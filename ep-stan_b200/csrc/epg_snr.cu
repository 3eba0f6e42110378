// Signal-to-noise statistics of the site updates: the inputs of the automatic damping selection
// (SURVEY 8f rank 1; reference experiment/find_damp.py:144-183 sweeps damping values off-line, and
// experiment/fit.py:176-186 hard-codes a schedule tuned for K <= 64 sites).
//
// At a fixed point of EP every site delta (dQi_k, dri_k) has zero expectation; what the K sites
// deliver is Monte Carlo noise of the moment estimates.  Far from the fixed point the deltas are
// coherent.  In the Fisher metric of the current global approximation N(m, S = Q^-1)
//     |(A, a)|^2 = 1/4 tr(S A S A) + 1/2 (a - A m)' S (a - A m)           (second-order KL)
// the kernels below return  sum_k |delta_k|^2  (this shard) and  |sum_k delta_k|^2  (after the
// all-reduce), from which the host estimates the fraction of the summed update that is signal.
#include "epg_internal.h"
#include "epg_linalg.cuh"

namespace {

// Q = L L' (packed lower, column by column) and m = Q^-1 r of the current global approximation
__global__ void k_fisher_prep(const double* __restrict__ Q, const double* __restrict__ r, double* __restrict__ Lp,
                              double* __restrict__ m, int* __restrict__ flag, int d) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Grp g;
    double* A = reinterpret_cast<double*>(smem_raw);
    double* vec = A + pk_size(d);
    for (int e = g.tid; e < d * d; e += g.n) {
        const int j = e / d, i = e - j * d;
        if (j >= i) A[pk(j, i, d)] = Q[e];
    }
    for (int i = g.tid; i < d; i += g.n) vec[i] = r[i];
    g.sync();
    const bool good = chol_packed(g, A, d);
    if (good) {
        for (int e = g.tid; e < pk_size(d); e += g.n) Lp[e] = A[e];
        fwd_solve_packed(g, A, vec, d);
        bwd_solve_packed(g, A, vec, d);
        for (int i = g.tid; i < d; i += g.n) m[i] = vec[i];
    }
    if (g.tid == 0) flag[0] = good ? 1 : 0;
}

// One CTA per delta (A = dQ, a = dr): out[b] = 1/4 |L^-1 A L^-T|_F^2 + 1/2 |L^-1 (a - A m)|^2.
// Y is a d x ld work matrix (ld odd: both access patterns below are bank-conflict free), in shared
// memory when it fits, else in global scratch (d > 128).
__global__ void k_fisher_norm(const double* __restrict__ dQ_all, const double* __restrict__ dr_all,
                              const double* __restrict__ Lp_g, const double* __restrict__ m_g,
                              double* __restrict__ out, double* __restrict__ Yglob, int y_in_smem, int d) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Grp g;
    const int ld = d | 1;
    double* L = reinterpret_cast<double*>(smem_raw);
    double* v = L + pk_size(d);
    double* mm = v + d;
    double* red = mm + d;
    double* Y = y_in_smem ? red + 48 : Yglob + (size_t)blockIdx.x * d * ld;
    const double* A = dQ_all + (size_t)blockIdx.x * d * d;
    const double* a = dr_all + (size_t)blockIdx.x * d;
    for (int e = g.tid; e < pk_size(d); e += g.n) L[e] = Lp_g[e];
    for (int i = g.tid; i < d; i += g.n) mm[i] = m_g[i];
    for (int e = g.tid; e < d * d; e += g.n) {
        const int j = e / d, i = e - j * d;
        Y[i * ld + j] = A[e];
    }
    __threadfence_block();
    g.sync();
    // v = a - A m  (A symmetric: row i of Y)
    for (int i = g.tid; i < d; i += g.n) {
        double acc = a[i];
        const double* row = Y + (size_t)i * ld;
        for (int j = 0; j < d; ++j) acc -= row[j] * mm[j];
        v[i] = acc;
    }
    g.sync();
    // stage 1: Y <- L^-1 Y, thread j owns column j (forward substitution down the rows)
    for (int j = g.tid; j < d; j += g.n) {
        for (int i = 0; i < d; ++i) {
            double acc0 = Y[i * ld + j], acc1 = 0.0;
            int idx = i;                                   // packed (i, l): l -> l+1 adds d - l - 1
            int l = 0;
            for (; l + 1 < i; l += 2) {
                acc0 -= L[idx] * Y[l * ld + j];
                const int idx1 = idx + d - l - 1;
                acc1 -= L[idx1] * Y[(l + 1) * ld + j];
                idx = idx1 + d - l - 2;
            }
            if (l < i) { acc0 -= L[idx] * Y[l * ld + j]; idx += d - l - 1; }
            Y[i * ld + j] = (acc0 + acc1) / L[idx];        // idx == pk(i, i)
        }
    }
    __threadfence_block();
    g.sync();
    // stage 2: rows of Y <- L^-1 (rows)', i.e. B = L^-1 A L^-T; thread j owns row j; sum of squares
    double ss = 0.0;
    for (int j = g.tid; j < d; j += g.n) {
        double* row = Y + (size_t)j * ld;
        for (int i = 0; i < d; ++i) {
            double acc0 = row[i], acc1 = 0.0;
            int idx = i;
            int l = 0;
            for (; l + 1 < i; l += 2) {
                acc0 -= L[idx] * row[l];
                const int idx1 = idx + d - l - 1;
                acc1 -= L[idx1] * row[l + 1];
                idx = idx1 + d - l - 2;
            }
            if (l < i) { acc0 -= L[idx] * row[l]; idx += d - l - 1; }
            const double z = (acc0 + acc1) / L[idx];
            row[i] = z;
            ss += z * z;
        }
    }
    const double trs = block_sum(g, ss, red);
    g.sync();
    fwd_solve_packed(g, L, v, d);
    double s2 = 0.0;
    for (int i = g.tid; i < d; i += g.n) s2 += v[i] * v[i];
    const double vs = block_sum(g, s2, red);
    if (g.tid == 0) out[blockIdx.x] = 0.25 * trs + 0.5 * vs;
}

// deterministic sum of n doubles (and count of non-zero flags) by one CTA
__global__ void k_sum_norms(const double* __restrict__ x, const int* __restrict__ ok, int n, double* __restrict__ out) {
    __shared__ double red[48];
    const Grp g;
    double s = 0.0, c = 0.0;
    for (int i = g.tid; i < n; i += g.n) {
        const bool good = ok[i] != 0;
        s += good ? x[i] : 0.0;
        c += good ? 1.0 : 0.0;
    }
    const double st = block_sum(g, s, red);
    const double ct = block_sum(g, c, red);
    if (g.tid == 0) { out[0] = st; out[1] = ct; }
}

__global__ void k_site_sum_partial2(const double* __restrict__ src, double* __restrict__ part, int K, int E, int ks) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const int kb = blockIdx.y * ks, ke = min(K, kb + ks);
    double s = 0.0;
    for (int k = kb; k < ke; ++k) s += src[(size_t)k * E + e];
    part[(size_t)blockIdx.y * E + e] = s;
}
__global__ void k_sum_chunks2(const double* __restrict__ part, double* __restrict__ out, int E, int nchunks) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    double s = 0.0;
    for (int c = 0; c < nchunks; ++c) s += part[(size_t)c * E + e];
    out[e] = s;
}

inline int fisher_threads(int d) { return d <= 64 ? 64 : (d <= 128 ? 128 : 256); }
inline size_t fisher_smem(int d, bool y_smem) {
    const size_t ld = (size_t)(d | 1);
    return sizeof(double) * ((size_t)pk_size(d) + 2 * (size_t)d + 48 + (y_smem ? (size_t)d * ld : 0));
}
inline size_t prep_smem(int d) { return sizeof(double) * ((size_t)pk_size(d) + 5 * (size_t)d + 48); }

#define SNR_LAUNCH_CHECK(c)                                                    \
    do {                                                                       \
        (c)->launches++;                                                       \
        cudaError_t _le = cudaGetLastError();                                  \
        if (_le != cudaSuccess) return epg_fail((c), "kernel launch", _le);    \
    } while (0)

// snr_buf layout (doubles): Lp[pk] | m[d] | norms[K+1] | flag (1) | chunk partials[nchunks*d*d] | Y slabs
struct SnrPlan {
    size_t o_L, o_m, o_norm, o_flag, o_part, o_Y, total;
    int nchunks, ks;
    bool y_smem;
};
SnrPlan snr_plan(int K, int d) {
    SnrPlan p;
    const size_t dd = (size_t)d * d;
    long want = (148L * 8 * 256) / (long)dd;
    if (want < 1) want = 1;
    if (want > K) want = K;
    p.ks = (int)((K + want - 1) / want);
    p.nchunks = (K + p.ks - 1) / p.ks;
    p.y_smem = fisher_smem(d, true) <= 200 * 1024;
    p.o_L = 0;
    p.o_m = p.o_L + pk_size(d);
    p.o_norm = p.o_m + d;
    p.o_flag = p.o_norm + K + 1;
    p.o_part = p.o_flag + 2;
    p.o_Y = p.o_part + (size_t)p.nchunks * dd;
    p.total = p.o_Y + (p.y_smem ? 0 : (size_t)K * d * (d | 1));
    return p;
}

// per site: mean of the draws, centred scatter and the outer product of the mean:
// out[k] = [m_k (d) | sum_t (x_t - m_k)(x_t - m_k)' (d*d) | m_k m_k' (d*d)]   (Master.mix_phi, method.py:1280-1298)
__global__ void k_site_scatter(const double* __restrict__ draws, int n, int d, double* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* mean = reinterpret_cast<double*>(smem_raw);
    const int k = blockIdx.x;
    const double* x = draws + (size_t)k * d * n;
    double* o = out + (size_t)k * (d + 2 * (size_t)d * d);
    for (int i = threadIdx.x; i < d; i += blockDim.x) {
        double s = 0.0;
        for (int t = 0; t < n; ++t) s += x[(size_t)i * n + t];
        mean[i] = s / n;
        o[i] = mean[i];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < d * d; e += blockDim.x) {
        const int j = e / d, i = e - j * d;
        if (j > i) continue;                                  // lower triangle, mirrored
        const double mi = mean[i], mj = mean[j];
        const double* xi = x + (size_t)i * n;
        const double* xj = x + (size_t)j * n;
        double a0 = 0.0, a1 = 0.0;
        int t = 0;
        for (; t + 2 <= n; t += 2) {
            a0 = fma(xi[t] - mi, xj[t] - mj, a0);
            a1 = fma(xi[t + 1] - mi, xj[t + 1] - mj, a1);
        }
        if (t < n) a0 = fma(xi[t] - mi, xj[t] - mj, a0);
        const double acc = a0 + a1;
        o[d + i + (size_t)j * d] = acc;
        o[d + j + (size_t)i * d] = acc;
        o[d + (size_t)d * d + i + (size_t)j * d] = mi * mj;
        o[d + (size_t)d * d + j + (size_t)i * d] = mi * mj;
    }
}

int launch_norms(epg_ctx* c, const SnrPlan& p, const double* dQ, const double* dr, double* out, int batch) {
    const int d = c->d;
    double* buf = c->snr_buf;
    const size_t sm = fisher_smem(d, p.y_smem);
    EPG_CHECK(c, cudaFuncSetAttribute((const void*)k_fisher_norm, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
    k_fisher_norm<<<batch, fisher_threads(d), sm, c->stream>>>(dQ, dr, buf + p.o_L, buf + p.o_m, out,
                                                                p.y_smem ? nullptr : buf + p.o_Y, p.y_smem ? 1 : 0, d);
    SNR_LAUNCH_CHECK(c);
    return 0;
}

}  // namespace

extern "C" {

int epg_delta_sums(epg_ctx* c) { return epg_delta_sums_ex(c, 1, nullptr, 0); }

int epg_delta_sums_ex(epg_ctx* c, int with_norms, const double* slots, int n_slots) {
    if (!c->arr[EPG_Q]) return epg_fail_msg(c, "state not initialised");
    if (n_slots < 0 || n_slots > EPG_XCHG_SLOTS || (n_slots > 0 && !slots)) return epg_fail_msg(c, "epg_delta_sums_ex: bad slots");
    const int d = c->d, K = c->K;
    const size_t dd = (size_t)d * d;
    const SnrPlan p = snr_plan(K, d);
    c->sums_valid = false;                                        // (until this call has completed)
    EPG_CHECK(c, epg_reserve((void**)&c->snr_buf, &c->snr_bytes, sizeof(double) * p.total));
    double* buf = c->snr_buf;
    int* flag = reinterpret_cast<int*>(buf + p.o_flag);
    const size_t psm = prep_smem(d);
    EPG_CHECK(c, cudaFuncSetAttribute((const void*)k_fisher_prep, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
    k_fisher_prep<<<1, d <= 32 ? 64 : (d <= 64 ? 128 : (d <= 128 ? 256 : 512)), psm, c->stream>>>(
        c->arr[EPG_Q], c->arr[EPG_R], buf + p.o_L, buf + p.o_m, flag, d);
    SNR_LAUNCH_CHECK(c);
    if (with_norms) {
        if (int rc = launch_norms(c, p, c->arr[EPG_DQI], c->arr[EPG_DRI], buf + p.o_norm, K)) return rc;
    } else {
        EPG_CHECK(c, cudaMemsetAsync(buf + p.o_norm, 0, sizeof(double) * (size_t)K, c->stream));
    }
    // the global (Q, r) these deltas refer to: epg_update_from_sums builds its proposals on them
    EPG_CHECK(c, epg_reserve((void**)&c->q_prev, &c->q_prev_bytes, sizeof(double) * (dd + d)));
    EPG_CHECK(c, cudaMemcpyAsync(c->q_prev, c->arr[EPG_Q], sizeof(double) * dd, cudaMemcpyDeviceToDevice, c->stream));
    EPG_CHECK(c, cudaMemcpyAsync(c->q_prev + dd, c->arr[EPG_R], sizeof(double) * d, cudaMemcpyDeviceToDevice, c->stream));
    // DSUM = [sum dQi | sum dri | sum |delta_k|^2 | n_ok | slots]   (failed sites hold zero deltas: method.py:460-465)
    double* dsum = c->arr[EPG_DSUM];
    {
        double h[EPG_XCHG_SLOTS];
        for (int i = 0; i < EPG_XCHG_SLOTS; ++i) h[i] = i < n_slots ? slots[i] : 0.0;
        EPG_CHECK(c, cudaMemcpyAsync(dsum + dd + d + 2, h, sizeof(h), cudaMemcpyHostToDevice, c->stream));
        EPG_CHECK(c, cudaStreamSynchronize(c->stream));             // (h is a local)
    }
    dim3 grid((unsigned)((dd + 255) / 256), p.nchunks);
    k_site_sum_partial2<<<grid, 256, 0, c->stream>>>(c->arr[EPG_DQI], buf + p.o_part, K, (int)dd, p.ks);
    SNR_LAUNCH_CHECK(c);
    k_sum_chunks2<<<(unsigned)((dd + 255) / 256), 256, 0, c->stream>>>(buf + p.o_part, dsum, (int)dd, p.nchunks);
    SNR_LAUNCH_CHECK(c);
    dim3 grid2((d + 255) / 256, p.nchunks);
    k_site_sum_partial2<<<grid2, 256, 0, c->stream>>>(c->arr[EPG_DRI], buf + p.o_part, K, d, p.ks);
    SNR_LAUNCH_CHECK(c);
    k_sum_chunks2<<<(d + 255) / 256, 256, 0, c->stream>>>(buf + p.o_part, dsum + dd, d, p.nchunks);
    SNR_LAUNCH_CHECK(c);
    k_sum_norms<<<1, 256, 0, c->stream>>>(buf + p.o_norm, c->site_ok, K, dsum + dd + d);
    SNR_LAUNCH_CHECK(c);
    c->sums_valid = true;
    return 0;
}

int epg_delta_snr(epg_ctx* c, double* stats_out) {
    if (!c->arr[EPG_Q] || !c->sums_valid) return epg_fail_msg(c, "epg_delta_snr: call epg_delta_sums(_ex) first");
    const int d = c->d, K = c->K;
    const size_t dd = (size_t)d * d;
    const SnrPlan p = snr_plan(K, d);
    double* buf = c->snr_buf;
    double* dsum = c->arr[EPG_DSUM];
    if (int rc = launch_norms(c, p, dsum, dsum + dd, buf + p.o_norm + K, 1)) return rc;
    double h[3];
    int hf = 0;
    EPG_CHECK(c, cudaMemcpyAsync(&h[0], buf + p.o_norm + K, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaMemcpyAsync(&h[1], dsum + dd + d, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaMemcpyAsync(&hf, buf + p.o_flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    if (!hf) return epg_fail_msg(c, "epg_delta_snr: the current global precision is not pos.def.");
    if (stats_out) { stats_out[0] = h[0]; stats_out[1] = h[1]; stats_out[2] = h[2]; }
    return 0;
}

// PARTIAL <- (Q_prev - Q0) + df * sum_k dQi  |  (r_prev - r0) + df * sum_k dri : what epg_update_finish adds to
// the prior, i.e. the proposal Q_prev + df * (summed site deltas), with no further exchange between the ranks
__global__ void k_partial_from_sums(const double* __restrict__ qprev, const double* __restrict__ Q0,
                                    const double* __restrict__ r0, const double* __restrict__ dsum,
                                    double* __restrict__ partial, double df, int d) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int dd = d * d;
    if (e >= dd + d) return;
    const double base = e < dd ? qprev[e] - Q0[e] : qprev[e] - r0[e - dd];
    partial[e] = base + df * dsum[e];
}

// Sums over the local sites of [m_k | scatter_k | m_k m_k'] of the phi draws in the device draw buffer
// (d + 2 d*d doubles): what Master.mix_phi pools (method.py:1250-1301); additive over ranks.
int epg_mix_phi_sums(epg_ctx* c, int n, double* sums_out) {
    if (!c->draws || n != c->draws_n || n < 2 || !sums_out) return epg_fail_msg(c, "epg_mix_phi_sums: no resident draws for this n");
    const int d = c->d, K = c->K;
    const size_t E = (size_t)d + 2 * (size_t)d * d;
    const SnrPlan p = snr_plan(K, d);
    const size_t need = sizeof(double) * (E * K + (size_t)p.nchunks * E + E);
    EPG_CHECK(c, epg_reserve((void**)&c->util_buf, &c->util_bytes, need));
    double* per = c->util_buf, *part = per + E * K, *tot = part + (size_t)p.nchunks * E;
    k_site_scatter<<<K, 256, sizeof(double) * d, c->stream>>>(c->draws, n, d, per);
    SNR_LAUNCH_CHECK(c);
    dim3 grid((unsigned)((E + 255) / 256), p.nchunks);
    k_site_sum_partial2<<<grid, 256, 0, c->stream>>>(per, part, K, (int)E, p.ks);
    SNR_LAUNCH_CHECK(c);
    k_sum_chunks2<<<(unsigned)((E + 255) / 256), 256, 0, c->stream>>>(part, tot, (int)E, p.nchunks);
    SNR_LAUNCH_CHECK(c);
    EPG_CHECK(c, cudaMemcpyAsync(sums_out, tot, sizeof(double) * E, cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int epg_update_from_sums(epg_ctx* c, double df) {
    if (!c->arr[EPG_Q] || !c->sums_valid) return epg_fail_msg(c, "epg_update_from_sums: call epg_delta_sums(_ex) first");
    const int d = c->d, E = d * d + d;
    k_partial_from_sums<<<(E + 255) / 256, 256, 0, c->stream>>>(c->q_prev, c->arr[EPG_Q0], c->arr[EPG_R0],
                                                               c->arr[EPG_DSUM], c->arr[EPG_PARTIAL], df, d);
    SNR_LAUNCH_CHECK(c);
    return 0;
}

}  // extern "C"

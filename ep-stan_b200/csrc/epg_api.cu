// C ABI of libepgpu (include/epgpu.h): context, device memory, dispatch.
#include "epg_internal.h"
#include <stdlib.h>
#include <string.h>
#include <vector>

size_t epg_array_site_stride(const epg_ctx* c, int a) {
    const size_t d = c->d;
    switch (a) {
        case EPG_QI: case EPG_QI2: case EPG_DQI: case EPG_CAVQ: return d * d;
        case EPG_RI: case EPG_RI2: case EPG_DRI: case EPG_CAVM: case EPG_TMEAN: return d;
        default: return 0;
    }
}

size_t epg_array_elems(const epg_ctx* c, int a) {
    const size_t d = c->d;
    const size_t st = epg_array_site_stride(c, a);
    if (st) return st * (size_t)c->K;
    switch (a) {
        case EPG_Q: case EPG_Q0: case EPG_S: return d * d;
        case EPG_R: case EPG_R0: case EPG_M: return d;
        case EPG_PARTIAL: return d * d + d + 1;
        case EPG_DSUM: return d * d + d + 2 + EPG_XCHG_SLOTS;
        default: return 0;
    }
}

int epg_fail(epg_ctx* c, const char* what, cudaError_t e) {
    if (c) c->err = std::string(what) + ": " + cudaGetErrorString(e);
    return -1;
}
int epg_fail_msg(epg_ctx* c, const std::string& msg) {
    if (c) c->err = msg;
    return -2;
}

cudaError_t epg_reserve(void** p, size_t* cap, size_t need) {
    if (*cap >= need && *p) return cudaSuccess;
    if (*p) { cudaError_t e = cudaFree(*p); *p = nullptr; *cap = 0; if (e != cudaSuccess) return e; }
    size_t want = need + need / 4 + 256;
    cudaError_t e = cudaMalloc(p, want);
    if (e == cudaSuccess) *cap = want;
    return e;
}

static int ensure_hflags(epg_ctx* c, size_t n) {
    if (c->h_flags_n >= n) return 0;
    if (c->h_flags) cudaFreeHost(c->h_flags);
    c->h_flags = nullptr;
    EPG_CHECK(c, cudaMallocHost((void**)&c->h_flags, sizeof(int32_t) * (n + 64)));
    c->h_flags_n = n + 64;
    return 0;
}

static void free_state(epg_ctx* c) {
    for (int a = 0; a < EPG_NARRAYS; ++a) { if (c->arr[a]) cudaFree(c->arr[a]); c->arr[a] = nullptr; }
    if (c->chol) cudaFree(c->chol); c->chol = nullptr;
    if (c->site_ok) cudaFree(c->site_ok); c->site_ok = nullptr;
    if (c->flags) cudaFree(c->flags); c->flags = nullptr;
    c->sums_valid = false;         // q_prev / snr_buf describe the old state (and may be too small for the new one)
}

extern void epg_sites_free(epg_ctx* c);

extern "C" {

int epg_version(void) { return EPG_VERSION; }

int epg_create(epg_ctx** out, int device, void* stream, int own_stream) {
    if (!out) return -2;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || device < 0 || device >= ndev) return -1;   // no CPU fallback: fail loudly
    if (cudaSetDevice(device) != cudaSuccess) return -1;
    epg_ctx* c = new epg_ctx();
    c->device = device;
    if (cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) c->num_sms = 148;
    { int l2 = 0; if (cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, device) == cudaSuccess && l2 > 0) c->l2_bytes = (size_t)l2; }
    if (!own_stream) { c->stream = (cudaStream_t)stream; c->own_stream = false; }
    else {
        if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return -1; }
        c->own_stream = true;
    }
    *out = c;
    return 0;
}

void epg_destroy(epg_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    free_state(c);
    epg_sites_free(c);
    if (c->draws) cudaFree(c->draws);
    if (c->scratch) cudaFree(c->scratch);
    if (c->util_buf) cudaFree(c->util_buf);
    if (c->snr_buf) cudaFree(c->snr_buf);
    if (c->mom_buf) cudaFree(c->mom_buf);
    if (c->q_prev) cudaFree(c->q_prev);
    if (c->h_flags) cudaFreeHost(c->h_flags);
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char* epg_last_error(const epg_ctx* c) { return c ? c->err.c_str() : "null context"; }

int epg_sync(epg_ctx* c) {
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int64_t epg_launch_count(const epg_ctx* c) { return c ? c->launches : 0; }

int epg_init_state(epg_ctx* c, int K, int d) {
    if (K < 1 || d < 1) return epg_fail_msg(c, "epg_init_state: K and d must be positive");
    if (d > 200) return epg_fail_msg(c, "epg_init_state: d > 200 exceeds the shared-memory resident design");
    EPG_CHECK(c, cudaSetDevice(c->device));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    free_state(c);
    c->K = K; c->d = d;
    for (int a = 0; a < EPG_NARRAYS; ++a) {
        const size_t n = epg_array_elems(c, a);
        if (!n) continue;
        EPG_CHECK(c, cudaMalloc((void**)&c->arr[a], sizeof(double) * n));
        EPG_CHECK(c, cudaMemsetAsync(c->arr[a], 0, sizeof(double) * n, c->stream));
    }
    EPG_CHECK(c, cudaMalloc((void**)&c->chol, sizeof(double) * (size_t)d * (d + 1) / 2));
    EPG_CHECK(c, cudaMalloc((void**)&c->site_ok, sizeof(int) * (size_t)K));
    EPG_CHECK(c, cudaMemsetAsync(c->site_ok, 0, sizeof(int) * (size_t)K, c->stream));   // no site has a result yet
    EPG_CHECK(c, cudaMalloc((void**)&c->flags, sizeof(int) * 8));
    EPG_CHECK(c, cudaMemsetAsync(c->flags, 0, sizeof(int) * 8, c->stream));
    if (ensure_hflags(c, (size_t)K + 8)) return -1;
    return 0;
}

static int check_range(epg_ctx* c, int a, int& k0, int& k1, size_t& off, size_t& cnt) {
    if (a < 0 || a >= EPG_NARRAYS || !c->arr[a]) return epg_fail_msg(c, "bad array id or state not initialised");
    const size_t st = epg_array_site_stride(c, a);
    if (st) {
        if (k0 < 0 || k1 > c->K || k0 >= k1) return epg_fail_msg(c, "bad site range");
        off = st * (size_t)k0; cnt = st * (size_t)(k1 - k0);
    } else { off = 0; cnt = epg_array_elems(c, a); }
    return 0;
}

int epg_upload(epg_ctx* c, int a, int k0, int k1, const double* host) {
    size_t off, cnt;
    if (int rc = check_range(c, a, k0, k1, off, cnt)) return rc;
    EPG_CHECK(c, cudaMemcpyAsync(c->arr[a] + off, host, sizeof(double) * cnt, cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int epg_download(epg_ctx* c, int a, int k0, int k1, double* host) {
    size_t off, cnt;
    if (int rc = check_range(c, a, k0, k1, off, cnt)) return rc;
    EPG_CHECK(c, cudaMemcpyAsync(host, c->arr[a] + off, sizeof(double) * cnt, cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int64_t epg_array_count(epg_ctx* c, int a, int k0, int k1) {
    if (!c || a < 0 || a >= EPG_NARRAYS) return -1;
    const size_t st = epg_array_site_stride(c, a);
    return (int64_t)(st ? st * (size_t)(k1 - k0) : epg_array_elems(c, a));
}

void* epg_device_ptr(epg_ctx* c, int a) {
    if (!c || a < 0 || a >= EPG_NARRAYS) return nullptr;
    return c->arr[a];
}

// copy `n` ints of site_ok[k0..] (or flags) to the host and wait
static int read_ints(epg_ctx* c, const int* dev, size_t n, int32_t* dst) {
    if (ensure_hflags(c, n)) return -1;
    EPG_CHECK(c, cudaMemcpyAsync(c->h_flags, dev, sizeof(int) * n, cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    if (dst) memcpy(dst, c->h_flags, sizeof(int32_t) * n);
    return 0;
}

int epg_cavity(epg_ctx* c, int k0, int k1, int proposal, int32_t* posdef_out, int* all_ok) {
    if (!c->arr[EPG_Q] || k0 < 0 || k1 > c->K || k0 >= k1) return epg_fail_msg(c, "epg_cavity: bad range/state");
    EPG_CHECK(c, epg_launch_cavity(c, k0, k1, proposal));
    if (int rc = read_ints(c, c->site_ok + k0, (size_t)(k1 - k0), posdef_out)) return rc;
    if (all_ok) {
        int ok = 1;
        for (int i = 0; i < k1 - k0; ++i) ok &= (c->h_flags[i] != 0);
        *all_ok = ok;
    }
    return 0;
}

static int reserve_draws(epg_ctx* c, int n) {
    const size_t need = (size_t)c->K * c->d * n;
    if (need > c->draws_cap || n != c->draws_n) {
        if (need > c->draws_cap) {
            if (c->draws) EPG_CHECK(c, cudaFree(c->draws));
            c->draws = nullptr; c->draws_cap = 0;
            EPG_CHECK(c, cudaMalloc((void**)&c->draws, sizeof(double) * need));
            c->draws_cap = need;
        }
        c->draws_n = n;
    }
    return 0;
}

int epg_reserve_draws(epg_ctx* c, int n) { return reserve_draws(c, n); }

int epg_set_draws(epg_ctx* c, int k0, int k1, int n, const double* draws) {
    if (!c->arr[EPG_Q] || k0 < 0 || k1 > c->K || k0 >= k1 || n < 1) return epg_fail_msg(c, "epg_set_draws: bad args");
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    if (int rc = reserve_draws(c, n)) return rc;
    const size_t st = (size_t)c->d * n;
    EPG_CHECK(c, cudaMemcpyAsync(c->draws + st * k0, draws, sizeof(double) * st * (k1 - k0),
                                 cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int epg_get_draws(epg_ctx* c, int k0, int k1, int n, double* draws) {
    if (!c->draws || n != c->draws_n || k0 < 0 || k1 > c->K || k0 >= k1) return epg_fail_msg(c, "epg_get_draws: bad args");
    const size_t st = (size_t)c->d * n;
    EPG_CHECK(c, cudaMemcpyAsync(draws, c->draws + st * k0, sizeof(double) * st * (k1 - k0),
                                 cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int epg_moments(epg_ctx* c, int k0, int k1, int n, int prec_estim, int32_t* ok_out, int* n_ok) {
    if (!c->draws || n != c->draws_n || k0 < 0 || k1 > c->K || k0 >= k1)
        return epg_fail_msg(c, "epg_moments: draws not resident for this n / bad range");
    if (prec_estim != EPG_PREC_SAMPLE && prec_estim != EPG_PREC_OLSE)
        return epg_fail_msg(c, "Invalid value for option `prec_estim`");
    EPG_CHECK(c, epg_launch_moments(c, k0, k1, n, prec_estim));
    if (int rc = read_ints(c, c->site_ok + k0, (size_t)(k1 - k0), ok_out)) return rc;
    if (n_ok) {
        int cnt = 0;
        for (int i = 0; i < k1 - k0; ++i) cnt += (c->h_flags[i] != 0);
        *n_ok = cnt;
    }
    return 0;
}

int epg_fail_sites(epg_ctx* c, int n, const int32_t* sites) {
    if (!c->arr[EPG_Q] || n < 0 || (n > 0 && !sites)) return epg_fail_msg(c, "epg_fail_sites: bad args/state");
    const size_t d = c->d;
    for (int i = 0; i < n; ++i) {
        const int k = sites[i];
        if (k < 0 || k >= c->K) return epg_fail_msg(c, "epg_fail_sites: bad site index");
        EPG_CHECK(c, cudaMemsetAsync(c->arr[EPG_DQI] + d * d * k, 0, sizeof(double) * d * d, c->stream));
        EPG_CHECK(c, cudaMemsetAsync(c->arr[EPG_DRI] + d * k, 0, sizeof(double) * d, c->stream));
        EPG_CHECK(c, cudaMemsetAsync(c->site_ok + k, 0, sizeof(int), c->stream));
    }
    return 0;
}

int epg_update_partial(epg_ctx* c, double df) {
    if (!c->arr[EPG_Q]) return epg_fail_msg(c, "state not initialised");
    EPG_CHECK(c, epg_launch_update_partial(c, df));
    return 0;
}

int epg_update_finish(epg_ctx* c, int* posdef) {
    if (!c->arr[EPG_Q]) return epg_fail_msg(c, "state not initialised");
    EPG_CHECK(c, epg_launch_update_finish(c));
    int32_t f = 0;
    if (int rc = read_ints(c, c->flags, 1, &f)) return rc;
    if (posdef) *posdef = f;
    return 0;
}

int epg_accept(epg_ctx* c) {
    if (!c->arr[EPG_Q]) return epg_fail_msg(c, "state not initialised");
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    double* t = c->arr[EPG_QI]; c->arr[EPG_QI] = c->arr[EPG_QI2]; c->arr[EPG_QI2] = t;
    t = c->arr[EPG_RI]; c->arr[EPG_RI] = c->arr[EPG_RI2]; c->arr[EPG_RI2] = t;
    return 0;
}

int epg_global_moments(epg_ctx* c, double* m_out, double* S_out) {
    if (!c->arr[EPG_Q]) return epg_fail_msg(c, "state not initialised");
    EPG_CHECK(c, epg_launch_global_moments(c));
    const size_t d = c->d;
    if (m_out) EPG_CHECK(c, cudaMemcpyAsync(m_out, c->arr[EPG_M], sizeof(double) * d, cudaMemcpyDeviceToHost, c->stream));
    if (S_out) EPG_CHECK(c, cudaMemcpyAsync(S_out, c->arr[EPG_S], sizeof(double) * d * d, cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int epg_force_pd(epg_ctx* c, double thr, double min_eig, int32_t* forced_out, double* lam_out) {
    if (!c->arr[EPG_Q]) return epg_fail_msg(c, "state not initialised");
    EPG_CHECK(c, epg_reserve((void**)&c->util_buf, &c->util_bytes, sizeof(double) * (size_t)c->K));
    EPG_CHECK(c, epg_launch_force_pd(c, thr, min_eig, c->util_buf));
    if (lam_out) EPG_CHECK(c, cudaMemcpyAsync(lam_out, c->util_buf, sizeof(double) * c->K, cudaMemcpyDeviceToHost, c->stream));
    return read_ints(c, c->site_ok, (size_t)c->K, forced_out);
}

int epg_damp_sweep(epg_ctx* c, int n_df, const double* dfs, const double* m_tgt, const double* S_tgt,
                   double* mse_out, double* kl_out) {
    if (!c->arr[EPG_Q] || n_df < 1) return epg_fail_msg(c, "epg_damp_sweep: bad args/state");
    const size_t d = c->d;
    const size_t n_in = (size_t)n_df + d + d * d, n_out = 3 * (size_t)n_df;
    EPG_CHECK(c, epg_reserve((void**)&c->util_buf, &c->util_bytes, sizeof(double) * (n_in + n_out)));
    double* dfs_d = c->util_buf;
    double* tgt_d = dfs_d + n_df;
    double* out_d = tgt_d + d + d * d;
    EPG_CHECK(c, cudaMemcpyAsync(dfs_d, dfs, sizeof(double) * n_df, cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, cudaMemcpyAsync(tgt_d, m_tgt, sizeof(double) * d, cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, cudaMemcpyAsync(tgt_d + d, S_tgt, sizeof(double) * d * d, cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, epg_launch_damp_sweep(c, n_df, dfs_d, tgt_d, out_d));
    if (mse_out) EPG_CHECK(c, cudaMemcpyAsync(mse_out, out_d, sizeof(double) * n_df, cudaMemcpyDeviceToHost, c->stream));
    if (kl_out) EPG_CHECK(c, cudaMemcpyAsync(kl_out, out_d + n_df, sizeof(double) * n_df, cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int epg_invert_normal_params(epg_ctx* c, int batch, int d, const double* A, const double* b, int cho_form,
                             double* out_A, double* out_b, int32_t* ok) {
    if (batch < 1 || d < 1 || d > 200 || !A || !out_A) return epg_fail_msg(c, "epg_invert_normal_params: bad args");
    const size_t dd = (size_t)d * d, nA = dd * batch, nb = (size_t)d * batch;
    const size_t ints = (batch + 1) / 2 + 1;
    EPG_CHECK(c, epg_reserve((void**)&c->util_buf, &c->util_bytes, sizeof(double) * (2 * nA + 2 * nb + ints)));
    double* dA = c->util_buf; double* dO = dA + nA; double* db = dO + nA; double* dob = db + nb;
    int* dok = reinterpret_cast<int*>(dob + nb);
    EPG_CHECK(c, cudaMemcpyAsync(dA, A, sizeof(double) * nA, cudaMemcpyHostToDevice, c->stream));
    if (b) EPG_CHECK(c, cudaMemcpyAsync(db, b, sizeof(double) * nb, cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, epg_launch_invert(c, batch, d, dA, b ? db : nullptr, cho_form, dO, dob, dok));
    EPG_CHECK(c, cudaMemcpyAsync(out_A, dO, sizeof(double) * nA, cudaMemcpyDeviceToHost, c->stream));
    if (b && out_b) EPG_CHECK(c, cudaMemcpyAsync(out_b, dob, sizeof(double) * nb, cudaMemcpyDeviceToHost, c->stream));
    return read_ints(c, dok, (size_t)batch, ok);
}

int epg_olse(epg_ctx* c, int batch, int d, const double* S, int n, const double* P, double* out, int32_t* ok) {
    if (batch < 1 || d < 1 || d > 200 || !S || !out) return epg_fail_msg(c, "epg_olse: bad args");
    const size_t nA = (size_t)d * d * batch;
    const size_t ints = (batch + 1) / 2 + 1;
    EPG_CHECK(c, epg_reserve((void**)&c->util_buf, &c->util_bytes, sizeof(double) * (3 * nA + ints)));
    double* dS = c->util_buf; double* dP = dS + nA; double* dO = dP + nA;
    int* dok = reinterpret_cast<int*>(dO + nA);
    EPG_CHECK(c, cudaMemcpyAsync(dS, S, sizeof(double) * nA, cudaMemcpyHostToDevice, c->stream));
    if (P) EPG_CHECK(c, cudaMemcpyAsync(dP, P, sizeof(double) * nA, cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, epg_launch_olse(c, batch, d, dS, n, P ? dP : nullptr, dO, dok));
    EPG_CHECK(c, cudaMemcpyAsync(out, dO, sizeof(double) * nA, cudaMemcpyDeviceToHost, c->stream));
    return read_ints(c, dok, (size_t)batch, ok);
}

}  // extern "C"

// Batched adaptive NUTS on the tilted densities of all sites x chains.
//
// Replaces the sampling half of Worker.tilted (reference epstan/method.py:338-408,
// _sample_stan :43-118, util.stan_sample_time util.py:692-724), i.e. one PyStan
// 2.17 `StanModel.sampling` call per site per EP iteration, by ONE persistent
// kernel launch: one CTA per site, all chains of the site advanced in lock-step
// at the granularity of a gradient evaluation ("tick").
//
//   tick = [per-chain warps]  consume the previous gradient, run the NUTS state
//                             machine until the chain needs the next gradient
//          [whole CTA]        likelihood pass for all chains at once:
//                               F = X B'      (rows x chains)      "forward"
//                               E = y - sigmoid(F), lp += y F - softplus(F)
//                               G = E' X      (chains x inputs)    "backward"
//                             X_k is read ONCE per tick for both products; it
//                             stays resident in shared memory when it fits,
//                             otherwise it is streamed L2->smem with cp.async
//                             double buffering.
//
// The densities are those of experiment/models/m{1,3,4}b[_sg].stan (see
// oracle/density.py for the formulas); the sampler is Stan 2.17's adaptive
// diag_e NUTS (multinomial trajectory sampling, generalised U-turn criterion,
// dual-averaging step size, windowed variance adaptation) restated as an
// iterative (stack based) tree builder so that it runs without recursion.
// Arithmetic: fp32 for positions/momenta/gradients and the two contractions,
// fp64 for the energies used in the accept/multinomial weights.
#include "epg_internal.h"
#include "epg_common.cuh"
#include <cuda.h>
#include <cuda_bf16.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <cmath>
#include <vector>

#define NTHR 256
#define NWARP (NTHR / 32)
#define MAXDEPTH_CAP 12
#define NCMAX 4

// ---------------------------------------------------------------------------
// site data
// ---------------------------------------------------------------------------
struct epg_site_data {
    int model = 0, D = 0, S = 0;        // S: padded row stride (floats), column D holds 1.0
    int K = 0;
    int64_t N = 0;
    float* X = nullptr;                 // [N][S]
    __nv_bfloat16* Xb = nullptr;        // [N][xb_pitch] bf16 copy for the tensor-core passes (column D = 1)
    int nkc = 1, xb_pitch = 64;         // 64-column sub-tiles per tile; row pitch: 64 (D+1 <= 64) or D+1 rounded up to 16
    float* gout_w = nullptr;            // wide pass scratch [K][2][32][256]
    float* xmean = nullptr;             // [K][64 nkc] per-site column means the bf16 copy is centred on (0 beyond column D-1)
    int* order = nullptr;               // [K] launch order of the sites: most expensive (gradient evaluations of the
    std::vector<double> h_cost;         //     previous run, h_cost) first, so that stragglers do not start last
    unsigned char* reinit = nullptr;    // [K] 1: the next init_prev run starts this site's chains at random (epg_reinit_sites)
    std::vector<unsigned char> h_reinit;
    float* inits = nullptr;             // [K][inits_C][Pmax] starting points of init mode "given" (epg_set_inits), NaN: random
    int inits_C = 0;
    std::vector<unsigned char> h_inits_set;   // [K] 1: epg_set_inits covered the site
    CUtensorMap tmap;                   // TMA descriptor of Xb: box 64 columns x 128 rows, 128-byte swizzle
    bool tc_ok = false;                 // tensor-core passes usable (single group, D+1 <= 256)
    int use_tc = 1;                     // option (epg_set_option "use_tc")
    double* tstats = nullptr;           // [K][2][P] per-site mean and sum of squared deviations of the transformed
    size_t tstats_bytes = 0;            //     parameters over the last run's draws (option "param_stats", Master.mix_pred)
    int param_stats = 0;
    int carry_adapt = 1;                // option "carry_adapt": init_prev runs start from the previous run's adapted metric / step size
    int pp_mode = 0;                    // option "pingpong": 0 never (default), 1 when sites > SMs and L2-resident, 2 always
    float metric_reg = 1e-3f;           // option "metric_reg": identity weight of the regularised dense_e window estimate
    float* y = nullptr;                 // [N]
    int64_t* row0 = nullptr;            // [K+1]
    int* grp_ptr = nullptr;             // [K+1] offsets into grp_rows
    int* grp_rows = nullptr;            // per site: J+1 row offsets relative to the site start
    std::vector<int64_t> h_row0;
    std::vector<int> h_J, h_p;
    int Pmax = 0, Jmax = 0;
    int64_t max_rows = 0;
    // sampler state
    float* chain_mem = nullptr;         // [K*C][NVEC][P]
    size_t chain_mem_bytes = 0;
    float* last_q = nullptr;            // [K*C][P] last draw of every chain (init_prev), then last_minv, last_eps, last_metric
    size_t last_q_bytes = 0;
    int last_C = 0;
    float* omega = nullptr;             // [K][d*d] fp32 copy of the cavity precision
    size_t omega_bytes = 0;
    double* out = nullptr;              // per-site analytics
    size_t out_bytes = 0;
    double* ld_buf = nullptr;           // logdensity staging
    size_t ld_bytes = 0;
    float* dense = nullptr;             // dense_e state [K*C][dense_floats(P)] (first dense_e run on)
    size_t dense_bytes = 0;
    double* dense_ws = nullptr;         // dense_e window-end factorisation scratch [K*C][P][P]
    size_t dense_ws_bytes = 0;
    int32_t plan[EPG_PLAN_FIELDS] = {}; // launch plan of the last epg_tilted_sample / epg_logdensity (epg_last_plan)
    // HMC diagnostics (epg_get_hmc_diag, epg_get_sampler_params)
    void* hmc = nullptr;                // HmcChain [K*hmc_C]
    int hmc_C = 0;
    std::vector<unsigned char> h_hmc_ok;      // [K] 1: the site's most recent run wrote its diagnostics
    int sampler_params = 0;             // option "sampler_params": record every transition
    double* rec = nullptr;              // [K][hmc_C][rec_n][HMC_REC]
    size_t rec_bytes = 0;
    int rec_iter = 0, rec_warmup = 0, rec_thin = 0, rec_n = 0, rec_nw = 0;   // shape of the records
    std::vector<unsigned char> h_rec_ok;      // [K] 1: the site's most recent run recorded
};

void epg_sites_free(epg_ctx* c) {
    epg_site_data* s = c->sites;
    if (!s) return;
    cudaFree(s->xmean); cudaFree(s->gout_w); cudaFree(s->order); cudaFree(s->reinit); cudaFree(s->tstats);
    cudaFree(s->X); cudaFree(s->Xb); cudaFree(s->y); cudaFree(s->row0); cudaFree(s->grp_ptr); cudaFree(s->grp_rows);
    cudaFree(s->chain_mem); cudaFree(s->last_q); cudaFree(s->omega); cudaFree(s->out); cudaFree(s->ld_buf);
    cudaFree(s->dense); cudaFree(s->dense_ws); cudaFree(s->inits); cudaFree(s->hmc); cudaFree(s->rec);
    delete s;
    c->sites = nullptr;
}

namespace {

__host__ __device__ inline bool model_four(int model) { return model == EPG_M4B || model == EPG_M5B; }
__host__ __device__ inline int model_dphi(int model, int D) {
    return model_four(model) ? 2 * D + 2 : (model == EPG_M2B ? 2 : D + 1);
}
// sampled parameters q = [phi (d) | eta (J) | etb]: etb is absent (m1b), one vector per site (m2b) or per group
__host__ __device__ inline int model_np(int model, int D, int J) {
    return model_dphi(model, D) + J + (model == EPG_M1B ? 0 : (model == EPG_M2B ? D : J * D));
}

__global__ void k_convert_x(const double* __restrict__ src, float* __restrict__ dst, int64_t rows, int D, int S) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * S) return;
    const int64_t r = idx / S;
    const int c = (int)(idx - r * S);
    dst[idx] = c < D ? (float)src[r * D + c] : (c == D ? 1.0f : 0.0f);
}
// bf16 copy for the tensor-core pass, CENTRED per site: dst = bf16(x - mean_k[col]) for the D input columns
// (column D stays 1, the rest 0).  bf16 keeps 8 significant bits: a column like 35.5 +- 0.02 (the simulators
// shift the inputs of groups with extreme intercepts, common.py:132-317) would otherwise lose all of its
// within-site variation.  The means re-enter exactly: f = (alpha + c'beta) + (x - c)'beta and
// G_col = sum_n e_n (x - c)_col + c_col sum_n e_n  (coefficient build / chain rule of likelihood_pass_tc).
__global__ void k_convert_xb(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t rows, int S, int D,
                             const float* __restrict__ xmean, const int64_t* __restrict__ row0, int K, int pitch,
                             int xm_stride) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= rows * pitch) return;
    const int64_t r = idx / pitch;
    const int c = (int)(idx - r * pitch);
    float v = c < S ? src[r * S + c] : 0.0f;
    if (c < D) {
        int lo = 0, hi = K;                       // site of row r: row0[lo] <= r < row0[lo + 1]
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (row0[mid] <= r) lo = mid; else hi = mid; }
        v -= xmean[(size_t)lo * xm_stride + c];
    }
    dst[idx] = __float2bfloat16(v);
}
__global__ void k_convert_y(const int64_t* __restrict__ src, float* __restrict__ dst, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[i] ? 1.0f : 0.0f;
}

// ---------------------------------------------------------------------------
// RNG: Philox4x32-10, counter based.  key = (site seed, chain), counter =
// (draw index, element, purpose).  Every lane of a warp can evaluate it
// independently and get identical streams.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += 0x9E3779B9u;
        key.y += 0xBB67AE85u;
    }
    return ctr;
}
// purposes: 1 tree uniforms, 2 momenta, 3 random inits, 4 step-size jitter, 5 re-initialisation around the cavity
__device__ __forceinline__ float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }
__device__ __forceinline__ float rng_uniform(uint2 key, uint32_t& ctr) {
    const uint4 r = philox4x32(make_uint4(ctr++, 0u, 1u, 0u), key);
    return u01(r.x);
}
__device__ __forceinline__ float rng_normal(uint2 key, uint32_t ctr, uint32_t elem) {
    const uint4 r = philox4x32(make_uint4(ctr, elem, 2u, 0u), key);
    const float u1 = u01(r.x), u2 = u01(r.y);
    return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

__device__ __forceinline__ double log_sum_exp(double a, double b) {
    if (a == -INFINITY) return b;
    if (b == -INFINITY) return a;
    // the correction term is < log 2: single precision is ample for it
    const double m = fmax(a, b);
    return m + (double)log1pf(__expf(-(float)fabs(a - b)));
}

// per-chain vectors (stride P floats).  The first `hot_nvec` of them (ordered by
// how often a tick touches them) live in shared memory, the rest in global memory.
enum {
    V_Q = 0,                      // working point z: position
    V_GL,                         // likelihood-gradient output of the batched pass
    V_G, V_P,                     // working point: gradient of the potential, momentum
    V_MINV,                       // inverse metric (diag)
    V_CRHO, V_CPSL,               // node being built: rho and left-end p_sharp
    V_QPROP, V_GPROP,             // proposal of the node being built
    V_RHO,                        // sum of momenta over the trajectory
    V_QS, V_GS,                   // current sample
    V_QM, V_PM, V_GM,             // minus end of the trajectory
    V_QP, V_PP, V_GP,             // plus end
    V_NHOT,                       // ---- vectors below are always in global memory ----
    V_WMEAN = V_NHOT, V_WM2,      // Welford accumulators
    V_RS0, V_RQ0, V_RS1, V_RQ1,   // split-Rhat sums / sums of squares per half
    V_TREF, V_TS, V_TQ,           // transformed parameters (alpha, beta): first draw, sums and sums of squares about it
    V_STACK                       // + 4*level : psl, rho, qprop, gprop
};
#define NVEC (V_STACK + 4 * MAXDEPTH_CAP)

enum { PH_START = 0, PH_START_WAIT, PH_SS_WAIT, PH_TREE_WAIT, PH_DONE, PH_DEAD };
// starting points: the public init modes of epg_sampler_opts (0-3), and the re-initialisation around the cavity
// of a site marked by epg_reinit_sites
enum { IM_RANDOM = 0, IM_ZERO = 1, IM_PREV = 2, IM_GIVEN = 3, IM_REINIT = 4 };

struct ChainS {
    int phase, iter, depth, nleaf, sign, n_leap_tr, ss_dir, ss_first, init_tries, restart_ss;
    int carried;                  // the warm-up started from the previous run's adapted metric / step size
    int init_mode;                // SamplerArgs::init_mode, or IM_REINIT for a site marked by epg_reinit_sites
    uint32_t rng;
    float eps;
    double V, H0, Vs, lsw, sum_metro, cur_lsw, Vprop;
    // dual averaging
    double s_bar, x_bar, mu;
    int da_count;
    // variance windows
    int win_count, win_next, win_size, w_n;
    float eps_tr;                 // step size of the current transition: eps (the nominal step size) with jitter applied
    // analytics
    double eps_sum;
    long long n_leap_total;
    int n_div;
};
// (the shared-memory plan is built from this size: new fields go into the two 4-byte alignment holes)
static_assert(sizeof(ChainS) == 184, "ChainS layout");
// per-level scalars of the tree stack live in shared memory next to ChainS
struct ChainStack { double lsw[MAXDEPTH_CAP], V[MAXDEPTH_CAP]; };
// HMC diagnostics of a chain, in global memory (the shared-memory plan has no room for them): the Hamiltonian
// H(q, p) of the current sample and of the proposal pending at each tree-stack level (energy__ is H of the
// selected sample), and the summary of the saved post-warm-up transitions.  Written by lane 0.
struct HmcChain {
    double Hs, Hstk[MAXDEPTH_CAP];
    double e0, se, see, sdd, eprev;     // energies: the first saved one, sums of E - e0, of (E - e0)^2, of
                                        // (E_t - E_t-1)^2, the previous one
    double n_saved, n_div, n_maxd, ebfmi;   // the EPG_DIAG_FIELDS of epg_get_hmc_diag, in order
};
#define HMC_REC 6                       // values of a per-transition record (PyStan's get_sampler_params order)

struct SamplerArgs {
    // site data
    const float* X; const float* y; const int64_t* row0; const int* grp_ptr; const int* grp_rows;
    const float* xmean;                // [K][64] column means of the centred bf16 copy (tensor-core pass)
    const int* order;                  // launch order: block b samples site k0 + order[b] (nullptr: identity)
    const unsigned char* reinit;       // [K] per local site: start the chains at random although init_mode == 2 (nullptr: none)
    int model, D, S, d;
    // cavity
    const double* cavQ; const double* cavm; float* omega;
    // chains
    float* chain_mem; float* last_q; int P, C;
    float* last_minv; float* last_eps;  // [K*C][P], [K*C]: adapted metric / step size at the end of the previous run
    float* last_metric;                 // [K*C]: the metric (EPG_METRIC_*) of that run
    int carry_adapt;                    // init_prev also starts the warm-up from them (option "carry_adapt")
    int metric;                         // EPG_METRIC_*
    float* dense; double* dense_ws;     // dense_e: per-chain state (dense_floats) and fp64 scratch [K*C][P][P]
    float metric_reg;                   // dense_e window estimate: n/(n+5) C + metric_reg 5/(n+5) I
    int iter, warmup, init_mode, max_depth;
    double delta;
    int win_init, win_term, win_base;
    double gamma, kappa, t0;           // dual averaging (epg_sampler_adapt)
    float stepsize, jitter, init_r;    // starting nominal step size, step-size jitter, radius of random inits
    int adapt_engaged;                 // 0: no step-size heuristic, dual averaging or metric windows
    int thin, n_save;                  // post-warm-up transition m is saved when m % thin == 0; n_save per chain
    const float* inits;                // init mode "given": [K][C][P] starting points, NaN = random
    const uint32_t* seeds;
    // outputs
    double* draws; int n_draws;     // [K][d][n]
    double* tstats;                 // [K][2][P] or nullptr (see epg_site_data)
    double* out;                    // [K][8]: mean eps, max rhat, n_leapfrog, n_divergent, clk chain, clk lik, ticks, -
    HmcChain* hmc;                  // [K*C] HMC diagnostics (always)
    double* rec;                    // [K][C][n_rec][HMC_REC] per-transition records (option "sampler_params"), or nullptr
    int n_rec, n_rec_warm;          // records per chain: ceil(warmup / thin) warm-up ones, then the n_save saved ones
    int k0;
    // shared-memory plan
    int R, resident, slices, NC, combos;
    float* gout_w;                     // wide tensor-core pass: [K][2][32][256] likelihood-gradient halves (global scratch)
    float* cavc_g;                     // wide pass: cavity terms [K][32][d] in global memory (shared memory goes to the TMA ring)
    int nkc, xm_stride;                // 64-column sub-tiles per tile; stride of xmean (64 * nkc)
    int use_tc, tc_nst, pp, hot_nvec, hot_levels, omega_smem;     // use_tc: 0 SIMT, 1 tensor-core pass, 2 wide tensor-core pass; tc_nst: X/E stages of the tensor-core pass     // hot_levels: tree-stack levels kept in shared memory
    size_t off_E, off_B, off_G, off_gphi, off_cavc, off_lp, off_cs, off_hot, off_omega, smem_total;
    size_t site_stride;                // ping-pong kernel: distance between the two per-site blocks
};

// One site as a CTA sees it: its index and the base of its block of shared memory (the per-site offsets of
// SamplerArgs are relative to `sm`; the ping-pong kernel keeps two such blocks).
struct SiteView { unsigned char* sm; int k; uint32_t off = 0; };   // off: sm minus the start of dynamic shared memory

__device__ __forceinline__ float* cvec(const SamplerArgs& a, const SiteView& sv, int c_local, int v) {
    const bool hot = v < a.hot_nvec;
    const bool hot_stack = v >= V_STACK && v < V_STACK + 4 * a.hot_levels;
    if (hot || hot_stack) {
        const int per_chain = a.hot_nvec + 4 * a.hot_levels;
        const int slot = hot ? v : a.hot_nvec + (v - V_STACK);
        return reinterpret_cast<float*>(sv.sm + a.off_hot) + ((size_t)c_local * per_chain + slot) * a.P;
    }
    return a.chain_mem + ((size_t)(sv.k * a.C + c_local) * NVEC + v) * a.P;
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// Bernoulli-logit pieces from ONE exp, ONE log and ONE reciprocal:
//   t = exp(-|f|);  softplus(f) = max(f,0) + log(1+t);  sigmoid(f) = f>=0 ? 1/(1+t) : t/(1+t)
// returns y*f - softplus(f) and writes e = y - sigmoid(f)
__device__ __forceinline__ float logit_terms(float f, float yv, float& e) {
    const float t = __expf(-fabsf(f));
    const float inv = __fdividef(1.0f, 1.0f + t);
    const float sg = f >= 0.0f ? inv : t * inv;
    e = yv - sg;
    return yv * f - (fmaxf(f, 0.0f) + __logf(1.0f + t));
}

#include "epg_lik_tc.cuh"
#include "epg_lik_tcw.cuh"

// shared-memory load through the shared window (ld.shared).  The pointers the sampler works with are generic
// (a vector lives in shared OR global memory depending on the launch plan), and generic loads take the L1TEX
// path: measured ~200 cycles per dependent step against ~30 for ld.shared.  Only for data that no thread
// writes while the caller runs (no memory clobber: the compiler may schedule the loads freely).
__device__ __forceinline__ float lds_ro(uint32_t saddr) {
    float v;
    asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(saddr));
    return v;
}

// Cavity term of every chain, c = Omega (phi - mu), by the whole CTA (one (chain,row)
// dot product per thread) into shared memory; consumed by finish_gradient.
__device__ __forceinline__ void cavity_term(const SamplerArgs& a, unsigned char* smem, const float* om, const float* muf,
                                            int k_local, int nchains, int nthr_workers) {
    float* cavc = a.cavc_g ? a.cavc_g + (size_t)k_local * tcw::NCH * a.d : reinterpret_cast<float*>(smem + a.off_cavc);
    const int d = a.d;
    const bool in_smem = a.omega_smem && a.hot_nvec > V_Q;
    for (int e = threadIdx.x; e < nchains * d; e += nthr_workers) {
        const int c = e / d, i = e - c * d;
        const float* q = cvec(a, SiteView{smem, k_local}, c, V_Q);
        // eight independent loads and four accumulators per step: the loop is latency-bound otherwise
        float acc0 = 0.0f, acc1 = 0.0f, acc2 = 0.0f, acc3 = 0.0f;
        int j = 0;
        if (in_smem) {
            const uint32_t oc = tc::smem_u32(om + i), qs = tc::smem_u32(q), ms = tc::smem_u32(muf);
            const uint32_t dd = 4u * (uint32_t)d;
            for (; j + 3 < d; j += 4) {
                const uint32_t ob = oc + (uint32_t)j * dd, jb = 4u * (uint32_t)j;
                const float o0 = lds_ro(ob), o1 = lds_ro(ob + dd), o2 = lds_ro(ob + 2 * dd), o3 = lds_ro(ob + 3 * dd);
                const float x0 = lds_ro(qs + jb) - lds_ro(ms + jb), x1 = lds_ro(qs + jb + 4) - lds_ro(ms + jb + 4);
                const float x2 = lds_ro(qs + jb + 8) - lds_ro(ms + jb + 8), x3 = lds_ro(qs + jb + 12) - lds_ro(ms + jb + 12);
                acc0 = fmaf(o0, x0, acc0); acc1 = fmaf(o1, x1, acc1);
                acc2 = fmaf(o2, x2, acc2); acc3 = fmaf(o3, x3, acc3);
            }
            for (; j < d; ++j)
                acc0 = fmaf(lds_ro(oc + (uint32_t)j * dd), lds_ro(qs + 4u * j) - lds_ro(ms + 4u * j), acc0);
        } else {
            const float* oc = om + i;
            for (; j + 3 < d; j += 4) {
                const float o0 = oc[(size_t)j * d], o1 = oc[(size_t)(j + 1) * d];
                const float o2 = oc[(size_t)(j + 2) * d], o3 = oc[(size_t)(j + 3) * d];
                const float x0 = q[j] - muf[j], x1 = q[j + 1] - muf[j + 1];
                const float x2 = q[j + 2] - muf[j + 2], x3 = q[j + 3] - muf[j + 3];
                acc0 = fmaf(o0, x0, acc0); acc1 = fmaf(o1, x1, acc1);
                acc2 = fmaf(o2, x2, acc2); acc3 = fmaf(o3, x3, acc3);
            }
            for (; j < d; ++j) acc0 = fmaf(oc[(size_t)j * d], q[j] - muf[j], acc0);
        }
        cavc[e] = (acc0 + acc2) + (acc1 + acc3);
    }
}

// ---------------------------------------------------------------------------
// Likelihood pass for all chains of one site: fills V_GL (likelihood part of
// grad log p wrt every sampled parameter) and lp_out[c] (likelihood log-density).
// ---------------------------------------------------------------------------
template <int CP>
__device__ void likelihood_pass(const SamplerArgs& a, unsigned char* smem, int site, int k_local, int nchains,
                                int J, int64_t row_begin, int n_rows, const int* grows, double* lp_out,
                                const float* om, const float* muf) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int S = a.S, D = a.D, d = a.d, model = a.model;
    float* Xs = reinterpret_cast<float*>(smem);
    float* Et = reinterpret_cast<float*>(smem + a.off_E);
    float* Bm = reinterpret_cast<float*>(smem + a.off_B);
    float* Gp = reinterpret_cast<float*>(smem + a.off_G);
    float* gphi = reinterpret_cast<float*>(smem + a.off_gphi);
    double* lpw = reinterpret_cast<double*>(smem + a.off_lp);      // [NWARP][CP]
    const int R = a.R;
    const int S4 = S >> 2;
    const int chain0 = k_local * a.C;
    const bool four = model_four(model);
    const int ia = four ? 1 : 0;                                    // index of log sigma_a in phi
    const int ib = four ? 2 + D : 1;                                // start of log sigma_b (m2b: the one scale)

    for (int e = tid; e < CP * d; e += NTHR) gphi[e] = 0.0f;
    if (model == EPG_M2B)                                           // slope gradient accumulates over the groups
        for (int e = tid; e < nchains * D; e += NTHR) {
            const int c = e / D, col = e - c * D;
            cvec(a, SiteView{smem, k_local}, c, V_GL)[d + J + col] = 0.0f;
        }
    cavity_term(a, smem, om, muf, k_local, nchains, NTHR);
    float lpacc[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) lpacc[c] = 0.0f;

    // B2 work assignment
    const int combos = a.combos, slices = a.slices, NC = a.NC;
    const int my_slice = (NC == 1) ? tid / combos : 0;
    const bool b2_active = (NC > 1) || (my_slice < slices);
    const int combo0 = (NC == 1) ? tid % combos : tid;

    int tile_parity = 0;
    for (int j = 0; j < J; ++j) {
        const int g_begin = grows[j], g_end = grows[j + 1];
        // ---- coefficients of group j: Bm[c][0..D) = beta_j(c), Bm[c][D] = alpha_j(c) ----
        __syncthreads();
        for (int e = tid; e < CP * S; e += NTHR) {
            const int c = e / S, col = e - c * S;
            float v = 0.0f;
            if (c < nchains && col <= D) {
                const float* q = cvec(a, SiteView{smem, k_local}, c, V_Q);
                if (col == D) {
                    const float sa = __expf(q[ia]);
                    v = q[d + j] * sa + (four ? q[0] : 0.0f);
                } else if (model == EPG_M1B) {
                    v = q[1 + col];
                } else if (model == EPG_M2B) {
                    v = q[d + J + col] * __expf(q[ib]);
                } else {
                    const float etb = q[d + J + j * D + col];
                    v = etb * __expf(q[ib + col]) + (four ? q[2 + col] : 0.0f);
                }
            }
            Bm[e] = v;
        }
        float acc[NCMAX][16];
#pragma unroll
        for (int u = 0; u < NCMAX; ++u)
#pragma unroll
            for (int q = 0; q < 16; ++q) acc[u][q] = 0.0f;

        const int n_tiles = (g_end - g_begin + R - 1) / R;
        // streaming: prefetch the first tile of the group
        if (!a.resident && n_tiles > 0) {
            const int rows = min(R, g_end - g_begin);
            const float4* src = reinterpret_cast<const float4*>(a.X + (size_t)(row_begin + g_begin) * S);
            float4* dst = reinterpret_cast<float4*>(Xs + (size_t)tile_parity * R * S);
            for (int e = tid; e < rows * S4; e += NTHR) cp_async16(dst + e, src + e);
            cp_async_commit();
        }
        for (int t = 0; t < n_tiles; ++t) {
            const int r0 = g_begin + t * R;
            const int rows = min(R, g_end - r0);
            const float* Xt;
            if (a.resident) {
                Xt = Xs + (size_t)r0 * S;
                __syncthreads();                       // Bm ready / previous tile's Et consumed
            } else {
                cp_async_wait<0>();
                __syncthreads();                       // tile t landed; everyone left tile t-1
                if (t + 1 < n_tiles) {
                    const int rows_n = min(R, g_end - (r0 + R));
                    const float4* src = reinterpret_cast<const float4*>(a.X + (size_t)(row_begin + r0 + R) * S);
                    float4* dst = reinterpret_cast<float4*>(Xs + (size_t)(tile_parity ^ 1) * R * S);
                    for (int e = tid; e < rows_n * S4; e += NTHR) cp_async16(dst + e, src + e);
                    cp_async_commit();
                }
                Xt = Xs + (size_t)tile_parity * R * S;
                tile_parity ^= 1;
            }
            // ---- B1: F = X B', E = y - sigmoid(F), lp ----
            if (tid < rows) {
                float f[CP];
#pragma unroll
                for (int c = 0; c < CP; ++c) f[c] = 0.0f;
                const float4* xr = reinterpret_cast<const float4*>(Xt + (size_t)tid * S);
                for (int i = 0; i < S4; ++i) {
                    const float4 x = xr[i];
#pragma unroll
                    for (int c = 0; c < CP; ++c) {
                        const float4 b = reinterpret_cast<const float4*>(Bm + c * S)[i];
                        f[c] = fmaf(x.x, b.x, fmaf(x.y, b.y, fmaf(x.z, b.z, fmaf(x.w, b.w, f[c]))));
                    }
                }
                const float yv = a.y[row_begin + r0 + tid];
#pragma unroll
                for (int c = 0; c < CP; ++c) {
                    float e;
                    lpacc[c] += logit_terms(f[c], yv, e);
                    f[c] = e;
                }
#pragma unroll
                for (int c4 = 0; c4 < CP / 4; ++c4)
                    reinterpret_cast<float4*>(Et + (size_t)tid * CP)[c4] =
                        make_float4(f[4 * c4], f[4 * c4 + 1], f[4 * c4 + 2], f[4 * c4 + 3]);
            }
            __syncthreads();
            // ---- B2: G += E' X  (4 inputs x 4 chains register tiles) ----
            if (b2_active) {
#pragma unroll
                for (int u = 0; u < NCMAX; ++u) {
                    const int combo = combo0 + u * NTHR;
                    if (u < NC && combo < combos) {
                        const int dq = combo % S4, cg = combo / S4;
                        for (int r = my_slice; r < rows; r += slices) {
                            const float4 x = reinterpret_cast<const float4*>(Xt + (size_t)r * S)[dq];
                            const float4 e = reinterpret_cast<const float4*>(Et + (size_t)r * CP)[cg];
                            acc[u][0] = fmaf(x.x, e.x, acc[u][0]);   acc[u][1] = fmaf(x.x, e.y, acc[u][1]);
                            acc[u][2] = fmaf(x.x, e.z, acc[u][2]);   acc[u][3] = fmaf(x.x, e.w, acc[u][3]);
                            acc[u][4] = fmaf(x.y, e.x, acc[u][4]);   acc[u][5] = fmaf(x.y, e.y, acc[u][5]);
                            acc[u][6] = fmaf(x.y, e.z, acc[u][6]);   acc[u][7] = fmaf(x.y, e.w, acc[u][7]);
                            acc[u][8] = fmaf(x.z, e.x, acc[u][8]);   acc[u][9] = fmaf(x.z, e.y, acc[u][9]);
                            acc[u][10] = fmaf(x.z, e.z, acc[u][10]); acc[u][11] = fmaf(x.z, e.w, acc[u][11]);
                            acc[u][12] = fmaf(x.w, e.x, acc[u][12]); acc[u][13] = fmaf(x.w, e.y, acc[u][13]);
                            acc[u][14] = fmaf(x.w, e.z, acc[u][14]); acc[u][15] = fmaf(x.w, e.w, acc[u][15]);
                        }
                    }
                }
            }
        }
        // ---- group end: G_part[slice][c][col] ----
        __syncthreads();
        if (b2_active) {
#pragma unroll
            for (int u = 0; u < NCMAX; ++u) {
                const int combo = combo0 + u * NTHR;
                if (u < NC && combo < combos) {
                    const int dq = combo % S4, cg = combo / S4;
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const int col = 4 * dq + (q >> 2), c = 4 * cg + (q & 3);
                        Gp[((size_t)my_slice * CP + c) * S + col] = acc[u][q];
                    }
                }
            }
        }
        __syncthreads();
        // ---- fixed-order slice reduction + chain rule of group j ----
        for (int e = tid; e < CP * S; e += NTHR) {
            const int c = e / S, col = e - c * S;
            if (c >= nchains || col > D) continue;
            float gsum = 0.0f;
            for (int sl = 0; sl < slices; ++sl) gsum += Gp[((size_t)sl * CP + c) * S + col];
            const float* q = cvec(a, SiteView{smem, k_local}, c, V_Q);
            float* gl = cvec(a, SiteView{smem, k_local}, c, V_GL);
            if (col == D) {
                // s_j = sum_n e_n
                const float sa = __expf(q[ia]);
                const float eta = q[d + j];
                gl[d + j] = sa * gsum;
                gphi[c * d + ia] += sa * eta * gsum;      // (c, col) pairs own distinct slots
                if (four) gphi[c * d + 0] += gsum;
            } else if (model == EPG_M1B) {
                gphi[c * d + 1 + col] += gsum;
            } else if (model == EPG_M2B) {
                gl[d + J + col] += __expf(q[ib]) * gsum;  // d/d etb = sigma_b sum_j g_j (log sigma_b: below)
            } else {
                const float sb = __expf(q[ib + col]);
                const float etb = q[d + J + j * D + col];
                gl[d + J + j * D + col] = sb * gsum;
                gphi[c * d + ib + col] += sb * etb * gsum;
                if (four) gphi[c * d + 2 + col] += gsum;
            }
        }
    }
    // ---- lp reduction (fp64) and phi gradient write-back ----
#pragma unroll
    for (int c = 0; c < CP; ++c) {
        const double v = warp_sum((double)lpacc[c]);
        if (lane == 0) lpw[warp * CP + c] = v;
    }
    __syncthreads();
    if (tid < nchains) {
        double s = 0.0;
        for (int w = 0; w < NWARP; ++w) s += lpw[w * CP + tid];
        lp_out[tid] = s;
        if (model == EPG_M2B) {
            // d/d log sigma_b = sum_i etb_i (sigma_b g_i), in a fixed order
            const float* q = cvec(a, SiteView{smem, k_local}, tid, V_Q);
            const float* gl = cvec(a, SiteView{smem, k_local}, tid, V_GL);
            float acc = 0.0f;
            for (int col = 0; col < D; ++col) acc = fmaf(q[d + J + col], gl[d + J + col], acc);
            gphi[tid * d + ib] = acc;
        }
    }
    __syncthreads();
    for (int e = tid; e < CP * d; e += NTHR) {
        const int c = e / d, i = e - c * d;
        if (c < nchains) cvec(a, SiteView{smem, k_local}, c, V_GL)[i] = gphi[e];
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------
// Tensor-core variant of the likelihood pass (single-group sites, D+1 <= 64,
// <= 16 chains): see epg_lik_tc.cuh.  Same outputs as likelihood_pass.
// ---------------------------------------------------------------------------
// barrier over the tc::NTHREADS likelihood threads only (== the whole CTA except in the ping-pong kernel)
__device__ __forceinline__ void lik_group_sync() { asm volatile("bar.sync 1, %0;\n" ::"n"(tc::NTHREADS) : "memory"); }

__device__ void likelihood_pass_tc(const SamplerArgs& a, unsigned char* smem, unsigned char* tcb, uint32_t tmem_base,
                                   const CUtensorMap* tmap, tc::State& st, int k_local, int nchains,
                                   int64_t row_begin, int n_rows, double* lp_out, const float* om, const float* muf) {
    const int tid = threadIdx.x;
    const bool worker = tid < NTHR;                  // warps 8, 9, 10 only drive MMA / TMA inside the pass
    const int D = a.D, d = a.d, model = a.model;
    double* lpw = reinterpret_cast<double*>(smem + a.off_lp);       // [NWARP][8]
    const int chain0 = k_local * a.C;
    const bool four = model_four(model);
    const int ia = four ? 1 : 0;
    const int ib = four ? 2 + D : 1;
    PROF_T(q0);
    const float* xm = a.xmean + (size_t)k_local * tc::KW;            // column means of the centred design matrix
    if (worker) {
        // coefficient operands B = B_hi + B_lo (bf16 each), K-major interleaved layout; one warp per chain,
        // lane l builds columns l and l + 32.  The design matrix is centred, so the intercept coefficient
        // (column D, which multiplies 1) carries the mean term:  alpha + sum_col mean_col * beta_col.
        const int lane = tid & 31;
        for (int c = tid >> 5; c < nchains; c += NWARP) {          // (rows of unused chains stay zero from setup)
            const float* q = cvec(a, SiteView{smem, k_local}, c, V_Q);
            float v[2];
            float mterm = 0.0f;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int col = lane + 32 * h;
                float b = 0.0f;
                if (col < D) {
                    if (model == EPG_M1B) b = q[1 + col];
                    else if (model == EPG_M2B) b = q[d + 1 + col] * __expf(q[ib]);
                    else b = q[d + 1 + col] * __expf(q[ib + col]) + (four ? q[2 + col] : 0.0f);
                    mterm = fmaf(xm[col], b, mterm);
                }
                v[h] = b;
            }
            mterm = warp_sum(mterm);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int col = lane + 32 * h;
                if (col == D) v[h] = q[d] * __expf(q[ia]) + (four ? q[0] : 0.0f) + mterm;
                const __nv_bfloat16 hi = __float2bfloat16(v[h]);
                const __nv_bfloat16 lo = __float2bfloat16(v[h] - __bfloat162float(hi));
                const int cc = tc::chain_col(c);
                *reinterpret_cast<__nv_bfloat16*>(tcb + tc::Smem::BM + tc::interleave_off32(cc, col)) = hi;
                *reinterpret_cast<__nv_bfloat16*>(tcb + tc::Smem::BM + tc::interleave_off32(tc::NCH + cc, col)) = lo;
            }
        }
        tc::fence_proxy_async();
    }
    lik_group_sync();
    PROF_T(q1);
    const int ksteps = (D + 1 + 15) / 16;           // 16 input columns per tcgen05.mma
    // the cavity term is independent of the pass: the epilogue warps compute it while the
    // first tiles are in flight
    auto prologue = [&]() { cavity_term(a, smem, om, muf, k_local, nchains, NTHR); };
    if (nchains <= 4) tc::pass<4>(tcb, tmem_base, tmap, st, row_begin, n_rows, ksteps, a.y, lpw, prologue);
    else if (nchains <= 8) tc::pass<8>(tcb, tmem_base, tmap, st, row_begin, n_rows, ksteps, a.y, lpw, prologue);
    else tc::pass<16>(tcb, tmem_base, tmap, st, row_begin, n_rows, ksteps, a.y, lpw, prologue);
    PROF_T(q2);
    lik_group_sync();
    PROF_T(q3);
    if (worker) {
        // chain rule (single group: every slot of the likelihood gradient gets exactly one term)
        const float* gout = reinterpret_cast<const float*>(tcb + tc::Smem::GOUT);
        for (int e = tid; e < nchains * tc::KW; e += NTHR) {
            const int c = e / tc::KW, col = e - c * tc::KW;
            if (col > D) continue;
            float gsum = gout[tc::chain_col(c) * tc::KW + col] + gout[(tc::NCH + tc::chain_col(c)) * tc::KW + col];
            if (col < D)                                   // centred inputs: + mean_col * sum_n e_n
                gsum = fmaf(xm[col], gout[tc::chain_col(c) * tc::KW + D] + gout[(tc::NCH + tc::chain_col(c)) * tc::KW + D], gsum);
            const float* q = cvec(a, SiteView{smem, k_local}, c, V_Q);
            float* gl = cvec(a, SiteView{smem, k_local}, c, V_GL);
            if (col == D) {
                const float sa = __expf(q[ia]);
                gl[d] = sa * gsum;
                gl[ia] = sa * q[d] * gsum;
                if (four) gl[0] = gsum;
            } else if (model == EPG_M1B) {
                gl[1 + col] = gsum;
            } else if (model == EPG_M2B) {
                gl[d + 1 + col] = __expf(q[ib]) * gsum;       // (log sigma_b: below, one thread per chain)
            } else {
                const float sb = __expf(q[ib + col]);
                const float etb = q[d + 1 + col];
                gl[d + 1 + col] = sb * gsum;
                gl[ib + col] = sb * etb * gsum;
                if (four) gl[2 + col] = gsum;
            }
        }
        if (tid < nchains) {
            double sum = 0.0;
            for (int w = 0; w < NWARP; ++w) sum += lpw[w * tc::NCH + tc::chain_col(tid)];
            lp_out[tid] = sum;
            if (model == EPG_M2B) {
                // d/d log sigma_b = sigma_b sum_i etb_i g_i, in a fixed order
                const float* gout = reinterpret_cast<const float*>(tcb + tc::Smem::GOUT);
                const float* q = cvec(a, SiteView{smem, k_local}, tid, V_Q);
                float acc = 0.0f;
                const float se = gout[tc::chain_col(tid) * tc::KW + D] + gout[(tc::NCH + tc::chain_col(tid)) * tc::KW + D];
                for (int col = 0; col < D; ++col)
                    acc = fmaf(q[d + 1 + col], fmaf(xm[col], se, gout[tc::chain_col(tid) * tc::KW + col] +
                                                                 gout[(tc::NCH + tc::chain_col(tid)) * tc::KW + col]), acc);
                cvec(a, SiteView{smem, k_local}, tid, V_GL)[ib] = __expf(q[ib]) * acc;
            }
        }
    }
    lik_group_sync();
    PROF_T(q4);
#ifdef EPG_TC_PROFILE
    if (threadIdx.x == 0) { PROF2_ADD(2, q0, q1); PROF2_ADD(3, q1, q2); PROF2_ADD(4, q2, q3); PROF2_ADD(5, q3, q4); PROF2_ADD(6, 0, 1); }
#endif
}

// ---------------------------------------------------------------------------
// Wide tensor-core variant (single-group sites, D+1 <= 256, <= 32 chains; config 5): see epg_lik_tcw.cuh.
// Same outputs as likelihood_pass.  The chain vectors may live in global memory here (generic pointers).
// ---------------------------------------------------------------------------
__device__ void likelihood_pass_tcw(const SamplerArgs& a, unsigned char* smem, unsigned char* tcb, uint32_t tmem_base,
                                    const CUtensorMap* tmap, tcw::State& st, int k_local, int nchains,
                                    int64_t row_begin, int n_rows, double* lp_out, const float* om, const float* muf) {
    const int tid = threadIdx.x;
    const bool worker = tid < NTHR;
    const int D = a.D, d = a.d, model = a.model;
    double* lpw = reinterpret_cast<double*>(smem + a.off_lp);       // [NWARP][32]
    const bool four = model_four(model);
    const int ia = four ? 1 : 0;
    const int ib = four ? 2 + D : 1;
    const int ncol = a.nkc * tc::KW;
    const float* xm = a.xmean + (size_t)k_local * a.xm_stride;
    float* gout = a.gout_w + (size_t)k_local * 2 * tcw::NCH * tcw::KWT;
    if (worker) {
        // coefficient operand B = B_hi + B_lo (bf16 each); one warp per chain, lane l builds columns l + 32 h.
        // Centred design matrix: the intercept coefficient (column D) carries  alpha + sum_col mean_col * beta_col.
        const int lane = tid & 31;
        for (int c = tid >> 5; c < nchains; c += NWARP) {
            const float* q = cvec(a, SiteView{smem, k_local}, c, V_Q);
            float v[tcw::KWT / 32];
            float mterm = 0.0f;
#pragma unroll
            for (int h = 0; h < tcw::KWT / 32; ++h) {
                const int col = lane + 32 * h;
                float b = 0.0f;
                if (col < D) {
                    if (model == EPG_M1B) b = q[1 + col];
                    else if (model == EPG_M2B) b = q[d + 1 + col] * __expf(q[ib]);
                    else b = q[d + 1 + col] * __expf(q[ib + col]) + (four ? q[2 + col] : 0.0f);
                    mterm = fmaf(xm[col], b, mterm);
                }
                v[h] = b;
            }
            mterm = warp_sum(mterm);
#pragma unroll
            for (int h = 0; h < tcw::KWT / 32; ++h) {
                const int col = lane + 32 * h;
                if (col >= ncol) continue;
                if (col == D) v[h] = q[d] * __expf(q[ia]) + (four ? q[0] : 0.0f) + mterm;
                const __nv_bfloat16 hi = __float2bfloat16(v[h]);
                const __nv_bfloat16 lo = __float2bfloat16(v[h] - __bfloat162float(hi));
                *reinterpret_cast<__nv_bfloat16*>(tcb + tcw::Smem::BM + tcw::b_off(c, col)) = hi;
                *reinterpret_cast<__nv_bfloat16*>(tcb + tcw::Smem::BM + tcw::b_off(tcw::NCH + c, col)) = lo;
            }
        }
        tc::fence_proxy_async();
    }
    lik_group_sync();
    const int ksteps = (D + 1 + 15) / 16;
    auto prologue = [&]() { cavity_term(a, smem, om, muf, k_local, nchains, NTHR); };
    tcw::pass(tcb, tmem_base, tmap, st, row_begin, n_rows, a.nkc, ksteps, a.y, lpw, gout, prologue);
    lik_group_sync();
    if (worker) {
        // chain rule (single group: every slot of the likelihood gradient gets exactly one term)
        const float* g0 = gout;
        const float* g1 = gout + (size_t)tcw::NCH * tcw::KWT;
        for (int e = tid; e < nchains * ncol; e += NTHR) {
            const int c = e / ncol, col = e - c * ncol;
            if (col > D) continue;
            const float se = g0[c * tcw::KWT + D] + g1[c * tcw::KWT + D];            // sum_n e_n
            float gsum = g0[c * tcw::KWT + col] + g1[c * tcw::KWT + col];
            if (col < D) gsum = fmaf(xm[col], se, gsum);                             // centred inputs
            const float* q = cvec(a, SiteView{smem, k_local}, c, V_Q);
            float* gl = cvec(a, SiteView{smem, k_local}, c, V_GL);
            if (col == D) {
                const float sa = __expf(q[ia]);
                gl[d] = sa * gsum;
                gl[ia] = sa * q[d] * gsum;
                if (four) gl[0] = gsum;
            } else if (model == EPG_M1B) {
                gl[1 + col] = gsum;
            } else if (model == EPG_M2B) {
                gl[d + 1 + col] = __expf(q[ib]) * gsum;       // (log sigma_b: below, one thread per chain)
            } else {
                const float sb = __expf(q[ib + col]);
                const float etb = q[d + 1 + col];
                gl[d + 1 + col] = sb * gsum;
                gl[ib + col] = sb * etb * gsum;
                if (four) gl[2 + col] = gsum;
            }
        }
        if (tid < nchains) {
            double sum = 0.0;
            for (int w = 0; w < NWARP; ++w) sum += lpw[w * tcw::NCH + tid];
            lp_out[tid] = sum;
            if (model == EPG_M2B) {
                // d/d log sigma_b = sigma_b sum_i etb_i g_i, in a fixed order
                const float* q = cvec(a, SiteView{smem, k_local}, tid, V_Q);
                float acc = 0.0f;
                const float se = g0[tid * tcw::KWT + D] + g1[tid * tcw::KWT + D];
                for (int col = 0; col < D; ++col)
                    acc = fmaf(q[d + 1 + col], fmaf(xm[col], se, g0[tid * tcw::KWT + col] + g1[tid * tcw::KWT + col]), acc);
                cvec(a, SiteView{smem, k_local}, tid, V_GL)[ib] = __expf(q[ib]) * acc;
            }
        }
    }
    lik_group_sync();
}

// ---------------------------------------------------------------------------
// per-chain (one warp) helpers
// ---------------------------------------------------------------------------
// ALLHOT = true (tensor-core kernels): the launch plan guarantees that every hot vector, the cavity term and
// the cavity mean live in shared memory; they are then addressed through the __shared__ symbol so that the
// compiler emits ld.shared / st.shared instead of generic loads (which take the L1TEX path: ~50 cycles more
// per dependent access, and the chain phase is one long dependency chain).
// DENSE = true: the chain runs Stan's dense_e metric; its p x p matrices and the p_sharp vectors of the
// trajectory live in the dense_e block (global memory), which the diag_e / unit_e instances never touch.
//   dense block of a chain: [Sigma][U^-1 stored by columns][window co-moment] (P x P each), then
//   p_sharp of the working point, of the minus end and of the plus end (P each)
enum { DN_SIGMA = 0, DN_UINV, DN_W2 };
enum { DV_PSH = 0, DV_PSM, DV_PSP };
__host__ __device__ inline size_t dense_floats(int P) { return 3 * (size_t)P * P + 3 * (size_t)P; }

template <bool ALLHOT, bool DENSE = false>
struct ChainCtxT {
    static constexpr bool kDense = DENSE;
    const SamplerArgs& a;
    int cg;          // global chain index (k_local*C + c)
    int p, d, J, D, lane;
    uint2 key;
    const float* omega;   // [d*d] fp32 cavity precision
    const float* muf_;    // [d] fp32 cavity mean
    ChainStack* stk;      // shared memory
    const float* cavc_;   // [d] cavity term Omega (phi - mu) of this chain (shared memory)
    float* hot;           // this chain's block of shared-memory vectors (hot vectors, then hot stack levels)
    float* cold;          // this chain's vectors in global memory
    uint32_t hot_off, cavc_off, muf_off;      // the same three as byte offsets into dynamic shared memory
    float* dn;            // dense_e block of this chain (DENSE only)
    double* ws;           // dense_e fp64 factorisation scratch [P][P] (DENSE only)
    __device__ __forceinline__ float* dm(int which) const { return dn + (size_t)which * a.P * a.P; }
    __device__ __forceinline__ float* dv(int which) const { return dn + 3 * (size_t)a.P * a.P + (size_t)which * a.P; }
    __device__ __forceinline__ float* v(int which) const {
        if constexpr (ALLHOT) {
            extern __shared__ __align__(1024) unsigned char smem_dyn[];
            float* h = reinterpret_cast<float*>(smem_dyn + hot_off);
            if (which < V_NHOT) return h + which * a.P;
            if (which >= V_STACK && which < V_STACK + 4 * a.hot_levels) return h + (V_NHOT + which - V_STACK) * a.P;
            return cold + (size_t)which * a.P;
        } else {
            if (which < a.hot_nvec) return hot + which * a.P;
            if (which >= V_STACK && which < V_STACK + 4 * a.hot_levels) return hot + (a.hot_nvec + which - V_STACK) * a.P;
            return cold + (size_t)which * a.P;
        }
    }
    __device__ __forceinline__ const float* cavc() const {
        if constexpr (ALLHOT) {
            extern __shared__ __align__(1024) unsigned char smem_dyn[];
            return reinterpret_cast<const float*>(smem_dyn + cavc_off);
        } else return cavc_;
    }
    __device__ __forceinline__ const float* muf() const {
        if constexpr (ALLHOT) {
            extern __shared__ __align__(1024) unsigned char smem_dyn[];
            return reinterpret_cast<const float*>(smem_dyn + muf_off);
        } else return muf_;
    }
};
template <bool ALLHOT, bool DENSE = false>
__device__ __forceinline__ ChainCtxT<ALLHOT, DENSE> make_chain_ctx(const SamplerArgs& a, const SiteView& sv, int c_local,
                                                                   int p, int d, int J, int D, int lane, uint2 key,
                                                                   const float* om, const float* muf, ChainStack* stk) {
    const int cg = sv.k * a.C + c_local;
    float* hot = cvec(a, sv, c_local, 0);    // slot 0 of the chain's shared block (when hot_nvec > 0)
    float* cold = a.chain_mem + (size_t)cg * NVEC * a.P;
    const float* cavc = (a.cavc_g ? a.cavc_g + (size_t)sv.k * tcw::NCH * d
                                  : reinterpret_cast<const float*>(sv.sm + a.off_cavc)) + (size_t)c_local * d;
    const uint32_t per_chain = (uint32_t)(a.hot_nvec + 4 * a.hot_levels);
    const uint32_t hot_off = sv.off + (uint32_t)a.off_hot + (uint32_t)c_local * per_chain * (uint32_t)a.P * 4u;
    const uint32_t cavc_off = sv.off + (uint32_t)a.off_cavc + (uint32_t)(c_local * d) * 4u;
    const uint32_t muf_off = sv.off + (uint32_t)a.off_omega + (uint32_t)(d * d) * 4u;
    float* dn = nullptr;
    double* ws = nullptr;
    if constexpr (DENSE) {
        dn = a.dense + (size_t)cg * dense_floats(a.P);
        ws = a.dense_ws + (size_t)cg * a.P * a.P;
    }
    return ChainCtxT<ALLHOT, DENSE>{a, cg, p, d, J, D, lane, key, om, muf, stk, cavc, hot, cold, hot_off, cavc_off,
                                    muf_off, dn, ws};
}

template <class CX>
__device__ __forceinline__ void vcopy(const CX& x, int dst, int src) {
    float4* D_ = reinterpret_cast<float4*>(x.v(dst));
    const float4* S_ = reinterpret_cast<const float4*>(x.v(src));
    for (int i = x.lane; 4 * i < x.p; i += 32) D_[i] = S_[i];       // vectors are padded to P (multiple of 32)
}
// the same for the p_sharp vectors of the dense_e block
template <class CX>
__device__ __forceinline__ void dcopy(const CX& x, int dst, int src) {
    float4* D_ = reinterpret_cast<float4*>(x.dv(dst));
    const float4* S_ = reinterpret_cast<const float4*>(x.dv(src));
    for (int i = x.lane; 4 * i < x.p; i += 32) D_[i] = S_[i];
}

// dense_e: out = M v on the chain's warp.  Entry (i, j) of M is stored at M[j P + i] (M symmetric, or stored
// by columns), so for each j the lanes read P consecutive floats while v_j is a broadcast: p^2/32 FMAs per lane.
// `upper`: entry (i, j) is zero for j < i, and the sum over j starts at the first row of the lane's chunk.
// The sum runs over increasing j from 0: for the identity it returns v exactly (the zero terms add +0).
// v must be visible to the whole warp (written before a __syncwarp) and must not alias out.
template <class CX>
__device__ __forceinline__ void warp_matvec(const CX& x, const float* M, const float* v, float* out, bool upper) {
    const size_t P = x.a.P;
    for (int i0 = 0; i0 < x.p; i0 += 32) {
        const int i = i0 + x.lane;                        // (< P: P is a multiple of 32)
        float acc = 0.0f;
        for (int j = upper ? i0 : 0; j < x.p; ++j) acc = fmaf(M[(size_t)j * P + i], v[j], acc);
        if (i < x.p) out[i] = acc;
    }
    __syncwarp();
}

// kinetic energy 0.5 p' M^-1 p  (dense_e: also leaves p_sharp = Sigma p of the working point in DV_PSH)
template <class CX>
__device__ __forceinline__ double kinetic(const CX& x, const float* p) {
    if constexpr (CX::kDense) {
        float* ps = x.dv(DV_PSH);
        warp_matvec(x, x.dm(DN_SIGMA), p, ps, false);
        float s = 0.0f;
        for (int i = x.lane; i < x.p; i += 32) s = fmaf(ps[i], p[i], s);
        return 0.5 * warp_sum((double)s);
    }
    const float* minv = x.v(V_MINV);
    float s = 0.0f;
    for (int i = x.lane; i < x.p; i += 32) s += minv[i] * p[i] * p[i];
    return 0.5 * warp_sum((double)s);
}

// full gradient / potential from the likelihood pass output:
//   V = -(lp_lik + lp_prior),  g = dV/dq
template <class CX>
__device__ double finish_gradient(const CX& x, double lp_lik) {
    const float* q = x.v(V_Q);
    const float* gl = x.v(V_GL);
    float* g = x.v(V_G);
    const int d = x.d;
    float quad = 0.0f, sq = 0.0f;
    for (int i = x.lane; i < d; i += 32) {
        const float ci = x.cavc()[i];               // Omega (phi - mu), computed by cavity_term()
        quad += ci * (q[i] - x.muf()[i]);
        g[i] = ci - gl[i];
    }
    const bool laplace = x.a.model == EPG_M5B;        // eta, etb ~ double_exponential(0,1): -|q| instead of -q^2/2
    for (int i = d + x.lane; i < x.p; i += 32) {
        const float qi = q[i];
        sq += laplace ? 2.0f * fabsf(qi) : qi * qi;
        g[i] = (laplace ? copysignf(qi != 0.0f ? 1.0f : 0.0f, qi) : qi) - gl[i];
    }
    const double prior = -0.5 * warp_sum((double)quad) - 0.5 * warp_sum((double)sq);
    __syncwarp();
    return -(lp_lik + prior);
}

// Fused consume step of a tree leaf: gradient/potential from the likelihood pass, second half
// of the leapfrog, kinetic energy and the leaf's node vectors (rho = p, p_sharp = M^-1 p,
// proposal = this point) in ONE pass over the parameter vector and ONE round of warp reductions.
template <class CX>
__device__ void leaf_fused(const CX& x, double lp_lik, float eps_signed, double& Vnew, double& kin) {
    const float* q = x.v(V_Q);
    const float* gl = x.v(V_GL);
    const float* minv = x.v(V_MINV);
    float* g = x.v(V_G); float* p = x.v(V_P);
    float* crho = x.v(V_CRHO); float* cpsl = x.v(V_CPSL);
    float* qp_ = x.v(V_QPROP); float* gp_ = x.v(V_GPROP);
    const int d = x.d;
    const bool laplace = x.a.model == EPG_M5B;
    float prior2 = 0.0f, kin2 = 0.0f;                 // (phi-mu)'Omega(phi-mu) + |latents|^2 ;  p'M^-1 p
    for (int i = x.lane; i < x.p; i += 32) {
        const float qi = q[i];
        float gi;
        if (i < d) {
            const float ci = x.cavc()[i];
            prior2 = fmaf(ci, qi - x.muf()[i], prior2);
            gi = ci - gl[i];
        } else if (laplace) {
            prior2 += 2.0f * fabsf(qi);
            gi = copysignf(qi != 0.0f ? 1.0f : 0.0f, qi) - gl[i];
        } else {
            prior2 = fmaf(qi, qi, prior2);
            gi = qi - gl[i];
        }
        const float pi = p[i] - 0.5f * eps_signed * gi;
        if constexpr (CX::kDense) {
            g[i] = gi; p[i] = pi;
            crho[i] = pi;
            qp_[i] = qi; gp_[i] = gi;
        } else {
            const float mp = minv[i] * pi;
            kin2 = fmaf(mp, pi, kin2);
            g[i] = gi; p[i] = pi;
            crho[i] = pi; cpsl[i] = mp;
            qp_[i] = qi; gp_[i] = gi;
        }
    }
    if constexpr (CX::kDense) {          // p_sharp = Sigma p needs all of p: a second pass
        __syncwarp();
        float* ps = x.dv(DV_PSH);
        warp_matvec(x, x.dm(DN_SIGMA), p, ps, false);
        for (int i = x.lane; i < x.p; i += 32) {
            const float mp = ps[i];
            kin2 = fmaf(mp, p[i], kin2);
            cpsl[i] = mp;
        }
    }
    // two reductions interleaved
    double a = (double)prior2, b = (double)kin2;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    __syncwarp();
    Vnew = -(lp_lik - 0.5 * a);
    kin = 0.5 * b;
}

template <class CX>
__device__ void sample_momentum(const CX& x, ChainS& s) {
    const float* minv = x.v(V_MINV);
    float* p = x.v(V_P);
    const uint32_t ctr = s.rng++;
    if constexpr (CX::kDense) {
        // p = U^-1 z with Sigma = U'U, z ~ N(0, I): p ~ N(0, Sigma^-1) (dense_e_metric.hpp sample_p).  z goes
        // through the minus-end p_sharp, which a transition / step-size trial sets only after this.
        float* z = x.dv(DV_PSM);
        for (int i = x.lane; i < x.p; i += 32) z[i] = rng_normal(x.key, ctr, (uint32_t)i);
        __syncwarp();
        warp_matvec(x, x.dm(DN_UINV), z, p, true);
        return;
    }
    for (int i = x.lane; i < x.p; i += 32) p[i] = rng_normal(x.key, ctr, (uint32_t)i) * rsqrtf(minv[i]);
    __syncwarp();
}

// first half of a leapfrog step from the working point: p -= e/2 g ; q += e M^-1 p
template <class CX>
__device__ void leapfrog_begin(const CX& x, float eps_signed) {
    float* q = x.v(V_Q); float* p = x.v(V_P); const float* g = x.v(V_G); const float* minv = x.v(V_MINV);
    if constexpr (CX::kDense) {          // q += e Sigma p, through the working point's p_sharp (recomputed at the leaf)
        for (int i = x.lane; i < x.p; i += 32) p[i] = p[i] - 0.5f * eps_signed * g[i];
        __syncwarp();
        float* ps = x.dv(DV_PSH);
        warp_matvec(x, x.dm(DN_SIGMA), p, ps, false);
        for (int i = x.lane; i < x.p; i += 32) q[i] += eps_signed * ps[i];
        __syncwarp();
        return;
    }
    for (int i = x.lane; i < x.p; i += 32) {
        const float ph = p[i] - 0.5f * eps_signed * g[i];
        p[i] = ph;
        q[i] += eps_signed * minv[i] * ph;
    }
    __syncwarp();
}
template <class CX>
__device__ void leapfrog_end(const CX& x, float eps_signed) {
    float* p = x.v(V_P); const float* g = x.v(V_G);
    for (int i = x.lane; i < x.p; i += 32) p[i] -= 0.5f * eps_signed * g[i];
    __syncwarp();
}

template <class CX>
__device__ void begin_ss_trial(const CX& x, ChainS& s) {
    vcopy(x, V_Q, V_QS);
    vcopy(x, V_G, V_GS);
    __syncwarp();
    sample_momentum(x, s);
    s.H0 = s.Vs + kinetic(x, x.v(V_P));
    leapfrog_begin(x, s.eps);
    s.phase = PH_SS_WAIT;
}

template <class CX>
__device__ void issue_leapfrog(const CX& x, ChainS& s) {
    leapfrog_begin(x, s.sign * s.eps_tr);
    s.phase = PH_TREE_WAIT;
}

template <class CX>
__device__ void begin_subtree(const CX& x, ChainS& s) {
    const float u = rng_uniform(x.key, s.rng);
    s.sign = (u > 0.5f) ? 1 : -1;
    if (s.sign > 0) { vcopy(x, V_Q, V_QP); vcopy(x, V_P, V_PP); vcopy(x, V_G, V_GP); }
    else            { vcopy(x, V_Q, V_QM); vcopy(x, V_P, V_PM); vcopy(x, V_G, V_GM); }
    __syncwarp();
    s.nleaf = 0;
    issue_leapfrog(x, s);
}

template <class CX>
__device__ void begin_transition(const CX& x, ChainS& s) {
    // base_hmc::sample_stepsize: eps = eps_nom (1 + jitter (2u - 1)) from its own stream (counter = transition), so
    // that jitter 0 draws exactly what a run without jitter draws
    s.eps_tr = s.eps;
    if (x.a.jitter > 0.0f) {
        const uint4 r = philox4x32(make_uint4((uint32_t)s.iter, 0u, 4u, 0u), x.key);
        s.eps_tr = s.eps * (1.0f + x.a.jitter * (2.0f * u01(r.x) - 1.0f));
    }
    vcopy(x, V_Q, V_QS);
    vcopy(x, V_G, V_GS);
    __syncwarp();
    sample_momentum(x, s);
    s.V = s.Vs;
    s.H0 = s.Vs + kinetic(x, x.v(V_P));
    if (x.lane == 0) x.a.hmc[x.cg].Hs = s.H0;           // the sample starts as the initial point
    vcopy(x, V_QM, V_Q); vcopy(x, V_PM, V_P); vcopy(x, V_GM, V_G);
    vcopy(x, V_QP, V_Q); vcopy(x, V_PP, V_P); vcopy(x, V_GP, V_G);
    vcopy(x, V_RHO, V_P);
    if constexpr (CX::kDense) { dcopy(x, DV_PSM, DV_PSH); dcopy(x, DV_PSP, DV_PSH); }   // (kinetic() set PSH)
    __syncwarp();
    s.lsw = 0.0;
    s.depth = 0;
    s.n_leap_tr = 0;
    s.sum_metro = 0.0;
    begin_subtree(x, s);
}

// Stan 2.17 windowed_adaptation::compute_next_window
__device__ void next_window(const SamplerArgs& a, ChainS& s) {
    const int last = a.warmup - a.win_term - 1;
    if (s.win_next == last) return;
    s.win_size *= 2;
    s.win_next = s.win_count + s.win_size;
    if (s.win_next == last) return;
    const int boundary = s.win_next + 2 * s.win_size;
    if (boundary >= a.warmup - a.win_term) s.win_next = last;
}

// dense_e window end (covar_adaptation.hpp learn_covariance + dense_e_metric): from the window's co-moment W2 of
// n draws, Sigma = n/(n+5) W2/(n-1) + reg 5/(n+5) I, formed and Cholesky-factored (Sigma = L L', U = L') in fp64
// in the chain's scratch, by the chain's warp.  On success Sigma (fp32, symmetric), U^-1 = (L^-1)' stored by
// columns and diag(Sigma) in V_MINV are replaced; a non-finite or non-positive pivot leaves all three as they were.
template <class CX>
__device__ void dense_window_end(const CX& x, int n) {
    const int p = x.p, lane = x.lane;
    const size_t P = x.a.P;
    double* A = x.ws;
    const float* w2 = x.dm(DN_W2);
    const double sc = (double)n / ((double)n + 5.0) / ((double)n - 1.0);
    const double reg = (double)x.a.metric_reg * (5.0 / ((double)n + 5.0));
    // lower triangle (Stan's LLT reads the lower triangle of the estimate too)
    for (int i = 0; i < p; ++i)
        for (int j = lane; j <= i; j += 32) A[i * P + j] = sc * (double)w2[i * P + j] + (i == j ? reg : 0.0);
    __syncwarp();
    // right-looking Cholesky, lane r owns rows r, r + 32, ...
    bool ok = true;
    for (int k = 0; k < p; ++k) {
        const double piv = A[k * P + k];
        if (!(piv > 0.0 && isfinite(piv))) { ok = false; break; }       // (the same value on every lane)
        const double lkk = sqrt(piv), rl = 1.0 / lkk;
        for (int i = k + 1 + lane; i < p; i += 32) A[i * P + k] *= rl;
        __syncwarp();
        if (lane == 0) A[k * P + k] = lkk;
        for (int i = k + 1 + lane; i < p; i += 32) {
            const double lik = A[i * P + k];
            for (int j = k + 1; j <= i; ++j) A[i * P + j] -= lik * A[j * P + k];
        }
        __syncwarp();
    }
    __syncwarp();
    if (!ok) return;
    // L^-1 column by column (lane r: columns r, r + 32, ...): L x = e_j, x_i (i > j) kept in the free upper
    // triangle A[j][i]
    for (int j = lane; j < p; j += 32) {
        const double xj = 1.0 / A[j * P + j];
        for (int i = j + 1; i < p; ++i) {
            double acc = A[i * P + j] * xj;
            for (int k = j + 1; k < i; ++k) acc += A[i * P + k] * A[j * P + k];
            A[j * P + i] = -acc / A[i * P + i];
        }
    }
    __syncwarp();
    // U^-1 (i, j) = L^-1 (j, i), nonzero for i <= j, stored at ui[j P + i]; Sigma recomputed from W2
    float* sig = x.dm(DN_SIGMA); float* ui = x.dm(DN_UINV); float* minv = x.v(V_MINV);
    for (int j = 0; j < p; ++j)
        for (int i = lane; i < p; i += 32) {
            ui[j * P + i] = i < j ? (float)A[i * P + j] : (i == j ? (float)(1.0 / A[i * P + i]) : 0.0f);
            const int r = i > j ? i : j, c = i > j ? j : i;
            sig[j * P + i] = (float)(sc * (double)w2[r * P + c] + (i == j ? reg : 0.0));
        }
    __syncwarp();
    for (int i = lane; i < p; i += 32) minv[i] = sig[i * P + i];
    __syncwarp();
}

// HMC diagnostics of the transition that ends (lane 0), with Stan 2.17's definitions (base_nuts::transition):
// the record of every transition Stan saves with save_warmup (warm-up or post-warm-up transition m with
// m % thin == 0), and over the saved post-warm-up ones the divergences, the transitions at max_treedepth and the
// energy sums of E-BFMI = sum (E_t - E_t-1)^2 / sum (E_t - mean E)^2 (PyStan's check_energy), shifted by the
// first saved energy
template <class CX>
__device__ void hmc_diagnostics(const CX& x, const ChainS& s, double accept, bool divergent) {
    const SamplerArgs& a = x.a;
    const bool warm = s.iter < a.warmup;
    const int m = warm ? s.iter : s.iter - a.warmup;
    if (x.lane != 0 || m % a.thin != 0) return;
    HmcChain& h = a.hmc[x.cg];
    const double E = h.Hs;
    const int t = m / a.thin;
    if (a.rec) {
        double* r = a.rec + ((size_t)x.cg * a.n_rec + (warm ? 0 : a.n_rec_warm) + t) * HMC_REC;
        r[0] = accept; r[1] = (double)s.eps_tr; r[2] = (double)s.depth; r[3] = (double)s.n_leap_tr;
        r[4] = divergent ? 1.0 : 0.0; r[5] = E;
    }
    if (warm) return;
    if (t == 0) { h.e0 = E; h.eprev = E; }
    const double dv = E - h.e0, de = E - h.eprev;
    h.se += dv; h.see += dv * dv; h.sdd += de * de; h.eprev = E;
    h.n_saved += 1.0;
    if (divergent) h.n_div += 1.0;
    if (s.depth >= a.max_depth) h.n_maxd += 1.0;
    if (t == a.n_save - 1) {
        const double var = h.see - h.se * h.se / h.n_saved;
        h.ebfmi = (h.n_saved >= 2.0 && var > 0.0) ? h.sdd / var : NAN;
    }
}

// bookkeeping at the end of a transition; returns with the next request issued
// (or the chain finished)
template <class CX>
__device__ void end_transition(const CX& x, ChainS& s, int c_local, int k_global_draw_site, bool divergent) {
    const SamplerArgs& a = x.a;
    const double accept = s.n_leap_tr > 0 ? s.sum_metro / (double)s.n_leap_tr : 0.0;
    hmc_diagnostics(x, s, accept, divergent);
    s.n_leap_total += s.n_leap_tr;
    const float* qs = x.v(V_QS);
    bool restart_ss = false;
    if (s.iter < a.warmup) {
      if (a.adapt_engaged) {           // (otherwise a warm-up transition is only discarded)
        // ---- dual averaging (stepsize_adaptation::learn_stepsize) ----
        s.da_count += 1;
        const double stat = accept > 1.0 ? 1.0 : accept;
        const double eta = 1.0 / (s.da_count + a.t0);
        s.s_bar = (1.0 - eta) * s.s_bar + eta * (a.delta - stat);
        const double xx = s.mu - s.s_bar * sqrt((double)s.da_count) / a.gamma;
        const double x_eta = pow((double)s.da_count, -a.kappa);
        s.x_bar = (1.0 - x_eta) * s.x_bar + x_eta * xx;
        s.eps = (float)exp(xx);
        // ---- variance windows (var_adaptation::learn_variance; dense_e: covar_adaptation; unit_e: none) ----
        const bool windows = a.warmup >= 20 && a.metric != EPG_METRIC_UNIT;
        const bool in_win = windows && s.win_count >= a.win_init &&
                            s.win_count < a.warmup - a.win_term && s.win_count != a.warmup;
        if (CX::kDense && in_win) {
            // Welford co-moment (welford_covar_estimator): m += d/n, W2 += (q - m) d'.  d and q - m go through the
            // p_sharp vectors of the ends, which the finished transition no longer needs.
            s.w_n += 1;
            float* wm = x.v(V_WMEAN); float* dl = x.dv(DV_PSM); float* dq = x.dv(DV_PSP);
            for (int i = x.lane; i < x.p; i += 32) {
                const float dlt = qs[i] - wm[i];
                wm[i] += dlt / (float)s.w_n;
                dl[i] = dlt; dq[i] = qs[i] - wm[i];
            }
            __syncwarp();
            float* w2 = x.dm(DN_W2);
            for (int i = 0; i < x.p; ++i) {
                const float di = dq[i];
                for (int j = x.lane; j < x.p; j += 32) w2[(size_t)i * a.P + j] += di * dl[j];
            }
            __syncwarp();
        } else if (in_win) {
            s.w_n += 1;
            float* wm = x.v(V_WMEAN); float* w2 = x.v(V_WM2);
            for (int i = x.lane; i < x.p; i += 32) {
                const float dlt = qs[i] - wm[i];
                wm[i] += dlt / (float)s.w_n;
                w2[i] += (qs[i] - wm[i]) * dlt;
            }
        }
        const bool win_end = windows && s.win_count == s.win_next && s.win_count != a.warmup;
        if (CX::kDense && win_end) {
            next_window(a, s);
            dense_window_end(x, s.w_n);
            float* wm = x.v(V_WMEAN); float* w2 = x.dm(DN_W2);
            for (int i = x.lane; i < x.p; i += 32) wm[i] = 0.0f;
            for (int i = 0; i < x.p; ++i)
                for (int j = x.lane; j < x.p; j += 32) w2[(size_t)i * a.P + j] = 0.0f;
            __syncwarp();
            s.w_n = 0;
            restart_ss = true;
        } else if (win_end) {
            next_window(a, s);
            const float n = (float)s.w_n;
            float* minv = x.v(V_MINV); float* wm = x.v(V_WMEAN); float* w2 = x.v(V_WM2);
            for (int i = x.lane; i < x.p; i += 32) {
                const float var = w2[i] / (n - 1.0f);
                // (Stan's regularisation towards the absolute scale 1e-3 is kept also when the metric is carried over
                //  between EP iterations: shrinking towards the carried value instead was measured -- shorter
                //  trees, 3.8 s instead of 5.8 s per config-4 iteration, but underestimated variances then feed
                //  back into the next run: median split-Rhat 1.02 -> 1.06 and the EP iteration became unstable)
                minv[i] = (n / (n + 5.0f)) * var + 1e-3f * (5.0f / (n + 5.0f));
                wm[i] = 0.0f; w2[i] = 0.0f;
            }
            s.w_n = 0;
            restart_ss = true;
        }
        s.win_count += 1;
      }
    } else if ((s.iter - a.warmup) % a.thin == 0) {
        // ---- store the draw of phi (saved draw t of n_save) and accumulate split-Rhat sums ----
        const int t = (s.iter - a.warmup) / a.thin;
        const int per = a.n_save;
        double* dst = a.draws + (size_t)k_global_draw_site * a.d * a.n_draws;
        for (int i = x.lane; i < a.d; i += 32) dst[(size_t)i * a.n_draws + c_local * per + t] = (double)qs[i];
        const int half = (t < per / 2) ? 0 : 1;
        if (t < 2 * (per / 2)) {
            float* rs = x.v(half ? V_RS1 : V_RS0); float* rq = x.v(half ? V_RQ1 : V_RQ0);
            // centred on the first draw for accuracy: stored in WMEAN after warm-up
            const float* ref = x.v(V_WMEAN);
            for (int i = x.lane; i < x.p; i += 32) {
                const float dv = qs[i] - ref[i];
                rs[i] += dv; rq[i] += dv * dv;
            }
        }
        s.eps_sum += s.eps_tr;
        if (t == per - 1) {
            // the last saved draw is what init_prev carries over (util.get_last_fit_sample reads the last saved
            // draw of a fit; with thin > 1 it need not be the final transition)
            float* lq = a.last_q + (size_t)x.cg * a.P;
            for (int i = x.lane; i < x.p; i += 32) lq[i] = qs[i];
        }
        if (a.tstats) {
            // transformed parameters of the Stan programs (m1b.stan:30-36 ...): slot i of q maps to
            // phi_i | alpha_j = [mu_a +] eta_j sigma_a | beta_ji = [mu_b,i +] etb_ji sigma_b,i
            float* tr = x.v(V_TREF); float* ts = x.v(V_TS); float* tq = x.v(V_TQ);
            const int D = x.D, J = x.J, d = a.d;
            const bool four = model_four(a.model);
            const int ia = four ? 1 : 0, ib = four ? 2 + D : 1;
            for (int i = x.lane; i < x.p; i += 32) {
                float T;
                if (i < d) T = qs[i];
                else if (i < d + J) T = qs[i] * __expf(qs[ia]) + (four ? qs[0] : 0.0f);
                else {
                    const int e = i - d - J;
                    const int col = a.model == EPG_M2B ? e : e % D;
                    const float lsb = a.model == EPG_M2B ? qs[ib] : qs[ib + col];
                    T = qs[i] * __expf(lsb) + (four ? qs[2 + col] : 0.0f);
                }
                if (t == 0) { tr[i] = T; ts[i] = 0.0f; tq[i] = 0.0f; }
                else { const float dv = T - tr[i]; ts[i] += dv; tq[i] += dv * dv; }
            }
        }
    }
    __syncwarp();
    s.iter += 1;
    if (s.iter == a.warmup && a.warmup > 0 && a.adapt_engaged) {
        s.eps = (float)exp(s.x_bar);                 // complete_adaptation
        restart_ss = false;
    }
    if (s.iter == a.warmup) {
        // reference point for the Rhat sums
        float* ref = x.v(V_WMEAN);
        for (int i = x.lane; i < x.p; i += 32) ref[i] = qs[i];
        __syncwarp();
    }
    if (s.iter >= a.iter) {
        float* lm = a.last_minv + (size_t)x.cg * a.P;
        const float* minv = x.v(V_MINV);
        for (int i = x.lane; i < x.p; i += 32) lm[i] = minv[i];
        if (x.lane == 0) { a.last_eps[x.cg] = s.eps; a.last_metric[x.cg] = (float)a.metric; }
        s.phase = PH_DONE;
        return;
    }
    if (restart_ss) {
        s.ss_first = 1;
        s.restart_ss = 1;
        begin_ss_trial(x, s);
    } else {
        begin_transition(x, s);
    }
}

// a given starting point (init mode "given") with an entry to draw at random (NaN)
template <class CX>
__device__ bool given_has_random(const CX& x, const float* gq) {
    float nr = 0.0f;
    for (int i = x.lane; i < x.p; i += 32) if (isnan(gq[i])) nr = 1.0f;
    return warp_sum(nr) > 0.0f;
}

// One step of the per-chain state machine: consume the gradient that was just
// evaluated at V_Q (lp_lik) and advance until the next evaluation is requested.
template <class CX>
__device__ void chain_step(const CX& x, ChainS& s, double lp_lik, int c_local, int site_draw) {
    const SamplerArgs& a = x.a;
    if (s.phase == PH_DONE || s.phase == PH_DEAD) return;
    if (s.phase == PH_START_WAIT) {
        const double V0 = finish_gradient(x, lp_lik);
        bool fin = isfinite(V0);
        const float* g = x.v(V_G);
        float bad = 0.0f;
        for (int i = x.lane; i < x.p; i += 32) if (!isfinite(g[i])) bad = 1.0f;
        fin = fin && (warp_sum(bad) == 0.0f);
        if (fin) {
            s.Vs = V0;
            vcopy(x, V_QS, V_Q);
            vcopy(x, V_GS, V_G);
            __syncwarp();
            if (!a.adapt_engaged) { begin_transition(x, s); return; }     // (run_sampler: no step-size heuristic)
            s.ss_first = 1;
            s.restart_ss = 0;
            begin_ss_trial(x, s);
            return;
        }
        // redraw a starting point with a random component (Stan: up to 100 attempts); one that is given in full
        // fails the chain at once
        const bool redraw = s.init_mode == IM_RANDOM || s.init_mode == IM_REINIT ||
                            (s.init_mode == IM_GIVEN && given_has_random(x, a.inits + (size_t)x.cg * a.P));
        if (redraw && s.init_tries < 100) { s.init_tries++; s.phase = PH_START; }   // redraw below
        else { s.phase = PH_DEAD; return; }
    }
    if (s.phase == PH_START) {
        float* q = x.v(V_Q);
        if (s.init_mode == IM_PREV) {
            const float* lq = a.last_q + (size_t)x.cg * a.P;
            for (int i = x.lane; i < x.p; i += 32) q[i] = lq[i];
        } else if (s.init_mode == IM_ZERO) {
            for (int i = x.lane; i < x.p; i += 32) q[i] = 0.0f;
        } else if (s.init_mode == IM_REINIT) {
            // re-initialisation of a site whose chains did not mix: phi within one conditional cavity standard
            // deviation of the cavity mean, latents in U(-1, 1).  (Late in an EP run the cavity is so tight that
            // Stan's U(-2, 2) starts thousands of standard deviations out and the step size collapses.)
            const uint32_t ctr = s.rng++;
            for (int i = x.lane; i < x.p; i += 32) {
                const uint4 r = philox4x32(make_uint4(ctr, (uint32_t)i, 5u, 0u), x.key);
                const float u = 2.0f * u01(r.x) - 1.0f;
                q[i] = i < x.d ? x.muf()[i] + u * rsqrtf(fmaxf(x.omega[i * x.d + i], 1e-12f)) : u;
            }
        } else {
            // Stan's random init U(-init_r, init_r) (default 2), for every entry of a given init that is NaN
            // (an init given in full draws nothing: it starts the chain's stream where init '0' does)
            const float* gq = s.init_mode == IM_GIVEN ? a.inits + (size_t)x.cg * a.P : nullptr;
            const uint32_t ctr = (!gq || given_has_random(x, gq)) ? s.rng++ : 0u;
            const float rr = a.init_r;
            for (int i = x.lane; i < x.p; i += 32) {
                const float g = gq ? gq[i] : NAN;
                if (!isnan(g)) { q[i] = g; continue; }
                const uint4 r = philox4x32(make_uint4(ctr, (uint32_t)i, 3u, 0u), x.key);
                q[i] = 2.0f * rr * u01(r.x) - rr;
            }
        }
        __syncwarp();
        s.phase = PH_START_WAIT;
        return;
    }
    // ---- consume ----
    double Vnew, kin_leaf = 0.0;
    const bool tree_leaf = s.phase == PH_TREE_WAIT;
    if (tree_leaf) leaf_fused(x, lp_lik, s.sign * s.eps_tr, Vnew, kin_leaf);
    else Vnew = finish_gradient(x, lp_lik);
    if (s.phase == PH_SS_WAIT) {
        leapfrog_end(x, s.eps);
        double h = Vnew + kinetic(x, x.v(V_P));
        if (isnan(h)) h = INFINITY;
        const double dH = s.H0 - h;
        const double thr = log(0.8);
        s.n_leap_total += 1;
        if (s.ss_first) {
            s.ss_dir = (dH > thr) ? 1 : -1;
            s.ss_first = 0;
            begin_ss_trial(x, s);
            return;
        }
        const bool stop = (s.ss_dir == 1) ? !(dH > thr) : !(dH < thr);
        if (stop || s.eps > 1e7f || s.eps < 1e-30f) {
            if (s.restart_ss) {            // after a metric update: restart dual averaging
                s.mu = log(10.0 * (double)s.eps);
                s.s_bar = 0.0; s.x_bar = 0.0; s.da_count = 0;
                s.restart_ss = 0;
            }
            begin_transition(x, s);
            return;
        }
        s.eps = (s.ss_dir == 1) ? 2.0f * s.eps : 0.5f * s.eps;
        begin_ss_trial(x, s);
        return;
    }
    // ---- PH_TREE_WAIT: a new leaf of the current subtree ----
    s.V = Vnew;
    double h = Vnew + kin_leaf;
    if (isnan(h)) h = INFINITY;
    s.n_leap_tr += 1;
    const double dH = s.H0 - h;
    s.sum_metro += (dH > 0.0) ? 1.0 : (double)__expf((float)dH);
    if (-dH > 1000.0) {                 // divergent: the subtree is discarded
        s.n_div += 1;
        end_transition(x, s, c_local, site_draw, true);
        return;
    }
    // (leaf node vectors -- rho = p, p_sharp(left) = M^-1 p, proposal = this point -- were
    //  written by leaf_fused)
    s.cur_lsw = dH;
    s.Vprop = Vnew;
    // Hamiltonian of the proposal, beside Vprop (only lane 0 keeps it: it feeds the HMC diagnostics alone): this
    // leaf's, or that of the highest stack level whose pending proposal wins a merge below, loaded once after the
    // merges and stored after the next stretch of work
    HmcChain& hm = a.hmc[x.cg];
    double hprop = h;
    int hsrc = -1;
    int l = 0;
    while ((s.nleaf >> l) & 1) {
        // merge the pending left sibling at level l with the node just completed
        const int base = V_STACK + 4 * l;
        const double lsw_sub = log_sum_exp(x.stk->lsw[l], s.cur_lsw);
        bool take_right = s.cur_lsw > lsw_sub;
        if (!take_right) take_right = rng_uniform(x.key, s.rng) < __expf((float)(s.cur_lsw - lsw_sub));
        const float* lpsl = x.v(base + 0); const float* lrho = x.v(base + 1);
        float* crho = x.v(V_CRHO); float* cpsl = x.v(V_CPSL);
        const float* p = x.v(V_P); const float* minv = x.v(V_MINV);
        float d1 = 0.0f, d2 = 0.0f;
        if constexpr (CX::kDense) {
            const float* ps = x.dv(DV_PSH);       // p_sharp of the new leaf (leaf_fused)
            for (int i = x.lane; i < x.p; i += 32) {
                const float rs = lrho[i] + crho[i];
                crho[i] = rs;
                const float pl = lpsl[i];
                cpsl[i] = pl;
                d1 += pl * rs;
                d2 = fmaf(ps[i], rs, d2);
            }
        } else
        for (int i = x.lane; i < x.p; i += 32) {
            const float rs = lrho[i] + crho[i];
            crho[i] = rs;
            const float pl = lpsl[i];
            cpsl[i] = pl;
            d1 += pl * rs;
            d2 += minv[i] * p[i] * rs;
        }
        d1 = warp_sum(d1); d2 = warp_sum(d2);
        if (!take_right) {
            vcopy(x, V_QPROP, base + 2);
            vcopy(x, V_GPROP, base + 3);
            s.Vprop = x.stk->V[l];
            hsrc = l;
        }
        __syncwarp();
        s.cur_lsw = lsw_sub;
        if (!(d1 > 0.0f && d2 > 0.0f)) {        // U-turn inside the new subtree: discard it
            end_transition(x, s, c_local, site_draw, false);
            return;
        }
        ++l;
    }
    if (x.lane == 0 && hsrc >= 0) hprop = hm.Hstk[hsrc];
    if (l < s.depth) {
        const int base = V_STACK + 4 * l;
        {
            float4* d0 = reinterpret_cast<float4*>(x.v(base + 0)); const float4* s0 = reinterpret_cast<const float4*>(x.v(V_CPSL));
            float4* d1 = reinterpret_cast<float4*>(x.v(base + 1)); const float4* s1 = reinterpret_cast<const float4*>(x.v(V_CRHO));
            float4* d2 = reinterpret_cast<float4*>(x.v(base + 2)); const float4* s2 = reinterpret_cast<const float4*>(x.v(V_QPROP));
            float4* d3 = reinterpret_cast<float4*>(x.v(base + 3)); const float4* s3 = reinterpret_cast<const float4*>(x.v(V_GPROP));
            for (int i = x.lane; 4 * i < x.p; i += 32) { d0[i] = s0[i]; d1[i] = s1[i]; d2[i] = s2[i]; d3[i] = s3[i]; }
        }
        if (x.lane == 0) { x.stk->lsw[l] = s.cur_lsw; x.stk->V[l] = s.Vprop; }
        __syncwarp();
        s.nleaf += 1;
        issue_leapfrog(x, s);
        if (x.lane == 0) hm.Hstk[l] = hprop;
        return;
    }
    // ---- the subtree of 2^depth leaves is complete and valid ----
    if (s.sign > 0) { vcopy(x, V_QP, V_Q); vcopy(x, V_PP, V_P); vcopy(x, V_GP, V_G); }
    else            { vcopy(x, V_QM, V_Q); vcopy(x, V_PM, V_P); vcopy(x, V_GM, V_G); }
    if constexpr (CX::kDense) dcopy(x, s.sign > 0 ? DV_PSP : DV_PSM, DV_PSH);
    s.depth += 1;
    bool take = s.cur_lsw > s.lsw;
    if (!take) take = rng_uniform(x.key, s.rng) < __expf((float)(s.cur_lsw - s.lsw));
    if (take) { vcopy(x, V_QS, V_QPROP); vcopy(x, V_GS, V_GPROP); s.Vs = s.Vprop; }
    s.lsw = log_sum_exp(s.lsw, s.cur_lsw);
    __syncwarp();
    float d1 = 0.0f, d2 = 0.0f;
    {
        float* rho = x.v(V_RHO); const float* crho = x.v(V_CRHO);
        const float* pm = x.v(V_PM); const float* pp = x.v(V_PP); const float* minv = x.v(V_MINV);
        if constexpr (CX::kDense) {
            const float* psm = x.dv(DV_PSM); const float* psp = x.dv(DV_PSP);
            for (int i = x.lane; i < x.p; i += 32) {
                const float r = rho[i] + crho[i];
                rho[i] = r;
                d1 = fmaf(psm[i], r, d1);
                d2 = fmaf(psp[i], r, d2);
            }
        } else
        for (int i = x.lane; i < x.p; i += 32) {
            const float r = rho[i] + crho[i];
            rho[i] = r;
            d1 += minv[i] * pm[i] * r;
            d2 += minv[i] * pp[i] * r;
        }
        d1 = warp_sum(d1); d2 = warp_sum(d2);
        __syncwarp();
    }
    if (take && x.lane == 0) hm.Hs = hprop;
    if (!(d1 > 0.0f && d2 > 0.0f) || s.depth >= a.max_depth) {
        end_transition(x, s, c_local, site_draw, false);
        return;
    }
    begin_subtree(x, s);
}

// ---------------------------------------------------------------------------
// pieces shared by the sampling kernels
// ---------------------------------------------------------------------------
// cavity precision / mean -> fp32 copies (read by every chain every tick); thread t of a group of nthr
__device__ __forceinline__ void load_cavity(const SamplerArgs& a, int k, float* om, int t, int nthr) {
    const int d = a.d;
    const double* cq = a.cavQ + (size_t)k * d * d;
    float* muf = om + d * d;
    for (int e = t; e < d * d; e += nthr) om[e] = (float)cq[e];
    for (int i = t; i < d; i += nthr) muf[i] = (float)a.cavm[(size_t)k * d + i];
}

// initial state of the site's chains; warp w of a group of nw warps
__device__ __forceinline__ void init_chains(const SamplerArgs& a, const SiteView& sv, ChainS* cs, int w, int nw, int lane) {
    const int im = (a.init_mode == IM_PREV && a.reinit && a.reinit[sv.k]) ? IM_REINIT : a.init_mode;
    for (int c = w; c < a.C; c += nw) {
        ChainS& s = cs[c];
        const int cg = sv.k * a.C + c;
        // Warm-up starting point.  Stan: unit metric, step size 1.  With init_prev (method.py:404-406 carries the
        // last draw over) the previous run's ADAPTED metric and step size are carried over as well: the tilted
        // distribution of a site changes little between EP iterations, while a unit metric makes the first
        // 90 % of every warm-up crawl at the scale of the tightest cavity direction with saturated trees.
        // A re-initialised site (mode 3) starts from the conditional cavity variances instead.
        // (only from a run of the same metric: a diag_e metric is no starting point for dense_e, nor vice versa)
        // The step size starts from control 'stepsize' (default 1).  Without adaptation (run_sampler) every chain
        // runs with that step size and the unit metric throughout.
        float eps0 = a.stepsize;
        bool carried = false;
        if (im == IM_PREV && a.carry_adapt && a.adapt_engaged && a.last_metric[cg] == (float)a.metric) {
            const float e = a.last_eps[cg];
            if (e > 0.0f && isfinite(e)) { eps0 = e; carried = true; }     // (written together with last_minv)
        }
        if (lane == 0) {
            memset(&s, 0, sizeof(ChainS));
            s.phase = PH_START;
            s.init_mode = im;
            s.carried = carried ? 1 : 0;
            s.eps = eps0;
            s.mu = log(10.0 * (double)eps0);
            s.rng = 0;
            s.win_next = a.win_init + a.win_base - 1;
            s.win_size = a.win_base;
            HmcChain& h = a.hmc[cg];
            memset(&h, 0, sizeof(HmcChain));
            h.ebfmi = NAN;
        }
        // starting inverse metric, element i of the diagonal (unit_e: always 1)
        auto start_minv = [&](int i) -> float {
            float mv = 1.0f;
            if (a.metric == EPG_METRIC_UNIT || !a.adapt_engaged) return mv;
            if (carried) {
                const float v = a.last_minv[(size_t)cg * a.P + i];
                if (v > 0.0f && isfinite(v)) mv = v;
            } else if (im == IM_REINIT && i < a.d) {
                const double om = a.cavQ[(size_t)sv.k * a.d * a.d + (size_t)i * a.d + i];
                if (om > 0.0 && isfinite(om)) mv = (float)(1.0 / om);
            }
            return mv;
        };
        const int vecs[] = {V_WMEAN, V_WM2, V_RS0, V_RQ0, V_RS1, V_RQ1};
        for (int i = lane; i < a.P; i += 32) {
            const float mv = start_minv(i);
            cvec(a, sv, c, V_MINV)[i] = mv;
            for (int v = 0; v < 6; ++v) cvec(a, sv, c, vecs[v])[i] = 0.0f;
        }
        if (a.metric == EPG_METRIC_DENSE) {
            // a carried chain keeps Sigma and U^-1 of its previous (dense_e) run; otherwise diagonal: Sigma = the
            // starting diagonal above, U^-1 = its inverse square root
            float* dn = a.dense + (size_t)cg * dense_floats(a.P);
            const size_t PP = (size_t)a.P * a.P;
            for (int i = 0; i < a.P; ++i) {
                const float mv = carried ? 0.0f : start_minv(i);
                for (int j = lane; j < a.P; j += 32) {
                    if (!carried) {
                        dn[DN_SIGMA * PP + (size_t)i * a.P + j] = i == j ? mv : 0.0f;
                        dn[DN_UINV * PP + (size_t)i * a.P + j] = i == j ? (float)(1.0 / sqrt((double)mv)) : 0.0f;
                    }
                    dn[DN_W2 * PP + (size_t)i * a.P + j] = 0.0f;
                }
            }
        }
    }
}

// one chain phase of a site: every chain advances to its next gradient request; warp w of nw
template <bool ALLHOT, bool DENSE = false>
__device__ __forceinline__ void chain_phase(const SamplerArgs& a, const SiteView& sv, ChainS* cs, ChainStack* cstk,
                                            const double* lp_lik, int* n_active, int p, int J, uint32_t site_seed,
                                            const float* om, const float* muf, int w, int nw, int lane) {
    for (int c = w; c < a.C; c += nw) {
        const ChainCtxT<ALLHOT, DENSE> x = make_chain_ctx<ALLHOT, DENSE>(a, sv, c, p, a.d, J, a.D, lane,
                                                                         make_uint2(site_seed, (uint32_t)c), om, muf,
                                                                         cstk + c);
        ChainS s = cs[c];                  // private copy: every lane runs the same scalar code
        const int before = s.phase;
        chain_step(x, s, lp_lik[c], c, sv.k);
        __syncwarp();
        if (lane == 0) {
            cs[c] = s;
            if ((s.phase == PH_DONE || s.phase == PH_DEAD) && !(before == PH_DONE || before == PH_DEAD))
                atomicSub(n_active, 1);
        }
    }
}

// per-site analytics by one warp: mean step size, max split-Rhat, leapfrogs
__device__ void site_analytics(const SamplerArgs& a, const SiteView& sv, const ChainS* cs, int p, int lane,
                               double clk_chain, double clk_lik, double n_ticks) {
    const int C = a.C;
    const int per = a.n_save;                    // saved draws per chain
    const int hn = per / 2;
    float worst = 0.0f;
    if (hn >= 2 && C >= 1) {
        for (int i = lane; i < p; i += 32) {
            // split chains: 2C sequences of hn draws
            float mean_all = 0.0f, W = 0.0f;
            int m = 0;
            for (int c = 0; c < C; ++c) {
                if (cs[c].phase != PH_DONE) continue;
                for (int h = 0; h < 2; ++h) {
                    const float sm = cvec(a, sv, c, h ? V_RS1 : V_RS0)[i];
                    const float sq = cvec(a, sv, c, h ? V_RQ1 : V_RQ0)[i];
                    const float ref = cvec(a, sv, c, V_WMEAN)[i];
                    const float mu = sm / hn;
                    W += (sq - hn * mu * mu) / (hn - 1);
                    mean_all += mu + ref;
                    ++m;
                }
            }
            if (m >= 2) {
                mean_all /= m; W /= m;
                float B = 0.0f;
                for (int c = 0; c < C; ++c) {
                    if (cs[c].phase != PH_DONE) continue;
                    for (int h = 0; h < 2; ++h) {
                        const float mu = cvec(a, sv, c, h ? V_RS1 : V_RS0)[i] / hn + cvec(a, sv, c, V_WMEAN)[i];
                        B += (mu - mean_all) * (mu - mean_all);
                    }
                }
                B = B * hn / (m - 1);
                const float var_plus = (hn - 1.0f) / hn * W + B / hn;
                const float rhat = W > 0.0f ? sqrtf(var_plus / W) : 1.0f;
                worst = fmaxf(worst, rhat);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) worst = fmaxf(worst, __shfl_xor_sync(0xffffffffu, worst, o));
    // a chain that never found a finite starting point (PH_DEAD) has written no draws: poison its slice of
    // the draw buffer so that moment matching fails the site (Stan raises on an initialisation failure;
    // the reference then zero-fills the site update, method.py:460-465) instead of matching stale draws
    for (int c = 0; c < C; ++c) {
        if (cs[c].phase == PH_DONE) continue;
        double* dst = a.draws + (size_t)sv.k * a.d * a.n_draws;
        for (int e = lane; e < a.d * per; e += 32) {
            const int i = e / per, t = e - i * per;
            dst[(size_t)i * a.n_draws + c * per + t] = NAN;
        }
        // nor sampler-parameter records (epg_get_sampler_params then returns NaN for it, not stale records)
        if (a.rec) {
            double* r = a.rec + (size_t)(sv.k * C + c) * a.n_rec * HMC_REC;
            for (int e = lane; e < a.n_rec * HMC_REC; e += 32) r[e] = NAN;
        }
    }
    if (a.tstats) {
        double* to = a.tstats + (size_t)sv.k * 2 * a.P;
        for (int i = lane; i < p; i += 32) {
            double msum = 0.0;
            int m = 0;
            for (int c = 0; c < C; ++c) {
                if (cs[c].phase != PH_DONE) continue;
                msum += (double)cvec(a, sv, c, V_TREF)[i] + (double)cvec(a, sv, c, V_TS)[i] / per;
                ++m;
            }
            const double mean = m ? msum / m : NAN;
            double ssd = 0.0;
            for (int c = 0; c < C; ++c) {
                if (cs[c].phase != PH_DONE) continue;
                const double s1 = cvec(a, sv, c, V_TS)[i], s2 = cvec(a, sv, c, V_TQ)[i];
                const double mc = (double)cvec(a, sv, c, V_TREF)[i] + s1 / per;
                ssd += (s2 - s1 * s1 / per) + per * (mc - mean) * (mc - mean);
            }
            to[i] = mean;
            to[a.P + i] = m ? ssd : NAN;
        }
    }
    if (lane == 0) {
        double eps_mean = 0.0, nl = 0.0, nd = 0.0;
        int ok = 0;
        for (int c = 0; c < C; ++c) {
            nl += (double)cs[c].n_leap_total;
            nd += cs[c].n_div;
            if (cs[c].phase == PH_DONE) { eps_mean += cs[c].eps_sum / (per > 0 ? per : 1); ++ok; }
        }
        double* o = a.out + (size_t)sv.k * 8;
        o[4] = clk_chain; o[5] = clk_lik; o[6] = n_ticks; o[7] = 0.0;
        o[0] = ok ? eps_mean / ok : NAN;
        o[1] = (ok == C) ? (double)worst : NAN;
        o[2] = nl;
        o[3] = (ok == C) ? nd : -1.0;
    }
}

// ---------------------------------------------------------------------------
// the persistent sampling kernel: one CTA per site
// ---------------------------------------------------------------------------
// TCM 0: fp32 SIMT likelihood pass (NTHR threads); 1: tensor-core pass, 2: wide tensor-core pass (tc::NTHREADS threads)
// DENSE: the dense_e chain phase (separate instances, so that the diag_e / unit_e ones carry none of its code)
template <int CP, int TCM, bool DENSE>
__global__ void __launch_bounds__(TCM ? tc::NTHREADS : NTHR, 1)
k_nuts(const SamplerArgs a, const __grid_constant__ CUtensorMap tmap) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr bool USE_TC = TCM == 1, USE_TCW = TCM == 2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int site_off = a.order ? a.order[blockIdx.x] : (int)blockIdx.x;    // most expensive sites first
    const int k_local = a.k0 + site_off;
    const int C = a.C, d = a.d, D = a.D, S = a.S;
    const int64_t row_begin = a.row0[k_local];
    const int n_rows = (int)(a.row0[k_local + 1] - row_begin);
    const int* grows = a.grp_rows + a.grp_ptr[k_local];
    const int J = a.grp_ptr[k_local + 1] - a.grp_ptr[k_local] - 1;
    const int p = model_np(a.model, D, J);
    const SiteView sv{smem, k_local};
    ChainS* cs = reinterpret_cast<ChainS*>(smem + a.off_cs);
    ChainStack* cstk = reinterpret_cast<ChainStack*>(smem + a.off_cs + sizeof(ChainS) * a.C);
    __shared__ double lp_lik[32];
    __shared__ int n_active;

    // (the tensor-core variant runs with three extra warps, 8/9 = MMA issue and 10 = TMA,
    //  which take part only in the barriers and in tc::pass)
    const bool worker = tid < NTHR;
    float* om = a.omega_smem ? reinterpret_cast<float*>(smem + a.off_omega)
                             : a.omega + (size_t)k_local * (d * d + d);
    float* muf = om + d * d;
    if (worker) load_cavity(a, k_local, om, tid, NTHR);
    // resident design matrix
    if (TCM == 0 && a.resident) {
        const float4* src = reinterpret_cast<const float4*>(a.X + (size_t)row_begin * S);
        float4* dst = reinterpret_cast<float4*>(smem);
        for (int e = tid; e < n_rows * (S >> 2); e += NTHR) dst[e] = src[e];
    }
    // tensor-core pass: barriers + tensor memory
    unsigned char* tcb = smem + ((1024u - (tc::smem_u32(smem) & 1023u)) & 1023u);
    uint32_t tmem_base = 0;
    tc::State tcst;
    tcw::State tcwst;
    if constexpr (USE_TC) {
        tcst.set_stages(a.tc_nst);
        tmem_base = tc::setup(tcb, a.tc_nst);
    }
    if constexpr (USE_TCW) {
        tcwst.nst = (uint32_t)a.tc_nst;
        tmem_base = tcw::setup(tcb);
    }
    if (worker) init_chains(a, sv, cs, warp, NWARP, lane);
    if (tid == 0) n_active = C;
    __threadfence_block();
    __syncthreads();

    const uint32_t site_seed = a.seeds[site_off];
    long long clk_chain = 0, clk_lik = 0, n_ticks = 0;
    for (;;) {
        const long long tk0 = clock64();
        if (worker) chain_phase<USE_TC, DENSE>(a, sv, cs, cstk, lp_lik, &n_active, p, J, site_seed, om, muf, warp, NWARP, lane);
        __threadfence_block();
        __syncthreads();
        if (n_active <= 0) break;
        const long long tk1 = clock64();
        if constexpr (USE_TC) likelihood_pass_tc(a, smem, tcb, tmem_base, &tmap, tcst, k_local, C, row_begin, n_rows, lp_lik, om, muf);
        else if constexpr (USE_TCW) likelihood_pass_tcw(a, smem, tcb, tmem_base, &tmap, tcwst, k_local, C, row_begin, n_rows, lp_lik, om, muf);
        else likelihood_pass<CP>(a, smem, k_local, k_local, C, J, row_begin, n_rows, grows, lp_lik, om, muf);
        clk_chain += tk1 - tk0;
        clk_lik += clock64() - tk1;
        ++n_ticks;
    }
    if constexpr (USE_TC) tc::teardown(tmem_base);
    if constexpr (USE_TCW) tcw::teardown(tmem_base);
    __syncthreads();
    if (warp == 0) site_analytics(a, sv, cs, p, lane, (double)clk_chain, (double)clk_lik, (double)n_ticks);
}

// ---------------------------------------------------------------------------
// "ping-pong" sampling kernel (tensor-core pass, more sites than SMs): a persistent CTA
// holds TWO sites.  While the likelihood warps (TMA / tcgen05 / epilogue, the first
// tc::NTHREADS threads) run the pass of one site, PP_NCW chain warps advance the
// chains of the other; the roles swap every half-tick, so the tensor-core pipeline
// and the per-chain dependency chains hide each other.  Finished sites are replaced
// from a global queue (no wave quantisation).
// ---------------------------------------------------------------------------
constexpr int PP_NCW = 4;
constexpr int PP_THREADS = tc::NTHREADS + 32 * PP_NCW;
struct PPSlot {
    int k, state, n_active, n_rows, p;       // state 0 = empty, 1 = sampling
    uint32_t seed;
    int64_t row_begin;
    long long clk_chain, clk_lik, n_ticks;
};
__device__ __forceinline__ void chain_group_sync() { asm volatile("bar.sync 2, %0;\n" ::"n"(32 * PP_NCW) : "memory"); }

template <bool DENSE>
__global__ void __launch_bounds__(PP_THREADS, 1)
k_nuts_pp(const SamplerArgs a, const __grid_constant__ CUtensorMap tmap, int n_sites, int* queue) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int C = a.C, d = a.d;
    __shared__ PPSlot slot[2];
    __shared__ double lp_lik[2][32];
    __shared__ int exhausted, go_on[2];
    const bool lik_thread = tid < tc::NTHREADS;
    const int cw = warp - tc::NTHREADS / 32, ct = tid - tc::NTHREADS;      // chain warp / thread index

    unsigned char* tcb = smem + ((1024u - (tc::smem_u32(smem) & 1023u)) & 1023u);
    tc::State tcst;
    tcst.set_stages(a.tc_nst);
    const uint32_t tmem_base = tc::setup(tcb, a.tc_nst);
    if (tid == 0) { slot[0].state = 0; slot[1].state = 0; exhausted = 0; }
    __syncthreads();

    for (uint32_t h = 0;; ++h) {
        const int sl = (int)(h & 1u), sc = sl ^ 1;
        if (lik_thread) {
            // ---- likelihood pass of slot sl ----
            if (slot[sl].state == 1) {
                const long long t0 = clock64();
                unsigned char* sm = smem + (size_t)sl * a.site_stride;
                float* om = reinterpret_cast<float*>(sm + a.off_omega);
                likelihood_pass_tc(a, sm, tcb, tmem_base, &tmap, tcst, slot[sl].k, C, slot[sl].row_begin,
                                   slot[sl].n_rows, lp_lik[sl], om, om + d * d);
                if (tid == 0) slot[sl].clk_lik += clock64() - t0;
            }
        } else {
            // ---- chain phase of slot sc (also: retire a finished site, start the next one) ----
            PPSlot& S = slot[sc];
            unsigned char* sm = smem + (size_t)sc * a.site_stride;
            ChainS* cs = reinterpret_cast<ChainS*>(sm + a.off_cs);
            ChainStack* cstk = reinterpret_cast<ChainStack*>(sm + a.off_cs + sizeof(ChainS) * a.C);
            float* om = reinterpret_cast<float*>(sm + a.off_omega);
            for (int round = 0; round < 2; ++round) {
                if (S.state == 0) {
                    const int ex = exhausted;
                    chain_group_sync();                 // everyone has read the flag before thread 0 may set it
                    if (ex) break;
                    if (ct == 0) {
                        const int qi = atomicAdd(queue, 1);
                        if (qi < n_sites) {
                            const int i = a.order ? a.order[qi] : qi;
                            const int k = a.k0 + i;
                            S.k = k; S.n_active = C; S.seed = a.seeds[i];
                            S.row_begin = a.row0[k];
                            S.n_rows = (int)(a.row0[k + 1] - a.row0[k]);
                            S.p = model_np(a.model, a.D, 1);
                            S.clk_chain = 0; S.clk_lik = 0; S.n_ticks = 0;
                            S.state = 1;
                        } else {
                            exhausted = 1;
                        }
                    }
                    chain_group_sync();
                    if (S.state == 0) break;
                    load_cavity(a, S.k, om, ct, 32 * PP_NCW);
                    init_chains(a, SiteView{sm, S.k}, cs, cw, PP_NCW, lane);
                    __threadfence_block();
                    chain_group_sync();
                }
                const long long t0 = clock64();
                const SiteView sv{sm, S.k, (uint32_t)((size_t)sc * a.site_stride)};
                chain_phase<true, DENSE>(a, sv, cs, cstk, lp_lik[sc], &S.n_active, S.p, 1, S.seed, om, om + d * d, cw,
                                         PP_NCW, lane);
                __threadfence_block();
                chain_group_sync();
                if (ct == 0) { S.clk_chain += clock64() - t0; S.n_ticks += 1; }
                if (S.n_active > 0) break;
                // every chain of the site has finished
                if (cw == 0) site_analytics(a, sv, cs, S.p, lane, (double)S.clk_chain, (double)S.clk_lik, (double)S.n_ticks);
                chain_group_sync();
                if (ct == 0) S.state = 0;
                chain_group_sync();
            }
            // (decided by one thread, double-buffered: the slot states change again in the next half-tick)
            if (ct == 0) go_on[h & 1u] = !(slot[0].state == 0 && slot[1].state == 0 && exhausted);
        }
        __threadfence_block();
        __syncthreads();
        if (!go_on[h & 1u]) break;
    }
    tc::teardown(tmem_base);
}

// log-density / gradient at caller-supplied points (parity tests): the likelihood pass of k_nuts<CP, TCM>, run
// `ticks` times, then the gradient finish of its chain phase (the same ChainCtxT)
template <int CP, int TCM>
__global__ void __launch_bounds__(TCM ? tc::NTHREADS : NTHR, 1)
k_logdensity(const SamplerArgs a, const __grid_constant__ CUtensorMap tmap, int nq, int ticks, double* lp_out,
             double* grad_out) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr bool USE_TC = TCM == 1, USE_TCW = TCM == 2;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k_local = a.k0;
    const int d = a.d, D = a.D, S = a.S;
    const int64_t row_begin = a.row0[k_local];
    const int n_rows = (int)(a.row0[k_local + 1] - row_begin);
    const int* grows = a.grp_rows + a.grp_ptr[k_local];
    const int J = a.grp_ptr[k_local + 1] - a.grp_ptr[k_local] - 1;
    const int p = model_np(a.model, D, J);
    __shared__ double lp_lik[32];
    const bool worker = tid < NTHR;
    float* om = a.omega_smem ? reinterpret_cast<float*>(smem + a.off_omega)
                             : a.omega + (size_t)k_local * (d * d + d);
    float* muf = om + d * d;
    if (worker) load_cavity(a, k_local, om, tid, NTHR);
    if (TCM == 0 && a.resident) {
        const float4* src = reinterpret_cast<const float4*>(a.X + (size_t)row_begin * S);
        float4* dst = reinterpret_cast<float4*>(smem);
        for (int e = tid; e < n_rows * (S >> 2); e += NTHR) dst[e] = src[e];
    }
    unsigned char* tcb = smem + ((1024u - (tc::smem_u32(smem) & 1023u)) & 1023u);
    uint32_t tmem_base = 0;
    tc::State tcst;
    tcw::State tcwst;
    if constexpr (USE_TC) {
        tcst.set_stages(a.tc_nst);
        tmem_base = tc::setup(tcb, a.tc_nst);
    }
    if constexpr (USE_TCW) {
        tcwst.nst = (uint32_t)a.tc_nst;
        tmem_base = tcw::setup(tcb);
    }
    // the evaluation points were staged in the global copy of V_Q (k_set_q)
    if (worker && a.hot_nvec > V_Q)
        for (int e = tid; e < nq * a.P; e += NTHR) {
            const int c = e / a.P, i = e - c * a.P;
            cvec(a, SiteView{smem, k_local}, c, V_Q)[i] = a.chain_mem[((size_t)(k_local * a.C + c) * NVEC + V_Q) * a.P + i];
        }
    __threadfence_block();
    __syncthreads();
    // (ticks > 1: the pipeline state of the tensor-core passes carries over from one pass to the next, as it
    //  does between the sampler's gradient evaluations)
    for (int t = 0; t < ticks; ++t) {
        if constexpr (USE_TC) likelihood_pass_tc(a, smem, tcb, tmem_base, &tmap, tcst, k_local, nq, row_begin, n_rows, lp_lik, om, muf);
        else if constexpr (USE_TCW) likelihood_pass_tcw(a, smem, tcb, tmem_base, &tmap, tcwst, k_local, nq, row_begin, n_rows, lp_lik, om, muf);
        else likelihood_pass<CP>(a, smem, k_local, k_local, nq, J, row_begin, n_rows, grows, lp_lik, om, muf);
        __syncthreads();
    }
    for (int c = warp; worker && c < nq; c += NWARP) {
        const ChainCtxT<USE_TC> x = make_chain_ctx<USE_TC>(a, SiteView{smem, k_local}, c, p, d, J, D, lane,
                                                           make_uint2(0u, 0u), om, muf, nullptr);
        const double V = finish_gradient(x, lp_lik[c]);
        const float* g = x.v(V_G);
        if (lane == 0) lp_out[c] = -V;
        for (int i = lane; i < p; i += 32) grad_out[(size_t)c * p + i] = -(double)g[i];
    }
    if constexpr (USE_TC) tc::teardown(tmem_base);
    if constexpr (USE_TCW) tcw::teardown(tmem_base);
}

__global__ void k_set_q(float* chain_mem, int chain0, int P, int p, int nq, const double* q) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nq * p) return;
    const int c = idx / p, i = idx - c * p;
    chain_mem[((size_t)(chain0 + c) * NVEC + V_Q) * P + i] = (float)q[idx];
}

// shared-memory plan for a launch
constexpr size_t SMEM_BUDGET_1 = 227 * 1024 - 1024;       // one CTA per SM
constexpr size_t SMEM_BUDGET_2 = 112 * 1024 - 256;        // two CTAs per SM: 2 x (dynamic + 1 KB static + 1 KB reserved) <= 228 KB
bool plan_smem(SamplerArgs& a, int CP, int64_t max_rows, int d, size_t budget = SMEM_BUDGET_1) {
    auto al16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
    const size_t sz_cs = al16((sizeof(ChainS) + sizeof(ChainStack)) * (size_t)a.C);
    const size_t sz_om = al16(sizeof(float) * ((size_t)d * d + d));
    const size_t per_vec = sizeof(float) * (size_t)a.C * a.P;          // one hot vector of every chain
    // tail regions shared by both variants: [omega][hot vectors]
    auto place_tail = [&](size_t o) -> size_t {
        a.omega_smem = 0; a.hot_nvec = 0; a.hot_levels = 0; a.off_omega = a.off_hot = 0;
        if (o + sz_om <= budget && sz_om <= 48 * 1024) { a.omega_smem = 1; a.off_omega = o; o += sz_om; }
        int nv = per_vec ? (int)((budget - o) / per_vec) : 0;
        int lv = 0;
        if (nv > V_NHOT) {                      // room left: keep the lowest tree-stack levels on chip too
            lv = (nv - V_NHOT) / 4;
            if (lv > MAXDEPTH_CAP) lv = MAXDEPTH_CAP;
            if (const char* e = getenv("EPGPU_LEVELS")) lv = std::min(lv, atoi(e));
            nv = V_NHOT;
        }
        a.hot_levels = 0;
        if (nv > 0) {
            a.hot_nvec = nv; a.hot_levels = lv; a.off_hot = o;
            o += al16((size_t)(nv + 4 * lv) * per_vec);
        }
        return o;
    };
    if (a.use_tc == 2) {
        // wide pass: [coefficients | barriers | 4 E buffers | nst X sub-tiles][lp][chain scalars][tail]; the cavity
        // terms live in global memory (cavc_g).  The ring is as deep as fits, at most min(NST, 4 nkc) stages (E-buffer
        // reuse rule of epg_lik_tcw.cuh): the pass is HBM-bound and lives on the TMA bytes in flight -- measured on
        // config 5: 7 stages 3.6k cycles per 64 kB tile (the last sub-tile of the next tile is issued only when the
        // first GEMM2 of this one retires), against 2.9k at the HBM roofline
        a.off_E = a.off_B = a.off_G = a.off_gphi = a.off_cavc = 0;
        a.R = 0; a.resident = 0; a.slices = 1; a.NC = 1; a.combos = 1;
        const size_t fixed = al16(sizeof(double) * (size_t)NWARP * tcw::NCH) + sz_cs;
        int nst = std::min(tcw::NST, 4 * a.nkc);
        if (const char* e = getenv("EPGPU_NST")) nst = std::max(2, std::min(nst, atoi(e)));
        while (nst >= 2 && al16(1024 + tcw::Smem::total(nst)) + fixed > budget) --nst;
        if (nst < 2 || nst < a.nkc) return false;
        a.tc_nst = nst;
        size_t o = al16(1024 + tcw::Smem::total(nst));
        a.off_lp = o; o += al16(sizeof(double) * (size_t)NWARP * tcw::NCH);
        a.off_cs = o; o += sz_cs;
        a.smem_total = place_tail(o);
        return true;
    }
    if (a.use_tc) {
        if (a.tc_nst < tc::NF || a.tc_nst > tc::NST) a.tc_nst = tc::NST;
        size_t o = al16(1024 + tc::Smem::total(a.tc_nst));      // 1024: alignment slack for the swizzled tiles
        a.off_E = a.off_B = a.off_G = 0;
        a.R = 0; a.resident = 0; a.slices = 1; a.NC = 1; a.combos = 1;
        a.off_gphi = o; o += al16(sizeof(float) * (size_t)tc::NCH * d);
        a.off_cavc = o; o += al16(sizeof(float) * (size_t)tc::NCH * d);
        a.off_lp = o; o += al16(sizeof(double) * (size_t)NWARP * tc::NCH);
        a.off_cs = o; o += sz_cs;
        if (o > budget) return false;
        a.smem_total = place_tail(o);
        return true;
    }
    const int S = a.S;
    const int S4 = S / 4;
    a.combos = S4 * (CP / 4);
    if (a.combos <= NTHR) { a.NC = 1; a.slices = NTHR / a.combos; if (a.slices > 16) a.slices = 16; }
    else { a.NC = (a.combos + NTHR - 1) / NTHR; a.slices = 1; if (a.NC > NCMAX) return false; }
    a.R = NTHR;
    // what we would like to keep on chip besides the design matrix
    const size_t want_tail = sz_om + al16((size_t)V_NHOT * per_vec);
    for (;;) {
        const size_t szE = al16(sizeof(float) * (size_t)a.R * CP);
        const size_t szB = al16(sizeof(float) * (size_t)CP * S);
        const size_t szG = al16(sizeof(float) * (size_t)a.slices * CP * S);
        const size_t szg = al16(sizeof(float) * (size_t)CP * d);
        const size_t szl = al16(sizeof(double) * (size_t)NWARP * CP);
        const size_t rest = szE + szB + szG + 2 * szg + szl + sz_cs;
        const size_t xres = al16(sizeof(float) * (size_t)max_rows * S);
        const size_t xstream = al16(2 * sizeof(float) * (size_t)a.R * S);
        size_t xbytes;
        // the resident design matrix wins over the hot chain vectors only if both fit
        if (xres + rest + (want_tail <= 96 * 1024 ? want_tail : 0) <= budget) { a.resident = 1; xbytes = xres; }
        else { a.resident = 0; xbytes = xstream; }
        if (xbytes + rest <= budget) {
            size_t o = xbytes;
            a.off_E = o; o += szE;
            a.off_B = o; o += szB;
            a.off_G = o; o += szG;
            a.off_gphi = o; o += szg;
            a.off_cavc = o; o += szg;
            a.off_lp = o; o += szl;
            a.off_cs = o; o += sz_cs;
            a.smem_total = place_tail(o);
            return true;
        }
        if (a.R <= 32) return false;
        a.R /= 2;
    }
}

// shared-memory plan of the ping-pong kernel: [tensor-core pass buffers][site block 0][site block 1];
// a site block = [cavc][lp][chain scalars][omega][hot vectors (+ low tree-stack levels)]
bool plan_smem_pp(SamplerArgs& a, int d) {
    auto al16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
    const size_t per_vec = sizeof(float) * (size_t)a.C * a.P;
    const size_t sz_g = al16(sizeof(float) * (size_t)a.C * d);                // cavity terms of the chains
    const size_t sz_lp = al16(sizeof(double) * (size_t)NWARP * tc::NCH);
    const size_t sz_cs = al16((sizeof(ChainS) + sizeof(ChainStack)) * (size_t)a.C);
    const size_t sz_om = al16(sizeof(float) * ((size_t)d * d + d));
    const size_t site_min = sz_g + sz_lp + sz_cs + sz_om + al16((size_t)V_NHOT * per_vec);
    int nst_max = tc::NST;
    if (const char* e = getenv("EPGPU_NST")) nst_max = std::max(tc::NF, std::min(tc::NST, atoi(e)));
    for (int nst = nst_max; nst >= tc::NF; --nst) {
        const size_t tcsz = al16(1024 + tc::Smem::total(nst));
        if (tcsz + 2 * site_min > SMEM_BUDGET_1) continue;
        int lv = (int)((SMEM_BUDGET_1 - tcsz - 2 * site_min) / (2 * 4 * per_vec));
        if (lv > MAXDEPTH_CAP) lv = MAXDEPTH_CAP;
        a.tc_nst = nst; a.pp = 1;
        a.off_E = a.off_B = a.off_G = 0;
        a.R = 0; a.resident = 0; a.slices = 1; a.NC = 1; a.combos = 1;
        a.omega_smem = 1; a.hot_nvec = V_NHOT; a.hot_levels = lv;
        size_t o = tcsz;
        a.off_gphi = 0;                            // (not used by the tensor-core pass)
        a.off_cavc = o; o += sz_g;
        a.off_lp = o; o += sz_lp;
        a.off_cs = o; o += sz_cs;
        a.off_omega = o; o += sz_om;
        a.off_hot = o; o += al16((size_t)(V_NHOT + 4 * lv) * per_vec);
        a.site_stride = o - tcsz;
        a.smem_total = o + a.site_stride;
        return true;
    }
    return false;
}

int pad_chains(int C) { return C <= 4 ? 4 : (C <= 8 ? 8 : (C <= 16 ? 16 : 32)); }

template <typename F>
cudaError_t set_smem_attr(F f, size_t bytes) {
    return cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

}  // namespace

extern "C" {

int epg_upload_sites(epg_ctx* c, int model, int D, const int64_t* k_lim, const double* X, const int64_t* y,
                     const int32_t* j_ind, const int32_t* Jk) {
    if (!c->arr[EPG_Q]) return epg_fail_msg(c, "epg_upload_sites: call epg_init_state first");
    if (model != EPG_M1B && model != EPG_M2B && model != EPG_M3B && model != EPG_M4B && model != EPG_M5B)
        return epg_fail_msg(c, "unknown model id");
    if (D < 1 || D > 1000) return epg_fail_msg(c, "bad D");
    if (model_dphi(model, D) != c->d) return epg_fail_msg(c, "dphi of the model does not match the state dimension");
    if ((j_ind == nullptr) != (Jk == nullptr)) return epg_fail_msg(c, "j_ind and Jk must be given together");
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    epg_sites_free(c);
    epg_site_data* s = new epg_site_data();
    c->sites = s;
    const int K = c->K;
    s->model = model; s->D = D; s->K = K;
    int S = ((D + 1 + 3) / 4) * 4;
    if (((S / 4) & 1) == 0) S += 4;            // S = 4 * odd: conflict-free 128-bit row reads
    s->S = S;
    s->h_row0.assign(k_lim, k_lim + K + 1);
    const int64_t base = s->h_row0[0];
    for (auto& v : s->h_row0) v -= base;
    const int64_t N = s->h_row0[K];
    s->N = N;
    if (N < 1) return epg_fail_msg(c, "no rows");
    // group structure
    std::vector<int> gptr(K + 1, 0), grows;
    s->h_J.resize(K); s->h_p.resize(K);
    for (int k = 0; k < K; ++k) {
        const int64_t lo = s->h_row0[k], hi = s->h_row0[k + 1];
        if (hi <= lo) return epg_fail_msg(c, "empty site");
        const int J = Jk ? Jk[k] : 1;
        if (J < 1) return epg_fail_msg(c, "bad group count");
        gptr[k] = (int)grows.size();
        if (!j_ind) { grows.push_back(0); grows.push_back((int)(hi - lo)); }
        else {
            int64_t r = lo;
            for (int j = 0; j < J; ++j) {
                grows.push_back((int)(r - lo));
                while (r < hi && j_ind[base + r] == j) ++r;
            }
            if (r != hi) return epg_fail_msg(c, "j_ind must be sorted and in [0, J) within every site");
            grows.push_back((int)(hi - lo));
        }
        s->h_J[k] = J;
        s->h_p[k] = model_np(model, D, J);
        s->Pmax = std::max(s->Pmax, s->h_p[k]);
        s->Jmax = std::max(s->Jmax, J);
        s->max_rows = std::max<int64_t>(s->max_rows, hi - lo);
    }
    gptr[K] = (int)grows.size();
    s->Pmax = (s->Pmax + 31) & ~31;
    EPG_CHECK(c, cudaMalloc((void**)&s->X, sizeof(float) * (size_t)N * S));
    EPG_CHECK(c, cudaMalloc((void**)&s->y, sizeof(float) * (size_t)N));
    EPG_CHECK(c, cudaMalloc((void**)&s->row0, sizeof(int64_t) * (K + 1)));
    EPG_CHECK(c, cudaMalloc((void**)&s->grp_ptr, sizeof(int) * (K + 1)));
    EPG_CHECK(c, cudaMalloc((void**)&s->grp_rows, sizeof(int) * grows.size()));
    EPG_CHECK(c, cudaMemcpyAsync(s->row0, s->h_row0.data(), sizeof(int64_t) * (K + 1), cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, cudaMemcpyAsync(s->grp_ptr, gptr.data(), sizeof(int) * (K + 1), cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, cudaMemcpyAsync(s->grp_rows, grows.data(), sizeof(int) * grows.size(), cudaMemcpyHostToDevice, c->stream));
    // X, y: staged fp64 -> fp32 conversion in chunks
    const int64_t chunk_rows = std::max<int64_t>(1, (int64_t)(128u << 20) / (sizeof(double) * D));
    double* stage = nullptr;
    EPG_CHECK(c, cudaMalloc((void**)&stage, sizeof(double) * (size_t)chunk_rows * D));
    for (int64_t r = 0; r < N; r += chunk_rows) {
        const int64_t rows = std::min(chunk_rows, N - r);
        EPG_CHECK(c, cudaMemcpyAsync(stage, X + (size_t)(base + r) * D, sizeof(double) * (size_t)rows * D,
                                     cudaMemcpyHostToDevice, c->stream));
        const int64_t tot = rows * S;
        k_convert_x<<<(unsigned)((tot + 255) / 256), 256, 0, c->stream>>>(stage, s->X + (size_t)r * S, rows, D, S);
        c->launches++;
        EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    }
    {
        int64_t* ys = reinterpret_cast<int64_t*>(stage);
        const int64_t ychunk = chunk_rows * D;    // same bytes
        for (int64_t r = 0; r < N; r += ychunk) {
            const int64_t rows = std::min(ychunk, N - r);
            EPG_CHECK(c, cudaMemcpyAsync(ys, y + base + r, sizeof(int64_t) * (size_t)rows, cudaMemcpyHostToDevice, c->stream));
            k_convert_y<<<(unsigned)((rows + 255) / 256), 256, 0, c->stream>>>(ys, s->y + r, rows);
            c->launches++;
            EPG_CHECK(c, cudaStreamSynchronize(c->stream));
        }
    }
    EPG_CHECK(c, cudaFree(stage));
    EPG_CHECK(c, cudaGetLastError());
    // tensor-core paths: bf16 copy [N][pitch] + TMA descriptor (single-group sites, D+1 <= 256).  D+1 <= 64: one
    // 64-column box per 128-row tile (pitch 64); wider: nkc boxes per tile, pitch = D+1 rounded up to 16 columns
    // (32-byte sectors); the columns of the last box beyond the pitch are out of bounds (zero-filled by TMA)
    s->tc_ok = false;
    memset(&s->tmap, 0, sizeof(s->tmap));
    if (s->Jmax == 1 && D + 1 <= tcw::KWT) {
        s->nkc = (D + 1 + tc::KW - 1) / tc::KW;
        s->xb_pitch = s->nkc == 1 ? tc::KW : ((D + 1 + 15) / 16) * 16;
        // (measured and not adopted: dense rows for D+1 < 57 -- pitch D+1 rounded up to 8 columns, the rest of the
        //  64-column box out of bounds -- cut the L2 -> SM bytes of a tile by 12 % (config 4) / 62 % (config 3) and
        //  changed nothing: 26.9k vs 27.0k and 13.6k vs 13.3k cycles per pass; the tile phase is not bound by L2 bytes)
        const int xm_stride = tc::KW * s->nkc;
        EPG_CHECK(c, cudaMalloc((void**)&s->Xb, sizeof(__nv_bfloat16) * (size_t)N * s->xb_pitch));
        // per-site column means (fp64 on the host, stored as fp32) the bf16 copy is centred on
        std::vector<float> xm((size_t)K * xm_stride, 0.0f);
        {
            std::vector<double> acc(D);
            for (int k = 0; k < K; ++k) {
                std::fill(acc.begin(), acc.end(), 0.0);
                const int64_t lo = s->h_row0[k], hi = s->h_row0[k + 1];
                for (int64_t r = lo; r < hi; ++r) {
                    const double* xr = X + (size_t)(base + r) * D;
                    for (int j = 0; j < D; ++j) acc[j] += xr[j];
                }
                for (int j = 0; j < D; ++j) xm[(size_t)k * xm_stride + j] = (float)(acc[j] / (double)(hi - lo));
            }
        }
        EPG_CHECK(c, cudaMalloc((void**)&s->xmean, sizeof(float) * xm.size()));
        EPG_CHECK(c, cudaMemcpyAsync(s->xmean, xm.data(), sizeof(float) * xm.size(), cudaMemcpyHostToDevice, c->stream));
        const int64_t tot = N * s->xb_pitch;
        k_convert_xb<<<(unsigned)((tot + 255) / 256), 256, 0, c->stream>>>(s->X, s->Xb, N, S, D, s->xmean, s->row0, K,
                                                                        s->xb_pitch, xm_stride);
        c->launches++;
        EPG_CHECK(c, cudaStreamSynchronize(c->stream));
        typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        EPG_CHECK(c, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (fn && qres == cudaDriverEntryPointSuccess) {
            const cuuint64_t gdim[2] = {(cuuint64_t)s->xb_pitch, (cuuint64_t)N};
            const cuuint64_t gstride[1] = {(cuuint64_t)s->xb_pitch * 2};
            const cuuint32_t box[2] = {(cuuint32_t)tc::KW, (cuuint32_t)tc::TILE_M};
            const cuuint32_t estr[2] = {1, 1};
            const CUresult r = ((encode_fn)fn)(&s->tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, s->Xb, gdim, gstride, box, estr,
                                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            s->tc_ok = (r == CUDA_SUCCESS);
        }
        if (s->tc_ok)        // wide pass scratch: gradient halves [K][2][32][256] + cavity terms [K][32][d]
            EPG_CHECK(c, cudaMalloc((void**)&s->gout_w, sizeof(float) * (size_t)K * tcw::NCH * (2 * tcw::KWT + c->d)));
    }
    return 0;
}

int epg_set_option(epg_ctx* c, const char* name, double value) {
    if (!name) return epg_fail_msg(c, "epg_set_option: null name");
    if (strcmp(name, "use_tc") == 0) {
        if (!c->sites) return epg_fail_msg(c, "epg_set_option(use_tc): upload the sites first");
        c->sites->use_tc = value != 0.0;
        return 0;
    }
    if (strcmp(name, "param_stats") == 0) {
        if (!c->sites) return epg_fail_msg(c, "epg_set_option(param_stats): upload the sites first");
        c->sites->param_stats = value != 0.0;
        return 0;
    }
    if (strcmp(name, "sampler_params") == 0) {
        if (!c->sites) return epg_fail_msg(c, "epg_set_option(sampler_params): upload the sites first");
        c->sites->sampler_params = value != 0.0;
        return 0;
    }
    if (strcmp(name, "carry_adapt") == 0) {
        if (!c->sites) return epg_fail_msg(c, "epg_set_option(carry_adapt): upload the sites first");
        c->sites->carry_adapt = value != 0.0;
        return 0;
    }
    if (strcmp(name, "metric_reg") == 0) {
        if (!c->sites) return epg_fail_msg(c, "epg_set_option(metric_reg): upload the sites first");
        c->sites->metric_reg = (float)value;
        return 0;
    }
    if (strcmp(name, "pingpong") == 0) {
        if (!c->sites) return epg_fail_msg(c, "epg_set_option(pingpong): upload the sites first");
        c->sites->pp_mode = (int)value;
        return 0;
    }
    return epg_fail_msg(c, std::string("epg_set_option: unknown option ") + name);
}

int epg_num_params(epg_ctx* c, int k) {
    if (!c->sites || k < 0 || k >= c->K) return -1;
    return c->sites->h_p[k];
}

static int fill_args(epg_ctx* c, SamplerArgs& a, int C, int CP, int n_sites = 1, bool need_allhot = false) {
    epg_site_data* s = c->sites;
    a.X = s->X; a.y = s->y; a.row0 = s->row0; a.grp_ptr = s->grp_ptr; a.grp_rows = s->grp_rows;
    a.xmean = s->xmean; a.order = nullptr;
    a.model = s->model; a.D = s->D; a.S = s->S; a.d = c->d;
    a.cavQ = c->arr[EPG_CAVQ]; a.cavm = c->arr[EPG_CAVM];
    a.P = s->Pmax; a.C = C;
    const size_t need = sizeof(float) * (size_t)c->K * C * NVEC * s->Pmax;
    if (need > s->chain_mem_bytes) {
        if (s->chain_mem) cudaFree(s->chain_mem);
        s->chain_mem = nullptr; s->chain_mem_bytes = 0;
        EPG_CHECK(c, cudaMalloc((void**)&s->chain_mem, need));
        s->chain_mem_bytes = need;
    }
    const size_t n_lq = (size_t)c->K * C * s->Pmax;               // last_q | last_minv | last_eps | last_metric
    const size_t need_lq = sizeof(float) * (2 * n_lq + 2 * (size_t)c->K * C);
    if (need_lq > s->last_q_bytes || s->last_C != C) {
        if (s->last_q) cudaFree(s->last_q);
        s->last_q = nullptr; s->last_q_bytes = 0;
        EPG_CHECK(c, cudaMalloc((void**)&s->last_q, need_lq));
        EPG_CHECK(c, cudaMemsetAsync(s->last_q, 0, need_lq, c->stream));
        s->last_q_bytes = need_lq; s->last_C = C;
    }
    EPG_CHECK(c, epg_reserve((void**)&s->omega, &s->omega_bytes, sizeof(float) * (size_t)c->K * (c->d * c->d + c->d)));
    EPG_CHECK(c, epg_reserve((void**)&s->out, &s->out_bytes, sizeof(double) * (size_t)c->K * 8 + sizeof(uint32_t) * ((size_t)c->K + 4)));
    a.chain_mem = s->chain_mem; a.last_q = s->last_q; a.omega = s->omega; a.out = s->out;
    a.last_minv = s->last_q + n_lq; a.last_eps = s->last_q + 2 * n_lq; a.carry_adapt = s->carry_adapt;
    a.last_metric = a.last_eps + (size_t)c->K * C;
    a.metric_reg = s->metric_reg;
    a.tstats = nullptr;
    if (s->param_stats) {
        EPG_CHECK(c, epg_reserve((void**)&s->tstats, &s->tstats_bytes, sizeof(double) * (size_t)c->K * 2 * s->Pmax));
        a.tstats = s->tstats;
    }
    // tensor-core pass: 1 = D+1 <= 64 and <= 16 chains (chain vectors in shared memory), 2 = wide (D+1 <= 256, <= 32 chains)
    a.use_tc = (s->tc_ok && s->use_tc) ? ((s->nkc == 1 && C <= tc::NCH) ? 1 : (C <= tcw::NCH ? 2 : 0)) : 0;
    a.nkc = s->nkc; a.xm_stride = tc::KW * s->nkc; a.gout_w = s->gout_w;
    a.cavc_g = a.use_tc == 2 ? s->gout_w + (size_t)c->K * 2 * tcw::NCH * tcw::KWT : nullptr;
    if (a.use_tc == 2) {
        if (!plan_smem(a, CP, s->max_rows, c->d)) { a.use_tc = 0; }
        else return 0;
    }
    // More sites than SMs: the ping-pong kernel (two sites per persistent CTA) if both per-site blocks fit.
    a.tc_nst = tc::NST;
    a.pp = 0;
    int mode = s->pp_mode;
    if (const char* e = getenv("EPGPU_PP")) mode = atoi(e);
    // (the kernel doubles the number of sites streamed concurrently: it only pays while the bf16 design
    //  matrices of 2 x SMs sites stay resident in L2 -- measured: config 4, 640 KB per site, does not)
    const double resident_bytes = 2.0 * c->num_sms * (double)s->max_rows * tc::KW * 2.0;
    const int pp = a.use_tc == 1 && s->Jmax == 1 && n_sites > 1 &&
                   (mode == 2 || (mode == 1 && n_sites > c->num_sms && resident_bytes <= 0.75 * c->l2_bytes));
    if (pp && plan_smem_pp(a, c->d)) return 0;
    a.pp = 0;
    // Ring depth vs tree-stack levels in shared memory (measured on config 4): the pass gains up to 5 stages
    // (29.2k -> 25.4k cycles per tick), the chain phase up to 5 levels (12.3k -> 7.3k): take the deepest ring
    // that still leaves 5 levels (or all the sampler can use) on chip.
    a.tc_nst = tc::NF;
    if (a.use_tc) {
        const int want = std::min(5, std::min(MAXDEPTH_CAP, a.max_depth > 0 ? a.max_depth : 10));
        for (int nst = tc::NST; nst > tc::NF; --nst) {
            a.tc_nst = nst;
            if (plan_smem(a, CP, s->max_rows, c->d) && a.hot_nvec >= V_NHOT && a.hot_levels >= want) break;
            a.tc_nst = tc::NF;
        }
    }
    if (const char* e = getenv("EPGPU_NST")) a.tc_nst = atoi(e);
    if (!plan_smem(a, CP, s->max_rows, c->d)) return epg_fail_msg(c, "sampler: shapes exceed the shared-memory plan");
    if (need_allhot && a.use_tc && !(a.omega_smem && a.hot_nvec >= V_NHOT)) {
        // the tensor-core kernels address the chain vectors as shared memory: without room for all of them the
        // fp32 SIMT kernel takes over
        a.use_tc = 0;
        if (!plan_smem(a, CP, s->max_rows, c->d)) return epg_fail_msg(c, "sampler: shapes exceed the shared-memory plan");
    }
    return 0;
}

// what epg_last_plan reports (field order: include/epgpu.h)
static void record_plan(epg_site_data* s, const SamplerArgs& a, int kernel, int CP) {
    const int chain_pad = a.use_tc == 2 ? tcw::NCH : (a.use_tc ? (a.C <= 4 ? 4 : (a.C <= 8 ? 8 : 16)) : CP);
    const int32_t v[EPG_PLAN_FIELDS] = {kernel, a.use_tc, chain_pad, a.use_tc ? a.tc_nst : 0, a.resident, a.R,
                                        a.slices, a.NC, a.hot_nvec, a.hot_levels, a.omega_smem, (int32_t)a.smem_total};
    memcpy(s->plan, v, sizeof(v));
}

int epg_reserve_draws(epg_ctx* c, int n);

int epg_set_inits(epg_ctx* c, int k0, int k1, int chains, const double* q) {
    if (!c->sites) return epg_fail_msg(c, "epg_set_inits: no site data (epg_upload_sites)");
    if (k0 < 0 || k1 > c->K || k0 >= k1 || !q) return epg_fail_msg(c, "epg_set_inits: bad args");
    if (chains < 1 || chains > 32) return epg_fail_msg(c, "chains must be in 1..32");
    epg_site_data* s = c->sites;
    const size_t P = s->Pmax;
    if (s->inits_C != chains || !s->inits) {
        // (a new chain count drops the starting points of every site)
        EPG_CHECK(c, cudaStreamSynchronize(c->stream));
        cudaFree(s->inits);
        s->inits = nullptr; s->inits_C = 0;
        EPG_CHECK(c, cudaMalloc((void**)&s->inits, sizeof(float) * (size_t)c->K * chains * P));
        s->inits_C = chains;
        s->h_inits_set.assign((size_t)c->K, 0);
    }
    std::vector<float> h((size_t)(k1 - k0) * chains * P);
    for (size_t i = 0; i < h.size(); ++i) h[i] = (float)q[i];
    EPG_CHECK(c, cudaMemcpyAsync(s->inits + (size_t)k0 * chains * P, h.data(), sizeof(float) * h.size(),
                                 cudaMemcpyHostToDevice, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));           // (h is a local)
    std::fill(s->h_inits_set.begin() + k0, s->h_inits_set.begin() + k1, (unsigned char)1);
    return 0;
}

static const epg_sampler_adapt k_stan_adapt = {1.0, 0.0, 0.05, 0.75, 10.0, 2.0, 1, 75, 50, 25, {0}};

int epg_tilted_sample(epg_ctx* c, int k0, int k1, const uint32_t* seeds, const epg_sampler_opts* o,
                      double* msteps_out, double* mrhat_out, int64_t* n_leapfrog_out, double* seconds) {
    return epg_tilted_sample_ex(c, k0, k1, seeds, o, nullptr, msteps_out, mrhat_out, n_leapfrog_out, seconds);
}

int epg_tilted_sample_ex(epg_ctx* c, int k0, int k1, const uint32_t* seeds, const epg_sampler_opts* o,
                         const epg_sampler_adapt* ad, double* msteps_out, double* mrhat_out,
                         int64_t* n_leapfrog_out, double* seconds) {
    if (!c->sites) return epg_fail_msg(c, "epg_tilted_sample: no site data (epg_upload_sites)");
    if (k0 < 0 || k1 > c->K || k0 >= k1 || !seeds || !o) return epg_fail_msg(c, "epg_tilted_sample: bad args");
    if (!ad) ad = &k_stan_adapt;
    if (o->chains < 1 || o->chains > 32) return epg_fail_msg(c, "chains must be in 1..32");
    if (o->thin < 1) return epg_fail_msg(c, "thin must be >= 1");
    if (o->iter < 1) return epg_fail_msg(c, "iter must be positive");
    if (o->metric < EPG_METRIC_DIAG || o->metric > EPG_METRIC_UNIT)
        return epg_fail_msg(c, "metric must be 0 (diag_e), 1 (dense_e) or 2 (unit_e)");
    if (o->init_mode < 0 || o->init_mode > 3) return epg_fail_msg(c, "init_mode must be 0, 1, 2 or 3");
    auto pos = [](double v) { return v > 0.0 && std::isfinite(v); };
    if (!pos(ad->stepsize) || !((float)ad->stepsize > 0.0f) || !std::isfinite((float)ad->stepsize))
        return epg_fail_msg(c, "stepsize must be positive and finite");
    if (!(ad->stepsize_jitter >= 0.0 && ad->stepsize_jitter <= 1.0))
        return epg_fail_msg(c, "stepsize_jitter must be in [0, 1]");
    if (!pos(ad->gamma)) return epg_fail_msg(c, "adapt_gamma must be positive");
    if (!pos(ad->kappa)) return epg_fail_msg(c, "adapt_kappa must be positive");
    if (!pos(ad->t0)) return epg_fail_msg(c, "adapt_t0 must be positive");
    if (!pos(ad->init_radius)) return epg_fail_msg(c, "init_radius must be positive and finite");
    if (ad->engaged != 0 && ad->engaged != 1) return epg_fail_msg(c, "engaged must be 0 or 1");
    if (ad->init_buffer < 0 || ad->term_buffer < 0) return epg_fail_msg(c, "adaptation buffers must be >= 0");
    if (ad->window < 1) return epg_fail_msg(c, "adapt_window must be >= 1");
    const int warm = o->warmup < 0 ? o->iter / 2 : o->warmup;
    if (warm >= o->iter) return epg_fail_msg(c, "warmup must be smaller than iter");
    const int C = o->chains, CP = pad_chains(C);
    const int n_save = (o->iter - warm + o->thin - 1) / o->thin;
    const int n = C * n_save;
    epg_site_data* s = c->sites;
    if (o->init_mode == 2 && (s->last_C != C || !s->last_q)) return epg_fail_msg(c, "init_prev without previous draws");
    if (o->init_mode == 3 && (s->inits_C != C || !s->inits ||
                              !std::all_of(s->h_inits_set.begin() + k0, s->h_inits_set.begin() + k1,
                                           [](unsigned char f) { return f != 0; })))
        return epg_fail_msg(c, "init mode 3 (given): epg_set_inits has not set these sites for this chain count");
    if (int rc = epg_reserve_draws(c, n)) return rc;
    SamplerArgs a;
    memset(&a, 0, sizeof(a));
    if (int rc = fill_args(c, a, C, CP, k1 - k0, true)) return rc;
    a.iter = o->iter; a.warmup = warm; a.init_mode = o->init_mode;
    a.thin = o->thin; a.n_save = n_save;
    a.gamma = ad->gamma; a.kappa = ad->kappa; a.t0 = ad->t0;
    a.stepsize = (float)ad->stepsize; a.jitter = (float)ad->stepsize_jitter; a.init_r = (float)ad->init_radius;
    a.adapt_engaged = ad->engaged;
    a.inits = o->init_mode == 3 ? s->inits : nullptr;
    a.metric = o->metric;
    if (a.metric == EPG_METRIC_DENSE) {
        // (allocated with the first dense_e run; a larger chain count reallocates them, and the carried state with
        //  them, but then last_q is reallocated and zeroed as well, so nothing is carried)
        const size_t nch = (size_t)c->K * C;
        EPG_CHECK(c, epg_reserve((void**)&s->dense, &s->dense_bytes, sizeof(float) * nch * dense_floats(s->Pmax)));
        EPG_CHECK(c, epg_reserve((void**)&s->dense_ws, &s->dense_ws_bytes, sizeof(double) * nch * s->Pmax * s->Pmax));
        a.dense = s->dense; a.dense_ws = s->dense_ws;
    }
    a.max_depth = o->max_treedepth > 0 ? std::min(o->max_treedepth, MAXDEPTH_CAP) : 10;
    a.delta = o->adapt_delta > 0 ? o->adapt_delta : 0.8;
    // Stan 2.17 windowed_adaptation::set_window_params: (init buffer, term buffer, window), 75 / 50 / 25 by
    // default, rescaled to 15 % / 10 % / the rest when they do not fit the warm-up
    a.win_init = ad->init_buffer; a.win_term = ad->term_buffer; a.win_base = ad->window;
    if (warm >= 20 && a.win_init + a.win_base + a.win_term > warm) {
        a.win_init = (int)(0.15 * warm); a.win_term = (int)(0.1 * warm);
        a.win_base = warm - (a.win_init + a.win_term);
    }
    // HMC diagnostics: one block per chain of this chain count (another count drops the diagnostics and records
    // of every site, as epg_set_inits drops its starting points); records of this shape (another shape drops
    // those of every other site)
    if (s->hmc_C != C || !s->hmc) {
        EPG_CHECK(c, cudaStreamSynchronize(c->stream));
        cudaFree(s->hmc);
        s->hmc = nullptr; s->hmc_C = 0;
        EPG_CHECK(c, cudaMalloc(&s->hmc, sizeof(HmcChain) * (size_t)c->K * C));
        s->hmc_C = C;
        s->h_hmc_ok.assign((size_t)c->K, 0);
        s->h_rec_ok.assign((size_t)c->K, 0);
    }
    a.hmc = static_cast<HmcChain*>(s->hmc);
    const int n_rec_warm = (warm + o->thin - 1) / o->thin;
    if (s->sampler_params) {
        if (s->rec_iter != o->iter || s->rec_warmup != warm || s->rec_thin != o->thin) {
            std::fill(s->h_rec_ok.begin(), s->h_rec_ok.end(), (unsigned char)0);
            s->rec_iter = o->iter; s->rec_warmup = warm; s->rec_thin = o->thin;
            s->rec_n = n_rec_warm + n_save; s->rec_nw = n_rec_warm;
        }
        const size_t need = sizeof(double) * HMC_REC * (size_t)c->K * C * s->rec_n;
        if (need > s->rec_bytes) EPG_CHECK(c, cudaStreamSynchronize(c->stream));     // (epg_reserve reallocates)
        EPG_CHECK(c, epg_reserve((void**)&s->rec, &s->rec_bytes, need));
        a.rec = s->rec; a.n_rec = s->rec_n; a.n_rec_warm = n_rec_warm;
    }
    uint32_t* dseeds = reinterpret_cast<uint32_t*>(s->out + (size_t)c->K * 8);
    EPG_CHECK(c, cudaMemcpyAsync(dseeds, seeds, sizeof(uint32_t) * (k1 - k0), cudaMemcpyHostToDevice, c->stream));
    a.seeds = dseeds;
    a.draws = c->draws; a.n_draws = n; a.k0 = k0;
    // launch order: sites that spent the most gradient evaluations in the previous run first (longest
    // processing time first): a straggler -- e.g. an ill-conditioned site that saturates the tree depth on
    // every transition -- must not start in the last wave
    if ((int)s->h_cost.size() == c->K && k1 - k0 > 1) {
        std::vector<int> ord(k1 - k0);
        for (int i = 0; i < k1 - k0; ++i) ord[i] = i;
        std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return s->h_cost[k0 + x] > s->h_cost[k0 + y]; });
        if (!s->order) EPG_CHECK(c, cudaMalloc((void**)&s->order, sizeof(int) * (size_t)c->K));
        EPG_CHECK(c, cudaMemcpyAsync(s->order, ord.data(), sizeof(int) * ord.size(), cudaMemcpyHostToDevice, c->stream));
        EPG_CHECK(c, cudaStreamSynchronize(c->stream));           // (ord is a local)
        a.order = s->order;
    }
    // sites marked by epg_reinit_sites: random starting points instead of the previous last draws (consumed here)
    if (o->init_mode == 2 && (int)s->h_reinit.size() == c->K &&
        std::any_of(s->h_reinit.begin() + k0, s->h_reinit.begin() + k1, [](unsigned char f) { return f != 0; })) {
        if (!s->reinit) EPG_CHECK(c, cudaMalloc((void**)&s->reinit, (size_t)c->K));
        EPG_CHECK(c, cudaMemcpyAsync(s->reinit, s->h_reinit.data(), (size_t)c->K, cudaMemcpyHostToDevice, c->stream));
        EPG_CHECK(c, cudaStreamSynchronize(c->stream));
        a.reinit = s->reinit;
    }
    if ((int)s->h_reinit.size() == c->K) std::fill(s->h_reinit.begin() + k0, s->h_reinit.begin() + k1, (unsigned char)0);
#ifdef EPG_TC_EXPERIMENT
    { int kn = getenv("EPGPU_KNOBS") ? atoi(getenv("EPGPU_KNOBS")) : 0; cudaMemcpyToSymbol(tc::g_knobs, &kn, sizeof(int)); }
#endif
    cudaEvent_t e0, e1;
    EPG_CHECK(c, cudaEventCreate(&e0));
    EPG_CHECK(c, cudaEventCreate(&e1));
    EPG_CHECK(c, cudaEventRecord(e0, c->stream));
    const bool dense = a.metric == EPG_METRIC_DENSE;
#define LAUNCH_NUTS_M(CPV, TC, DN)                                                \
    {                                                                             \
        EPG_CHECK(c, set_smem_attr(k_nuts<CPV, TC, DN>, a.smem_total));           \
        k_nuts<CPV, TC, DN><<<k1 - k0, TC ? tc::NTHREADS : NTHR, a.smem_total, c->stream>>>(a, s->tmap); \
    }
#define LAUNCH_NUTS(CPV, TC) { if (dense) LAUNCH_NUTS_M(CPV, TC, true) else LAUNCH_NUTS_M(CPV, TC, false) }
    if (a.pp) {
        int* queue = reinterpret_cast<int*>(dseeds + c->K);
        EPG_CHECK(c, cudaMemsetAsync(queue, 0, sizeof(int), c->stream));
        auto kpp = dense ? k_nuts_pp<true> : k_nuts_pp<false>;
        EPG_CHECK(c, set_smem_attr(kpp, a.smem_total));
        int grid = (k1 - k0) > c->num_sms ? c->num_sms : (k1 - k0 + 1) / 2;     // (forced mode: two sites per CTA)
        if (const char* e = getenv("EPGPU_PP_GRID")) grid = std::max(1, std::min(atoi(e), k1 - k0));
        kpp<<<grid, PP_THREADS, a.smem_total, c->stream>>>(a, s->tmap, k1 - k0, queue);
    }
    else if (a.use_tc == 2) LAUNCH_NUTS(32, 2)
    else if (a.use_tc) LAUNCH_NUTS(32, 1)
    else if (CP == 4) LAUNCH_NUTS(4, 0) else if (CP == 8) LAUNCH_NUTS(8, 0)
    else if (CP == 16) LAUNCH_NUTS(16, 0) else LAUNCH_NUTS(32, 0)
    c->launches++;
    record_plan(s, a, a.pp ? 2 : 1, CP);
    EPG_CHECK(c, cudaGetLastError());
    EPG_CHECK(c, cudaEventRecord(e1, c->stream));
    EPG_CHECK(c, cudaEventSynchronize(e1));
    float ms = 0.f;
    EPG_CHECK(c, cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (seconds) *seconds = ms * 1e-3;
    std::vector<double> out((size_t)(k1 - k0) * 8);
    EPG_CHECK(c, cudaMemcpyAsync(out.data(), s->out + (size_t)k0 * 8, sizeof(double) * out.size(),
                                 cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    std::fill(s->h_hmc_ok.begin() + k0, s->h_hmc_ok.begin() + k1, (unsigned char)1);
    std::fill(s->h_rec_ok.begin() + k0, s->h_rec_ok.begin() + k1, (unsigned char)(a.rec ? 1 : 0));
    if ((int)s->h_cost.size() != c->K) s->h_cost.assign((size_t)c->K, 0.0);
    for (int i = 0; i < k1 - k0; ++i) {
        s->h_cost[k0 + i] = out[8 * i + 6];                      // ticks = the site's sequential length
        if (msteps_out) msteps_out[i] = out[8 * i + 0];
        if (mrhat_out) mrhat_out[i] = out[8 * i + 1];
        if (n_leapfrog_out) n_leapfrog_out[i] = (int64_t)out[8 * i + 2];
    }
#ifdef EPG_TC_PROFILE
    if (getenv("EPGPU_TRACE")) {
        long long hp[8];
        cudaMemcpyFromSymbol(hp, tc::g_prof, sizeof(hp));
        fprintf(stderr, "[epgpu] epilogue cycles/tile: wait_f %.0f ld %.0f math %.0f wait_e %.0f sts %.0f fence %.0f arrive %.0f (tiles %lld)\n",
                (double)hp[0] / hp[7], (double)hp[1] / hp[7], (double)hp[2] / hp[7], (double)hp[3] / hp[7], (double)hp[4] / hp[7], (double)hp[5] / hp[7], (double)hp[6] / hp[7], hp[7]);
        cudaMemcpyFromSymbol(hp, tc::g_prof2, sizeof(hp));
        fprintf(stderr, "[epgpu] lik pass cycles/tick (thread 0): build %.0f pass %.0f sync %.0f chainrule+tail %.0f\n", (double)hp[2] / hp[6], (double)hp[3] / hp[6], (double)hp[4] / hp[6], (double)hp[5] / hp[6]);
        fprintf(stderr, "[epgpu] mma thread cycles/tile: wait_e %.0f issue_g2 %.0f commits %.0f gemm1(wait full+issue) %.0f (tiles %lld)\n",
                (double)hp[0] / hp[7], (double)hp[1] / hp[7], (double)hp[2] / hp[7], (double)hp[3] / hp[7], hp[7]);
    }
#endif
#ifdef EPG_TC_TIMELINE
    if (getenv("EPGPU_TRACE"))
        {
            long long tl[8][64], tx[8];
            cudaMemcpyFromSymbol(tl, tc::g_tl, sizeof(tl));
            cudaMemcpyFromSymbol(tx, tc::g_tlx, sizeof(tx));
            const long long z = tx[0];
            fprintf(stderr, "[epgpu] timeline (cycles from pass start): prologue_end %lld tiles_done %lld gready %lld end %lld\n",
                    tx[1] - z, tx[2] - z, tx[3] - z, tx[4] - z);
            fprintf(stderr, "[epgpu] tile: tma_issue full_seen g1_issued f_seen e_arrived e_seen g2_issued\n");
            for (int t = 0; t < 44; ++t) {
                fprintf(stderr, "[epgpu] %2d:", t);
                for (int e = 0; e < 7; ++e) fprintf(stderr, " %7lld", tl[e][t] ? tl[e][t] - z : -1);
                fprintf(stderr, "\n");
            }
        }
#endif
    if (getenv("EPGPU_TRACE")) {
        double cc = 0, cl = 0, nt = 0;
        for (int i = 0; i < k1 - k0; ++i) { cc += out[8 * i + 4]; cl += out[8 * i + 5]; nt += out[8 * i + 6]; }
        fprintf(stderr, "[epgpu] sampler %d sites: %.3f s, ticks/site %.0f, cycles/tick chain %.0f lik %.0f (tc=%d pp=%d nst=%d levels=%d smem=%zu)\n",
                k1 - k0, ms * 1e-3, nt / (k1 - k0), cc / nt, cl / nt, a.use_tc, a.pp, a.tc_nst, a.hot_levels, a.smem_total);
    }
    return 0;
}

int epg_get_param_stats(epg_ctx* c, int k0, int k1, double* mean_out, double* ssd_out) {
    if (!c->sites || !c->sites->tstats || k0 < 0 || k1 > c->K || k0 >= k1 || !mean_out || !ssd_out)
        return epg_fail_msg(c, "epg_get_param_stats: enable option param_stats before sampling");
    epg_site_data* s = c->sites;
    const size_t P = s->Pmax;
    std::vector<double> h((size_t)(k1 - k0) * 2 * P);
    EPG_CHECK(c, cudaMemcpyAsync(h.data(), s->tstats + (size_t)k0 * 2 * P, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    for (int k = 0; k < k1 - k0; ++k)
        for (size_t i = 0; i < P; ++i) {
            mean_out[(size_t)k * P + i] = h[(size_t)k * 2 * P + i];
            ssd_out[(size_t)k * P + i] = h[(size_t)k * 2 * P + P + i];
        }
    return 0;
}

int epg_get_hmc_diag(epg_ctx* c, int k0, int k1, double* out) {
    epg_site_data* s = c->sites;
    if (!s || k0 < 0 || k1 > c->K || k0 >= k1) return epg_fail_msg(c, "epg_get_hmc_diag: bad args");
    if ((int)s->h_hmc_ok.size() != c->K ||
        !std::all_of(s->h_hmc_ok.begin() + k0, s->h_hmc_ok.begin() + k1, [](unsigned char f) { return f != 0; }))
        return epg_fail_msg(c, "epg_get_hmc_diag: no sampling run of these sites at the current chain count");
    const int C = s->hmc_C;
    if (!out) return C;
    std::vector<HmcChain> h((size_t)(k1 - k0) * C);
    EPG_CHECK(c, cudaMemcpyAsync(h.data(), static_cast<HmcChain*>(s->hmc) + (size_t)k0 * C, sizeof(HmcChain) * h.size(),
                                 cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    for (size_t i = 0; i < h.size(); ++i) {
        out[EPG_DIAG_FIELDS * i + 0] = h[i].n_saved;
        out[EPG_DIAG_FIELDS * i + 1] = h[i].n_div;
        out[EPG_DIAG_FIELDS * i + 2] = h[i].n_maxd;
        out[EPG_DIAG_FIELDS * i + 3] = h[i].ebfmi;
    }
    return C;
}

int epg_get_sampler_params(epg_ctx* c, int k0, int k1, int inc_warmup, double* out) {
    epg_site_data* s = c->sites;
    if (!s || k0 < 0 || k1 > c->K || k0 >= k1) return epg_fail_msg(c, "epg_get_sampler_params: bad args");
    if ((int)s->h_rec_ok.size() != c->K || !s->rec ||
        !std::all_of(s->h_rec_ok.begin() + k0, s->h_rec_ok.begin() + k1, [](unsigned char f) { return f != 0; }))
        return epg_fail_msg(c, "epg_get_sampler_params: the most recent run of these sites did not record "
                               "(option sampler_params), or a later recording run had another shape");
    const int skip = inc_warmup ? 0 : s->rec_nw, n = s->rec_n - skip;
    if (!out) return n;
    const size_t nch = (size_t)(k1 - k0) * s->hmc_C, row = (size_t)HMC_REC * s->rec_n;
    std::vector<double> h(nch * row);
    EPG_CHECK(c, cudaMemcpyAsync(h.data(), s->rec + (size_t)k0 * s->hmc_C * row, sizeof(double) * h.size(),
                                 cudaMemcpyDeviceToHost, c->stream));
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    for (size_t ch = 0; ch < nch; ++ch)
        memcpy(out + ch * HMC_REC * n, h.data() + ch * row + (size_t)HMC_REC * skip, sizeof(double) * HMC_REC * n);
    return n;
}

int epg_max_params(epg_ctx* c) { return c->sites ? c->sites->Pmax : -1; }

int epg_get_adapt(epg_ctx* c, int k, float* minv_out, float* eps_out) {
    if (!c->sites || k < 0 || k >= c->K || !c->sites->last_q || c->sites->last_C < 1)
        return epg_fail_msg(c, "epg_get_adapt: no finished sampling run");
    epg_site_data* s = c->sites;
    const int C = s->last_C;
    const size_t n_lq = (size_t)c->K * C * s->Pmax;
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    if (minv_out) EPG_CHECK(c, cudaMemcpy(minv_out, s->last_q + n_lq + (size_t)k * C * s->Pmax, sizeof(float) * (size_t)C * s->Pmax, cudaMemcpyDeviceToHost));
    if (eps_out) EPG_CHECK(c, cudaMemcpy(eps_out, s->last_q + 2 * n_lq + (size_t)k * C, sizeof(float) * C, cudaMemcpyDeviceToHost));
    return 0;
}

int epg_get_metric(epg_ctx* c, int k, float* out) {
    if (!c->sites || k < 0 || k >= c->K || !c->sites->last_q || c->sites->last_C < 1 || !out)
        return epg_fail_msg(c, "epg_get_metric: no finished sampling run");
    epg_site_data* s = c->sites;
    const int C = s->last_C;
    const size_t P = s->Pmax, n_lq = (size_t)c->K * C * P;
    std::vector<float> minv((size_t)C * P), met(C);
    EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    EPG_CHECK(c, cudaMemcpy(minv.data(), s->last_q + n_lq + (size_t)k * C * P, sizeof(float) * minv.size(), cudaMemcpyDeviceToHost));
    EPG_CHECK(c, cudaMemcpy(met.data(), s->last_q + 2 * n_lq + (size_t)c->K * C + (size_t)k * C, sizeof(float) * C,
                            cudaMemcpyDeviceToHost));
    for (int ch = 0; ch < C; ++ch) {
        float* o = out + (size_t)ch * P * P;
        if (met[ch] == (float)EPG_METRIC_DENSE && s->dense) {
            const float* src = s->dense + ((size_t)k * C + ch) * dense_floats((int)P) + DN_SIGMA * P * P;
            EPG_CHECK(c, cudaMemcpy(o, src, sizeof(float) * P * P, cudaMemcpyDeviceToHost));
        } else {
            std::fill(o, o + P * P, 0.0f);
            for (size_t i = 0; i < P; ++i) o[i * P + i] = minv[(size_t)ch * P + i];
        }
    }
    return 0;
}

int epg_reinit_sites(epg_ctx* c, int n, const int32_t* sites) {
    if (!c->sites || n < 0 || (n > 0 && !sites)) return epg_fail_msg(c, "epg_reinit_sites: bad args / no site data");
    epg_site_data* s = c->sites;
    if ((int)s->h_reinit.size() != c->K) s->h_reinit.assign((size_t)c->K, 0);
    for (int i = 0; i < n; ++i) {
        if (sites[i] < 0 || sites[i] >= c->K) return epg_fail_msg(c, "epg_reinit_sites: bad site index");
        s->h_reinit[sites[i]] = 1;
    }
    return 0;
}

int epg_logdensity(epg_ctx* c, int k, int nq, const double* q, double* lp_out, double* grad_out, int chains,
                   int ticks) {
    if (!c->sites || k < 0 || k >= c->K || nq < 1 || chains > 32 || ticks < 1)
        return epg_fail_msg(c, "epg_logdensity: bad args");
    epg_site_data* s = c->sites;
    const int p = s->h_p[k];
    SamplerArgs a;
    int C = chains;
    if (C <= 0) {
        // default: the most chains (<= 16) at which the sampler keeps the single-box tensor-core pass when that
        // pass may serve the sites; otherwise 32 (the wide tensor-core pass where it applies, else SIMT)
        C = 32;
        if (s->tc_ok && s->use_tc && s->nkc == 1)
            for (int n = tc::NCH; n >= 1; --n) {
                memset(&a, 0, sizeof(a));
                if (fill_args(c, a, n, pad_chains(n), 1, true) == 0 && a.use_tc == 1) { C = n; break; }
            }
    }
    const int CP = pad_chains(C);
    memset(&a, 0, sizeof(a));
    // the plan of epg_tilted_sample for C chains on one site
    if (int rc = fill_args(c, a, C, CP, 1, true)) return rc;
    s->last_C = 0;                                   // chain memory was repurposed
    a.k0 = k;
    const size_t need = sizeof(double) * ((size_t)C * p * 2 + C);
    EPG_CHECK(c, epg_reserve((void**)&s->ld_buf, &s->ld_bytes, need));
    double* dq = s->ld_buf; double* dlp = dq + (size_t)C * p; double* dg = dlp + C;
#define LAUNCH_LD(CPV, TC)                                                                              \
    {                                                                                                   \
        EPG_CHECK(c, set_smem_attr(k_logdensity<CPV, TC>, a.smem_total));                              \
        k_logdensity<CPV, TC><<<1, TC ? tc::NTHREADS : NTHR, a.smem_total, c->stream>>>(a, s->tmap, nb, ticks, dlp, dg); \
    }
    record_plan(s, a, 3, CP);
    for (int q0 = 0; q0 < nq; q0 += C) {
        const int nb = std::min(C, nq - q0);
        EPG_CHECK(c, cudaMemcpyAsync(dq, q + (size_t)q0 * p, sizeof(double) * (size_t)nb * p, cudaMemcpyHostToDevice, c->stream));
        k_set_q<<<(nb * p + 255) / 256, 256, 0, c->stream>>>(s->chain_mem, k * C, s->Pmax, p, nb, dq);
        // the six instances k_nuts is launched as (epg_tilted_sample)
        if (a.use_tc == 2) LAUNCH_LD(32, 2)
        else if (a.use_tc) LAUNCH_LD(32, 1)
        else if (CP == 4) LAUNCH_LD(4, 0) else if (CP == 8) LAUNCH_LD(8, 0)
        else if (CP == 16) LAUNCH_LD(16, 0) else LAUNCH_LD(32, 0)
        c->launches += 2;
        EPG_CHECK(c, cudaGetLastError());
        EPG_CHECK(c, cudaMemcpyAsync(lp_out + q0, dlp, sizeof(double) * nb, cudaMemcpyDeviceToHost, c->stream));
        EPG_CHECK(c, cudaMemcpyAsync(grad_out + (size_t)q0 * p, dg, sizeof(double) * (size_t)nb * p, cudaMemcpyDeviceToHost, c->stream));
        EPG_CHECK(c, cudaStreamSynchronize(c->stream));
    }
#undef LAUNCH_LD
    return 0;
}

int epg_last_plan(epg_ctx* c, int32_t* out, int n) {
    if (!c->sites || !c->sites->plan[0] || !out || n < 1)
        return epg_fail_msg(c, "epg_last_plan: no sampling or log-density launch yet");
    memcpy(out, c->sites->plan, sizeof(int32_t) * std::min(n, EPG_PLAN_FIELDS));
    return 0;
}

}  // extern "C"

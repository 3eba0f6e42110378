/*
 * epgpu.h -- C ABI of libepgpu.so: the B200 (sm_100a) implementation of the
 * data-parallel EP inner loop of gelman/ep-stan.
 *
 * The reference exposes this path as a Python class API (epstan/method.py:19,
 * Master / Worker) on top of NumPy/SciPy-LAPACK/Cython/PyStan calls; it has no
 * FFI of its own.  Every entry point below therefore cites the reference code
 * it replaces (file:line under the reference tree).  A maintainer binds these
 * with ctypes (see INTEGRATION.md); ep-stan_b200/epstan/_lib.py is that binding.
 *
 * Conventions
 *   - plain C types, caller-owned HOST buffers, fp64 unless noted;
 *   - matrices are d x d column-major (they are symmetric, so NumPy 'F' or 'C'
 *     order hold the same bytes); batched site arrays are site-major:
 *     element (i,j) of site k at  i + j*d + k*d*d  == NumPy (d,d,K) order='F',
 *     vectors (d,K) order='F'  ->  [K][d]  (reference method.py:838-851);
 *   - draws of one site are an (n,d) order='F' array (reference util.py:446),
 *     i.e. [d][n]; K sites are concatenated -> [K][d][n];
 *   - site ranges are [k0,k1) in LOCAL site indices of this context (one
 *     context == one GPU == one shard of sites);
 *   - return value: 0 ok; <0 CUDA/usage error (text via epg_last_error);
 *     no exceptions cross the ABI.  Numerical outcomes (not pos.def. etc.) are
 *     reported through flag outputs, never through the return value.
 */
#ifndef EPGPU_H
#define EPGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct epg_ctx epg_ctx;

#define EPG_VERSION 1
#define EPG_XCHG_SLOTS 64      /* caller-defined doubles that ride on the per-iteration all-reduce */

/* ---- device-resident arrays (ids for epg_upload / epg_download / epg_device_ptr) ---- */
enum epg_array {
    EPG_Q = 0,      /* global precision            d*d      method.py:841  */
    EPG_R = 1,      /* global shift                d        method.py:842  */
    EPG_Q0 = 2,     /* prior precision             d*d      method.py:779-788 */
    EPG_R0 = 3,     /* prior shift                 d                       */
    EPG_QI = 4,     /* site precisions             K*d*d    method.py:844  */
    EPG_RI = 5,     /* site shifts                 K*d      method.py:845  */
    EPG_QI2 = 6,    /* proposal site precisions    K*d*d    method.py:847  */
    EPG_RI2 = 7,    /* proposal site shifts        K*d      method.py:848  */
    EPG_DQI = 8,    /* site precision deltas       K*d*d    method.py:850  */
    EPG_DRI = 9,    /* site shift deltas           K*d      method.py:851  */
    EPG_CAVQ = 10,  /* cavity precisions (Worker.Mat after cavity)  K*d*d  method.py:288 */
    EPG_CAVM = 11,  /* cavity means      (Worker.vec after cavity)  K*d    method.py:295 */
    EPG_S = 12,     /* global covariance           d*d      method.py:838  */
    EPG_M = 13,     /* global mean                 d        method.py:839  */
    EPG_PARTIAL = 14, /* [sum_k Qi2 | sum_k ri2 | n_ok] of this shard, d*d+d+1: the
                         NCCL all-reduce payload (method.py:1073-1074)     */
    EPG_TMEAN = 15, /* tilted means of the last moment matching  K*d (Worker.vec after tilted) */
    EPG_DSUM = 16,  /* [sum_k dQi | sum_k dri | sum_k |delta_k|^2 | n_ok | EPG_XCHG_SLOTS caller slots] of this
                       shard, d*d+d+2+EPG_XCHG_SLOTS doubles (epg_delta_sums[_ex]): THE buffer the ranks
                       all-reduce (sum) once per EP iteration (method.py:1073-1074, SURVEY 8e)  */
    EPG_NARRAYS = 17
};

/* ---- tilted log-density families (experiment/models/<name>[_sg].stan) ---- */
enum epg_model {
    EPG_M1B = 1,    /* m1b.stan:21-42, m1b_sg.stan:19-35: phi=[log sigma_a, beta]           */
    EPG_M2B = 2,    /* m2b.stan:21-46, m2b_sg.stan:19-38: phi=[log sigma_a, log sigma_b], one slope vector etb(D) per site */
    EPG_M3B = 3,    /* m3b.stan:21-49, m3b_sg.stan:19-39: phi=[log sigma_a, log sigma_b]    */
    EPG_M4B = 4,    /* m4b.stan:21-53, m4b_sg.stan:19-43: phi=[mu_a,log sigma_a,mu_b,log sigma_b] */
    EPG_M5B = 5     /* m5b.stan:21-53, m5b_sg.stan:19-45: m4b with double_exponential(0,1) latents */
};

enum epg_prec_estim { EPG_PREC_SAMPLE = 0, EPG_PREC_OLSE = 1 };  /* method.py:163 */

/* ---- lifetime ---- */
int epg_version(void);
/* device: CUDA ordinal.  own_stream != 0: the context creates a private
 * non-blocking stream (`stream` is ignored).  own_stream == 0: every kernel and
 * copy is issued on the caller's cudaStream_t `stream` (NULL = the legacy
 * default stream) -- required when the caller interleaves its own work, e.g.
 * NCCL collectives issued by torch.distributed on torch's current stream. */
int epg_create(epg_ctx** out, int device, void* stream, int own_stream);
void epg_destroy(epg_ctx* ctx);
const char* epg_last_error(const epg_ctx* ctx);
int epg_sync(epg_ctx* ctx);
/* number of kernels this context has launched so far (bench.py "gpu_launches") */
int64_t epg_launch_count(const epg_ctx* ctx);

/* ---- state (Master.__init__, method.py:836-851) ---- */
int epg_init_state(epg_ctx* ctx, int K, int d);
int epg_upload(epg_ctx* ctx, int array, int k0, int k1, const double* host);
int epg_download(epg_ctx* ctx, int array, int k0, int k1, double* host);
void* epg_device_ptr(epg_ctx* ctx, int array);
/* number of doubles epg_upload / epg_download move for this array and site range (k0,k1 ignored for global arrays) */
int64_t epg_array_count(epg_ctx* ctx, int array, int k0, int k1);

/* ---- cavity: Worker.cavity, method.py:267-302 (batched over sites) ----
 * proposal==0 uses (Qi,ri), 1 uses (Qi2,ri2).  Writes EPG_CAVQ / EPG_CAVM for
 * sites whose cavity is pos.def.; posdef_out[k1-k0] (may be NULL); *all_ok.
 *
 * Site flags: the context keeps ONE per-site flag vector, written by the last
 * per-site call that covered the site -- epg_moments (moment estimate ok),
 * epg_fail_sites (cleared), epg_cavity (cavity pos.def.) and epg_force_pd
 * (site forced).  epg_delta_sums(_ex) counts it as n_ok and skips the Fisher
 * norms of flagged-off sites, so call it right after epg_moments/epg_fail_sites. */
int epg_cavity(epg_ctx* ctx, int k0, int k1, int proposal, int32_t* posdef_out, int* all_ok);

/* ---- moment matching: Worker.tilted second half, method.py:408-468 ----
 * epg_set_draws copies host draws [k1-k0][d][n] to the device draw buffer;
 * epg_moments turns the device-resident draws of sites [k0,k1) into
 * (dQi, dri) = tilted natural parameters - (Q, r)   (method.py:413-458),
 * zero-filling failed sites (method.py:460-465).  ok_out[k1-k0] may be NULL. */
int epg_set_draws(epg_ctx* ctx, int k0, int k1, int n, const double* draws);
int epg_get_draws(epg_ctx* ctx, int k0, int k1, int n, double* draws);
int epg_moments(epg_ctx* ctx, int k0, int k1, int n, int prec_estim, int32_t* ok_out, int* n_ok);

/* Mark local sites as failed for this EP iteration: zero-fills their (dQi, dri) and clears their
 * flags exactly as a failed moment estimate does (method.py:460-465).  Used by the host when a
 * site's chains did not mix (Master option `rhat_max`, an extension). */
int epg_fail_sites(epg_ctx* ctx, int n, const int32_t* sites);

/* ---- damped update + aggregation: method.py:1071-1081 ----
 * epg_update_partial: Qi2 = Qi + df*dQi, ri2 = ri + df*dri for the local sites
 *   and EPG_PARTIAL = [sum Qi2 | sum ri2 | (unchanged)]            (a11)
 * (multi-GPU: the caller all-reduces EPG_PARTIAL over the ranks here)
 * epg_update_finish: Q = Q0 + partial, r = r0 + partial; Cholesky of Q kept
 *   for epg_global_moments; *posdef = 0 if Q is not pos.def.       (a12) */
int epg_update_partial(epg_ctx* ctx, double df);
int epg_update_finish(epg_ctx* ctx, int* posdef);
/* accept the proposal: swap (Qi,Qi2), (ri,ri2)  -- method.py:1148-1157 */
int epg_accept(epg_ctx* ctx);
/* (S, m) from the kept Cholesky factor -- method.py:1211-1219; outputs may be NULL */
int epg_global_moments(epg_ctx* ctx, double* m_out, double* S_out);
/* force improper sites proper -- method.py:1119-1132 / 1194-1207:
 * lam = lambda_min(Qi2_k); if lam < thr: diag(Qi_k) += min_eig - lam.
 * forced_out[K], lam_out[K] may be NULL. */
int epg_force_pd(epg_ctx* ctx, double thr, double min_eig, int32_t* forced_out, double* lam_out);

/* ---- automatic damping selection (SURVEY 8f rank 1; find_damp.py:144-183, fit.py:176-186) ----
 * Signal-to-noise statistics of the site updates in the Fisher metric of the
 * current global approximation N(m, S = Q^-1):
 *     |(A, a)|^2 = 1/4 tr(S A S A) + 1/2 (a - A m)' S (a - A m)
 * epg_delta_sums (call right after epg_moments): EPG_DSUM = [sum_k dQi | sum_k dri |
 *   sum_k |delta_k|^2 | n_ok] over the local sites.  The caller all-reduces EPG_DSUM.
 * epg_delta_snr: stats_out[3] = { |sum_k delta_k|^2, sum_k |delta_k|^2, n_ok } of the
 *   (reduced) EPG_DSUM.  At an EP fixed point the first is the K-site sum of
 *   independent zero-mean noise, i.e. about equal to the second. */
int epg_delta_sums(epg_ctx* ctx);
int epg_delta_snr(epg_ctx* ctx, double* stats_out);

/* ---- one exchange per EP iteration (SURVEY 8e; method.py:1073-1074 sums the sites on one host) ----
 * epg_delta_sums_ex: epg_delta_sums with the Fisher norms optional (with_norms == 0: the sum_k |delta_k|^2
 *   entry is 0) and `n_slots` <= EPG_XCHG_SLOTS caller-defined doubles appended (the rest zero) -- the host
 *   puts its per-rank scalars there (failed-site counts, analytics maxima in per-rank slots), so that ONE
 *   all-reduce(sum) of EPG_DSUM carries everything an iteration exchanges.  Also snapshots the current
 *   global (Q, r).
 * epg_update_from_sums: with EPG_DSUM all-reduced, sets EPG_PARTIAL so that the following
 *   epg_update_finish yields the proposal Q = Q_prev + df * sum_k dQi, r = r_prev + df * sum_k dri --
 *   identical on every rank, so damping retries need no further exchange of matrices
 *   (epg_update_partial(df) still forms the local Qi2 = Qi + df dQi for the proposal cavities).
 * epg_delta_snr and epg_update_from_sums fail (return < 0) unless epg_delta_sums(_ex) has run since the
 *   last epg_init_state: the snapshot and the sums belong to one state. */
int epg_delta_sums_ex(epg_ctx* ctx, int with_norms, const double* slots, int n_slots);

/* ---- Master.mix_phi, method.py:1250-1301: pool the last tilted draws of phi over the sites ----
 * sums_out [d + 2 d*d] = sum over the local sites of [ mean_k | sum_t (x_t - mean_k)(x_t - mean_k)' | mean_k mean_k' ]
 * of the n draws per site in the device draw buffer; the host combines (and sums over ranks):
 *   m = sum mean_k / K,   S = (sum scatter_k + n (sum mean_k mean_k' - K m m')) / (K n - 1). */
int epg_mix_phi_sums(epg_ctx* ctx, int n, double* sums_out);
int epg_update_from_sums(epg_ctx* ctx, double df);

/* ---- damping sweep: experiment/find_damp.py:144-174 + kl_mvn :32-51 ----
 * For each dfs[i]: rebuild the global approximation from (Qi,ri,dQi,dri),
 * require it and all K cavities pos.def., and score it against the target
 * N(m_tgt,S_tgt): mse_out[i] = mean((m-m_tgt)^2), kl_out[i] = KL(target||approx);
 * NaN where a factorisation failed.  (single-context sweep) */
int epg_damp_sweep(epg_ctx* ctx, int n_df, const double* dfs, const double* m_tgt,
                   const double* S_tgt, double* mse_out, double* kl_out);

/* ---- stand-alone batched utilities (no EP state needed) ----
 * epg_invert_normal_params: util.py:51-125 (+ copy_triu_to_tril pyx:86-106).
 *   A [batch][d*d], b [batch][d] or NULL; cho_form: A holds the upper factor.
 *   ok[batch]=0 where not pos.def. (outputs of that item are then undefined). */
int epg_invert_normal_params(epg_ctx* ctx, int batch, int d, const double* A, const double* b,
                             int cho_form, double* out_A, double* out_b, int32_t* ok);
/* epg_olse: util.py:128-194 (+ fro_norm_squared pyx:17-40). P may be NULL (naive prior). */
int epg_olse(epg_ctx* ctx, int batch, int d, const double* S, int n, const double* P,
             double* out, int32_t* ok);
/* epg_cv_moments: util.py:245-411 (+ auto_outer/ravel_triu/unravel_triu pyx:45-183).
 *   draws [batch][d][n], lp [batch][n], Q_tilde [batch][d*d], r_tilde [batch][d];
 *   regulate_a / max_a <= 0 mean "None"; m_treshold <= 0 means no treshold.
 *   used_cv[batch]: 1 control-variate estimate, 0 plain fallback (util.py:353-367),
 *   -1 factorisation/solve failed. */
int epg_cv_moments(epg_ctx* ctx, int batch, int n, int d, const double* draws, const double* lp,
                   const double* Q_tilde, const double* r_tilde, int multiple_cv,
                   double regulate_a, double max_a, double m_treshold,
                   double* S_hat, double* m_hat, int32_t* used_cv);
/* the same, additionally returning the control-variate coefficients (cv_moments(..., ret_a=True), util.py:396-410):
 *   a_m_out [batch][d*d] and a_S_out [batch][d2*d2] (row-major, first index = control feature) with multiple_cv,
 *   [batch][d] and [batch][d2] without; zeros for items that took the plain fallback; either may be NULL. */
int epg_cv_moments_ex(epg_ctx* ctx, int batch, int n, int d, const double* draws, const double* lp,
                      const double* Q_tilde, const double* r_tilde, int multiple_cv,
                      double regulate_a, double max_a, double m_treshold,
                      double* S_hat, double* m_hat, int32_t* used_cv, double* a_S_out, double* a_m_out);

/* ---- site data + tilted sampling: Worker.tilted first half, method.py:338-408,
 *      _sample_stan :43-118, stan_sample_time util.py:692-724 (PyStan NUTS) ----
 * epg_upload_sites: X [N][D] row-major fp64 (method.py:733), y [N] in {0,1},
 *   k_lim[K+1] row offsets of the local sites (method.py:700),
 *   j_ind [N] 0-based group index within its site and Jk[K] groups per site
 *   (fit.py:318-319; both NULL for the single-group *_sg models). */
int epg_upload_sites(epg_ctx* ctx, int model, int D, const int64_t* k_lim, const double* X,
                     const int64_t* y, const int32_t* j_ind, const int32_t* Jk);

typedef struct epg_sampler_opts {
    int32_t chains;        /* method.py:155 */
    int32_t iter;          /* method.py:156 */
    int32_t warmup;        /* <0: iter/2  (method.py:567-569) */
    int32_t thin;          /* >= 1: post-warm-up transition m (0-based) is saved when m % thin == 0, i.e.
                              ceil((iter - warmup) / thin) draws per chain (Stan's generate_transitions); the
                              chain itself, its transitions and random numbers, do not depend on it (fit.py:304) */
    int32_t init_mode;     /* 0: 'random' U(-init_radius, init_radius); 1: zeros; 2: previous last draws (init_prev,
                              method.py:404-406); 3: given by epg_set_inits (PyStan init=dict / list / function) */
    int32_t max_treedepth; /* Stan default 10 */
    double adapt_delta;    /* Stan default 0.8 */
    int32_t metric;        /* EPG_METRIC_*; 0 (diag_e) is Stan's default.  Other values: the call fails (< 0) */
    int32_t reserved[7];
} epg_sampler_opts;

/* Euclidean metrics of the sampler (PyStan `control={'metric': ...}`), with Sigma the p x p inverse metric:
 *   EPG_METRIC_DIAG  diag_e: Sigma diagonal, adapted from the variances of the draws of each warm-up window
 *                    (stan/mcmc/hmc/hamiltonians/diag_e_metric.hpp, stan/mcmc/var_adaptation.hpp);
 *   EPG_METRIC_DENSE dense_e: Sigma = U'U full, momentum p = U^-1 z (z ~ N(0, I)), kinetic energy p'Sigma p / 2,
 *                    position update q += eps Sigma p; each window end sets Sigma = n/(n+5) C + 1e-3 5/(n+5) I from
 *                    the window's sample covariance C (stan/mcmc/hmc/hamiltonians/dense_e_metric.hpp,
 *                    stan/mcmc/covar_adaptation.hpp).  A window whose Sigma has no Cholesky factor (fp64) leaves
 *                    the chain's previous Sigma in place;
 *   EPG_METRIC_UNIT  unit_e: Sigma = I, step-size adaptation only (stan/mcmc/hmc/nuts/adapt_unit_e_nuts.hpp).
 * carry_adapt carries Sigma and the step size over only between runs of a chain with the same metric; otherwise
 * the warm-up starts from Sigma = I and step size 1. */
enum epg_metric { EPG_METRIC_DIAG = 0, EPG_METRIC_DENSE = 1, EPG_METRIC_UNIT = 2 };

/* Stan 2.17's remaining NUTS settings (PyStan `control`, `init_r`); epg_tilted_sample_ex with adapt == NULL, and
 * epg_tilted_sample, use the defaults in brackets.  Fill in every field: an out-of-range value fails the call (< 0).
 *   stepsize         starting nominal step size [1]; the step-size heuristic and dual averaging start from it
 *                    (mu = log(10 stepsize)).  A chain that carries its adaptation (init_mode 2, carry_adapt) starts
 *                    from its carried step size instead.  > 0, finite
 *   stepsize_jitter  j in [0, 1] [0]: every transition (warm-up and sampling) uses eps = eps_nom (1 + j (2u - 1)),
 *                    u ~ U(0, 1) (base_hmc::sample_stepsize); adaptation works on eps_nom, the mean step size
 *                    (msteps_out) averages the eps of the saved transitions, like Stan's stepsize__, and the step
 *                    size carried over is eps_nom
 *   gamma, kappa, t0 dual-averaging constants of stepsize_adaptation [0.05, 0.75, 10], each > 0
 *   init_radius      r > 0 [2]: random inits (init_mode 0, and the NaN entries of init_mode 3) are U(-r, r)
 *   engaged          1 [1]: adaptive NUTS (run_adaptive_sampler); 0: run_sampler -- no step-size heuristic, no
 *                    dual averaging, no metric windows: eps_nom = stepsize and the inverse metric is the identity
 *                    throughout, for every metric, init mode and carried state; warm-up transitions still run and
 *                    are discarded
 *   init_buffer, term_buffer, window   windowed_adaptation [75, 50, 25]: buffers >= 0, window >= 1.  No windows
 *                    below 20 warm-up iterations; when init_buffer + window + term_buffer exceeds the warm-up they
 *                    become 15 % / 10 % / the rest of it (set_window_params); window ends by compute_next_window
 * (C99) */
typedef struct epg_sampler_adapt {
    double stepsize;
    double stepsize_jitter;
    double gamma;
    double kappa;
    double t0;
    double init_radius;
    int32_t engaged;
    int32_t init_buffer;
    int32_t term_buffer;
    int32_t window;
    int32_t reserved[8];
} epg_sampler_adapt;

/* Runs adaptive NUTS for sites [k0,k1) x chains on their tilted densities
 * (cavity from EPG_CAVQ/EPG_CAVM x site likelihood), leaves the post-warm-up
 * draws of phi in the device draw buffer ([d][n] per site, chain-major rows,
 * util.py:475-484) and the per-chain last states for init_prev.
 * seeds[k1-k0]: the per-site Stan seeds (method.py:342-346).
 * Analytics (all may be NULL): msteps_out[k] mean step size (method.py:99-102),
 * mrhat_out[k] max split-Rhat (method.py:104), n_leapfrog_out[k] gradient
 * evaluations spent, *seconds = device time of the sampling kernel. */
int epg_tilted_sample(epg_ctx* ctx, int k0, int k1, const uint32_t* seeds,
                      const epg_sampler_opts* opts, double* msteps_out, double* mrhat_out,
                      int64_t* n_leapfrog_out, double* seconds);
/* the same with the settings of `adapt` (NULL: Stan's defaults, as epg_tilted_sample) */
int epg_tilted_sample_ex(epg_ctx* ctx, int k0, int k1, const uint32_t* seeds,
                         const epg_sampler_opts* opts, const epg_sampler_adapt* adapt, double* msteps_out,
                         double* mrhat_out, int64_t* n_leapfrog_out, double* seconds);

/* Starting points of init_mode 3 (PyStan init = dict, list of dicts or function): q [k1-k0][chains][Pmax]
 * (Pmax = epg_max_params) in the layout q = [phi (d) | eta (J) | etb] of epg_get_param_stats.  A NaN entry is
 * drawn U(-init_radius, init_radius) as init_mode 0 draws it; entries beyond a site's epg_num_params are
 * ignored.  A chain whose start has a random entry redraws up to 100 times when its density is not finite; one
 * given in full fails its site at once, as Stan fails such a user init.  The values stay until the next
 * epg_set_inits or epg_upload_sites; a call with another chain count drops those of every site.  An init_mode 3
 * run fails unless every one of its sites was set for its chain count. */
int epg_set_inits(epg_ctx* ctx, int k0, int k1, int chains, const double* q);

/* Marks local sites whose chains the next epg_tilted_sample with init_mode 2 starts afresh -- phi within one
 * conditional cavity standard deviation of the cavity mean, the site-local latents in U(-1,1) -- instead of
 * from their previous last draws (an extension: with init_prev, method.py:404-406, a chain that got stuck,
 * e.g. far out with a collapsed step size, would otherwise stay stuck for the rest of the EP run; Stan's
 * U(-2,2) is no remedy late in a run, when the cavity is thousands of times narrower than that).
 * The marks are consumed by that call. */
int epg_reinit_sites(epg_ctx* ctx, int n, const int32_t* sites);

/* ---- Master.mix_pred, method.py:1304-1478: moments of the site parameters over the last draws ----
 * With option "param_stats" = 1 the sampler accumulates, for every sampled slot i of a site's parameter vector
 * q = [phi (d) | eta (J) | etb], the TRANSFORMED parameter of the Stan programs (m1b.stan:30-36 ...):
 * phi_i | alpha_j = [mu_a +] eta_j sigma_a | beta_ji = [mu_b,i +] etb_ji sigma_b,i.
 * epg_get_param_stats returns per site the mean and the sum of squared deviations over all retained draws of all
 * chains, [k1-k0][Pmax] each (Pmax = epg_max_params; slots beyond a site's epg_num_params are undefined). */
int epg_get_param_stats(epg_ctx* ctx, int k0, int k1, double* mean_out, double* ssd_out);
int epg_max_params(epg_ctx* ctx);

/* ---- HMC diagnostics of the sampler (PyStan 2.17 get_sampler_params and check_hmc_diagnostics) ----
 * Per-site summary, always kept: out [k1-k0][chains][EPG_DIAG_FIELDS] for each site's most recent run, over
 * the SAVED post-warm-up transitions of each chain (those whose draws are written; thin applies), fields
 *   n_saved          saved transitions (0 for a chain that found no finite starting point)
 *   n_divergent      saved transitions with divergent__ = 1 (PyStan check_div)
 *   n_max_treedepth  saved transitions with treedepth__ >= max_treedepth (PyStan check_treedepth)
 *   ebfmi            sum_t (E_t - E_t-1)^2 / sum_t (E_t - mean E)^2 over the saved energy__ values (PyStan
 *                    check_energy); NaN with fewer than 2 saved transitions or zero variance
 * Returns the chain count (> 0; out may be NULL to ask for it only); fails (< 0) unless every site of the range
 * has run at the chain count of the most recent run (a run with another chain count drops every site's). */
#define EPG_DIAG_FIELDS 4
int epg_get_hmc_diag(epg_ctx* ctx, int k0, int k1, double* out);
/* Per-transition records (option "sampler_params" = 1 when the run was launched): out [k1-k0][chains][n][6],
 * per transition PyStan's get_sampler_params() columns in its order, with Stan 2.17's definitions
 * (base_nuts::transition):
 *   accept_stat__  sum of min(1, exp(H0 - H)) over the transition's leapfrog steps / n_leapfrog__ (what dual
 *                  averaging sees, before it is clamped)
 *   stepsize__     the transition's step size (jitter applied)
 *   treedepth__    subtrees merged into the trajectory (one that diverges or U-turns internally does not count)
 *   n_leapfrog__   leapfrog steps, including those of a discarded subtree
 *   divergent__    1 when the transition ended on H - H0 > 1000
 *   energy__       H(q, p) of the selected sample, its momentum included
 * Records are the transitions Stan saves with save_warmup: warm-up transition m with m % thin == 0
 * (ceil(warmup / thin) of them, dropped when inc_warmup = 0), then the ceil((iter - warmup) / thin) saved ones;
 * step-size-heuristic leapfrogs are not transitions.  Returns n (out may be NULL to ask for it only); fails
 * (< 0) for a site whose most recent run did not record.  A recording run of another chains, iter, warmup or
 * thin drops the records of every other site; a run with another chain count drops every site's. */
int epg_get_sampler_params(epg_ctx* ctx, int k0, int k1, int inc_warmup, double* out);

/* Diagnostics: the diagonal inverse metric [chains][Pmax] (fp32, Pmax = the largest epg_num_params of the
 * context) and the step size [chains] site k's chains ended their last run with (what carry_adapt carries over). */
int epg_get_adapt(epg_ctx* ctx, int k, float* minv_out, float* eps_out);
/* The inverse metric Sigma site k's chains ended their last run with, as full matrices [chains][Pmax][Pmax]
 * (fp32, row-major, Pmax = epg_max_params; entries beyond the site's epg_num_params are undefined): diag_e gives
 * a diagonal matrix, unit_e the identity, dense_e the adapted Sigma (whose diagonal epg_get_adapt returns).
 * Fails before the first sampling run. */
int epg_get_metric(epg_ctx* ctx, int k, float* out);

/* Options.  "carry_adapt" (default 1): a run with init_mode 2 (init_prev) starts its warm-up from the metric
 * and step size the previous run of the same chain ended with, instead of Stan's unit metric and step size 1
 * (an extension in the spirit of init_prev, method.py:404-406; the warm-up itself -- dual averaging, variance
 * windows -- still runs in full); 0 = Stan's defaults.  "use_tc" (default 1): use the tcgen05/TMA likelihood pass when the
 * shapes allow it (single-group sites; D+1 <= 64 and chains <= 16: design matrix from L2, chain state in shared memory;
 * otherwise D+1 <= 256 and chains <= 32: the wide pass, design matrix streamed from HBM -- config 5); 0 forces the
 * fp32 SIMT pass.  "pingpong" (default 0): 1 = with the tensor-core pass, more
 * sites than SMs and design matrices that stay L2-resident, run the persistent
 * two-sites-per-CTA kernel (likelihood pass of one site overlapped with the chain
 * phase of the other); 2 = always; 0 = never (measured gain on B200 is <= 15 %).
 * Draws do not depend on these two kernels' choice.  "metric_reg" (default 1e-3, Stan's value): the weight of
 * the identity in the regularised dense_e window estimate (n/(n+5) C + metric_reg 5/(n+5) I); a value <= 0
 * lets a window that is (numerically) singular fail its factorisation.  "sampler_params" (default 0): 1 = record
 * every transition of the following runs for epg_get_sampler_params (6 doubles per record, kept for every
 * site and chain: about 39 MB at config 4's shape); the draws do not depend on it.  Call after epg_upload_sites. */
int epg_set_option(epg_ctx* ctx, const char* name, double value);

/* Direct evaluation of the tilted log-density and its gradient for site k at
 * `nq` points q [nq][p] (p = epg_num_params); used by the parity tests against
 * the fp64 oracle.  lp_out[nq], grad_out[nq][p].
 * The points are evaluated in batches of `chains` (1..32) under the launch plan epg_tilted_sample makes for
 * that many chains: the same likelihood pass (SIMT, tensor-core or wide tensor-core, including the fall-back
 * to SIMT when the chain vectors do not fit in shared memory), the same shared-memory layout, ring depth and
 * chain-vector addressing.  chains <= 0: when the single-box tensor-core pass may serve the sites, the most
 * chains (<= 16) at which the sampler keeps it; otherwise 32.
 * `ticks` (>= 1): how many times the likelihood pass runs before the read-out (the sampler runs it once per
 * gradient evaluation and carries the pipeline state of the tensor-core passes from one to the next). */
int epg_num_params(epg_ctx* ctx, int k);
int epg_logdensity(epg_ctx* ctx, int k, int nq, const double* q, double* lp_out, double* grad_out,
                   int chains, int ticks);

/* Launch plan of the most recent epg_tilted_sample or epg_logdensity, as EPG_PLAN_FIELDS int32 in this order:
 *   kernel      1 = per-site sampling kernel, 2 = two-sites-per-CTA sampling kernel, 3 = log-density kernel
 *   use_tc      0 = fp32 SIMT pass, 1 = tensor-core pass (D+1 <= 64, <= 16 chains), 2 = wide tensor-core pass
 *   chain_pad   SIMT: chains padded to 4, 8, 16 or 32; tensor-core pass: chain columns processed (4, 8 or 16);
 *               wide pass: 32
 *   tc_nst      X-tile stages of the tensor-core ring (0 on the SIMT pass)
 *   resident    SIMT: the design matrix stays in shared memory (1) or is streamed in tiles (0)
 *   R, slices, NC   SIMT: rows per tile, row slices of the gradient product, chain-column blocks per thread
 *   hot_nvec, hot_levels   per-chain vectors and tree-stack levels kept in shared memory
 *   omega_smem  the cavity precision lives in shared memory
 *   smem_total  dynamic shared memory of the launch (bytes)
 * Writes min(n, EPG_PLAN_FIELDS) values; fails before the first such call. */
#define EPG_PLAN_FIELDS 12
int epg_last_plan(epg_ctx* ctx, int32_t* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* EPGPU_H */

// Internal context of libepgpu (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include "../../include/epgpu.h"

struct epg_site_data;      // sampler-side site data (epg_sampler.cu)

struct epg_ctx {
    int device = 0;
    int num_sms = 148;
    size_t l2_bytes = 126u << 20;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    int64_t launches = 0;

    // EP state
    int K = 0, d = 0;
    double* arr[EPG_NARRAYS] = {nullptr};
    double* chol = nullptr;        // packed lower Cholesky factor of the global Q (d(d+1)/2)
    int* site_ok = nullptr;        // [K] per-site flags of the last batched kernel
    int* flags = nullptr;          // [8] scalar device flags
    double* scratch = nullptr;     // update partials etc.
    size_t scratch_bytes = 0;
    int32_t* h_flags = nullptr;    // pinned host mirror for small read-backs
    size_t h_flags_n = 0;

    // draws [K][d][n_cap]
    double* draws = nullptr;
    size_t draws_cap = 0;          // doubles
    int draws_n = 0;

    // staging for the stand-alone utilities
    double* util_buf = nullptr;
    size_t util_bytes = 0;

    // per-site packed Gram + shift between the two moment-matching kernels (epg_moments.cu)
    double* mom_buf = nullptr;
    size_t mom_bytes = 0;

    // global (Q, r) at the time of the last epg_delta_sums: base of epg_update_from_sums
    double* q_prev = nullptr;
    size_t q_prev_bytes = 0;
    // q_prev, snr_buf and EPG_DSUM were filled by epg_delta_sums(_ex) for the current state (K, d);
    // cleared by epg_init_state, required by epg_update_from_sums and epg_delta_snr
    bool sums_valid = false;

    // scratch of the damping-selection statistics (epg_snr.cu)
    double* snr_buf = nullptr;
    size_t snr_bytes = 0;

    epg_site_data* sites = nullptr;
};

size_t epg_array_elems(const epg_ctx* c, int array);       // total element count
size_t epg_array_site_stride(const epg_ctx* c, int array); // 0 for global arrays
int epg_fail(epg_ctx* c, const char* what, cudaError_t e);
int epg_fail_msg(epg_ctx* c, const std::string& msg);
cudaError_t epg_reserve(void** p, size_t* cap, size_t need);

// kernel launchers (each returns the launch status; all asynchronous on c->stream)
int epg_moments_threads(int d);
cudaError_t epg_launch_moments(epg_ctx* c, int k0, int k1, int n, int mode);
cudaError_t epg_launch_cavity(epg_ctx* c, int k0, int k1, int proposal);
cudaError_t epg_launch_update_partial(epg_ctx* c, double df);
cudaError_t epg_launch_update_finish(epg_ctx* c);
cudaError_t epg_launch_global_moments(epg_ctx* c);
cudaError_t epg_launch_force_pd(epg_ctx* c, double thr, double min_eig, double* lam_dev);
cudaError_t epg_launch_damp_sweep(epg_ctx* c, int n_df, const double* dfs_dev, const double* tgt_dev,
                                  double* out_dev);
cudaError_t epg_launch_invert(epg_ctx* c, int batch, int d, const double* A, const double* b,
                              int cho_form, double* outA, double* outb, int* ok);
cudaError_t epg_launch_olse(epg_ctx* c, int batch, int d, const double* S, int n, const double* P,
                            double* out, int* ok);

#define EPG_CHECK(c, call)                                      \
    do {                                                        \
        cudaError_t _e = (call);                                \
        if (_e != cudaSuccess) return epg_fail((c), #call, _e); \
    } while (0)

"""ctypes binding of libepgpu.so (include/epgpu.h).

There is deliberately no CPU fallback: if the shared library is missing or no
CUDA device is usable, constructing a :class:`Context` raises.
"""

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), 'libepgpu.so')

# enum epg_array
(Q, R, Q0, R0, QI, RI, QI2, RI2, DQI, DRI, CAVQ, CAVM, S, M, PARTIAL, TMEAN, DSUM) = range(17)
XCHG_SLOTS = 64           # EPG_XCHG_SLOTS: caller-defined doubles at the end of DSUM
MODEL_IDS = {'m1b': 1, 'm2b': 2, 'm3b': 3, 'm4b': 4, 'm5b': 5}
PREC_ESTIM = {'sample': 0, 'olse': 1}
METRICS = {'diag_e': 0, 'dense_e': 1, 'unit_e': 2}     # enum epg_metric (Stan's `metric` names)

_c_double_p = C.POINTER(C.c_double)
_c_int32_p = C.POINTER(C.c_int32)
_c_int64_p = C.POINTER(C.c_int64)
_c_uint32_p = C.POINTER(C.c_uint32)


class SamplerOpts(C.Structure):
    _fields_ = [('chains', C.c_int32), ('iter', C.c_int32), ('warmup', C.c_int32),
                ('thin', C.c_int32), ('init_mode', C.c_int32), ('max_treedepth', C.c_int32),
                ('adapt_delta', C.c_double), ('metric', C.c_int32), ('reserved', C.c_int32 * 7)]


class SamplerAdapt(C.Structure):
    """epg_sampler_adapt: Stan's step-size, adaptation and init-radius settings"""
    _fields_ = [('stepsize', C.c_double), ('stepsize_jitter', C.c_double), ('gamma', C.c_double),
                ('kappa', C.c_double), ('t0', C.c_double), ('init_radius', C.c_double), ('engaged', C.c_int32),
                ('init_buffer', C.c_int32), ('term_buffer', C.c_int32), ('window', C.c_int32),
                ('reserved', C.c_int32 * 8)]


INIT_GIVEN = 3            # init_mode of starting points set by Context.set_inits


class EpgError(RuntimeError):
    pass


_lib = None

# every symbol include/epgpu.h declares: (name, restype, argtypes)
SYMBOLS = [
    ('epg_version', C.c_int, []),
    ('epg_create', C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_int]),
    ('epg_destroy', None, [C.c_void_p]),
    ('epg_last_error', C.c_char_p, [C.c_void_p]),
    ('epg_sync', C.c_int, [C.c_void_p]),
    ('epg_launch_count', C.c_int64, [C.c_void_p]),
    ('epg_init_state', C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    ('epg_upload', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _c_double_p]),
    ('epg_download', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _c_double_p]),
    ('epg_array_count', C.c_int64, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    ('epg_device_ptr', C.c_void_p, [C.c_void_p, C.c_int]),
    ('epg_cavity', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _c_int32_p, C.POINTER(C.c_int)]),
    ('epg_set_draws', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _c_double_p]),
    ('epg_get_draws', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _c_double_p]),
    ('epg_moments', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, _c_int32_p, C.POINTER(C.c_int)]),
    ('epg_fail_sites', C.c_int, [C.c_void_p, C.c_int, _c_int32_p]),
    ('epg_reinit_sites', C.c_int, [C.c_void_p, C.c_int, _c_int32_p]),
    ('epg_get_param_stats', C.c_int, [C.c_void_p, C.c_int, C.c_int, _c_double_p, _c_double_p]),
    ('epg_max_params', C.c_int, [C.c_void_p]),
    ('epg_get_adapt', C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    ('epg_get_metric', C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_float)]),
    ('epg_update_partial', C.c_int, [C.c_void_p, C.c_double]),
    ('epg_update_finish', C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    ('epg_accept', C.c_int, [C.c_void_p]),
    ('epg_global_moments', C.c_int, [C.c_void_p, _c_double_p, _c_double_p]),
    ('epg_force_pd', C.c_int, [C.c_void_p, C.c_double, C.c_double, _c_int32_p, _c_double_p]),
    ('epg_delta_sums', C.c_int, [C.c_void_p]),
    ('epg_delta_snr', C.c_int, [C.c_void_p, _c_double_p]),
    ('epg_delta_sums_ex', C.c_int, [C.c_void_p, C.c_int, _c_double_p, C.c_int]),
    ('epg_update_from_sums', C.c_int, [C.c_void_p, C.c_double]),
    ('epg_mix_phi_sums', C.c_int, [C.c_void_p, C.c_int, _c_double_p]),
    ('epg_damp_sweep', C.c_int, [C.c_void_p, C.c_int, _c_double_p, _c_double_p, _c_double_p,
                                 _c_double_p, _c_double_p]),
    ('epg_invert_normal_params', C.c_int, [C.c_void_p, C.c_int, C.c_int, _c_double_p, _c_double_p, C.c_int,
                                           _c_double_p, _c_double_p, _c_int32_p]),
    ('epg_olse', C.c_int, [C.c_void_p, C.c_int, C.c_int, _c_double_p, C.c_int, _c_double_p, _c_double_p,
                           _c_int32_p]),
    ('epg_cv_moments', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _c_double_p, _c_double_p, _c_double_p,
                                 _c_double_p, C.c_int, C.c_double, C.c_double, C.c_double, _c_double_p,
                                 _c_double_p, _c_int32_p]),
    ('epg_cv_moments_ex', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _c_double_p, _c_double_p, _c_double_p,
                                 _c_double_p, C.c_int, C.c_double, C.c_double, C.c_double, _c_double_p,
                                 _c_double_p, _c_int32_p, _c_double_p, _c_double_p]),
    ('epg_upload_sites', C.c_int, [C.c_void_p, C.c_int, C.c_int, _c_int64_p, _c_double_p, _c_int64_p,
                                   _c_int32_p, _c_int32_p]),
    ('epg_tilted_sample', C.c_int, [C.c_void_p, C.c_int, C.c_int, _c_uint32_p, C.POINTER(SamplerOpts),
                                    _c_double_p, _c_double_p, _c_int64_p, _c_double_p]),
    ('epg_tilted_sample_ex', C.c_int, [C.c_void_p, C.c_int, C.c_int, _c_uint32_p, C.POINTER(SamplerOpts),
                                       C.POINTER(SamplerAdapt), _c_double_p, _c_double_p, _c_int64_p,
                                       _c_double_p]),
    ('epg_set_inits', C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _c_double_p]),
    ('epg_set_option', C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    ('epg_num_params', C.c_int, [C.c_void_p, C.c_int]),
    ('epg_logdensity', C.c_int, [C.c_void_p, C.c_int, C.c_int, _c_double_p, _c_double_p, _c_double_p,
                                 C.c_int, C.c_int]),
    ('epg_last_plan', C.c_int, [C.c_void_p, _c_int32_p, C.c_int]),
]

# fields of epg_last_plan, in order (include/epgpu.h)
PLAN_FIELDS = ('kernel', 'use_tc', 'chain_pad', 'tc_nst', 'resident', 'R', 'slices', 'NC', 'hot_nvec',
               'hot_levels', 'omega_smem', 'smem_total')


def load():
    """Load libepgpu.so and attach prototypes (no device needed for this)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EpgError(
            "libepgpu.so not found at {} -- build it with `python ep-stan_b200/build.py` "
            "(there is no CPU fallback)".format(LIB_PATH))
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(_c_double_p)


def _f64(a, order=None):
    return np.require(a, dtype=np.float64, requirements=['A'] + ([order] if order else []))


class Context:
    """One GPU == one shard of sites.  Thin, typed wrapper over the C ABI."""

    def __init__(self, device=0, stream=None):
        self._lib = load()
        h = C.c_void_p()
        # stream None -> private stream; an int (0 == the default stream) -> caller's stream
        own = stream is None
        rc = self._lib.epg_create(C.byref(h), int(device), None if own else C.c_void_p(int(stream)), int(own))
        if rc != 0 or not h:
            raise EpgError("epg_create failed on device {}: no usable CUDA device "
                           "(libepgpu has no CPU fallback)".format(device))
        self._h = h
        self.device = int(device)
        self.stream = None if own else int(stream)
        self.K = self.d = 0

    def on_torch_stream(self):
        """True when the context issues its work on torch's current stream of its device (so that
        torch.distributed collectives are stream-ordered with the kernels)."""
        if self.stream is None:
            return False
        import torch
        return int(torch.cuda.current_stream(self.device).cuda_stream) == self.stream

    def close(self):
        if getattr(self, '_h', None):
            self._lib.epg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise EpgError(self._lib.epg_last_error(self._h).decode())

    # ---- state ----
    def init_state(self, K, d):
        self._ck(self._lib.epg_init_state(self._h, K, d))
        self.K, self.d = K, d

    def upload(self, array, host, k0=0, k1=None):
        host = _f64(host, 'F')
        k1 = self.K if k1 is None else k1
        self._check_count(array, k0, k1, host)
        self._ck(self._lib.epg_upload(self._h, array, k0, k1, _dp(host)))

    def download(self, array, out, k0=0, k1=None):
        assert out.dtype == np.float64 and (out.flags.f_contiguous or out.flags.c_contiguous)
        k1 = self.K if k1 is None else k1
        self._check_count(array, k0, k1, out)
        self._ck(self._lib.epg_download(self._h, array, k0, k1, _dp(out)))
        return out

    def _check_count(self, array, k0, k1, buf):
        n = int(self._lib.epg_array_count(self._h, array, k0, k1))
        if n >= 0 and buf.size != n:
            raise ValueError("host buffer of %d doubles for device array %d, which holds %d" % (buf.size, array, n))

    def device_ptr(self, array):
        return self._lib.epg_device_ptr(self._h, array)

    def partial_tensor(self):
        """torch view (no copy) of EPG_PARTIAL = [sum Qi2 | sum ri2 | n_ok]: the
        buffer the ranks all-reduce with NCCL (method.py:1073-1074)."""
        import torch

        class _Alias(object):
            pass
        a = _Alias()
        a.__cuda_array_interface__ = {
            'shape': (self.d * self.d + self.d + 1,), 'typestr': '<f8',
            'data': (int(self.device_ptr(PARTIAL)), False), 'version': 2}
        return torch.as_tensor(a, device=torch.device('cuda', self.device))

    def _alias(self, array, n):
        import torch

        class _Alias(object):
            pass
        a = _Alias()
        a.__cuda_array_interface__ = {'shape': (n,), 'typestr': '<f8',
                                      'data': (int(self.device_ptr(array)), False), 'version': 2}
        return torch.as_tensor(a, device=torch.device('cuda', self.device))

    def dsum_tensor(self):
        """torch view (no copy) of EPG_DSUM = [sum dQi | sum dri | sum |delta_k|^2 | n_ok | slots]:
        the buffer the ranks all-reduce once per EP iteration."""
        return self._alias(DSUM, self.d * self.d + self.d + 2 + XCHG_SLOTS)

    def delta_sums(self, with_norms=True, slots=None):
        if slots is None:
            slots = np.zeros(0)
        slots = np.ascontiguousarray(slots, dtype=np.float64)
        self._ck(self._lib.epg_delta_sums_ex(self._h, 1 if with_norms else 0, _dp(slots) if len(slots) else None,
                                             len(slots)))

    def read_exchange(self):
        """(sum |delta_k|^2, n_ok, slots) of the (all-reduced) EPG_DSUM."""
        d = self.d
        buf = self.download(DSUM, np.empty(d * d + d + 2 + XCHG_SLOTS))
        return float(buf[d * d + d]), int(round(buf[d * d + d + 1])), buf[d * d + d + 2:]

    def mix_phi_sums(self, n):
        out = np.empty(self.d + 2 * self.d * self.d)
        self._ck(self._lib.epg_mix_phi_sums(self._h, int(n), _dp(out)))
        return out

    def update_from_sums(self, df):
        self._ck(self._lib.epg_update_from_sums(self._h, float(df)))

    def delta_snr(self):
        """(|sum_k delta_k|^2, sum_k |delta_k|^2, n_ok) of the (all-reduced) EPG_DSUM."""
        out = np.empty(3)
        self._ck(self._lib.epg_delta_snr(self._h, _dp(out)))
        return float(out[0]), float(out[1]), int(round(out[2]))

    def sync(self):
        self._ck(self._lib.epg_sync(self._h))

    def launch_count(self):
        return int(self._lib.epg_launch_count(self._h))

    # ---- EP path ----
    def cavity(self, k0=0, k1=None, proposal=False):
        k1 = self.K if k1 is None else k1
        flags = np.empty(k1 - k0, dtype=np.int32)
        all_ok = C.c_int(0)
        self._ck(self._lib.epg_cavity(self._h, k0, k1, int(proposal),
                                      flags.ctypes.data_as(_c_int32_p), C.byref(all_ok)))
        return flags.astype(bool), bool(all_ok.value)

    def set_draws(self, draws, n, k0=0, k1=None):
        """draws: (k1-k0, d, n) C-contiguous == per-site (n,d) F-order."""
        k1 = self.K if k1 is None else k1
        draws = _f64(draws, 'C')
        assert draws.size == (k1 - k0) * self.d * n
        self._ck(self._lib.epg_set_draws(self._h, k0, k1, n, _dp(draws)))

    def get_draws(self, n, k0=0, k1=None):
        k1 = self.K if k1 is None else k1
        out = np.empty((k1 - k0, self.d, n))
        self._ck(self._lib.epg_get_draws(self._h, k0, k1, n, _dp(out)))
        return out

    def moments(self, n, prec_estim='sample', k0=0, k1=None):
        k1 = self.K if k1 is None else k1
        flags = np.empty(k1 - k0, dtype=np.int32)
        n_ok = C.c_int(0)
        mode = PREC_ESTIM[prec_estim] if isinstance(prec_estim, str) else int(prec_estim)
        self._ck(self._lib.epg_moments(self._h, k0, k1, n, mode,
                                       flags.ctypes.data_as(_c_int32_p), C.byref(n_ok)))
        return flags.astype(bool), n_ok.value

    def fail_sites(self, sites):
        sites = np.ascontiguousarray(sites, dtype=np.int32)
        self._ck(self._lib.epg_fail_sites(self._h, len(sites), sites.ctypes.data_as(_c_int32_p)))

    def reinit_sites(self, sites):
        sites = np.ascontiguousarray(sites, dtype=np.int32)
        self._ck(self._lib.epg_reinit_sites(self._h, len(sites), sites.ctypes.data_as(_c_int32_p)))

    def param_stats(self, k0=0, k1=None):
        """(mean, sum of squared deviations), each [k1-k0, Pmax], of the transformed site parameters over
        the draws of the last sampling run (option 'param_stats')"""
        k1 = self.K if k1 is None else k1
        P = int(self._lib.epg_max_params(self._h))
        mean = np.empty((k1 - k0, P)); ssd = np.empty((k1 - k0, P))
        self._ck(self._lib.epg_get_param_stats(self._h, k0, k1, _dp(mean), _dp(ssd)))
        return mean, ssd

    def get_adapt(self, k, chains, pmax):
        """(inverse metric [chains, pmax], step size [chains]) site k's chains ended their last run with"""
        minv = np.empty((chains, pmax), dtype=np.float32)
        eps = np.empty(chains, dtype=np.float32)
        self._ck(self._lib.epg_get_adapt(self._h, int(k), minv.ctypes.data_as(C.POINTER(C.c_float)),
                                         eps.ctypes.data_as(C.POINTER(C.c_float))))
        return minv, eps

    def get_metric(self, k, chains):
        """inverse metric [chains, Pmax, Pmax] (fp32) site k's chains ended their last run with: diagonal
        (diag_e), the identity (unit_e) or the adapted full matrix (dense_e)"""
        P = int(self._lib.epg_max_params(self._h))
        out = np.empty((chains, P, P), dtype=np.float32)
        self._ck(self._lib.epg_get_metric(self._h, int(k), out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def update_partial(self, df):
        self._ck(self._lib.epg_update_partial(self._h, float(df)))

    def update_finish(self):
        pd = C.c_int(0)
        self._ck(self._lib.epg_update_finish(self._h, C.byref(pd)))
        return bool(pd.value)

    def accept(self):
        self._ck(self._lib.epg_accept(self._h))

    def global_moments(self, m_out=None, S_out=None):
        self._ck(self._lib.epg_global_moments(self._h, _dp(m_out), _dp(S_out)))

    def force_pd(self, thr, min_eig):
        forced = np.empty(self.K, dtype=np.int32)
        lam = np.empty(self.K)
        self._ck(self._lib.epg_force_pd(self._h, thr, min_eig, forced.ctypes.data_as(_c_int32_p), _dp(lam)))
        return forced.astype(bool), lam

    def damp_sweep(self, dfs, m_tgt, S_tgt):
        dfs = _f64(dfs, 'C')
        mse = np.empty(len(dfs))
        kl = np.empty(len(dfs))
        self._ck(self._lib.epg_damp_sweep(self._h, len(dfs), _dp(dfs), _dp(_f64(m_tgt, 'C')),
                                          _dp(_f64(S_tgt, 'F')), _dp(mse), _dp(kl)))
        return mse, kl

    # ---- stand-alone utilities ----
    def invert_normal_params(self, A, b=None, cho_form=False):
        """A: (batch, d, d) (each symmetric / upper factor), b: (batch, d) or None."""
        A = _f64(A, 'C')
        batch, d = A.shape[0], A.shape[1]
        # NumPy C-order (d,d) of a matrix M is the column-major image of M'; the
        # kernels read the UPPER triangle column-major, so hand them M' of M' = M
        # by transposing each item (upper factors are not symmetric).
        At = np.ascontiguousarray(A.transpose(0, 2, 1))
        outA = np.empty_like(At)
        outb = None
        if b is not None:
            b = _f64(b, 'C')
            outb = np.empty_like(b)
        ok = np.empty(batch, dtype=np.int32)
        self._ck(self._lib.epg_invert_normal_params(self._h, batch, d, _dp(At), _dp(b), int(cho_form),
                                                    _dp(outA), _dp(outb), ok.ctypes.data_as(_c_int32_p)))
        return outA, outb, ok.astype(bool)

    def olse(self, S, n, P=None):
        S = _f64(S, 'C')
        batch, d = S.shape[0], S.shape[1]
        out = np.empty_like(S)
        ok = np.empty(batch, dtype=np.int32)
        Pp = None if P is None else _f64(P, 'C')
        self._ck(self._lib.epg_olse(self._h, batch, d, _dp(S), int(n), _dp(Pp), _dp(out),
                                    ok.ctypes.data_as(_c_int32_p)))
        return out, ok.astype(bool)

    def cv_moments(self, draws, lp, Q_tilde, r_tilde, multiple_cv=True, regulate_a=None, max_a=None,
                   m_treshold=0.9, ret_a=False):
        """draws: (batch, d, n); lp: (batch, n); Q_tilde: (batch,d,d); r_tilde: (batch,d).
        ret_a: also return the coefficient arrays (a_S, a_m) of every item."""
        draws = _f64(draws, 'C')
        batch, d, n = draws.shape
        lp = _f64(lp, 'C')
        Qt = _f64(Q_tilde, 'C')
        rt = _f64(r_tilde, 'C')
        S_hat = np.empty((batch, d, d))
        m_hat = np.empty((batch, d))
        used = np.empty(batch, dtype=np.int32)
        d2 = d * (d + 1) // 2
        a_S = a_m = None
        if ret_a:
            a_S = np.empty((batch, d2, d2) if multiple_cv else (batch, d2))
            a_m = np.empty((batch, d, d) if multiple_cv else (batch, d))
        self._ck(self._lib.epg_cv_moments_ex(
            self._h, batch, n, d, _dp(draws), _dp(lp), _dp(Qt), _dp(rt), int(bool(multiple_cv)),
            float(regulate_a or 0.0), float(max_a or 0.0), float(m_treshold or 0.0),
            _dp(S_hat), _dp(m_hat), used.ctypes.data_as(_c_int32_p),
            _dp(a_S) if ret_a else None, _dp(a_m) if ret_a else None))
        if ret_a:
            return S_hat, m_hat, used, a_S, a_m
        return S_hat, m_hat, used

    # ---- sampler ----
    def upload_sites(self, model, D, k_lim, X, y, j_ind=None, Jk=None):
        k_lim = np.ascontiguousarray(k_lim, dtype=np.int64)
        X = _f64(X, 'C')
        y = np.ascontiguousarray(y, dtype=np.int64)
        ji = None if j_ind is None else np.ascontiguousarray(j_ind, dtype=np.int32)
        jk = None if Jk is None else np.ascontiguousarray(Jk, dtype=np.int32)
        self._ck(self._lib.epg_upload_sites(
            self._h, int(model), int(D), k_lim.ctypes.data_as(_c_int64_p), _dp(X),
            y.ctypes.data_as(_c_int64_p),
            None if ji is None else ji.ctypes.data_as(_c_int32_p),
            None if jk is None else jk.ctypes.data_as(_c_int32_p)))

    def tilted_sample(self, seeds, chains, iter, warmup=None, init_mode=0, k0=0, k1=None,
                      max_treedepth=10, adapt_delta=0.8, metric='diag_e', thin=1, stepsize=1.0,
                      stepsize_jitter=0.0, adapt_engaged=True, adapt_gamma=0.05, adapt_kappa=0.75, adapt_t0=10.0,
                      adapt_init_buffer=75, adapt_term_buffer=50, adapt_window=25, init_r=2.0):
        """metric: 'diag_e' (Stan's default), 'dense_e' or 'unit_e'; init_mode 0 random, 1 zeros, 2 previous
        last draws, INIT_GIVEN the starting points of set_inits.  The rest are PyStan's `thin`, `init_r` and
        `control` settings (include/epgpu.h, epg_sampler_adapt); draws per chain: ceil((iter - warmup) / thin)."""
        k1 = self.K if k1 is None else k1
        if metric not in METRICS:
            raise ValueError("metric must be one of %s, not %r" % (sorted(METRICS), metric))
        seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
        assert seeds.size == k1 - k0
        opts = SamplerOpts(chains=chains, iter=iter, warmup=-1 if warmup is None else warmup, thin=thin,
                           init_mode=init_mode, max_treedepth=max_treedepth, adapt_delta=adapt_delta,
                           metric=METRICS[metric])
        adapt = SamplerAdapt(stepsize=stepsize, stepsize_jitter=stepsize_jitter, gamma=adapt_gamma,
                             kappa=adapt_kappa, t0=adapt_t0, init_radius=init_r, engaged=1 if adapt_engaged else 0,
                             init_buffer=adapt_init_buffer, term_buffer=adapt_term_buffer, window=adapt_window)
        msteps = np.empty(k1 - k0)
        mrhat = np.empty(k1 - k0)
        nleap = np.empty(k1 - k0, dtype=np.int64)
        secs = C.c_double(0.0)
        self._ck(self._lib.epg_tilted_sample_ex(
            self._h, k0, k1, seeds.ctypes.data_as(_c_uint32_p), C.byref(opts), C.byref(adapt), _dp(msteps),
            _dp(mrhat), nleap.ctypes.data_as(_c_int64_p), C.byref(secs)))
        return msteps, mrhat, nleap, secs.value

    def set_inits(self, q, chains, k0=0, k1=None):
        """starting points of init_mode INIT_GIVEN: q [k1-k0, chains, <= Pmax] (NaN: drawn at random; padded
        with NaN to Pmax = epg_max_params)"""
        k1 = self.K if k1 is None else k1
        q = np.asarray(q, dtype=np.float64)
        P = int(self._lib.epg_max_params(self._h))
        if q.ndim != 3 or q.shape[:2] != (k1 - k0, chains) or q.shape[2] > P:
            raise ValueError("inits of shape %s, expected %s" % (q.shape, (k1 - k0, chains, P)))
        full = np.full((k1 - k0, chains, P), np.nan)
        full[:, :, :q.shape[2]] = q
        q = full
        self._ck(self._lib.epg_set_inits(self._h, k0, k1, int(chains), _dp(q)))

    def set_option(self, name, value):
        self._ck(self._lib.epg_set_option(self._h, name.encode(), float(value)))

    def num_params(self, k):
        return int(self._lib.epg_num_params(self._h, k))

    def logdensity(self, k, q, chains=None, ticks=2):
        """Tilted log-density and gradient of site k at the rows of q, evaluated in batches of `chains` under
        the launch plan tilted_sample makes for that many chains (None: when the single-box tensor-core pass
        may serve the sites, the most chains <= 16 at which the sampler keeps it, else 32); the likelihood pass
        runs `ticks` times before the read-out."""
        q = _f64(np.atleast_2d(q), 'C')
        nq, p = q.shape
        lp = np.empty(nq)
        grad = np.empty((nq, p))
        self._ck(self._lib.epg_logdensity(self._h, k, nq, _dp(q), _dp(lp), _dp(grad),
                                          0 if chains is None else int(chains), int(ticks)))
        return lp, grad

    def last_plan(self):
        """Launch plan of the last tilted_sample or logdensity: a dict over PLAN_FIELDS."""
        out = np.zeros(len(PLAN_FIELDS), dtype=np.int32)
        self._ck(self._lib.epg_last_plan(self._h, out.ctypes.data_as(_c_int32_p), len(out)))
        return dict(zip(PLAN_FIELDS, (int(v) for v in out)))

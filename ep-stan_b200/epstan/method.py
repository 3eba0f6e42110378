"""Distributed EP ("Expectation propagation as a way of life", arXiv:1412.4869)
-- the data-parallel inner loop on B200 GPUs.

Drop-in for the reference's ``epstan/method.py``: same ``Master`` / ``Worker``
classes, keyword arguments, defaults, return tuples, ``INFO_*`` codes and
F-order fp64 host arrays (``Q, r, Qi, ri, Qi2, ri2, dQi, dri, S, m``).  The
arithmetic of every EP iteration -- tilted sampling of all sites x chains,
moment matching, damped update, cavities, global moments -- runs in hand-written
sm_100a kernels behind the C ABI of ``libepgpu.so`` (include/epgpu.h); sites
are sharded in contiguous blocks over the ranks of a ``torch.distributed``
group with one all-reduce of the summed site parameters per update attempt.

There is no CPU fallback: without the library or a CUDA device construction
fails.
"""

__all__ = ['Worker', 'Master']

import sys
import time

import numpy as np

from . import _lib
from . import _comm
from . import util
from .util import (LinAlgError, BuiltinModel, load_stan, copy_fit_samples,
                   get_last_fit_sample)

# pystan.constants.MAX_UINT (reference method.py:40): upper bound of the seeds
MAX_UINT = 2 ** 31 - 1

_default_stream = None


def set_default_stream(cuda_stream_ptr):
    """Run subsequently created contexts on this cudaStream_t (an int, e.g.
    ``torch.cuda.current_stream().cuda_stream``); None -> private stream."""
    global _default_stream
    _default_stream = cuda_stream_ptr


def _pick_device():
    import os
    return int(os.environ.get('EPGPU_DEVICE', os.environ.get('LOCAL_RANK', 0)))


def _pick_stream(comm):
    if _default_stream is not None:
        return _default_stream
    if comm.size > 1 and getattr(comm, 'backend', None) == 'nccl':
        import torch
        torch.cuda.set_device(_pick_device())
        return torch.cuda.current_stream().cuda_stream    # NCCL orders against this stream
    return None


class _Shard(object):
    """The sites [k_begin, k_end) of one rank and the context that holds them."""

    def __init__(self, ctx, k_begin, k_end, K, comm):
        self.ctx, self.k_begin, self.k_end, self.K, self.comm = ctx, k_begin, k_end, K, comm
        self.n_local = k_end - k_begin
        self.sites_uploaded = False
        self.inits_set = set()          # local sites whose dict / list / function `init` is on the device

    def local(self, k):
        if not (self.k_begin <= k < self.k_end):
            raise RuntimeError("site {} lives on another rank".format(k))
        return k - self.k_begin


def _into(dst, src):
    """copy src into the caller-owned array dst (any strides)."""
    np.copyto(dst, src.reshape(dst.shape, order='F'))


class Worker(object):
    """Worker responsible of calculations for each site (reference
    method.py:121-475; same constructor, ``cavity`` and ``tilted``).

    ``stan_model`` may be a model path / name string (its base name selects a
    built-in CUDA density: m1b, m2b, m3b, m4b, m5b and their ``_sg`` variants), a
    ``util.BuiltinModel``, or any object with a PyStan-2 style
    ``sampling(data=, chains=, iter=, warmup=, thin=, init=, seed=, refresh=)``
    method, in which case its draws are moment-matched on the GPU.
    """

    DEFAULT_OPTIONS = {
        'init_prev'       : True,
        # extension: with init_prev the built-in sampler also starts each warm-up from the metric and step
        # size its previous run adapted (False: Stan's unit metric and step size 1 every EP iteration)
        'adapt_prev'      : True,
        'prec_estim'      : 'sample',
        'prec_estim_skip' : 0,
        'verbose'         : False
    }

    DEFAULT_STAN_PARAMS = {
        'chains'          : 4,
        'iter'            : 1000,
        'warmup'          : None,
        'thin'            : 1,
        'init'            : 'random',
        # extension (PyStan's own `sampling` keyword, which the reference never sets): radius of the random
        # inits U(-init_r, init_r); None = Stan's 2 (and not passed to a caller-supplied sampler)
        'init_r'          : None,
        # extension (PyStan's own `sampling` keyword, which the reference never sets): NUTS controls of the
        # built-in sampler, any of CONTROL_KEYS; None = Stan's defaults
        'control'         : None
    }

    # PyStan 2.17's `control` keys (Stan's defaults): max_treedepth 10, adapt_delta 0.8, metric 'diag_e'
    # ('dense_e', 'unit_e'), stepsize 1, stepsize_jitter 0, adapt_engaged True, adapt_gamma 0.05, adapt_kappa 0.75,
    # adapt_t0 10, adapt_init_buffer 75, adapt_term_buffer 50, adapt_window 25 (include/epgpu.h, epg_sampler_adapt)
    CONTROL_KEYS = ('max_treedepth', 'adapt_delta', 'metric', 'stepsize', 'stepsize_jitter', 'adapt_engaged',
                    'adapt_gamma', 'adapt_kappa', 'adapt_t0', 'adapt_init_buffer', 'adapt_term_buffer',
                    'adapt_window')

    PREC_ESTIM_OPTIONS = ('sample', 'olse')

    RESERVED_STAN_PARAMETER_NAMES = ['X', 'y', 'N', 'D', 'mu_phi', 'Omega_phi']

    def __init__(self, index, stan_model, dphi, X, y, A=None, **options):
        shard = options.pop('_shard', None)
        Mat = options.pop('_Mat', None)
        vec = options.pop('_vec', None)
        for (kw, default) in self.DEFAULT_OPTIONS.items():
            options.setdefault(kw, default)
        for (kw, default) in self.DEFAULT_STAN_PARAMS.items():
            options.setdefault(kw, default)
        self.stan_params = {}
        for (kw, val) in options.items():
            if kw in self.DEFAULT_STAN_PARAMS:
                self.stan_params[kw] = val
            elif kw not in self.DEFAULT_OPTIONS:
                raise TypeError("Unexpected option '{}'".format(kw))
        if A is None:
            A = {}

        # cavity precision / mean after `cavity`; the tilted mean lands in `vec`
        # after `tilted` (reference method.py:190-196)
        self.Mat = np.empty((dphi, dphi), order='F') if Mat is None else Mat
        self.vec = np.empty(dphi) if vec is None else vec
        self.phase = 0
        self.nsamp = None
        self.Q = None
        self.r = None

        self.X, self.y, self.A = X, y, A
        self.data = dict(N=X.shape[0], X=X, y=y, mu_phi=self.vec, Omega_phi=self.Mat.T, **A)
        if len(X.shape) == 2:
            self.data['D'] = X.shape[1]

        self.index = index
        if isinstance(stan_model, str):
            stan_model = load_stan(stan_model)
        self.stan_model = stan_model
        self.builtin = isinstance(stan_model, BuiltinModel)
        if not self.builtin and not hasattr(stan_model, 'sampling'):
            raise TypeError("`stan_model` must be a model name or an object with a `sampling` method")
        self.dphi = dphi
        self.iteration = 0
        self.last_time = None
        self.last_msteps = None
        self.last_mrhat = None
        self.last_n_leapfrog = 0
        self.saved_samples = None

        self.init_prev = options['init_prev']
        self.adapt_prev = bool(options['adapt_prev'])
        if self.builtin:
            self._check_sampler_args()
        self.init_orig = self.stan_params['init']
        if self.init_prev and not isinstance(self.init_orig, str):
            raise ValueError("Arg. `init` has to be a string if `init_prev` is True")
        self._have_prev = False

        self.prec_estim = options['prec_estim']
        if self.prec_estim not in self.PREC_ESTIM_OPTIONS:
            raise ValueError("Invalid value for option `prec_estim`")
        self.prec_estim_skip = options['prec_estim_skip'] if self.prec_estim != 'sample' else 0
        self.verbose = options['verbose']

        if shard is None:
            # stand-alone worker: a private one-site context
            ctx = Master._context_factory(_pick_device(), _default_stream)
            ctx.init_state(1, dphi)
            shard = _Shard(ctx, index, index + 1, index + 1, _comm.Comm())
            if self.builtin:
                _upload_site_block(shard, self.stan_model, [self])
        self._shard = shard

    # -- helpers -------------------------------------------------------------
    def _check_sampler_args(self):
        """ValueError for a sampling argument the built-in sampler cannot honour as PyStan would"""
        sp = self.stan_params

        def is_int(v):
            return isinstance(v, (int, np.integer)) and not isinstance(v, bool)

        def is_pos(v):
            return isinstance(v, (int, float, np.integer, np.floating)) and not isinstance(v, bool) and \
                np.isfinite(v) and v > 0
        if not (is_int(sp['thin']) and sp['thin'] >= 1):
            raise ValueError("`thin` must be an integer >= 1 (got {!r})".format(sp['thin']))
        init = sp['init']
        if isinstance(init, str):
            if init not in ('random', '0'):
                raise ValueError("`init` must be 'random', '0', a dict, a list of dicts or a function "
                                 "(got {!r})".format(init))
        elif isinstance(init, (list, tuple)):
            if len(init) != sp['chains'] or not all(isinstance(v, dict) for v in init):
                raise ValueError("`init` as a list needs one dict per chain ({})".format(sp['chains']))
        elif not (isinstance(init, dict) or callable(init) or (is_int(init) and init == 0)):
            raise ValueError("`init` must be 'random', '0', a dict, a list of dicts or a function")
        if sp['init_r'] is not None and not is_pos(sp['init_r']):
            raise ValueError("`init_r` must be positive (got {!r})".format(sp['init_r']))
        ctl = sp['control']
        if ctl is None:
            return
        if not isinstance(ctl, dict) or set(ctl) - set(self.CONTROL_KEYS):
            raise ValueError("built-in sampler: `control` may hold {} only".format(', '.join(self.CONTROL_KEYS)))
        if ctl.get('metric', 'diag_e') not in _lib.METRICS:
            raise ValueError("built-in sampler: control['metric'] must be one of {} (got {!r})".format(
                sorted(_lib.METRICS), ctl['metric']))
        for key in ('stepsize', 'adapt_gamma', 'adapt_kappa', 'adapt_t0'):
            if key in ctl and not is_pos(ctl[key]):
                raise ValueError("control['{}'] must be positive and finite (got {!r})".format(key, ctl[key]))
        if 'stepsize_jitter' in ctl:
            j = ctl['stepsize_jitter']
            if not (isinstance(j, (int, float, np.integer, np.floating)) and not isinstance(j, bool)
                    and 0 <= j <= 1):
                raise ValueError("control['stepsize_jitter'] must be in [0, 1] (got {!r})".format(j))
        if 'adapt_engaged' in ctl and not (isinstance(ctl['adapt_engaged'], (bool, np.bool_)) or
                                           (is_int(ctl['adapt_engaged']) and ctl['adapt_engaged'] in (0, 1))):
            raise ValueError("control['adapt_engaged'] must be a bool (got {!r})".format(ctl['adapt_engaged']))
        for key, lo in (('adapt_init_buffer', 0), ('adapt_term_buffer', 0), ('adapt_window', 1)):
            if key in ctl and not (is_int(ctl[key]) and ctl[key] >= lo):
                raise ValueError("control['{}'] must be an integer >= {} (got {!r})".format(key, lo, ctl[key]))
        if 'stepsize' in ctl and self.init_prev and self.adapt_prev and ctl.get('adapt_engaged', True):
            # every run after the first starts from the carried step size: the value would apply once only
            raise ValueError("control['stepsize'] with init_prev and adapt_prev (the defaults) would set the "
                             "first EP iteration's step size only: pass adapt_prev=False")

    def _sampler_kw(self):
        """keyword arguments of Context.tilted_sample beyond the run's shape"""
        sp = self.stan_params
        kw = dict(sp['control'] or {})
        kw['thin'] = int(sp['thin'])
        if sp['init_r'] is not None:
            kw['init_r'] = float(sp['init_r'])
        return kw

    def _site_layout(self):
        """(family, D, J) of the site: what util.init_values needs"""
        J = 1 if self.stan_model.single_group else int(self.A['J'])
        return (self.stan_model.family, self.X.shape[1], J)

    def _nsamp(self):
        sp = self.stan_params
        warm = sp['iter'] // 2 if sp['warmup'] is None else sp['warmup']
        return sp['chains'] * (-(-(sp['iter'] - warm) // sp['thin']))

    def _mode_now(self):
        """prec_estim to use this iteration (method.py:413,436-437)."""
        if self.prec_estim == 'sample' or self.prec_estim_skip > 0:
            return 'sample'
        return self.prec_estim

    def _init_mode(self):
        if self.init_prev and self._have_prev:
            return 2
        init = self.stan_params['init']
        if isinstance(init, str):
            if init == 'random':
                return 0
            if init == '0':
                return 1
        elif isinstance(init, (dict, list, tuple)) or callable(init):
            return _lib.INIT_GIVEN
        elif init == 0:
            return 1
        raise ValueError("`init` must be 'random', '0', a dict, a list of dicts or a function")

    def _host_sample(self, seed_stan, save_samples):
        """Draws from a caller-supplied PyStan-style sampler object
        (the reference's in-process branch, method.py:369-397)."""
        t0 = time.perf_counter()
        params = dict(self.stan_params, seed=seed_stan, refresh=-1)
        for kw in ('control', 'init_r'):
            if params.get(kw) is None:
                params.pop(kw, None)               # (the reference never passes them)
        fit = self.stan_model.sampling(data=self.data, **params)
        self.last_time = time.perf_counter() - t0
        self.last_msteps = float(np.mean([np.mean(p['stepsize__']) for p in fit.get_sampler_params()]))
        self.last_mrhat = float(np.max(fit.summary()['summary'][:-1, -1]))
        samp = copy_fit_samples(fit, 'phi')
        if self.init_prev:
            self.stan_params['init'] = get_last_fit_sample(fit)
        if save_samples:
            self.saved_samp = {par: fit.extract(pars=par)[par] for par in save_samples}
        return samp

    # -- API -----------------------------------------------------------------
    def cavity(self, Q, r, Qi, ri):
        """Form the cavity distribution and convert it to moment parameters
        (reference method.py:267-302).  Returns True if it is pos.def."""
        sh = self._shard
        kl = sh.local(self.index)
        self.Q = Q
        self.r = r
        ctx = sh.ctx
        ctx.upload(_lib.Q, Q)
        ctx.upload(_lib.R, r)
        ctx.upload(_lib.QI, np.asfortranarray(Qi), kl, kl + 1)
        ctx.upload(_lib.RI, np.ascontiguousarray(ri), kl, kl + 1)
        flags, _ = ctx.cavity(kl, kl + 1, proposal=False)
        buf = np.empty((self.dphi, self.dphi), order='F')
        _into(self.Mat, ctx.download(_lib.CAVQ, buf, kl, kl + 1))
        _into(self.vec, ctx.download(_lib.CAVM, np.empty(self.dphi), kl, kl + 1))
        self.phase = 1 if flags[0] else 0
        return bool(flags[0])

    def tilted(self, dQi, dri, save_samples=None, seed=None):
        """Estimate the tilted distribution parameters and write the site
        parameter updates into the caller's ``dQi``, ``dri`` (reference
        method.py:305-475).  ``cavity`` must have been called before."""
        if self.phase != 1:
            raise RuntimeError('Cavity has to be calculated before tilted.')
        rng = seed if isinstance(seed, np.random.RandomState) else np.random.RandomState(seed)
        seed_stan = int(rng.randint(0, MAX_UINT))
        self.stan_params['seed'] = seed_stan
        sh = self._shard
        ctx = sh.ctx
        kl = sh.local(self.index)
        n = self._nsamp()
        ctx.upload(_lib.Q, self.Q)
        ctx.upload(_lib.R, self.r)
        ctx.upload(_lib.CAVQ, np.asfortranarray(self.Mat), kl, kl + 1)
        ctx.upload(_lib.CAVM, np.ascontiguousarray(self.vec), kl, kl + 1)
        if self.builtin:
            sp = self.stan_params
            mode = self._init_mode()
            if mode == _lib.INIT_GIVEN:
                _upload_inits(sh, [self])
            msteps, mrhat, nleap, secs = ctx.tilted_sample(
                [seed_stan], sp['chains'], sp['iter'], sp['warmup'], mode, kl, kl + 1, **self._sampler_kw())
            self.last_time, self.last_msteps, self.last_mrhat = secs, float(msteps[0]), float(mrhat[0])
            self.last_n_leapfrog = int(nleap[0])
            self._have_prev = True
            if save_samples and 'phi' in save_samples:
                self.saved_samp = {'phi': np.asfortranarray(ctx.get_draws(n, kl, kl + 1)[0].T)}
        else:
            samp = self._host_sample(seed_stan, save_samples)
            n = samp.shape[0]
            ctx.set_draws(np.ascontiguousarray(samp.T)[None], n, kl, kl + 1)
        if self.verbose:
            print('\n   sampling runtime: {:.4}'.format(self.last_time))
            print('    mean stepsize: {:.4}'.format(self.last_msteps))
            print('    max Rhat: {:.4}'.format(self.last_mrhat))
        self.nsamp = n
        mode = self._mode_now()
        flags, _ = ctx.moments(n, mode, kl, kl + 1)
        if mode == 'sample' and self.prec_estim_skip > 0:
            self.prec_estim_skip -= 1
        d = self.dphi
        _into(dQi, ctx.download(_lib.DQI, np.empty((d, d), order='F'), kl, kl + 1))
        _into(dri, ctx.download(_lib.DRI, np.empty(d), kl, kl + 1))
        _into(self.vec, ctx.download(_lib.TMEAN, np.empty(d), kl, kl + 1))
        pos_def = bool(flags[0])
        self.phase = 2 if pos_def else 0
        self.iteration += 1
        return pos_def


def _upload_site_block(shard, model, workers):
    """Ship the design matrices of the local sites to the GPU (built-in models)."""
    D = workers[0].X.shape[1]
    k_lim = np.concatenate(([0], np.cumsum([w.X.shape[0] for w in workers])))
    X = np.ascontiguousarray(np.concatenate([w.X for w in workers], axis=0), dtype=np.float64)
    y = np.concatenate([np.asarray(w.y) for w in workers]).astype(np.int64)
    j_ind = Jk = None
    if not model.single_group:
        for w in workers:
            if 'j_ind' not in w.A or 'J' not in w.A:
                raise ValueError("multi-group model '{}' needs A_n['j_ind'] (1-based) and A_k['J']"
                                 .format(model.name))
        j_ind = np.concatenate([np.asarray(w.A['j_ind']) - 1 for w in workers]).astype(np.int32)
        Jk = np.array([int(w.A['J']) for w in workers], dtype=np.int32)
        for w, J in zip(workers, Jk):
            ji = np.asarray(w.A['j_ind']) - 1
            if ji.min() < 0 or ji.max() >= J or np.any(np.diff(ji) < 0):
                raise ValueError("`j_ind` must be sorted and within 1..J for every site")
    shard.ctx.upload_sites(model.model_id, D, k_lim, X, y, j_ind, Jk)
    shard.ctx.set_option('carry_adapt', 1 if workers[0].adapt_prev else 0)
    shard.sites_uploaded = True
    shard.inits_set = set()


def _upload_inits(shard, workers):
    """Starting points of a dict / list / function `init` for a contiguous block of local sites, once per
    context (a function is called once per chain here, not once per EP iteration)."""
    kls = [shard.local(w.index) for w in workers]
    if all(k in shard.inits_set for k in kls):
        return
    sp = workers[0].stan_params
    q = util.init_values(sp['init'], sp['chains'], [w._site_layout() for w in workers])
    shard.ctx.set_inits(q, sp['chains'], kls[0], kls[-1] + 1)
    shard.inits_set.update(kls)


class Master(object):
    """Manages the distributed EP algorithm (reference method.py:478-1478).

    Parameters are those of the reference ``Master`` (see its docstring,
    method.py:480-617): ``site_model, X, y`` and the keyword arguments ``A``,
    ``A_n``, ``A_k``, ``site_ind`` / ``site_ind_ord`` / ``site_sizes``, ``dphi``,
    ``prior``, ``init_site``, ``df0``, ``df_decay``, ``df_treshold``,
    ``overwrite_model`` plus the worker options ``init_prev``, ``prec_estim``,
    ``prec_estim_skip``, ``verbose``, ``chains``, ``iter``, ``warmup``, ``thin``,
    ``init``.

    Differences that matter to a caller:
      * ``site_model`` given as a path selects a built-in CUDA density by its
        base name (there is no Stan compiler); a sampler object is accepted too.
      * when a multi-rank ``torch.distributed`` group is initialised, each rank
        keeps a contiguous block of sites on its own GPU; the host arrays are
        made complete on every rank when ``run`` returns.
    """

    INFO_OK = 0
    INFO_INVALID_PRIOR = 1
    INFO_DF_TRESHOLD_REACHED_GLOBAL = 2
    INFO_DF_TRESHOLD_REACHED_CAVITY = 3
    INFO_ALL_SITES_FAIL = 4

    MIN_EIG_TRESHOLD = 1e-5
    MIN_EIG = 0.5

    DEFAULT_KWARGS = dict(
        A                 = {},
        A_n               = {},
        A_k               = {},
        site_ind          = None,
        site_ind_ord      = None,
        site_sizes        = None,
        dphi              = None,
        prior             = None,
        init_site         = None,
        df0               = None,
        df_decay          = 0.8,
        df_treshold       = 1e-6,
        overwrite_model   = False,
        # extensions (not in the reference): automatic damping selection, see `_select_df`
        df_select         = None,
        df_min            = None,
        df_snr_z          = 3.0,
        df_snr_min        = 0.5,
        # extension: a site whose max split-Rhat exceeds this is treated as failed for the iteration
        # (its update is skipped like a failed moment estimate, method.py:460-465); None = never
        rhat_max          = None
    )

    # hooks (tests substitute a CPU double for the context / a communicator)
    _context_factory = staticmethod(lambda device, stream: _lib.Context(device, stream))
    _comm_factory = staticmethod(_comm.default_comm)

    def __init__(self, site_model, X, y, **kwargs):
        self.worker_options = {}
        for (kw, val) in kwargs.items():
            if kw in Worker.DEFAULT_OPTIONS or kw in Worker.DEFAULT_STAN_PARAMS:
                self.worker_options[kw] = val
            elif kw not in self.DEFAULT_KWARGS:
                raise TypeError("Unexpected keyword argument '{}'".format(kw))
        for (kw, default) in self.DEFAULT_KWARGS.items():
            kwargs.setdefault(kw, default)
        for (kw, default) in Worker.DEFAULT_OPTIONS.items():
            self.worker_options.setdefault(kw, default)
        for (kw, default) in Worker.DEFAULT_STAN_PARAMS.items():
            self.worker_options.setdefault(kw, default)

        if isinstance(site_model, str):
            site_model = load_stan(site_model, kwargs['overwrite_model'])
        self.site_model = site_model

        self.N = X.shape[0]
        if len(X.shape) == 2:
            self.D = X.shape[1]
        elif len(X.shape) == 1:
            self.D = None
        else:
            raise ValueError("Argument `X` should be one or two dimensional")
        self.X = X
        if len(y.shape) != 1:
            raise ValueError("Argument `y` should be one dimensional")
        if y.shape[0] != self.N:
            raise ValueError("The shapes of `y` and `X` does not match")
        self.y = y

        # site partition (reference method.py:691-730)
        if kwargs['site_sizes'] is not None:
            self.Nk = np.asarray(kwargs['site_sizes'])
            self.K = len(self.Nk)
            self.k_lim = np.concatenate(([0], np.cumsum(self.Nk)))
            self.k_ind = np.repeat(np.arange(self.K), self.Nk).astype(np.int64)
        elif kwargs['site_ind_ord'] is not None:
            self.k_ind = kwargs['site_ind_ord']
            self.Nk = np.bincount(self.k_ind)
            self.K = len(self.Nk)
            self.k_lim = np.concatenate(([0], np.cumsum(self.Nk)))
        elif kwargs['site_ind'] is not None:
            k_ind = kwargs['site_ind']
            k_sort = k_ind.argsort(kind='mergesort')
            self.k_ind = k_ind[k_sort]
            self.Nk = np.bincount(self.k_ind)
            self.K = len(self.Nk)
            self.k_lim = np.concatenate(([0], np.cumsum(self.Nk)))
            self.X = self.X[k_sort]
            self.y = self.y[k_sort]
        else:
            raise NotImplementedError("Auto clustering not yet implemented")
        if self.k_lim[-1] != self.N:
            raise ValueError("Site definition does not match with `X`")
        if np.any(self.Nk == 0):
            raise ValueError("Empty sites: {}. Index the sites from 1 to K-1"
                             .format(np.nonzero(self.Nk == 0)[0]))
        if self.K < 2:
            raise ValueError("Distributed EP should be run with at least two sites.")
        self.X = np.ascontiguousarray(self.X)
        self.y = np.ascontiguousarray(self.y)

        # additional data (reference method.py:736-769)
        reserved = Worker.RESERVED_STAN_PARAMETER_NAMES
        self.A = kwargs['A']
        for key in self.A:
            if key in reserved:
                raise ValueError("Additional data name {} clashes.".format(key))
        self.A_n = dict(kwargs['A_n'])
        for (key, val) in kwargs['A_n'].items():
            if val.shape[0] != self.N:
                raise ValueError("The shapes of `A_n[{}]` and `X` does not match".format(repr(key)))
            if key in reserved or key in self.A:
                raise ValueError("Additional data name {} clashes.".format(key))
            if not val.flags['CARRAY']:
                self.A_n[key] = np.ascontiguousarray(val)
        self.A_k = kwargs['A_k']
        for (key, val) in self.A_k.items():
            if len(val) != self.K:
                raise ValueError("Array-like length mismatch in `A_k` (should be: {}, found: {})"
                                 .format(self.K, len(val)))
            if key in reserved or key in self.A or key in self.A_n:
                raise ValueError("Additional data name {} clashes.".format(key))

        # prior (reference method.py:771-797)
        prior = kwargs['prior']
        self.dphi = kwargs['dphi']
        if prior is None:
            if self.dphi is None:
                raise ValueError("If arg. `prior` is not provided, arg. `dphi` has to be given")
            self.Q0 = np.eye(self.dphi).T
            self.r0 = np.zeros(self.dphi)
        else:
            if not isinstance(prior, dict):
                raise TypeError("Argument `prior` is of wrong type")
            if 'Q' in prior and 'r' in prior:
                self.Q0 = np.asfortranarray(prior['Q'], dtype=np.float64)
                self.r0 = np.asarray(prior['r'], dtype=np.float64)
            elif 'S' in prior and 'm' in prior:
                from .util import invert_normal_params
                self.Q0, self.r0 = invert_normal_params(prior['S'], prior['m'])
            else:
                raise ValueError("Argument `prior` is not appropriate")
            if self.dphi is None:
                self.dphi = self.Q0.shape[0]
            if self.Q0.shape[0] != self.dphi or self.r0.shape[0] != self.dphi:
                raise ValueError("Arg. `dphi` does not match with `prior`")
        d, K = self.dphi, self.K

        # damping (reference method.py:799-814)
        self.df_decay = kwargs['df_decay']
        self.df_treshold = kwargs['df_treshold']
        if kwargs['df0'] is None:
            default_df = 1 / self.K
            self.df0 = lambda i: default_df
        elif isinstance(kwargs['df0'], (float, int)):
            if kwargs['df0'] <= 0 or kwargs['df0'] > 1:
                raise ValueError("Constant initial damping factor has to be in (0,1]")
            self.df0 = lambda i: kwargs['df0']
        else:
            self.df0 = kwargs['df0']

        self.df_select = kwargs['df_select']
        if self.df_select not in (None, 'snr'):
            raise ValueError("Arg. `df_select` has to be None or 'snr'")
        if self.df_select == 'snr' and kwargs['df0'] is None:
            self.df0 = lambda i: 1.0              # the selection rule picks below this cap
        self.df_min = min(1.0 / self.K, 0.2) if kwargs['df_min'] is None else float(kwargs['df_min'])
        self.df_snr_z = float(kwargs['df_snr_z'])
        self.df_snr_min = float(kwargs['df_snr_min'])
        self.rhat_max = kwargs['rhat_max']
        # per-iteration record of the last run(): damping used, update attempts, selection statistics
        self.history = dict(df=[], attempts=[], snr=[], n_ok=[], rhat_sites=[], n_fail=[], rejected=[])
        self._last_rejected = []

        # host mirrors (reference method.py:836-851), F-order as the reference
        self.S = np.empty((d, d), order='F')
        self.m = np.empty(d)
        self.Q = self.Q0.copy(order='F')
        self.r = self.r0.copy()
        self.Qi = np.zeros((d, d, K), order='F')
        self.ri = np.zeros((d, K), order='F')
        self.Qi2 = np.zeros((d, d, K), order='F')
        self.ri2 = np.zeros((d, K), order='F')
        self.dQi = np.zeros((d, d, K), order='F')
        self.dri = np.zeros((d, K), order='F')
        self._cavQ = np.zeros((d, d, K), order='F')   # workers' Mat are views of this
        self._cavm = np.zeros((d, K), order='F')      # workers' vec are views of this
        if kwargs['init_site'] is not None:
            if isinstance(kwargs['init_site'], np.ndarray):
                self.Qi[:] = kwargs['init_site'][:, :, None]
            else:
                self.Qi[np.arange(d), np.arange(d), :] = self.K / (kwargs['init_site'] ** 2)
        self.iter = 0
        # when True, run() leaves the state on the GPU between calls: the host
        # mirrors are neither uploaded first nor refreshed afterwards (sync_host())
        self.keep_on_device = False
        self._host_stale = False      # the device state is newer than the host mirrors (keep_on_device runs)
        self.n_leapfrog_total = 0     # gradient evaluations spent by the built-in sampler (local sites)

        # shard + device context
        self.comm = self._comm_factory()
        if K < self.comm.size:
            raise ValueError("Fewer sites ({}) than ranks ({}): every rank needs at least one site"
                             .format(K, self.comm.size))
        k_begin, k_end = self.comm.shard(K)
        ctx = self._context_factory(_pick_device(), _pick_stream(self.comm))
        ctx.init_state(k_end - k_begin, d)
        self._shard = _Shard(ctx, k_begin, k_end, K, self.comm)
        ctx.upload(_lib.Q0, self.Q0)
        ctx.upload(_lib.R0, self.r0)

        # workers (reference method.py:816-834; it slices the *unsorted* X there,
        # we slice the sorted copy, which is what the algorithm needs)
        self.workers = []
        for k in range(K):
            lo, hi = self.k_lim[k], self.k_lim[k + 1]
            A = dict((key, val[lo:hi]) for (key, val) in self.A_n.items())
            A.update(self.A)
            for (key, val) in self.A_k.items():
                A[key] = val[k]
            self.workers.append(Worker(
                k, self.site_model, d, self.X[lo:hi], self.y[lo:hi], A=A,
                _shard=self._shard, _Mat=self._cavQ[:, :, k], _vec=self._cavm[:, k],
                **self.worker_options))
        self.builtin = self.workers[0].builtin
        if self.builtin and self._shard.n_local > 0:
            _upload_site_block(self._shard, self.site_model, self.workers[k_begin:k_end])

        # initial global approximation and cavities (reference method.py:866-882)
        self._push_state()
        ctx.update_partial(0.0)
        self._allreduce_partial()
        if not ctx.update_finish():
            raise ValueError("Initial approximation is not pos.def.")
        ok = self._all_ranks(ctx.cavity(proposal=False)[1])
        if not ok:
            raise ValueError("Initial cavity is not pos.def.")
        self._pull_state()
        for w in self.workers:
            w.Q, w.r, w.phase = self.Q, self.r, 1

    # ---- host <-> device mirrors ---------------------------------------------
    def _loc(self, arr, axis):
        sl = [slice(None)] * arr.ndim
        sl[axis] = slice(self._shard.k_begin, self._shard.k_end)
        return np.asfortranarray(arr[tuple(sl)])

    def _push_state(self, with_cavity=False):
        """host arrays are the truth at API boundaries: ship them to the device"""
        ctx = self._shard.ctx
        if self._shard.n_local == 0:
            return
        ctx.upload(_lib.Q, self.Q)
        ctx.upload(_lib.R, self.r)
        for aid, arr, ax in ((_lib.QI, self.Qi, 2), (_lib.RI, self.ri, 1),
                             (_lib.DQI, self.dQi, 2), (_lib.DRI, self.dri, 1)):
            ctx.upload(aid, self._loc(arr, ax))
        if with_cavity:
            ctx.upload(_lib.CAVQ, self._loc(self._cavQ, 2))
            ctx.upload(_lib.CAVM, self._loc(self._cavm, 1))

    def _pull_state(self):
        """refresh every host mirror from the device (and the other ranks)"""
        sh = self._shard
        ctx, d = sh.ctx, self.dphi
        ctx.download(_lib.Q, self.Q)
        ctx.download(_lib.R, self.r)
        for aid, arr, ax in ((_lib.QI, self.Qi, 2), (_lib.RI, self.ri, 1),
                             (_lib.QI2, self.Qi2, 2), (_lib.RI2, self.ri2, 1),
                             (_lib.DQI, self.dQi, 2), (_lib.DRI, self.dri, 1),
                             (_lib.CAVQ, self._cavQ, 2), (_lib.CAVM, self._cavm, 1)):
            shape = (d, d, sh.n_local) if ax == 2 else (d, sh.n_local)
            loc = ctx.download(aid, np.empty(shape, order='F')) if sh.n_local else np.empty(shape, order='F')
            if self.comm.size > 1:
                arr[...] = self.comm.allgather_sites(loc, self.K, ax)
            else:
                arr[...] = loc
        self._host_stale = False

    def _allreduce_device(self, tensor):
        """Sum a device buffer of the context over the ranks.  The collective runs on torch's
        current stream; when the context works on another stream the two are ordered explicitly."""
        if self.comm.size <= 1:
            return
        ctx = self._shard.ctx
        same = getattr(ctx, 'on_torch_stream', lambda: True)()
        if not same:
            ctx.sync()                       # kernels that wrote the buffer have finished
        self.comm.allreduce_sum_(tensor)
        if not same:
            self.comm.sync_device()          # the reduced values are visible to the context's stream

    def _allreduce_partial(self):
        if self.comm.size > 1:
            self._allreduce_device(self._shard.ctx.partial_tensor())

    def _select_df(self, cap, exchanged=False):
        """Automatic damping (`df_select='snr'`; extension, SURVEY 8f rank 1).

        At an EP fixed point every site delta has zero mean: the summed update is the sum of K
        independent Monte Carlo errors.  With T2 = |sum_k delta_k|^2 and N2 = the K/(K-1)-corrected
        sum_k |delta_k - mean|^2 in the Fisher metric of the current approximation, 1 - N2/T2 is
        the positive-part shrinkage estimate of the fraction of the summed update that is signal
        (the damping that minimises the expected squared distance to the fixed point).  The
        estimate is taken `df_snr_z` standard errors low, capped by `df0(iter)` and floored at
        `df_min` (default min(1/K, 0.2), the reference's asymptotic damping, fit.py:176-186).

        Below `df_snr_min` (default 0.5: noise power above signal power) the floor is used outright.
        A small apparent signal fraction is not trustworthy: the unbiased-precision factor
        (n-d-2) of method.py:431-434 assumes independent Gaussian draws, and a relative bias b of
        the per-site precision estimate (autocorrelated draws: b ~ (tau-1)/n) is COHERENT over the
        sites -- it enters the summed update K times and looks like signal.  At the floor 1/K the
        update is the average of the sites' tilted estimates and such a bias passes through once."""
        ctx = self._shard.ctx
        if not exchanged:                       # (several ranks: `_exchange` has reduced the sums already)
            ctx.delta_sums()
            self._allreduce_device(ctx.dsum_tensor())
        T2, S2, n_ok = ctx.delta_snr()
        d = self.dphi
        dof = d * (d + 1) / 2.0 + d
        raw = 0.0
        N2 = float('nan')
        if n_ok >= 2 and T2 > 0.0:
            N2 = max(S2 - T2 / n_ok, 0.0) * n_ok / (n_ok - 1.0)
            raw = 1.0 - (1.0 + self.df_snr_z * np.sqrt(2.0 / dof)) * N2 / T2
        df = min(cap, max(self.df_min, raw)) if raw >= self.df_snr_min else min(cap, self.df_min)
        self.history['snr'].append((T2, N2, raw))
        return df

    def _exchange(self, with_norms, n_fail, maxima):
        """THE exchange of an EP iteration (SURVEY 8e): one all-reduce(sum) of EPG_DSUM =
        [sum_k dQi | sum_k dri | sum_k |delta_k|^2 | n_ok | slots].  The slots carry this rank's count of
        failed sites and, in a per-rank block, its analytics maxima (summing blocks that are zero on every
        other rank gathers them).  Returns (n_ok, n_fail, [max sampling time, max step size, max Rhat])."""
        ctx, comm = self._shard.ctx, self.comm
        slots = np.zeros(_lib.XCHG_SLOTS)
        per = len(maxima) + 1
        if 1 + per * comm.size > _lib.XCHG_SLOTS:
            raise ValueError("too many ranks for the exchange slots")
        slots[0] = n_fail
        base = 1 + per * comm.rank              # this rank's block: [bit i set = value i present, values ...]
        bits = 0
        for i, v in enumerate(maxima):
            if v is not None and np.isfinite(v):
                bits |= 1 << i
                slots[base + 1 + i] = v
        slots[base] = float(bits)
        ctx.delta_sums(with_norms=with_norms, slots=slots)
        self._allreduce_device(ctx.dsum_tensor())
        _, n_ok, red = ctx.read_exchange()
        out = []
        for i in range(len(maxima)):
            vals = [red[1 + per * rk + 1 + i] for rk in range(comm.size)
                    if (int(round(red[1 + per * rk])) >> i) & 1]
            out.append(max(vals) if vals else -np.inf)
        return n_ok, int(round(red[0])), out

    def _update_without_exchange(self, df_first, verbose):
        """Damped update after `_exchange` (several ranks).  Every rank forms the same proposal
        Q_prev + df * sum_k dQi from the reduced sums and checks it and its OWN cavities, walking down the
        damping ladder df, df*decay, ... without talking to the others.  Positive definiteness of the global
        matrix and of every cavity is linear in df and holds at df = 0 (the current state), so a rank that
        accepts df also accepts every smaller one: the consensus is the maximum of the local ladder
        positions -- ONE scalar all-reduce per iteration however many retries there were
        (reference method.py:1066-1146 broadcasts per attempt by construction: it is one process).
        Returns (status, df, attempts): status 0 accepted, 1 invalid prior, 2 the ladder ran below
        `df_treshold` somewhere (the caller falls back to the exchanging loop with its forcing branch)."""
        ctx = self._shard.ctx
        BIG = 1 << 30

        def attempt(df):
            ctx.update_partial(df)              # local Qi2 = Qi + df dQi (the cavities of the proposal need them)
            ctx.update_from_sums(df)
            if not ctx.update_finish():
                return -1
            return 1 if ctx.cavity(proposal=True)[1] else 0

        j, df = 0, df_first
        invalid = False
        while True:
            res = attempt(df)
            if res == 1:
                break
            if res == -1 and self.iter == 1:
                invalid = True                  # (the global matrix is the same on every rank: so is this flag)
                break
            df *= self.df_decay
            j += 1
            if verbose:
                sys.stdout.write("\rNon pos. def. {}, reducing df to {:.3}".format(
                    "posterior cov" if res == -1 else "cavity", df) + " " * 5 + "\b" * 5)
                sys.stdout.flush()
            if df < self.df_treshold:
                j = BIG
                break
        if invalid:
            return 1, df, j + 1
        j_all = int(round(self.comm.allreduce_scalar(float(j), 'max')))
        if j_all >= BIG:
            return 2, df_first, 0
        if j_all != j:
            # the damping the ladder reaches at position j_all, bit for bit: the ranks whose own ladder stopped
            # there multiplied by df_decay j_all times (df_first * df_decay ** j_all rounds differently)
            df = df_first
            for _ in range(j_all):
                df *= self.df_decay
            if attempt(df) != 1:
                raise RuntimeError("damping consensus: a smaller damping factor failed where a larger one passed")
        return 0, df, j_all + 1

    def _all_ranks(self, flag):
        if self.comm.size > 1:
            return self.comm.allreduce_scalar(1.0 if flag else 0.0, 'min') > 0.5
        return bool(flag)

    def sync_host(self):
        """Refresh every host mirror (Q, r, Qi, ... workers' Mat/vec) from the device."""
        self._pull_state()

    def cur_approx(self):
        """Current posterior approximation moments ``(S, m)`` (method.py:884-896)."""
        from .util import invert_normal_params
        return invert_normal_params(self.Q, self.r)

    # ---- one batch of tilted distributions -------------------------------------
    def _tilted_all(self, seeds_row, save_last_param):
        """Tilted step for every local site (reference method.py:1005-1023),
        batched: one sampler launch + one moment-matching launch."""
        sh = self._shard
        ctx = sh.ctx
        workers = self.workers[sh.k_begin:sh.k_end]
        for w in workers:
            if w.phase != 1:
                raise RuntimeError('Cavity has to be calculated before tilted.')
        stan_seeds = [int(np.random.RandomState(int(s)).randint(0, MAX_UINT))
                      for s in seeds_row[sh.k_begin:sh.k_end]]
        for w, s in zip(workers, stan_seeds):
            w.stan_params['seed'] = s
        n = workers[0]._nsamp() if workers else 0
        if self.builtin and workers:
            sp = workers[0].stan_params
            modes = set(w._init_mode() for w in workers)
            if len(modes) != 1:
                raise RuntimeError("sites disagree on the initialisation mode")
            mode = modes.pop()
            if mode == _lib.INIT_GIVEN:
                _upload_inits(sh, workers)
            msteps, mrhat, nleap, secs = ctx.tilted_sample(
                stan_seeds, sp['chains'], sp['iter'], sp['warmup'], mode, **workers[0]._sampler_kw())
            for i, w in enumerate(workers):
                w.last_time, w.last_msteps, w.last_mrhat = secs, float(msteps[i]), float(mrhat[i])
                w.last_n_leapfrog = int(nleap[i])
                w._have_prev = True
            self.n_leapfrog_total += int(np.sum(nleap))
            if save_last_param and 'phi' in save_last_param:
                dr = ctx.get_draws(n)
                for i, w in enumerate(workers):
                    w.saved_samp = {'phi': np.asfortranarray(dr[i].T)}
        elif workers:
            # a caller-supplied sampler reads the cavity from the workers' host
            # arrays (data['mu_phi'], data['Omega_phi']): refresh them first
            dd = self.dphi
            self._cavQ[:, :, sh.k_begin:sh.k_end] = ctx.download(
                _lib.CAVQ, np.empty((dd, dd, sh.n_local), order='F'))
            self._cavm[:, sh.k_begin:sh.k_end] = ctx.download(
                _lib.CAVM, np.empty((dd, sh.n_local), order='F'))
            draws = None
            for i, (w, s) in enumerate(zip(workers, stan_seeds)):
                samp = w._host_sample(s, save_last_param)
                if draws is None:
                    n = samp.shape[0]
                    draws = np.empty((len(workers), self.dphi, n))
                draws[i] = samp.T
            ctx.set_draws(draws, n)
        # moment matching, grouped by the estimator each site uses this round
        oks = np.zeros(len(workers), dtype=bool)
        i = 0
        while i < len(workers):
            mode = workers[i]._mode_now()
            j = i
            while j < len(workers) and workers[j]._mode_now() == mode:
                j += 1
            oks[i:j], _ = ctx.moments(n, mode, i, j)
            i = j
        if self.rhat_max is not None and workers:
            # chains that did not mix give unreliable moments: skip the site's update this round
            bad = [i for i, w in enumerate(workers)
                   if oks[i] and not (w.last_mrhat is not None and w.last_mrhat <= self.rhat_max)]
            if bad:
                ctx.fail_sites(bad)
                oks[bad] = False
                if self.builtin:
                    # init_prev would restart the chains where they got stuck: next time these sites
                    # start from Stan's random initialisation instead
                    ctx.reinit_sites(bad)
            self._last_rejected = [sh.k_begin + i for i in bad]
        for w, ok in zip(workers, oks):
            w.nsamp = n
            if w._mode_now() == 'sample' and w.prec_estim_skip > 0:
                w.prec_estim_skip -= 1
            w.phase = 2 if ok else 0
            w.iteration += 1
        return oks

    def _force_pos_def(self, verbose):
        forced, _ = self._shard.ctx.force_pd(self.MIN_EIG_TRESHOLD, self.MIN_EIG)
        if verbose:
            print("Force sites {} pos_def.".format(np.nonzero(forced)[0] + self._shard.k_begin))

    # ---- the EP loop -----------------------------------------------------------
    def run(self, niter, calc_moments=True, save_last_param=None, verbose=True,
            return_analytics=False, seed=None):
        """Run the distributed EP algorithm (reference method.py:899-1247).

        Returns ``info`` alone or a tuple ``(info[, (m_phi_s, cov_phi_s)]
        [, (stimes, msteps, mrhats, othertimes)])`` exactly as the reference.
        """
        if niter < 1:
            if verbose:
                print("Nothing to do here as provided arg. `niter` is {}".format(niter))
            out = [self.INFO_OK]
            if calc_moments:
                out.append((None, None))
            if return_analytics:
                out.append((None, None, None, None))
            return tuple(out) if len(out) > 1 else out[0]

        rng = seed if isinstance(seed, np.random.RandomState) else np.random.RandomState(seed=seed)
        seeds = rng.randint(0, MAX_UINT, size=(niter, self.K))

        sh = self._shard
        ctx, comm = sh.ctx, self.comm
        d = self.dphi
        m_phi_s = np.zeros((niter, d)) if calc_moments else None
        cov_phi_s = np.zeros((niter, d, d)) if calc_moments else None
        stimes = np.zeros(niter)
        msteps = np.zeros(niter)
        mrhats = np.zeros(niter)
        othertimes = np.zeros(niter)

        def result(info):
            if not self.keep_on_device:
                self._pull_state()
            else:
                self._host_stale = True
            out = [info]
            if calc_moments:
                out.append((m_phi_s, cov_phi_s))
            if return_analytics:
                out.append((stimes, msteps, mrhats, othertimes))
            return tuple(out) if len(out) > 1 else out[0]

        if not self.keep_on_device:
            if self._host_stale:
                # an earlier keep_on_device run left newer state on the device: refresh the mirrors
                # first instead of overwriting the device with the stale host copies
                self._pull_state()
            self._push_state(with_cavity=True)
        self.history = dict(df=[], attempts=[], snr=[], n_ok=[], rhat_sites=[], n_fail=[], rejected=[])
        local_workers = self.workers[sh.k_begin:sh.k_end]
        if self.builtin and sh.n_local:
            # moments of the transformed site parameters for mix_pred (the reference saves the samples:
            # method.py:1012-1016 `save_last_param`)
            ctx.set_option('param_stats', 1 if save_last_param else 0)

        for cur_iter in range(niter):
            self.iter += 1
            if verbose:
                print("Iter {} starting. Process tilted distributions".format(self.iter))
            oks = self._tilted_all(seeds[cur_iter], save_last_param)
            n_ok = int(oks.sum())
            n_fail = len(oks) - n_ok

            def lmax(vals):
                # (NaN = a site whose chains could not be initialised: it is a failed site, not a maximum)
                vals = [v for v in vals if v is not None and np.isfinite(v)]
                return max(vals) if vals else None
            maxima = [lmax([w.last_time for w in local_workers]), lmax([w.last_msteps for w in local_workers]),
                      lmax([w.last_mrhat for w in local_workers])]
            exchanged = False
            if comm.size > 1 and hasattr(ctx, 'update_from_sums'):
                # one all-reduce carries the summed site deltas, the counts and the analytics maxima
                n_ok, n_fail, maxima = self._exchange(self.df_select == 'snr', n_fail, maxima)
                exchanged = True
            elif comm.size > 1:
                n_ok = int(round(comm.allreduce_scalar(n_ok, 'sum')))
                n_fail = int(round(comm.allreduce_scalar(n_fail, 'sum')))
                maxima = [comm.allreduce_scalar(-np.inf if v is None else v, 'max') for v in maxima]
            if verbose:
                print("All sites ok" if n_fail == 0 else
                      ("Some sites failed and are not updated" if n_ok else "Every site failed"))
            if n_ok == 0:
                return result(self.INFO_ALL_SITES_FAIL)
            stimes[cur_iter], msteps[cur_iter], mrhats[cur_iter] = [-np.inf if v is None else v for v in maxima]
            # distribution of the per-site max split-Rhat behind that maximum (local shard)
            rh = np.array([w.last_mrhat for w in local_workers if w.last_mrhat is not None], dtype=np.float64)
            rh = rh[np.isfinite(rh)]
            self.history['rejected'].append(list(self._last_rejected))   # (local shard) sites over rhat_max
            self.history['rhat_sites'].append(
                (float(np.median(rh)), float(np.percentile(rh, 90)), float(np.mean(rh > 1.1))) if rh.size
                else (float('nan'),) * 3)
            if verbose:
                print("Sampling done, max sampling time {}".format(stimes[cur_iter]))

            start_othertime = time.time()
            df = self.df0(self.iter)
            if self.df_select == 'snr':
                df = self._select_df(df, exchanged)
            df_first = df
            if verbose:
                print("Iter {}, starting df {:.3g}".format(self.iter, df))
            failed_force_pos_def = False
            attempts = 0
            fast = 2
            if exchanged:
                fast, df_acc, attempts_acc = self._update_without_exchange(df_first, verbose)
                if fast == 1:
                    if verbose:
                        print("\nInvalid prior.")
                    return result(self.INFO_INVALID_PRIOR)
                if fast == 0:
                    ctx.accept()
                    self.history['df'].append(df_acc)
                    self.history['attempts'].append(attempts_acc)
                    self.history['n_ok'].append(n_ok)
                    self.history['n_fail'].append(n_fail)
            while fast == 2:
                attempts += 1
                # Qi2 = Qi + df dQi, Q = Q0 + sum_k Qi2 (method.py:1071-1074); the
                # all-reduce is the only exchange between GPUs
                ctx.update_partial(df)
                self._allreduce_partial()
                ok = ctx.update_finish()
                if ok:
                    ok = self._all_ranks(ctx.cavity(proposal=True)[1])
                    if ok:
                        ctx.accept()
                        self.history['df'].append(df)
                        self.history['attempts'].append(attempts)
                        self.history['n_ok'].append(n_ok)
                        self.history['n_fail'].append(n_fail)
                        break
                    what = "cavity"
                else:
                    what = "posterior cov"
                    if self.iter == 1:
                        if verbose:
                            print("\nInvalid prior.")
                        return result(self.INFO_INVALID_PRIOR)
                df *= self.df_decay
                if verbose:
                    sys.stdout.write("\rNon pos. def. {}, reducing df to {:.3}".format(what, df) + " " * 5 + "\b" * 5)
                    sys.stdout.flush()
                if df < self.df_treshold:
                    if verbose:
                        print("\nDamping factor reached minimum.")
                    df = df_first
                    ctx.update_partial(df)          # Qi2 = Qi + df0 dQi  (method.py:1105-1107)
                    if failed_force_pos_def:
                        if verbose:
                            print("Failed to force pos_def.")
                        return result(self.INFO_DF_TRESHOLD_REACHED_CAVITY)
                    failed_force_pos_def = True
                    self._force_pos_def(verbose)

            if calc_moments:
                ctx.global_moments(self.m, self.S)
                m_phi_s[cur_iter] = self.m
                cov_phi_s[cur_iter] = self.S.T
                if verbose:
                    print("Mean and std of phi[0]: {:.3}, {:.3}".format(
                        m_phi_s[cur_iter, 0], np.sqrt(cov_phi_s[cur_iter, 0, 0])))
            for w in local_workers:
                w.phase = 1
            othertimes[cur_iter] = time.time() - start_othertime
            if verbose:
                print("Iter {} done.".format(self.iter))

        if verbose:
            print("{} iterations done\nTotal limiting sampling time: {}".format(niter, stimes.sum()))
        res = result(self.INFO_OK)
        for w in self.workers:
            w.Q, w.r = self.Q, self.r
        return res

    def mix_phi(self, out_S=None, out_m=None):
        """Posterior approximation of phi by pooling the last tilted draws of every site
        (reference method.py:1250-1301; there the method is unreachable because `saved_samp` is never
        filled -- here the draws of the last `run()` are still in the device draw buffer, so no
        `save_last_param` is needed).  Returns ``(S, m)``: the pooled covariance and mean."""
        if self.iter == 0:
            raise RuntimeError("Can not mix samples before at least one iteration has been done.")
        d, K = self.dphi, self.K
        workers = self.workers[self._shard.k_begin:self._shard.k_end]
        n = workers[0].nsamp if workers else None
        if n is None:
            raise RuntimeError("No samples to mix")
        sums = self._shard.ctx.mix_phi_sums(n)
        if self.comm.size > 1:
            sums = self.comm.allreduce_array(sums)
        sm = sums[:d]
        sS = sums[d:d + d * d].reshape(d, d, order='F')
        sMM = sums[d + d * d:].reshape(d, d, order='F')
        m = sm / K
        S = (sS + n * (sMM - K * np.outer(m, m))) / (K * n - 1)
        if out_m is None:
            out_m = np.zeros(d)
        if out_S is None:
            out_S = np.zeros((d, d), order='F')
        out_m[...] = m
        out_S[...] = S
        return out_S, out_m

    # ---- parameter slots of the built-in models in a site's sampled vector q = [phi | eta | etb] ----
    def _param_slots(self, k, par):
        """(first slot, shape) of transformed parameter `par` of site k (see epg_get_param_stats)."""
        w = self.workers[k]
        fam = self.site_model.family
        D = w.X.shape[1]
        J = 1 if self.site_model.single_group else int(w.A['J'])
        d = self.dphi
        if par == 'phi':
            return 0, (d,)
        if par == 'alpha':
            return d, (J,)
        if par == 'beta':
            if fam == 'm1b':
                return 1, (D,)
            if fam == 'm2b':
                return d + J, (D,)
            return d + J, (J, D)
        raise ValueError("built-in models provide 'phi', 'alpha' and 'beta' (got {})".format(repr(par)))

    def mix_pred(self, params, smap=None, param_shapes=None):
        """Mean and variance of site parameters by pooling the last tilted draws of every site
        (reference method.py:1304-1478; unreachable there, `workers[k].fit` is never assigned).

        For the built-in models the sampler accumulates the moments of the transformed parameters
        ``'alpha'`` and ``'beta'`` (and ``'phi'``) on the device when the last ``run`` was given
        ``save_last_param``; `params`, `smap`, `param_shapes` and the pooling rules are the reference's:
        ``smap[k]`` maps the indices of site k's parameter to the global one (None: every site
        contributes to the whole parameter)."""
        if self.iter == 0:
            raise RuntimeError("Can not mix samples before at least one iteration has been done.")
        if not self.builtin:
            raise NotImplementedError("mix_pred needs the built-in sampler's parameter statistics")
        if isinstance(params, str):
            only_one_param = True
            params, smap, param_shapes = [params], [smap], [param_shapes]
        else:
            only_one_param = False
        sh = self._shard
        try:
            mean_l, ssd_l = sh.ctx.param_stats(0, sh.n_local)
        except Exception as e:
            raise RuntimeError("No parameter statistics: call run(..., save_last_param=[...]) first ({})".format(e))
        if self.comm.size > 1:
            mean_all = self.comm.allgather_sites(mean_l.T, self.K, 1).T
            ssd_all = self.comm.allgather_sites(ssd_l.T, self.K, 1).T
        else:
            mean_all, ssd_all = mean_l, ssd_l
        K = self.K
        ns = np.array([w.nsamp for w in self.workers], dtype=np.int64)
        ms_all, vs_all = [], []
        for par in params:
            ms, vs = [], []
            for k in range(K):
                o, shp = self._param_slots(k, par)
                cnt = int(np.prod(shp))
                ms.append(mean_all[k, o:o + cnt].reshape(shp))
                vs.append(ssd_all[k, o:o + cnt].reshape(shp))          # sum of squared deviations
            ms_all.append(ms)
            vs_all.append(vs)
        mean, var = pool_site_moments(ns, ms_all, vs_all, smap, param_shapes)
        if only_one_param:
            return mean[0], var[0]
        return mean, var


def pool_site_moments(ns, ms_all, vs_all, smap, param_shapes):
    """The pooling rules of the reference's `Master.mix_pred` (method.py:1375-1471) on per-site moments:
    ns[k] draws, ms_all[ip][k] the mean and vs_all[ip][k] the sum of squared deviations of parameter ip in
    site k; smap[ip] None (every site contributes to the whole parameter) or a per-site index into the
    global parameter of shape param_shapes[ip]."""
    K = len(ns)
    mean, var = [], []
    for ip in range(len(ms_all)):
        ms, vs = ms_all[ip], vs_all[ip]
        sit = smap[ip] if smap is not None else None
        if sit is None:
            ms_a, vs_a = np.array(ms), np.array(vs)
            n = ns.sum()
            mc = (ms_a.T * ns).T.sum(axis=0) / n
            vc = ((((ms_a - mc) ** 2).T * ns).T + vs_a).sum(axis=0) / (n - 1)
        else:
            par_shape = param_shapes[ip]
            count = np.zeros(par_shape)
            for k in range(K):
                count[sit[k]] += 1
            if np.count_nonzero(count) != count.size:
                raise ValueError("Arg. `smap` does not fill the parameter")
            onecont = count == 1
            mc = np.zeros(par_shape)
            vc = np.zeros(par_shape)
            if np.all(onecont):
                for k in range(K):
                    mc[sit[k]] = ms[k]
                    vc[sit[k]] = vs[k] / (ns[k] - 1)
            else:
                nc = np.zeros(par_shape, dtype=np.int64)
                for k in range(K):
                    nc[sit[k]] += ns[k]
                    mc[sit[k]] += ns[k] * ms[k]
                mc /= nc
                for k in range(K):
                    vc[sit[k]] += ns[k] * (np.asarray(ms[k] - mc[sit[k]]) ** 2) + vs[k]
                vc /= (nc - 1)
                if np.any(onecont):
                    # (method.py:1464-1469: as soon as one index has a single contribution the reference
                    #  re-assigns every site's own moments in site order; kept as it is)
                    for k in range(K):
                        mc[sit[k]] = ms[k]
                        vc[sit[k]] = vs[k] / (ns[k] - 1)
        mean.append(mc)
        var.append(vc)
    return mean, var

"""Utilities of the EP path, B200 edition.

Mirrors the public surface of the reference's ``epstan/util.py`` (``__all__``
at util.py:15-19) for the functions on the EP path.  The numerical ones run on
the GPU through libepgpu (there is no CPU fallback); the host-side ones
(``distribute_groups``, fit readers, ``load_stan``) stay in Python as the
reference's do (SURVEY 8a row a14).
"""

import itertools
import os

import numpy as np

from . import _lib

__all__ = [
    'invert_normal_params', 'olse', 'cv_moments', 'copy_fit_samples',
    'get_last_fit_sample', 'load_stan', 'distribute_groups', 'LinAlgError',
]

from numpy.linalg import LinAlgError   # the reference raises scipy's, which is this class

_ctx = None


def default_context():
    """Process-wide context for the stand-alone utilities (device from
    EPGPU_DEVICE / LOCAL_RANK, default 0)."""
    global _ctx
    if _ctx is None:
        dev = int(os.environ.get('EPGPU_DEVICE', os.environ.get('LOCAL_RANK', 0)))
        _ctx = _lib.Context(dev)
    return _ctx


def _resolve_out(arr, out, order=None):
    """Reference convention: None -> new array, 'in-place' -> the input."""
    if not isinstance(out, np.ndarray) and out == 'in-place':
        return arr
    if out is None:
        return None
    return out


def invert_normal_params(A, b=None, out_A=None, out_b=None, cho_form=False):
    """Invert moment parameters into natural parameters or vice versa.

    Same contract as reference util.py:51-125: returns ``(out_A, out_b)`` with
    ``out_A`` the full symmetric inverse (F-order), ``out_b = A^-1 b`` or None;
    ``out_*`` may be None (new array), an ndarray, or ``'in-place'``;
    ``cho_form=True`` means ``A`` holds the upper Cholesky factor.  Raises
    ``LinAlgError`` if ``A`` is not positive definite.
    """
    A = np.asarray(A)
    if A.ndim != 2 or A.shape[0] != A.shape[1]:
        raise ValueError('Provided array A is inappropriate')
    d = A.shape[0]
    # for cho_form the factor is the *upper* triangle of A in matrix terms
    Ainv, binv, ok = default_context().invert_normal_params(
        np.ascontiguousarray(A, dtype=np.float64)[None],
        None if b is None else np.ascontiguousarray(b, dtype=np.float64)[None],
        cho_form=cho_form)
    if not ok[0]:
        raise LinAlgError("matrix is not positive definite")
    res_A = _resolve_out(A, out_A)
    if res_A is None:
        res_A = np.empty((d, d), order='F')
    np.copyto(res_A, Ainv[0])
    if not res_A.flags['FARRAY']:
        res_A = res_A.T            # symmetric: same values, F-order view (util.py:95-99)
    res_b = None
    if b is not None:
        res_b = _resolve_out(b, out_b)
        if res_b is None:
            res_b = np.empty(d)
        np.copyto(res_b, binv[0])
    return res_A, res_b


def olse(S, n, P=None, out=None):
    """Optimal linear shrinkage precision estimator (reference util.py:128-194).

    ``P`` None uses the naive prior 1/d I.  ``out``: None, ndarray or 'in-place'.
    """
    S = np.asarray(S)
    d = S.shape[0]
    res, ok = default_context().olse(
        np.ascontiguousarray(S, dtype=np.float64)[None], n,
        None if P is None else np.ascontiguousarray(P, dtype=np.float64)[None])
    if not ok[0]:
        raise LinAlgError("matrix is not positive definite")
    dst = _resolve_out(S, out)
    if dst is None:
        dst = np.empty((d, d), order='F')
    np.copyto(dst, res[0])
    if not dst.flags['FARRAY']:
        dst = dst.T
    return dst


def cv_moments(samp, lp, Q_tilde, r_tilde, S_tilde=None, m_tilde=None,
               ldet_Q_tilde=None, multiple_cv=True, regulate_a=None, max_a=None,
               m_treshold=0.9, S_hat=None, m_hat=None, ret_a=False):
    """Approximate moments using a Gaussian control variate (reference
    util.py:245-411).  ``lp`` must be normalised.  ``S_tilde``, ``m_tilde`` and
    ``ldet_Q_tilde`` are accepted for signature compatibility and recomputed on
    the device from ``(Q_tilde, r_tilde)``.

    Returns ``(S_hat, m_hat, treshold_exceeded)`` and, with ``ret_a``, the
    coefficient arrays ``a_S, a_m`` (0, 0 when the plain estimates were returned).
    """
    samp = np.asarray(samp, dtype=np.float64)
    if samp.ndim == 1:
        samp = samp[:, None]
    n, d = samp.shape
    res = default_context().cv_moments(
        np.ascontiguousarray(samp.T)[None], np.asarray(lp, dtype=np.float64)[None],
        np.asarray(Q_tilde, dtype=np.float64)[None], np.asarray(r_tilde, dtype=np.float64)[None],
        multiple_cv=multiple_cv, regulate_a=regulate_a, max_a=max_a, m_treshold=m_treshold, ret_a=ret_a)
    S, m, used = res[:3]
    if used[0] < 0:
        raise LinAlgError("control variate system is singular or Q_tilde not positive definite")
    if S_hat is None:
        S_hat = np.empty((d, d), order='F')
    if m_hat is None:
        m_hat = np.empty(d)
    np.copyto(S_hat, S[0])
    np.copyto(m_hat, m[0])
    if ret_a:
        if not used[0]:
            return S_hat, m_hat, False, 0, 0
        return S_hat, m_hat, True, res[3][0], res[4][0]
    return S_hat, m_hat, bool(used[0])


# ---------------------------------------------------------------------------
# readers for PyStan-style fit objects (used when the caller supplies its own
# sampler object instead of a built-in model name)
# ---------------------------------------------------------------------------

def copy_fit_samples(fit, param_name, out=None):
    """Post-warm-up draws of one parameter of a PyStan-2-style fit as an
    F-order array (nsamp, *dims), chains stacked (reference util.py:414-486)."""
    dims = tuple(fit.par_dims[fit.model_pars.index(param_name)])
    sim = fit.sim
    nchains = sim['chains']
    warmup = sim['warmup2'][0]
    per_chain = len(sim['samples'][0]['chains']['lp__']) - warmup
    shape = (nchains * per_chain,) + dims
    if out is None:
        out = np.empty(shape, order='F')
    elif out.shape != shape or not out.flags.farray:
        raise ValueError('Invalid output array')
    if dims:
        index_sets = (tuple(reversed(ix)) for ix in itertools.product(*(range(n) for n in reversed(dims))))
    else:
        index_sets = ((),)
    for ix in index_sets:
        name = '{}[{}]'.format(param_name, ','.join(str(i) for i in ix)) if ix else param_name
        for c in range(nchains):
            rows = slice(c * per_chain, (c + 1) * per_chain)
            out[(rows,) + ix] = sim['samples'][c]['chains'][name][warmup:]
    return out


def get_last_fit_sample(fit, out=None):
    """Last draw of every chain as a list of {param: ndarray} dicts, the form
    ``StanModel.sampling(init=...)`` accepts (reference util.py:489-537)."""
    nchains = fit.sim['chains']
    if out is None:
        out = [{p: np.empty(tuple(dims), order='F') for p, dims in zip(fit.model_pars, fit.par_dims)}
               for _ in range(nchains)]
    for c in range(nchains):
        chains = fit.sim['samples'][c]['chains']
        for p, dims in zip(fit.model_pars, fit.par_dims):
            if not dims:
                out[c][p][()] = chains[p][-1]
                continue
            for ix in np.ndindex(*dims):
                out[c][p][ix] = chains['{}[{}]'.format(p, ','.join(str(i) for i in ix))][-1]
    return out


# ---------------------------------------------------------------------------
# host-side helpers
# ---------------------------------------------------------------------------

BUILTIN_MODELS = ('m1b', 'm2b', 'm3b', 'm4b', 'm5b')


class BuiltinModel(object):
    """What ``load_stan`` returns here: a handle on a built-in CUDA density.

    The reference compiles ``<name>.stan`` with PyStan (util.py:642-689); the
    GPU build has no Stan compiler, so the file's base name selects one of the
    hand-written tilted densities (SURVEY 8b)."""

    def __init__(self, name):
        base = name[:-3] if name.endswith('_sg') else name
        if base not in BUILTIN_MODELS:
            raise ValueError("no built-in CUDA density for model '{}' (available: {} and their _sg variants)"
                             .format(name, ', '.join(BUILTIN_MODELS)))
        self.name = name
        self.family = base
        self.single_group = name.endswith('_sg')
        self.model_id = _lib.MODEL_IDS[base]

    def dphi(self, D):
        return {'m1b': D + 1, 'm2b': 2, 'm3b': D + 1, 'm4b': 2 * D + 2, 'm5b': 2 * D + 2}[self.family]

    def __repr__(self):
        return "BuiltinModel('{}')".format(self.name)


def load_stan(filename, overwrite=False):
    """Resolve a model path / name (with or without '.stan' / '.pkl') to a
    built-in CUDA density (reference util.py:642-689 loads or compiles Stan)."""
    for ext in ('.pkl', '.stan'):
        if filename.endswith(ext):
            filename = filename[:-len(ext)]
    return BuiltinModel(os.path.basename(filename))


def _init_dict(init, c):
    """the init dict of chain c: PyStan calls a function as init(chain_id=c) if it takes that argument"""
    if callable(init):
        import inspect
        try:
            params = inspect.signature(init).parameters
        except (TypeError, ValueError):
            params = {}
        return init(chain_id=c) if 'chain_id' in params else init()
    if isinstance(init, dict):
        return init
    return init[c]


def init_values(init, chains, sites, Pmax=None):
    """Starting points of the built-in sampler for PyStan's ``init`` = dict, list of ``chains`` dicts or a
    function returning a dict, as the array ``[len(sites)][chains][Pmax]`` that ``Context.set_inits`` takes.

    ``sites`` holds ``(family, D, J)`` per site (family: 'm1b' ... 'm5b'); Pmax None: the largest number of
    parameters of these sites (Context.set_inits pads to its own).  A site's row is laid out as the
    sampler's parameter vector ``q = [phi (d) | eta (J) | etb]`` with ``etb`` (J, D) row-major for m3b, m4b and
    m5b, (D,) for m2b and absent for m1b; a single-group site (J = 1) also takes ``eta`` as a scalar and
    ``etb`` as (D,).  A parameter missing from the dict is NaN (drawn at random by the sampler), unknown names
    are ignored as Stan ignores them, and a value of the wrong shape raises ``ValueError``.
    """
    if isinstance(init, (list, tuple)):
        if len(init) != chains:
            raise ValueError("init: a list of {} dicts for {} chains".format(len(init), chains))
    elif not (isinstance(init, dict) or callable(init)):
        raise ValueError("init must be 'random', '0', a dict, a list of dicts or a function returning a dict")
    dicts = [_init_dict(init, c) for c in range(chains)]
    for c, dc in enumerate(dicts):
        if not isinstance(dc, dict):
            raise ValueError("init of chain {} is not a dict".format(c))
    layouts = []
    for family, D, J in sites:
        d = {'m1b': D + 1, 'm2b': 2, 'm3b': D + 1, 'm4b': 2 * D + 2, 'm5b': 2 * D + 2}[family]
        layout = [('phi', (d,)), ('eta', (J,))]
        if family == 'm2b':
            layout.append(('etb', (D,)))
        elif family != 'm1b':
            layout.append(('etb', (J, D)))
        layouts.append(layout)
    n_par = [sum(int(np.prod(shp)) for _, shp in layout) for layout in layouts]
    if Pmax is None:
        Pmax = max(n_par)
    elif max(n_par) > Pmax:
        raise ValueError("init: a site has more parameters ({}) than Pmax = {}".format(max(n_par), Pmax))
    out = np.full((len(sites), chains, Pmax), np.nan)
    for k, ((family, D, J), layout) in enumerate(zip(sites, layouts)):
        for c, dc in enumerate(dicts):
            off = 0
            for name, shp in layout:
                size = int(np.prod(shp))
                if name in dc:
                    v = np.asarray(dc[name], dtype=np.float64)
                    grouped = name == 'eta' or (name == 'etb' and family != 'm2b')
                    if v.shape != shp and not (J == 1 and grouped and v.shape == shp[1:]):
                        raise ValueError("init: site {}, parameter '{}': shape {}, expected {}"
                                         .format(k, name, v.shape, shp))
                    out[k, c, off:off + size] = v.ravel()
                off += size
    return out


def distribute_groups(J, K, Nj):
    """Distribute J groups to K sites (reference util.py:540-639).

    Returns ``(Nk, Nj_k, j_ind_k)`` for K < J (adjacent groups are merged,
    always the pair with the smallest combined size, first on ties),
    ``(Nj, None, None)`` for K == J and ``(Nk, parts_per_group, None)`` for
    J < K <= N (largest groups are split).
    """
    if isinstance(Nj, (int, np.integer)):
        Nj = np.full(J, int(Nj), dtype=np.int64)
    else:
        Nj = np.asarray(Nj)
        if Nj.ndim != 1 or Nj.shape[0] != J:
            raise ValueError("Invalid shape of arg. `Nj`.")
    if np.any(Nj <= 0):
        raise ValueError("Every group must have at least one item")
    N = int(Nj.sum())
    if K < 2:
        raise ValueError("K should be at least 2.")
    if K == J:
        return Nj, None, None
    if K < J:
        sizes = [int(v) for v in Nj]
        count = [1] * J
        while len(sizes) > K:
            best, best_i = None, 0
            for i in range(len(sizes) - 1):
                s = sizes[i] + sizes[i + 1]
                if best is None or s < best:
                    best, best_i = s, i
            sizes[best_i:best_i + 2] = [best]
            count[best_i:best_i + 2] = [count[best_i] + count[best_i + 1]]
        j_ind_k = np.empty(N, dtype=np.int32)
        row = 0
        grp = 0
        for c in count:
            for ji in range(c):
                j_ind_k[row:row + Nj[grp]] = ji
                row += int(Nj[grp])
                grp += 1
        return np.array(sizes), np.array(count), j_ind_k
    if K <= N:
        parts = np.ones(J, dtype=np.int64)
        cur = Nj.astype(np.float64)
        for _ in range(K - J):
            j = int(cur.argmax())
            parts[j] += 1
            cur[j] = Nj[j] / parts[j]
        base, rem = Nj // parts, Nj % parts
        Nk = np.concatenate([np.where(np.arange(parts[j]) < rem[j], base[j] + 1, base[j]) for j in range(J)])
        return Nk.astype(np.int64), parts, None
    raise ValueError("K cant be greater than number of samples")

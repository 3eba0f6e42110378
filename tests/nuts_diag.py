"""fp64 NumPy restatement of the per-transition sampler parameters of Stan 2.17's NUTS, beside the oracles of
oracle/nuts.py and tests/nuts_control.py.

TEST INFRASTRUCTURE ONLY.  oracle/nuts.py stays as it is; this module restates its transition so that it also
returns what PyStan's `get_sampler_params()` reports for it (base_nuts::transition):

  * accept_stat__  sum_metro / n_leapfrog of the transition (before dual averaging clamps it);
  * stepsize__     the step size of the transition (jitter applied);
  * treedepth__    the number of valid subtrees merged;
  * n_leapfrog__   leapfrog steps, including those of a discarded subtree;
  * divergent__    1 when a leaf had H - H0 > 1000;
  * energy__       H(q, p) of the selected sample, its momentum included;

and the summary PyStan's check_hmc_diagnostics draws from them (divergences, transitions at max_treedepth,
E-BFMI per chain) over the saved post-warm-up transitions.
"""
import numpy as np

from oracle import nuts
import nuts_control

FIELDS = ('accept_stat__', 'stepsize__', 'treedepth__', 'n_leapfrog__', 'divergent__', 'energy__')


class _Recording(nuts.NUTS):
    """oracle.nuts.NUTS.transition, restated to keep the selected sample's momentum and record the transition"""

    def transition(self, q, V, g):
        p = self._sample_p()
        z0 = (q, p, V, g)
        H0 = self._H(V, p)
        z_minus = z_plus = z_sample = z0
        rho = p.copy()
        lsw = 0.0
        depth = 0
        st = {'n_leapfrog': 0, 'sum_metro': 0.0, 'divergent': False}
        while depth < self.max_depth:
            if self.rng.uniform() > 0.5:
                ok, z_plus, prop, rho_sub, lsw_sub, _, _ = self._build(depth, z_plus, 1, H0, st)
            else:
                ok, z_minus, prop, rho_sub, lsw_sub, _, _ = self._build(depth, z_minus, -1, H0, st)
            if not ok:
                break
            depth += 1
            if lsw_sub > lsw or self.rng.uniform() < np.exp(lsw_sub - lsw):
                z_sample = prop
            lsw = np.logaddexp(lsw, lsw_sub)
            rho = rho + rho_sub
            if not self._criterion(self.minv * z_minus[1], self.minv * z_plus[1], rho):
                break
        accept = st['sum_metro'] / max(st['n_leapfrog'], 1)
        self.H0 = H0
        self.record = (accept, self.eps, depth, st['n_leapfrog'], 1.0 if st['divergent'] else 0.0,
                       self._H(z_sample[2], z_sample[1]))
        return z_sample[0], z_sample[2], z_sample[3], accept, st


class DiagNUTS(nuts_control.ControlNUTS, _Recording):
    """the recording transition with step-size jitter (ControlNUTS wraps _Recording.transition)"""


def ebfmi(energy):
    """PyStan's check_energy ratio: sum (E_t - E_t-1)^2 / sum (E_t - mean E)^2; NaN below 2 draws or at zero
    variance"""
    e = np.asarray(energy, dtype=np.float64)
    if e.size < 2:
        return float('nan')
    var = np.sum((e - e.mean()) ** 2)
    return float(np.sum(np.diff(e) ** 2) / var) if var > 0 else float('nan')


def sample_chain(lp_grad, dim, n_iter, n_warmup, rng, stepsize=1.0, jitter=0.0, adapt_engaged=True, thin=1,
                 max_depth=10, q0=None):
    """One chain with Stan's default adaptation (or none).  Returns dict(records [n_rec, 6] of every transition
    Stan saves with save_warmup (warm-up first), n_warm (warm-up records), draws, n_divergent, n_max_treedepth,
    ebfmi (the last three over the saved post-warm-up transitions), H0 [n_iter] (the Hamiltonian each transition
    started from))."""
    s = DiagNUTS(lp_grad, dim, rng, max_depth, jitter)
    while True:
        q = rng.uniform(-2, 2, size=dim) if q0 is None else np.array(q0, dtype=np.float64)
        V, g = s._vg(q)
        if np.isfinite(V) and np.all(np.isfinite(g)):
            break
    s.eps = stepsize
    if adapt_engaged:
        da = nuts.DualAveraging()
        da.mu = np.log(10 * stepsize)
        win = nuts.VarWindows(n_warmup, dim)
        s.init_stepsize(q, V, g)
    warm, post, draws, h0 = [], [], [], []
    for it in range(n_iter):
        q, V, g, accept, st = s.transition(q, V, g)
        h0.append(s.H0)
        if it < n_warmup:
            if it % thin == 0:
                warm.append(s.record)
            if not adapt_engaged:
                continue
            s.eps = da.learn(accept)
            new_minv = win.learn(q)
            if new_minv is not None:
                s.minv = new_minv
                s.init_stepsize(q, V, g)
                da.mu = np.log(10 * s.eps)
                da.restart()
            if it == n_warmup - 1:
                s.eps = da.final()
        elif (it - n_warmup) % thin == 0:
            post.append(s.record)
            draws.append(q)
    rec = np.array(warm + post, dtype=np.float64).reshape(-1, len(FIELDS))
    saved = rec[len(warm):]
    return dict(records=rec, n_warm=len(warm), draws=np.array(draws).reshape(-1, dim),
                n_divergent=int(np.sum(saved[:, 4])), n_max_treedepth=int(np.sum(saved[:, 2] >= max_depth)),
                ebfmi=ebfmi(saved[:, 5]), H0=np.array(h0))


def sample(lp_grad, dim, chains, n_iter, n_warmup=None, seed=0, **kw):
    """`chains` independent chains of sample_chain"""
    if n_warmup is None:
        n_warmup = n_iter // 2
    return [sample_chain(lp_grad, dim, n_iter, n_warmup, np.random.RandomState([seed, c]), **kw)
            for c in range(chains)]

"""fp64 NumPy restatement of Stan 2.17's dense_e and unit_e NUTS, beside the diag_e oracle (oracle/nuts.py).

TEST INFRASTRUCTURE ONLY.  oracle/nuts.py stays as it is, so that the cached diag_e references keep their
meaning; this module subclasses its sampler and swaps the Hamiltonian pieces for the chosen metric:

  * dense_e (stan/mcmc/hmc/hamiltonians/dense_e_metric.hpp): Sigma = U'U, momentum p = U^-1 z, kinetic
    energy p'Sigma p / 2, dtau/dp = Sigma p (position update and p_sharp of the U-turn criterion);
    covariance windows (stan/mcmc/covar_adaptation.hpp) on the variance-window schedule:
    Sigma = n/(n+5) C + 1e-3 5/(n+5) I from the window's sample covariance C;
  * unit_e (adapt_unit_e_nuts.hpp): Sigma = I, step-size dual averaging only.
"""
import numpy as np
from scipy.linalg import solve_triangular

from oracle import nuts

METRICS = ('diag_e', 'dense_e', 'unit_e')


class CovarWindows(nuts.VarWindows):
    def __init__(self, num_warmup, dim):
        super().__init__(num_warmup, dim)
        self.m2 = np.zeros((dim, dim))

    def learn(self, q):
        """returns the new inverse metric (p x p) at the end of a window, else None"""
        out = None
        if self.enabled:
            in_window = (self.init_buffer <= self.counter < self.num_warmup - self.term_buffer
                         and self.counter != self.num_warmup)
            if in_window:
                self.n += 1
                delta = q - self.mean
                self.mean += delta / self.n
                self.m2 += np.outer(q - self.mean, delta)
            if self.counter == self.next_window and self.counter != self.num_warmup:
                self._compute_next_window()
                n = float(self.n)
                covar = self.m2 / (n - 1.0)
                covar = np.tril(covar) + np.tril(covar, -1).T          # (Stan's LLT reads the lower triangle)
                out = (n / (n + 5.0)) * covar + 1e-3 * (5.0 / (n + 5.0)) * np.eye(len(q))
                self.n = 0
                self.mean[:] = 0.0
                self.m2[:] = 0.0
        self.counter += 1
        return out


class MetricNUTS(nuts.NUTS):
    """One chain of oracle NUTS with metric 'diag_e', 'dense_e' or 'unit_e'."""

    def __init__(self, lp_grad, dim, rng, max_depth=10, metric='diag_e'):
        super().__init__(lp_grad, dim, rng, max_depth)
        if metric not in METRICS:
            raise ValueError(metric)
        self.metric = metric
        self.set_sigma(np.eye(dim))

    def set_sigma(self, S):
        self.Sigma = np.array(S, dtype=np.float64)
        U = np.linalg.cholesky(self.Sigma).T
        self.Uinv = solve_triangular(U, np.eye(self.dim), lower=False)
        self.minv = np.diag(self.Sigma).copy()

    def _dtau(self, p):
        return self.Sigma @ p if self.metric == 'dense_e' else self.minv * p

    def _H(self, V, p):
        h = V + 0.5 * np.dot(p, self._dtau(p))
        return np.inf if np.isnan(h) else h

    def _leapfrog(self, z, eps):
        q, p, V, g = z
        p = p - 0.5 * eps * g
        q = q + eps * self._dtau(p)
        V, g = self._vg(q)
        p = p - 0.5 * eps * g
        return (q, p, V, g)

    def _sample_p(self):
        z = self.rng.standard_normal(self.dim)
        return self.Uinv @ z if self.metric == 'dense_e' else z / np.sqrt(self.minv)

    def _build(self, depth, z, sign, H0, st):
        if depth == 0:
            z = self._leapfrog(z, sign * self.eps)
            st['n_leapfrog'] += 1
            h = self._H(z[2], z[1])
            dH = H0 - h
            st['sum_metro'] += 1.0 if dH > 0 else np.exp(dH)
            if -dH > nuts.MAX_DELTA_H:
                st['divergent'] = True
                return False, z, z, z[1], dH, None, None
            ps = self._dtau(z[1])
            return True, z, z, z[1].copy(), dH, ps, ps
        ok, z, prop_l, rho_l, lsw_l, psl, _ = self._build(depth - 1, z, sign, H0, st)
        if not ok:
            return False, z, prop_l, rho_l, lsw_l, None, None
        ok, z, prop_r, rho_r, lsw_r, _, psr = self._build(depth - 1, z, sign, H0, st)
        if not ok:
            return False, z, prop_l, rho_l, lsw_l, None, None
        lsw = np.logaddexp(lsw_l, lsw_r)
        prop = prop_r if (lsw_r > lsw or self.rng.uniform() < np.exp(lsw_r - lsw)) else prop_l
        rho = rho_l + rho_r
        return self._criterion(psl, psr, rho), z, prop, rho, lsw, psl, psr

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
            if not self._criterion(self._dtau(z_minus[1]), self._dtau(z_plus[1]), rho):
                break
        accept = st['sum_metro'] / max(st['n_leapfrog'], 1)
        return z_sample[0], z_sample[2], z_sample[3], accept, st


def sample_chain(lp_grad, dim, n_iter, n_warmup, rng, metric='diag_e', q0=None, delta=0.8, max_depth=10):
    """Adaptive NUTS run with the given metric.  Returns dict(draws, stepsize, n_grad, last, Sigma, n_divergent)."""
    s = MetricNUTS(lp_grad, dim, rng, max_depth, metric)
    tries = 0
    while True:
        q = rng.uniform(-2, 2, size=dim) if q0 is None else np.array(q0, dtype=np.float64)
        V, g = s._vg(q)
        if np.isfinite(V) and np.all(np.isfinite(g)):
            break
        tries += 1
        if q0 is not None or tries > 100:
            raise RuntimeError("initialisation failed")
    da = nuts.DualAveraging(delta=delta)
    win = None if metric == 'unit_e' else (CovarWindows if metric == 'dense_e' else nuts.VarWindows)(n_warmup, dim)
    s.init_stepsize(q, V, g)
    draws = np.empty((n_iter - n_warmup, dim))
    eps_used = []
    n_div = 0
    for it in range(n_iter):
        q, V, g, accept, st = s.transition(q, V, g)
        n_div += st['divergent'] and it >= n_warmup
        if it < n_warmup:
            s.eps = da.learn(accept)
            new = win.learn(q) if win is not None else None
            if new is not None:
                s.set_sigma(new if metric == 'dense_e' else np.diag(new))
                s.init_stepsize(q, V, g)
                da.mu = np.log(10 * s.eps)
                da.restart()
            if it == n_warmup - 1:
                s.eps = da.final()
        else:
            draws[it - n_warmup] = q
            eps_used.append(s.eps)
    return dict(draws=draws, stepsize=float(np.mean(eps_used)) if eps_used else s.eps,
                n_grad=s.n_grad, last=q, Sigma=s.Sigma.copy(), n_divergent=n_div)


def sample(lp_grad, dim, chains, n_iter, n_warmup=None, seed=0, metric='diag_e', **kw):
    """`chains` independent chains (as oracle.nuts.sample) with the given metric."""
    if n_warmup is None:
        n_warmup = n_iter // 2
    res = [sample_chain(lp_grad, dim, n_iter, n_warmup, np.random.RandomState([seed, c]), metric=metric, **kw)
           for c in range(chains)]
    return dict(draws=np.concatenate([r['draws'] for r in res], axis=0),
                per_chain=[r['draws'] for r in res],
                stepsize=float(np.mean([r['stepsize'] for r in res])),
                n_grad=sum(r['n_grad'] for r in res), Sigma=[r['Sigma'] for r in res],
                n_divergent=sum(r['n_divergent'] for r in res))

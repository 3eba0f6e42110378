"""fp64 NumPy restatement of Stan 2.17's remaining NUTS sampling settings, beside the diag_e oracle (oracle/nuts.py).

TEST INFRASTRUCTURE ONLY.  oracle/nuts.py stays as it is, so that the cached diag_e references keep their
meaning; this module reuses its sampler and adds what PyStan's `sampling(thin=, init=, init_r=, control=)` sets:

  * the window schedule (windowed_adaptation::set_window_params, compute_next_window) with any
    (init buffer, term buffer, window);
  * the dual-averaging constants gamma / kappa / t0 and the starting step size (mu = log(10 stepsize), set
    before the step-size heuristic);
  * step-size jitter (base_hmc::sample_stepsize): eps = eps_nom (1 + j (2u - 1)) at the start of every
    transition, adaptation on eps_nom, stepsize__ = the eps used;
  * adaptation off (run_sampler): no heuristic, no dual averaging, no windows, unit metric;
  * thinning (generate_transitions): post-warm-up transition m is saved when m % thin == 0;
  * given inits with NaN entries drawn U(-init_r, init_r), one attempt when nothing is random.
"""
import numpy as np

from oracle import nuts


class Windows(nuts.VarWindows):
    """diag_e variance windows with Stan's (init_buffer, term_buffer, window) arguments"""

    def __init__(self, num_warmup, dim, init_buffer=75, term_buffer=50, window=25):
        self.num_warmup = num_warmup
        self.init_buffer, self.term_buffer, self.base_window = init_buffer, term_buffer, window
        self.enabled = num_warmup >= 20
        if self.enabled and init_buffer + window + term_buffer > num_warmup:
            self.init_buffer = int(0.15 * num_warmup)
            self.term_buffer = int(0.1 * num_warmup)
            self.base_window = num_warmup - (self.init_buffer + self.term_buffer)
        self.counter = 0
        self.window_size = self.base_window
        self.next_window = self.init_buffer + self.base_window - 1
        self.n = 0
        self.mean = np.zeros(dim)
        self.m2 = np.zeros(dim)


def window_ends(num_warmup, init_buffer=75, term_buffer=50, window=25):
    """0-based warm-up iterations at which Windows ends a window (its metric update)"""
    w = Windows(num_warmup, 1, init_buffer, term_buffer, window)
    ends = []
    with np.errstate(invalid='ignore', divide='ignore'):       # (a window of one draw has no variance)
        for it in range(num_warmup):
            if w.learn(np.zeros(1)) is not None:
                ends.append(it)
    return ends


class ControlNUTS(nuts.NUTS):
    """oracle diag_e NUTS whose transitions jitter the step size"""

    def __init__(self, lp_grad, dim, rng, max_depth=10, jitter=0.0):
        super().__init__(lp_grad, dim, rng, max_depth)
        self.jitter = jitter
        self.eps_used = self.eps

    def transition(self, q, V, g):
        nom = self.eps
        if self.jitter:
            self.eps = nom * (1.0 + self.jitter * (2.0 * self.rng.uniform() - 1.0))
        try:
            return super().transition(q, V, g)
        finally:
            self.eps_used = self.eps
            self.eps = nom


def sample_chain(lp_grad, dim, n_iter, n_warmup, rng, q0=None, init_r=2.0, delta=0.8, gamma=0.05, kappa=0.75,
                 t0=10.0, init_buffer=75, term_buffer=50, window=25, stepsize=1.0, jitter=0.0,
                 adapt_engaged=True, thin=1, max_depth=10):
    """One chain.  q0: given init (NaN entries drawn at random) or None.  Returns dict(draws (n_save, dim),
    stepsize (mean eps of the saved transitions), eps (final nominal step size), minv, n_grad, last (last saved
    draw), eps_used (of the saved transitions))."""
    s = ControlNUTS(lp_grad, dim, rng, max_depth, jitter)
    given = None if q0 is None else np.array(q0, dtype=np.float64)
    random_part = given is None or np.any(np.isnan(given))
    tries = 0
    while True:
        q = rng.uniform(-init_r, init_r, size=dim)
        if given is not None:
            q = np.where(np.isnan(given), q, given)
        V, g = s._vg(q)
        if np.isfinite(V) and np.all(np.isfinite(g)):
            break
        tries += 1
        if not random_part or tries > 100:
            raise RuntimeError("initialisation failed")
    s.eps = stepsize
    da = win = None
    if adapt_engaged:
        da = nuts.DualAveraging(delta=delta, gamma=gamma, t0=t0, kappa=kappa)
        da.mu = np.log(10 * stepsize)
        win = Windows(n_warmup, dim, init_buffer, term_buffer, window)
        s.init_stepsize(q, V, g)
    draws, eps_used = [], []
    last = q
    for it in range(n_iter):
        q, V, g, accept, st = s.transition(q, V, g)
        if it < n_warmup:
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
            draws.append(q)
            eps_used.append(s.eps_used)
            last = q
    return dict(draws=np.array(draws).reshape(-1, dim), stepsize=float(np.mean(eps_used)) if eps_used else s.eps,
                eps=s.eps, minv=s.minv.copy(), n_grad=s.n_grad, last=last, eps_used=np.array(eps_used))


def sample(lp_grad, dim, chains, n_iter, n_warmup=None, seed=0, inits=None, **kw):
    """`chains` independent chains (as oracle.nuts.sample); kw: the settings of sample_chain"""
    if n_warmup is None:
        n_warmup = n_iter // 2
    res = [sample_chain(lp_grad, dim, n_iter, n_warmup, np.random.RandomState([seed, c]),
                        q0=None if inits is None else inits[c], **kw) for c in range(chains)]
    return dict(draws=np.concatenate([r['draws'] for r in res], axis=0),
                per_chain=[r['draws'] for r in res],
                stepsize=float(np.mean([r['stepsize'] for r in res])),
                eps=np.array([r['eps'] for r in res]), minv=[r['minv'] for r in res],
                n_grad=sum(r['n_grad'] for r in res), last=[r['last'] for r in res],
                eps_used=[r['eps_used'] for r in res])

"""The per-transition sampler parameters of the tests-side oracle (tests/nuts_diag.py) on small targets, and the
HMC diagnostics Worker derives from a caller-supplied sampler's fit (CPU only)."""
import numpy as np

from oracle import fakes
import nuts_diag
from epstan import method


def gauss(scales):
    s = np.asarray(scales, dtype=np.float64)
    return lambda q: (-0.5 * np.sum((q / s) ** 2), -q / s ** 2)


def test_huge_fixed_step_diverges_on_the_first_leaf():
    res = nuts_diag.sample(gauss([1.0, 2.0]), 2, chains=2, n_iter=40, n_warmup=10, seed=1, stepsize=1e3,
                           adapt_engaged=False)
    for r in res:
        rec = r['records']
        assert rec.shape == (40, 6) and r['n_warm'] == 10
        assert np.all(rec[:, 4] == 1.0)                     # divergent__
        assert np.all(rec[:, 3] == 1.0)                     # n_leapfrog__
        assert np.all(rec[:, 2] == 0.0)                     # treedepth__
        assert np.all(rec[:, 1] == 1e3)                     # stepsize__
        assert np.all(rec[:, 0] == 0.0)                     # accept_stat__ = exp(-huge)
        assert r['n_divergent'] == 30
        assert np.allclose(r['draws'], r['draws'][0])       # the chain never moves


def test_max_treedepth_saturates():
    # a tiny fixed step on a wide target: the trajectory never turns within 2^2 leapfrogs
    res = nuts_diag.sample(gauss([1.0, 1.0, 1.0]), 3, chains=2, n_iter=30, n_warmup=0, seed=2, stepsize=1e-3,
                           adapt_engaged=False, max_depth=2)
    for r in res:
        rec = r['records']
        assert np.all(rec[:, 2] == 2) and np.all(rec[:, 3] == 3)
        assert r['n_max_treedepth'] == 30 and r['n_divergent'] == 0


def test_definitions_with_adaptation():
    res = nuts_diag.sample(gauss([0.5, 1.0, 3.0, 0.1]), 4, chains=2, n_iter=300, n_warmup=150, seed=3, thin=2,
                           jitter=0.2)
    for r in res:
        rec = r['records']
        assert r['n_warm'] == 75 and rec.shape == (150, 6)
        t, nl = rec[:, 2], rec[:, 3]
        ok = rec[:, 4] == 0
        # a transition of depth t merged 2^t - 1 leaves; a discarded subtree adds at most 2^t more
        assert np.all(2 ** t[ok] - 1 <= nl[ok]) and np.all(nl <= 2 ** (t + 1) - 1)
        assert np.all((rec[:, 0] >= 0) & (rec[:, 0] <= 1))
        assert np.all(np.isfinite(rec[:, 5]))
        post = rec[r['n_warm']:]
        assert np.ptp(post[:, 1]) > 0                       # jittered step sizes
        assert r['ebfmi'] == nuts_diag.ebfmi(post[:, 5]) and 0.3 < r['ebfmi'] < 3.0


def test_ebfmi_edge_cases():
    assert np.isnan(nuts_diag.ebfmi([1.0])) and np.isnan(nuts_diag.ebfmi([2.0, 2.0, 2.0]))
    e = np.array([1.0, 3.0, 2.0, 5.0])
    assert np.isclose(nuts_diag.ebfmi(e), (4 + 1 + 9) / np.sum((e - e.mean()) ** 2))
    assert method._ebfmi(e) == nuts_diag.ebfmi(e)


class FullFit(object):
    """a PyStan fit with every sampler parameter (warm-up included, as get_sampler_params() returns them)"""

    def __init__(self, records, warmup2):
        self.sim = {'warmup2': list(warmup2)}
        self._rec = records

    def get_sampler_params(self, inc_warmup=True):
        assert inc_warmup is True
        return [dict(zip(nuts_diag.FIELDS, r.T)) for r in self._rec]


def test_host_path_summary_from_a_full_fit():
    res = nuts_diag.sample(gauss([1.0, 0.3]), 2, chains=3, n_iter=120, n_warmup=60, seed=4, max_depth=3)
    fit = FullFit([r['records'] for r in res], [r['n_warm'] for r in res])
    h = method._fit_hmc(fit, fit.get_sampler_params(), 3)
    assert list(h['n_divergent']) == [r['n_divergent'] for r in res]
    assert list(h['n_max_treedepth']) == [r['n_max_treedepth'] for r in res]
    assert np.array_equal(h['ebfmi'], [r['ebfmi'] for r in res])


def test_host_path_without_sampler_params_gives_none():
    fit = fakes.FakeFit(np.zeros((8, 2)), chains=2, niter=8, warmup=4)
    assert method._fit_hmc(fit, fit.get_sampler_params(), 10) is None

    class NoWarmup(FullFit):
        def __init__(self, records):
            self.sim = {}
            self._rec = records
    res = nuts_diag.sample(gauss([1.0]), 1, chains=1, n_iter=20, n_warmup=10, seed=5)
    fit = NoWarmup([res[0]['records']])
    assert method._fit_hmc(fit, fit.get_sampler_params(), 10) is None


def test_transient_reference_tells_the_sample_from_the_start():
    """the cached TRANSIENT run (tests/oracle_refs_diag.py) separates energy__ = H(selected sample) from H0 by
    many standard errors at its first transition, so the GPU comparison with it checks which H is recorded"""
    import oracle_refs_diag
    ref = oracle_refs_diag.transient_reference()
    (e, se_e), (h0, se_h0) = ref['energy'][0], ref['H0'][0]
    assert h0 - e > 8 * 4 * np.hypot(se_e, se_h0)

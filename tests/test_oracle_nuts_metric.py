"""The fp64 dense_e / unit_e oracle (tests/nuts_metric.py) on exact Gaussian targets, and one cached entry of
tests/golden/nuts_metric_ref.npz re-derived."""
import numpy as np
import pytest

from oracle import nuts
import nuts_metric
import oracle_refs_metric


def _gauss(S):
    P = np.linalg.inv(S)
    return lambda q: (-0.5 * q @ P @ q, -P @ q)


ISO = np.diag([1.0, 4.0, 0.25])
# correlation 0.99, scales 1 and 30: condition number 4.5e4
CORR = np.array([[1.0, 0.99], [0.99, 1.0]]) * np.outer([1.0, 30.0], [1.0, 30.0])


def _check_moments(r, S):
    ess, mcse = nuts.ess_mcse(r['per_chain'])
    x = r['draws']
    assert np.all(np.abs(x.mean(axis=0)) < 4 * mcse)
    v = x.var(axis=0, ddof=1)
    assert np.all(np.abs(v / np.diag(S) - 1.0) < 4.0 * np.sqrt(2.0 / np.maximum(0.5 * ess, 10)))


@pytest.mark.parametrize('metric', ['dense_e', 'unit_e'])
def test_isotropic_gaussian(metric):
    r = nuts_metric.sample(_gauss(ISO), 3, chains=4, n_iter=1000, n_warmup=500, seed=2, metric=metric)
    _check_moments(r, ISO)
    for S in r['Sigma']:
        if metric == 'unit_e':
            assert np.array_equal(S, np.eye(3))
        else:   # the last window holds 225 draws: ~ sqrt(2/225) = 0.09 relative error per variance
            assert np.all(np.abs(np.diag(S) / np.diag(ISO) - 1.0) < 0.45)
            assert np.all(np.abs(S - np.diag(np.diag(S))) < 0.45 * np.sqrt(np.outer(np.diag(ISO), np.diag(ISO))))


def test_correlated_gaussian_dense_beats_diag():
    assert np.linalg.cond(CORR) > 1e3
    r = {m: nuts_metric.sample(_gauss(CORR), 2, chains=4, n_iter=1000, n_warmup=500, seed=1, metric=m)
         for m in ('diag_e', 'dense_e')}
    _check_moments(r['dense_e'], CORR)
    for S in r['dense_e']['Sigma']:
        # the adapted Sigma within Monte-Carlo error of the true covariance (last window: 225 draws)
        assert np.all(np.abs(S - CORR) < 0.45 * np.sqrt(np.outer(np.diag(CORR), np.diag(CORR))))
    # gradient evaluations per draw: the condition number predicted ~4x fewer for dense_e; measured 24.5 vs
    # 12.7 (1.9x) with 4 x 2000 iterations; the bound leaves room for the shorter runs here
    ratio = r['diag_e']['n_grad'] / r['dense_e']['n_grad']
    assert ratio > 1.3, ratio
    assert r['dense_e']['stepsize'] > 3 * r['diag_e']['stepsize']


def test_diag_e_path_matches_oracle_nuts():
    """metric='diag_e' of the subclass is the diag_e oracle: the same draws for the same seed"""
    lpg = _gauss(ISO)
    a = nuts.sample(lpg, 3, chains=2, n_iter=200, n_warmup=100, seed=4)
    b = nuts_metric.sample(lpg, 3, chains=2, n_iter=200, n_warmup=100, seed=4, metric='diag_e')
    assert np.allclose(a['draws'], b['draws'], rtol=1e-12, atol=1e-12)
    assert a['n_grad'] == b['n_grad']


def test_cached_dense_reference_rederived():
    shape = oracle_refs_metric.SHAPES[0]
    cached = oracle_refs_metric.reference(*shape)
    fresh = oracle_refs_metric.compute(*shape)
    for k in ('stepsize', 'evals_per_draw'):
        assert np.isclose(float(cached[k]), float(fresh[k]), rtol=1e-9), k

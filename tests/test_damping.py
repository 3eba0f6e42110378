"""Automatic damping selection (`Master(df_select='snr')`, SURVEY 8f rank 1).

The reference's damping schedule (experiment/fit.py:176-186) was tuned for K <= 64
sites; replayed through the pinned oracle on K = 256 Gaussian sites, d = 50, 400
draws per site it DIVERGES (the pos.def. retry loop cuts df every iteration and the
approximation drifts away from the exact posterior).  These tests pin

  * the selection statistic (epg_delta_sums / epg_delta_snr) against its NumPy
    restatement (oracle.ep_linalg.fisher_norm2) at <= 1e-10,
  * Master.run with the selection against the oracle replay of the same rule,
  * convergence to the analytic fixed point of Gaussian sites (SURVEY 4 KAT):
    Q* = Q0 + sum_k Q_k, at K = 256, d = 50, >= 15 iterations.
"""
import os
import sys

import numpy as np
import pytest

from conftest import relerr
import golden_inputs as gi
from oracle import ep_linalg as orc
from oracle import fakes

TESTS = os.path.dirname(os.path.abspath(__file__))


def _scenario(K, d, chains, it, niter, seed, df0):
    return dict(K=K, d=d, fseed=seed + 100, chains=chains, iter=it, niter=niter, seed=seed,
                df0=df0, prec_estim='sample', skip=0, prior=None)


def _oracle_run(sc, **sel):
    """oracle.run_ep on the scenario's exact Gaussian draws (same seeds as FakeModel sees)."""
    Qs, rs = fakes.gaussian_site_factors(sc['fseed'], sc['K'], sc['d'])
    st = orc.EPState(np.eye(sc['d']), np.zeros(sc['d']), sc['K'])
    seeds = gi.run_seeds(sc['seed'], sc['niter'], sc['K'])
    n = sc['chains'] * (sc['iter'] - sc['iter'] // 2)
    df0 = sc['df0']
    df0f = df0 if callable(df0) else (lambda i, v=df0: v)

    def draw_fn(it, k, cm, cP):
        return fakes.gaussian_tilted_draws(gi.stan_seed(seeds[it - 1, k]), cm, cP, Qs[:, :, k], rs[:, k], n)
    info, ms, Ss = orc.run_ep(st, draw_fn, sc['niter'], df0f, **sel)
    return info, ms, Ss, st, (Qs, rs)


def _exact(Qs, rs, d):
    S, m = orc.invert_normal_params(np.eye(d) + Qs.sum(axis=2), rs.sum(axis=1))
    return m, S


def _master(method, sc, **kw):
    Qs, rs = fakes.gaussian_site_factors(sc['fseed'], sc['K'], sc['d'])
    model = fakes.FakeModel(Qs, rs)
    model.quiet = True
    K, d = sc['K'], sc['d']
    return method.Master(model, np.zeros((2 * K, 2)), np.zeros(2 * K), site_sizes=np.full(K, 2), dphi=d,
                         A_k={'site_id': list(range(K))}, chains=sc['chains'], iter=sc['iter'],
                         df0=sc['df0'], **kw)


def test_reference_schedule_diverges_selection_converges_oracle():
    """The finding that motivates the selector, on the pinned oracle alone (CPU): with the fit.py
    schedule the KL to the exact posterior GROWS at K=96, d=24, n=200 (the summed Monte Carlo error
    of 96 sites is several times the global precision itself); with the selection it never grows:
    a half step (cap = the schedule) or a full step (no cap), then the noise floor."""
    sc = _scenario(K=96, d=24, chains=4, it=100, niter=8, seed=3, df0=orc.default_df0(96))
    _, ms, Ss, _, (Qs, rs) = _oracle_run(sc)
    mt, St = _exact(Qs, rs, sc['d'])
    kl_ref = np.array([orc.kl_mvn(mt, St, ms[i], Ss[i]) for i in range(sc['niter'])])
    _, ms2, Ss2, _, _ = _oracle_run(sc, df_select='snr')
    kl_sel = np.array([orc.kl_mvn(mt, St, ms2[i], Ss2[i]) for i in range(sc['niter'])])
    sc1 = dict(sc, df0=1.0)
    _, ms3, Ss3, _, _ = _oracle_run(sc1, df_select='snr')
    kl_full = np.array([orc.kl_mvn(mt, St, ms3[i], Ss3[i]) for i in range(sc['niter'])])
    assert kl_ref[-1] > 1.5 * kl_ref[0]                            # the schedule drifts away
    assert np.all(np.diff(kl_sel) < 0.05) and kl_sel[-1] < kl_ref[0]    # the selection does not
    assert kl_full[0] < 0.5 * kl_ref[0] and kl_full.max() < 0.6 * kl_ref[0]


def test_master_selection_matches_oracle_cpu(monkeypatch):
    """Host logic of df_select='snr' (fake device context) == oracle replay of the same rule."""
    sys.path.insert(0, TESTS)
    import epstan.method as method
    import fake_backend
    monkeypatch.setattr(method.Master, '_context_factory',
                        staticmethod(lambda dev, stream: fake_backend.OracleContext(dev, stream)))
    sc = _scenario(K=12, d=6, chains=4, it=60, niter=6, seed=11, df0=orc.default_df0(12))
    m = _master(method, sc, df_select='snr')
    info, (ms, Ss) = m.run(sc['niter'], verbose=False, seed=sc['seed'])
    oinfo, oms, oSs, st, _ = _oracle_run(sc, df_select='snr')
    assert info == oinfo == 0
    assert relerr(ms, oms) < 1e-10 and relerr(Ss, oSs) < 1e-10
    assert len(m.history['df']) == sc['niter'] and len(m.history['snr']) == sc['niter']
    assert all(m.df_min <= v <= 0.5 for v in m.history['df'])
    # bad option values
    with pytest.raises(ValueError):
        _master(method, sc, df_select='best')


def test_host_state_is_not_rewound_cpu(monkeypatch):
    """ADVICE r1: a keep_on_device run leaves the host mirrors stale; the next host-state run must
    refresh them instead of uploading the stale copies over the newer device state."""
    sys.path.insert(0, TESTS)
    import epstan.method as method
    import fake_backend
    monkeypatch.setattr(method.Master, '_context_factory',
                        staticmethod(lambda dev, stream: fake_backend.OracleContext(dev, stream)))
    sc = _scenario(K=6, d=5, chains=4, it=60, niter=3, seed=5, df0=0.3)
    a = _master(method, sc)
    b = _master(method, sc)
    a.run(2, verbose=False, seed=1)
    a.run(2, verbose=False, seed=2)
    ia, (ma, Sa) = a.run(2, verbose=False, seed=3)
    b.run(2, verbose=False, seed=1)
    b.keep_on_device = True
    b.run(2, verbose=False, seed=2)
    assert b._host_stale
    b.keep_on_device = False
    ib, (mb, Sb) = b.run(2, verbose=False, seed=3)
    assert ia == ib == 0 and not b._host_stale
    assert relerr(mb, ma) < 1e-12 and relerr(Sb, Sa) < 1e-12 and relerr(b.Qi, a.Qi) < 1e-12


# ------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize('K,d', [(7, 5), (40, 20), (12, 50), (5, 200)])
def test_delta_snr_statistic(K, d):
    from epstan import _lib
    rng = np.random.RandomState(K * 1000 + d)
    ctx = _lib.Context(0)
    ctx.init_state(K, d)
    Q = np.asfortranarray(fakes.random_spd(rng, d, scale=3.0))
    r = rng.standard_normal(d)
    dQ = np.zeros((d, d, K), order='F')
    for k in range(K):
        A = rng.standard_normal((d, d))
        dQ[:, :, k] = 0.3 * (A + A.T)
    dr = np.asfortranarray(rng.standard_normal((d, K)))
    ctx.upload(_lib.Q, Q)
    ctx.upload(_lib.R, r)
    ctx.upload(_lib.DQI, dQ)
    ctx.upload(_lib.DRI, dr)
    # site flags as epg_moments would leave them: all ok (cavity of Q - 0 is pos.def.)
    flags, _ = ctx.cavity(proposal=False)
    assert flags.all()
    ctx.delta_sums()
    T2, S2, n_ok = ctx.delta_snr()
    oS2 = sum(orc.fisher_norm2(Q, r, dQ[:, :, k], dr[:, k]) for k in range(K))
    oT2 = orc.fisher_norm2(Q, r, dQ.sum(axis=2), dr.sum(axis=1))
    assert n_ok == K
    assert abs(S2 - oS2) <= 1e-10 * oS2 and abs(T2 - oT2) <= 1e-10 * oT2
    ds = ctx.download(_lib.DSUM, np.empty(d * d + d + 2 + _lib.XCHG_SLOTS))
    assert relerr(ds[:d * d].reshape(d, d, order='F'), dQ.sum(axis=2)) < 1e-13
    assert relerr(ds[d * d:d * d + d], dr.sum(axis=1)) < 1e-13


@pytest.mark.gpu
def test_master_selection_matches_oracle_gpu():
    import epstan.method as method
    sc = _scenario(K=12, d=6, chains=4, it=60, niter=6, seed=11, df0=orc.default_df0(12))
    m = _master(method, sc, df_select='snr')
    info, (ms, Ss) = m.run(sc['niter'], verbose=False, seed=sc['seed'])
    oinfo, oms, oSs, st, _ = _oracle_run(sc, df_select='snr')
    assert info == oinfo == 0
    assert relerr(ms, oms) < 1e-9 and relerr(Ss, oSs) < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize('cap', ['schedule', 'none'])
def test_ep_converges_to_gaussian_fixed_point_K256_d50(cap):
    """VERDICT r1 item 1: >= 15 EP iterations at K >= 256, d = 50, 400 draws per site.  Gaussian sites have
    the analytic fixed point Q* = Q0 + sum_k Q_k.  The reference schedule on this problem reaches KL 5.6 after
    iteration 1 and then GROWS (14.8 after 12 iterations: VERDICT r1, reproduced by
    test_reference_schedule_diverges_selection_converges_oracle at a smaller size).  With the automatic
    selection the KL to the fixed point never grows and the damping settles at its floor; without a cap the
    first (nearly full) step lands within the Monte Carlo error of one iteration."""
    import epstan.method as method
    K, d, niter = 256, 50, 16
    sc = _scenario(K=K, d=d, chains=4, it=200, niter=niter, seed=21,
                   df0=orc.default_df0(K) if cap == 'schedule' else None)
    m = _master(method, sc, df_select='snr')
    info, (ms, Ss) = m.run(niter, verbose=False, seed=sc['seed'])
    assert info == 0
    Qs, rs = fakes.gaussian_site_factors(sc['fseed'], K, d)
    mt, St = _exact(Qs, rs, d)
    kl = np.array([orc.kl_mvn(mt, St, ms[i], Ss[i]) for i in range(niter)])
    kl0 = orc.kl_mvn(mt, St, np.zeros(d), np.eye(d))          # the prior
    dfs = np.array(m.history['df'])
    assert kl0 > 100
    if cap == 'schedule':
        assert dfs[0] == pytest.approx(0.5, rel=0.02)
        assert kl[0] < 7.0 and np.all(np.diff(kl) < 0.1) and kl[-1] < kl[0], kl
    else:
        assert dfs[0] > 0.95
        assert kl[0] < 2.5 and kl.max() < 3.0, kl
    assert np.all(dfs[3:] < 0.05), dfs
    assert all(a == 1 for a in m.history['attempts'])        # no pos.def. retries at all
    # step-to-step KL (the health metric of bench.py) falls to the noise floor
    step = np.array([orc.kl_mvn(ms[i], Ss[i], ms[i - 1], Ss[i - 1]) for i in range(1, niter)])
    assert step[4:].max() < 0.2, step

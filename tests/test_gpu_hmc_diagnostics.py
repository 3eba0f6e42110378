"""PyStan's per-transition sampler parameters and per-site HMC diagnostics of the built-in sampler on the GPU.

On every launch plan of tests/metric_cases.py:
  1. recording (option "sampler_params") changes neither the draws nor the launch plan;
  2. the records agree with the run's other outputs and with the always-on summary (epg_get_hmc_diag);
  3. thinned records are every thin-th record of the unthinned run, warm-up included;
  4. forced regimes: no adaptation, jitter, a huge fixed step, max_treedepth = 2.
Then the statistics of the records against the tests-side oracle (tests/nuts_diag.py, cached by
tests/oracle_refs_diag.py) on the SIMT, tensor-core and wide passes, and Master end to end.
"""
import numpy as np
import pytest

import metric_cases
import nuts_diag
import oracle_refs_diag
from test_gpu_sampler_metric import PARENT

pytestmark = pytest.mark.gpu

NAMES = list(metric_cases.CASES)
ACC, EPS, TD, NL, DIV, EN = range(6)


def _lib():
    from epstan import _lib as L
    return L


def _case(name, record=True):
    model, J, n, D, ns, use_tc, pp, C, it, wu = metric_cases.CASES[name]
    ctx = metric_cases.make_ctx(_lib(), model, metric_cases.case_sites(name), use_tc=use_tc)
    ctx.set_option('pingpong', pp)
    ctx.set_option('sampler_params', 1 if record else 0)
    return ctx, ns, C, it, wu


def _n_rec(it, wu, thin=1):
    return -(-wu // thin), -(-(it - wu) // thin)


@pytest.mark.parametrize('name', NAMES)
def test_recording_keeps_draws_and_plan(name):
    ctx, ns, C, it, wu = _case(name)
    seeds = [1000 + 7 * k for k in range(ns)]
    out = ctx.tilted_sample(seeds, C, it, wu)
    assert metric_cases.digest(ctx, C * (it - wu), out) == PARENT[name]['digest']
    assert ctx.last_plan() == PARENT[name]['plan']
    if name == 'tc_4':
        out = ctx.tilted_sample([s + 1 for s in seeds], C, it, wu, 2)
        assert metric_cases.digest(ctx, C * (it - wu), out) == PARENT['tc_4_carried']['digest']
        assert ctx.last_plan() == PARENT['tc_4_carried']['plan']
    assert ctx.sampler_params().shape == (ns, C, sum(_n_rec(it, wu)), 6)
    for met in ('dense_e', 'unit_e'):
        res = []
        for rec in (1, 0):
            ctx.set_option('sampler_params', rec)
            out = ctx.tilted_sample(seeds, C, it, wu, metric=met)
            res.append((ctx.get_draws(C * (it - wu)), out[:3], ctx.last_plan()))
        assert np.array_equal(res[0][0], res[1][0]), met
        for a, b in zip(res[0][1], res[1][1]):
            assert np.array_equal(a, b), met
        assert res[0][2] == res[1][2]
    ctx.close()


def _check_consistent(ctx, out, C, it, wu, max_depth=10):
    msteps, _, nleap, _ = out
    rec = ctx.sampler_params()
    nw, ns_ = _n_rec(it, wu)
    assert rec.shape[1:] == (C, nw + ns_, 6)
    assert np.array_equal(ctx.sampler_params(inc_warmup=False), rec[:, :, nw:])
    diag = ctx.hmc_diagnostics()
    post = rec[:, :, nw:]
    assert np.all(diag['n_saved'] == ns_)
    assert np.allclose(post[..., EPS].mean(axis=2).mean(axis=1), msteps, rtol=1e-12, atol=0)
    assert np.array_equal(post[..., DIV].sum(axis=2), diag['n_divergent'])
    assert np.array_equal((post[..., TD] >= max_depth).sum(axis=2), diag['n_max_treedepth'])
    host = np.array([[nuts_diag.ebfmi(post[k, c, :, EN]) for c in range(C)] for k in range(rec.shape[0])])
    assert np.allclose(diag['ebfmi'], host, rtol=1e-9, atol=0, equal_nan=True)
    t, nl = rec[..., TD], rec[..., NL]
    assert np.all(2 ** t - 1 <= nl) and np.all(nl <= 2 ** (t + 1) - 1)
    assert np.all(t <= max_depth) and np.all(np.isin(rec[..., DIV], (0.0, 1.0)))
    assert np.all((rec[..., ACC] >= 0) & (rec[..., ACC] <= 1)) and np.all(np.isfinite(rec[..., EN]))
    assert np.all(nl.sum(axis=(1, 2)) <= nleap)
    return rec, diag


@pytest.mark.parametrize('name', NAMES)
def test_records_agree_with_the_run(name):
    ctx, ns, C, it, wu = _case(name)
    out = ctx.tilted_sample([50 + k for k in range(ns)], C, it, wu)
    _check_consistent(ctx, out, C, it, wu)
    ctx.close()


@pytest.mark.parametrize('name', NAMES)
def test_thinned_records(name):
    ctx, ns, C, it, wu = _case(name)
    seeds = [300 + k for k in range(ns)]
    ctx.tilted_sample(seeds, C, it, wu)
    r1 = ctx.sampler_params()
    ctx.tilted_sample(seeds, C, it, wu, thin=3)
    r3 = ctx.sampler_params()
    want = np.concatenate([r1[:, :, 0:wu:3], r1[:, :, wu::3]], axis=2)
    assert r3.shape == want.shape and np.array_equal(r3, want)
    assert np.array_equal(ctx.sampler_params(inc_warmup=False), r1[:, :, wu::3])
    ctx.close()


@pytest.mark.parametrize('name', NAMES)
def test_forced_regimes(name):
    ctx, ns, C, it, wu = _case(name)
    seeds = [70 + k for k in range(ns)]
    I, W = 60, 20
    out = ctx.tilted_sample(seeds, C, I, W, adapt_engaged=False, stepsize=0.05)
    rec, _ = _check_consistent(ctx, out, C, I, W)
    assert np.all(rec[..., EPS] == float(np.float32(0.05)))
    out = ctx.tilted_sample(seeds, C, I, W, adapt_engaged=False, stepsize=0.05, stepsize_jitter=0.3)
    rec, _ = _check_consistent(ctx, out, C, I, W)
    e = rec[..., EPS]
    assert np.all(e >= 0.05 * 0.7 * (1 - 1e-6)) and np.all(e <= 0.05 * 1.3 * (1 + 1e-6)) and np.ptp(e) > 0.01
    out = ctx.tilted_sample(seeds, C, I, W, adapt_engaged=False, stepsize=1e3)
    rec, diag = _check_consistent(ctx, out, C, I, W)
    assert np.all(rec[..., DIV] == 1) and np.all(rec[..., NL] == 1) and np.all(rec[..., TD] == 0)
    assert np.all(diag['n_divergent'] == I - W)
    out = ctx.tilted_sample(seeds, C, it, wu, max_treedepth=2)
    rec, diag = _check_consistent(ctx, out, C, it, wu, max_depth=2)
    assert diag['n_max_treedepth'].sum() > 0
    # the summary is kept without recording; the records of a run that did not record are refused
    ctx.set_option('sampler_params', 0)
    out = ctx.tilted_sample(seeds, C, it, wu, max_treedepth=2)
    assert np.array_equal(ctx.hmc_diagnostics()['n_max_treedepth'], diag['n_max_treedepth'])
    with pytest.raises(_lib().EpgError):
        ctx.sampler_params()
    ctx.close()


@pytest.mark.parametrize('name', ['simt_single', 'tc_4'])
def test_dead_chain_records_are_nan(name):
    """a chain without a finite starting point writes no transitions: its records are NaN, not stale ones"""
    ctx, ns, C, it, wu = _case(name)
    seeds = [90 + k for k in range(ns)]
    ctx.tilted_sample(seeds, C, it, wu)
    P = max(ctx.num_params(k) for k in range(ns))
    q = np.full((ns, C, P), np.nan)
    q[0, 1, :] = 1e30                    # given in full, non-finite density: one attempt, the chain dies
    ctx.set_inits(q, C)
    ctx.tilted_sample(seeds, C, it, wu, _lib().INIT_GIVEN)
    rec, diag = ctx.sampler_params(), ctx.hmc_diagnostics()
    assert np.all(np.isnan(rec[0, 1])) and diag['n_saved'][0, 1] == 0 and np.isnan(diag['ebfmi'][0, 1])
    assert np.all(np.isfinite(rec[0, 0])) and np.all(np.isfinite(rec[1:]))
    ctx.close()


# name: (reference run of oracle_refs_diag, use_tc, expected pass, replicas of the site)
STAT_RUNS = {'simt': ('narrow', 0, 0, 4), 'tc': ('narrow', 1, 1, 4), 'wide': ('wide', 1, 2, 2)}


@pytest.mark.parametrize('which', list(STAT_RUNS))
def test_statistics_against_the_oracle(which):
    ref_name, use_tc, want_tc, reps = STAT_RUNS[which]
    case, C, it, wu = oracle_refs_diag.RUNS[ref_name]
    model = metric_cases.CASES[case][0]
    site = metric_cases.case_sites(case)[0]
    ctx = metric_cases.make_ctx(_lib(), model, [site] * reps, use_tc=use_tc)
    ctx.set_option('sampler_params', 1)
    out = ctx.tilted_sample([20 + k for k in range(reps)], C, it, wu)
    assert ctx.last_plan()['use_tc'] == want_tc
    rec = ctx.sampler_params()
    _check_consistent(ctx, out, C, it, wu)
    nw = _n_rec(it, wu)[0]
    got = oracle_refs_diag.summarise([r for r in rec.reshape(-1, *rec.shape[2:])], [nw] * (reps * C))
    ref = oracle_refs_diag.reference(ref_name)
    for s, (m_ref, se_ref) in ref.items():
        m, se = got[s]
        print(which, s, m, m_ref, se, se_ref)
        assert abs(m - m_ref) <= 4 * np.hypot(se, se_ref), (s, m, m_ref, se, se_ref)
    ctx.close()


@pytest.mark.parametrize('use_tc', [0, 1])
def test_energy_is_that_of_the_selected_sample(use_tc):
    """from q = 0 at a fixed, large step the first transitions' energy__ follow the oracle's H(selected sample),
    which differs from the starting H0 by many standard errors (oracle_refs_diag.TRANSIENT)"""
    case, chains, n_iter, eps, depth = oracle_refs_diag.TRANSIENT
    model = metric_cases.CASES[case][0]
    C, reps = 16, 8
    ctx = metric_cases.make_ctx(_lib(), model, [metric_cases.case_sites(case)[0]] * reps, use_tc=use_tc)
    ctx.set_option('sampler_params', 1)
    ctx.tilted_sample([400 + k for k in range(reps)], C, n_iter, 0, 1, adapt_engaged=False, stepsize=eps,
                      max_treedepth=depth)
    assert ctx.last_plan()['use_tc'] == use_tc
    E = ctx.sampler_params()[..., EN].reshape(reps * C, n_iter)
    ref = oracle_refs_diag.transient_reference()['energy']
    for t in range(n_iter):
        m, se = E[:, t].mean(), E[:, t].std(ddof=1) / np.sqrt(reps * C)
        print(use_tc, t, m, se, ref[t])
        assert abs(m - ref[t, 0]) <= 4 * np.hypot(se, ref[t, 1]), (t, m, se, ref[t])
    ctx.close()


def test_master_end_to_end():
    import epstan.method as method
    import oracle_refs
    K, n_k, D, C, siter, niter = 4, 150, 3, 4, 200, 3
    X, y, prior, d = oracle_refs.ep_problem('m1b', K, n_k, D, seed=9)
    kw = dict(site_sizes=np.full(K, n_k), prior=prior, chains=C, iter=siter, df0=0.6)
    res = {}
    for save in (False, True):
        m = method.Master('experiment/models/m1b_sg', X, y, save_sampler_params=save, **kw)
        ret = m.run(niter, calc_moments=False, verbose=False, seed=1)
        assert (ret[0] if isinstance(ret, tuple) else ret) == 0
        res[save] = (m.Q.copy(), m.r.copy())
        assert len(m.history['hmc']) == niter
        for h in m.history['hmc']:
            n_div, s_div, s_td, eb = h
            assert 0 <= s_div <= K and 0 <= s_td <= K and n_div >= s_div and eb > 0
        for w in m.workers:
            assert set(w.last_hmc) == {'n_divergent', 'n_max_treedepth', 'ebfmi'}
            assert w.last_hmc['ebfmi'].shape == (C,)
        last = m
    assert np.array_equal(res[False][0], res[True][0]) and np.array_equal(res[False][1], res[True][1])
    w0, w1 = last.workers[0], last.workers[1]
    sp = w0.get_sampler_params()
    assert len(sp) == C and list(sp[0]) == list(nuts_diag.FIELDS)
    assert all(len(v) == siter for p in sp for v in p.values())
    sp_post = w0.get_sampler_params(inc_warmup=False)
    assert all(len(v) == siter // 2 for p in sp_post for v in p.values())
    n_div = [int(np.sum(p['divergent__'])) for p in sp_post]
    assert n_div == list(w0.last_hmc['n_divergent'])
    assert np.allclose([nuts_diag.ebfmi(p['energy__']) for p in sp_post], w0.last_hmc['ebfmi'], rtol=1e-9)
    # a per-site run of another site keeps site 0's records readable
    before = [p['energy__'] for p in w0.get_sampler_params()]
    dQi, dri = np.empty((d, d), order='F'), np.empty(d)
    w1.cavity(last.Q, last.r, np.zeros((d, d), order='F'), np.zeros(d))
    w1.tilted(dQi, dri, seed=5)
    assert w1.last_hmc is not None
    after = [p['energy__'] for p in w0.get_sampler_params()]
    assert all(np.array_equal(a, b) for a, b in zip(before, after))
    assert not np.array_equal(w1.get_sampler_params()[0]['energy__'], before[0])

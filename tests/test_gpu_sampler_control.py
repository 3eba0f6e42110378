"""PyStan's `thin`, `init`, `init_r` and NUTS `control` settings of the built-in sampler on the GPU.

Deterministic, bitwise, on every launch plan of tests/metric_cases.py:
  1. every new argument passed at its default reproduces the digests of the library before they existed;
  2. thinning keeps every thin-th draw of the unthinned chain; 3. init_prev starts from the last saved draw;
  4. adaptation off: warm-up transitions are discarded transitions, and the metric choice does not matter;
  5. window arguments follow Stan's schedule (with its rescaling); 6. given inits and init_r.
Statistical, against Stan's formulas and the tests-side oracle (tests/nuts_control.py): jitter, dual-averaging
constants, a one-window schedule; then Master end to end, and kernel coverage.
"""
import numpy as np
import pytest

from oracle import nuts
import metric_cases
import oracle_refs_control
import synth
from test_gpu_sampler_metric import PARENT

pytestmark = pytest.mark.gpu

DEFAULTS = dict(thin=1, stepsize=1.0, stepsize_jitter=0.0, adapt_engaged=True, adapt_gamma=0.05, adapt_kappa=0.75,
                adapt_t0=10.0, adapt_init_buffer=75, adapt_term_buffer=50, adapt_window=25, init_r=2.0)
NAMES = list(metric_cases.CASES)
_COVER = {}             # (kernel, use_tc) -> {'thin', 'jitter', 'adapt_off'} seen by this module


def _lib():
    from epstan import _lib as L
    return L


def _record(ctx, *features):
    pl = ctx.last_plan()
    _COVER.setdefault((pl['kernel'], pl['use_tc']), set()).update(features)
    return pl


def _case(name):
    model, J, n, D, ns, use_tc, pp, C, it, wu = metric_cases.CASES[name]
    ctx = metric_cases.make_ctx(_lib(), model, metric_cases.case_sites(name), use_tc=use_tc)
    ctx.set_option('pingpong', pp)
    return ctx, ns, C, it, wu


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize('name', NAMES)
def test_explicit_defaults_reproduce_parent(name):
    res = metric_cases.run_case(_lib(), name, **DEFAULTS)
    for k, (dg, plan) in res.items():
        assert plan == PARENT[k]['plan'], (plan, PARENT[k]['plan'])
        assert dg == PARENT[k]['digest'], k


@pytest.mark.parametrize('name', NAMES)
def test_thin_and_last_saved_draw(name):
    ctx, ns, C, it, wu = _case(name)
    seeds = [300 + k for k in range(ns)]
    per, thin = it - wu, 3
    n3 = -(-per // thin)
    out1 = ctx.tilted_sample(seeds, C, it, wu)
    d1 = ctx.get_draws(C * per)
    out3 = ctx.tilted_sample(seeds, C, it, wu, thin=thin)
    _record(ctx, 'thin')
    d3 = ctx.get_draws(C * n3)
    for c in range(C):
        assert np.array_equal(d3[:, :, c * n3:(c + 1) * n3], d1[:, :, c * per:(c + 1) * per:thin]), c
    assert np.array_equal(out3[0], out1[0]) and np.array_equal(out3[2], out1[2])      # msteps, n_leapfrog
    assert not np.array_equal(out3[1], out1[1])
    for k in range(ns):
        chains = [d3[k][:, c * n3:(c + 1) * n3].T for c in range(C)]
        ref = np.max(nuts.split_rhat(chains))
        assert out3[1][k] >= ref * (1 - 1e-4), (k, out3[1][k], ref)
    # init_prev carries the last SAVED draw: a thinned run and an unthinned run that ends at that draw's
    # transition give the same follow-up run
    follow = [900 + k for k in range(ns)]
    ctx.tilted_sample(seeds, C, it, wu, thin=thin)
    ctx.tilted_sample(follow, C, 40, 20, 2)
    a = ctx.get_draws(C * 20)
    ctx.tilted_sample(seeds, C, wu + thin * (n3 - 1) + 1, wu)
    ctx.tilted_sample(follow, C, 40, 20, 2)
    assert np.array_equal(ctx.get_draws(C * 20), a)
    ctx.close()


@pytest.mark.parametrize('name', NAMES)
def test_adaptation_off(name):
    ctx, ns, C, _, _ = _case(name)
    seeds = [40 + k for k in range(ns)]
    I, W = 60, 25
    kw = dict(adapt_engaged=False, stepsize=0.05, stepsize_jitter=0.3)
    ctx.tilted_sample(seeds, C, I, 0, **kw)
    full = ctx.get_draws(C * I)
    res = {}
    for met in ('diag_e', 'dense_e', 'unit_e'):
        out = ctx.tilted_sample(seeds, C, I, W, metric=met, **kw)
        _record(ctx, 'adapt_off', 'jitter')
        res[met] = (ctx.get_draws(C * (I - W)), out[:3])
        assert np.all(np.isfinite(res[met][0]))
    for c in range(C):
        assert np.array_equal(res['diag_e'][0][:, :, c * (I - W):(c + 1) * (I - W)],
                              full[:, :, c * I + W:(c + 1) * I]), c
    for met in ('dense_e', 'unit_e'):
        assert np.array_equal(res[met][0], res['diag_e'][0]), met
        _same(res[met][1], res['diag_e'][1])
    # the carried state is what the run used: the step size and the identity
    P = _lib().load().epg_max_params(ctx._h)
    p = ctx.num_params(0)
    minv, eps = ctx.get_adapt(0, C, P)
    assert np.all(eps == np.float32(0.05)) and np.all(minv[:, :p] == 1.0)
    ctx.close()


@pytest.mark.parametrize('name', NAMES)
def test_window_arguments(name):
    ctx, ns, C, _, _ = _case(name)
    seeds = [70 + k for k in range(ns)]
    I, W = 130, 100
    runs = []
    for win in ((75, 50, 25), (15, 10, 75), (200, 200, 200), (15, 10, 74)):
        out = ctx.tilted_sample(seeds, C, I, W, adapt_init_buffer=win[0], adapt_term_buffer=win[1],
                                adapt_window=win[2])
        runs.append((ctx.get_draws(C * (I - W)), out[:3]))
    for r in runs[1:3]:
        assert np.array_equal(r[0], runs[0][0])
        _same(r[1], runs[0][1])
    assert not np.array_equal(runs[3][0], runs[0][0])
    ctx.close()


@pytest.mark.parametrize('name', NAMES)
def test_inits(name):
    L = _lib()
    ctx, ns, C, _, _ = _case(name)
    seeds = [110 + k for k in range(ns)]
    P = L.load().epg_max_params(ctx._h)
    d = ctx.d
    I, W = 40, 20

    def run(mode, **kw):
        out = ctx.tilted_sample(seeds, C, I, W, mode, **kw)
        return ctx.get_draws(C * (I - W)), out[:3]
    zero, rand = run(1), run(0)
    ctx.set_inits(np.zeros((ns, C, P)), C)
    g = run(L.INIT_GIVEN)
    assert np.array_equal(g[0], zero[0]); _same(g[1], zero[1])
    ctx.set_inits(np.full((ns, C, P), np.nan), C)
    g = run(L.INIT_GIVEN)
    assert np.array_equal(g[0], rand[0]); _same(g[1], rand[1])
    # a given phi comes back after one tiny step
    rng = np.random.RandomState(1)
    q = np.full((ns, C, P), np.nan)
    q[:, :, :d] = rng.uniform(-1, 1, size=(ns, C, d))
    ctx.set_inits(q, C)
    tiny = dict(adapt_engaged=False, stepsize=1e-4, max_treedepth=1)
    ctx.tilted_sample(seeds, C, 1, 0, L.INIT_GIVEN, **tiny)
    dr = ctx.get_draws(C)
    assert np.max(np.abs(dr - q[:, :, :d].transpose(0, 2, 1))) < 1e-2
    # init_r: random starts inside (-r, r) with a spread over sites x chains
    for r in (0.1, 5.0):
        ctx.tilted_sample(seeds, C, 1, 0, 0, init_r=r, **tiny)
        dr = ctx.get_draws(C)
        assert np.all(np.abs(dr) < r + 1e-2), r
        assert np.all(np.ptp(dr.transpose(1, 0, 2).reshape(d, -1), axis=1) > r / 2), r
    # a start given in full at a non-finite density fails its site, and only its site
    q = np.zeros((ns, C, P))
    q[0, :, :d] = 3e38
    ctx.set_inits(q, C)
    ms, mr, nl, _ = ctx.tilted_sample(seeds, C, I, W, L.INIT_GIVEN)
    dr = ctx.get_draws(C * (I - W))
    assert np.all(np.isnan(dr[0])) and np.all(np.isfinite(dr[1:]))
    ok, _ = ctx.moments(C * (I - W))
    assert not ok[0] and np.all(ok[1:]) and np.isnan(mr[0])
    # a given run needs inits for its chain count
    with pytest.raises(L.EpgError):
        ctx.tilted_sample(seeds, C + 1 if C < 32 else C - 1, I, W, L.INIT_GIVEN)
    ctx.close()


def _gauss_beta_site(sd, seed=5, n=200):
    """m1b with X = 0: beta leaves the likelihood, and with a block-diagonal cavity its tilted distribution is
    exactly the cavity's N(0, diag(sd^2))"""
    D = len(sd)
    site = synth.make_site('m1b', n, D, 1, seed=seed)
    site['X'][:] = 0.0
    Om = np.eye(D + 1)
    Om[1:, 1:] = np.diag(1.0 / np.asarray(sd) ** 2)
    site['Omega'] = Om
    site['mu'] = np.zeros(D + 1)
    return site


@pytest.mark.parametrize('use_tc', [0, 1])
def test_jitter_moments_and_mean_step(use_tc):
    sd = np.array([1.0, 0.5, 2.0])
    ctx = metric_cases.make_ctx(_lib(), 'm1b', [_gauss_beta_site(sd)], use_tc=use_tc)
    C, I, eps, j = 8, 1500, 0.3, 0.5
    ms, _, _, _ = ctx.tilted_sample([3], C, I, 0, adapt_engaged=False, stepsize=eps, stepsize_jitter=j)
    _record(ctx, 'jitter', 'adapt_off')
    se = eps * j / np.sqrt(3.0) / np.sqrt(C * I)
    assert abs(ms[0] - eps) < 4 * se, (ms[0], se)
    dr = ctx.get_draws(C * I)[0].T[:, 1:]
    chains = [dr[c * I:(c + 1) * I] for c in range(C)]
    ess, mcse = nuts.ess_mcse(chains)
    assert np.all(np.abs(dr.mean(axis=0)) < 4 * mcse)
    v = dr.var(axis=0, ddof=1)
    assert np.all(np.abs(v / sd ** 2 - 1.0) < 4.0 * np.sqrt(2.0 / np.maximum(0.5 * ess, 10)))
    ctx.close()


def test_dual_averaging_constants_vs_oracle():
    L = _lib()
    site = synth.make_site(*oracle_refs_control.SITE)
    ctx = metric_cases.make_ctx(L, oracle_refs_control.SITE[0], [site] * 4)
    C = oracle_refs_control.CHAINS
    P = L.load().epg_max_params(ctx._h)
    got = {}
    for name, kw in oracle_refs_control.SETTINGS.items():
        ctx.tilted_sample([11, 12, 13, 14], C, oracle_refs_control.ITER, oracle_refs_control.WARM,
                          **{'adapt_' + k: v for k, v in kw.items()})
        got[name] = np.median([ctx.get_adapt(k, C, P)[1] for k in range(4)])
        ref = oracle_refs_control.reference(name)
        print(name, 'step size GPU %.4g oracle %.4g' % (got[name], ref))
        assert 0.6 < got[name] / ref < 1.6, (name, got[name], ref)
    ctx.close()


def test_one_window_schedule_metric():
    """warm-up 150 with buffers 50 / 50 and window 50: one window of 50 draws, whose regularised variance
    n/(n+5) var + 1e-3 5/(n+5) is the adapted inverse metric; beta scales 0.03 ... 30 (10^3 apart)"""
    L = _lib()
    sd = np.array([0.03, 0.3, 3.0, 30.0])
    ctx = metric_cases.make_ctx(L, 'm1b', [_gauss_beta_site(sd)], use_tc=0)
    C = 16
    ctx.tilted_sample([9], C, 160, 150, adapt_init_buffer=50, adapt_term_buffer=50, adapt_window=50)
    P = L.load().epg_max_params(ctx._h)
    minv, _ = ctx.get_adapt(0, C, P)
    n = 50.0
    want = n / (n + 5) * sd ** 2 + 1e-3 * 5 / (n + 5)
    med = np.median(minv[:, 1:1 + len(sd)], axis=0)
    print('median window variance / expected', med / want)
    assert np.all(np.abs(med / want - 1.0) < 0.35), med / want
    # the default schedule at this warm-up has three windows: a different metric
    ctx.tilted_sample([9], C, 160, 150)
    assert not np.array_equal(ctx.get_adapt(0, C, P)[0], minv)
    ctx.close()


def test_master_end_to_end():
    import epstan.method as method
    import oracle_refs
    K, n_k, D, C, siter, thin = 4, 150, 3, 4, 300, 2
    X, y, prior, d = oracle_refs.ep_problem('m1b', K, n_k, D, seed=9)
    control = dict(max_treedepth=8, adapt_delta=0.85, metric='diag_e', stepsize=0.5, stepsize_jitter=0.1,
                   adapt_engaged=True, adapt_gamma=0.06, adapt_kappa=0.8, adapt_t0=8.0, adapt_init_buffer=30,
                   adapt_term_buffer=20, adapt_window=20)
    kw = dict(site_sizes=np.full(K, n_k), prior=prior, chains=C, iter=siter, df0=0.6)
    m = method.Master('experiment/models/m1b_sg', X, y, thin=thin, init_prev=False, adapt_prev=False,
                      init={'phi': np.zeros(d)}, init_r=1.5, control=control, **kw)
    info, (ms, Ss), _ = m.run(2, verbose=False, seed=1, return_analytics=True)
    assert info == 0 and np.all(np.isfinite(ms))
    n = C * -(-(siter - siter // 2) // thin)
    assert all(w.nsamp == n for w in m.workers)
    S, mm = m.mix_phi()
    dr = m._shard.ctx.get_draws(n)
    assert np.allclose(mm, dr.mean(axis=2).mean(axis=0), rtol=1e-9, atol=1e-12)
    with pytest.raises(ValueError, match='adapt_prev=False'):
        method.Master('experiment/models/m1b_sg', X, y, control={'stepsize': 0.1}, **kw)
    for bad in (dict(thin=0), dict(init_r=-1.0), dict(control={'stepsize_jitter': 2.0}, adapt_prev=False),
                dict(control={'adapt_window': 0}), dict(control={'adapt_gamma': 0.0}),
                dict(init={'phi': np.zeros(d)})):           # (a dict init needs init_prev=False)
        with pytest.raises(ValueError):
            method.Master('experiment/models/m1b_sg', X, y, **dict(kw, **bad))


def test_every_kernel_ran_each_setting():
    """runs last: thin > 1, jitter > 0 and adaptation off went through the per-site kernel with the SIMT,
    tensor-core and wide passes and through the two-sites-per-CTA kernel"""
    for want in [(1, 0), (1, 1), (1, 2), (2, 1)]:
        assert _COVER.get(want, set()) >= {'thin', 'jitter', 'adapt_off'}, (want, _COVER)

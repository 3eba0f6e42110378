"""The likelihood pass and the gradient finish of the sampler kernel, in every launch plan the sampler uses,
against the fp64 density (oracle/density.py).

`Context.logdensity(k, q, chains)` plans its launch exactly as `tilted_sample` does for `chains` chains (likelihood
pass, chain padding, shared-memory layout, tensor-core ring depth, chain-vector addressing) and `last_plan()`
reports that plan.  The tests sweep the chain counts, ring depths (EPGPU_NST) and site shapes that select the
different arms:
  SIMT pass           chains padded to 4/8/16/32, design matrix resident in shared memory or streamed, NC > 1
  tensor-core pass    tc::pass<4|8|16> x ring depth 4..8, ragged and single-tile sites
  wide tensor-core    D+1 in 65..256, every ring depth the plan admits
The tensor-core passes are compared with the oracle on the inputs they store (centred, bf16) and with the
residuals rounded to bf16 as the epilogue stores them (synth.tc_oracle), so that their gradient tolerance can be
tight.  Tolerances: lp 5e-5 relative (all passes); gradient 2e-4 (SIMT) and TC_GRAD_TOL (tensor-core passes)
of the largest entry.
"""

import numpy as np
import pytest

import synth

pytestmark = pytest.mark.gpu

LP_TOL = 5e-5
SIMT_GRAD_TOL = 2e-4
TC_GRAD_TOL = 5e-4

SIMT_CHAINS = (1, 4, 5, 8, 12, 16, 17, 32)
TC_CHAINS = (1, 3, 4, 5, 8, 9, 16)
TC_NST = (4, 5, 6, 7, 8)
TC_ROWS = (1, 127, 128, 129, 641, 5000)
TC_SHAPES = [('m1b', 19), ('m2b', 63), ('m3b', 8), ('m4b', 3), ('m5b', 31)]
WIDE_CHAINS = (1, 17, 32)
WIDE_SHAPES = [('m4b', 64), ('m3b', 128), ('m1b', 199), ('m2b', 255)]      # D + 1 = 65, 129, 200, 256
WIDE_ROWS = (129, 700)


def make_ctx(model, sites, use_tc):
    from epstan import _lib
    d = sites[0]['d']
    D = sites[0]['X'].shape[1]
    ctx = _lib.Context(0)
    ctx.init_state(len(sites), d)
    k_lim = np.concatenate(([0], np.cumsum([s['X'].shape[0] for s in sites])))
    multi = any(s['J'] > 1 for s in sites)
    ctx.upload_sites(_lib.MODEL_IDS[model], D, k_lim, np.concatenate([s['X'] for s in sites]),
                     np.concatenate([s['y'] for s in sites]),
                     np.concatenate([s['j_ind'] for s in sites]) if multi else None,
                     [s['J'] for s in sites] if multi else None)
    ctx.upload(_lib.CAVQ, np.asfortranarray(np.stack([s['Omega'] for s in sites], axis=2)))
    ctx.upload(_lib.CAVM, np.asfortranarray(np.stack([s['mu'] for s in sites], axis=1)))
    ctx.set_option('use_tc', use_tc)
    return ctx


def site_of(model, n, D, J=1, seed=0, sizes=None):
    s = synth.make_site(model, n, D, J, seed)
    if sizes is not None:                        # explicit group sizes (sorted group index)
        s['sizes'] = np.asarray(sizes)
        s['j_ind'] = np.repeat(np.arange(J), sizes)
    if s['d'] > 64:                              # keep the cavity term moderate at large d
        s['Omega'] = s['Omega'] / max(1.0, np.abs(s['Omega']).max()) + np.eye(s['d'])
    return s


def points(rng, p, nq, D, scale=0.4):
    return (scale / np.sqrt(max(D, 16) / 16.0)) * rng.standard_normal((nq, p))


def errors(lp, grad, ref):
    olp, og = ref
    assert np.all(np.isfinite(lp)) and np.all(np.isfinite(grad))
    return (float(np.max(np.abs(lp - olp) / np.maximum(1.0, np.abs(olp)))),
            float(np.max(np.abs(grad - og)) / max(1.0, np.max(np.abs(og)))))


def check(ctx, k, model, site, q, chains, ticks=2, worst=None):
    """logdensity of site k at q with `chains`, against the oracle of the pass the plan picked; returns the plan"""
    lp, grad = ctx.logdensity(k, q, chains=chains, ticks=ticks)
    plan = ctx.last_plan()
    assert plan['kernel'] == 3
    if plan['use_tc']:
        elp, eg = errors(lp, grad, synth.tc_oracle(model, site)(q))
        tol = TC_GRAD_TOL
    else:
        elp, eg = errors(lp, grad, synth.oracle_density(model, site).lp_grad(q))
        tol = SIMT_GRAD_TOL
    where = (model, site['X'].shape, chains, plan)
    assert elp < LP_TOL, (elp, where)
    assert eg < tol, (eg, where)
    if worst is not None:
        key = ('simt', 'tc', 'wide')[plan['use_tc']]
        w = worst.setdefault(key, [0.0, 0.0])
        w[0], w[1] = max(w[0], elp), max(w[1], eg)
    return plan


def report(name, worst):
    for arm, (elp, eg) in sorted(worst.items()):
        print('\n[likelihood-plans] %s %s: worst lp rel err %.2e, worst grad err %.2e' % (name, arm, elp, eg))


# ---- SIMT pass ----

def simt_sites():
    """(model, D, sites) of the SIMT arm for C chains: single- and multi-group sites on both sides of the
    residency limit of the design matrix for pad(C), and a wide shape whose chain columns need NC > 1 blocks
    per thread at 32 padded chains.  The limits (rows) follow plan_smem: m1b / m3b at D = 5 about 2.9k (32
    padded chains) to 6.9k (4); m4b at D = 12, J = 2 about 1.3k to 3.3k."""
    small = [('m1b', 5, [site_of('m1b', 300, 5, seed=1), site_of('m1b', 1100, 5, seed=2)]),
             ('m3b', 5, [site_of('m3b', 700, 5, 3, seed=3, sizes=[300, 1, 399]),
                         site_of('m3b', 900, 5, 4, seed=4, sizes=[255, 257, 129, 259])]),
             ('m4b', 12, [site_of('m4b', 1000, 12, 2, seed=5, sizes=[513, 487])])]
    big = [('m1b', 5, [site_of('m1b', 7500, 5, seed=6)]),
           ('m3b', 5, [site_of('m3b', 7400, 5, 3, seed=7, sizes=[2000, 2900, 2500])]),
           ('m4b', 12, [site_of('m4b', 3700, 12, 2, seed=8, sizes=[1800, 1900])]),
           ('m5b', 8, [site_of('m5b', 1500, 8, 2, seed=9)])]
    wide = [('m1b', 150, [site_of('m1b', 200, 150, seed=10), site_of('m1b', 500, 150, seed=11)])]
    return small + big + wide


@pytest.mark.parametrize('C', SIMT_CHAINS)
def test_simt_pass_every_plan(C):
    rng = np.random.RandomState(100 + C)
    worst = {}
    seen = set()
    for model, D, sites in simt_sites():
        ctx = make_ctx(model, sites, use_tc=0)
        for k, site in enumerate(sites):
            q = points(rng, ctx.num_params(k), 2 * C + 1, D)          # two full batches and a partial one
            plan = check(ctx, k, model, site, q, C, worst=worst)
            assert plan['use_tc'] == 0 and plan['chain_pad'] == max(4, 1 << (C - 1).bit_length())
            seen.add((plan['resident'], plan['NC'] > 1))
        ctx.close()
    assert {(1, False), (0, False)} <= seen, seen
    if C >= 17:
        assert any(nc for _, nc in seen), seen
    report('simt C=%d' % C, worst)


# ---- tensor-core pass ----

@pytest.mark.parametrize('nst', TC_NST)
@pytest.mark.parametrize('model,D', TC_SHAPES)
def test_tensor_core_pass_every_plan(model, D, nst, monkeypatch):
    monkeypatch.setenv('EPGPU_NST', str(nst))
    sites = [site_of(model, n, D, seed=200 + i) for i, n in enumerate(TC_ROWS)]
    ctx = make_ctx(model, sites, use_tc=1)
    rng = np.random.RandomState(nst)
    worst = {}
    n_tc = 0
    for C in TC_CHAINS:
        for k, site in enumerate(sites):
            q = points(rng, ctx.num_params(k), 2 * C, D)
            plan = check(ctx, k, model, site, q, C, worst=worst)
            if plan['use_tc']:
                assert plan['use_tc'] == 1 and plan['tc_nst'] == nst
                assert plan['chain_pad'] == (4 if C <= 4 else 8 if C <= 8 else 16)
                assert plan['omega_smem'] == 1 and plan['hot_nvec'] >= 18
                n_tc += 1
    ctx.close()
    assert n_tc > 0
    report('tc %s D=%d nst=%d' % (model, D, nst), worst)


def test_tensor_core_gradient_tolerance_is_tight():
    """Config 4's shape (m3b, D = 49, 4 chains: tc::pass<4>).  Against the bf16-E oracle the gradient must be
    within TC_GRAD_TOL; a gradient product that drops one 32-row slice of one tile (rows 96..127 of the first)
    moves the gradient by more than twice that, so such a fault cannot hide inside the tolerance."""
    model, n, D = 'm3b', 5000, 49
    site = site_of(model, n, D, seed=300)
    ctx = make_ctx(model, [site], use_tc=1)
    q = points(np.random.RandomState(3), ctx.num_params(0), 4, D)
    lp, grad = ctx.logdensity(0, q, chains=4)
    plan = ctx.last_plan()
    assert plan['use_tc'] == 1 and plan['chain_pad'] == 4
    olp, og = synth.tc_oracle(model, site)(q)
    scale = max(1.0, np.max(np.abs(og)))
    assert np.max(np.abs(lp - olp) / np.maximum(1.0, np.abs(olp))) < LP_TOL
    assert np.max(np.abs(grad - og)) < TC_GRAD_TOL * scale

    def drop_slice(e):
        e = synth.bf16_round(e)
        e[:, 96:128] = 0.0
        return e
    td = synth.oracle_density(model, dict(site, X=synth.tc_stored_X(site['X'])))
    _, og_cut = td.lp_grad(q, e_map=drop_slice)
    assert np.max(np.abs(og_cut - og)) > 2 * TC_GRAD_TOL * scale
    ctx.close()


# ---- wide tensor-core pass ----

@pytest.mark.parametrize('model,D', WIDE_SHAPES)
def test_wide_pass_every_ring_depth(model, D, monkeypatch):
    sites = [site_of(model, n, D, seed=400 + i) for i, n in enumerate(WIDE_ROWS)]
    ctx = make_ctx(model, sites, use_tc=1)
    rng = np.random.RandomState(D)
    nkc = (D + 1 + 63) // 64
    worst = {}
    # the plan's own depth first, then every depth from nkc (the least the pass admits) up to it
    monkeypatch.delenv('EPGPU_NST', raising=False)
    check(ctx, 0, model, sites[0], points(rng, ctx.num_params(0), 1, D), 32)
    deepest = ctx.last_plan()['tc_nst']
    assert ctx.last_plan()['use_tc'] == 2 and deepest >= nkc
    depths = set()
    for nst in range(nkc, deepest + 1):
        monkeypatch.setenv('EPGPU_NST', str(nst))
        for C in WIDE_CHAINS:
            for k, site in enumerate(sites):
                q = points(rng, ctx.num_params(k), C + 1, D)
                plan = check(ctx, k, model, site, q, C, worst=worst)
                assert plan['use_tc'] == 2 and plan['chain_pad'] == 32 and plan['tc_nst'] == max(nst, 2)
                depths.add(plan['tc_nst'])
    assert depths == set(range(max(nkc, 2), deepest + 1))
    ctx.close()
    report('wide %s D=%d' % (model, D), worst)


# ---- ticks ----

@pytest.mark.parametrize('arm', ['simt', 'tc4', 'tc16', 'wide'])
def test_ticks_give_identical_results(arm, monkeypatch):
    """The pipeline state the tensor-core passes carry from one gradient evaluation to the next (ring slot,
    barrier phases, accumulator buffers) must not change the result: ticks in {1, 2, 3, 2 nst + 1} give
    bit-identical lp and gradient, on a one-tile site and on a site whose tile count is not a multiple of
    the ring depth."""
    model, D, use_tc, C, nst = {'simt': ('m3b', 5, 0, 8, None), 'tc4': ('m3b', 8, 1, 4, 6),
                                'tc16': ('m1b', 19, 1, 16, 5), 'wide': ('m1b', 70, 1, 17, 3)}[arm]
    if nst:
        monkeypatch.setenv('EPGPU_NST', str(nst))
    sites = [site_of(model, 100, D, seed=500), site_of(model, 128 * 7 + 5, D, seed=501)]   # 1 tile; 8 tiles
    ctx = make_ctx(model, sites, use_tc=use_tc)
    rng = np.random.RandomState(5)
    for k, site in enumerate(sites):
        q = points(rng, ctx.num_params(k), C, D)
        ref = ctx.logdensity(k, q, chains=C, ticks=1)
        plan = ctx.last_plan()
        assert plan['use_tc'] == {'simt': 0, 'tc4': 1, 'tc16': 1, 'wide': 2}[arm]
        if nst:
            assert plan['tc_nst'] == nst
            tiles = (site['X'].shape[0] + 127) // 128
            assert tiles == 1 or tiles % nst != 0
        for ticks in (2, 3, 2 * max(plan['tc_nst'], 1) + 1):
            lp, grad = ctx.logdensity(k, q, chains=C, ticks=ticks)
            assert np.array_equal(lp, ref[0]) and np.array_equal(grad, ref[1]), ticks
        check(ctx, k, model, site, q, C, ticks=1)
    ctx.close()


# ---- extreme inputs ----

def edge_points(model, site, D, nq, fmax, rng):
    """q with alpha = 0 and slopes beta scaled so that max |x' beta| = fmax (m1b: beta = phi[1:]; m4b:
    beta = mu_b, sigma_b small); y then follows the sign of f except on the flipped rows."""
    td = synth.oracle_density(model, site)
    q = np.zeros((nq, td.p))
    for i in range(nq):
        beta = rng.standard_normal(D)
        beta *= fmax / np.max(np.abs(site['X'] @ beta))
        if model == 'm1b':
            q[i, 1:1 + D] = beta
        else:
            q[i, 2:2 + D] = beta
            q[i, 2 + D:2 + 2 * D] = -3.0                    # log sigma_b
            q[i, td.d + td.J:] = 0.1 * rng.standard_normal(td.p - td.d - td.J)
    return q


@pytest.mark.parametrize('use_tc', [0, 1])
@pytest.mark.parametrize('fmax', [20.0, 45.0, 100.0])
def test_large_linear_predictors(fmax, use_tc):
    worst = {}
    for model, D, C in (('m1b', 7, 8), ('m4b', 5, 4)):
        site = site_of(model, 641, D, seed=600)
        site['Omega'] = 1e-3 * site['Omega']
        rng = np.random.RandomState(int(fmax))
        q = edge_points(model, site, D, C, fmax, rng)
        # y follows the sign of f of the first point, opposed on a fifth of the rows
        f0 = site['X'] @ (q[0, 1:1 + D] if model == 'm1b' else q[0, 2:2 + D])
        y = (f0 > 0).astype(np.int64)
        flip = rng.uniform(size=len(y)) < 0.2
        y[flip] = 1 - y[flip]
        site['y'] = y
        ctx = make_ctx(model, [site], use_tc=use_tc)
        plan = check(ctx, 0, model, site, q, C, worst=worst)
        assert plan['use_tc'] == use_tc
        ctx.close()
    report('edges |f|<=%g use_tc=%d' % (fmax, use_tc), worst)


@pytest.mark.parametrize('use_tc', [0, 1])
def test_degenerate_sites(use_tc):
    """y all 0, y all 1, a single-row site, and (SIMT) single-row groups and groups across tile boundaries."""
    model, D, C = 'm4b', 6, 5
    sites = [site_of(model, 300, D, seed=700), site_of(model, 300, D, seed=701), site_of(model, 1, D, seed=702),
             site_of(model, 129, D, seed=703), site_of(model, 257, D, seed=704)]
    sites[0]['y'][:] = 0
    sites[1]['y'][:] = 1
    if not use_tc:
        # single-row groups; groups that straddle the 256-row (R) and 128-row boundaries
        sites[3] = site_of(model, 129, D, 4, seed=703, sizes=[1, 126, 1, 1])
        sites[4] = site_of(model, 600, D, 5, seed=704, sizes=[1, 300, 1, 169, 129])
    ctx = make_ctx(model, sites, use_tc=use_tc)
    rng = np.random.RandomState(7)
    worst = {}
    for k, site in enumerate(sites):
        q = points(rng, ctx.num_params(k), 2 * C, D)
        plan = check(ctx, k, model, site, q, C, worst=worst)
        assert plan['use_tc'] == use_tc
    ctx.close()
    report('degenerate use_tc=%d' % use_tc, worst)


# ---- the plans the sampler uses ----

@pytest.mark.parametrize('model', ['m1b', 'm2b', 'm3b', 'm4b', 'm5b'])
@pytest.mark.parametrize('n,D', [(37, 3), (128, 8), (700, 19), (5000, 49), (1300, 63)])
def test_default_chains_keep_a_tensor_core_pass(model, n, D):
    """Without a chain count, logdensity evaluates single-box-eligible sites with the most chains (<= 16) at
    which the sampler keeps the tensor-core pass; where no such count exists (m4b / m5b at D = 63: the cavity
    precision alone exceeds its share of shared memory) with 32 chains, on the wide pass."""
    site = site_of(model, n, D, seed=31)
    ctx = make_ctx(model, [site], use_tc=1)
    q = points(np.random.RandomState(2), ctx.num_params(0), 21, D)
    plan = check(ctx, 0, model, site, q, None)
    assert plan['use_tc'] == (2 if model in ('m4b', 'm5b') and D == 63 else 1), plan
    ctx.close()


@pytest.mark.parametrize('model,n,D,J,C,use_tc', [
    ('m1b', 300, 5, 1, 1, 0), ('m3b', 700, 5, 3, 12, 0), ('m1b', 7500, 5, 1, 17, 0), ('m1b', 500, 150, 1, 32, 0),
    ('m3b', 641, 8, 1, 3, 1), ('m1b', 641, 19, 1, 9, 1), ('m3b', 5000, 49, 1, 4, 1), ('m2b', 641, 63, 1, 16, 1),
    ('m4b', 300, 49, 1, 16, 1), ('m1b', 300, 70, 1, 17, 1), ('m4b', 700, 64, 1, 32, 1)])
def test_sampler_plan_matches_logdensity_plan(model, n, D, J, C, use_tc):
    """A short tilted_sample (iter 4) launches with the plan logdensity reports for the same chain count,
    including the fall-back from the tensor-core pass to SIMT when the chain vectors do not all fit in shared
    memory (m4b, D = 49, 16 chains)."""
    site = site_of(model, n, D, J, seed=800)
    ctx = make_ctx(model, [site, site], use_tc=use_tc)
    q = points(np.random.RandomState(8), ctx.num_params(0), C, D)
    check(ctx, 0, model, site, q, C)
    ld = ctx.last_plan()
    ctx.tilted_sample([3, 4], C, 4)
    smp = ctx.last_plan()
    assert smp['kernel'] == 1
    assert {k: v for k, v in smp.items() if k != 'kernel'} == {k: v for k, v in ld.items() if k != 'kernel'}
    ctx.close()


def test_every_arm_is_reached(monkeypatch):
    """The shapes of the tests above reach every arm of the plan: each padded chain count resident and
    streamed, NC > 1, tc::pass<4|8|16> at every ring depth 4..8, and several wide ring depths."""
    seen = set()
    for C in SIMT_CHAINS:
        for model, D, sites in simt_sites():
            ctx = make_ctx(model, sites, use_tc=0)
            for k in range(len(sites)):
                ctx.logdensity(k, np.zeros((1, ctx.num_params(k))), chains=C)
                pl = ctx.last_plan()
                seen.add(('simt', pl['chain_pad'], pl['resident']))
                if pl['NC'] > 1:
                    seen.add(('NC>1',))
            ctx.close()
    for model, D in TC_SHAPES:
        ctx = make_ctx(model, [site_of(model, 129, D, seed=1)], use_tc=1)
        for nst in TC_NST:
            monkeypatch.setenv('EPGPU_NST', str(nst))
            for C in TC_CHAINS:
                ctx.logdensity(0, np.zeros((1, ctx.num_params(0))), chains=C)
                pl = ctx.last_plan()
                if pl['use_tc'] == 1:
                    seen.add(('tc', pl['chain_pad'], pl['tc_nst']))
        ctx.close()
    monkeypatch.delenv('EPGPU_NST')
    wide = set()
    for model, D in WIDE_SHAPES:
        ctx = make_ctx(model, [site_of(model, 129, D, seed=1)], use_tc=1)
        ctx.logdensity(0, np.zeros((1, ctx.num_params(0))), chains=32)
        wide.add(ctx.last_plan()['tc_nst'])
        ctx.close()
    want = {('simt', cp, r) for cp in (4, 8, 16, 32) for r in (0, 1)} | {('NC>1',)}
    want |= {('tc', ncp, nst) for ncp in (4, 8, 16) for nst in TC_NST}
    assert want <= seen, sorted(want - seen)
    assert len(wide) >= 2, wide

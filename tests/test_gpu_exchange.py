"""The one-exchange update path of the C ABI (include/epgpu.h: epg_delta_sums_ex, the all-reduced EPG_DSUM,
epg_update_from_sums) on the real kernels, call for call against tests/fake_backend.OracleContext.

The multi-rank host logic is tested on CPU with the oracle stand-in (tests/test_distributed_gloo.py); that evidence
is only as good as the stand-in's likeness to the kernels.  Here both are driven with the same inputs through the
calls Master issues in one exchanged iteration (moments on two sub-ranges, a rejected site, the exchange, the damping
ladder with a non-pos.def. global matrix and a failing cavity, accept, global moments), and every return value and
every device array is compared after every call.  Where a call consumes the result of an earlier one, the stand-in is
given the kernel's copy, so each call is compared on identical inputs at its own tolerance."""
import numpy as np
import pytest

from conftest import relerr
import fake_backend as fb
from oracle import fakes

TOL_MOM = 1e-10        # moments, cavities, Fisher norms
TOL_SUM = 1e-12        # sums and updates

SITE3 = ('QI', 'QI2', 'DQI', 'CAVQ')
SITE2 = ('RI', 'RI2', 'DRI', 'CAVM', 'TMEAN')
GLOB = ('Q', 'R', 'PARTIAL', 'DSUM')
ARRAYS = SITE3 + SITE2 + GLOB


def test_array_ids_and_slots_match_the_c_abi():
    """the stand-in indexes the same device arrays and carries as many exchange slots as libepgpu"""
    from epstan import _lib
    names = ('Q', 'R', 'Q0', 'R0', 'QI', 'RI', 'QI2', 'RI2', 'DQI', 'DRI', 'CAVQ', 'CAVM', 'S', 'M', 'PARTIAL',
             'TMEAN', 'DSUM')
    assert [getattr(fb, n) for n in names] == [getattr(_lib, n) for n in names] == list(range(17))
    assert fb.XCHG_SLOTS == _lib.XCHG_SLOTS == 64


def _shape(name, K, d):
    if name in SITE3:
        return (d, d, K)
    if name in SITE2:
        return (d, K)
    return {'Q': (d, d), 'R': (d,), 'PARTIAL': (d * d + d + 1,), 'DSUM': (d * d + d + 2 + 64,)}[name]


def _get(ctx, name, K, d):
    from epstan import _lib
    return ctx.download(getattr(_lib, name), np.empty(_shape(name, K, d), order='F'))


def _site_relerr(a, b):
    """max over the sites (last axis) of relerr of that site"""
    a = a.reshape(-1, a.shape[-1])
    b = b.reshape(-1, b.shape[-1])
    den = np.max(np.abs(b), axis=0)
    num = np.max(np.abs(a - b), axis=0)
    return float(np.max(num / np.where(den > 0, den, 1.0)))


class Pair(object):
    """the real context and the stand-in, driven together"""

    def __init__(self, real, fake, K, d):
        self.real, self.fake, self.K, self.d = real, fake, K, d
        self.cav_ok = None                     # flags of the last cavity call (EPG_CAVM is defined there)

    def call(self, name, *args, **kw):
        a = getattr(self.real, name)(*args, **kw)
        b = getattr(self.fake, name)(*args, **kw)
        return a, b

    def check(self, step, tol=None):
        """compare every array; tol: name -> tolerance (default TOL_SUM; moment-type arrays TOL_MOM)"""
        K, d = self.K, self.d
        tol = dict(tol or {})
        out = {}
        for name in ARRAYS:
            a, b = _get(self.real, name, K, d), _get(self.fake, name, K, d)
            out[name] = a
            t = tol.get(name, TOL_MOM if name in ('DQI', 'DRI', 'TMEAN', 'CAVQ', 'CAVM') else TOL_SUM)
            if name == 'CAVM' and self.cav_ok is not None:
                a, b = a[:, self.cav_ok], b[:, self.cav_ok]
            if name == 'DSUM':
                dd = d * d + d
                assert relerr(a[:dd], b[:dd]) <= t, (step, name)
                assert abs(a[dd] - b[dd]) <= TOL_MOM * max(abs(b[dd]), 1e-300), (step, 'DSUM norms', a[dd], b[dd])
                assert np.array_equal(a[dd + 1:], b[dd + 1:]), (step, 'DSUM n_ok/slots')
                continue
            err = _site_relerr(a, b) if name in SITE3 + SITE2 else relerr(a, b)
            assert err <= t, (step, name, err)
        return out

    def sync_fake(self, names):
        """hand the stand-in the kernel's copy of arrays that the next calls consume"""
        from epstan import _lib
        for name in names:
            self.fake.upload(getattr(_lib, name), _get(self.real, name, self.K, self.d))


def _inputs(K, d, n, seed):
    """SPD global state whose site deltas (from the draws) shrink it: the ladder can reach a non-pos.def. global
    matrix; site f carries a large Qi (its cavity fails first), site c has a constant coordinate in its draws."""
    rng = np.random.RandomState(seed)
    Q0 = fakes.random_spd(rng, d) + 30.0 * np.eye(d)
    r0 = rng.standard_normal(d)
    Qi = np.stack([0.05 * fakes.random_spd(rng, d) for _ in range(K)], axis=2)
    f, c = 0, K - 1
    Qi[:, :, f] = 15.0 * np.eye(d)
    ri = 0.05 * rng.standard_normal((d, K))
    scale = np.exp(0.3 * rng.standard_normal((K, d, 1)))
    draws = rng.standard_normal((K, d, n)) * scale * 0.3 + 3.0 * rng.standard_normal((K, d, 1))
    draws[c, d // 2, :] = 2.0          # exactly representable: the centred coordinate is exactly 0
    return dict(Q0=Q0, r0=r0, Qi=np.asfortranarray(Qi), ri=np.asfortranarray(ri),
                Q=Q0 + Qi.sum(axis=2), r=r0 + ri.sum(axis=1), draws=draws, f=f, c=c)


def _min_eig_rel(A, ref):
    return np.linalg.eigvalsh(A)[..., 0] / ref


def _ladder(inp, dQ, margin=1e-3):
    """damping values: (global not pos.def., only site f's cavity fails, all pos.def.), each at least `margin`
    (relative to |Q_prev|) away from every pos.def. boundary"""
    Qp, Qi, f = inp['Q'], inp['Qi'], inp['f']
    ref = np.linalg.norm(Qp, 2)
    SdQ = dQ.sum(axis=2)
    L = np.linalg.cholesky(Qp)
    Li = np.linalg.inv(L)
    lam = np.linalg.eigvalsh(-Li @ SdQ @ Li.T)[-1]
    assert lam > 0, "the summed deltas never make the global matrix indefinite"
    df_g = 1.0 / lam

    def state(df):
        g = _min_eig_rel(Qp + df * SdQ, ref)
        cav = _min_eig_rel(np.moveaxis((Qp + df * SdQ)[:, :, None] - Qi - df * dQ, 2, 0), ref)
        return g, cav

    big = 1.5 * df_g
    assert state(big)[0] < -margin
    grid = df_g * np.linspace(0.02, 0.98, 49)
    mid, small = [], []
    for df in grid:
        g, cav = state(df)
        if g < margin:
            continue
        others = np.delete(cav, f)
        if np.all(np.abs(cav) > margin) and np.all(others > 0):
            (small if cav[f] > 0 else mid).append(df)
    assert mid and small, "no damping window with exactly one failing cavity"
    return [big, mid[len(mid) // 2], small[len(small) // 2]]


def drive(real, fake, K, d, n, seed=7):
    """one exchanged iteration of Master, call for call; returns the damping values used"""
    from epstan import _lib
    inp = _inputs(K, d, n, seed)
    P = Pair(real, fake, K, d)
    P.call('init_state', K, d)
    for aid, v in ((_lib.Q0, inp['Q0']), (_lib.R0, inp['r0']), (_lib.Q, inp['Q']), (_lib.R, inp['r']),
                   (_lib.QI, inp['Qi']), (_lib.RI, inp['ri'])):
        P.call('upload', aid, v)
    P.call('set_draws', inp['draws'], n)
    P.check('set_draws', tol={n_: 0.0 for n_ in ARRAYS})
    f, c = inp['f'], inp['c']

    # moments on [0, j) with the sample estimate and on [j, K) with olse (k0 > 0)
    j = max(1, K // 2)
    for k0, k1, mode in ((0, j, 'sample'), (j, K, 'olse')):
        (fa, na), (fo, no) = P.call('moments', n, mode, k0, k1)
        assert np.array_equal(fa, fo) and na == no, (mode, fa, fo)
        assert na == (k1 - k0) - (1 if k0 <= c < k1 else 0)
        P.check('moments ' + mode)
    got = P.check('moments')
    assert not got['DQI'][:, :, c].any() and not got['DRI'][:, c].any()      # failed estimate: zero deltas
    P.sync_fake(('DQI', 'DRI', 'TMEAN'))

    P.call('fail_sites', [f])
    got = P.check('fail_sites')
    assert not got['DQI'][:, :, f].any() and not got['DRI'][:, f].any()
    n_ok = K - 2

    # the exchange: without norms and a short slot vector, then as Master does with norms and all 64 slots
    rng = np.random.RandomState(seed + 1)
    short = np.arange(1, 8) * 0.5
    P.call('delta_sums', with_norms=False, slots=short)
    got = P.check('delta_sums short')
    dd = d * d + d
    assert got['DSUM'][dd] == 0.0 and got['DSUM'][dd + 1] == n_ok
    assert np.array_equal(got['DSUM'][dd + 2:dd + 9], short) and not got['DSUM'][dd + 9:].any()
    full = rng.standard_normal(64)
    P.call('delta_sums', with_norms=True, slots=full)
    got = P.check('delta_sums full')
    assert np.array_equal(got['DSUM'][dd + 2:], full)
    (S2a, na, sa), (S2b, nb, sb) = P.call('read_exchange')
    assert na == nb == n_ok and np.array_equal(sa, full) and np.array_equal(sb, full)
    assert abs(S2a - S2b) <= TOL_MOM * S2b and S2a > 0
    snr_a, snr_b = P.call('delta_snr')
    assert snr_a[2] == snr_b[2] == n_ok and snr_a[1] == S2a
    assert abs(snr_a[0] - snr_b[0]) <= TOL_MOM * snr_b[0] and abs(snr_a[1] - snr_b[1]) <= TOL_MOM * snr_b[1]
    P.check('delta_snr')

    # the damping ladder of Master._update_without_exchange
    dQ = got['DQI']
    SdQ, Sdr = dQ.sum(axis=2), got['DRI'].sum(axis=1)
    dfs = _ladder(inp, dQ)
    outcomes = []
    for i, df in enumerate(dfs):
        P.call('update_partial', df)
        got = P.check('update_partial %g' % df)
        a_pd, b_pd = P.call('update_finish')           # (Q from the local Qi2: the single-rank proposal)
        assert a_pd == b_pd
        Q_loc, r_loc = _get(real, 'Q', K, d), _get(real, 'R', K, d)
        P.call('update_from_sums', df)
        got = P.check('update_from_sums %g' % df)
        # built on the (Q, r) of delta_sums, also after a failed attempt overwrote Q
        part = np.concatenate([(inp['Q'] - inp['Q0'] + df * SdQ).ravel(order='F'), inp['r'] - inp['r0'] + df * Sdr])
        assert relerr(got['PARTIAL'][:d * d + d], part) <= TOL_SUM, ('partial from sums', df)
        pd_a, pd_b = P.call('update_finish')
        assert pd_a == pd_b == a_pd
        got = P.check('update_finish %g' % df)
        assert relerr(got['Q'], Q_loc) <= 1e-13 and relerr(got['R'], r_loc) <= 1e-13
        if not pd_a:
            outcomes.append('global')
            # the statistics keep the metric of the snapshot, not of the overwritten Q
            again = P.call('delta_snr')
            assert again[0] == snr_a and again[1][0] == pytest.approx(snr_b[0], rel=1e-14)
            continue
        (fa, oka), (fo, oko) = P.call('cavity', proposal=True)
        assert np.array_equal(fa, fo) and oka == oko
        P.cav_ok = fa
        P.check('cavity %g' % df)
        outcomes.append('ok' if oka else tuple(np.nonzero(~fa)[0]))
    assert outcomes == ['global', (f,), 'ok'], outcomes

    P.call('accept')
    P.check('accept')
    m_a, S_a = np.empty(d), np.empty((d, d), order='F')
    m_b, S_b = np.empty(d), np.empty((d, d), order='F')
    real.global_moments(m_a, S_a)
    fake.global_moments(m_b, S_b)
    assert relerr(m_a, m_b) <= TOL_MOM and relerr(S_a, S_b) <= TOL_MOM
    P.check('global_moments')

    # epg_cavity writes the site flags that epg_delta_sums counts (include/epgpu.h)
    (fa, _), (fo, _) = P.call('cavity', proposal=False)
    assert fa.all() and fo.all()
    P.call('delta_sums')
    got = P.check('delta_sums after cavity')
    assert got['DSUM'][dd + 1] == K
    return dfs


@pytest.mark.gpu
@pytest.mark.parametrize('K,d,n', [(3, 5, 40), (64, 20, 400), (1024, 50, 200), (8, 200, 2400)])
def test_exchange_calls_match_oracle_context(K, d, n):
    from epstan import _lib
    real = _lib.Context(0)
    try:
        drive(real, fb.OracleContext(), K, d, n)
    finally:
        real.close()


@pytest.mark.gpu
@pytest.mark.parametrize('K2,d2', [(8, 6), (5, 4)])
def test_init_state_invalidates_the_exchange(K2, d2):
    """a new state has no delta sums: update_from_sums / delta_snr must refuse instead of building on the
    previous state's snapshot (same or smaller shape only: a larger one would be read out of bounds)"""
    from epstan import _lib
    real = _lib.Context(0)
    try:
        for ctx in (real, fb.OracleContext()):
            K, d = 8, 6
            inp = _inputs(K, d, 40, 3)
            ctx.init_state(K, d)
            for aid, v in ((_lib.Q0, inp['Q0']), (_lib.R0, inp['r0']), (_lib.Q, inp['Q']), (_lib.R, inp['r']),
                           (_lib.QI, inp['Qi']), (_lib.RI, inp['ri'])):
                ctx.upload(aid, v)
            ctx.set_draws(inp['draws'], 40)
            ctx.moments(40, 'sample')
            ctx.delta_sums()
            ctx.update_from_sums(0.1)
            ctx.delta_snr()
            ctx.init_state(K2, d2)
            with pytest.raises(_lib.EpgError):
                ctx.update_from_sums(0.1)
            with pytest.raises(_lib.EpgError):
                ctx.delta_snr()
            # fresh sums of the new state make both usable again
            Q = np.eye(d2) * 2.0
            ctx.upload(_lib.Q, Q)
            ctx.upload(_lib.Q0, np.eye(d2))
            ctx.delta_sums()
            ctx.update_from_sums(0.5)
            assert ctx.update_finish()
            out = ctx.download(_lib.Q, np.empty((d2, d2), order='F'))
            assert np.array_equal(out, Q)
            assert ctx.delta_snr() == (0.0, 0.0, 0)        # (epg_init_state clears the site flags)
    finally:
        real.close()

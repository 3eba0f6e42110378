"""The tests-side oracle of PyStan's remaining sampling settings (tests/nuts_control.py) and the host-side
conversion of a dict / list / function `init` into the sampler's starting points (epstan.util.init_values)."""
import numpy as np
import pytest

from oracle import nuts
import nuts_control


def _direct_window_ends(W, init, term, window):
    """windowed_adaptation restated directly: set_window_params, then the window ends compute_next_window
    produces from the end of the first window"""
    if W < 20:
        return []
    if init + window + term > W:
        init, term = int(0.15 * W), int(0.1 * W)
        window = W - (init + term)
    last = W - term - 1
    ends = []
    size, nxt = window, init + window - 1
    for counter in range(W):
        if counter == nxt:
            ends.append(counter)
            if nxt != last:
                size *= 2
                nxt = counter + size
                if nxt != last and nxt + 2 * size >= W - term:
                    nxt = last
    return ends


@pytest.mark.parametrize('W,init,term,window', [
    (1000, 75, 50, 25), (500, 75, 50, 25), (150, 75, 50, 25), (149, 75, 50, 25), (100, 75, 50, 25),
    (19, 75, 50, 25), (20, 75, 50, 25), (10, 0, 0, 1), (100, 15, 10, 75), (100, 15, 10, 74),
    (100, 200, 200, 200), (300, 0, 50, 25), (300, 100, 0, 25), (300, 10, 10, 1), (1000, 0, 0, 1),
    (400, 50, 50, 300), (64, 0, 0, 64)])
def test_window_ends_follow_compute_next_window(W, init, term, window):
    assert nuts_control.window_ends(W, init, term, window) == _direct_window_ends(W, init, term, window)


def test_default_window_ends_match_the_diag_e_oracle():
    for W in (30, 100, 149, 150, 500, 1000):
        w = nuts.VarWindows(W, 1)
        ends = []
        for it in range(W):
            if w.learn(np.zeros(1) + it % 3) is not None:
                ends.append(it)
        assert nuts_control.window_ends(W) == ends, W


def _gauss(S):
    P = np.linalg.inv(S)
    return lambda q: (-0.5 * q @ P @ q, -P @ q)


S3 = np.diag([1.0, 4.0, 0.25])


def test_adaptation_off_warmup_is_discarded_transitions():
    I, W = 120, 40
    a = nuts_control.sample(_gauss(S3), 3, 2, I, W, seed=5, adapt_engaged=False, stepsize=0.4)
    b = nuts_control.sample(_gauss(S3), 3, 2, I, 0, seed=5, adapt_engaged=False, stepsize=0.4)
    for ca, cb in zip(a['per_chain'], b['per_chain']):
        assert np.array_equal(ca, cb[W:])
    assert np.all(a['eps'] == 0.4) and all(np.array_equal(m, np.ones(3)) for m in a['minv'])


def test_thinned_draws_are_every_thin_th_draw():
    for thin in (2, 3, 7):
        a = nuts_control.sample(_gauss(S3), 3, 2, 200, 100, seed=2, thin=thin)
        b = nuts_control.sample(_gauss(S3), 3, 2, 200, 100, seed=2)
        for ca, cb in zip(a['per_chain'], b['per_chain']):
            assert ca.shape[0] == -(-100 // thin)
            assert np.array_equal(ca, cb[::thin])
        assert all(np.array_equal(la, ca[-1]) for la, ca in zip(a['last'], a['per_chain']))


def test_jittered_step_sizes_average_to_the_nominal():
    j, eps = 0.5, 0.7
    r = nuts_control.sample(_gauss(S3), 3, 4, 1500, 0, seed=3, adapt_engaged=False, stepsize=eps, jitter=j)
    e = np.concatenate(r['eps_used'])
    assert np.all(np.abs(e / eps - 1.0) <= j)
    se = eps * j / np.sqrt(3.0) / np.sqrt(len(e))          # sd of eps (1 + j U(-1, 1)) over the saved draws
    assert abs(e.mean() - eps) < 4 * se, (e.mean(), se)
    assert e.std() > 0.8 * eps * j / np.sqrt(3.0)
    # the jittered chain still targets the Gaussian
    ess, mcse = nuts.ess_mcse(r['per_chain'])
    assert np.all(np.abs(r['draws'].mean(axis=0)) < 4 * mcse)


def test_given_inits_and_radius():
    q0 = np.array([0.5, np.nan, -0.25])
    r = nuts_control.sample_chain(_gauss(S3), 3, 1, 0, np.random.RandomState(0), q0=q0, init_r=0.1,
                                  adapt_engaged=False, stepsize=1e-6, max_depth=1)
    assert abs(r['draws'][0, 0] - 0.5) < 1e-3 and abs(r['draws'][0, 2] + 0.25) < 1e-3
    assert abs(r['draws'][0, 1]) < 0.1 + 1e-3
    # an init given in full with a non-finite density has one attempt
    bad = lambda q: (np.nan, np.zeros_like(q))
    with pytest.raises(RuntimeError):
        nuts_control.sample_chain(bad, 2, 10, 5, np.random.RandomState(0), q0=np.zeros(2))


# ---- epstan.util.init_values ----

def _iv(*a, **k):
    from epstan import util
    return util.init_values(*a, **k)


def test_init_values_dict_list_callable():
    sites = [('m1b', 3, 1)]                                       # p = 4 + 1
    phi = np.array([0.1, 0.2, 0.3, 0.4])
    q = _iv({'phi': phi, 'eta': [0.5]}, 2, sites)
    assert q.shape == (1, 2, 5)
    assert np.array_equal(q[0, 0], np.r_[phi, 0.5]) and np.array_equal(q[0, 1], q[0, 0])
    q = _iv({'eta': 0.5, 'bogus': 1.0, 'etb': np.ones(3)}, 1, sites)     # scalar eta at J = 1; m1b has no etb
    assert np.all(np.isnan(q[0, 0, :4])) and q[0, 0, 4] == 0.5
    q = _iv([{'phi': phi}, {}], 2, sites)
    assert np.array_equal(q[0, 0, :4], phi) and np.all(np.isnan(q[0, 0, 4:])) and np.all(np.isnan(q[0, 1]))
    q = _iv(lambda chain_id: {'phi': phi + chain_id}, 3, sites)
    for c in range(3):
        assert np.array_equal(q[0, c, :4], phi + c)
    q = _iv(lambda: {'phi': phi}, 2, sites)
    assert np.array_equal(q[0, 1, :4], phi)
    with pytest.raises(ValueError):
        _iv([{}], 2, sites)
    with pytest.raises(ValueError):
        _iv('random', 2, sites)


def test_init_values_layouts():
    # m2b: phi (2), eta (J), etb (D) one vector per site; m4b multi-group sites with different J: etb (J, D)
    q = _iv({'phi': [1.0, 2.0], 'eta': [3.0, 4.0, 5.0], 'etb': [6.0, 7.0]}, 1, [('m2b', 2, 3)])
    assert np.array_equal(q[0, 0], [1, 2, 3, 4, 5, 6, 7])
    sites = [('m4b', 2, 2), ('m4b', 2, 3)]                        # p = 6 + 2 + 4 and 6 + 3 + 6
    etb2 = np.arange(4.0).reshape(2, 2)
    q = _iv(lambda chain_id: {'etb': etb2} if chain_id == 0 else {}, 2, sites[:1])
    assert q.shape == (1, 2, 12)
    assert np.array_equal(q[0, 0, 8:], [0, 1, 2, 3]) and np.all(np.isnan(q[0, 0, :8])) and np.all(np.isnan(q[0, 1]))
    with pytest.raises(ValueError, match="site 1, parameter 'etb'"):
        _iv({'etb': etb2}, 1, sites)                            # (2, 2) does not fit J = 3
    q = _iv({'eta': [1.0, 2.0]}, 1, sites[:1], Pmax=20)
    assert q.shape == (1, 1, 20) and np.array_equal(q[0, 0, 6:8], [1, 2]) and np.all(np.isnan(q[0, 0, 8:]))
    with pytest.raises(ValueError, match="parameter 'phi'"):
        _iv({'phi': np.zeros(5)}, 1, sites[:1])
    with pytest.raises(ValueError, match="parameter 'phi'"):
        _iv({'phi': 0.0}, 1, [('m1b', 3, 1)])                     # (no scalar phi at J = 1)
    # m3b single group: etb (1, D) or (D,)
    a = _iv({'etb': [[1.0, 2.0]]}, 1, [('m3b', 2, 1)])
    b = _iv({'etb': [1.0, 2.0]}, 1, [('m3b', 2, 1)])
    assert np.array_equal(a, b, equal_nan=True) and np.array_equal(a[0, 0, 4:], [1, 2])

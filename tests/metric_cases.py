"""Fixed-seed diag_e sampling runs on every launch plan of the sampler, reduced to SHA-256 digests.

tests/test_gpu_sampler_metric.py compares the digests with the ones recorded before the sampler learnt the
dense_e and unit_e metrics (tools/metric_digests.py records them); both use only calls the earlier library
had, so the same code runs against either build.
"""
import hashlib

import numpy as np

import synth


def make_ctx(_lib, model, sites, use_tc=None):
    K = len(sites)
    d = sites[0]['d']
    D = sites[0]['X'].shape[1]
    ctx = _lib.Context(0)
    ctx.init_state(K, d)
    k_lim = np.concatenate(([0], np.cumsum([s['X'].shape[0] for s in sites])))
    X = np.concatenate([s['X'] for s in sites])
    y = np.concatenate([s['y'] for s in sites])
    multi = any(s['J'] > 1 for s in sites)
    ctx.upload_sites(_lib.MODEL_IDS[model], D, k_lim, X, y,
                     np.concatenate([s['j_ind'] for s in sites]) if multi else None,
                     [s['J'] for s in sites] if multi else None)
    ctx.upload(_lib.CAVQ, np.asfortranarray(np.stack([s['Omega'] for s in sites], axis=2)))
    ctx.upload(_lib.CAVM, np.asfortranarray(np.stack([s['mu'] for s in sites], axis=1)))
    if use_tc is not None:
        ctx.set_option('use_tc', use_tc)
    return ctx


# name: (model, J, n, D, sites, use_tc, pingpong, chains, iter, warmup)
CASES = {
    'simt_single': ('m1b', 1, 700, 19, 2, 0, 0, 4, 200, 100),
    'simt_multi': ('m1b', 4, 400, 5, 2, 0, 0, 8, 200, 100),
    'tc_4': ('m1b', 1, 700, 19, 2, 1, 0, 4, 200, 100),
    'tc_16': ('m1b', 1, 700, 19, 2, 1, 0, 16, 200, 100),
    'wide_70': ('m1b', 1, 300, 70, 2, 1, 0, 32, 120, 60),
    'pingpong': ('m1b', 1, 300, 8, 5, 1, 2, 8, 200, 100),
}


def case_sites(name):
    model, J, n, D, ns = CASES[name][:5]
    sites = [synth.make_site(model, n + 31 * k, D, J, seed=70 + k) for k in range(ns)]
    if D > 64:                                          # (keep the cavity term moderate at large d)
        for s in sites:
            s['Omega'] = s['Omega'] / max(1.0, np.abs(s['Omega']).max()) + np.eye(s['d'])
    return sites


def digest(ctx, n, out):
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(ctx.get_draws(n)).tobytes())
    for a in out[:3]:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def run_case(_lib, name, **kw):
    """-> (digest of the run, plan) and, for 'tc_4', also a second run with carried adaptation
    (name + '_carried').  kw goes to tilted_sample (e.g. metric=...)."""
    model, J, n, D, ns, use_tc, pp, C, it, wu = CASES[name]
    ctx = make_ctx(_lib, model, case_sites(name), use_tc=use_tc)
    ctx.set_option('pingpong', pp)
    seeds = [1000 + 7 * k for k in range(ns)]
    res = {}
    out = ctx.tilted_sample(seeds, C, it, wu, **kw)
    res[name] = (digest(ctx, C * (it - wu), out), ctx.last_plan())
    if name == 'tc_4':
        out = ctx.tilted_sample([s + 1 for s in seeds], C, it, wu, 2, **kw)
        res[name + '_carried'] = (digest(ctx, C * (it - wu), out), ctx.last_plan())
    ctx.close()
    return res

"""Cached fp64 oracle dense_e NUTS runs (tests/nuts_metric.py) on the synthetic sites of the GPU sampler tests.

    python tests/oracle_refs_metric.py        # rewrites tests/golden/nuts_metric_ref.npz

Each entry holds the mean step size and the gradient evaluations per draw of 4 chains x 1000 iterations
(500 warm-up) of the oracle dense_e sampler on synth.make_site(model, n, D, J, seed=21), the site of
test_gpu_sampler.py::test_sampler_vs_oracle_nuts.  The moments of that target are the cached diag_e summaries
of tests/oracle_refs.py: the metric does not change the distribution.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import nuts_metric  # noqa: E402
import synth  # noqa: E402

PATH = os.path.join(HERE, 'golden', 'nuts_metric_ref.npz')
# (model, J, n, D)
SHAPES = [('m1b', 1, 300, 4), ('m1b', 5, 250, 6), ('m4b', 2, 300, 3), ('m5b', 1, 300, 3)]
CHAINS, ITER, WARM, SEED = 4, 1000, 500, 3


def key(model, J, n, D):
    return 'dense_%s_%d_%d_%d_' % (model, J, n, D)


def compute(model, J, n, D, chains=CHAINS, n_iter=ITER, n_warmup=WARM, seed=SEED):
    site = synth.make_site(model, n, D, J, seed=21)
    td = synth.oracle_density(model, site)
    ref = nuts_metric.sample(lambda q: tuple(v[0] for v in td.lp_grad(q[None])), td.p, chains=chains,
                             n_iter=n_iter, n_warmup=n_warmup, seed=seed, metric='dense_e')
    return dict(stepsize=np.float64(ref['stepsize']),
                evals_per_draw=np.float64(ref['n_grad'] / float(chains * n_iter)))


def reference(model, J, n, D):
    k = key(model, J, n, D)
    c = dict(np.load(PATH)) if os.path.exists(PATH) else {}
    if k + 'stepsize' in c:
        return {f: c[k + f] for f in ('stepsize', 'evals_per_draw')}
    return compute(model, J, n, D)


def main():
    out = {}
    for shp in SHAPES:
        r = compute(*shp)
        print(shp, {f: float(v) for f, v in r.items()}, flush=True)
        for f, v in r.items():
            out[key(*shp) + f] = v
    np.savez(PATH, **out)


if __name__ == '__main__':
    main()

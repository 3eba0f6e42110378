"""Cached tests-side oracle runs (tests/nuts_control.py) for tests/test_gpu_sampler_control.py.

    python tests/oracle_refs_control.py        # rewrites tests/golden/nuts_control_ref.npz

Each entry is the median over chains of the adapted nominal step size of CHAINS x ITER iterations (WARM warm-up)
of the oracle on synth.make_site(*SITE), with the dual-averaging constants of SETTINGS[name].
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import nuts_control  # noqa: E402
import synth  # noqa: E402

PATH = os.path.join(HERE, 'golden', 'nuts_control_ref.npz')
SITE = ('m1b', 300, 4, 1, 21)                 # synth.make_site(model, n, D, J, seed)
CHAINS, ITER, WARM, SEED = 4, 600, 300, 3
SETTINGS = {'default': dict(gamma=0.05, kappa=0.75, t0=10.0),
            'custom': dict(gamma=0.1, kappa=0.9, t0=5.0)}


def compute(name):
    site = synth.make_site(*SITE)
    td = synth.oracle_density(SITE[0], site)
    r = nuts_control.sample(lambda q: tuple(v[0] for v in td.lp_grad(q[None])), td.p, chains=CHAINS,
                            n_iter=ITER, n_warmup=WARM, seed=SEED, **SETTINGS[name])
    return np.float64(np.median(r['eps']))


def reference(name):
    c = dict(np.load(PATH)) if os.path.exists(PATH) else {}
    return float(c[name]) if name in c else float(compute(name))


def main():
    out = {}
    for name in SETTINGS:
        out[name] = compute(name)
        print(name, float(out[name]), flush=True)
    np.savez(PATH, **out)


if __name__ == '__main__':
    main()

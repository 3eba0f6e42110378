"""Cached tests-side oracle runs (tests/nuts_diag.py) for tests/test_gpu_hmc_diagnostics.py.

    python tests/oracle_refs_diag.py        # rewrites tests/golden/nuts_diag_ref.npz

For each entry of RUNS (a site of tests/metric_cases.py, chains, iter, warm-up) the oracle samples the first site
of the case with Stan's default adaptation; stored are the mean over the saved post-warm-up transitions of all
chains of accept_stat__, treedepth__, n_leapfrog__ and energy__, and the mean over chains of E-BFMI, each with
its Monte Carlo standard error, sd / sqrt(chains) of the per-chain values (each chain adapts its own step size
and metric: the chains are the independent replicates).

TRANSIENT: from q = 0, without adaptation, at a fixed step size large enough for a visible energy error, the
mean and its standard error over chains of energy__ of each of the first transitions, and of the Hamiltonian H0
each transition starts from.  energy__ is H of the SELECTED sample: its mean differs from that of H0 by many
standard errors there (at stationarity the two would agree), so a comparison of energy__ with this reference
tells the selected sample's H from the initial one's.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

import metric_cases  # noqa: E402
import nuts_diag  # noqa: E402
import synth  # noqa: E402

PATH = os.path.join(HERE, 'golden', 'nuts_diag_ref.npz')
# name: (metric_cases case, chains, iter, warm-up)
RUNS = {'narrow': ('tc_16', 16, 400, 200),
        'wide': ('wide_70', 32, 200, 100)}
STATS = ('accept_stat__', 'treedepth__', 'n_leapfrog__', 'energy__')
SEED = 11
# (metric_cases case, chains, transitions, fixed step size, max_treedepth)
TRANSIENT = ('tc_16', 128, 3, 0.1, 6)


def summarise(records, n_warm):
    """{stat: (mean, mcse)} of per-chain record arrays [n_rec, 6] (the first n_warm of each are warm-up)"""
    post = [r[w:] for r, w in zip(records, n_warm)]
    per_chain = {s: np.array([p[:, nuts_diag.FIELDS.index(s)].mean() for p in post]) for s in STATS}
    per_chain['ebfmi'] = np.array([nuts_diag.ebfmi(p[:, 5]) for p in post])
    return {s: (float(v.mean()), float(v.std(ddof=1) / np.sqrt(len(v)))) for s, v in per_chain.items()}


def compute(name):
    case, chains, n_iter, warm = RUNS[name]
    model = metric_cases.CASES[case][0]
    site = metric_cases.case_sites(case)[0]
    td = synth.oracle_density(model, site)
    res = nuts_diag.sample(lambda q: tuple(v[0] for v in td.lp_grad(q[None])), td.p, chains=chains,
                           n_iter=n_iter, n_warmup=warm, seed=SEED)
    return summarise([r['records'] for r in res], [r['n_warm'] for r in res])


def compute_transient():
    case, chains, n_iter, eps, depth = TRANSIENT
    model = metric_cases.CASES[case][0]
    site = metric_cases.case_sites(case)[0]
    td = synth.oracle_density(model, site)
    res = nuts_diag.sample(lambda q: tuple(v[0] for v in td.lp_grad(q[None])), td.p, chains=chains,
                           n_iter=n_iter, n_warmup=0, seed=SEED, stepsize=eps, adapt_engaged=False,
                           max_depth=depth, q0=np.zeros(td.p))
    out = {}
    for key, v in (('energy', np.array([r['records'][:, 5] for r in res])), ('H0', np.array([r['H0'] for r in res]))):
        out['transient/' + key] = np.stack([v.mean(axis=0), v.std(axis=0, ddof=1) / np.sqrt(chains)], axis=1)
    return out


def transient_reference():
    """{'energy', 'H0'}: [transitions, 2] arrays of (mean, standard error) of TRANSIENT, from the cache"""
    c = np.load(PATH)
    return {k: c['transient/' + k] for k in ('energy', 'H0')}


def reference(name):
    """{stat: (mean, mcse)} of RUNS[name], from the cache"""
    c = np.load(PATH)
    return {s: tuple(float(v) for v in c[name + '/' + s]) for s in STATS + ('ebfmi',)}


def main():
    out = {}
    for name in RUNS:
        for s, v in compute(name).items():
            out[name + '/' + s] = np.array(v)
            print(name, s, v, flush=True)
    out.update(compute_transient())
    print('transient', out['transient/energy'].tolist(), out['transient/H0'].tolist(), flush=True)
    np.savez(PATH, **out)


if __name__ == '__main__':
    main()

"""diag_e against dense_e in EP iterations through Master (adapt_prev on), alternated in one process.

    python tools/metric_workload.py [--iters 4] [--reps 2] [--problems cfg3,cfg4s] [--out DIR]

Problems: cfg3 = bench.simulate_problem('m1b', 64, 2000, 19), 8 chains x 200 iterations; cfg4s = a 148-site
slice of config 4, simulate_problem('m3b', 148, 5000, 49), 4 chains x 200 iterations.  For every problem and
repetition, two Masters on the same data (one per metric) advance one EP iteration at a time, alternately.
The first iteration of each is warm-up (module load, first allocation) and is reported but not summarised.

Per iteration and metric: sampler device seconds (Master's sampling time), leapfrogs per retained draw, mean
step size, median / max split-Rhat of phi over the sites, median ESS/s of phi (oracle.nuts.ess_mcse on the
draw buffer, per site, over the sampler seconds) and the chain-phase / likelihood-pass cycles per tick
(EPGPU_TRACE).  Prints one JSON line per iteration and a summary table (median and spread over the measured
iterations and repetitions); the card's name and power limit are read in the same process.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'ep-stan_b200')]

PROBLEMS = {'cfg3': ('m1b', 64, 2000, 19, 8, 200), 'cfg4s': ('m3b', 148, 5000, 49, 4, 200)}
TRACE = re.compile(r'cycles/tick chain (\d+) lik (\d+)')


def card():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:          # (reported, not fatal)
        return 'unknown (%s)' % e


class StderrCapture(object):
    """captures what the library writes to file descriptor 2 (EPGPU_TRACE lines)"""

    def __enter__(self):
        sys.stderr.flush()
        self.f = tempfile.TemporaryFile(mode='w+')
        self.saved = os.dup(2)
        os.dup2(self.f.fileno(), 2)
        return self

    def __exit__(self, *exc):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.f.seek(0)
        self.text = self.f.read()
        self.f.close()


def one_iteration(m, metric, it, C, siter):
    from oracle import nuts
    ctx = m._shard.ctx
    l0 = m.n_leapfrog_total
    with StderrCapture() as cap:
        info, _, (st, ms, mr, _) = m.run(1, verbose=False, seed=4321 + m.iter, return_analytics=True)
    if info != 0:
        raise RuntimeError('EP stopped (info=%d) with metric %s' % (info, metric))
    per = siter - siter // 2
    n = C * per
    draws = ctx.get_draws(n)                                # (K, d, n)
    rh, ess = [], []
    for k in range(draws.shape[0]):
        chains = [draws[k][:, c * per:(c + 1) * per].T for c in range(C)]
        rh.append(np.max(nuts.split_rhat(chains)))
        ess.append(np.median(nuts.ess_mcse(chains)[0]))
    tr = [tuple(map(float, t)) for t in TRACE.findall(cap.text)]
    secs = float(st[0])
    return dict(metric=metric, iter=it, sampler_s=secs,
                leapfrog_per_draw=(m.n_leapfrog_total - l0) / float(draws.shape[0] * n),     # (warm-up included)
                mean_stepsize=float(ms[0]), rhat_median=float(np.median(rh)), rhat_max=float(np.max(rh)),
                ess_per_s_median=float(np.median(ess)) / secs,
                chain_cycles_per_tick=tr[-1][0] if tr else None, lik_cycles_per_tick=tr[-1][1] if tr else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=4)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--problems', default='cfg3,cfg4s')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    os.environ['EPGPU_TRACE'] = '1'
    import bench
    import epstan.method as method
    print(json.dumps({'card': card()}), flush=True)
    rows = []
    for name in args.problems.split(','):
        model, K, n_k, D, C, siter = PROBLEMS[name]
        X, y, prior = bench.simulate_problem(model, K, n_k, D)
        for rep in range(args.reps):
            ms = {met: method.Master('experiment/models/%s_sg' % model, X, y, site_sizes=np.full(K, n_k),
                                     prior=prior, chains=C, iter=siter, df0=bench.default_df0(K),
                                     control={'metric': met})
                  for met in ('diag_e', 'dense_e')}
            for it in range(args.iters + 1):
                for met in (('diag_e', 'dense_e') if (it + rep) % 2 == 0 else ('dense_e', 'diag_e')):
                    r = one_iteration(ms[met], met, it, C, siter)
                    r.update(problem=name, rep=rep, warm=it == 0)
                    rows.append(r)
                    print(json.dumps(r), flush=True)
            for m in ms.values():
                m._shard.ctx.close()
    keys = ['sampler_s', 'leapfrog_per_draw', 'mean_stepsize', 'rhat_median', 'rhat_max', 'ess_per_s_median',
            'chain_cycles_per_tick', 'lik_cycles_per_tick']
    print('\n| problem | metric | ' + ' | '.join(keys) + ' |')
    print('|---|---|' + '---|' * len(keys))
    for name in args.problems.split(','):
        for met in ('diag_e', 'dense_e'):
            sel = [r for r in rows if r['problem'] == name and r['metric'] == met and not r['warm']]
            cells = []
            for k in keys:
                v = np.array([r[k] for r in sel if r[k] is not None], dtype=float)
                cells.append('%.4g (%.4g–%.4g)' % (np.median(v), v.min(), v.max()) if v.size else 'not measured')
            print('| %s | %s | %s |' % (name, met, ' | '.join(cells)))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, 'metric_workload.json'), 'w') as f:
            json.dump(rows, f, indent=1)


if __name__ == '__main__':
    main()

"""Cost of recording every transition (option "sampler_params") on a bench workload.

    python tools/sampler_params_cost.py cfg4 3      # workload, EP iterations per arm and round

Runs Master.run on the workload with save_sampler_params False and True, alternating (two rounds, after one
untimed warm-up run of each), and prints the wall time per EP iteration of each run and that the two arms
computed the same Q and r.
"""
import sys
import time

sys.path.insert(0, '.'); sys.path.insert(0, 'ep-stan_b200')
import numpy as np  # noqa: E402
import bench  # noqa: E402
import epstan.method as method  # noqa: E402

work = sys.argv[1] if len(sys.argv) > 1 else 'cfg4'
niter = int(sys.argv[2]) if len(sys.argv) > 2 else 3
model, K, n_k, D, chains, siter = bench.WORKLOADS[work]
X, y, prior = bench.build_problem(model, K, n_k, D, 0, K)


def run(save):
    m = method.Master('experiment/models/%s_sg' % model, X, y, site_sizes=np.full(K, n_k), prior=prior,
                      chains=chains, iter=siter, df0=bench.default_df0(K), save_sampler_params=save)
    m._shard.ctx.sync()
    t0 = time.perf_counter()
    m.run(niter, calc_moments=False, verbose=False, seed=1)
    m._shard.ctx.sync()
    dt = (time.perf_counter() - t0) / niter
    out = (m.Q.copy(), m.r.copy())
    del m
    return dt, out


run(False), run(True)                     # warm-up
res = {False: [], True: []}
ref = None
for rnd in range(2):
    for save in (False, True):
        dt, out = run(save)
        res[save].append(dt)
        same = ref is None or (np.array_equal(out[0], ref[0]) and np.array_equal(out[1], ref[1]))
        ref = ref or out
        print('%s round %d save_sampler_params=%s: %.3f s per EP iteration (same Q, r: %s)'
              % (work, rnd, save, dt, same), flush=True)
print('%s mean s/iteration: off %.3f, on %.3f (%+.1f %%)' % (
    work, np.mean(res[False]), np.mean(res[True]), 100 * (np.mean(res[True]) / np.mean(res[False]) - 1)))

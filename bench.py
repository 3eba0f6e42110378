#!/usr/bin/env python
"""Benchmark of the EP inner loop (BASELINE.json metric: EP iterations/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg3|cfg4|cfg5|cfg1like] [--sites K] [--chains C] [--siter I]
                    [--damp auto|schedule] [--data sim|synth] [--max-treedepth T] [--rhat-max R]
                    [--dump-outputs DIR]

    python bench.py --workload cfg5 --sites 148 --siter 100 --max-treedepth 6 --rhat-max 0 --no-cpu-baseline
        BASELINE.json configs[4] (K=256, n_k=200 000, D=199, 32 chains), bounded: one wave of sites, 100
        sampling iterations, tree depth <= 6 (a full-depth transition streams the site's 83 MB design matrix
        1023 times); `roofline.bound` is "hbm" there (the wide tcgen05 pass streams X from HBM).

A "step" is one full EP iteration over all K sites: tilted NUTS sampling of
every site x chain (all draws), moment matching, damping selection, damped
update with the natural-parameter all-reduce, cavities and global moments.
Default workload is BASELINE.json configs[3] (SURVEY 8d "config 4"):
varying-slope logistic model m3b_sg, K=1024 sites, n_k=5000, D=49 (d=50),
data from the repository's m3b simulator with seed_data=100 (the reference's
fit.py default), sharded by site over the ranks (strong scaling: K is fixed,
each of N GPUs owns K/N sites).

Prints ONE JSON line (rank 0).  `value` = EP iterations/s with the state
resident in HBM; `e2e` = the same through one Master.run(1) call per step with
host state buffers (upload of Q,r,Qi,ri,dQi,dri,cavities before, download of
all mirrors and the moments after, every step); `roofline` = the sampler kernel
(dominant) against the measured bf16 tensor peak, algorithmic flops = 4*n_k*D
per gradient evaluation (SURVEY 8d) times the evaluations counted on the
device; `health` = per-iteration EP diagnostics (damping used, update
attempts, max split-Rhat, mean step size, KL between successive global
approximations); `cpu_baseline` = the fp64 NumPy oracle (oracle/nuts.py +
oracle/ep_linalg.py) timed on this box's host cores on a bounded sample of the
same sites at the cavities the GPU run ended with.
"""

import argparse
import json
import os
import subprocess
import sys
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'ep-stan_b200'))

WORKLOADS = {
    # name: (model, K, n_k, D, chains, siter)
    'cfg4': ('m3b', 1024, 5000, 49, 4, 200),      # BASELINE configs[3]
    'cfg3': ('m1b', 64, 2000, 19, 8, 200),        # BASELINE configs[2]
    'cfg5': ('m1b', 256, 200000, 199, 32, 200),   # BASELINE configs[4] (use --sites to bound the step time)
    'cfg1like': ('m1b', 4, 320, 16, 4, 200),      # shape of configs[0] (single group per site)
}


def dphi(model, D):
    return 2 * D + 2 if model in ('m4b', 'm5b') else D + 1


def simulate_problem(model, K, n_k, D, seed=100):
    """The reference's data recipe (SURVEY 8d): experiment/models/<model>.py simulate_data with
    Sigma_x='rand', seed_data=100 (fit.py:136-140,235-238), one group per site (K == J, the *_sg
    Stan programs), and the model's own prior (get_prior)."""
    import importlib
    sys.path.insert(0, os.path.join(ROOT, 'ep-stan_b200', 'experiment'))
    mod = importlib.import_module('models.' + model)
    mdl = mod.model(K, D, n_k)
    data = mdl.simulate_data(Sigma_x='rand', rng=seed)
    _, _, Q0, r0 = mdl.get_prior()
    return data.X, data.y.astype(np.int64), {'Q': Q0, 'r': r0}


def synth_site(model, k, n_k, D, seed=100):
    """Cheap per-site generator for shapes whose full simulation does not fit the host
    (config 5: 51 M rows x 199 inputs): standardised correlated inputs, group intercept/slopes.
    (float32 normals from a counter-free SFC64 stream per site: 40 M normals per config-5 site)"""
    rng = np.random.Generator(np.random.SFC64([seed, k]))
    g = np.random.RandomState(seed)                       # shared truth
    beta = g.standard_normal(D) * (0.5 if model != 'm1b' else 1.0) / np.sqrt(D / 4.0)
    sigma_b = np.exp(0.3 * g.standard_normal(D) - 1.0)
    alpha = rng.standard_normal() * 1.0
    bk = beta + (rng.standard_normal(D) * sigma_b if model != 'm1b' else 0.0)
    X = rng.standard_normal((n_k, D), dtype=np.float32)
    X += 0.3 * rng.standard_normal((n_k, 1), dtype=np.float32)   # common factor -> correlated inputs
    f = alpha + X @ bk.astype(np.float32)
    y = (rng.random(n_k) < 1.0 / (1.0 + np.exp(-f.astype(np.float64)))).astype(np.int64)
    return X, y


# (kept under its old name for tests/test_host_logic.py)
site_data = synth_site


def build_problem(model, K, n_k, D, k_begin, k_end, data='synth'):
    """Full-shape X, y with (at least) the local sites' rows filled in, and the prior."""
    d = dphi(model, D)
    if data == 'sim':
        return simulate_problem(model, K, n_k, D)
    X = np.zeros((K * n_k, D))
    y = np.zeros(K * n_k, dtype=np.int64)

    def fill(k):
        X[k * n_k:(k + 1) * n_k], y[k * n_k:(k + 1) * n_k] = synth_site(model, k, n_k, D)

    if (k_end - k_begin) * n_k * D > 1 << 26:             # large: the generator releases the GIL
        import concurrent.futures
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
            list(ex.map(fill, range(k_begin, k_end)))
    else:
        for k in range(k_begin, k_end):
            fill(k)
    prior = {'Q': np.eye(d) / 1.5 ** 2, 'r': np.zeros(d)}
    return X, y, prior


def default_df0(K):
    """experiment/fit.py:176-186"""
    b = min(1.0 / K, 0.2)
    a = 0.5 - b
    t = -np.log(0.1) / (K - 1)
    return lambda it: a * np.exp(-t * (it - 1)) + b


def kl_mvn(m0, S0, m1, S1):
    """KL(N(m0,S0) || N(m1,S1)) (reference experiment/find_damp.py:32-51)."""
    L0 = np.linalg.cholesky(S0)
    L1 = np.linalg.cholesky(S1)
    dm = m1 - m0
    sol = np.linalg.solve(S1, S0)
    return float(0.5 * (np.trace(sol) + dm.dot(np.linalg.solve(S1, dm)) - len(m0))
                 - np.sum(np.log(np.diag(L0))) + np.sum(np.log(np.diag(L1))))


class ClockSampler(object):
    FIELDS = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
              'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
              'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.proc = None
        self.rows = []
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(gpu_index), '--query-gpu=' + self.FIELDS,
                 '--format=csv,noheader,nounits', '-lms', '200'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ''
        sm, smax, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [v.strip() for v in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': float(max(smax)) if smax else None, 'reasons': sorted(reasons)}


def load_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p.get('hbm_gbs', 6650.0), p.get('bf16_tflops_sustained', 1400.0), 'measured'
    return 6650.0, 1590.0, 'fallback'


def load_traffic(workload, world):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of the
    same workload (profiles/traffic.json, written by tools/profile_round.sh); None when there is none."""
    path = os.path.join(ROOT, 'profiles', 'traffic.json')
    try:
        with open(path) as f:
            return json.load(f).get('%s_n%d' % (workload, world))
    except Exception:
        return None


# ---------------------------------------------------------------------------
# CPU baseline: the fp64 oracle on a bounded sample of sites
# ---------------------------------------------------------------------------
def _cpu_site(args):
    """One site's tilted step with the oracle: NUTS draws + moment matching + cavity."""
    model, Xk, yk, chains, siter, cav_m, cav_Q, Q, r, seed = args
    from oracle import density as dens, nuts, ep_linalg as orc
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(1)                  # one BLAS thread per worker process
    except Exception:
        pass
    d = Q.shape[0]
    td = dens.TiltedDensity(model, Xk, yk, cav_m, cav_Q)
    t0 = time.perf_counter()
    res = nuts.sample(lambda q: tuple(v[0] for v in td.lp_grad(q[None])), td.p, chains=chains,
                      n_iter=siter, seed=seed)
    if res['draws'].shape[0] > d + 2:
        ok, dQ, dr_ = orc.tilted_moments(res['draws'][:, :d], Q, r, 'sample')
        orc.cavity(Q + 0.1 * dQ, r + 0.1 * dr_, 0.1 * dQ, 0.1 * dr_)
    return time.perf_counter() - t0, res['n_grad']


def cpu_baseline(model, K, chains, siter, sites, procs, Q, r):
    """Bounded sample: ONE chain of `siter` iterations on each of the given sites
    [(X_k, y_k, cavity mean, cavity precision)], one process per core, scaled to K sites x `chains`."""
    import multiprocessing as mp
    jobs = [(model, Xk, yk, 1, siter, cm, cQ, Q, r, k) for k, (Xk, yk, cm, cQ) in enumerate(sites)]
    t0 = time.perf_counter()
    if procs > 1:
        with mp.get_context('fork').Pool(procs) as pool:
            out = pool.map(_cpu_site, jobs)
    else:
        out = [_cpu_site(j) for j in jobs]
    wall = time.perf_counter() - t0
    n_grad = sum(o[1] for o in out)
    its = 1.0 / (wall * (K * chains) / float(len(sites)))   # EP iterations/s for K sites x chains at this rate
    return its, n_grad / wall, wall


def cpu_linalg_baseline(d, n, n_sites=32):
    """Moment matching + cavity of the oracle (fp64 NumPy/LAPACK restatement of method.py:267-302,413-468)
    on `n_sites` sites of n draws, one core: microseconds per site."""
    from oracle import ep_linalg as orc
    rng = np.random.RandomState(0)
    Q = np.eye(d) * 3.0
    r = rng.standard_normal(d)
    Qi = np.eye(d) * 0.5
    ri = np.zeros(d)
    samps = [rng.standard_normal((n, d)) for _ in range(n_sites)]
    from threadpoolctl import threadpool_limits
    with threadpool_limits(1):                          # one BLAS thread: these are 50 x 800 problems
        orc.tilted_moments(samps[0], Q, r, 'sample')   # (library warm-up)
        orc.cavity(Q, r, Qi, ri)
        t0 = time.perf_counter()
        for sm in samps:
            orc.tilted_moments(sm, Q, r, 'sample')
        t1 = time.perf_counter()
        for _ in samps:
            orc.cavity(Q, r, Qi, ri)
        t2 = time.perf_counter()
    return 1e6 * (t1 - t0) / n_sites, 1e6 * (t2 - t1) / n_sites


def _sample_sites(model, K, n_k, D, n_sample, data):
    """(X_k, y_k, prior-cavity) of the first n_sample sites and the prior, for the reference arm."""
    if data == 'sim':
        X, y, prior = simulate_problem(model, K, n_k, D)
    else:
        X, y, prior = build_problem(model, K, n_k, D, 0, n_sample, 'synth')
    Q0 = np.asarray(prior['Q'], dtype=np.float64)
    r0 = np.asarray(prior['r'], dtype=np.float64)
    m0 = np.linalg.solve(Q0, r0)
    sites = [(X[k * n_k:(k + 1) * n_k].copy(), y[k * n_k:(k + 1) * n_k].copy(), m0, Q0) for k in range(n_sample)]
    return sites, Q0, r0


def run_reference(args, model, K, n_k, D, chains, siter):
    """--impl reference: the reference's CPU path for this workload.  PyStan (un-vendored dependency,
    README.md:5-10) is probed at run time; without it this is the oracle port (kind "port"), one
    process per host core over sites."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    try:
        import pystan  # noqa: F401
        have_pystan = True
    except Exception:
        have_pystan = False
    cores = os.cpu_count() or 1
    n_sample = min(K, max(cores, 2))
    sites, Q0, r0 = _sample_sites(model, K, n_k, D, n_sample, args.data)
    # Bounded sample: a step = ONE chain on each of n_sample sites at the first EP iteration's cavity (the
    # prior).  The warm-up steps (siter/4 iterations) also calibrate the cost per sampling iteration; the timed
    # steps run the full `siter` when --steps of them fit in REF_BUDGET_S, otherwise fewer iterations per chain,
    # scaled to `siter` (stated in `sample`).
    REF_BUDGET_S = 240.0
    t_begin = time.perf_counter()
    siter_w = max(20, siter // 4)
    wall_w = None
    for i in range(max(args.warmup, 1)):
        _, _, wall_w = cpu_baseline(model, K, chains, siter_w, sites, cores, Q0, r0)
    per_iter = wall_w / siter_w
    remaining = max(REF_BUDGET_S - (time.perf_counter() - t_begin), 30.0)
    siter_step = siter if per_iter * siter * args.steps <= remaining else \
        max(20, min(siter, int(remaining / (args.steps * per_iter))))
    vals = []
    for i in range(args.steps):
        its, gps, wall = cpu_baseline(model, K, chains, siter_step, sites, cores, Q0, r0)
        vals.append((its * siter_step / float(siter), gps, wall))
    its = float(np.mean([v[0] for v in vals]))
    line = {
        'impl': 'reference', 'metric': 'EP iterations/sec (K sites, all draws)', 'value': its,
        'unit': 'it/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 / its, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': args.workload, 'model': model + '_sg', 'K': K, 'n_k': n_k, 'D': D,
                   'chains': chains, 'siter': siter, 'data': args.data},
        'grad_evals_per_s': float(np.mean([v[1] for v in vals])),
        'pystan_available': have_pystan,
        'cpu_baseline': {'value': its, 'unit': 'it/s', 'cores': cores, 'kind': 'port',
                         'sample': 'one chain of %d (of %d) iterations on each of %d sites per step (of %d sites x %d '
                                   'chains), fp64 NumPy oracle NUTS, one process per core; scaled to the full workload'
                                   % (siter_step, siter, n_sample, K, chains)},
        'e2e': {'value': its, 'unit': 'it/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, m, m_phi, cov_phi):
    """What the last timed EP iteration computed, as float64 .npy files in `out_dir`, so that two builds run
    with the same arguments can be compared output for output: the global approximation Master.run returned
    (m_phi, cov_phi), its natural parameters (Q, r) and the site natural parameters (site_Qi [d, d, n],
    site_ri [d, n]) of the sites in site_index -- all K sites, or a fixed seeded sample of them when all would
    exceed DUMP_BYTES in all."""
    d, K = m.dphi, m.K
    per_site = 8 * (d * d + d + 1)
    n = min(K, (DUMP_BYTES - 16 * (d * d + d) - 7 * 128) // per_site)      # (128: an .npy header)
    idx = np.arange(K) if n == K else np.sort(np.random.RandomState(0).choice(K, n, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (('m_phi', m_phi), ('cov_phi', cov_phi), ('Q', m.Q), ('r', m.r),
                    ('site_Qi', m.Qi[:, :, idx]), ('site_ri', m.ri[:, idx]), ('site_index', idx)):
        np.save(os.path.join(out_dir, name + '.npy'), np.asarray(a, dtype=np.float64))


def run_ours(args, model, K, n_k, D, chains, siter):
    import torch
    import torch.distributed as dist
    if os.environ.get('BENCH_DEBUG'):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ['BENCH_DEBUG']), exit=True)
    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank),
                                timeout=datetime.timedelta(seconds=int(os.environ.get('BENCH_NCCL_TIMEOUT', 900))))
    import epstan.method as method
    method.set_default_stream(torch.cuda.current_stream().cuda_stream)

    d = dphi(model, D)
    base, rem = divmod(K, world)
    k_begin = rank * base + min(rank, rem)
    k_end = k_begin + base + (1 if rank < rem else 0)
    t_data = time.perf_counter()
    X, y, prior = build_problem(model, K, n_k, D, k_begin, k_end, args.data)
    t_data = time.perf_counter() - t_data
    kw = dict(df0=default_df0(K))
    if args.damp in ('auto', 'auto1'):
        kw['df_select'] = 'snr'
        if args.damp == 'auto1':
            kw['df0'] = None                   # no cap: the selection may take a full step
    if args.rhat_max > 0:
        kw['rhat_max'] = args.rhat_max
    if args.no_adapt_prev:
        kw['adapt_prev'] = False
    if args.max_treedepth:
        kw['control'] = {'max_treedepth': args.max_treedepth}
    m = method.Master('experiment/models/%s_sg' % model, X, y, site_sizes=np.full(K, n_k), prior=prior,
                      chains=chains, iter=siter, **kw)
    n_sample = min(K, max(os.cpu_count() or 1, 2))
    cpu_sites = [(X[k * n_k:(k + 1) * n_k].copy(), y[k * n_k:(k + 1) * n_k].copy()) for k in range(n_sample)] \
        if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None
    del X, y
    ctx = m._shard.ctx

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    hist = dict(df=[], attempts=[], mrhat=[], mstep=[], stime=[], other=[], m=[], S=[], rhat_sites=[], snr=[], n_fail=[],
                rejected=[])

    def timed_run(nsteps, per_step_calls=False):
        """nsteps EP iterations: one run(nsteps) call, or nsteps calls of run(1) (the e2e leg: host state in and
        out every step).  Returns (iterations completed, device ms, wall ms, kernel launches)."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launch_count()
        t0 = time.perf_counter()
        e0.record()
        done = 0
        for call in range(nsteps if per_step_calls else 1):
            n_it = 1 if per_step_calls else nsteps
            info, (ms_, Ss_), (st_, mst_, mrh_, oth_) = m.run(n_it, verbose=False, seed=1234 + m.iter,
                                                              return_analytics=True)
            n_done = len(m.history['df'])
            done += n_done
            hist['df'] += list(m.history['df'])
            hist['attempts'] += list(m.history['attempts'])
            hist['rhat_sites'] += list(m.history['rhat_sites'][:n_done])
            hist['snr'] += list(m.history['snr'][:n_done])
            hist['n_fail'] += list(m.history['n_fail'][:n_done])
            hist['rejected'] += list(m.history['rejected'][:n_done])
            hist['mrhat'] += list(mrh_[:n_done])
            hist['mstep'] += list(mst_[:n_done])
            hist['stime'] += list(st_[:n_done])
            hist['other'] += list(oth_[:n_done])
            hist['m'] += [ms_[i].copy() for i in range(n_done)]
            hist['S'] += [Ss_[i].copy() for i in range(n_done)]
            if info != 0:
                raise RuntimeError("EP stopped with info=%d after %d of %d iterations (EP iteration %d)"
                                   % (info, done, nsteps, m.iter))
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return done, float(t[0]), float(t[1]), ctx.launch_count() - l0

    # ---- warm-up (untimed) ----
    m.keep_on_device = False
    timed_run(args.warmup)

    # ---- value: state resident in HBM ----
    m.keep_on_device = True
    m.n_leapfrog_total = 0
    i_timed = len(hist['df'])
    clocks = ClockSampler(local_rank) if rank == 0 else None
    done, ms_dev, ms_wall, launches = timed_run(args.steps)
    clk = clocks.stop() if clocks else None
    if args.dump_outputs:
        m.sync_host()                  # (every rank: the site arrays are gathered over the ranks)
        if rank == 0:
            dump_outputs(args.dump_outputs, m, hist['m'][-1], hist['S'][-1])
    samp_s = float(np.sum(hist['stime'][i_timed:]))
    evals = torch.tensor([float(m.n_leapfrog_total)], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(evals, op=dist.ReduceOp.SUM)
    n_leap = float(evals[0])

    # ---- e2e: one Master.run(1) call per step, host state buffers in and out every step ----
    m.keep_on_device = False           # (run() first refreshes the host mirrors: they are stale after the resident leg)
    e2e_steps = args.steps if ms_wall / max(done, 1) < 5e3 else min(args.steps, 3)
    done2, ms_dev2, ms_wall2, _ = timed_run(e2e_steps, per_step_calls=True)
    n_loc = k_end - k_begin
    h2d = 8 * ((d * d + d) + n_loc * 3 * (d * d + d))               # Q,r + Qi,ri,dQi,dri + cavities, per step
    d2h = 8 * ((d * d + d) + n_loc * 4 * (d * d + d)) + 8 * (d * d + d)   # all mirrors + the moments, per step

    cpu_line = None
    if cpu_sites is not None:
        # the CPU arm samples the same sites at the cavities the GPU run ended with
        cores = os.cpu_count() or 1
        sites = [(Xk, yk, np.array(m.workers[k].vec), np.array(m.workers[k].Mat)) for k, (Xk, yk) in enumerate(cpu_sites)]
        cits, cgps, cwall = cpu_baseline(model, K, chains, siter, sites, cores, np.array(m.Q), np.array(m.r))
        cpu_line = {
            'value': cits, 'unit': 'it/s', 'cores': cores, 'kind': 'port', 'grad_evals_per_s': cgps,
            'sample': 'one chain of %d iterations on each of %d sites (of %d sites x %d chains) at the cavities of EP '
                      'iteration %d, fp64 NumPy oracle NUTS + moment matching, one process per core (%.1f s); scaled '
                      'to the full workload' % (siter, len(sites), K, chains, m.iter, cwall)}
        mom_us, cav_us = cpu_linalg_baseline(d, chains * (siter - siter // 2))
        cpu_line['moments_us_per_site'] = mom_us       # one core; the GPU kernels: profiles/*linalg_timing*
        cpu_line['cavity_us_per_site'] = cav_us

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    hbm_peak, tf_peak, peak_src = load_peaks()
    its = done / (ms_wall * 1e-3)
    its_e2e = done2 / (ms_wall2 * 1e-3)
    flops_per_eval = 4.0 * n_k * D
    # sampler kernel time = stimes (device events around the kernel), max over ranks per step
    tf_achieved = (n_leap / max(world, 1)) * flops_per_eval / max(samp_s, 1e-9) / 1e12   # per GPU
    kl_step = [kl_mvn(hist['m'][i], hist['S'][i], hist['m'][i - 1], hist['S'][i - 1]) for i in range(1, len(hist['m']))]
    rh = np.array(hist['mrhat'])
    x_bytes = n_loc * n_k * ((D + 3) * 4 + 64 * 2)
    # A site whose bf16 design matrix exceeds what stays on chip / in L2 next to the other sites' (config 5: 83 MB per
    # site) is streamed from HBM once per gradient evaluation of the site's chains: the sampler is HBM-bound there.
    # Algorithmic bytes per evaluation of all chains (SURVEY 8d): n_k * (2 D + 4) (bf16 X once + fp32 y once);
    # evaluations = leapfrogs / chains (the chains of a site advance in lock-step).
    hbm_roofline = None
    site_bytes = n_k * (2.0 * D + 4.0)
    if site_bytes * min(n_loc, 148) > 126e6 * 2:
        gbs = (n_leap / chains / max(world, 1)) * site_bytes / max(samp_s, 1e-9) / 1e9
        hbm_roofline = {'bound': 'hbm', 'achieved': gbs, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': gbs / hbm_peak,
                        'traffic': load_traffic(args.workload, world), 'kernel': 'k_nuts<32,2> (wide tcgen05 pass)',
                        'peak_source': peak_src + ' HBM copy bandwidth',
                        'tensor': {'achieved': tf_achieved, 'peak': tf_peak, 'unit': 'TFLOP/s',
                                   'frac': tf_achieved / tf_peak}}
    line = {
        'metric': 'EP iterations/sec (K sites, all draws)', 'value': its, 'unit': 'it/s',
        'n_gpus': world, 'steps': done, 'warmup': args.warmup, 'ms_per_step': ms_wall / max(done, 1),
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'bf16',
        'dtype_detail': 'sampler contractions bf16 x bf16 -> f32 on tcgen05, energies f64; moments/updates f64',
        'data': 'synthetic',
        'config': {'workload': args.workload, 'model': model + '_sg', 'K': K, 'n_k': n_k, 'D': D, 'd': d,
                   'chains': chains, 'siter': siter, 'parallelism': 'sites sharded %d-way' % world,
                   'data': ("experiment/models/%s.py simulate_data(Sigma_x='rand', seed 100) + get_prior (%.0f s)"
                            % (model, t_data)) if args.data == 'sim' else 'per-site generator synth_site (bench.py)',
                   'damping': {'auto': 'fit.py default_df0 as cap + automatic selection (df_select=snr)',
                               'auto1': 'automatic selection (df_select=snr), no cap',
                               'schedule': 'fit.py default_df0'}[args.damp],
                   'rhat_max': args.rhat_max if args.rhat_max > 0 else None,
                   'max_treedepth': args.max_treedepth or 10,
                   'warmup_start': ("Stan defaults (unit metric, step size 1) every EP iteration" if args.no_adapt_prev else
                                    "init_prev carries the last draw AND the adapted metric / step size of each chain "
                                    "(adapt_prev=True, an extension; --no-adapt-prev for Stan's defaults)"),
                   'l2': ('inputs larger than L2 (X %.0f MB fp32 + bf16 per GPU)' if x_bytes > 126e6
                          else 'inputs smaller than L2 (X %.0f MB fp32 + bf16 per GPU); not flushed: a step re-reads '
                               'each site\'s X thousands of times by design, the first touch is <0.1 %% of a step')
                         % (x_bytes / 1e6)},
        'grad_evals_per_s': n_leap / max(samp_s, 1e-9),
        'sampling_share': samp_s / (ms_wall * 1e-3),
        'device_ms_per_step': ms_dev / max(done, 1),
        'e2e': {'value': its_e2e, 'unit': 'it/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'steps': done2, 'ms_per_step': ms_wall2 / max(done2, 1)},
        'gpu_launches': launches,
        'clocks': clk,
        'roofline': hbm_roofline if hbm_roofline else {'bound': 'tensor', 'achieved': tf_achieved, 'peak': tf_peak, 'unit': 'TFLOP/s',
                     'frac': tf_achieved / tf_peak, 'traffic': load_traffic(args.workload, world), 'kernel': 'k_nuts',
                     'peak_source': peak_src + ' bf16 sustained; contractions on tcgen05 (bf16 in, fp32 accumulate)',
                     # supplementary view: every gradient evaluation of a site's chains streams the site's bf16
                     # design matrix (64 padded columns) + responses once, from L2
                     'x_stream': {'achieved': (n_leap / chains / max(world, 1)) * n_k * (64 * 2 + 4) / max(samp_s, 1e-9) / 1e9,
                                  'unit': 'GB/s per GPU (L2 -> shared memory)', 'hbm_peak': hbm_peak}},
        'info': 0, 'mean_stepsize': float(np.mean(hist['mstep'][i_timed:i_timed + done])),
        'max_rhat': float(np.max(rh[i_timed:i_timed + done])),
        'health': {
            'ep_iterations_total': len(hist['df']),
            'df_used': [round(float(v), 6) for v in hist['df']],
            'update_attempts': [int(v) for v in hist['attempts']],
            'sites_skipped': [int(v) for v in hist['n_fail']],     # failed moment estimate or Rhat > rhat_max
            # (rank 0's shard) the sites over rhat_max: they restart from a random initialisation next time
            'sites_rejected_rank0': [[int(k) for k in v] for v in hist['rejected']],
            'max_rhat': [round(float(v), 4) for v in hist['mrhat']],
            'mean_stepsize': [round(float(v), 5) for v in hist['mstep']],
            'sampling_s': [round(float(v), 3) for v in hist['stime']],
            'kl_step': [round(v, 5) for v in kl_step],       # KL(iteration i || i-1) of the global approximation
            'all_rhat_below_1p1': bool(np.all(rh < 1.1)),
            # per-site max split-Rhat over the site's sampled parameters (rank 0's shard): median, 90th
            # percentile, share of sites above 1.1 -- `max_rhat` is the maximum of these over all sites
            'rhat_sites_median_p90_frac_gt_1p1': [[round(float(x), 3) for x in t] for t in hist['rhat_sites']],
            # damping selection: |sum_k delta_k|^2, noise estimate, raw signal fraction
            'snr_T2_N2_raw': [[float('%.4g' % x) for x in t] for t in hist['snr']],
        },
    }
    if cpu_line is not None:
        line['cpu_baseline'] = cpu_line
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg4', choices=sorted(WORKLOADS))
    ap.add_argument('--sites', type=int, default=None)
    ap.add_argument('--chains', type=int, default=None)
    ap.add_argument('--siter', type=int, default=None)
    ap.add_argument('--damp', default='auto', choices=['auto', 'auto1', 'schedule'])
    ap.add_argument('--data', default=None, choices=['sim', 'synth'])
    ap.add_argument('--rhat-max', type=float, default=2.0,
                    help='skip the update of sites whose max split-Rhat exceeds this (0: never, the reference)')
    ap.add_argument('--no-adapt-prev', action='store_true',
                    help="Stan's unit metric / step size 1 at the start of every warm-up (the reference's behaviour)")
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--max-treedepth', type=int, default=None,
                    help="NUTS control (Stan's default 10); bounds the step time of --workload cfg5, stated in config")
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed EP iteration computed to DIR/<name>.npy (float64, <= 64 MB)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs needs --impl ours (the reference arm times sampling only)')
    model, K, n_k, D, chains, siter = WORKLOADS[args.workload]
    K = args.sites or K
    chains = args.chains or chains
    siter = args.siter or siter
    if args.data is None:
        args.data = 'synth' if args.workload == 'cfg5' else 'sim'
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get('RANK', 0))
    try:
        if args.impl == 'reference':
            run_reference(args, model, K, n_k, D, chains, siter)
        else:
            run_ours(args, model, K, n_k, D, chains, siter)
    except BaseException as e:                     # every rank reports its own failure before torchrun reaps it
        if not isinstance(e, SystemExit) or e.code not in (0, None):
            sys.stderr.write("[bench.py rank %d] FAILED: %s\n%s\n" % (rank, repr(e), traceback.format_exc()))
            sys.stderr.flush()
        raise


if __name__ == '__main__':
    main()

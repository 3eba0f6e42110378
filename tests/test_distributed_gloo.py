"""The N>1 path: two or three gloo ranks, each owning a contiguous block of the sites, must reproduce the
single-process reference results (golden Master.run scenarios).

On CPU the device context is replaced by the oracle-backed double in tests/fake_backend.py -- what is under test
is the host logic of the sharded Master: contiguous site shards, ONE all-reduce of the summed site deltas per EP
iteration, consensus on the damping, gathering of the mirrors.  The `gpu` cases run the same scenarios on the real
kernels, every rank on device 0 (gloo all-reduces the CUDA buffers), and record which branches of the exchanged
update (`Master._update_without_exchange`) the runs took."""
import os
import sys

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, 'tests')
SCENARIOS = ['runA', 'runB', 'runC', 'runD', 'runE', 'runF']


def _setup(rank, world, port, real):
    for p in (ROOT, os.path.join(ROOT, 'ep-stan_b200'), TESTS):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    if real:
        os.environ['EPGPU_DEVICE'] = '0'           # every rank shares the one GPU
    dist.init_process_group('gloo', rank=rank, world_size=world)
    import epstan.method as method
    if not real:
        import fake_backend
        method.Master._context_factory = staticmethod(lambda dev, stream: fake_backend.OracleContext(dev, stream))
    return method


def _record_branches(method):
    """count the branches of the exchanged update that a run takes: ladder retries (more than one proposal in one
    call), consensus re-attempts (the agreed ladder position is not this rank's), the fallback to the exchanging
    loop (status 2) and an invalid prior found under the exchange (status 1)"""
    seen = dict(calls=0, retry=0, reattempt=0, fallback=0, invalid=0)
    inner = method.Master._update_without_exchange

    def wrapped(self, df_first, verbose):
        ctx, comm = self._shard.ctx, self.comm
        n = [0]
        maxes = []
        f_ctx, f_comm = ctx.update_from_sums, comm.allreduce_scalar

        def ufs(df):
            n[0] += 1
            return f_ctx(df)

        def ars(value, op='sum'):
            out = f_comm(value, op)
            if op == 'max':
                maxes.append((value, out))
            return out
        ctx.update_from_sums, comm.allreduce_scalar = ufs, ars
        try:
            status, df, att = inner(self, df_first, verbose)
        finally:
            del ctx.update_from_sums, comm.allreduce_scalar
        seen['calls'] += 1
        seen['retry'] += n[0] > 1
        seen['reattempt'] += any(v != o for v, o in maxes) and status == 0
        seen['fallback'] += status == 2
        seen['invalid'] += status == 1
        return status, df, att
    method.Master._update_without_exchange = wrapped
    return seen


def _worker(rank, world, port, tag, ret, real=False):
    method = _setup(rank, world, port, real)
    try:
        import golden_inputs as gi
        from test_gpu_linalg import build_master
        seen = _record_branches(method)

        class _Ep(object):
            pass
        ep = _Ep()
        ep.method = method
        scs = gi.master_scenarios()
        sc = scs[tag]
        m = build_master(ep, sc)
        assert m.comm.size == world and m._shard.n_local in (sc['K'] // world, sc['K'] // world + 1)
        info, (ms, Ss) = m.run(sc['niter'], verbose=False, seed=sc['seed'])
        out = dict(info=info, m=ms, S=Ss, Q=m.Q.copy(), Qi=m.Qi.copy(), ri=m.ri.copy(),
                   k=(m._shard.k_begin, m._shard.k_end), df=list(m.history['df']))
        if tag == 'runC':
            sc2 = scs['runC2']
            res = m.run(sc2['niter'], verbose=False, seed=sc2['seed'])
            out.update(info2=res[0], m2=res[1][0], S2=res[1][1])
        out['seen'] = dict(seen)
        ret[rank] = out
    finally:
        dist.destroy_process_group()


def _worker_snr(rank, world, port, ret, real=False):
    method = _setup(rank, world, port, real)
    try:
        import test_damping as td
        from oracle import ep_linalg as orc
        sc = td._scenario(K=9, d=5, chains=4, it=60, niter=5, seed=17, df0=orc.default_df0(9))
        m = td._master(method, sc, df_select='snr')
        info, (ms, Ss) = m.run(sc['niter'], verbose=False, seed=sc['seed'])
        S_mix, m_mix = m.mix_phi()
        n = sc['chains'] * (sc['iter'] - sc['iter'] // 2)
        ret[rank] = dict(info=info, m=ms, S=Ss, df=list(m.history['df']), n_local=m._shard.n_local,
                         S_mix=S_mix.copy(), m_mix=m_mix.copy(),
                         draws=m._shard.ctx.get_draws(n), k=(m._shard.k_begin, m._shard.k_end))
    finally:
        dist.destroy_process_group()


def _spawn(target, world, args, timeout=180):
    """run `target(rank, world, *args, ret)` in `world` spawned processes; returns {rank: result}.  Whatever
    happens, no process outlives the call."""
    ctx = mp.get_context('spawn')
    mgr = ctx.Manager()
    procs = []
    try:
        ret = mgr.dict()
        procs = [ctx.Process(target=target, args=(r, world) + tuple(args[:-1]) + (ret,) + tuple(args[-1:]))
                 for r in range(world)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(timeout)
            assert p.exitcode == 0, p.exitcode
        assert sorted(ret.keys()) == list(range(world))
        return dict(ret)
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(10)
            if p.is_alive():
                p.kill()
                p.join()
        mgr.shutdown()


def _check_snr(world, ret, oinfo, oms, oSs, tol):
    from conftest import relerr
    assert sum(ret[r]['n_local'] for r in range(world)) == 9
    for r in range(world):
        assert ret[r]['info'] == oinfo == 0
        assert relerr(ret[r]['m'], oms) < tol and relerr(ret[r]['S'], oSs) < tol
        assert ret[r]['df'] == ret[0]['df']
    # Master.mix_phi over the ranks == the reference's pooling formula (method.py:1280-1298) on all the draws
    draws = np.concatenate([ret[r]['draws'][:ret[r]['k'][1] - ret[r]['k'][0]] for r in range(world)], axis=0)
    K, d, n = draws.shape
    assert K == 9
    means = draws.mean(axis=2)
    m_ref = means.mean(axis=0)
    S_ref = np.zeros((d, d))
    for k in range(K):
        xc = draws[k] - means[k][:, None]
        S_ref += xc @ xc.T + n * np.outer(means[k] - m_ref, means[k] - m_ref)
    S_ref /= K * n - 1
    for r in range(world):
        assert relerr(ret[r]['m_mix'], m_ref) < 1e-12 and relerr(ret[r]['S_mix'], S_ref) < 1e-10


def _snr_reference():
    sys.path.insert(0, TESTS)
    import test_damping as td
    from oracle import ep_linalg as orc
    sc = td._scenario(K=9, d=5, chains=4, it=60, niter=5, seed=17, df0=orc.default_df0(9))
    oinfo, oms, oSs, _, _ = td._oracle_run(sc, df_select='snr')
    return oinfo, oms, oSs


def test_two_and_three_rank_damping_selection():
    """df_select='snr' over 2 and 3 ranks (uneven shards): the all-reduced statistics give every rank the
    same damping as the single-process oracle replay."""
    oinfo, oms, oSs = _snr_reference()
    for world in (2, 3):
        port = 29700 + (os.getpid() % 2000) + world
        _check_snr(world, _spawn(_worker_snr, world, (port, False)), oinfo, oms, oSs, 1e-10)


@pytest.mark.gpu
def test_two_and_three_rank_damping_selection_real_context():
    """the same on the kernels, every rank on device 0"""
    oinfo, oms, oSs = _snr_reference()
    for world in (2, 3):
        port = 31700 + (os.getpid() % 2000) + world
        _check_snr(world, _spawn(_worker_snr, world, (port, True)), oinfo, oms, oSs, 1e-10)


def _check_golden(g, tag, world, ret):
    from conftest import relerr
    assert all(ret[r]['k'][1] == ret[r + 1]['k'][0] for r in range(world - 1))      # contiguous shards
    assert ret[0]['k'][0] == 0
    for r in range(world):
        o = ret[r]
        assert o['info'] == int(g[tag + '_info'])
        assert relerr(o['m'], g[tag + '_m']) < 1e-10 and relerr(o['S'], g[tag + '_S']) < 1e-10
        assert o['df'] == ret[0]['df']
        if o['info'] == 0:
            # host mirrors are complete on every rank
            assert relerr(o['Q'], g[tag + '_Q']) < 1e-10
            assert relerr(o['Qi'], g[tag + '_Qi']) < 1e-10 and relerr(o['ri'], g[tag + '_ri']) < 1e-10
        if tag == 'runC':
            assert o['info2'] == int(g['runC2_info'])
            assert relerr(o['m2'], g['runC2_m']) < 1e-10 and relerr(o['S2'], g['runC2_S']) < 1e-10


@pytest.mark.parametrize('tag', ['runA', 'runC', 'runD', 'runF'])
def test_two_rank_master_matches_reference(golden, tag):
    world = 2
    port = 29500 + (os.getpid() % 2000) + {'runA': 0, 'runC': 1, 'runD': 2, 'runF': 3}[tag]
    _check_golden(golden['master'], tag, world, _spawn(_worker, world, (port, tag, False)))


@pytest.mark.gpu
def test_multirank_real_context_matches_reference(golden):
    """every golden scenario over 2 and 3 ranks on the kernels (gloo, every rank on device 0) == the reference;
    together the runs take every branch of the exchanged update"""
    seen = {}
    for world in (2, 3):
        for i, tag in enumerate(SCENARIOS):
            port = 30000 + (os.getpid() % 2000) + 10 * i + world
            ret = _spawn(_worker, world, (port, tag, True))
            _check_golden(golden['master'], tag, world, ret)
            for r in range(world):
                for key, v in ret[r]['seen'].items():
                    seen[key] = seen.get(key, 0) + v
    assert seen['calls'] > 0
    for key in ('retry', 'reattempt', 'fallback', 'invalid'):
        assert seen[key] > 0, (key, seen)

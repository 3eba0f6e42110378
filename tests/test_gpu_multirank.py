"""Real-GPU, multi-rank runs of the EP loop against the single-rank result (SURVEY 8e).

The NCCL cases need >= 2 visible GPUs (skipped otherwise).  The gloo cases run 2 and 3 ranks on device 0 whatever
the GPU count: the same exchanged update (`Master._exchange`, `Master._update_without_exchange`) on the real kernels,
with gloo all-reducing the device buffers.  Sampling is deterministic per site, so sharding only changes the order
of the site sum: results must agree to ~1e-9."""
import os
import signal
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _ngpu():
    import torch
    return torch.cuda.device_count()


def _launch(tmp_path, nproc, mode, K, port, env_extra=None, timeout=600):
    """torchrun in its own session: on a timeout or any other exit the whole process group goes"""
    tag = '_'.join('%s%s' % kv for kv in sorted((env_extra or {}).items()))
    out = str(tmp_path / ('mr_%d_%s_%d%s.npz' % (nproc, mode, K, tag)))
    env = dict(os.environ)
    env.update(env_extra or {})
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(nproc),
           '--master-addr', '127.0.0.1', '--master-port', str(port), os.path.join(HERE, 'mr_worker.py'), out, mode, str(K)]
    p = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env,
                         start_new_session=True)
    try:
        so, se = p.communicate(timeout=timeout)
    finally:
        try:
            os.killpg(p.pid, signal.SIGKILL)
        except ProcessLookupError:
            pass
        p.wait()
    assert p.returncode == 0, so[-2000:] + se[-4000:]
    return np.load(out)


def _close(a, b, what):
    assert np.max(np.abs(a - b)) <= 1e-9 * max(1.0, np.max(np.abs(b))), what


@pytest.mark.parametrize('mode', ['current', 'side', 'private'])
def test_nccl_ranks_match_single_rank(tmp_path, mode):
    n = _ngpu()
    if n < 2:
        pytest.skip('needs >= 2 GPUs')
    import mr_worker
    K = 10
    m, info, ms, Ss, _ = mr_worker.run(K)
    assert info == 0
    for nproc in sorted(set([2, min(n, 4)])):
        res = _launch(tmp_path, nproc, mode, K, 29600 + nproc)
        assert int(res['info']) == 0 and int(res['size']) == nproc
        for a, b in ((res['ms'], ms), (res['Ss'], Ss), (res['Q'], m.Q), (res['Qi'], m.Qi), (res['cavm'], m._cavm)):
            _close(a, b, (mode, nproc))


def test_nccl_selection_and_uneven_shards(tmp_path):
    """automatic damping selection (its own all-reduce) with K not divisible by the rank count"""
    n = _ngpu()
    if n < 2:
        pytest.skip('needs >= 2 GPUs')
    import mr_worker
    K = 11
    m, info, ms, Ss, _ = mr_worker.run(K, df_select='snr')
    nproc = min(n, 4)
    res = _launch(tmp_path, nproc, 'current', K, 29650, {'MR_SELECT': '1'})
    assert int(res['info']) == info == 0
    assert np.allclose(res['df'], m.history['df'], rtol=1e-9)
    assert np.max(np.abs(res['ms'] - ms)) <= 1e-9 * max(1.0, np.max(np.abs(ms)))
    assert np.max(np.abs(res['Ss'] - Ss)) <= 1e-9 * max(1.0, np.max(np.abs(Ss)))


def _compare_single(res, single, nproc, what):
    m, info, ms, Ss, an = single
    assert int(res['info']) == info == 0 and int(res['size']) == nproc, what
    for a, b in ((res['ms'], ms), (res['Ss'], Ss), (res['Q'], m.Q), (res['r'], m.r), (res['Qi'], m.Qi),
                 (res['ri'], m.ri), (res['cavm'], m._cavm)):
        _close(a, b, what)
    assert np.allclose(res['df'], m.history['df'], rtol=1e-12, atol=0), what
    assert list(res['attempts']) == list(m.history['attempts']), what
    assert list(res['rejected']) == sorted(set(k for it in m.history['rejected'] for k in it)), what
    # the analytics maxima travel through the exchange slots
    assert np.array_equal(res['msteps'], an[1]) and np.array_equal(res['mrhats'], an[2]), what


@pytest.mark.parametrize('mode', ['private', 'current'])
def test_gloo_ranks_on_one_gpu_match_single_rank(tmp_path, mode):
    """2 and 3 ranks sharing device 0 over gloo: the exchanged update on the real kernels == one rank"""
    import mr_worker
    K = 10
    single = mr_worker.run(K)
    for nproc in (2, 3):
        res = _launch(tmp_path, nproc, mode, K, 29700 + 10 * nproc + (mode == 'current'), {'MR_BACKEND': 'gloo'})
        _compare_single(res, single, nproc, (mode, nproc))


def test_gloo_uneven_shards_with_rejected_sites(tmp_path):
    """K = 11 over 2 and 3 ranks with `rhat_max` between the two largest first-iteration Rhats: at least one site
    is rejected (epg_fail_sites, epg_reinit_sites, the failed-site count in the exchange slots)"""
    import mr_worker
    K = 11
    m1 = mr_worker.master(K)
    m1.run(1, verbose=False, seed=5)
    rh = np.sort([w.last_mrhat for w in m1.workers])
    assert np.all(np.isfinite(rh)) and rh[-1] > rh[-2]
    rhat_max = 0.5 * (rh[-1] + rh[-2])
    single = mr_worker.run(K, rhat_max=rhat_max)
    rejected = single[0].history['rejected']
    assert rejected[0] and any(rejected)
    assert single[0].history['n_fail'][0] >= 1
    for nproc in (2, 3):
        res = _launch(tmp_path, nproc, 'current', K, 29760 + nproc,
                      {'MR_BACKEND': 'gloo', 'MR_RHAT_MAX': repr(float(rhat_max))})
        _compare_single(res, single, nproc, ('rhat', nproc))

"""Worker of tests/test_gpu_multirank.py: one rank of a torchrun launch on real GPUs.

    torchrun --nproc-per-node N tests/mr_worker.py OUT.npz [side|current|private] [K]

Runs a small EP problem sharded over the ranks and lets rank 0 save the result.  Environment:
MR_BACKEND=gloo creates the process group with gloo and puts every rank on device 0 (so several ranks can share
one GPU; gloo all-reduces the CUDA buffers), else NCCL with one GPU per rank; MR_SELECT=1 selects
df_select='snr'; MR_RHAT_MAX sets the Master option rhat_max."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, os.path.join(ROOT, 'ep-stan_b200'), HERE):
    if p not in sys.path:
        sys.path.insert(0, p)


def problem(K=10, n_k=120, D=3, seed=3):
    rng = np.random.RandomState(seed)
    X = rng.standard_normal((K * n_k, D))
    beta = rng.standard_normal(D) * 0.7
    alpha = rng.standard_normal(K)
    f = alpha[np.repeat(np.arange(K), n_k)] + X @ beta
    y = (rng.uniform(size=K * n_k) < 1 / (1 + np.exp(-f))).astype(np.int64)
    d = D + 1
    return X, y, {'Q': np.eye(d) / 1.5 ** 2, 'r': np.zeros(d)}, n_k


def master(K, **kw):
    import epstan.method as method
    X, y, prior, n_k = problem(K)
    return method.Master('experiment/models/m1b_sg', X, y, site_sizes=np.full(K, n_k), prior=prior,
                         chains=4, iter=80, df0=0.4, **kw)


def run(K, niter=3, **kw):
    """(Master, info, per-iteration means, covariances, analytics (stimes, msteps, mrhats, othertimes))"""
    m = master(K, **kw)
    info, (ms, Ss), an = m.run(niter, verbose=False, seed=5, return_analytics=True)
    return m, info, ms, Ss, an


def main():
    import torch
    import torch.distributed as dist
    out, mode = sys.argv[1], sys.argv[2]
    K = int(sys.argv[3]) if len(sys.argv) > 3 else 10
    if os.environ.get('MR_BACKEND') == 'gloo':
        os.environ['EPGPU_DEVICE'] = '0'
        torch.cuda.set_device(0)
        dist.init_process_group('gloo')
    else:
        lr = int(os.environ['LOCAL_RANK'])
        torch.cuda.set_device(lr)
        dist.init_process_group('nccl', device_id=torch.device('cuda', lr))
    import epstan.method as method
    side = None
    if mode == 'side':            # the context works on a stream that is NOT the one NCCL is ordered on
        side = torch.cuda.Stream()
        method.set_default_stream(side.cuda_stream)
    elif mode == 'current':
        method.set_default_stream(torch.cuda.current_stream().cuda_stream)
    kw = dict(df_select='snr') if os.environ.get('MR_SELECT') else {}
    if os.environ.get('MR_RHAT_MAX'):
        kw['rhat_max'] = float(os.environ['MR_RHAT_MAX'])
    m, info, ms, Ss, an = run(K, **kw)
    # (history['rejected'] lists the sites of the local shard)
    rejected = [None] * dist.get_world_size()
    dist.all_gather_object(rejected, sorted(set(k for it in m.history['rejected'] for k in it)))
    if dist.get_rank() == 0:
        np.savez(out, info=info, ms=ms, Ss=Ss, Q=m.Q, r=m.r, Qi=m.Qi, ri=m.ri, cavm=m._cavm,
                 df=np.array(m.history['df']), attempts=np.array(m.history['attempts']),
                 rejected=np.array(sorted(set(k for r in rejected for k in r)), dtype=np.int64),
                 msteps=an[1], mrhats=an[2], size=dist.get_world_size())
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()

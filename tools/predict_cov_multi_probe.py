"""Cost of cgpcm_predict_f_cov on one or several ranks: the bench shape (N = 1e5, M = 200, frozen regime, default
cull) at n_star = 1000, smf = 1, for B in {1, 64}, with and without draws.  Each rank holds its shard_bounds slice.

    python tools/predict_cov_multi_probe.py [--out FILE] [--reps R]                     (one GPU)
    torchrun --nproc-per-node G tools/predict_cov_multi_probe.py [--out FILE] [--reps R]

Per row: the host-clock time of R calls that each end in a device synchronise (after one warm-up call of the same
shape), as median, min and max over the calls and over the ranks; then, from one more call under torch.profiler, the
device time of the gather (pcov_pack_kernel, pcov_unpack_kernel and the NCCL kernels) against all kernels of the call,
and the kernels that took the most time.  Rank 0 writes one JSON document."""
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, '.')
import cgpcm_b200
from cgpcm_b200.cgpcm import shard_bounds
from tools.predict_batch_probe import gpu_info
from tools.predict_cov_probe import counts
from tests.workload import sweep_workload

GATHER = ('pcov_pack_kernel', 'pcov_unpack_kernel', 'nccl')


def kernel_split(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, 'device_time_total', None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            per[e.key] = per.get(e.key, 0.0) + t / 1e3
    total = sum(per.values())
    gather = sum(v for k, v in per.items() if any(g in k for g in GATHER))
    top = sorted(per.items(), key=lambda kv: -kv[1])[:8]
    return dict(kernels_ms=total, gather_ms=gather, top_kernels_ms=[[k[:80], v] for k, v in top])


def main():
    out_path = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else 'profiles/r07_predict_multi.json'
    reps = int(sys.argv[sys.argv.index('--reps') + 1]) if '--reps' in sys.argv else 5
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group('gloo')
    wl = sweep_workload(100000, 200)
    n, n_star = wl['t'].shape[0], 1000
    eng = cgpcm_b200.Engine(wl['nh'], wl['nx'], device=local)
    if world > 1:
        box = [cgpcm_b200.Engine.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        eng.comm_init(box[0], rank, world)
    lo, hi = shard_bounds(n, rank, world)
    eng.set_data(wl['t'][lo:hi], wl['y'][lo:hi], wl['th'], wl['tx'])
    eng.precompute(*wl['hyp'], reg=wl['reg'])
    p, reg, nh = wl['params'], wl['reg'], wl['nh']
    rng = np.random.default_rng(1)
    S = np.stack([p[5:5 + nh] * (1 + .2 * rng.standard_normal(nh)) for _ in range(64)])
    t_star = np.linspace(wl['t'].min(), wl['t'].max(), n_star)
    rows = []
    for B in (1, 64):
        for draws in (False, True):
            noise = rng.standard_normal((n_star, B)) if draws else None
            call = lambda: eng.predict_f_cov(p, t_star, S[:B], smf=True, reg=reg, noise=noise)
            call()
            ts = []
            for _ in range(reps):
                t0 = time.perf_counter()
                call()
                ts.append(time.perf_counter() - t0)
            split = kernel_split(call)
            mine = dict(rank=rank, call_s=ts, **split)
            if world > 1:
                allr = [None] * world
                dist.all_gather_object(allr, mine)
            else:
                allr = [mine]
            every = [t for r in allr for t in r['call_s']]
            row = dict(B=B, draws=draws, calls=len(every), median_s=float(np.median(every)), min_s=float(min(every)),
                       max_s=float(max(every)), ranks=allr)
            rows.append(row)
            if rank == 0:
                print('world %d B %d draws %d: median %.3f s [%.3f, %.3f]; kernels %.1f ms, gather %.2f ms' % (
                    world, B, draws, row['median_s'], row['min_s'], row['max_s'], split['kernels_ms'],
                    split['gather_ms']), flush=True)
    if rank == 0:
        res = dict(gpu=gpu_info(), world=world, shape=dict(n=n, nx=wl['nx'], nh=nh, n_star=n_star, smf=1,
                                                             cull='default (80)'),
                   counts=counts(n_star, wl['nx'], nh), reps=reps,
                   method='host clock around calls that end in cudaStreamSynchronize, after one warm-up call of the '
                          'same shape; kernel split from one further call under torch.profiler', rows=rows)
        os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
        with open(out_path, 'w') as f:
            json.dump(res, f, indent=1)
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()

"""torchrun --nproc-per-node 2 tools/check_smf_batch_multi.py : cgpcm_elbo_smf_batch on observation shards (one
all-reduce of the per-sample C1 slabs) against the same call on one GPU with the whole series."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, '.')
import cgpcm_b200
from cgpcm_b200.cgpcm import shard_bounds
from tests.cases import make_case

rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
torch.cuda.set_device(local)
dist.init_process_group('nccl', device_id=torch.device('cuda', local))
c = make_case('toy_test', n=900)
rng = np.random.default_rng(3)
nh = c['nh']
S = np.stack([c['params'][5:5 + nh] * (1 + .2 * rng.standard_normal(nh)) for _ in range(9)])
eng = cgpcm_b200.Engine(nh, c['nx'], device=local)
box = [cgpcm_b200.Engine.unique_id() if rank == 0 else None]
dist.broadcast_object_list(box, src=0)
eng.comm_init(box[0], rank, world)
lo, hi = shard_bounds(len(c['t']), rank, world)
eng.set_data(c['t'][lo:hi], c['y'][lo:hi], c['th'], c['tx'])
eng.precompute(*c['hyp'], reg=c['reg'])
e, t, ll = eng.elbo_smf_batch(c['params'], S, reg=c['reg'])
got = [None] * world
dist.all_gather_object(got, (e.tobytes(), ll.tobytes()))
assert all(g == got[0] for g in got), 'ranks disagree'
if rank == 0:
    one = cgpcm_b200.Engine(nh, c['nx'], device=local)
    one.set_data(c['t'], c['y'], c['th'], c['tx'])
    one.precompute(*c['hyp'], reg=c['reg'])
    e1, t1, ll1 = one.elbo_smf_batch(c['params'], S, reg=c['reg'])
    scale = max(np.abs(e1).max(), np.abs(t1).max())
    err_e, err_l = np.abs(e - e1).max() / scale, np.abs(ll - ll1).max() / max(np.abs(ll1).max(), np.abs(t1[:, 2:4]).max())
    print('world %d: sharded vs one GPU: elbo rel %.2e, loglik rel %.2e' % (world, err_e, err_l))
    assert err_e <= 1e-9 and err_l <= 1e-9
    print('OK')
dist.barrier()
dist.destroy_process_group()

"""torchrun --nproc-per-node G tools/check_multi_predict.py : the sharded prediction paths (cgpcm_predict_f_cov with and
without draws, cgpcm_predict_logpdf, cgpcm_predict_f_batch; smf = 0 and 1) against a one-GPU Engine on the same data.

1. Rank 0 holds every observation and the other ranks none, so every all-reduced training-side sum is the one-GPU
   value: every output on every rank must be bitwise what the one-GPU engine returns (-0.0 == 0.0).
2. Balanced shards (shard_bounds): every rank returns byte-identical outputs, which agree with one GPU to 1e-6
   relative (lp_s and the whitened residuals within a bar derived from that agreement).
3. A sample owned by rank 1 whose C_b + d I is not positive definite: every rank raises -3 with the one-GPU message.

The shapes cover a tile count that is not a multiple of the world size, a single tile (n_star <= the tile side), B = 1
and B not a multiple of the world size, the bench's M = 200, and a call of two sample groups.  Object collectives run
over gloo; the library's own NCCL communicator carries the sharded work."""
import hashlib
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, '.')
import cgpcm_b200
from cgpcm_b200 import _lib
from cgpcm_b200.cgpcm import shard_bounds
from tests.cases import make_case
from tests.test_gpu_predict_cov import _draws, _trained
from tests.test_gpu_predict_logpdf import _check_scoring, _oracle_bound
from tests.workload import named_workload, sweep_workload

rank, world, local = int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), int(os.environ['LOCAL_RANK'])
dev = local % torch.cuda.device_count()
torch.cuda.set_device(dev)
dist.init_process_group('gloo')
EPS = np.finfo(np.float64).eps
NAMES = ['mean_s', 'cov_s', 'cov', 'draws', 'cov_nodraw', 'mean_s_nodraw', 'lp', 'lp_s', 'white', 'mean', 'var',
         'mean_b', 'var_b']


def bcast(obj):
    box = [obj]
    dist.broadcast_object_list(box, src=0)
    return box[0]


def digest(a, exact):
    """sha256 of the bytes; exact=False first maps -0.0 to 0.0 (np.array_equal's equality for finite values)."""
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    return hashlib.sha256((a if exact else a + 0.0).tobytes()).hexdigest()


def engine(wl, lo, hi, comm):
    eng = cgpcm_b200.Engine(wl['nh'], wl['nx'], causal=wl.get('causal', True), causal_id=wl.get('causal_id', False),
                            device=dev)
    if comm:
        eng.comm_init(bcast(cgpcm_b200.Engine.unique_id() if rank == 0 else None), rank, world)
    eng.set_data(wl['t'][lo:hi], wl['y'][lo:hi], wl['th'], wl['tx'])
    eng.precompute(*wl['hyp'], reg=wl['reg'])
    return eng


def inputs(wl, n_star, B, seed=1):
    rng = np.random.default_rng(seed)
    p, nh = wl['params'], wl['nh']
    S = np.stack([p[5:5 + nh] * (1 + .2 * rng.standard_normal(nh)) for _ in range(B)])
    t_star = np.linspace(wl['t'].min(), wl['t'].max(), n_star)
    y = np.interp(t_star, wl['t'], wl['y']) + .3 * rng.standard_normal(n_star)
    return t_star, S, rng.standard_normal((n_star, B)), y


def outputs(eng, wl, case, smf):
    t_star, S, noise, y = case
    p, reg = wl['params'], wl['reg']
    o = {}
    _, o['cov'], o['mean_s'], o['cov_s'], o['draws'] = eng.predict_f_cov(p, t_star, S, smf=smf, reg=reg,
                                                                         per_sample=True, noise=noise)
    _, o['cov_nodraw'], o['mean_s_nodraw'], _, _ = eng.predict_f_cov(p, t_star, S, smf=smf, reg=reg)
    lp, o['lp_s'], o['white'] = eng.predict_logpdf(p, t_star, y, S, smf=smf, reg=reg, noise=True, white=True)
    o['lp'] = np.array([lp])
    o['mean'], o['var'], o['mean_b'], o['var_b'] = eng.predict_f_batch(p, t_star, S, smf=smf, reg=reg)
    return o


def rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def check_balanced(label, wl, case, one, sh):
    """Rank 0: the balanced-shard outputs against one GPU."""
    t_star, S, noise, y = case
    d = np.exp(wl['params'][0])
    worst = {}
    for k in ('mean_s', 'cov_s', 'cov', 'draws', 'cov_nodraw', 'mean_s_nodraw', 'mean', 'var', 'mean_b', 'var_b'):
        worst[k] = rel(sh[k], one[k])
        assert worst[k] < 1e-6, (label, k, worst[k])
    # lp_s: the bound of tests/test_gpu_predict_logpdf.py with the measured agreement of the means and covariances
    # (at most four samples: the bound and the host scoring take seconds per sample at n_star = 2000)
    B = S.shape[0]
    bs = sorted({0, 1 % B, B - 2 if B > 1 else 0, B - 1})
    em = np.abs(sh['mean_s'] - one['mean_s']).max()
    for b in bs:
        eC = np.abs(sh['cov_s'][b] - one['cov_s'][b]).max()
        bound = 2 * _oracle_bound(y, one['mean_s'][:, b], one['cov_s'][b], (em, eC), d) + 1e-10 * abs(one['lp_s'][b])
        assert abs(sh['lp_s'][b] - one['lp_s'][b]) <= bound, (label, b, sh['lp_s'][b], one['lp_s'][b], bound)
    # the scoring stage on the sharded run's own m_b and C_b
    _check_scoring(sh['lp_s'][bs], sh['white'][:, bs], y, sh['mean_s'][:, bs], sh['cov_s'][bs], d)
    print('%s balanced: max rel %s' % (label, ' '.join('%s %.1e' % kv for kv in worst.items())), flush=True)


def run_shape(label, wl, n_star, B):
    case = inputs(wl, n_star, B)
    n = wl['t'].shape[0]
    one = None
    if rank == 0:
        eng1 = engine(wl, 0, n, False)
    eng_a = engine(wl, 0, n if rank == 0 else 0, True)          # rank 0 holds everything
    lo, hi = shard_bounds(n, rank, world)
    eng_b = engine(wl, lo, hi, True)
    for smf in (0, 1):
        tag = '%s smf=%d n_star=%d B=%d' % (label, smf, n_star, B)
        if rank == 0:
            one = outputs(eng1, wl, case, smf)
            ref = {k: digest(one[k], False) for k in NAMES}
        ref = bcast(ref if rank == 0 else None)
        a = outputs(eng_a, wl, case, smf)
        bad = [k for k in NAMES if digest(a[k], False) != ref[k]]
        res = [None] * world
        dist.all_gather_object(res, bad)
        assert all(not r for r in res), (tag, 'differs from one GPU', res)
        b = outputs(eng_b, wl, case, smf)
        res = [None] * world
        dist.all_gather_object(res, {k: digest(b[k], True) for k in NAMES})
        assert all(r == res[0] for r in res), (tag, 'ranks differ')
        if rank == 0:
            print('%s: bitwise equal to one GPU on %d ranks' % (tag, world), flush=True)
            check_balanced(tag, wl, case, one, b)
    for e in (eng_a, eng_b) + ((eng1,) if rank == 0 else ()):
        e.close()


def run_errors():
    """toy_small (trained), f scored with d = reg at a test input repeated 16 times, so that C_b is singular; a filter
    sample scaled up makes C_b grow with the square of the scale until its rounding outweighs reg.  Samples [passing,
    failing] under the first of smf = 0, 1 that has both: the failing one is sample 1, owned by rank 1."""
    c = make_case('toy_small')
    p, reg, nh = _trained(c), c['reg'], c['nh']
    t_star = np.linspace(c['t'].min(), c['t'].max(), 20)
    t_star = np.concatenate([np.full(16, t_star[8]), t_star])
    y = np.interp(t_star, c['t'], c['y']) + .3 * np.random.default_rng(0).standard_normal(t_star.size)
    draws = _draws(p, nh, reg, 2)
    cand = np.concatenate([draws, np.array([1e2, 1e4, 1e6, 1e8])[:, None] * draws[1:]])
    n = c['t'].shape[0]
    S = smf = msg = None
    if rank == 0:
        eng1 = engine(c, 0, n, False)
        for smf in (False, True):
            ok = []
            for b in range(cand.shape[0]):
                try:
                    eng1.predict_logpdf(p, t_star, y, cand[b:b + 1], smf=smf, reg=reg, noise=False)
                    ok.append(True)
                except _lib.CgpcmError as e:
                    ok.append(False if 'C_b + d I' in str(e) else None)
            print('error case: smf %d, samples alone pass: %s' % (smf, ok), flush=True)
            if True in ok and False in ok:
                break
        assert True in ok and False in ok, ok
        S = np.stack([cand[ok.index(True)], cand[ok.index(False)]])
        try:
            eng1.predict_logpdf(p, t_star, y, S, smf=smf, reg=reg, noise=False)
        except _lib.CgpcmError as e:
            msg = (e.code, str(e))
        assert msg and msg[0] == -3 and 'sample 1 ' in msg[1], msg
        eng1.close()
    S, smf, msg = bcast((S, smf, msg))
    for lo, hi in ((0, n if rank == 0 else 0), shard_bounds(n, rank, world)):
        eng = engine(c, lo, hi, True)
        got = None
        try:
            eng.predict_logpdf(p, t_star, y, S, smf=smf, reg=reg, noise=False)
        except _lib.CgpcmError as e:
            got = (e.code, str(e))
        res = [None] * world
        dist.all_gather_object(res, got)
        if lo == 0 and hi == (n if rank == 0 else 0):
            assert all(r == msg for r in res), (res, msg)
        else:
            assert all(r == res[0] and r[0] == -3 and 'sample 1 ' in r[1] for r in res), res
        eng.close()
    if rank == 0:
        print('errors: every rank raises %r' % (msg,), flush=True)


small = sweep_workload(1200, 16)          # nx = 16: tile side 64, cheap pair blocks
run_shape('toy', named_workload('toy'), 50, 3)          # tile side 48: 3 tiles
run_shape('toy', named_workload('toy'), 40, 1)          # one tile: ranks > 0 own none
run_shape('m200', sweep_workload(4000, 200), 100, 5)    # tile side 32: 10 tiles
run_shape('nx16', small, 2000, 65)                      # two groups of samples (64 + 1)
run_errors()
if rank == 0:
    print('OK multi predict')
dist.barrier()
dist.destroy_process_group()

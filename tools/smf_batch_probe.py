"""Per-sample cost of scoring filter samples under the SMF bound: cgpcm_elbo_smf (one frozen forward sweep with
H = h h^T per sample) against cgpcm_elbo_smf_batch (W = H_B A and the rank-one contraction, B samples per call), at
the toy shape (n = 400, nx = 150, nh = 41) and the bench shape (N = 1e5, M = 200, frozen regime, default cull), for
B in {1, 8, 64, 256}; and the toy experiment's sampling phase with one chain and with 8 chains at the same number of
states.  Times are host clock around a call that ends in a device synchronise, after warm-up.  One JSON document.

    python tools/smf_batch_probe.py [--out profiles/r03_smf_batch.json]
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, '.')
import cgpcm_b200
from cgpcm_b200 import MODE_FROZEN, VCGPCM, Data, Session, config
from tests.workload import named_workload, sweep_workload

BS = (1, 8, 64, 256)


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, pl, clk = [x.strip() for x in q.split(',')]
        return dict(name=name, power_limit=pl, sm_max_clock=clk)
    except Exception as ex:                          # the name from the runtime at least
        import torch
        return dict(name=torch.cuda.get_device_name(0), power_limit='unavailable (%s)' % ex)


def timed(fn, reps):
    fn()                                             # warm-up of this exact call
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps


def probe_shape(name, wl, single_reps):
    eng = cgpcm_b200.Engine(wl['nh'], wl['nx'])
    eng.set_data(wl['t'], wl['y'], wl['th'], wl['tx'])
    eng.precompute(*wl['hyp'], reg=wl['reg'])
    p, reg, nh = wl['params'], wl['reg'], wl['nh']
    rng = np.random.default_rng(1)
    S = np.stack([p[5:5 + nh] * (1 + .2 * rng.standard_normal(nh)) for _ in range(max(BS))])
    # the single-sample path costs the same for every sample: time `single_reps` calls, report per sample
    t_single = timed(lambda: [eng.elbo_smf(p, S[b], mode=MODE_FROZEN, reg=reg) for b in range(single_reps)], 1)
    t_single /= single_reps
    rows = []
    for B in BS:
        reps = max(1, min(10, 64 // B))
        t_call = timed(lambda: eng.elbo_smf_batch(p, S[:B], reg=reg), reps)
        t_ll = timed(lambda: eng.elbo_smf_batch(p, S[:B], reg=reg, want_elbo=False), reps)
        rows.append(dict(B=B, batch_call_s=t_call, batch_per_sample_s=t_call / B,
                         batch_loglik_only_per_sample_s=t_ll / B, single_per_sample_s=t_single,
                         speedup=t_single / (t_call / B)))
        print(name, rows[-1], flush=True)
    # agreement at the timed inputs (first 4 samples)
    e, t, ll = eng.elbo_smf_batch(p, S[:4], reg=reg)
    dev = 0.0
    for b in range(4):
        e1, t1, ll1 = eng.elbo_smf(p, S[b], mode=MODE_FROZEN, reg=reg)
        dev = max(dev, abs(e[b] - e1) / max(abs(e1), np.abs(t1).max()))
    eng.close()
    return dict(shape=name, n=int(wl['t'].shape[0]), nx=wl['nx'], nh=wl['nh'], cull='default (80)',
                single_calls_timed=single_reps, rows=rows, max_rel_elbo_dev_batch_vs_single=dev)


def probe_sampler(states):
    wl = named_workload('toy')
    config.reg = wl['reg']
    np.random.seed(1005)
    sess = Session()
    mod = VCGPCM.from_recipe(sess, Data(wl['t'], wl['y']), nx=wl['nx'], nh=wl['nh'], tau_w=.1, tau_f=.05, causal=True,
                             noise_init=1e-2)
    mod.precompute()
    mod.fpi(50)
    out = {}
    mod.sample(iters=2, burn=0)                      # warm-up of both paths
    mod.sample(iters=2, burn=0, chains=8)
    half = states // 2
    t0 = time.perf_counter()
    s1 = mod.sample(iters=half, burn=half)
    out['chains_1'] = dict(burn=half, iters=half, states=2 * half, seconds=time.perf_counter() - t0)
    per = states // 8 // 2
    t0 = time.perf_counter()
    s8 = mod.sample(iters=per, burn=per, chains=8)
    out['chains_8'] = dict(burn=per, iters=per, states=8 * 2 * per, seconds=time.perf_counter() - t0)
    assert len(s1) == half and len(s8) == 8 and all(np.all(np.isfinite(x)) for ch in s8 for x in ch)
    out['speedup'] = out['chains_1']['seconds'] / out['chains_8']['seconds']
    out['note'] = ('toy shape (n = 400, nx = 150, nh = 41) after precompute + 50 fixed-point rounds, no L-BFGS phases; '
                   'states include burn-in')
    print('sampler', out, flush=True)
    return out


def main():
    out_path = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else 'profiles/r03_smf_batch.json'
    res = dict(gpu=gpu_info(), method='host clock around calls that end in cudaStreamSynchronize, after one warm-up '
                                      'call of the same shape; batch_call_s is the mean of min(10, 64 / B) calls')
    res['shapes'] = [probe_shape('toy', named_workload('toy'), 16),
                     probe_shape('bench', sweep_workload(100000, 200), 3)]
    res['sampler'] = probe_sampler(1000)
    os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
    with open(out_path, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()

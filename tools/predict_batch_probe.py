"""Per-sample cost of predict_f's SMF prediction: cgpcm_predict_f (a frozen forward sweep, a blocked inverse and one
launch per sample and test chunk that reads the chunk's whole Bxx* block) against cgpcm_predict_f_batch (the rank-one C1
stage, one CTA per sample for q(z | h_b), and the test side as DMMA contractions over batches of samples), at the toy
shape (n = 400, nx = 150, nh = 41) and the bench shape (N = 1e5, M = 200, frozen regime, default cull) with
n_star = 10 000 test points, for B in {1, 8, 64, 256}; and the toy experiment's SMF predict_f with its 200 samples on
both paths.  Times are host clock around a call that ends in a device synchronise, after warm-up.  One JSON document.

    python tools/predict_batch_probe.py [--out profiles/r04_predict_f_batch.json]
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, '.')
import cgpcm_b200
from cgpcm_b200 import VCGPCM, Data, Session, config
from tests.workload import named_workload, sweep_workload

BS = (1, 8, 64, 256)
N_STAR = 10000


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


def rel_dev(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def probe_shape(name, wl, single_samples):
    eng = cgpcm_b200.Engine(wl['nh'], wl['nx'])
    eng.set_data(wl['t'], wl['y'], wl['th'], wl['tx'])
    eng.precompute(*wl['hyp'], reg=wl['reg'])
    p, reg, nh = wl['params'], wl['reg'], wl['nh']
    rng = np.random.default_rng(1)
    S = np.stack([p[5:5 + nh] * (1 + .2 * rng.standard_normal(nh)) for _ in range(max(BS))])
    t_star = np.linspace(wl['t'].min(), wl['t'].max(), N_STAR)
    # the single path costs the same for every sample: time `single_samples` samples in one call, report per sample
    t_single = timed(lambda: eng.predict_f(p, t_star, S[:single_samples], smf=True, reg=reg), 1) / single_samples
    rows = []
    for B in BS:
        reps = max(1, min(5, 64 // B))
        t_call = timed(lambda: eng.predict_f_batch(p, t_star, S[:B], smf=True, reg=reg), reps)
        rows.append(dict(B=B, batch_call_s=t_call, batch_per_sample_s=t_call / B, single_per_sample_s=t_single,
                         speedup=t_single / (t_call / B)))
        print(name, rows[-1], flush=True)
    # agreement at the timed inputs: averages and per-sample moments of the first samples against the single path
    m, v, ms, vs = eng.predict_f_batch(p, t_star, S[:single_samples], smf=True, reg=reg)
    m1, v1 = eng.predict_f(p, t_star, S[:single_samples], smf=True, reg=reg)
    dev = dict(mean=rel_dev(m, m1), var=rel_dev(v, v1))
    mb, vb = eng.predict_f(p, t_star, S[:1], smf=True, reg=reg)
    dev.update(mean_s_0=rel_dev(ms[:, 0], mb), var_s_0=rel_dev(vs[:, 0], vb))
    eng.close()
    return dict(shape=name, n=int(wl['t'].shape[0]), nx=wl['nx'], nh=wl['nh'], n_star=N_STAR, cull='default (80)',
                single_samples_timed=single_samples, rows=rows, max_rel_dev_batch_vs_single=dev)


def probe_toy_experiment():
    """The toy experiment's SMF prediction: its 200 posterior samples at the 400 inputs of the series."""
    wl = named_workload('toy')
    config.reg = wl['reg']
    np.random.seed(1005)
    mod = VCGPCM.from_recipe(Session(), Data(wl['t'], wl['y']), nx=wl['nx'], nh=wl['nh'], tau_w=.1, tau_f=.05,
                             causal=True, noise_init=1e-2)
    mod.precompute()
    mod.fpi(50)
    chains = mod.sample(iters=25, burn=25, chains=8)
    samples = [s for ch in chains for s in ch]
    t = wl['t']
    mod.predict_f(t, samples_h=samples[:2])           # warm-up of both paths
    mod.predict_f_samples(t, samples_h=samples[:2])
    t0 = time.perf_counter()
    pred = mod.predict_f(t, samples_h=samples)
    t_single = time.perf_counter() - t0
    t0 = time.perf_counter()
    mean, var = mod.predict_f_samples(t, samples_h=samples)
    t_batch = time.perf_counter() - t0
    out = dict(samples=len(samples), n_star=int(t.shape[0]), predict_f_s=t_single, predict_f_samples_s=t_batch,
               speedup=t_single / t_batch, max_rel_dev_mean=rel_dev(mean.mean(1), pred.mean.y),
               note='toy shape (n = 400, nx = 150, nh = 41) after precompute + 50 fixed-point rounds; 200 states of '
                    'sample(chains=8); the frozen statistics stay in place for both calls')
    print('toy_experiment', out, flush=True)
    return out


def main():
    out_path = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else 'profiles/r04_predict_f_batch.json'
    res = dict(gpu=gpu_info(), method='host clock around calls that end in cudaStreamSynchronize, after one warm-up '
                                      'call of the same shape; batch_call_s is the mean of min(5, 64 / B) calls')
    res['shapes'] = [probe_shape('toy', named_workload('toy'), 8),
                     probe_shape('bench', sweep_workload(100000, 200), 2)]
    res['toy_experiment'] = probe_toy_experiment()
    os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
    with open(out_path, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()

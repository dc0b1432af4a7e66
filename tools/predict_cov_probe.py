"""Cost of the joint predictive covariance of f (cgpcm_predict_f_cov, smf = 1, with draws): the toy shape (n = 400,
nx = 150, nh = 41) at n_star = 400 for B in {1, 8, 64, 200}, and the bench shape (N = 1e5, M = 200, frozen regime,
default cull) at n_star = 1000 for B in {1, 64}.  Per row: the call's time (host clock around a call that ends in a
device synchronise, after a warm-up call of the same shape), the time of cgpcm_predict_f_batch at the same inputs, and
the counts the test side needs: BVN evaluations of the pair blocks (tiles p >= q, full tiles) and flops of the fold
GEMMs.  One JSON document.

    python tools/predict_cov_probe.py [--out profiles/r05_predict_f_cov.json]
"""
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, '.')
import cgpcm_b200
from tests.workload import named_workload, sweep_workload
from tools.predict_batch_probe import gpu_info, timed


def counts(n_star, nx, nh):
    """Pair-block elements and fold flops of the lower-triangle tiles (tile side as pcov_tile in csrc/cgpcm.cu)."""
    nxp, nhp = -(-nx // 8) * 8, -(-nh // 8) * 8
    tp = max(8, min(64, int((6e7 / (nxp * nxp)) ** .5) // 8 * 8))
    nt = -(-n_star // tp)
    pairs = 0
    fold = 0.0
    for pt in range(nt):
        P = min(tp, n_star - pt * tp)
        for qt in range(pt + 1):
            Q = min(tp, n_star - qt * tp)
            pairs += P * Q
            fold += 2.0 * (P * nxp) * (Q * nxp) * nhp
    return dict(tile=tp, pair_blocks=pairs, bvn_evaluations=pairs * nx * nx, fold_gemm_flop=fold)


def probe_shape(name, wl, n_star, bs):
    eng = cgpcm_b200.Engine(wl['nh'], wl['nx'])
    eng.set_data(wl['t'], wl['y'], wl['th'], wl['tx'])
    eng.precompute(*wl['hyp'], reg=wl['reg'])
    p, reg, nh = wl['params'], wl['reg'], wl['nh']
    rng = np.random.default_rng(1)
    S = np.stack([p[5:5 + nh] * (1 + .2 * rng.standard_normal(nh)) for _ in range(max(bs))])
    t_star = np.linspace(wl['t'].min(), wl['t'].max(), n_star)
    rows = []
    for B in bs:
        noise = rng.standard_normal((n_star, B))
        reps = 2 if B <= 8 else 1
        t_cov = timed(lambda: eng.predict_f_cov(p, t_star, S[:B], smf=True, reg=reg, noise=noise), reps)
        t_batch = timed(lambda: eng.predict_f_batch(p, t_star, S[:B], smf=True, reg=reg), reps)
        _, cov, ms, _, dr = eng.predict_f_cov(p, t_star, S[:B], smf=True, reg=reg, noise=noise)
        _, v1, ms1, _ = eng.predict_f_batch(p, t_star, S[:B], smf=True, reg=reg)
        scale = max(np.abs(v1).max(), np.abs(ms1).max() ** 2)
        rows.append(dict(B=B, cov_call_s=t_cov, cov_per_sample_s=t_cov / B, predict_f_batch_call_s=t_batch,
                         max_rel_dev_diag_vs_batch=float(np.abs(np.diag(cov) - v1).max() / scale),
                         finite=bool(np.all(np.isfinite(cov)) and np.all(np.isfinite(dr)))))
        print(name, rows[-1], flush=True)
    eng.close()
    return dict(shape=name, n=int(wl['t'].shape[0]), nx=wl['nx'], nh=wl['nh'], n_star=n_star, cull='default (80)',
                counts=counts(n_star, wl['nx'], wl['nh']), rows=rows)


def main():
    out_path = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else 'profiles/r05_predict_f_cov.json'
    res = dict(gpu=gpu_info(), method='host clock around calls that end in cudaStreamSynchronize, after one warm-up '
                                      'call of the same shape; mean of 2 calls for B <= 8, else 1; smf = 1 with draws')
    res['shapes'] = [probe_shape('toy', named_workload('toy'), 400, (1, 8, 64, 200)),
                     probe_shape('bench', sweep_workload(100000, 200), 1000, (1, 64))]
    os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
    with open(out_path, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()

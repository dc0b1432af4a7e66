"""Cost of held-out scoring (cgpcm_predict_logpdf, smf = 1, noise = 1) beside the joint covariance it is built on
(cgpcm_predict_f_cov, smf = 1, with draws and without): the toy shape (n = 400, nx = 150, nh = 41) at n_star = 400 for
B in {1, 8, 64, 200}, and the bench shape (N = 1e5, M = 200, frozen regime, default cull) at n_star = 1000 for B in
{1, 64}.  Per row: each call's time (host clock around a call that ends in a device synchronise, after a warm-up call
of the same shape) and launch count.  scoring_increment_s = logpdf - f_cov without draws (the bordered factorisations
and the scoring kernels); draws_increment_s = f_cov with draws - without.  Not separated: the factorisations from the
border and scoring kernels, and the pair blocks from the fold GEMMs.  The card's name and power limit are read in the
same process.  One JSON document.

    python tools/predict_logpdf_probe.py [--out profiles/r06_predict_logpdf.json]
"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, '.')
import cgpcm_b200
from tests.workload import named_workload, sweep_workload
from tools.predict_batch_probe import gpu_info, timed


def probe_shape(name, wl, n_star, bs):
    eng = cgpcm_b200.Engine(wl['nh'], wl['nx'])
    eng.set_data(wl['t'], wl['y'], wl['th'], wl['tx'])
    eng.precompute(*wl['hyp'], reg=wl['reg'])
    p, reg, nh = wl['params'], wl['reg'], wl['nh']
    rng = np.random.default_rng(1)
    S = np.stack([p[5:5 + nh] * (1 + .2 * rng.standard_normal(nh)) for _ in range(max(bs))])
    t_star = np.linspace(wl['t'].min(), wl['t'].max(), n_star)
    y_star = np.interp(t_star, wl['t'], wl['y'])
    rows = []
    for B in bs:
        noise = rng.standard_normal((n_star, B))
        reps = 2 if B <= 8 else 1
        calls = dict(
            logpdf=lambda: eng.predict_logpdf(p, t_star, y_star, S[:B], smf=True, reg=reg, white=True),
            f_cov_draws=lambda: eng.predict_f_cov(p, t_star, S[:B], smf=True, reg=reg, noise=noise),
            f_cov=lambda: eng.predict_f_cov(p, t_star, S[:B], smf=True, reg=reg))
        row = dict(B=B)
        for k, fn in calls.items():
            row[k + '_s'] = timed(fn, reps)
            row[k + '_launches'] = eng.last_timing()['launches']
        lp, lp_s, white = eng.predict_logpdf(p, t_star, y_star, S[:B], smf=True, reg=reg, white=True)
        row.update(scoring_increment_s=row['logpdf_s'] - row['f_cov_s'],
                   draws_increment_s=row['f_cov_draws_s'] - row['f_cov_s'],
                   lp=lp, lp_s_range=[float(lp_s.min()), float(lp_s.max())],
                   white_mean=float(white.mean()), white_var=float(white.var()),
                   finite=bool(np.isfinite(lp) and np.all(np.isfinite(lp_s)) and np.all(np.isfinite(white))))
        rows.append(row)
        print(name, row, flush=True)
    eng.close()
    return dict(shape=name, n=int(wl['t'].shape[0]), nx=wl['nx'], nh=wl['nh'], n_star=n_star, cull='default (80)',
                rows=rows)


def main():
    out_path = sys.argv[sys.argv.index('--out') + 1] if '--out' in sys.argv else 'profiles/r06_predict_logpdf.json'
    res = dict(gpu=gpu_info(), method='host clock around calls that end in cudaStreamSynchronize, after one warm-up '
                                      'call of the same shape; mean of 2 calls for B <= 8, else 1; smf = 1; logpdf with '
                                      'noise = 1 and the whitened residuals',
               not_measured='the split of the scoring increment between the per-sample factorisations and the border / '
                            'scoring kernels; the split of the shared covariance between pair blocks and fold GEMMs')
    res['shapes'] = [probe_shape('toy', named_workload('toy'), 400, (1, 8, 64, 200)),
                     probe_shape('bench', sweep_workload(100000, 200), 1000, (1, 64))]
    os.makedirs(os.path.dirname(out_path) or '.', exist_ok=True)
    with open(out_path, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()

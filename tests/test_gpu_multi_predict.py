"""The sharded prediction paths (cgpcm_predict_f_cov, cgpcm_predict_logpdf, cgpcm_predict_f_batch) on 2 ranks against
one GPU: bitwise when rank 0 holds every observation, byte-identical ranks and 1e-6 agreement under balanced shards,
and the same -3 on every rank for an indefinite sample owned by rank 1.  Self-launches tools/check_multi_predict.py
under torchrun when at least two GPUs are visible.  On one GPU: a handle without observations (what a rank of a series
shorter than the world size holds) runs precompute and the three prediction paths."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
import cgpcm_b200
from tests.workload import named_workload

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_ranks_predict_like_one_gpu():
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(_free_port()), os.path.join(ROOT, 'tools', 'check_multi_predict.py')]
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
    assert p.returncode == 0, p.stdout[-3000:]
    assert 'OK multi predict' in p.stdout, p.stdout[-3000:]


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_no_observations(smf):
    """Every frozen training-side sum is zero and the three prediction paths run: finite outputs, exactly symmetric
    covariances, and the mixture score the log-sum-exp of the per-sample scores."""
    wl = named_workload('toy')
    eng = cgpcm_b200.Engine(wl['nh'], wl['nx'])
    eng.set_data(wl['t'][:0], wl['y'][:0], wl['th'], wl['tx'])
    eng.precompute(*wl['hyp'], reg=wl['reg'])
    fm = eng.frozen_mats()
    assert all(not np.any(np.asarray(fm[k])) for k in ('sum_Bxx', 'sum_Bhh', 'sum_b', 'sum_Ahx_y'))
    p, nh = wl['params'], wl['nh']
    rng = np.random.default_rng(0)
    S = np.stack([p[5:5 + nh] * (1 + .2 * rng.standard_normal(nh)) for _ in range(3)])
    t_star = np.linspace(0, 1, 30)
    _, cov, ms, cs, dr = eng.predict_f_cov(p, t_star, S, smf=smf, reg=wl['reg'], per_sample=True,
                                           noise=rng.standard_normal((30, 3)))
    mean, var, mb, vb = eng.predict_f_batch(p, t_star, S, smf=smf, reg=wl['reg'])
    lp, lp_s, white = eng.predict_logpdf(p, t_star, rng.standard_normal(30), S, smf=smf, reg=wl['reg'], white=True)
    for a in (cov, ms, cs, dr, mean, var, mb, vb, lp_s, white):
        assert np.all(np.isfinite(a))
    for b in range(3):
        assert np.array_equal(cs[b], cs[b].T)
    top = lp_s.max()
    assert abs(lp - (top + np.log(np.exp(lp_s - top).mean()))) <= 1e-12 * abs(lp)
    eng.close()

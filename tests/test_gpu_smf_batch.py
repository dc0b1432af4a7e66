"""cgpcm_elbo_smf_batch / Engine.elbo_smf_batch: the SMF bound and the slice sampler's log-likelihood for many filter
samples per call (rank-one contraction C1_b = sum_n w_bn w_bn^T, w_bn = A_n^T h_b) against the oracle and against the
single-sample cgpcm_elbo_smf in MODE_FROZEN; bitwise independence of the batch; VCGPCM.sample(chains=C)."""
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
import cgpcm_b200
from cgpcm_b200 import VCGPCM, Data, Session, config, MODE_FROZEN
from oracle import model as om
from tests.cases import make_case, ulp_noise

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = ['toy_small', 'toy_test', 'sweep_hi', 'crude', 'toy_acausal_model', 'toy_small_cid', 'ou', 'hrir']


def _engine(c, **opts):
    eng = cgpcm_b200.Engine(c['nh'], c['nx'], causal=c['causal'], causal_id=c['causal_id'])
    for k, v in opts.items():
        eng.set_option(k, v)
    eng.set_data(c['t'], c['y'], c['th'], c['tx'])
    return eng


def _samples(c, B, seed=5):
    rng = np.random.default_rng(seed)
    nh = c['nh']
    mu = c['params'][5:5 + nh]
    return np.stack([mu * (1 + .2 * rng.standard_normal(nh)) + .01 * rng.standard_normal(nh) for _ in range(B)])


def _check_against_single(eng, c, S, e, t, ll):
    for b in range(S.shape[0]):
        e1, t1, ll1 = eng.elbo_smf(c['params'], S[b], mode=MODE_FROZEN, reg=c['reg'])
        scale = max(abs(e1), np.abs(t1).max())
        assert abs(e[b] - e1) <= 1e-9 * scale and np.abs(t[b] - t1).max() <= 1e-9 * scale, (b, e[b], e1)
        assert abs(ll[b] - ll1) <= 1e-9 * max(abs(ll1), np.abs(t1[2:4]).max()), (b, ll[b], ll1)


@pytest.mark.parametrize('name', CASES)
def test_batch_matches_oracle_and_single_sample(name):
    c = make_case(name)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    S = _samples(c, 3)
    e, t, ll = eng.elbo_smf_batch(c['params'], S, reg=c['reg'])
    assert e.shape == (3,) and t.shape == (3, 7) and ll.shape == (3,)
    for b in range(S.shape[0]):
        om.PW_DISTS_EXACT = True
        try:
            (e0, t0, ll0), (en, tn, lln) = ulp_noise(
                lambda p, th: om.elbo_smf(p, c['t'], c['y'], th, c['tx'], c['reg'], S[b], causal=c['causal'],
                                          causal_id=c['causal_id']), c['params'], c['th'])
        finally:
            om.PW_DISTS_EXACT = False
        scale = max(abs(e0), np.abs(t0).max())
        assert abs(e[b] - e0) <= 1e-9 * scale + 3 * en and np.abs(t[b] - t0).max() <= 1e-9 * scale + 3 * tn
        assert abs(ll[b] - ll0) <= 1e-9 * max(abs(ll0), np.abs(t0[2:4]).max()) + 3 * lln
    _check_against_single(eng, c, S, e, t, ll)
    # loglik only / elbo only
    _, _, ll2 = eng.elbo_smf_batch(c['params'], S, reg=c['reg'], want_elbo=False)
    assert np.array_equal(ll2, ll)


def test_batch_with_narrow_windows_matches_oracle(capfd, monkeypatch):
    """'sweep_wide': 3000 observations over 40 inducing inputs in chunks of 256 observations, so the chunks contract
    narrow windows, at k_lo > 0 past the first, and neighbouring chunks add overlapping windows into the same C1 slab."""
    c = make_case('sweep_wide')
    monkeypatch.setenv('CGPCM_DEBUG_PLAN', '1')
    eng = _engine(c, chunk=256)
    eng.precompute(*c['hyp'], reg=c['reg'])
    capfd.readouterr()
    S = _samples(c, 2)
    e, t, ll = eng.elbo_smf_batch(c['params'], S, reg=c['reg'])
    plan = [tuple(int(v) for v in m) for m in re.findall(r'\((\d+) x (\d+) @(\d+)\)', capfd.readouterr().err)]
    assert len(plan) > 1 and all(kwp < c['nx'] for _, kwp, _ in plan) and any(k_lo > 0 for _, _, k_lo in plan), plan
    om.PW_DISTS_EXACT = True
    try:
        (e0, t0, ll0), (en, tn, lln) = ulp_noise(
            lambda p, th: om.elbo_smf(p, c['t'], c['y'], th, c['tx'], c['reg'], S[0]), c['params'], c['th'], trials=1)
    finally:
        om.PW_DISTS_EXACT = False
    scale = max(abs(e0), np.abs(t0).max())
    assert abs(e[0] - e0) <= 1e-9 * scale + 3 * en and np.abs(t[0] - t0).max() <= 1e-9 * scale + 3 * tn
    assert abs(ll[0] - ll0) <= 1e-9 * max(abs(ll0), np.abs(t0[2:4]).max()) + 3 * lln
    _check_against_single(eng, c, S, e, t, ll)


def test_batch_invariance_is_bitwise():
    c = make_case('toy_test')
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    S = _samples(c, 200, seed=7)
    e64, t64, ll64 = eng.elbo_smf_batch(c['params'], S[:64], reg=c['reg'])
    er, tr, llr = eng.elbo_smf_batch(c['params'], S[:64][::-1].copy(), reg=c['reg'])
    e1, t1, ll1 = eng.elbo_smf_batch(c['params'], S[5:6].copy(), reg=c['reg'])
    assert e64[5] == er[58] == e1[0] and ll64[5] == llr[58] == ll1[0]
    assert np.array_equal(t64[5], tr[58]) and np.array_equal(t64[5], t1[0])
    assert np.array_equal(e64, er[::-1]) and np.array_equal(ll64, llr[::-1])
    # other companions, other sizes, one size above the internal batch (200 > 64 samples per batch at this shape)
    for B in (1, 7, 64, 200):
        e, t, ll = eng.elbo_smf_batch(c['params'], S[:B], reg=c['reg'])
        assert np.array_equal(e, e64[:B]) if B <= 64 else np.array_equal(e[:64], e64)
        assert np.all(np.isfinite(e)) and np.all(np.isfinite(ll))
    e200, _, ll200 = eng.elbo_smf_batch(c['params'], S, reg=c['reg'])
    e_tail, _, ll_tail = eng.elbo_smf_batch(c['params'], S[150:].copy(), reg=c['reg'])
    assert np.array_equal(e200[150:], e_tail) and np.array_equal(ll200[150:], ll_tail)
    # run to run
    e2, t2, ll2 = eng.elbo_smf_batch(c['params'], S[:64], reg=c['reg'])
    assert np.array_equal(e2, e64) and np.array_equal(t2, t64) and np.array_equal(ll2, ll64)
    _check_against_single(eng, c, S[190:], e200[190:], eng.elbo_smf_batch(c['params'], S[190:], reg=c['reg'])[1],
                          ll200[190:])


@pytest.mark.parametrize('opts', [{'store': 0}, {'cull': 0}, {'gram': 2}], ids=['store0', 'cull0', 'gram2'])
def test_batch_with_options(opts):
    c = make_case('toy_test')
    eng = _engine(c, **opts)
    eng.precompute(*c['hyp'], reg=c['reg'])
    S = _samples(c, 4)
    e, t, ll = eng.elbo_smf_batch(c['params'], S, reg=c['reg'])
    om.PW_DISTS_EXACT = True
    try:
        (e0, t0, ll0), (en, tn, lln) = ulp_noise(
            lambda p, th: om.elbo_smf(p, c['t'], c['y'], th, c['tx'], c['reg'], S[0]), c['params'], c['th'])
    finally:
        om.PW_DISTS_EXACT = False
    scale = max(abs(e0), np.abs(t0).max())
    assert abs(e[0] - e0) <= 1e-9 * scale + 3 * en and np.abs(t[0] - t0).max() <= 1e-9 * scale + 3 * tn
    assert abs(ll[0] - ll0) <= 1e-9 * max(abs(ll0), np.abs(t0[2:4]).max()) + 3 * lln
    if opts.get('gram'):
        # the single-sample path contracts with the Psi tensor here: its noise is ~sqrt(N) larger (gram_kernels.cuh)
        for b in range(S.shape[0]):
            e1, t1, ll1 = eng.elbo_smf(c['params'], S[b], mode=MODE_FROZEN, reg=c['reg'])
            assert abs(e[b] - e1) <= 1e-8 * max(abs(e1), np.abs(t1).max())
    else:
        _check_against_single(eng, c, S, e, t, ll)


def test_batch_error_paths():
    c = make_case('toy_small')
    eng = _engine(c)
    S = _samples(c, 2)
    with pytest.raises(ValueError, match='precompute'):
        eng.elbo_smf_batch(c['params'], S, reg=c['reg'])
    eng.precompute(*c['hyp'], reg=c['reg'])
    L = cgpcm_b200.lib()
    e, t, ll = np.empty(1), np.empty(7), np.empty(1)
    assert L.cgpcm_elbo_smf_batch(eng._h, c['params'].ctypes.data, c['reg'], S.ctypes.data, 0, e.ctypes.data,
                                  t.ctypes.data, ll.ctypes.data) == -1
    with pytest.raises(ValueError):
        eng.elbo_smf_batch(c['params'], np.zeros((2, c['nh'] + 1)), reg=c['reg'])
    with pytest.raises(ValueError):
        eng.elbo_smf_batch(c['params'], np.zeros((0, c['nh'])), reg=c['reg'])
    bad = S.copy()
    bad[1, 3] = np.nan
    with pytest.raises(ValueError, match='sample 1'):
        eng.elbo_smf_batch(c['params'], bad, reg=c['reg'])
    p = c['params'].copy()
    p[0] = np.inf
    with pytest.raises(ValueError):
        eng.elbo_smf_batch(p, S, reg=c['reg'])
    # still usable after the errors
    e, _, ll = eng.elbo_smf_batch(c['params'], S, reg=c['reg'])
    assert np.all(np.isfinite(e)) and np.all(np.isfinite(ll))


def test_bench_order_batch_matches_single_sample():
    f = os.path.join(ROOT, 'tests', 'golden', 'bench_m200.npz')
    d = dict(np.load(f))
    reg = float(d['reg'])
    nh, nx = len(d['th']), len(d['tx'])
    eng = cgpcm_b200.Engine(nh, nx, causal=True)
    eng.set_data(d['t'], d['y'], d['th'], d['tx'])
    eng.precompute(*np.exp(d['params'][2:5]), reg=reg)
    c = dict(params=d['params'], nh=nh, reg=reg)
    S = _samples(c, 16)
    e, t, ll = eng.elbo_smf_batch(d['params'], S, reg=reg)
    _check_against_single(eng, c, S, e, t, ll)


def test_sampler_with_several_chains():
    c = make_case('toy_small')
    config.reg = c['reg']
    try:
        np.random.seed(11)
        sess = Session()
        mod = VCGPCM.from_recipe(sess, Data(c['t'], c['y']), nx=c['nx'], nh=c['nh'], tau_w=.1, tau_f=.05, causal=True,
                                 noise_init=1e-2)
        mod.precompute()
        mod.fpi(5)
        mod.undo_precompute()
        out = mod.sample(iters=12, burn=4, chains=3)
        assert len(out) == 3 and all(len(ch) == 12 for ch in out)
        assert all(s.shape == (c['nh'], 1) and np.all(np.isfinite(s)) for ch in out for s in ch)
        assert not np.array_equal(out[0][-1], out[1][-1]) and not np.array_equal(out[1][-1], out[2][-1])
        assert not mod._precomputed                  # the frozen statistics were temporary
        est, se = mod.elbo_smf([s for ch in out for s in ch])
        assert np.isfinite(est) and se >= 0
    finally:
        config.reg = 1e-8


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs two GPUs')
def test_two_ranks_batch_agrees_with_one_gpu():
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', str(_free_port()), os.path.join(ROOT, 'tools', 'check_smf_batch_multi.py')]
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:]
    assert 'OK\n' in p.stdout, p.stdout[-3000:]

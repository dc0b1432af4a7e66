"""Batched SMF scoring (cgpcm_elbo_smf_batch) at the bench's M = nh = nx = 200 against the oracle, on a 97-observation
slice of the sweep workload (inducing inputs on both sides; the last chunk of every plan is ragged and padded): windows
of 7 DMMA tiles with a ragged last tile, several chunks adding windows at k_lo > 0, the 200 x 200 factorisations.  Also
the single-sample cgpcm_elbo_smf in both regimes, batch invariance above the internal batch of 64 samples, the
resident Ahx blocks across interleaved calls of other kinds, and device-pointer arguments."""
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
import cgpcm_b200
from cgpcm_b200 import _lib, MODE_FROZEN, MODE_FULL
from oracle import model as om
from tests.cases import ulp_noise
from tests.workload import sweep_workload

M, N_OBS = 200, 97
OPTS = [dict(cull=0.0, chunk=48, store=1), dict(cull=80.0, chunk=64, store=0), dict(cull=80.0, chunk=32)]
OPT_IDS = ['dense_store', 'cull_nostore', 'cull_narrow']


def _samples(params, B, seed=5):
    rng = np.random.default_rng(seed)
    mu = params[5:5 + M]
    return np.stack([mu * (1 + .2 * rng.standard_normal(M)) + .01 * rng.standard_normal(M) for _ in range(B)])


@pytest.fixture(scope='module')
def case():
    w = sweep_workload(4000, M, seed=3)
    sl = slice(1000, 1000 + N_OBS)
    t, y = np.ascontiguousarray(w['t'][sl]), np.ascontiguousarray(w['y'][sl])
    S = _samples(w['params'], 3)
    oracle = []
    om.PW_DISTS_EXACT = True
    try:
        for b in range(S.shape[0]):
            oracle.append(ulp_noise(lambda p, th: om.elbo_smf(p, t, y, th, w['tx'], w['reg'], S[b]), w['params'],
                                    w['th'], trials=1))
    finally:
        om.PW_DISTS_EXACT = False
    return dict(w=w, t=t, y=y, S=S, oracle=oracle)


def _engine(c, **opts):
    eng = cgpcm_b200.Engine(M, M)
    for k, v in opts.items():
        eng.set_option(k, v)
    eng.set_data(c['t'], c['y'], c['w']['th'], c['w']['tx'])
    return eng


def _check_oracle(c, b, e, t, ll, what):
    (e0, t0, ll0), (en, tn, lln) = c['oracle'][b]
    scale = max(abs(e0), np.abs(t0).max())
    assert abs(e - e0) <= 1e-9 * scale + 3 * en, (what, b, e, e0)
    assert np.abs(t - t0).max() <= 1e-9 * scale + 3 * tn, (what, b, t, t0)
    assert abs(ll - ll0) <= 1e-9 * max(abs(ll0), np.abs(t0[2:4]).max()) + 3 * lln, (what, b, ll, ll0)


@pytest.fixture(scope='module')
def dense_flops(case):
    eng = _engine(case, **OPTS[0])
    w = case['w']
    eng.precompute(*w['hyp'], reg=w['reg'])
    eng.elbo_smf_batch(w['params'], case['S'], reg=w['reg'])
    f = eng.last_timing()['gemm_flops']
    eng.close()
    return f


@pytest.mark.parametrize('opts', OPTS, ids=OPT_IDS)
def test_batch_and_single_sample_match_oracle_at_m200(case, opts, dense_flops, capfd, monkeypatch):
    w, S = case['w'], case['S']
    monkeypatch.setenv('CGPCM_DEBUG_PLAN', '1')
    eng = _engine(case, **opts)
    try:
        for b in range(S.shape[0]):                       # the full regime needs no precompute
            e1, t1, ll1 = eng.elbo_smf(w['params'], S[b], mode=MODE_FULL, reg=w['reg'])
            _check_oracle(case, b, e1, t1, ll1, 'single, full regime')
        eng.precompute(*w['hyp'], reg=w['reg'])
        capfd.readouterr()
        e, t, ll = eng.elbo_smf_batch(w['params'], S, reg=w['reg'])
        flops = eng.last_timing()['gemm_flops']
        plan = [tuple(int(v) for v in m) for m in re.findall(r'\((\d+) x (\d+) @(\d+)\)', capfd.readouterr().err)]
        assert len(plan) > 1 and sum(nv for nv, _, _ in plan) == N_OBS, plan
        for b in range(S.shape[0]):
            _check_oracle(case, b, e[b], t[b], ll[b], 'batch')
            e1, t1, ll1 = eng.elbo_smf(w['params'], S[b], mode=MODE_FROZEN, reg=w['reg'])
            _check_oracle(case, b, e1, t1, ll1, 'single, frozen regime')
        if opts['cull']:
            assert flops < dense_flops                    # the culled plans contract narrower windows
            if opts['chunk'] == 32:
                assert any(0 < k_lo and kwp < M for _, kwp, k_lo in plan), plan
        else:
            assert flops == dense_flops
            assert all(kwp == M and k_lo == 0 for _, kwp, k_lo in plan), plan
    finally:
        eng.close()


def test_batch_invariance_above_the_internal_batch_at_m200(case):
    """B = 70 > 64 samples per internal batch: every sample's results are bitwise those of sub-batches and of the
    reversed batch."""
    w = case['w']
    eng = _engine(case, cull=80.0)
    eng.precompute(*w['hyp'], reg=w['reg'])
    S = _samples(w['params'], 70, seed=9)
    e, t, ll = eng.elbo_smf_batch(w['params'], S, reg=w['reg'])
    assert np.all(np.isfinite(e)) and np.all(np.isfinite(ll))
    er, tr, llr = eng.elbo_smf_batch(w['params'], S[::-1].copy(), reg=w['reg'])
    assert np.array_equal(er[::-1], e) and np.array_equal(tr[::-1], t) and np.array_equal(llr[::-1], ll)
    for a, b in ((0, 64), (64, 70), (3, 10), (69, 70)):
        es, ts, lls = eng.elbo_smf_batch(w['params'], S[a:b].copy(), reg=w['reg'])
        assert np.array_equal(es, e[a:b]) and np.array_equal(ts, t[a:b]) and np.array_equal(lls, ll[a:b]), (a, b)
    _, _, ll_only = eng.elbo_smf_batch(w['params'], S, reg=w['reg'], want_elbo=False)
    assert np.array_equal(ll_only, ll)
    eng.close()


def test_resident_blocks_survive_interleaved_calls(case):
    """With the sweep stores the batch path reuses the frozen regime's resident Ahx blocks.  Calls that overwrite them
    (full-regime sweeps at other hyper-parameters) or re-freeze must make it regenerate them: after each call the batch
    result is bitwise the recorded one, and a fresh engine's."""
    w, S = case['w'], case['S']
    reg = w['reg']
    other = w['params'].copy()
    other[2:5] += np.log([1.3, 0.8, 1.2])                # other alpha, gamma, omega: other Ahx blocks
    eng = _engine(case, store=1)
    eng.precompute(*w['hyp'], reg=reg)
    rec = eng.elbo_smf_batch(w['params'], S, reg=reg)

    def fresh():
        f = _engine(case, store=1)
        f.precompute(*w['hyp'], reg=reg)
        out = f.elbo_smf_batch(w['params'], S, reg=reg)
        f.close()
        return out

    def same(step):
        got = eng.elbo_smf_batch(w['params'], S, reg=reg)
        for g, r in zip(got, rec):
            assert np.array_equal(g, r), step

    steps = [
        ('full elbo_grad', lambda: eng.elbo_grad(other, mode=MODE_FULL, reg=reg)),
        ('elbo_smf full', lambda: eng.elbo_smf(other, S[0], mode=MODE_FULL, reg=reg)),
        ('frozen elbo_grad', lambda: eng.elbo_grad(w['params'], mode=MODE_FROZEN, reg=reg)),
        ('predict_f', lambda: eng.predict_f(w['params'], case['t'][::7].copy(), S[:2], smf=True, reg=reg)),
        ('precompute elsewhere and back', lambda: (eng.precompute(*np.exp(other[2:5]), reg=reg),
                                                   eng.precompute(*w['hyp'], reg=reg))),
    ]
    for name, fn in steps:
        fn()
        same(name)
    for g, r in zip(fresh(), rec):
        assert np.array_equal(g, r)
    eng.close()


def test_device_pointer_arguments(case):
    """params, samples and outputs as CUDA tensors: bitwise the host-array results, with and without loglik, and with
    loglik alone."""
    w, S = case['w'], case['S']
    reg = w['reg']
    eng = _engine(case)
    eng.precompute(*w['hyp'], reg=reg)
    e, t, ll = eng.elbo_smf_batch(w['params'], S, reg=reg)
    L = _lib.lib()
    B = S.shape[0]
    dev = lambda a: torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')
    dp, dS = dev(w['params']), dev(S)
    for with_elbo, with_ll in ((True, True), (True, False), (False, True)):
        de = torch.full((B,), np.nan, dtype=torch.float64, device='cuda') if with_elbo else None
        dt = torch.full((B, 7), np.nan, dtype=torch.float64, device='cuda') if with_elbo else None
        dl = torch.full((B,), np.nan, dtype=torch.float64, device='cuda') if with_ll else None
        rc = L.cgpcm_elbo_smf_batch(eng._h, dp.data_ptr(), reg, dS.data_ptr(), B, _lib.ptr(de), _lib.ptr(dt),
                                    _lib.ptr(dl))
        assert rc == 0
        if with_elbo:
            assert np.array_equal(de.cpu().numpy(), e) and np.array_equal(dt.cpu().numpy(), t)
        if with_ll:
            assert np.array_equal(dl.cpu().numpy(), ll)
    eng.close()

"""cgpcm_predict_logpdf / Engine.predict_logpdf / VCGPCM.log_predictive_density: the log predictive density of a
held-out block per filter sample and for the mixture of the samples.  The scoring stage against numpy on the GPU's own
means and covariances, lp_s against tests.pair_oracle.predict_f_cov, the joint density at one input against the
marginal path, the mixture's log-sum-exp, the calibration of the whitened residuals, bitwise independence of the batch,
the bench's M = 200 with device pointers, the error paths and the model API."""
import numpy as np
import pytest
from scipy.linalg import solve_triangular
from scipy.stats import norm

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
from cgpcm_b200 import _lib, VCGPCM, Data, Session, config
from tests.cases import make_case
from tests.test_gpu_predict_cov import _draws, _engine, _oracle, _t_star, _trained
from tests.workload import sweep_workload

EPS = np.finfo(np.float64).eps
LOG2PI = np.log(2 * np.pi)
CASES = ['toy_small', 'crude', 'toy_acausal_model', 'hrir']


def _y_star(c, t_star, seed=0):
    """Held-out values at t_star: the observations interpolated (held at the ends past the series) plus noise."""
    rng = np.random.default_rng(seed)
    return np.interp(t_star, c['t'], c['y']) + .3 * rng.standard_normal(t_star.size)


def _numpy_score(y, m, C, d):
    """lp = log N(y; m, C + d I), z = L^-1 (y - m) and cond(C + d I), all in float64 on the host."""
    S = C + d * np.eye(y.size)
    L = np.linalg.cholesky(S)
    z = solve_triangular(L, y - m, lower=True)
    lp = -.5 * (y.size * LOG2PI + 2 * np.log(np.diag(L)).sum() + z @ z)
    w = np.linalg.eigvalsh(S)                 # cond of a symmetric positive definite S: seconds at n = 4096
    return lp, z, w[-1] / w[0]


def _check_scoring(lp_s, white, y, ms, cs, d):
    """lp_s to 1e-10 relative, plus the conditioning term below (which is far smaller on these cases).  The whitened
    residuals: the GPU's and numpy's factors of S_b are each backward stable (|dS| <= n eps |S|), so the two z differ
    by at most about |L^-1 dL z| <= n eps cond(S_b) |z|; held to 4 n eps cond(S_b) |z| (absolute, per entry)."""
    n = y.size
    for b in range(ms.shape[1]):
        ref, z, cond = _numpy_score(y, ms[:, b], cs[b], d)
        tol = 1e-10 * abs(ref) + 4 * n * EPS * cond * (z @ z + n)
        assert abs(lp_s[b] - ref) <= tol, (b, lp_s[b], ref, abs(lp_s[b] - ref) / abs(ref))
        wtol = 4 * n * EPS * cond * np.linalg.norm(z)
        assert np.abs(white[:, b] - z).max() <= wtol, (b, np.abs(white[:, b] - z).max(), wtol)


def _lse(lp_s):
    top = lp_s.max()
    acc = 0.0
    for v in lp_s:
        acc += np.exp(v - top)
    return top + np.log(acc) - np.log(lp_s.size)


def _oracle_bound(y, m0, C0, noise, d):
    """Bound on |lp(m, C) - lp(m0, C0)| for |m - m0| <= em and max |C - C0| <= eC (the documented agreement of the
    means and covariances with the oracle, tests/test_gpu_predict_cov.py: 1e-8 of max |m0| and of max(|C0|, m0^2),
    plus three times the oracle's own 2-ulp sensitivity).  With S = C0 + d I, u = S^-1 (y - m0) and |dC|_2 <= n eC:
        |d log det S| = |tr(S^-1 dC)| <= n |dC|_2 / lambda_min(S),
        |d (y - m)^T S^-1 (y - m)| <= 2 |dm| |u| + |u|^2 |dC|_2   (first order),
    and lp = -(n log 2 pi + log det S + (y - m)^T S^-1 (y - m)) / 2; doubled for the second-order terms."""
    (em, eC) = noise
    n = y.size
    S = C0 + d * np.eye(n)
    lam = np.linalg.eigvalsh(S).min()
    u = np.linalg.solve(S, y - m0)
    dC = n * eC
    return (n * dC / lam + 2 * np.sqrt(n) * em * np.linalg.norm(u) + (u @ u) * dC)


_ORACLE = {}


@pytest.mark.parametrize('noise', [True, False], ids=['noise', 'f'])
@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
@pytest.mark.parametrize('name', CASES)
def test_scoring_matches_numpy_and_the_oracle(name, smf, noise):
    c = make_case(name)
    p = _trained(c)
    S = _draws(p, c['nh'], c['reg'], 3)
    t_star = _t_star(c['t'])                  # 19 points across the series and one past each end
    y = _y_star(c, t_star)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    d = np.exp(p[0]) if noise else c['reg']
    _, _, ms, cs, _ = eng.predict_f_cov(p, t_star, S, smf=smf, reg=c['reg'], per_sample=True)
    lp, lp_s, white = eng.predict_logpdf(p, t_star, y, S, smf=smf, reg=c['reg'], noise=noise, white=True)
    assert lp_s.shape == (3,) and white.shape == (t_star.size, 3)
    # 1. the scoring stage on the GPU's own m_b and C_b
    _check_scoring(lp_s, white, y, ms, cs, d)
    assert abs(lp - _lse(lp_s)) <= 1e-15 * abs(lp)
    # 2. against the oracle's mean and covariance
    key = (name, smf)
    if key not in _ORACLE:
        _ORACLE[key] = _oracle(c, p, t_star, S, smf)
    (m0, C0), (mn, cn) = _ORACLE[key]
    em = 1e-8 * np.abs(m0).max() + 3 * mn
    eC = 1e-8 * max(np.abs(C0).max(), np.abs(m0).max() ** 2) + 3 * cn
    for b in range(3):
        ref = _numpy_score(y, m0[:, b], C0[b], d)[0]
        bound = 2 * _oracle_bound(y, m0[:, b], C0[b], (em, eC), d)
        assert abs(lp_s[b] - ref) <= bound, (b, lp_s[b], ref, bound)
    # the outputs one by one are the same bits
    L = _lib.lib()
    one = np.full(1, np.nan)
    only = np.full(3, np.nan)
    assert L.cgpcm_predict_logpdf(eng._h, p.ctypes.data, c['reg'], t_star.ctypes.data, y.ctypes.data, t_star.size,
                                  S.ctypes.data, 3, int(smf), int(noise), one.ctypes.data, only.ctypes.data,
                                  None) == 0
    assert one[0] == lp and np.array_equal(only, lp_s)


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_causal_id_indefinite_covariance_is_refused(smf):
    """The causal_id toy at its untrained parameters (training it fails: the oracle's q(z) is indefinite) has C_b with
    eigenvalues far below -d: numpy's Cholesky of C_b + d I fails, and so does the call, naming the first such sample."""
    c = make_case('toy_small_cid')
    p = c['params']
    S = _draws(p, c['nh'], c['reg'], 3)
    t_star = _t_star(c['t'])
    y = _y_star(c, t_star)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    _, _, ms, cs, _ = eng.predict_f_cov(p, t_star, S, smf=smf, reg=c['reg'], per_sample=True)
    for noise, d in ((True, np.exp(p[0])), (False, c['reg'])):
        first = None
        for b in range(3):
            try:
                _numpy_score(y, ms[:, b], cs[b], d)
            except np.linalg.LinAlgError:
                first = b
                break
        assert first is not None, 'expected an indefinite C_b + d I'
        with pytest.raises(_lib.CgpcmError,
                           match=r'C_b \+ d I of sample %d is not positive definite \(pivot \d+\)' % first) as e:
            eng.predict_logpdf(p, t_star, y, S, smf=smf, reg=c['reg'], noise=noise)
        assert e.value.code == -3


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_one_input_matches_the_marginal(smf):
    """At n_star = 1 the joint density is the marginal N(y; m_b, v_b + d).  diag(C_b) agrees with predict_f_batch's
    var_s to 1e-8 of max(|var|, mean^2), and the means to 1e-8 of |mean| (tests/test_gpu_predict_cov.py); with
    s = v + d and first-order propagation, |dlp| <= (dv / s) (1 + (y - m)^2 / s) / 2 + |y - m| dm / s."""
    c = make_case('toy_small')
    p = _trained(c)
    S = _draws(p, c['nh'], c['reg'], 4, seed=5)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    s2 = np.exp(p[0])
    lo, hi = c['t'].min(), c['t'].max()
    for t0, y0 in ((.37 * (lo + hi), .4), (hi + .05 * (hi - lo), -1.3)):
        ts, ys = np.array([t0]), np.array([y0])
        _, lp_s, _ = eng.predict_logpdf(p, ts, ys, S, smf=smf, reg=c['reg'])
        _, _, m, v = eng.predict_f_batch(p, ts, S, smf=smf, reg=c['reg'])
        m, v = m[0], v[0]
        sv = v + s2
        ref = -.5 * (LOG2PI + np.log(sv) + (y0 - m) ** 2 / sv)
        dv = 1e-8 * max(np.abs(v).max(), np.abs(m).max() ** 2)
        dm = 1e-8 * np.abs(m).max()
        bound = (dv / sv) * (1 + (y0 - m) ** 2 / sv) / 2 + np.abs(y0 - m) * dm / sv
        assert np.all(np.abs(lp_s - ref) <= 2 * bound), (lp_s, ref, bound)


def test_mixture_of_far_apart_densities():
    """A 400-point block of observations scored as f (noise = 0, d = reg): every lp_s is far below -800, where
    exp(lp_s) underflows; the mixture is still the host's shifted log-sum-exp, and lies in [max - log B, max]."""
    c = make_case('toy_small')
    p = _trained(c)
    S = _draws(p, c['nh'], c['reg'], 6, seed=8)
    t_star = np.linspace(c['t'].min() - .02, c['t'].max() + .02, 400)
    y = _y_star(c, t_star, seed=3)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    for smf in (False, True):
        lp, lp_s, _ = eng.predict_logpdf(p, t_star, y, S, smf=smf, reg=c['reg'], noise=False)
        assert np.all(lp_s < -800) and np.isfinite(lp)
        assert abs(lp - _lse(lp_s)) <= 1e-15 * abs(lp)
        assert lp_s.max() - np.log(6) <= lp <= lp_s.max()
        assert np.exp(lp_s).sum() == 0.0          # the naive mixture would be log 0


def test_whitened_residuals_are_calibrated():
    """y drawn from sample b's own predictive distribution (a posterior path of f plus sqrt(s2) noise, seeded): the
    whitened residuals of that sample have mean within 4 / sqrt(n) of 0 and variance within 4 sqrt(2 / n) of 1."""
    c = make_case('toy_small')
    p = _trained(c)
    S = _draws(p, c['nh'], c['reg'], 3, seed=12)
    n = 400
    t_star = np.linspace(c['t'].min(), c['t'].max(), n)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    rng = np.random.default_rng(21)
    draws = eng.predict_f_cov(p, t_star, S, smf=True, reg=c['reg'], noise=rng.standard_normal((n, 3)))[4]
    s2 = np.exp(p[0])
    for b in range(3):
        y = draws[:, b] + np.sqrt(s2) * rng.standard_normal(n)
        _, lp_s, white = eng.predict_logpdf(p, t_star, y, S, smf=True, reg=c['reg'], white=True)
        z = white[:, b]
        assert abs(z.mean()) <= 4 / np.sqrt(n), (b, z.mean())
        assert abs(z.var() - 1) <= 4 * np.sqrt(2 / n), (b, z.var())


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_batch_invariance_is_bitwise(smf):
    """At n_star = 2048 a sample's covariance and bordered slabs take 67 MB, so a group (~4 GB of them, at least one
    internal batch of at most 64 samples) holds at most 64: the 70 samples cross the internal batch and a group
    boundary."""
    c = make_case('toy_small')
    p = _trained(c)
    S = _draws(p, c['nh'], c['reg'], 70, seed=7)
    t_star = np.linspace(c['t'].min() - .05, c['t'].max() + .05, 2048)
    y = _y_star(c, t_star, seed=4)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    run = lambda SS: eng.predict_logpdf(p, t_star, y, SS, smf=smf, reg=c['reg'], white=True)
    lp, lp_s, white = run(S)
    assert np.all(np.isfinite(lp_s)) and np.all(np.isfinite(white))
    for b in (0, 63, 64, 69):
        _, a, aw = run(S[b:b + 1].copy())
        assert a[0] == lp_s[b] and np.array_equal(aw[:, 0], white[:, b]), b
    perm = np.random.default_rng(9).permutation(70)
    _, a, aw = run(S[perm].copy())
    assert np.array_equal(a, lp_s[perm]) and np.array_equal(aw, white[:, perm])


@pytest.fixture(scope='module')
def m200():
    w = sweep_workload(4000, 200, seed=3)
    sl = slice(1000, 1097)
    c = dict(t=np.ascontiguousarray(w['t'][sl]), y=np.ascontiguousarray(w['y'][sl]), th=w['th'], tx=w['tx'],
             reg=w['reg'], hyp=w['hyp'], causal=True, causal_id=False, nh=200, nx=200)
    S = _draws(w['params'], 200, w['reg'], 2, seed=4)
    t_star = _t_star(c['t'], n=13)
    return dict(c=c, p=w['params'], S=S, t_star=t_star, y=_y_star(c, t_star, seed=6))


@pytest.mark.parametrize('noise', [True, False], ids=['noise', 'f'])
@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_m200_with_device_pointers(m200, smf, noise):
    c, p, S, t_star, y = m200['c'], m200['p'], m200['S'], m200['t_star'], m200['y']
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    n = t_star.size
    _, _, ms, cs, _ = eng.predict_f_cov(p, t_star, S, smf=smf, reg=c['reg'], per_sample=True)
    dp, dt, dy, dS = (torch.tensor(a, dtype=torch.float64, device='cuda') for a in (p, t_star, y, S))
    dlp = torch.full((1,), np.nan, dtype=torch.float64, device='cuda')
    dls = torch.full((2,), np.nan, dtype=torch.float64, device='cuda')
    dw = torch.full((n, 2), np.nan, dtype=torch.float64, device='cuda')
    assert _lib.lib().cgpcm_predict_logpdf(eng._h, dp.data_ptr(), c['reg'], dt.data_ptr(), dy.data_ptr(), n,
                                           dS.data_ptr(), 2, int(smf), int(noise), dlp.data_ptr(), dls.data_ptr(),
                                           dw.data_ptr()) == 0
    lp_s, white = dls.cpu().numpy(), dw.cpu().numpy()
    _check_scoring(lp_s, white, y, ms, cs, np.exp(p[0]) if noise else c['reg'])
    lp, hs, hw = eng.predict_logpdf(p, t_star, y, S, smf=smf, reg=c['reg'], noise=noise, white=True)
    assert float(dlp.cpu()[0]) == lp and np.array_equal(hs, lp_s) and np.array_equal(hw, white)


def test_error_paths():
    c = make_case('toy_small')
    eng = _engine(c)
    p = _trained(c)
    S = _draws(p, c['nh'], c['reg'], 3)
    t_star = _t_star(c['t'], n=9)
    y = _y_star(c, t_star)
    n = t_star.size
    L = _lib.lib()
    lp, lps, wh = np.full(1, np.nan), np.full(3, np.nan), np.full(n * 3, np.nan)
    call = lambda ts, ys, nn, B=3, noise=1, reg=c['reg']: L.cgpcm_predict_logpdf(
        eng._h, p.ctypes.data, reg, ts.ctypes.data, ys.ctypes.data, nn, S.ctypes.data, B, 1, noise, lp.ctypes.data,
        lps.ctypes.data, wh.ctypes.data)
    good = lambda: eng.predict_logpdf(p, t_star, y, S, reg=c['reg'], white=True)
    # not precomputed
    assert call(t_star, y, n) == -1 and 'precompute' in L.cgpcm_last_error(eng._h).decode()
    with pytest.raises(ValueError, match='precompute'):
        good()
    eng.precompute(*c['hyp'], reg=c['reg'])
    ref = good()
    assert np.isfinite(ref[0])
    # bad arguments
    assert call(t_star, y, n, B=0) == -1
    big = np.linspace(0, 1, 4097)
    assert call(big, big, 4097) == -1 and '4096' in L.cgpcm_last_error(eng._h).decode()
    assert call(t_star, y, n, noise=2) == -1 and 'noise' in L.cgpcm_last_error(eng._h).decode()
    # non-finite y_star
    yb = y.copy()
    yb[3] = np.nan
    assert call(t_star, yb, n) == -4 and 'y_star' in L.cgpcm_last_error(eng._h).decode()
    with pytest.raises(ValueError, match='y_star'):
        eng.predict_logpdf(p, t_star, yb, S, reg=c['reg'])
    # n_star = 0: the empty block has density 1
    assert call(t_star, y, 0) == 0 and lp[0] == 0.0 and np.all(lps == 0.0)
    # a singular S_b: f scored with d = reg = 0 at a test input repeated 16 times
    ts = np.concatenate([np.full(16, t_star[4]), t_star])
    ys = _y_star(c, ts, seed=1)
    with pytest.raises(_lib.CgpcmError, match=r'matrix C_b \+ d I of sample \d+ is not positive definite \(pivot \d+\)') \
            as e:
        eng.predict_logpdf(p, ts, ys, S, smf=True, reg=0.0, noise=False)
    assert e.value.code == -3
    # the handle works after each error, with the same bits
    got = good()
    assert got[0] == ref[0] and np.array_equal(got[1], ref[1]) and np.array_equal(got[2], ref[2])


def test_vcgpcm_log_predictive_density():
    c = make_case('toy_small')
    config.reg = c['reg']
    try:
        np.random.seed(4)
        mod = VCGPCM.from_recipe(Session(), Data(c['t'], c['y']), nx=c['nx'], nh=c['nh'], tau_w=.1, tau_f=.05,
                                 causal=True, noise_init=1e-2)
        mod.precompute()
        mod.fpi(10)
        mod.undo_precompute()
        t = np.linspace(c['t'].min() - .05, c['t'].max() + .05, 31)
        y = _y_star(c, t, seed=2) * .3
        flat = [s for ch in mod.sample(iters=3, burn=2, chains=2) for s in ch]
        B = len(flat)
        s2 = float(np.exp(mod._pack()[0]))
        # joint=False: the mixture of the marginals, point by point
        for noise, d in ((True, s2), (False, config.reg)):
            lp, lp_s = mod.log_predictive_density(t, y, samples_h=flat, joint=False, noise=noise, per_sample=True)
            mean, var = mod.predict_f_samples(t, samples_h=flat)
            ref_s = norm.logpdf(y[:, None], mean, np.sqrt(var + d))
            assert np.abs(lp_s - ref_s).max() <= 1e-12 * np.abs(ref_s).max()
            from scipy.special import logsumexp
            ref = logsumexp(ref_s, axis=1) - np.log(B)
            assert lp.shape == (31,) and np.abs(lp - ref).max() <= 1e-12 * np.abs(ref).max()
            assert np.array_equal(mod.log_predictive_density(t, y, samples_h=flat, joint=False, noise=noise), lp)
        # joint=True: the Engine call
        lp, lp_s, white = mod.log_predictive_density(Data(t, y), Data(t, y), samples_h=flat, per_sample=True)
        assert not mod._precomputed and lp_s.shape == (B,) and white.shape == (31, B)
        mod.precompute()
        try:
            ref = mod.engine.predict_logpdf(mod._pack(), t, y, np.stack([s.ravel() for s in flat]), smf=True,
                                            reg=config.reg, noise=True, white=True)
        finally:
            mod.undo_precompute()
        assert lp == ref[0] and np.array_equal(lp_s, ref[1]) and np.array_equal(white, ref[2])
        assert mod.log_predictive_density(t, y, samples_h=flat) == lp
        # numeric samples_h: draws from q(u) under one q(z)
        assert np.isfinite(mod.log_predictive_density(t, y, samples_h=4))
        # a non-positive predictive variance is named
        eng_batch = mod.engine.predict_f_batch

        def neg(*a, **k):
            m, v, ms, vs = eng_batch(*a, **k)
            vs = vs.copy()
            vs[7, 2] = -1.0
            return m, v, ms, vs
        mod.engine.predict_f_batch = neg
        try:
            with pytest.raises(ValueError, match='sample 2 at point 7'):
                mod.log_predictive_density(t, y, samples_h=flat, joint=False)
        finally:
            del mod.engine.predict_f_batch
    finally:
        config.reg = 1e-8

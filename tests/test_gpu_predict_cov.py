"""cgpcm_predict_f_cov / Engine.predict_f_cov / VCGPCM.predict_f_cov / VCGPCM.sample_f: the joint predictive
covariance of f per filter sample and posterior draws of f.  Per sample against tests.pair_oracle.predict_f_cov, the
diagonal and the means against the shipped marginal paths, the structure of C_b, the draws against numpy, bitwise
independence of the batch, the bench's M = 200 with device pointers, the error paths, and the pair-block kernel against
float64 through its C-ABI hook."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
import cgpcm_b200
from cgpcm_b200 import _lib, VCGPCM, Data, Session, config
from oracle import model as om
from tests import pair_oracle as po
from tests.cases import make_case, ulp_noise
from tests.workload import sweep_workload

EPS = np.finfo(np.float64).eps
CASES = ['toy_small', 'crude', 'sweep_hi', 'toy_acausal_model', 'toy_small_cid', 'hrir']


def _engine(c, **opts):
    eng = cgpcm_b200.Engine(c['nh'], c['nx'], causal=c.get('causal', True), causal_id=c.get('causal_id', False))
    for k, v in opts.items():
        eng.set_option(k, v)
    eng.set_data(c['t'], c['y'], c['th'], c['tx'])
    return eng


def _trained(c, rounds=6):
    om.PW_DISTS_EXACT = True
    try:
        mu, var, _, _ = om.fpi(c['params'], c['t'], c['y'], c['th'], c['tx'], c['reg'], rounds,
                               causal=c['causal'], causal_id=c['causal_id'])
    finally:
        om.PW_DISTS_EXACT = False
    p = c['params'].copy()
    p[5:5 + c['nh']] = mu
    p[5 + c['nh']:] = var
    return p


def _draws(p, nh, reg, B, seed=2):
    rng = np.random.default_rng(seed)
    L = om.vec_to_tril(om.T(p[5 + nh:])).numpy()
    Lc = np.linalg.cholesky(L @ L.T + reg * np.eye(nh))
    return np.stack([p[5:5 + nh] + Lc @ rng.standard_normal(nh) for _ in range(B)])


def _t_star(t, n=19):
    lo, hi = t.min(), t.max()
    return np.concatenate([np.linspace(lo, hi, n), [lo - .05 * (hi - lo), hi + .05 * (hi - lo)]])


def _oracle(c, p, t_star, S, smf):
    om.PW_DISTS_EXACT = True
    try:
        return ulp_noise(lambda pp, th: po.predict_f_cov(pp, c['t'], c['y'], th, c['tx'], c['reg'], t_star, S, smf=smf,
                                                         causal=c['causal'], causal_id=c['causal_id']),
                         p, c['th'], trials=1)
    finally:
        om.PW_DISTS_EXACT = False


def _close_to_oracle(ms, cs, ref):
    (m0, C0), (mn, cn) = ref
    assert np.abs(ms - m0).max() <= 1e-8 * np.abs(m0).max() + 3 * mn, np.abs(ms - m0).max()
    scale = max(np.abs(C0).max(), np.abs(m0).max() ** 2)
    assert np.abs(cs - C0).max() <= 1e-8 * scale + 3 * cn, np.abs(cs - C0).max() / scale


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
@pytest.mark.parametrize('name', CASES)
def test_per_sample_matches_oracle(name, smf):
    c = make_case(name)
    p = c['params'] if c['causal_id'] else _trained(c)    # (the oracle's q(z) of the untrained causal_id toy is indefinite)
    S = _draws(p, c['nh'], c['reg'], 3)
    t_star = _t_star(c['t'])
    ref = _oracle(c, p, t_star, S, smf)
    eng = _engine(c)
    with pytest.raises(ValueError, match='precompute'):
        eng.predict_f_cov(p, t_star, S, smf=smf, reg=c['reg'])
    eng.precompute(*c['hyp'], reg=c['reg'])
    m, cov, ms, cs, dr = eng.predict_f_cov(p, t_star, S, smf=smf, reg=c['reg'], per_sample=True)
    n = t_star.size
    assert m.shape == (n,) and cov.shape == (n, n) and ms.shape == (n, 3) and cs.shape == (3, n, n) and dr is None
    _close_to_oracle(ms, cs, ref)
    # off the diagonal as well as on it: the pairs with t_p != t_q carry most of the entries
    off = ~np.eye(n, dtype=bool)
    assert np.abs(ref[0][1][:, off]).max() > 1e-3 * np.abs(ref[0][1]).max()


def _consistency_case(name, smf, B=5):
    c = make_case(name)
    p = _trained(c)
    S = _draws(p, c['nh'], c['reg'], B, seed=3)
    t_star = _t_star(c['t'], n=53)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    return c, p, S, t_star, eng


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
@pytest.mark.parametrize('name', ['toy_small', 'crude', 'hrir'])
def test_diagonal_and_means_match_the_marginal_paths(name, smf):
    c, p, S, t_star, eng = _consistency_case(name, smf)
    m, cov, ms, cs, _ = eng.predict_f_cov(p, t_star, S, smf=smf, reg=c['reg'], per_sample=True)
    mb, vb, msb, vsb = eng.predict_f_batch(p, t_star, S, smf=smf, reg=c['reg'])
    m1, v1 = eng.predict_f(p, t_star, S, smf=smf, reg=c['reg'])
    # The second moment is a difference of large terms (h h^T against iKh, Axx against A^T iKh A): two summation orders
    # of it differ by far more than 1e-12 of the variance (the oracle's own predict_f and predict_f_cov diagonals by up
    # to 6e-8 on these toys).  The diagonal is held to the tolerance between the batch and single paths
    # (tests/test_gpu_predict_batch.py).  The means cancel too (h_b^T A* over filter samples of mixed sign, on a GEMM
    # of another width than the batch call's): same tolerance.
    scale = max(np.abs(vsb).max(), np.abs(msb).max() ** 2)
    assert np.abs(ms - msb).max() <= 1e-8 * np.abs(msb).max(), np.abs(ms - msb).max() / np.abs(msb).max()
    for b in range(S.shape[0]):
        assert np.abs(np.diag(cs[b]) - vsb[:, b]).max() <= 1e-8 * scale, (b, np.abs(np.diag(cs[b]) - vsb[:, b]).max())
    assert np.abs(np.diag(cov) - v1).max() <= 1e-8 * scale, np.abs(np.diag(cov) - v1).max() / scale
    assert np.abs(m - m1).max() <= 1e-8 * np.abs(m1).max()
    # structure: exactly symmetric, positive semi-definite to rounding, cov = the average of the C_b
    for b in range(S.shape[0]):
        assert np.array_equal(cs[b], cs[b].T)
        assert np.linalg.eigvalsh(cs[b]).min() >= -1e-10 * np.abs(cs[b]).max()
    assert np.array_equal(cov, cov.T)
    assert np.abs(cov - cs.mean(0)).max() <= 1e-14 * np.abs(cs).max()
    # the outputs one by one (NULL elsewhere) are the same bits
    m2, cov2, ms2, cs2, _ = eng.predict_f_cov(p, t_star, S, smf=smf, reg=c['reg'])
    assert cs2 is None and np.array_equal(cov2, cov) and np.array_equal(ms2, ms)


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_draws_match_numpy(smf):
    c, p, S, t_star, eng = _consistency_case('toy_small', smf, B=4)
    reg = 1e-6
    eng.precompute(*c['hyp'], reg=reg)
    noise = np.random.default_rng(11).standard_normal((t_star.size, S.shape[0]))
    m, cov, ms, cs, dr = eng.predict_f_cov(p, t_star, S, smf=smf, reg=reg, per_sample=True, noise=noise)
    n = t_star.size
    for b in range(S.shape[0]):
        L = np.linalg.cholesky(cs[b] + reg * np.eye(n))
        ref = ms[:, b] + L @ noise[:, b]
        scale = np.abs(ms[:, b]).max() + np.abs(L).max() * np.abs(noise[:, b]).sum()
        assert np.abs(dr[:, b] - ref).max() <= 1e-10 * scale, (b, np.abs(dr[:, b] - ref).max() / scale)
    # the draws are the same with the other outputs absent
    L_ = _lib.lib()
    d2 = np.full((n, S.shape[0]), np.nan)
    assert L_.cgpcm_predict_f_cov(eng._h, p.ctypes.data, reg, t_star.ctypes.data, n, S.ctypes.data, S.shape[0],
                                  int(smf), None, None, None, noise.ctypes.data, d2.ctypes.data) == 0
    assert np.array_equal(d2, dr)


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_batch_invariance_is_bitwise(smf):
    c = make_case('toy_test')
    eng = _engine(c, chunk=64)
    reg = 1e-6
    eng.precompute(*c['hyp'], reg=reg)
    p = c['params']
    S = _draws(p, c['nh'], reg, 70, seed=7)
    t_star = _t_star(c['t'], n=41)
    noise = np.random.default_rng(5).standard_normal((t_star.size, 70))
    run = lambda SS, nn: eng.predict_f_cov(p, t_star, SS, smf=smf, reg=reg, per_sample=True, noise=nn)
    m, cov, ms, cs, dr = run(S, noise)
    assert np.all(np.isfinite(cs)) and np.all(np.isfinite(dr))
    # alone
    for b in (0, 65):
        _, _, a, ac, ad = run(S[b:b + 1].copy(), noise[:, b:b + 1].copy())
        assert np.array_equal(a[:, 0], ms[:, b]) and np.array_equal(ac[0], cs[b]) and np.array_equal(ad[:, 0], dr[:, b])
    # shuffled positions
    perm = np.random.default_rng(9).permutation(70)
    _, _, a, ac, ad = run(S[perm].copy(), noise[:, perm].copy())
    assert np.array_equal(a, ms[:, perm]) and np.array_equal(ac, cs[perm]) and np.array_equal(ad, dr[:, perm])
    # run to run
    m2, cov2, ms2, cs2, dr2 = run(S, noise)
    assert np.array_equal(cov2, cov) and np.array_equal(cs2, cs) and np.array_equal(dr2, dr)


@pytest.fixture(scope='module')
def m200():
    w = sweep_workload(4000, 200, seed=3)
    sl = slice(1000, 1097)
    c = dict(t=np.ascontiguousarray(w['t'][sl]), y=np.ascontiguousarray(w['y'][sl]), th=w['th'], tx=w['tx'],
             reg=w['reg'], hyp=w['hyp'], causal=True, causal_id=False, nh=200, nx=200)
    S = _draws(w['params'], 200, w['reg'], 2, seed=4)
    t_star = _t_star(c['t'], n=13)
    ref = {smf: _oracle(c, w['params'], t_star, S, smf) for smf in (False, True)}
    return dict(c=c, p=w['params'], S=S, t_star=t_star, ref=ref)


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_m200_matches_oracle_with_device_pointers(m200, smf):
    c, p, S, t_star = m200['c'], m200['p'], m200['S'], m200['t_star']
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    m, cov, ms, cs, _ = eng.predict_f_cov(p, t_star, S, smf=smf, reg=c['reg'], per_sample=True)
    _close_to_oracle(ms, cs, m200['ref'][smf])
    n = t_star.size
    dp, dt, dS = (torch.tensor(a, dtype=torch.float64, device='cuda') for a in (p, t_star, S))
    dms = torch.empty((n, 2), dtype=torch.float64, device='cuda')
    dcs = torch.empty((2, n, n), dtype=torch.float64, device='cuda')
    dcov = torch.empty((n, n), dtype=torch.float64, device='cuda')
    assert _lib.lib().cgpcm_predict_f_cov(eng._h, dp.data_ptr(), c['reg'], dt.data_ptr(), n, dS.data_ptr(), 2, int(smf),
                                          dms.data_ptr(), dcs.data_ptr(), dcov.data_ptr(), None, None) == 0
    assert np.array_equal(dms.cpu().numpy(), ms) and np.array_equal(dcs.cpu().numpy(), cs)
    assert np.array_equal(dcov.cpu().numpy(), cov)


def test_error_paths():
    c = make_case('toy_small')
    eng = _engine(c)
    p = c['params']
    S = _draws(p, c['nh'], c['reg'], 3)
    t_star = _t_star(c['t'], n=9)
    n = t_star.size
    noise = np.zeros((n, 3))
    with pytest.raises(ValueError, match='precompute'):
        eng.predict_f_cov(p, t_star, S, reg=c['reg'])
    eng.precompute(*c['hyp'], reg=c['reg'])
    L = _lib.lib()
    outs = [np.full(n * 3 * n, np.nan) for _ in range(4)]
    args = lambda: [o.ctypes.data for o in outs[:3]] + [noise.ctypes.data, outs[3].ctypes.data]
    assert L.cgpcm_predict_f_cov(eng._h, p.ctypes.data, c['reg'], t_star.ctypes.data, n, S.ctypes.data, 0, 1,
                                 *args()) == -1
    big = np.linspace(0, 1, 4097)
    assert L.cgpcm_predict_f_cov(eng._h, p.ctypes.data, c['reg'], big.ctypes.data, 4097, S.ctypes.data, 3, 1,
                                 *args()) == -1
    assert L.cgpcm_predict_f_cov(eng._h, p.ctypes.data, c['reg'], t_star.ctypes.data, n, S.ctypes.data, 3, 1,
                                 None, None, None, None, outs[3].ctypes.data) == -1          # draws without noise
    assert L.cgpcm_predict_f_cov(eng._h, p.ctypes.data, c['reg'], t_star.ctypes.data, 0, S.ctypes.data, 3, 1,
                                 *args()) == 0
    assert all(np.all(np.isnan(o)) for o in outs)           # n_star = 0 writes nothing
    m, cov, ms, cs, dr = eng.predict_f_cov(p, np.zeros(0), S, reg=c['reg'], per_sample=True)
    assert cov.shape == (0, 0) and ms.shape == (0, 3)
    bad = S.copy()
    bad[1, 3] = np.nan
    with pytest.raises(ValueError, match='sample 1'):
        eng.predict_f_cov(p, t_star, bad, reg=c['reg'])
    pb = p.copy()
    pb[1] = np.inf
    with pytest.raises(ValueError, match='parameter'):
        eng.predict_f_cov(pb, t_star, S, reg=c['reg'])
    tb = t_star.copy()
    tb[2] = np.nan
    with pytest.raises(ValueError, match='test input'):
        eng.predict_f_cov(p, tb, S, reg=c['reg'])
    nb = noise.copy()
    nb[4, 2] = np.inf
    with pytest.raises(ValueError, match='noise'):
        eng.predict_f_cov(p, t_star, S, reg=c['reg'], noise=nb)
    # a failing P_b (smf) and a failing C_b + reg I (one q(z); the huge sample makes C_b NaN) name the sample
    huge = S.copy()
    huge[2] *= 1e160
    with pytest.raises(_lib.CgpcmError, match=r'matrix P of sample 2 is not positive definite \(pivot \d+\)') as e:
        eng.predict_f_cov(p, t_star, huge, smf=True, reg=c['reg'], noise=noise)
    assert e.value.code == -3
    with pytest.raises(_lib.CgpcmError, match=r'C_b \+ reg I of sample 2 is not positive definite \(pivot \d+\)') as e:
        eng.predict_f_cov(p, t_star, huge, smf=False, reg=c['reg'], noise=noise)
    assert e.value.code == -3
    # still usable after the errors
    m2, cov2, _, _, dr2 = eng.predict_f_cov(p, t_star, S, smf=True, reg=c['reg'], noise=np.ones((n, 3)))
    assert np.all(np.isfinite(cov2)) and np.all(np.isfinite(dr2))


# ---- the pair-block kernel against float64

def _dev(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


@pytest.mark.parametrize('model', [dict(causal=True, causal_id=False), dict(causal=False, causal_id=False),
                                   dict(causal=True, causal_id=True)], ids=['causal', 'acausal', 'causal_id'])
@pytest.mark.parametrize('nx,np_,nq', [(1, 1, 1), (7, 5, 3), (8, 8, 8), (33, 7, 9), (200, 3, 5), (203, 2, 1),
                                       (640, 2, 2)])
@pytest.mark.parametrize('fold', [False, True], ids=['axx', 'fold'])
def test_pair_kernel_matches_float64(nx, np_, nq, fold, model):
    rng = np.random.default_rng(nx * 7 + np_ + nq)
    hyp = np.array([5., 30., 4. * nx])
    tx = np.linspace(0., 1., nx) if nx > 1 else np.array([.4])
    tp = rng.uniform(-.2, 1.2, np_)
    tq = rng.uniform(-.2, 1.2, nq)
    tq[0] = tp[0]                                      # one pair with t_p = t_q
    pad = lambda a: np.concatenate([a, np.full(3, np.nan)])   # entries past the counts are never read
    ref = po.psi_axx_pairs(tp, tq, tx, *hyp, **model).numpy().reshape(np_ * nq, nx, nx)
    gk = nx + 3
    ldg = nq * gk + 5
    G = None
    if fold:
        Gd = rng.standard_normal((np_, nx, nq, nx)) * np.abs(ref).max()
        G = np.full((np_ * gk, ldg), np.nan)            # NaN in the padding rows / columns of the fold
        for i in range(np_):
            for j in range(nq):
                G[i * gk:i * gk + nx, j * gk:j * gk + nx] = Gd[i, :, j, :]
        ref = ref - Gd.transpose(0, 2, 1, 3).reshape(np_ * nq, nx, nx)
    total = np_ * nq * nx * nx
    X = torch.full((total + 64,), np.nan, dtype=torch.float64, device='cuda')
    dG = _dev(G) if fold else None
    dtp, dtq, dtx = _dev(pad(tp)), _dev(pad(tq)), _dev(pad(tx))      # held: a freed block would be reused
    rc = _lib.lib().cgpcm_predict_pair_test(dtp.data_ptr(), np_, dtq.data_ptr(), nq,
                                            dtx.data_ptr(), nx, hyp.ctypes.data, int(model['causal']),
                                            int(model['causal_id']), dG.data_ptr() if fold else None,
                                            ldg if fold else 0, gk if fold else 0, X.data_ptr(), None)
    assert rc == 0
    out = X.cpu().numpy()
    assert np.all(np.isnan(out[total:]))                # nothing past the blocks is written
    got = out[:total].reshape(np_ * nq, nx, nx)
    assert np.all(np.isfinite(got))
    # the tolerance of the per-observation Axx against the oracle (tests/test_gpu_psi.py), plus the rounding of the fold
    atol = 1e-13 + (4 * EPS * np.abs(G[np.isfinite(G)]).max() if fold else 0.0)
    np.testing.assert_allclose(got, ref, rtol=1e-11, atol=atol)


def test_pair_hook_rejects_bad_shapes():
    L = _lib.lib()
    x = _dev(np.zeros(64))
    p = x.data_ptr()
    hyp = np.array([5., 30., 40.])
    assert L.cgpcm_predict_pair_test(p, 0, p, 1, p, 4, hyp.ctypes.data, 1, 0, None, 0, 0, p, None) == -1
    assert L.cgpcm_predict_pair_test(p, 1, p, 1, p, 4, hyp.ctypes.data, 1, 0, p, 8, 3, p, None) == -1     # gk < nx
    assert L.cgpcm_predict_pair_test(p, 1, p, 2, p, 4, hyp.ctypes.data, 1, 0, p, 6, 4, p, None) == -1     # ldg < nq gk
    bad = np.array([5., -1., 40.])
    assert L.cgpcm_predict_pair_test(p, 1, p, 1, p, 4, bad.ctypes.data, 1, 0, None, 0, 0, p, None) == -4


def test_vcgpcm_predict_f_cov_and_sample_f():
    c = make_case('toy_small')
    config.reg = c['reg']
    try:
        np.random.seed(4)
        mod = VCGPCM.from_recipe(Session(), Data(c['t'], c['y']), nx=c['nx'], nh=c['nh'], tau_w=.1, tau_f=.05,
                                 causal=True, noise_init=1e-2)
        mod.precompute()
        mod.fpi(10)
        mod.undo_precompute()
        t = np.linspace(c['t'].min(), c['t'].max(), 23)
        chains = mod.sample(iters=4, burn=2, chains=3)
        flat = [s for ch in chains for s in ch]
        mean, mix, ms, cs = mod.predict_f_cov(t, samples_h=flat, per_sample=True)
        assert mix.shape == (23, 23) and ms.shape == (23, 12) and cs.shape == (12, 23, 23) and not mod._precomputed
        mod.precompute()
        try:
            _, cov, ms2, _, _ = mod.engine.predict_f_cov(mod._pack(), t, np.stack([s.ravel() for s in flat]),
                                                         smf=True, reg=config.reg)
        finally:
            mod.undo_precompute()
        assert np.array_equal(ms2, ms)
        assert np.abs(mix - (cov + np.cov(ms, bias=True))).max() <= 1e-15 * np.abs(mix).max()
        # the sample-averaged part has predict_f's variance on its diagonal
        pred = mod.predict_f(t, samples_h=flat)
        assert np.abs(np.maximum(np.diag(cov), 0) ** .5 - pred.std.y).max() <= 1e-7 * max(pred.std.y.max(),
                                                                                           np.abs(pred.mean.y).max())
        assert np.abs(mean - pred.mean.y).max() <= 1e-8 * np.abs(pred.mean.y).max()
        # sample_f: one path per filter sample, the noise from the model's generator
        st = mod._rng.get_state()
        paths = mod.sample_f(t, samples_h=flat)
        mod._rng.set_state(st)
        noise = mod._rng.randn(t.size, len(flat))
        assert paths.shape == (23, 12) and np.all(np.isfinite(paths))
        mod.precompute()
        try:
            ref = mod.engine.predict_f_cov(mod._pack(), t, np.stack([s.ravel() for s in flat]), smf=True,
                                           reg=config.reg, noise=noise)[4]
        finally:
            mod.undo_precompute()
        assert np.array_equal(paths, ref)
        # numeric samples_h: draws from q(u), one q(z)
        m5, mix5 = mod.predict_f_cov(t, samples_h=5)
        assert mix5.shape == (23, 23) and m5.shape == (23,)
        assert np.abs(mix5 - mix5.T).max() <= 1e-14 * np.abs(mix5).max()
    finally:
        config.reg = 1e-8

"""cgpcm_predict_f_batch / Engine.predict_f_batch / VCGPCM.predict_f_samples: predict_f's moments per filter sample.
Per sample against the oracle's predict_f with that one sample, the averages against the single-sample path
cgpcm_predict_f, the bench's M = 200, bitwise independence of the batch, the error paths, and the two new kernels
(smf_posterior_kernel, predict_quad_kernel / predict_qb_kernel) against float64 numpy through their C-ABI hooks."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
import cgpcm_b200
from cgpcm_b200 import _lib, VCGPCM, Data, Session, config
from oracle import model as om
from tests.cases import make_case, ulp_noise
from tests.workload import sweep_workload

EPS = np.finfo(np.float64).eps
CASES = ['toy_small', 'crude', 'sweep_hi', 'toy_acausal_model', 'toy_small_cid', 'hrir']


def _engine(c, nh=None, nx=None, **opts):
    eng = cgpcm_b200.Engine(nh or c['nh'], nx or c['nx'], causal=c.get('causal', True),
                            causal_id=c.get('causal_id', False))
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


def _t_star(t, n=37):
    lo, hi = t.min(), t.max()
    return np.concatenate([np.linspace(lo, hi, n), [lo - .05 * (hi - lo), hi + .05 * (hi - lo)]])


def _oracle(c, p, t_star, S, smf):
    om.PW_DISTS_EXACT = True
    try:
        return [ulp_noise(lambda pp, th: om.predict_f(pp, c['t'], c['y'], th, c['tx'], c['reg'], t_star, S[b:b + 1],
                                                      smf=smf, causal=c['causal'], causal_id=c['causal_id']),
                          p, c['th'], trials=1) for b in range(S.shape[0])]
    finally:
        om.PW_DISTS_EXACT = False


def _close(m, v, m0, v0, mn, vn, what):
    assert np.abs(m - m0).max() <= 1e-8 * np.abs(m0).max() + 3 * mn, (what, np.abs(m - m0).max())
    assert np.abs(v - v0).max() <= 1e-8 * max(np.abs(v0).max(), np.abs(m0).max() ** 2) + 3 * vn, \
        (what, np.abs(v - v0).max())


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
        eng.predict_f_batch(p, t_star, S, smf=smf, reg=c['reg'])
    eng.precompute(*c['hyp'], reg=c['reg'])
    m, v, ms, vs = eng.predict_f_batch(p, t_star, S, smf=smf, reg=c['reg'])
    assert ms.shape == vs.shape == (t_star.size, 3) and m.shape == v.shape == (t_star.size,)
    for b, ((m0, v0), (mn, vn)) in enumerate(ref):
        _close(ms[:, b], vs[:, b], m0, v0, mn, vn, ('sample', b))
    # the averages against the single-sample path (and the oracle's bar of the samples)
    m1, v1 = eng.predict_f(p, t_star, S, smf=smf, reg=c['reg'])
    mn, vn = max(r[1][0] for r in ref), max(r[1][1] for r in ref)
    _close(m, v, m1, v1, mn, vn, 'single path')
    m2, v2, ms2, vs2 = eng.predict_f_batch(p, t_star, S, smf=smf, reg=c['reg'], per_sample=False)
    assert ms2 is None and vs2 is None and np.array_equal(m2, m) and np.array_equal(v2, v)


@pytest.mark.parametrize('name,opts', [('toy_small', {'store': 0}), ('toy_small', {'chunk': 32}),
                                       ('crude', {'gram': 1}), ('sweep_wide', {'chunk': 256})],
                         ids=['store0', 'chunk32', 'gram1', 'sweep_wide_chunk256'])
@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_averages_match_single_path(name, opts, smf):
    c = make_case(name)
    p = c['params'] if name == 'sweep_wide' else _trained(c)
    S = _draws(p, c['nh'], c['reg'], 5, seed=3)
    t_star = _t_star(c['t'], n=83)                     # chunk = 32: three chunks, a ragged last one
    eng = _engine(c, **opts)
    eng.precompute(*c['hyp'], reg=c['reg'])
    m, v, ms, vs = eng.predict_f_batch(p, t_star, S, smf=smf, reg=c['reg'])
    m1, v1 = eng.predict_f(p, t_star, S, smf=smf, reg=c['reg'])
    tol = 1e-8 if opts.get('gram') is None else 1e-7   # gram: the single path's noise is ~sqrt(N) larger
    assert np.abs(m - m1).max() <= tol * np.abs(m1).max(), np.abs(m - m1).max()
    assert np.abs(v - v1).max() <= tol * max(np.abs(v1).max(), np.abs(m1).max() ** 2), np.abs(v - v1).max()
    # per sample: the single path with that one sample
    for b in (0, 4):
        mb, vb = eng.predict_f(p, t_star, S[b:b + 1], smf=smf, reg=c['reg'])
        assert np.abs(ms[:, b] - mb).max() <= tol * np.abs(mb).max()
        assert np.abs(vs[:, b] - vb).max() <= tol * max(np.abs(vb).max(), np.abs(mb).max() ** 2)


@pytest.fixture(scope='module')
def m200():
    w = sweep_workload(4000, 200, seed=3)
    sl = slice(1000, 1097)
    c = dict(t=np.ascontiguousarray(w['t'][sl]), y=np.ascontiguousarray(w['y'][sl]), th=w['th'], tx=w['tx'],
             reg=w['reg'], hyp=w['hyp'], causal=True, causal_id=False, nh=200, nx=200)
    S = _draws(w['params'], 200, w['reg'], 2, seed=4)
    t_star = _t_star(c['t'], n=45)
    ref = {smf: _oracle(c, w['params'], t_star, S, smf) for smf in (False, True)}
    return dict(c=c, p=w['params'], S=S, t_star=t_star, ref=ref)


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
@pytest.mark.parametrize('opts', [dict(), dict(chunk=32, store=0, cull=0.0)], ids=['default', 'chunk32_dense'])
def test_m200_matches_oracle_and_single_path(m200, smf, opts):
    c, p, S, t_star = m200['c'], m200['p'], m200['S'], m200['t_star']
    eng = _engine(c, **opts)
    eng.precompute(*c['hyp'], reg=c['reg'])
    m, v, ms, vs = eng.predict_f_batch(p, t_star, S, smf=smf, reg=c['reg'])
    for b, ((m0, v0), (mn, vn)) in enumerate(m200['ref'][smf]):
        _close(ms[:, b], vs[:, b], m0, v0, mn, vn, ('sample', b))
    m1, v1 = eng.predict_f(p, t_star, S, smf=smf, reg=c['reg'])
    mn, vn = max(r[1][0] for r in m200['ref'][smf]), max(r[1][1] for r in m200['ref'][smf])
    _close(m, v, m1, v1, mn, vn, 'single path')
    # device pointers in, device pointers out
    dp, dt, dS = (torch.tensor(a, dtype=torch.float64, device='cuda') for a in (p, t_star, S))
    dm, dv = (torch.empty(t_star.size, dtype=torch.float64, device='cuda') for _ in range(2))
    dms, dvs = (torch.empty((t_star.size, 2), dtype=torch.float64, device='cuda') for _ in range(2))
    assert _lib.lib().cgpcm_predict_f_batch(eng._h, dp.data_ptr(), c['reg'], dt.data_ptr(), t_star.size,
                                            dS.data_ptr(), 2, int(smf), dm.data_ptr(), dv.data_ptr(),
                                            dms.data_ptr(), dvs.data_ptr()) == 0
    assert np.array_equal(dms.cpu().numpy(), ms) and np.array_equal(dvs.cpu().numpy(), vs)
    assert np.array_equal(dm.cpu().numpy(), m) and np.array_equal(dv.cpu().numpy(), v)


@pytest.mark.parametrize('smf', [False, True], ids=['qu', 'smf'])
def test_batch_invariance_is_bitwise(smf):
    c = make_case('toy_test')
    eng = _engine(c, chunk=64)
    eng.precompute(*c['hyp'], reg=c['reg'])
    p = c['params']
    S = _draws(p, c['nh'], c['reg'], 200, seed=7)
    t_star = _t_star(c['t'], n=150)
    m, v, ms, vs = eng.predict_f_batch(p, t_star, S, smf=smf, reg=c['reg'])
    assert np.all(np.isfinite(ms)) and np.all(np.isfinite(vs))
    # the averages are the per-sample moments averaged
    assert np.abs(m - ms.mean(1)).max() <= 1e-14 * np.abs(ms).max()
    assert np.abs(v - vs.mean(1)).max() <= 1e-14 * np.abs(vs).max()
    # alone, reversed, at another position, and run to run
    _, _, a, av = eng.predict_f_batch(p, t_star, S[130:131], smf=smf, reg=c['reg'])
    assert np.array_equal(a[:, 0], ms[:, 130]) and np.array_equal(av[:, 0], vs[:, 130])
    _, _, r, rv = eng.predict_f_batch(p, t_star, S[::-1].copy(), smf=smf, reg=c['reg'])
    assert np.array_equal(r[:, ::-1], ms) and np.array_equal(rv[:, ::-1], vs)
    _, _, q, qv = eng.predict_f_batch(p, t_star, S[120:].copy(), smf=smf, reg=c['reg'])
    assert np.array_equal(q, ms[:, 120:]) and np.array_equal(qv, vs[:, 120:])
    m2, v2, ms2, vs2 = eng.predict_f_batch(p, t_star, S, smf=smf, reg=c['reg'])
    assert np.array_equal(ms2, ms) and np.array_equal(vs2, vs) and np.array_equal(m2, m) and np.array_equal(v2, v)


def test_error_paths():
    c = make_case('toy_small')
    eng = _engine(c)
    p = c['params']
    S = _draws(p, c['nh'], c['reg'], 3)
    t_star = _t_star(c['t'], n=9)
    with pytest.raises(ValueError, match='precompute'):
        eng.predict_f_batch(p, t_star, S, reg=c['reg'])
    eng.precompute(*c['hyp'], reg=c['reg'])
    L = _lib.lib()
    out = [np.full(t_star.size * 3, np.nan) for _ in range(4)]
    assert L.cgpcm_predict_f_batch(eng._h, p.ctypes.data, c['reg'], t_star.ctypes.data, t_star.size, S.ctypes.data, 0,
                                   1, *[o.ctypes.data for o in out]) == -1
    assert L.cgpcm_predict_f_batch(eng._h, p.ctypes.data, c['reg'], t_star.ctypes.data, 0, S.ctypes.data, 3, 1,
                                   *[o.ctypes.data for o in out]) == 0
    assert all(np.all(np.isnan(o)) for o in out)           # n_star = 0 writes nothing
    m, v, ms, vs = eng.predict_f_batch(p, np.zeros(0), S, reg=c['reg'])
    assert m.shape == (0,) and ms.shape == (0, 3)
    bad = S.copy()
    bad[1, 3] = np.nan
    with pytest.raises(ValueError, match='sample 1'):
        eng.predict_f_batch(p, t_star, bad, reg=c['reg'])
    pb = p.copy()
    pb[1] = np.inf
    with pytest.raises(ValueError, match='parameter'):
        eng.predict_f_batch(pb, t_star, S, reg=c['reg'])
    tb = t_star.copy()
    tb[2] = np.nan
    with pytest.raises(ValueError, match='test input'):
        eng.predict_f_batch(p, tb, S, reg=c['reg'])
    with pytest.raises(ValueError):
        eng.predict_f_batch(p, t_star, np.zeros((2, c['nh'] + 1)), reg=c['reg'])
    # still usable after the errors
    m2, v2, _, _ = eng.predict_f_batch(p, t_star, S, smf=True, reg=c['reg'])
    assert np.all(np.isfinite(m2)) and np.all(np.isfinite(v2))


def test_failed_sample_is_reported_by_index():
    """A finite sample of magnitude 1e160 makes C1_b overflow, so that the factorisation of its P_b meets a NaN pivot:
    the call fails naming that sample, and the handle gives the same results as before afterwards."""
    c = make_case('toy_small')
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    p = c['params']
    S = _draws(p, c['nh'], c['reg'], 3)
    t_star = _t_star(c['t'], n=9)
    m0, v0, ms0, vs0 = eng.predict_f_batch(p, t_star, S, smf=True, reg=c['reg'])
    big = S.copy()
    big[2] *= 1e160
    with pytest.raises(_lib.CgpcmError, match=r'sample 2 is not positive definite \(pivot \d+\)') as e:
        eng.predict_f_batch(p, t_star, big, smf=True, reg=c['reg'])
    assert e.value.code == -3
    m, v, ms, vs = eng.predict_f_batch(p, t_star, S, smf=True, reg=c['reg'])
    assert np.array_equal(m, m0) and np.array_equal(v, v0) and np.array_equal(ms, ms0) and np.array_equal(vs, vs0)


# ---- kernel hooks against float64 numpy

def _dev(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _sym_rand(rng, n, scale=1.0):
    A = rng.standard_normal((n, n))
    return scale * (A @ A.T) / n


def _posterior_inputs(nx, nh, B, seed=0):
    rng = np.random.default_rng(seed)
    ld = max(((max(nx, nh) + 7) // 8) * 8, 8)
    nan = lambda shape: np.full(shape, np.nan)
    kx_f = _sym_rand(rng, nx) + np.eye(nx)
    sxx_f = _sym_rand(rng, nx, .3)
    c1_f = np.stack([_sym_rand(rng, nx, .5) for _ in range(B)])
    ikx_f = _sym_rand(rng, nx, .2)

    def lower(M):           # lower triangle at ld; the upper triangle and the padding are never read
        out = nan((ld, ld))
        il = np.tril_indices(nx)
        out[il] = M[il]
        return out
    kx, sxx, ikx = lower(kx_f), lower(sxx_f), lower(ikx_f)
    c1 = np.stack([lower(c1_f[b]) for b in range(B)])
    fy = nan((ld, ld))
    fy[:nh, :nx] = rng.standard_normal((nh, nx))
    ahh = nan((ld, ld))
    ahh[:nh, :nh] = _sym_rand(rng, nh)
    ldh = ((nh + 7) // 8) * 8 + 8
    hs = nan((B, ldh))
    hs[:, :nh] = rng.standard_normal((B, nh))
    return dict(nx=nx, nh=nh, B=B, ld=ld, ldh=ldh, kx=kx, sxx=sxx, c1=c1, fy=fy, ahh=ahh, ikx=ikx, hs=hs,
                full=dict(kx=kx_f, sxx=sxx_f, c1=c1_f, ikx=ikx_f), r=.7, c0=1.3, reg=1e-3, a=.4, tr=.25)


def _posterior_gpu(d, nslots=None):
    B, ld, nx = d['B'], d['ld'], d['nx']
    mx = torch.full((B, ld * ld), np.nan, dtype=torch.float64, device='cuda')
    xm = torch.full((B, ld), np.nan, dtype=torch.float64, device='cuda')
    q1 = torch.full((B,), np.nan, dtype=torch.float64, device='cuda')
    info = torch.full((B,), -7, dtype=torch.int32, device='cuda')
    ins = [_dev(d[k]) for k in ('kx', 'sxx', 'c1', 'fy', 'ahh', 'ikx')] + [_dev([d['tr']]), _dev(d['hs'])]
    rc = _lib.lib().cgpcm_smf_posterior_test(*[x.data_ptr() for x in ins], B, nslots or B, nx, d['nh'], ld, d['ldh'],
                                             d['r'], d['c0'], d['reg'], d['a'], mx.data_ptr(), xm.data_ptr(),
                                             q1.data_ptr(), info.data_ptr(), None)
    assert rc == 0
    return (mx.cpu().numpy()[:, :nx * nx].reshape(B, nx, nx), xm.cpu().numpy()[:, :nx], q1.cpu().numpy(),
            info.cpu().numpy(), mx.cpu().numpy()[:, nx * nx:], xm.cpu().numpy()[:, nx:])


def _posterior_ref(d, b):
    f, nx, nh = d['full'], d['nx'], d['nh']
    P = f['kx'] + d['r'] * (f['sxx'] + f['c1'][b]) + d['reg'] * np.eye(nx)
    h = d['hs'][b, :nh]
    lam = d['c0'] * d['fy'][:nh, :nx].T @ h
    Pi = np.linalg.inv(P)
    xm = Pi @ lam
    mx = Pi + np.outer(xm, xm) - f['ikx']
    q1 = d['a'] + h @ d['ahh'][:nh, :nh] @ h - d['tr']
    return mx, xm, q1, np.linalg.cond(P)


@pytest.mark.parametrize('nx,nh,B', [(1, 1, 1), (7, 3, 3), (8, 17, 3), (31, 40, 1), (33, 1, 3), (64, 200, 3),
                                     (200, 200, 3), (203, 64, 1), (640, 41, 1), (96, 96, 64)])
def test_posterior_kernel_matches_float64(nx, nh, B):
    d = _posterior_inputs(nx, nh, B, seed=nx + nh)
    mx, xm, q1, info, mx_pad, xm_pad = _posterior_gpu(d, nslots=max(B, 8))
    assert np.all(info == 0)
    assert np.all(np.isnan(mx_pad)) and np.all(np.isnan(xm_pad))       # nothing past the nx x nx block is written
    for b in range(B):
        mr, xr, qr, cond = _posterior_ref(d, b)
        tol = 50 * nx * EPS * cond
        assert np.abs(mx[b] - mr).max() <= tol * (np.abs(mr).max() + np.abs(xr).max() ** 2), (b, np.abs(mx[b] - mr).max())
        assert np.array_equal(mx[b], mx[b].T)
        assert np.abs(xm[b] - xr).max() <= tol * np.abs(xr).max()
        h = d['hs'][b, :nh]
        assert abs(q1[b] - qr) <= 10 * nh * EPS * (d['a'] + np.abs(h) @ np.abs(d['ahh'][:nh, :nh]) @ np.abs(h) + d['tr'])


@pytest.mark.parametrize('pivot', [0, 5, 63])
def test_posterior_kernel_reports_the_failed_pivot(pivot):
    nx, B = 64, 3
    d = _posterior_inputs(nx, 12, B, seed=pivot)
    good = _posterior_gpu(d)
    # sample 1: make pivot `pivot` negative (the leading block stays positive definite)
    bad = d['c1'].copy()
    kxp = d['full']['kx'][pivot, pivot] + d['r'] * (d['full']['sxx'][pivot, pivot] + 1e3)
    bad[1, pivot, pivot] = -kxp / d['r'] - 1e3
    d['c1'] = bad
    mx, xm, q1, info, _, _ = _posterior_gpu(d)
    assert info[1] == pivot + 1 and info[0] == 0 and info[2] == 0
    for b in (0, 2):
        assert np.array_equal(mx[b], good[0][b]) and np.array_equal(xm[b], good[1][b]) and q1[b] == good[2][b]
    assert np.all(np.isnan(mx[1])) and np.isnan(q1[1])                  # a failed sample writes nothing else


def _quad_case(nv, nx, B, shared=False, seed=0):
    rng = np.random.default_rng(seed)
    ldv = ((nx + 7) // 8) * 8 + 8
    v_stride = nv * ldv + 16
    V = np.full(B * v_stride, np.nan)
    Vd = rng.standard_normal((B, nv, nx))
    for b in range(B):
        blk = np.full((nv, ldv), np.nan)
        blk[:, :nx] = Vd[b]
        V[b * v_stride:b * v_stride + nv * ldv] = blk.ravel()
    nm = 1 if shared else B
    mx_stride = 0 if shared else nx * nx + 8
    Md = rng.standard_normal((nm, nx, nx))
    mx = np.full(max(nm * (nx * nx + 8), 1), np.nan)
    for b in range(nm):
        mx[b * (nx * nx + 8):b * (nx * nx + 8) + nx * nx] = Md[b].ravel()
    xm_stride = 0 if shared else nx + 3
    Xd = rng.standard_normal((nm, nx))
    xm = np.full(nm * (nx + 3), np.nan)
    for b in range(nm):
        xm[b * (nx + 3):b * (nx + 3) + nx] = Xd[b]
    Bxx = rng.standard_normal((nv, nx, nx))
    return dict(nv=nv, nx=nx, B=B, ldv=ldv, v_stride=v_stride, V=V, Vd=Vd, mx=mx, Md=Md, mx_stride=mx_stride,
                xm=xm, Xd=Xd, xm_stride=xm_stride, Bxx=Bxx, shared=shared)


def _quad_gpu(q, nslots=None, with_qb=True):
    nv, B = q['nv'], q['B']
    outs = [torch.full((nv, B), np.nan, dtype=torch.float64, device='cuda') for _ in range(3)]
    dV, dmx, dxm, dB = _dev(q['V']), _dev(q['mx']), _dev(q['xm']), _dev(q['Bxx'])
    rc = _lib.lib().cgpcm_predict_quad_test(dV.data_ptr(), q['v_stride'], q['ldv'], dmx.data_ptr(), q['mx_stride'],
                                            dxm.data_ptr(), q['xm_stride'], dB.data_ptr(), nv, q['nx'], B,
                                            nslots or B, outs[0].data_ptr(), outs[1].data_ptr(),
                                            outs[2].data_ptr() if with_qb else None, None)
    assert rc == 0
    return [o.cpu().numpy() for o in outs]


@pytest.mark.parametrize('nv,nx,B', [(1, 1, 1), (31, 7, 3), (33, 8, 3), (70, 31, 1), (64, 32, 64), (45, 33, 3),
                                     (97, 200, 3), (40, 203, 1), (33, 640, 1), (65, 96, 64)])
@pytest.mark.parametrize('shared', [False, True], ids=['per_sample', 'shared'])
def test_quad_kernels_match_float64(nv, nx, B, shared):
    q = _quad_case(nv, nx, B, shared=shared, seed=nv * nx + B)
    quad, lin, qb = _quad_gpu(q, nslots=max(B, 64))
    for b in range(B):
        m = 0 if shared else b
        M, x, Vb = q['Md'][m], q['Xd'][m], q['Vd'][b]
        ref_quad = np.einsum('nk,kl,nl->n', Vb, M, Vb)
        bound = np.einsum('nk,kl,nl->n', np.abs(Vb), np.abs(M), np.abs(Vb))
        assert np.all(np.abs(quad[:, b] - ref_quad) <= 4 * nx * EPS * bound + 1e-300)
        assert np.all(np.abs(lin[:, b] - Vb @ x) <= 2 * nx * EPS * (np.abs(Vb) @ np.abs(x)) + 1e-300)
        ref_qb = np.einsum('nkl,kl->n', q['Bxx'], M)
        bq = np.einsum('nkl,kl->n', np.abs(q['Bxx']), np.abs(M))
        assert np.all(np.abs(qb[:, b] - ref_qb) <= 4 * nx * EPS * bq + 1e-300)
    # a sample's outputs do not depend on the batch: alone and in a batch of other size
    if B > 1 and not shared:
        one = _quad_case(nv, nx, B, seed=nv * nx + B)
        one['V'] = one['V'][one['v_stride']:2 * one['v_stride']].copy()
        one['Vd'], one['Md'], one['Xd'] = one['Vd'][1:2], one['Md'][1:2], one['Xd'][1:2]
        one['mx'] = one['mx'][one['mx_stride']:2 * one['mx_stride']].copy()
        one['xm'] = one['xm'][one['xm_stride']:2 * one['xm_stride']].copy()
        one['B'] = 1
        q1_, l1_, b1_ = _quad_gpu(one, nslots=max(B, 64))
        assert np.array_equal(q1_[:, 0], quad[:, 1]) and np.array_equal(l1_[:, 0], lin[:, 1])
        assert np.array_equal(b1_[:, 0], qb[:, 1])


def test_hooks_reject_bad_shapes():
    L = _lib.lib()
    x = _dev(np.zeros(64))
    p = x.data_ptr()
    # ldv < nx, nslots < B, overlapping V slabs, mx stride shorter than nx^2
    assert L.cgpcm_predict_quad_test(p, 64, 4, p, 0, p, 0, None, 2, 8, 1, 1, p, p, None, None) == -1
    assert L.cgpcm_predict_quad_test(p, 64, 8, p, 0, p, 0, None, 2, 8, 2, 1, p, p, None, None) == -1
    assert L.cgpcm_predict_quad_test(p, 8, 8, p, 0, p, 0, None, 2, 8, 2, 2, p, p, None, None) == -1
    assert L.cgpcm_predict_quad_test(p, 64, 8, p, 10, p, 0, None, 2, 8, 2, 2, p, p, None, None) == -1
    assert L.cgpcm_predict_quad_test(p, 64, 8, p, 0, p, 0, None, 2, 8, 2, 2, p, p, p, None) == -1   # qb without bxx
    # ld < nx, nslots < B, nx beyond the shared-memory budget
    args = [p] * 8
    assert L.cgpcm_smf_posterior_test(*args, 1, 1, 16, 4, 8, 8, 1., 1., 0., 0., p, p, p, p, None) == -1
    assert L.cgpcm_smf_posterior_test(*args, 2, 1, 8, 4, 8, 8, 1., 1., 0., 0., p, p, p, p, None) == -1
    assert L.cgpcm_smf_posterior_test(*args, 1, 1, 4096, 4, 4096, 8, 1., 1., 0., 0., p, p, p, p, None) == -1


def test_predict_f_samples_api():
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
        chains = mod.sample(iters=6, burn=2, chains=4)
        flat = [s for ch in chains for s in ch]
        mean, var = mod.predict_f_samples(t, samples_h=flat)
        assert mean.shape == var.shape == (23, 24) and not mod._precomputed
        pred = mod.predict_f(t, samples_h=flat)
        m1 = pred.mean.y
        assert np.abs(mean.mean(1) - m1).max() <= 1e-8 * np.abs(m1).max()
        s1 = pred.std.y
        assert np.abs(np.maximum(var.mean(1), 0) ** .5 - s1).max() <= 1e-7 * max(s1.max(), np.abs(m1).max())
        mix = var.mean(1) + mean.var(1)
        assert np.all(mix >= var.mean(1))
        # numeric samples_h: draws from q(u), all under one q(z)
        st = mod._rng.get_state()
        mq, vq = mod.predict_f_samples(t, samples_h=5)
        mod._rng.set_state(st)
        pq = mod.predict_f(t, samples_h=5)
        assert mq.shape == (23, 5)
        assert np.abs(mq.mean(1) - pq.mean.y).max() <= 1e-8 * np.abs(pq.mean.y).max()
    finally:
        config.reg = 1e-8

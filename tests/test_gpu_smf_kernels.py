"""The kernels of batched SMF scoring (csrc/smf_batch.cuh) against float64 numpy, through the C-ABI hooks
cgpcm_smf_c1_test / cgpcm_smf_algebra_test, which launch them with the shapes cgpcm_elbo_smf_batch uses.

smf_c1_kernel + smf_reduce_kernel: C1_b = sum over windows of W_b^T W_b at (k_lo, k_lo), lower triangle of the leading
nx x nx block, at every window width (ragged last 32-wide tile), observation count (empty slices) and window position,
several windows overlapping in one slab, and bitwise independence of the batch.  smf_algebra_kernel: log det and
|L^-1 lam|^2 of P = Kx + r (sum_Bxx + C1) (+ reg I) and h^T sum_Bhh h across the 512-thread row stride, and the exit of
a factorisation that meets a non-positive pivot."""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
from cgpcm_b200 import _lib

EPS = np.finfo(np.float64).eps
NX, LD = 203, 208                    # nx not a multiple of 8: rows / columns nx..ld-1 of every slab must stay 0
KWPS = [8, 16, 24, 32, 40, 64, 72, 104, 200]
NCS = [8, 16, 24, 32, 40, 264, 2056]  # 8..24: slices 1..3 of the chunk are empty; 32, 40: slice 3 is empty


def _dev(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _c1_gpu(W, w_stride, B, windows, nx=NX, ld=LD):
    """c1 [B, ld, ld] from the hook; W is the host array of B samples at stride w_stride."""
    win = np.ascontiguousarray(np.asarray(windows, dtype=np.int64).reshape(-1, 4))
    dW = _dev(W)
    out = torch.full((B, ld, ld), np.nan, dtype=torch.float64, device='cuda')   # an element left unwritten stays NaN
    rc = _lib.lib().cgpcm_smf_c1_test(dW.data_ptr(), w_stride, B, win.shape[0], win.ctypes.data, nx, ld,
                                      out.data_ptr(), None)
    assert rc == 0
    return out.cpu().numpy()


def _c1_ref(W, w_stride, B, windows, nx=NX, ld=LD):
    """(reference, |W|^T |W| bound, mask of the elements the kernel computes)."""
    ref, bound = np.zeros((B, ld, ld)), np.zeros((B, ld, ld))
    for b in range(B):
        for k_lo, kwp, nc, off in windows:
            Wb = W[b * w_stride + off:b * w_stride + off + nc * kwp].reshape(nc, kwp)
            ref[b, k_lo:k_lo + kwp, k_lo:k_lo + kwp] += Wb.T @ Wb
            bound[b, k_lo:k_lo + kwp, k_lo:k_lo + kwp] += np.abs(Wb).T @ np.abs(Wb)
    mask = np.tril(np.ones((ld, ld), bool))
    mask[nx:, :] = False
    mask[:, nx:] = False
    return ref, bound, mask


def _check_c1(got, W, w_stride, B, windows):
    ref, bound, mask = _c1_ref(W, w_stride, B, windows)
    assert not np.any(np.isnan(got))
    assert np.all(got[:, ~mask] == 0.0)                  # upper triangle, rows and columns >= nx
    err = np.abs(got - ref)[:, mask]
    assert np.all(err <= 4e-15 * bound[:, mask] + 1e-300), err.max()


@pytest.mark.parametrize('nc', NCS)
@pytest.mark.parametrize('kwp', KWPS)
def test_c1_one_window(kwp, nc):
    """One window at k_lo = 0, 2 and the last position (nxp - kwp); 3 samples."""
    rng = np.random.default_rng(kwp * 10000 + nc)
    B, stride = 3, nc * kwp
    W = rng.standard_normal(B * stride)
    for k_lo in sorted({0, 2, LD - kwp}):
        win = [(k_lo, kwp, nc, 0)]
        _check_c1(_c1_gpu(W, stride, B, win), W, stride, B, win)


def _windows(nwin, big, rng):
    """nwin windows that all contain inducing input 100 (so every pair overlaps), packed one after another in a
    sample's W; one 2056-observation window when `big`."""
    out, off = [], 0
    for w in range(nwin):
        kwp = int(rng.choice(KWPS))
        nc = 2056 if big and w == nwin // 2 else int(rng.choice(NCS[:-1]))
        lo, hi = max(0, 100 - kwp + 2), min(100, LD - kwp)
        k_lo = int(rng.integers(lo // 2, hi // 2 + 1)) * 2
        out.append((k_lo, kwp, nc, off))
        off += nc * kwp
    return out, off


@pytest.mark.parametrize('B', [1, 3, 64])
@pytest.mark.parametrize('nwin', [1, 3, 7])
def test_c1_overlapping_windows_and_batch_invariance(nwin, B):
    """Several chunks add overlapping windows into one slab (k_lo > 0).  A sample's slab is bitwise the same alone, in
    the batch, and at the mirrored position of the reversed batch."""
    rng = np.random.default_rng(100 * nwin + B)
    win, stride = _windows(nwin, B <= 3, rng)
    stride += 8                                           # a gap between samples
    W = rng.standard_normal(B * stride)
    got = _c1_gpu(W, stride, B, win)
    _check_c1(got, W, stride, B, win)
    if B > 1:
        Wr = W.reshape(B, stride)[::-1].ravel()
        assert np.array_equal(_c1_gpu(Wr, stride, B, win)[::-1], got)
        for b in (0, B // 2, B - 1):
            assert np.array_equal(_c1_gpu(W[b * stride:(b + 1) * stride], stride, 1, win)[0], got[b])
        assert np.array_equal(_c1_gpu(W[stride:], stride, B - 1, win), got[1:])


def test_c1_hook_rejects_bad_windows():
    W = _dev(np.zeros(64 * 64))
    c1 = torch.zeros((1, LD, LD), dtype=torch.float64, device='cuda')
    L = _lib.lib()
    for win in [(0, 12, 8, 0), (0, 8, 12, 0), (1, 8, 8, 0), (LD - 6, 8, 8, 0), (0, 8, 8, 4090), (0, 0, 8, 0)]:
        w = np.array(win, dtype=np.int64)
        assert L.cgpcm_smf_c1_test(W.data_ptr(), 64 * 64, 1, 1, w.ctypes.data, NX, LD, c1.data_ptr(), None) == -1, win
    w = np.array((0, 8, 8, 0), dtype=np.int64)
    assert L.cgpcm_smf_c1_test(W.data_ptr(), 64 * 64, 1, 1, w.ctypes.data, NX, LD - 4, c1.data_ptr(), None) == -1
    assert L.cgpcm_smf_c1_test(W.data_ptr(), 64 * 64, 1, 1, w.ctypes.data, 210, LD, c1.data_ptr(), None) == -1


# ---- smf_algebra_kernel

R, C0 = 0.7, 1.3


def _alg_gpu(inp, want_p, want_p0):
    """(out [B, 5], info [B, 2]); every element the kernel must not read is NaN, as is every output not written."""
    kx, sxx, c1, fy, bhh, hs, nx, nh, ld, ldh, reg = (inp[k] for k in ('kx', 'sxx', 'c1', 'fy', 'bhh', 'hs', 'nx', 'nh',
                                                                      'ld', 'ldh', 'reg'))
    B = hs.shape[0]
    d = [_dev(a) for a in (kx, sxx, c1, fy, bhh, hs)]
    out = torch.full((B, 5), np.nan, dtype=torch.float64, device='cuda')
    info = torch.full((B, 2), -7, dtype=torch.int32, device='cuda')
    rc = _lib.lib().cgpcm_smf_algebra_test(*[a.data_ptr() for a in d], B, nx, nh, ld, ldh, R, C0, reg, want_p,
                                           want_p0, out.data_ptr(), info.data_ptr(), None)
    assert rc == 0
    return out.cpu().numpy(), info.cpu().numpy()


def _pad(a, shape, lower=False):
    """a in the top-left corner of a NaN array of `shape` (only its lower triangle when `lower`)."""
    out = np.full(shape, np.nan)
    v = np.where(np.tril(np.ones(a.shape[-2:], bool)), a, np.nan) if lower else a
    out[(Ellipsis,) + tuple(slice(0, s) for s in a.shape[-2:])] = v
    return out


def _spd(rng, n, floor):
    """A random SPD matrix: half its eigenvalues equal `floor`, the others O(1)."""
    G = rng.standard_normal((n, max(1, n // 2)))
    return G @ G.T / n + floor * np.eye(n)


def _indefinite(rng, n, size):
    """Symmetric, spectral norm `size`, smallest eigenvalue -size."""
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    e = rng.uniform(-1, 1, n)
    e[0] = -1.0
    return size * (Q * e) @ Q.T


def _alg_inputs(nx, nh, B, seed, reg=1e-3):
    """Kx SPD with jitter 1e-3; sum_Bxx indefinite with |r sum_Bxx| = lambda_min(Kx) / 2, so P0 = Kx + r (sum_Bxx + C1)
    stays positive definite for any C1 >= 0; C1_b = W_b^T W_b; random sum_Ahx_y, symmetric sum_Bhh, samples."""
    rng = np.random.default_rng(seed)
    ld, ldh = (max(nx, nh) + 7) // 8 * 8 + 8, (nh + 7) // 8 * 8 + 8
    kx = _spd(rng, nx, 1e-3)
    sxx = _indefinite(rng, nx, .5 * np.linalg.eigvalsh(kx)[0] / R)
    W = .3 * rng.standard_normal((B, 12, nx))
    c1 = np.einsum('bni,bnj->bij', W, W)
    fy = rng.standard_normal((nh, nx))
    bhh = rng.standard_normal((nh, nh))
    bhh = bhh + bhh.T
    hs = rng.standard_normal((B, nh))
    return dict(nx=nx, nh=nh, ld=ld, ldh=ldh, reg=reg, kx_m=kx, sxx_m=sxx, c1_m=c1, fy_m=fy, bhh_m=bhh, hs_m=hs,
                kx=_pad(kx, (ld, ld), True), sxx=_pad(sxx, (ld, ld), True), c1=_pad(c1, (B, ld, ld), True),
                fy=_pad(fy, (nh, ld)), bhh=_pad(bhh, (nh, ld)), hs=_pad(hs, (B, ldh)))


def _p_matrix(inp, b, kind):
    """P_b (kind 0, with reg) or P0_b (kind 1) formed as the kernel forms it: Kx + r (sum_Bxx + C1_b) (+ reg I)."""
    c1 = np.tril(inp['c1_m'][b]) + np.tril(inp['c1_m'][b], -1).T
    return inp['kx_m'] + R * (inp['sxx_m'] + c1) + (inp['reg'] * np.eye(inp['nx']) if kind == 0 else 0.0)


def _alg_ref(inp):
    """Per sample and kind: (log det, |L^-1 lam|^2, cond(P), bound of the rounding of lam_b's dot products propagated
    into |L^-1 lam|^2); per sample: (h^T sum_Bhh h, |h|^T |sum_Bhh| |h|)."""
    import scipy.linalg as sl
    B, nh = inp['hs_m'].shape
    res, hbh = np.zeros((B, 2, 4)), np.zeros((B, 2))
    for b in range(B):
        h = inp['hs_m'][b]
        lam = C0 * inp['fy_m'].T @ h
        # lam_k = c0 sum_i fy[i][k] h[i] in any order: |error| <= nh eps c0 (|fy|^T |h|)_k + eps |lam_k|
        dlam = nh * EPS * C0 * (np.abs(inp['fy_m']).T @ np.abs(h)) + EPS * np.abs(lam)
        for kind in range(2):
            P = _p_matrix(inp, b, kind)
            Lc = np.linalg.cholesky(P)
            z = sl.solve_triangular(Lc, lam, lower=True)
            x = sl.solve_triangular(Lc.T, z, lower=False)        # P^-1 lam: d(lam^T P^-1 lam) = 2 x^T dlam
            ev = np.linalg.eigvalsh(P)
            assert ev[0] > 0
            res[b, kind] = 2 * np.log(np.diag(Lc)).sum(), z @ z, ev[-1] / ev[0], 2 * np.abs(x) @ dlam
        hbh[b] = h @ inp['bhh_m'] @ h, np.abs(h) @ np.abs(inp['bhh_m']) @ np.abs(h)
    return res, hbh


def _mp_ref(inp, b, kind, dps=40):
    """(log det, |L^-1 lam|^2, h^T sum_Bhh h) in mpmath from the same float64 inputs."""
    import mpmath as mp
    with mp.workdps(dps):
        n, nh = inp['nx'], inp['nh']
        c1 = inp['c1_m'][b]
        P = mp.matrix(n, n)
        for i in range(n):
            for j in range(i + 1):
                v = mp.mpf(inp['kx_m'][i, j]) + mp.mpf(R) * (mp.mpf(inp['sxx_m'][i, j]) + mp.mpf(c1[i, j]))
                if i == j and kind == 0:
                    v += mp.mpf(inp['reg'])
                P[i, j] = P[j, i] = v
        h = [mp.mpf(x) for x in inp['hs_m'][b]]
        lam = mp.matrix([mp.mpf(C0) * mp.fsum(mp.mpf(inp['fy_m'][i, k]) * h[i] for i in range(nh)) for k in range(n)])
        Lc = mp.cholesky(P)
        z = mp.lu_solve(Lc, lam)
        logdet = 2 * mp.fsum(mp.log(Lc[i, i]) for i in range(n))
        hbh = mp.fsum(h[i] * mp.mpf(inp['bhh_m'][i, k]) * h[k] for i in range(nh) for k in range(nh))
        return float(logdet), float(mp.fsum(x * x for x in z)), float(hbh)


@functools.lru_cache(maxsize=None)
def _alg_case(nx, nh):
    inp = _alg_inputs(nx, nh, 3, seed=nx * 1000 + nh)
    return inp, _alg_ref(inp), _alg_gpu(inp, 1, 1)


def _close_alg(got, want, n):
    """want = (log det, |L^-1 lam|^2, cond(P), lam term).  log det to 4 n eps cond (absolute: a sum of log pivots);
    |L^-1 lam|^2 to 4 n eps cond relative -- the backward error of the factorisation is O(n eps |P|), and
    lam^T P^-1 lam moves by at most cond(P) times that, relatively -- plus twice the propagated rounding of lam (the GPU
    and the reference each round it once)."""
    tol = 4 * n * EPS * want[2]
    return (abs(got[0] - want[0]) <= tol * max(1.0, abs(want[0]) / n) and
            abs(got[1] - want[1]) <= tol * abs(want[1]) + 2 * want[3])


@pytest.mark.parametrize('wants', [(1, 1), (1, 0), (0, 1)], ids=['p_p0', 'p', 'p0'])
@pytest.mark.parametrize('nh', [1, 31, 32, 33, 200])
@pytest.mark.parametrize('nx', [1, 7, 8, 31, 33, 200, 511, 512, 513, 640])
def test_algebra_matches_float64(nx, nh, wants):
    """Right-looking Cholesky of P_b / P0_b with the fused forward solve, and h^T sum_Bhh h, against numpy / scipy
    (and mpmath at 40 digits for nx <= 24).  Each pass of a one-pass launch is bitwise the pass of the two-pass launch;
    the outputs of a pass not run are not touched."""
    inp, (ref, hbh), (out2, info2) = _alg_case(nx, nh)
    want_p, want_p0 = wants
    out, info = _alg_gpu(inp, want_p, want_p0) if wants != (1, 1) else (out2, info2)
    B = out.shape[0]
    assert np.all(info == 0)
    for b in range(B):
        for kind, want in ((0, want_p), (1, want_p0)):
            if not want:
                assert np.all(np.isnan(out[b, 2 * kind:2 * kind + 2]))
                continue
            got = out[b, 2 * kind:2 * kind + 2]
            assert np.array_equal(got, out2[b, 2 * kind:2 * kind + 2])
            assert _close_alg(got, ref[b, kind], nx), (b, kind, got, ref[b, kind])
            if nx <= 24 and b == 0:
                mp_ld, mp_q, mp_h = _mp_ref(inp, b, kind)
                assert _close_alg(got, (mp_ld, mp_q) + tuple(ref[b, kind, 2:]), nx), (b, kind, got, mp_ld, mp_q)
                if kind == 1:
                    assert abs(out[b, 4] - mp_h) <= 4 * nh * EPS * hbh[b, 1]
        if want_p0:
            assert abs(out[b, 4] - hbh[b, 0]) <= 4 * nh * EPS * hbh[b, 1], (b, out[b, 4], hbh[b, 0])
            assert out[b, 4] == out2[b, 4]
        else:
            assert np.isnan(out[b, 4])


@pytest.mark.parametrize('j', [0, 5, 200])
def test_algebra_reports_the_failed_pivot(j):
    """P0_1 = Lu D Lu^T (Lu unit lower triangular) with D[j] = -1: its leading j x j block is positive definite and the
    next Schur complement is -1, so the factorisation stops at pivot j: info[1][1] == j + 1.  reg lifts P_1 = P0_1 + reg I
    above 1, so info[1][0] == 0.  The other samples of the launch are bitwise those of a launch without sample 1."""
    nx, nh = 256, 33
    inp = _alg_inputs(nx, nh, 3, seed=j + 17)
    rng = np.random.default_rng(j)
    Lu = np.tril(.2 * rng.standard_normal((nx, nx)) / np.sqrt(nx), -1) + np.eye(nx)
    D = rng.uniform(.5, 1.5, nx)
    D[j] = -1.0
    T = (Lu * D) @ Lu.T
    T = (T + T.T) / 2
    assert np.all(np.linalg.eigvalsh(T[:j, :j]) > 0) if j else True
    c1 = inp['c1_m'].copy()
    c1[1] = (T - inp['kx_m']) / R - inp['sxx_m']
    inp['c1_m'] = c1
    inp['c1'] = _pad(c1, (3, inp['ld'], inp['ld']), True)
    inp['reg'] = 1.0 - np.linalg.eigvalsh(T)[0]
    assert np.linalg.eigvalsh(_p_matrix(inp, 1, 1))[0] < 0 < np.linalg.eigvalsh(_p_matrix(inp, 1, 0))[0]
    out, info = _alg_gpu(inp, 1, 1)
    assert info[1, 1] == j + 1 and info[1, 0] == 0
    assert np.all(info[[0, 2]] == 0)
    ref, _ = _alg_ref(dict(inp, c1_m=c1[[0, 2]], hs_m=inp['hs_m'][[0, 2]]))
    for k, b in enumerate((0, 2)):
        assert _close_alg(out[b, 0:2], ref[k, 0], nx) and _close_alg(out[b, 2:4], ref[k, 1], nx)
    # the same launch without the bad sample
    sub = dict(inp, c1=inp['c1'][[0, 2]], hs=inp['hs'][[0, 2]])
    out2, info2 = _alg_gpu(sub, 1, 1)
    assert np.all(info2 == 0)
    assert np.array_equal(out2, out[[0, 2]])

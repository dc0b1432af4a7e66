"""GPU building blocks through the C-ABI against numpy / the oracle: the stand-alone bvn_cdf op (the
reference's only native FFI, src/core/exponentiated_quadratic.py:552), the DMMA GEMM and the Cholesky /
inverse / log-det kernels."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
import cgpcm_b200
from cgpcm_b200 import _lib
from oracle import bvn as obvn

RHOS = [0.0, 0.032, 0.122, 0.29, 0.31, 0.422, 0.65, 0.74, 0.76, 0.86, 0.92, 0.93, 0.969, 0.999, -0.5, -0.95]


def test_bvn_cdf_matches_oracle_host_buffers():
    rng = np.random.default_rng(0)
    n = 4000
    x1, x2 = rng.uniform(-6, 6, n), rng.uniform(-6, 6, n)
    rho = rng.choice(RHOS, n)
    got = cgpcm_b200.bvn_cdf(x1, x2, rho)
    want = obvn.bvn_cdf(x1, x2, rho)
    np.testing.assert_allclose(got, want, atol=3e-16, rtol=2e-14)


def test_bvn_cdf_device_buffers_and_edge_cases():
    x1 = torch.tensor([0., 40., -40., 1e-300, 3., -3., 0.], dtype=torch.float64, device='cuda')
    x2 = torch.tensor([0., 40., 0., -1e-300, -3., 3., 0.], dtype=torch.float64, device='cuda')
    rho = torch.tensor([.5, .5, .5, .3, .97, -.97, 0.], dtype=torch.float64, device='cuda')
    got = cgpcm_b200.bvn_cdf(x1, x2, rho).cpu().numpy()
    want = obvn.bvn_cdf(x1.cpu().numpy(), x2.cpu().numpy(), rho.cpu().numpy())
    np.testing.assert_allclose(got, want, atol=3e-16, rtol=2e-14)
    assert got[1] == pytest.approx(1.0, abs=1e-15) and got[2] == 0.0 and got[6] == pytest.approx(.25, abs=1e-16)
    empty = cgpcm_b200.bvn_cdf(np.zeros(0), np.zeros(0), np.zeros(0))
    assert empty.shape == (0,)
    with pytest.raises(ValueError):
        cgpcm_b200.bvn_cdf(np.zeros(3), np.zeros(2), np.zeros(3))


def _dgemm(a_kc, b_kc, c_tr, A, B, C, alpha, beta, splits=1, lower=0):
    """A: logical M x K, B: logical K x N, C: logical M x N numpy; stored per the layout flags."""
    M, K = A.shape
    N = B.shape[1]
    dev = lambda x: torch.tensor(np.ascontiguousarray(x), dtype=torch.float64, device='cuda')
    As = dev(A if a_kc else A.T)
    Bs = dev(B.T if b_kc else B)
    if splits > 1:
        Cs = torch.zeros(splits, M, N, dtype=torch.float64, device='cuda')
        stride = M * N
    else:
        Cs = dev(C.T if c_tr else C)
        stride = 0
    rc = _lib.lib().cgpcm_dgemm(int(a_kc), int(b_kc), int(c_tr), M, N, K, alpha, As.data_ptr(), As.shape[1],
                                 Bs.data_ptr(), Bs.shape[1], beta, Cs.data_ptr(), Cs.shape[-1], splits, stride,
                                 lower, None)
    assert rc == 0
    out = Cs.cpu().numpy()
    if splits > 1:
        return out.sum(0)
    return out.T if c_tr else out


@pytest.mark.parametrize('a_kc', [0, 1])
@pytest.mark.parametrize('b_kc', [0, 1])
@pytest.mark.parametrize('c_tr', [0, 1])
@pytest.mark.parametrize('shape', [(8, 8, 2), (200, 200, 200), (104, 136, 50), (216, 8, 34), (40, 264, 1026)])
def test_dgemm_layouts(a_kc, b_kc, c_tr, shape):
    M, N, K = shape
    rng = np.random.default_rng(M + N + K)
    A, B, C = rng.standard_normal((M, K)), rng.standard_normal((K, N)), rng.standard_normal((M, N))
    got = _dgemm(a_kc, b_kc, c_tr, A, B, C, 1.25, -0.5)
    want = 1.25 * A @ B - 0.5 * C
    np.testing.assert_allclose(got, want, atol=1e-12 * np.sqrt(K) * 10)


def test_dgemm_split_k_and_lower_only():
    rng = np.random.default_rng(5)
    M, K = 200, 5000
    A = rng.standard_normal((M, K))
    got = _dgemm(1, 1, 0, A, A.T.copy(), np.zeros((M, M)), 1.0, 0.0, splits=7)
    np.testing.assert_allclose(got, A @ A.T, atol=1e-10)
    low = _dgemm(1, 1, 0, A, A.T.copy(), np.zeros((M, M)), 1.0, 0.0, splits=5, lower=1)
    np.testing.assert_allclose(np.tril(low), np.tril(A @ A.T), atol=1e-10)


@pytest.mark.parametrize('b_kc', [0, 1])
@pytest.mark.parametrize('M,K,N', [(200, 200, 64 * 148 + 64 * 37), (200, 184, 64 * 150 + 8), (168, 200, 64 * 148),
                                   (208, 24, 64 * 149 + 40),
                                   # windows of inducing inputs (one half, 5 / 9 / 12 / 13 row blocks) and 104 + a short half
                                   (96, 96, 64 * 148 + 64 * 5), (40, 40, 64 * 300 + 16), (16, 16, 64 * 148),
                                   (72, 56, 64 * 150 + 24), (104, 104, 64 * 148), (88, 200, 64 * 149),
                                   (112, 112, 64 * 148 + 8), (136, 136, 64 * 151)])
def test_dgemm_small_left(b_kc, M, K, N):
    """Persistent small-left-operand kernel (dgemm_sl.cuh: resident S, bulk-copy ring, mbarriers) against numpy,
    both layouts (left multiply / transposed right multiply), ragged N tiles, short last k-tile, M = 104 + 96,
    the zero-padded generic halves and the single-half windows (M <= 104)."""
    rng = np.random.default_rng(M + K + N + b_kc)
    S = rng.standard_normal((M, K))
    B = rng.standard_normal((K, N))
    want = 1.5 * (S @ B)
    dev = lambda x: torch.tensor(np.ascontiguousarray(x), dtype=torch.float64, device='cuda')
    Sd = dev(S)
    if b_kc:
        Bd = dev(B.T)                                   # B(k, n) at Bd[n * K + k]
        C = torch.full((N, M), np.nan, dtype=torch.float64, device='cuda')
        rc = _lib.lib().cgpcm_dgemm(1, 1, 1, M, N, K, 1.5, Sd.data_ptr(), K, Bd.data_ptr(), K, 0.0, C.data_ptr(), M,
                                    1, 0, 0, None)
        got = C.cpu().numpy().T
    else:
        Bd = dev(B)
        C = torch.full((M, N), np.nan, dtype=torch.float64, device='cuda')
        rc = _lib.lib().cgpcm_dgemm(1, 0, 0, M, N, K, 1.5, Sd.data_ptr(), K, Bd.data_ptr(), N, 0.0, C.data_ptr(), N,
                                    1, 0, 0, None)
        got = C.cpu().numpy()
    assert rc == 0
    scale = 1.5 * (np.abs(S) @ np.abs(B))
    assert np.all(np.abs(got - want) <= 4e-15 * scale)


@pytest.mark.parametrize('kc', [1, 0])
@pytest.mark.parametrize('M,K', [(200, 4096), (200, 50), (168, 1234), (184, 16 * 148 * 3 + 6),
                                 # windows: 4 / 3 / 2 / 1 warp-block rows, the last three with k-sub-sliced warps
                                 (160, 2000), (136, 778), (96, 16 * 148 * 2 + 10), (120, 64), (80, 5000), (48, 334),
                                 (40, 16 * 200), (8, 100), (64, 1000), (128, 1500), (32, 640), (104, 900), (152, 320)])
def test_dgemm_sym(kc, M, K):
    """Symmetric-output split-K DMMA kernel (dgemm_sym.cuh): C = X S X^T with S symmetric, computed as A B^T with
    A = X, B = X S, against numpy; ragged K, orders below the 200-row panel, both operand layouts."""
    rng = np.random.default_rng(M + K + kc)
    X = rng.standard_normal((M, K))
    d = rng.uniform(.5, 2., K)
    Bm = X * d                                   # (X D)  ->  X (X D)^T = X D X^T is symmetric
    want = X @ Bm.T
    dev = lambda x: torch.tensor(np.ascontiguousarray(x), dtype=torch.float64, device='cuda')
    if kc:
        As, Bs, lda = dev(X), dev(Bm), K
    else:
        As, Bs, lda = dev(X.T), dev(Bm.T), M
    C = torch.full((M, M), np.nan, dtype=torch.float64, device='cuda')
    rc = _lib.lib().cgpcm_dgemm_sym(kc, M, K, As.data_ptr(), lda, Bs.data_ptr(), lda, C.data_ptr(), M, None, None)
    assert rc == 0
    got = C.cpu().numpy()
    scale = np.abs(X) @ np.abs(Bm).T
    assert np.all(np.abs(got - want) <= 4e-15 * scale + 1e-300)
    assert np.array_equal(got, got.T)


@pytest.mark.parametrize('n,ld', [(1, 8), (1, 24), (5, 8), (32, 32), (33, 40), (41, 48), (41, 64), (150, 152),
                                  (200, 200), (301, 304), (301, 320)])
def test_cholinv(n, ld):
    """cgpcm_cholinv against float64 bars: the factor's backward error |L L^T - A| <= 4 (n + 1) eps |L| |L|^T, the
    residual and forward error of the inverse within 4 n eps cond(A), the padding rows / columns [n, np) of the inverse
    exactly 0, and logdet within n eps of 2 sum log L_ii of the GPU's own factor and within 1e-12 of slogdet.  Every
    element outside the logical n x n block starts as NaN: the identity padding must be put in by the call."""
    import math
    eps = np.finfo(np.float64).eps
    rng = np.random.default_rng(n)
    X = rng.standard_normal((n, n + 3))
    A = X @ X.T + 1e-3 * np.eye(n)
    np_ = (n + 7) // 8 * 8
    buf = np.full((ld, ld), np.nan)
    buf[:n, :n] = A
    dA = torch.tensor(buf, device='cuda')
    dI = torch.full_like(dA, np.nan)
    logdet = np.zeros(1)
    info = ctypes.c_int(0)
    rc = _lib.lib().cgpcm_cholinv(dA.data_ptr(), dI.data_ptr(), logdet.ctypes.data, n, ld, ctypes.byref(info))
    assert rc == 0 and info.value == 0
    L = dA.cpu().numpy()[:n, :n]
    assert np.all(np.triu(L, 1) == 0.0) and np.all(np.diag(L) > 0)
    assert np.all(np.abs(L @ L.T - A) <= 4 * (n + 1) * eps * (np.abs(L) @ np.abs(L).T))
    full = dI.cpu().numpy()
    inv = full[:n, :n]
    w = np.linalg.eigvalsh(A)
    cond = w[-1] / w[0]
    assert np.abs(A @ inv - np.eye(n)).max() <= 4 * n * eps * cond
    ref = np.linalg.inv(A)
    assert np.abs(inv - ref).max() <= 4 * n * eps * cond * np.abs(ref).max()
    assert np.all(full[:np_, n:np_] == 0.0) and np.all(full[n:np_, :np_] == 0.0)
    own = 2 * math.fsum(np.log(np.diag(L)))
    assert abs(logdet[0] - own) <= (n + 2) * eps * 2 * math.fsum(np.abs(np.log(np.diag(L)))) + 1e-300
    assert logdet[0] == pytest.approx(np.linalg.slogdet(A)[1], rel=1e-12, abs=1e-12)


def test_cholinv_reports_non_positive_definite():
    n, ld = 16, 16
    A = np.eye(n)
    A[7, 7] = -1.0
    dA = torch.tensor(A, device='cuda')
    info = ctypes.c_int(0)
    rc = _lib.lib().cgpcm_cholinv(dA.data_ptr(), None, None, n, ld, ctypes.byref(info))
    assert rc == -3 and info.value == 8


def test_in_register_exp_and_erfc_against_mpmath():
    """csrc/cgmath.cuh (the lock-step exp / erfc of the Ahx kernels) against mpmath: <= 2 ulp for exp on [-745, 0],
    <= 4 ulp for erfc on [-8, 27] (relative to the result, i.e. also where erfc is 1e-300), exact limits, and the
    four-at-a-time evaluation gives the same bits as one at a time."""
    import ctypes
    import mpmath as mp
    mp.mp.dps = 40
    rng = np.random.default_rng(11)
    x = np.concatenate([-rng.uniform(0, 745, 1500), -10.0 ** rng.uniform(-12, 0, 300), [0.0, -1e-300, -744.4, -708.4],
                        rng.uniform(-8, 27, 1500), rng.normal(0, 1.5, 700), [-6.5, -30.0, 26.5, 27.2, 0.5, 4.0]])
    x = np.ascontiguousarray(x)
    oe, oc = np.empty_like(x), np.empty_like(x)
    mism = ctypes.c_int(-1)
    rc = _lib.lib().cgpcm_math_test(_lib.ptr(x), x.shape[0], _lib.ptr(oe), _lib.ptr(oc), ctypes.byref(mism))
    assert rc == 0 and mism.value == 0

    def ulps(got, want):
        want_f = float(want)
        if want_f == 0.0 or abs(want_f) < 2.3e-308:          # subnormal results: absolute, in units of the least subnormal
            return abs(got - want_f) / 5e-324 / 2 ** 3
        return abs(mp.mpf(got) - want) / mp.mpf(np.spacing(abs(want_f)))

    worst_e = max(ulps(oe[i], mp.exp(mp.mpf(min(x[i], 0.0)))) for i in range(x.shape[0]))
    worst_c = max(ulps(oc[i], mp.erfc(mp.mpf(x[i]))) for i in range(x.shape[0]) if x[i] < 26.0)
    assert worst_e <= 2.0, worst_e
    assert worst_c <= 4.0, worst_c
    i0 = int(np.where(x == 0.0)[0][0])
    assert oe[i0] == 1.0 and oc[i0] == 1.0
    assert oc[np.where(x == -30.0)[0][0]] == 2.0 and oc[np.where(x == -6.5)[0][0]] == 2.0
    assert 0.0 <= oc[np.where(x == 27.2)[0][0]] <= 1e-320


def test_flushing_exp_and_erfcx_against_mpmath():
    """The variants the separable Psi kernels use (csrc/cgmath.cuh): exp with one integer scaling step -- bit-identical
    to the two-step version wherever the result is normal, exactly 0 below 2^-1021 -- and erfcx(|x|) = exp(x^2) erfc(|x|),
    the rational part of erfc, <= 5 ulp against mpmath on [0, 27] (measured: 4.5)."""
    import ctypes
    import mpmath as mp
    mp.mp.dps = 40
    rng = np.random.default_rng(12)
    x = np.concatenate([-rng.uniform(0, 745, 1500), -10.0 ** rng.uniform(-12, 0, 300), [0.0, -1e-300, -707.0, -708.0, -709.0, -744.4],
                        rng.uniform(-27, 27, 1500), rng.normal(0, 1.5, 700), [-6.5, 26.5, 27.2, 0.5, 4.0]])
    x = np.ascontiguousarray(x)
    oe, oc, oe2, oc2 = np.empty_like(x), np.empty_like(x), np.empty_like(x), np.empty_like(x)
    mism = ctypes.c_int(-1)
    assert _lib.lib().cgpcm_math_test_fast(_lib.ptr(x), x.shape[0], _lib.ptr(oe), _lib.ptr(oc)) == 0
    assert _lib.lib().cgpcm_math_test(_lib.ptr(x), x.shape[0], _lib.ptr(oe2), _lib.ptr(oc2), ctypes.byref(mism)) == 0
    xe = np.minimum(x, 0.0)
    normal = oe2 >= 2.0 ** -1021
    assert np.array_equal(oe[normal], oe2[normal])               # same bits as the exact-scaling version
    assert np.all(oe[xe < -708.1] == 0.0) and np.all(oe[~normal] <= 2.0 ** -1021)
    worst = 0.0
    for xi, got in zip(x, oc):
        a = abs(float(xi))
        if a > 27.3:                                             # the argument is clamped there (erfc underflows)
            continue
        want = mp.erfc(mp.mpf(a)) * mp.exp(mp.mpf(a) ** 2)
        worst = max(worst, float(abs(mp.mpf(float(got)) - want) / mp.mpf(float(np.spacing(float(want))))))
    assert worst <= 5.0, worst


@pytest.mark.parametrize('M', [40, 72, 88, 96, 104])
def test_triangular_right_multiply_against_torch(M):
    """dgemm_sl_tri (csrc/dgemm_sl.cuh): C[n][m] = sum_{k >= m} S[m][k] B[n][k] for an upper-triangular resident operand,
    with the DMMA blocks below the diagonal skipped -- the right-multiply by the transposed Cholesky factor of a window
    block (Q = sum A iKx A^T as V' V'^T).  Against torch on the full columns, ragged tail included."""
    import torch
    N = 64 * 148 + 8 * 37
    g = torch.Generator(device='cpu').manual_seed(M)
    S = torch.triu(torch.randn(M, M, dtype=torch.float64, generator=g)).cuda()
    B = torch.randn(N, M, dtype=torch.float64, generator=g).cuda()
    C = torch.full((N, M), float('nan'), dtype=torch.float64, device='cuda')
    rc = _lib.lib().cgpcm_dgemm_tri(M, N, S.data_ptr(), M, B.data_ptr(), M, C.data_ptr(), M, None)
    assert rc == 0
    ref = B @ S.t()
    err = float((C - ref).abs().max() / ref.abs().max())
    assert err < 1e-14, err

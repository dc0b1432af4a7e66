"""The dense factorisation of csrc/linalg.cuh against float64 references: potrf_lower and trtri_lower through their
C-ABI hooks (cgpcm_potrf_test, cgpcm_trtri_test), cholinv through cgpcm_cholinv (tests/test_gpu_kernels.py), and the
callers that factorise the largest matrices -- filter draws (order <= 8192), AKM draws (<= 4096), predictive draws
(<= 4096) and held-out scoring (the bordered matrix, order 4097 padded to 4104) -- once each at their documented limits.

The factor is held to the componentwise backward-error bar |L L^T - A| <= 4 (n + 1) eps |L| |L|^T, which does not depend
on the conditioning, on random and squared-exponential Gram matrices (cond ~ 1e3 .. 1e10) at every order 8 .. 296 and at
1000 .. 8192 (a row sample from 2048 on).  Every buffer carries a guard: the ld padding beyond np and 32 rows past the
matrix hold a sentinel that must keep its bits.  A factor of D A D with D = diag(2^k) must be D L bitwise: every step is
a correctly rounded product, quotient, square root or FMA of terms that all scale alike, so an element read from the
wrong row or column shows as a changed bit.  The info word must name the FIRST non-positive pivot."""
import ctypes

import numpy as np
import pytest
from scipy.linalg import cho_solve, solve_triangular

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
import cgpcm_b200
from cgpcm_b200 import _lib
from oracle import model as om
from tests.cases import make_case
from tests.test_gpu_predict_cov import _draws, _engine, _trained
from tests.test_gpu_predict_logpdf import _check_scoring, _y_star

EPS = np.finfo(np.float64).eps
NB, ROWS = 32, 128                     # LA_NB (panel width) and LA_ROWS (panel rows per CTA) of linalg.cuh
GUARD = 32                             # sentinel rows past the matrix
SENT = -3.0e301                        # the sentinel: finite, and fails any pivot it reaches
SMALL = list(range(8, 297, 8))         # np % 32 in {0, 8, 16, 24}; rows below a panel at 1, 2 and 3 CTAs of 128 rows
LARGE = [1000, 2048, 4096, 4104, 8192]
WORST = {}                             # largest error / bar per check (printed with -s)


def _note(key, v):
    WORST[key] = max(WORST.get(key, 0.0), float(v))
    print('%s: %.3g of the bar' % (key, WORST[key]))


# ------------------------------------------------------------------------------------------------------ matrices
def _dd(n, seed):
    """Random symmetric, diagonally dominant (cond ~ 10): O(n^2)."""
    rng = np.random.default_rng(seed)
    A = rng.uniform(-1, 1, (n, n))
    A += A.T
    A *= .5
    A[np.diag_indices(n)] = np.abs(A).sum(1) + 1.0
    return A


def _xxt(n, seed):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, n + 3))
    return X @ X.T + 1e-3 * np.eye(n)


def _se(n, cond, seed):
    """Squared-exponential Gram matrix at sorted inputs on [0, 1] (length scale .05: numerically rank ~100) plus
    lambda_max / cond on the diagonal, the kind of matrix the sampling and scoring paths factorise: O(n^2)."""
    t = np.sort(np.random.default_rng(seed).uniform(0, 1, n))
    A = np.subtract.outer(t, t)
    A *= A
    A *= -1.0 / (2 * .05 ** 2)
    np.exp(A, out=A)
    lam = A.sum() / n                  # 1^T A 1 / n: within a small factor of lambda_max for these inputs
    A[np.diag_indices(n)] += lam / cond
    return A


def _matrix(kind, n, seed=0):
    if kind == 'dd':
        return _dd(n, seed)
    if kind == 'xxt':
        return _xxt(n, seed)
    return _se(n, {'se3': 1e3, 'se6': 1e6, 'se10': 1e10}[kind], seed)


# -------------------------------------------------------------------------------------------------------- hooks
def _guarded(A, ld, fill=SENT):
    """A (n x n) in the top-left of a (n + GUARD) x ld buffer of sentinels."""
    n = A.shape[0]
    buf = np.full((n + GUARD, ld), fill)
    buf[:n, :n] = A
    return buf


def _sentinel_kept(buf, n):
    s = np.float64(SENT).view(np.int64)
    return bool(np.all(buf[:n, n:].view(np.int64) == s) and np.all(buf[n:].view(np.int64) == s))


def potrf_gpu(A, ld=None, tag=5):
    """L of A through cgpcm_potrf_test (lower triangle read), the raw info word; the guard is checked here."""
    n = A.shape[0]
    ld = ld or n
    d = torch.from_numpy(_guarded(A, ld)).cuda()
    info = ctypes.c_int(-7)
    assert _lib.lib().cgpcm_potrf_test(d.data_ptr(), n, ld, tag, ctypes.byref(info), None) == 0
    out = d.cpu().numpy()
    del d
    assert _sentinel_kept(out, n), 'potrf wrote outside the np x np block'
    return np.ascontiguousarray(out[:n, :n]), info.value


def trtri_gpu(L, ld=None):
    n = L.shape[0]
    ld = ld or n
    dL = torch.from_numpy(_guarded(L, ld)).cuda()
    dX = torch.from_numpy(_guarded(np.full((n, n), np.nan), ld)).cuda()
    assert _lib.lib().cgpcm_trtri_test(dL.data_ptr(), dX.data_ptr(), n, ld, None) == 0
    Lb, X = dL.cpu().numpy(), dX.cpu().numpy()
    assert np.array_equal(Lb[:n, :n], L) and _sentinel_kept(Lb, n), 'trtri changed its input'
    assert _sentinel_kept(X, n), 'trtri wrote outside the np x np block'
    return np.ascontiguousarray(X[:n, :n])


def _sample_rows(n, seed=1):
    """Every row at a panel edge (j0 - 1, j0, j0 + 31; the CTA edges j0 + 32 + 128 b are panel edges too) and ~200
    random rows."""
    r = set()
    for j0 in range(0, n, NB):
        r.update((j0 - 1, j0, j0 + NB - 1))
    r.update(np.random.default_rng(seed).integers(0, n, 200).tolist())
    r.add(n - 1)
    return np.array(sorted(i for i in r if 0 <= i < n))


def _rows_product(R, M, absolute=False):
    """R @ M.T, in column blocks of M (bounded memory at n = 8192)."""
    out = np.empty((R.shape[0], M.shape[0]))
    Ra = np.abs(R) if absolute else R
    for c0 in range(0, M.shape[0], 1024):
        blk = M[c0:c0 + 1024]
        out[:, c0:c0 + 1024] = Ra @ (np.abs(blk) if absolute else blk).T
    return out


def check_factor(L, A, key, rows=None):
    """The upper triangle exactly 0, a positive diagonal, and |L L^T - A| <= 4 (n + 1) eps |L| |L|^T element-wise
    (rows: a row sample; None: every row).  The host's own product adds at most n eps |L| |L|^T of the bar."""
    n = A.shape[0]
    assert not np.isnan(L).any()
    assert np.all(np.triu(L, 1) == 0.0)
    assert np.all(np.diag(L) > 0.0)
    rows = np.arange(n) if rows is None else rows
    R = L[rows]
    err = np.abs(_rows_product(R, L) - A[rows])
    bar = 4 * (n + 1) * EPS * _rows_product(R, L, absolute=True)
    ratio = (err / np.maximum(bar, 1e-300)).max()
    _note(key, ratio)
    assert ratio <= 1.0, (n, ratio)


# ------------------------------------------------------------------------------------------------ potrf: accuracy
@pytest.mark.parametrize('kind', ['dd', 'xxt', 'se3', 'se6', 'se10'])
def test_potrf_backward_error_every_small_order(kind):
    for n in SMALL:
        A = _matrix(kind, n, seed=n)
        for ld in (n, n + 8) if n % 16 else (n,):
            L, info = potrf_gpu(A, ld)
            assert info == 0, (n, ld, info)
            check_factor(L, A, 'potrf backward error, n <= 296')


@pytest.mark.parametrize('n,ld', [(200, 208), (200, 4096), (1000, 1000), (1000, 1016)])
def test_potrf_leading_dimension(n, ld):
    for kind in ('dd', 'se6'):
        A = _matrix(kind, n, seed=3)
        L, info = potrf_gpu(A, ld)
        assert info == 0
        check_factor(L, A, 'potrf backward error, ld > np')
        if n == 1000 and ld == 1000:
            continue
        assert np.array_equal(L, potrf_gpu(A)[0]), 'the factor depends on ld'


@pytest.mark.parametrize('n', LARGE)
def test_potrf_backward_error_large_orders(n):
    kinds = ('dd', 'se3', 'se6', 'se10') if n < 8192 else ('dd', 'se6', 'se10')
    rows = None if n < 2048 else _sample_rows(n)
    for kind in kinds:
        A = _matrix(kind, n, seed=n)
        L, info = potrf_gpu(A)
        assert info == 0, (kind, info)
        check_factor(L, A, 'potrf backward error, n >= 1000', rows)
        del L, A


def test_potrf_upper_triangle_is_not_read():
    """NaN in the strict upper triangle changes no bit of the factor and is not reported."""
    for n in (40, 168, 296, 1000):
        A = _matrix('dd', n, seed=n + 1)
        L, info = potrf_gpu(A)
        B = A.copy()
        B[np.triu_indices(n, 1)] = np.nan
        L2, info2 = potrf_gpu(B)
        assert info == 0 and info2 == 0 and np.array_equal(L.view(np.int64), L2.view(np.int64)), n


def _pow2(n, seed):
    return np.random.default_rng(seed).integers(-60, 61, n)


@pytest.mark.parametrize('n', [8, 24, 40, 128, 160, 200, 264, 296, 1000, 4104])
def test_potrf_power_of_two_scaling_is_exact(n):
    """L(D A D) = D L(A) bitwise for D = diag(2^k), k in [-60, 60]; at 4104 also two calls give the same bits."""
    A = _matrix('dd' if n % 16 else 'xxt', n, seed=n + 2)
    k = _pow2(n, n)
    L, info = potrf_gpu(A)
    S = np.ldexp(np.ldexp(A, k[:, None]), k[None, :])
    LS, info2 = potrf_gpu(S)
    assert info == 0 and info2 == 0
    want = np.ldexp(L, k[:, None])
    bad = LS.view(np.int64) != want.view(np.int64)
    assert not bad.any(), (n, np.argwhere(bad)[:5])
    if n == 4104:
        assert np.array_equal(potrf_gpu(A)[0].view(np.int64), L.view(np.int64)), 'two calls differ'


# ------------------------------------------------------------------------------------------------ potrf: info word
def _banded(n, bad, seed=0, w=3):
    """A = L0 diag(s) L0^T with a unit lower L0 of bandwidth w, entries in {-1/4, .., 1/4}, s_j in {1, 4} and s_j = -1
    at the pivots `bad`: every step is exact, so the pivots of those rows are exactly -1 (and those after them stay
    positive after a failed one is replaced by 1)."""
    rng = np.random.default_rng(seed)
    s = rng.choice([1.0, 4.0], n)
    s[list(bad)] = -1.0
    L0 = np.eye(n)
    for d in range(1, w + 1):
        idx = np.arange(d, n)
        L0[idx, idx - d] = rng.integers(-2, 3, n - d) / 8.0
    A = (L0 * s) @ L0.T
    return A


@pytest.mark.parametrize('n', [8, 40, 168, 4104])
def test_potrf_reports_the_failed_pivot(n):
    for j in (0, 1, 30, 31, 32, 33, 127, 128, 159, 160, n - 1):
        if j >= n:
            continue
        L, info = potrf_gpu(_banded(n, [j], seed=j), tag=6)
        assert info == 6 * 100000 + j + 1, (n, j, info)


@pytest.mark.parametrize('j1,j2', [(33, 40), (32, 63), (0, 1), (5, 70), (31, 32)],
                         ids=['one-panel', 'panel-ends', 'first-two', 'two-panels', 'panel-boundary'])
def test_potrf_reports_the_first_of_two_failed_pivots(j1, j2):
    L, info = potrf_gpu(_banded(168, [j1, j2], seed=j1 + j2), tag=7)
    assert info == 7 * 100000 + j1 + 1, (j1, j2, info)


@pytest.mark.parametrize('i,j', [(5, 5), (40, 40), (200, 200), (20, 10), (40, 3), (200, 150), (295, 0)])
def test_potrf_reports_nan_at_its_row(i, j):
    """NaN at A[i][j] (j <= i): the first pivot that cannot be formed is i's."""
    A = _banded(296, [], seed=3)
    A[i, j] = np.nan
    L, info = potrf_gpu(A, tag=8)
    assert info == 8 * 100000 + i + 1, (i, j, info)


def test_potrf_hook_rejects_bad_shapes():
    d = torch.zeros(64 * 64, dtype=torch.float64, device='cuda')
    info = ctypes.c_int(0)
    f = _lib.lib().cgpcm_potrf_test
    assert f(d.data_ptr(), 60, 64, 5, ctypes.byref(info), None) == -1          # np % 8 != 0
    assert f(d.data_ptr(), 64, 56, 5, ctypes.byref(info), None) == -1          # np > ld
    assert f(d.data_ptr(), 56, 63, 5, ctypes.byref(info), None) == -1          # odd ld
    assert _lib.lib().cgpcm_trtri_test(d.data_ptr(), d.data_ptr(), 64, 56, None) == -1


# ------------------------------------------------------------------------------------------------------- trtri
def check_inverse(X, L, key, cols=None):
    """X exactly lower triangular and |L X - I| <= 4 n eps |L| |X| element-wise (cols: a column sample).  The left
    residual is the one the algorithm bounds: each diagonal block comes from column solves L_ii x = e_c, and a float64
    emulation of the blocking exceeds a bar on the right residual X L - I already at n = 32 on a cond-1e3 Gram factor
    (and ~100-fold at cond 1e6), so the factors here have cond(A) <= 1e5."""
    n = L.shape[0]
    assert not np.isnan(X).any()
    assert np.all(np.triu(X, 1) == 0.0)
    cols = np.arange(n) if cols is None else cols
    C = X[:, cols]
    E = L @ C
    E[cols, np.arange(cols.size)] -= 1.0
    bar = 4 * n * EPS * (np.abs(L) @ np.abs(C))
    ratio = (np.abs(E) / np.maximum(bar, 1e-300)).max()
    _note(key, ratio)
    assert ratio <= 1.0, (n, ratio)


@pytest.mark.parametrize('kind', ['dd', 'xxt', 'se3'])
def test_trtri_every_small_order(kind):
    for n in SMALL:
        L = np.linalg.cholesky(_matrix(kind, n, seed=n))
        for ld in (n, n + 8) if n % 16 else (n,):
            check_inverse(trtri_gpu(L, ld), L, 'trtri residual, n <= 296')


@pytest.mark.parametrize('n,ld', [(1000, 1000), (1000, 1032), (4104, 4104)])
def test_trtri_large_orders(n, ld):
    L = np.linalg.cholesky(_matrix('se3', n, seed=n))
    cols = None if n < 2048 else np.union1d(_sample_rows(n), np.arange(n - n % NB, n))   # the last partial block
    check_inverse(trtri_gpu(L, ld), L, 'trtri residual, n >= 1000', cols)


# -------------------------------------------------------------------------------- the callers at their limits
@pytest.fixture(scope='module')
def toy():
    c = make_case('toy_small')
    eng = cgpcm_b200.Engine(c['nh'], c['nx'], causal=c['causal'])
    eng.set_data(c['t'], c['y'], c['th'], c['tx'])
    return c, eng


def _cond(S):
    w = np.linalg.eigvalsh(S)
    assert w[0] > 0
    return w[-1] / w[0]


def _check_whitened(S, d, e, key, cond=None, Lh=None):
    """d = L e for the GPU's factor L of S: |L_host^-1 d - e| <= 4 n eps cond(S) |e| (both factors are backward
    stable, so they differ by about L^-1 dL with |dS| <= n eps |S|)."""
    n = S.shape[0]
    Lh = np.linalg.cholesky(S) if Lh is None else Lh
    cond = _cond(S) if cond is None else cond
    for b in range(d.shape[1]):
        z = solve_triangular(Lh, d[:, b], lower=True)
        bar = 4 * n * EPS * cond * np.linalg.norm(e[:, b])
        ratio = np.abs(z - e[:, b]).max() / bar
        _note(key, ratio)
        assert ratio <= 1.0, (b, ratio)


def test_filter_samples_at_8192(toy):
    """The conditional mean against the oracle at a subset of the inputs (row p only depends on t_p), the noise part
    L e against the host's factor of S = reg(k_h(t, t) - A^T A); 8193 inputs are refused."""
    c, eng = toy
    n, B, nh = 8192, 2, c['nh']
    rng = np.random.default_rng(3)
    samples = c['params'][5:5 + nh] + .3 * rng.standard_normal((B, nh))
    lo, hi = c['th'].min(), c['th'].max()
    t = np.linspace(lo - .3 * (hi - lo), hi + .3 * (hi - lo), n)
    noise = rng.standard_normal((n, B))
    got0 = eng.filter_samples(c['params'], t, samples, np.zeros_like(noise), reg=c['reg'])
    got = eng.filter_samples(c['params'], t, samples, noise, reg=c['reg'])
    sub = np.union1d(np.arange(0, n, 37), [n - 1])
    om.PW_DISTS_EXACT = True
    try:
        mean_only = om.filter_samples(c['params'], c['th'], c['reg'], t[sub], samples, np.zeros((sub.size, B)))
        with torch.no_grad():                   # S as oracle.model.filter_samples forms it, at all 8192 inputs
            s2, s2_f, alpha, gamma, omega, _, _ = om.unpack(om.T(c['params']), nh)
            thT, tt = om.T(c['th']), om.T(t)
            Lh = torch.linalg.cholesky(om.reg(om.deq(1., alpha, gamma, thT), c['reg']))
            A = om.trisolve(Lh, om.deq(1., alpha, gamma, thT, tt))
            S = om.reg(om.deq(1., alpha, gamma, tt) - A.T @ A, c['reg']).numpy()
    finally:
        om.PW_DISTS_EXACT = False
    assert np.abs(got0[sub] - mean_only).max() <= 1e-12 * np.abs(mean_only).max()
    # cond(S) without an eigen-decomposition at n = 8192: lambda_max <= |S|_1, lambda_min by inverse iteration
    Lh = np.linalg.cholesky(S)
    v = rng.standard_normal(n)
    for _ in range(30):
        v = cho_solve((Lh, True), v)
        v /= np.linalg.norm(v)
    cond = np.abs(S).sum(1).max() / (v @ S @ v)
    _check_whitened(S, got - got0, noise, 'filter_samples whitened noise', cond=cond, Lh=Lh)
    del S
    L = _lib.lib()
    t1 = np.linspace(0, 1, n + 1)
    nz = np.zeros((n + 1) * B)
    out = np.empty((n + 1) * B)
    assert L.cgpcm_filter_samples(eng._h, c['params'][:5].copy().ctypes.data, c['reg'], t1.ctypes.data, n + 1,
                                  samples.ctypes.data, B, nz.ctypes.data, out.ctypes.data) == -1
    assert '8192' in L.cgpcm_last_error(eng._h).decode()


def test_akm_sample_at_4096(toy):
    """K symmetric to the accuracy of its entries (K[p][q] and K[q][p] are evaluated at the lags +-(t_p - t_q); the
    factorisation reads the lower triangle only), 196 entries against the oracle's pair statistics (entry (p, q) only
    depends on t_p, t_q), f against the host's factor of K; 4097 inputs are refused."""
    c, eng = toy
    n, nh = 4096, c['nh']
    rng = np.random.default_rng(4)
    t = np.sort(rng.uniform(0., 1., n))
    h = c['params'][5:5 + nh] + .3 * rng.standard_normal(nh)
    e = rng.standard_normal(n)
    f, K = eng.akm_sample(c['params'], t, h, e, reg=c['reg'], want_cov=True)
    assert np.abs(K - K.T).max() <= 1e-6 * np.abs(K).max()                     # as tests/test_gpu_akm.py
    K = np.tril(K) + np.tril(K, -1).T                                           # the matrix potrf factorises
    idx = np.sort(rng.choice(n, 14, replace=False))
    om.PW_DISTS_EXACT = True
    try:
        _, K0 = om.akm_f(c['params'], c['th'], c['reg'], t[idx], h, e[idx], causal=c['causal'])
    finally:
        om.PW_DISTS_EXACT = False
    assert np.abs(K[np.ix_(idx, idx)] - K0).max() <= 1e-6 * np.abs(K0).max()    # as tests/test_gpu_akm.py
    _check_whitened(K, f[:, None] / np.sqrt(np.exp(c['params'][1])), e[:, None], 'akm_sample whitened draw')
    L = _lib.lib()
    t1 = np.linspace(0, 1, n + 1)
    out = np.empty(n + 1)
    assert L.cgpcm_akm_sample(eng._h, c['params'][:5].copy().ctypes.data, c['reg'], t1.ctypes.data, n + 1,
                              h.ctypes.data, t1.ctypes.data, out.ctypes.data, None) == -1
    assert '4096' in L.cgpcm_last_error(eng._h).decode()


def test_predict_draws_and_scoring_at_4096():
    """Draws at 4096 test inputs against the host's factor of the GPU's own C_b + reg I, and held-out scoring (the
    bordered matrix of order 4097, padded to 4104) through tests/test_gpu_predict_logpdf._check_scoring; 4097 test
    inputs are refused by predict_f_cov."""
    c = make_case('toy_small')
    p = _trained(c)
    S = _draws(p, c['nh'], c['reg'], 2, seed=5)
    n = 4096
    t_star = np.linspace(c['t'].min() - .05, c['t'].max() + .05, n)
    y = _y_star(c, t_star, seed=2)
    eng = _engine(c)
    eng.precompute(*c['hyp'], reg=c['reg'])
    noise = np.random.default_rng(6).standard_normal((n, 2))
    _, _, ms, cs, draws = eng.predict_f_cov(p, t_star, S, smf=True, reg=c['reg'], per_sample=True, noise=noise)
    for b in range(2):
        Sb = cs[b] + c['reg'] * np.eye(n)
        _check_whitened(Sb, (draws[:, b] - ms[:, b])[:, None], noise[:, b:b + 1], 'predict_f_cov whitened draw')
    lp, lp_s, white = eng.predict_logpdf(p, t_star, y, S, smf=True, reg=c['reg'], noise=True, white=True)
    _check_scoring(lp_s, white, y, ms, cs, np.exp(p[0]))
    big = np.linspace(0, 1, n + 1)
    L = _lib.lib()
    assert L.cgpcm_predict_f_cov(eng._h, p.ctypes.data, c['reg'], big.ctypes.data, n + 1, S.ctypes.data, 2, 1, None,
                                 None, None, None, None) == -1
    assert '4096' in L.cgpcm_last_error(eng._h).decode()

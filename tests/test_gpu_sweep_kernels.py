"""The kernels of the ELBO sweeps against float64 references, one kernel at a time, through the C-ABI hooks that run the
sweeps' own launch code (cgpcm_ahx_gen_test, cgpcm_ahx_dot_test, cgpcm_axx_sum_test, cgpcm_window_chol_test,
cgpcm_sym_accum_test), and the windowed products through cgpcm_dgemm / cgpcm_dgemm_tri as the sweeps call them; then
every contraction route of the sweeps against the CPU oracle at M = 200 and against the default route at N = 1e5.

Shapes are the bench's (N = 1e5 observations on [0, 100], nh = nx = 200, rho = gamma / (alpha + gamma + omega) = 0.968)
plus the edges where the kernels branch: window widths past one 256-thread pass (two k per thread), windows against the
end of the inducing grid with nx % 8 != 0, short last 16-observation slices, n_valid < nc, nh < nhp, fully culled CTAs
and elements within a hair of the cull threshold."""
import ctypes
import functools
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')
from scipy.special import erfcx

import cgpcm_b200
from cgpcm_b200 import _lib
from tests.workload import named_workload, sweep_workload

EPS = np.finfo(np.float64).eps
TINY = 2.0 ** -1021          # the separable kernels flush exp() results below this to 0 (cgmath.cuh)

# Distinct (kwp, nc, nv) of the chunks the planner makes at the bench shape (N = 1e5, M = 200, option chunk = 0), from
# CGPCM_DEBUG_PLAN=1 on one B200: 23 chunks at cull 746, 47 at cull 80, 49 dense.  The Ahx cases below take these window
# widths (and the first / last chunks' window positions) with up to 2048 observations, so that the float64 reference
# stays in memory; nc only sets the number of 16-observation slices.
BENCH_CHUNKS = {
    746.0: [(56, 5984, 5984), (56, 6112, 6112), (64, 4032, 4032), (72, 4000, 4000), (72, 5664, 5664), (80, 4032, 4032),
            (80, 5120, 5120), (88, 4032, 4032), (88, 4640, 4640), (96, 3936, 3936), (96, 4256, 4256)],
    80.0: [(24, 2336, 2336), (24, 3200, 3200), (32, 1984, 1984), (32, 2016, 2016), (32, 2464, 2464), (32, 3200, 3200)],
    0.0: [(200, 1696, 1696), (200, 2048, 2048)],
}


@functools.lru_cache(None)
def bench():
    return sweep_workload(100000, 200, seed=0)


@functools.lru_cache(None)
def toy():
    return named_workload('toy')


def _dev(a):
    return torch.tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _hyp(src):
    return np.array((bench() if src == 'bench' else toy())['hyp'], dtype=np.float64)


# ---------------------------------------------------------------------------------------------------------- Ahx gen
def _chunk(src, nh, nx, n0, nv):
    """(t of the chunk, y, th, tx) from the bench (nh / nx inducing points on its grid) or the toy workload."""
    w = bench() if src == 'bench' else toy()
    t, y = w['t'][n0:n0 + nv], w['y'][n0:n0 + nv]
    th = np.linspace(w['th'][0], w['th'][-1], nh)
    tx = np.linspace(w['tx'][0], w['tx'][-1], nx)
    return np.ascontiguousarray(t), np.ascontiguousarray(y), th, tx


def _ahx_terms(t, th, tx, k_lo, kwp, nhp, nc, hyp, causal_id):
    """E, z, the exponent of the separable factorisation c = -(alpha + gamma) th^2 - omega d^2, and the sum of the
    magnitudes of the exponent's terms, on the padded [nhp][nc][kwp] block (padding: NaN)."""
    a, g, o = hyp
    A = a + g + o
    nv, nh, nx = len(t), len(th), len(tx)
    kk = k_lo + np.arange(kwp)
    d = np.full((1, nc, kwp), np.nan)
    ok = kk < nx
    d[0, :nv, ok] = (t[:, None] - tx[kk[ok]][None, :]).T
    thi = np.full((nhp, 1, 1), np.nan)
    thi[:nh, 0, 0] = th
    e_hh, e_dd, e_hd = ((a + g) * A - g * g) / A, o * (a + g) / A, 2 * g * o / A
    E = -e_hh * thi ** 2 - e_dd * d ** 2 + e_hd * thi * d
    z = -(g * thi + o * d) / math.sqrt(A)
    if causal_id:
        z = z + np.maximum(d, 0.0) * math.sqrt(A)
    c = -(a + g) * thi ** 2 - o * d ** 2
    S = e_hh * thi ** 2 + e_dd * d ** 2 + np.abs(e_hd * thi * d) + np.abs(c)
    return E, z, c, S


def ahx_ref(t, th, tx, k_lo, kwp, nhp, nc, hyp, causal, causal_id):
    """float64 Ahx = pref exp(E) erfc(z) (oracle/model.py::psi_Ahx) on the padded block, written in the separable form
    that stays accurate where exp(E) or erfc(z) alone would under- / overflow; also E and the term magnitudes."""
    a, g, o = hyp
    A = a + g + o
    E, z, c, S = _ahx_terms(t, th, tx, k_lo, kwp, nhp, nc, hyp, causal_id)
    pref = (0.5 if causal else 1.0) * math.sqrt(math.pi / A)
    with np.errstate(over='ignore', under='ignore', invalid='ignore'):
        if not causal:
            v = pref * np.exp(E)
        elif causal_id:
            # exp(E) erfc(z) = exp(E - z^2) erfcx(z) for z >= 0
            v = np.where(z >= 0, pref * np.exp(E - z * z) * erfcx(np.abs(z)),
                         pref * (2 * np.exp(E) - np.exp(E - z * z) * erfcx(np.abs(z))))
        else:
            v = np.where(z >= 0, pref * np.exp(c) * erfcx(np.abs(z)),
                         pref * (2 * np.exp(E) - np.exp(c) * erfcx(np.abs(z))))
    return v, E, S, pref


def ahx_mp(th, d, hyp, causal, causal_id):
    """Ahx of one element in 40-digit arithmetic."""
    import mpmath
    mpmath.mp.dps = 40
    a, g, o = (mpmath.mpf(float(x)) for x in hyp)
    th, d = mpmath.mpf(float(th)), mpmath.mpf(float(d))
    A = a + g + o
    b = -2 * g * th - 2 * o * d
    E = -(a + g) * th ** 2 - o * d ** 2 + b ** 2 / (4 * A)
    v = mpmath.sqrt(mpmath.pi / A) * mpmath.exp(E)
    if causal:
        z = b / (2 * mpmath.sqrt(A))
        if causal_id and d > 0:
            z += d * mpmath.sqrt(A)
        v = v * mpmath.erfc(z) / 2
    return float(v)


def ahx_gen_gpu(t, y, th, tx, nhp, nc, k_lo, kwp, hyp, causal, causal_id, cull, sep, ld):
    nv, nh, nx = len(t), len(th), len(tx)
    slices = (nc + 15) // 16
    A = torch.full((nhp, nc, kwp), float('nan'), dtype=torch.float64, device='cuda')
    yp = torch.full((slices, nhp, ld), float('nan'), dtype=torch.float64, device='cuda')
    tp = np.zeros(nc)
    tp[:nv] = t
    yy = np.zeros(nc)
    yy[:nv] = y
    dt, dy, dth, dtx = _dev(tp), _dev(yy), _dev(th), _dev(tx)
    hp = np.ascontiguousarray(hyp, dtype=np.float64)
    rc = _lib.lib().cgpcm_ahx_gen_test(dt.data_ptr(), dy.data_ptr(), nv, nc, dth.data_ptr(), nh, nhp, dtx.data_ptr(), nx,
                                       k_lo, kwp, hp.ctypes.data, int(causal), int(causal_id), cull, int(sep), ld,
                                       A.data_ptr(), yp.data_ptr(), None)
    assert rc == 0
    return A.cpu().numpy(), yp.cpu().numpy()


def _centred(src, nx, nc, n0):
    """k_lo of a window of the grid centred on the chunk's observations (even, inside the padded grid)."""
    w = bench() if src == 'bench' else toy()
    tx = np.linspace(w['tx'][0], w['tx'][-1], nx)
    return int(np.clip(np.searchsorted(tx, w['t'][n0 + nc // 2]), 0, nx)) // 2 * 2


# name: (hyper-parameter source, nh, nhp, nx, ld, n0, nv, nc, k_lo ('mid' = centred on the chunk, 'end' = nxp - kwp), kwp,
#        causal, causal_id, cull)
AHX_CASES = {
    # the bench's own chunks (BENCH_CHUNKS), windows centred on the observations (z changes sign inside)
    'bench_746': ('bench', 200, 200, 200, 208, 49500, 1024, 1024, 'mid', 96, 1, 0, 746.0),
    'bench_746_last': ('bench', 200, 200, 200, 208, 98000, 1000, 1000, 144, 56, 1, 0, 746.0),
    'bench_80': ('bench', 200, 200, 200, 208, 49500, 2016, 2016, 'mid', 32, 1, 0, 80.0),
    'bench_80_first': ('bench', 200, 200, 200, 208, 0, 2048, 2048, 0, 24, 1, 0, 80.0),
    'bench_dense': ('bench', 200, 200, 200, 208, 49800, 512, 512, 0, 200, 1, 0, 0.0),
    # window edges: narrowest window; window at the end of a grid with nx % 8 != 0; two k per thread (kwp > 256)
    'kwp8_short_slice': ('bench', 41, 48, 203, 208, 50000, 37, 40, 'mid', 8, 1, 0, 80.0),
    'end_of_grid_nx203': ('bench', 203, 208, 203, 208, 99000, 1000, 1000, 'end', 48, 1, 0, 80.0),
    'kwp304_two_k_per_thread': ('bench', 203, 208, 299, 304, 49000, 200, 200, 0, 304, 1, 0, 0.0),
    # observations far outside the window: every CTA takes the culled branch
    'fully_culled': ('bench', 200, 200, 200, 208, 0, 512, 512, 96, 104, 1, 0, 80.0),
    # the toy's hyper-parameters (rho well below the bench's), acausal and causal_id (generic kernel only)
    'toy_causal': ('toy', 41, 48, 150, 152, 100, 250, 256, 'mid', 40, 1, 0, 80.0),
    'toy_acausal': ('toy', 41, 48, 150, 152, 100, 247, 256, 'mid', 40, 0, 0, 80.0),
    'toy_causal_id': ('toy', 41, 48, 150, 152, 100, 247, 256, 'mid', 40, 1, 1, 746.0),
    # cull set to -E of one element: that element sits on the threshold
    'on_the_threshold': ('bench', 200, 200, 200, 208, 49500, 512, 512, 'mid', 40, 1, 0, 'edge'),
}


def _ahx_case(name):
    src, nh, nhp, nx, ld, n0, nv, nc, k_lo, kwp, causal, causal_id, cull = AHX_CASES[name]
    t, y, th, tx = _chunk(src, nh, nx, n0, nv)
    nxp = -(-nx // 8) * 8
    if k_lo == 'mid':
        k_lo = min(max(0, _centred(src, nx, nv, n0) - kwp // 2 // 2 * 2), nxp - kwp)
    elif k_lo == 'end':
        k_lo = nxp - kwp
    hyp = _hyp(src)
    if cull == 'edge':
        E = _ahx_terms(t, th, tx, k_lo, kwp, nhp, nc, hyp, causal_id)[0]
        e = E[:nh, :nv, :][np.isfinite(E[:nh, :nv, :])]
        cull = float(-np.sort(e)[len(e) // 3])       # a third of the block below the threshold
    return dict(t=t, y=y, th=th, tx=tx, nhp=nhp, nc=nc, k_lo=k_lo, kwp=kwp, hyp=hyp, causal=causal,
                causal_id=causal_id, cull=cull, ld=ld)


def _ahx_bar(v, E, S, pref):
    """Per-element bound on |kernel - exact|: the exponent carries ~eps per unit of its terms' magnitude (S), exp /
    erfc / erfcx of cgmath.cuh are within a few ulp, the z < 0 branch cancels 2 exp(E) against the erfcx term (bounded
    by 2 pref exp(E)), and the flushing exp() drops results below 2^-1021."""
    with np.errstate(over='ignore', under='ignore', invalid='ignore'):
        mag = np.maximum(np.abs(v), 2 * pref * np.exp(np.minimum(E, 0)))
    return 16 * EPS * (8 + S) * mag + 4 * pref * TINY


@pytest.mark.parametrize('name', sorted(AHX_CASES))
def test_ahx_gen_matches_float64(name):
    c = _ahx_case(name)
    t, y, th, tx, nhp, nc, k_lo, kwp, ld = c['t'], c['y'], c['th'], c['tx'], c['nhp'], c['nc'], c['k_lo'], c['kwp'], c['ld']
    nv, nh, nx = len(t), len(th), len(tx)
    cull = c['cull'] if c['cull'] > 0 else 746.0
    seps = [True, False] if (c['causal'] and not c['causal_id']) else [False]
    ref, E, S, pref = ahx_ref(t, th, tx, k_lo, kwp, nhp, nc, c['hyp'], c['causal'], c['causal_id'])
    live = np.isfinite(E)
    band = 1e-12 * cull
    culled = live & (E < -cull - band)
    kept = live & (E > -cull + band)
    bar = _ahx_bar(ref, E, S, pref)
    got = {}
    for sep in seps:
        A, yp = ahx_gen_gpu(t, y, th, tx, nhp, nc, k_lo, kwp, c['hyp'], c['causal'], c['causal_id'], c['cull'], sep, ld)
        got[sep] = A
        assert not np.isnan(A).any(), 'elements left unwritten'
        assert np.all(A[~live] == 0.0), 'padding (rows >= nh, observations >= n_valid, k_lo + k >= nx) must be 0'
        assert np.all(A[culled] == 0.0), 'elements with E < -cull must be 0'
        err = np.abs(A - ref)
        assert np.all(err[kept] <= bar[kept]), (sep, (err[kept] / bar[kept]).max())
        edge = live & ~culled & ~kept                        # within the band: either 0 or the value
        assert np.all((A[edge] == 0.0) | (np.abs(A[edge] - ref[edge]) <= bar[edge]))
        # Y slice partials: sum over slices of the rows i < nh at columns k_lo + k < nx is sum_n y_n A; 0 elsewhere
        slices = (nc + 15) // 16
        assert yp.shape[0] == slices and not np.isnan(yp).any()
        # (slices and the reference summed in extended precision: what is left is the kernel's own sum of 16
        # observations per slice, 20 roundings at most.  The absolute floor covers sums whose terms are within a few
        # hundred binades of the subnormals: there the generic kernel's sums were seen off by up to 1.5e-300 against
        # Y ~ 1e-290 (not understood yet; the elements of A themselves pass the element-wise bar there))
        Y = yp.astype(np.longdouble).sum(0)
        kk = np.arange(k_lo, min(k_lo + kwp, nx))
        Yr = np.zeros_like(Y)
        Yb = np.zeros(Y.shape)
        yy = np.zeros(nc)
        yy[:nv] = y
        Yr[:nh, kk] = np.einsum('n,ink->ik', yy.astype(np.longdouble), A[:nh, :, :len(kk)].astype(np.longdouble))
        Yb[:nh, kk] = np.einsum('n,ink->ik', np.abs(yy), np.abs(A[:nh, :, :len(kk)]))
        assert np.all(Y[Yb == 0] == 0.0)
        yerr = np.abs(Y - Yr).astype(np.float64)
        print('%s sep=%d: max err / bar %.3g, %d kept, %d culled; Y: max err / (eps sum|y||A|) %.3g'
              % (name, sep, (err[kept] / bar[kept]).max() if kept.any() else 0.0, kept.sum(), culled.sum(),
                 (yerr / (EPS * Yb + 1e-300)).max()))
        assert np.all(yerr <= 12 * EPS * Yb + 1e-290), (sep, (yerr / (EPS * Yb + 1e-300)).max())
    if len(seps) == 2:
        d = np.abs(got[True] - got[False])
        assert np.all(d[kept] <= 2 * bar[kept]), (d[kept] / bar[kept]).max()
        assert np.array_equal(got[True][~kept & ~(live & ~culled)], got[False][~kept & ~(live & ~culled)])
    # a seeded sample of elements, and every element next to the threshold or a sign change of z, in 40 digits
    rng = np.random.default_rng(0)
    idx = list(zip(*np.nonzero(kept)))
    pick = [idx[j] for j in rng.choice(len(idx), min(48, len(idx)), replace=False)] if idx else []
    near = np.argwhere(live & (np.abs(E + cull) < 1e-3 * cull) & (E > -cull + band))
    pick += [tuple(p) for p in near[:16]]
    for sep, A in got.items():
        for i, n, k in pick:
            d = t[n] - tx[k_lo + k]
            v = ahx_mp(th[i], d, c['hyp'], c['causal'], c['causal_id'])
            assert abs(A[i, n, k] - v) <= bar[i, n, k], (sep, i, n, k, A[i, n, k], v)


# ---------------------------------------------------------------------------------------------------------- Ahx dot
def ahx_torch(t, th, tx, k_lo, kwp, nhp, nc, hyp_t, causal, causal_id):
    """oracle/model.py::psi_Ahx on the padded block (padding: 0), differentiable in hyp_t."""
    from oracle import model as om
    nv, nh, nx = len(t), len(th), len(tx)
    kv = max(0, min(kwp, nx - k_lo))
    out = torch.zeros(nhp, nc, kwp, dtype=torch.float64)
    a = om.psi_Ahx(t, th, tx[k_lo:k_lo + kv], hyp_t[0], hyp_t[1], hyp_t[2], bool(causal), bool(causal_id))  # [n, i, k]
    out = out.index_put((torch.arange(nh)[:, None, None], torch.arange(nv)[None, :, None],
                         torch.arange(kv)[None, None, :]), a.permute(1, 0, 2))
    return out


@pytest.mark.parametrize('name', ['bench_80', 'end_of_grid_nx203', 'kwp304_two_k_per_thread', 'toy_causal',
                                  'toy_acausal', 'toy_causal_id', 'kwp8_short_slice'])
def test_ahx_dot_matches_autograd(name):
    c = _ahx_case(name)
    t, y, th, tx, nhp, nc, k_lo, kwp, ld = c['t'], c['y'], c['th'], c['tx'], c['nhp'], c['nc'], c['k_lo'], c['kwp'], c['ld']
    nv, nh, nx = len(t), len(th), len(tx)
    if nc > 512:                                    # the reference holds the block with its autograd graph
        nv = nc = 512
        t, y = t[:nv], y[:nv]
    cull = c['cull'] if c['cull'] > 0 else 746.0
    rng = np.random.default_rng(1)
    E = _ahx_terms(t, th, tx, k_lo, kwp, nhp, nc, c['hyp'], c['causal_id'])[0]
    live = np.isfinite(E)
    W = rng.standard_normal((nhp, nc, kwp))
    Ybar = rng.standard_normal((nhp, ld))
    kk = np.arange(ld)
    Ybar[nh:, :] = np.nan                           # every position the kernels must not read
    Ybar[:, (kk < k_lo) | (kk >= min(k_lo + kwp, nx))] = np.nan
    W[~live] = np.nan
    for sep in ([True, False] if (c['causal'] and not c['causal_id']) else [False]):
        A, _ = ahx_gen_gpu(t, y, th, tx, nhp, nc, k_lo, kwp, c['hyp'], c['causal'], c['causal_id'], c['cull'], sep, ld)
        tp, yy = np.zeros(nc), np.zeros(nc)
        tp[:nv], yy[:nv] = t, y
        dt, dy, dth, dtx = _dev(tp), _dev(yy), _dev(th), _dev(tx)
        dA, dW, dYb = _dev(A), _dev(W), _dev(Ybar)
        g3 = torch.full((3,), float('nan'), dtype=torch.float64, device='cuda')
        hp = np.ascontiguousarray(c['hyp'])
        rc = _lib.lib().cgpcm_ahx_dot_test(dt.data_ptr(), dy.data_ptr(), nv, nc, dth.data_ptr(), nh, nhp,
                                           dtx.data_ptr(), nx, k_lo, kwp, hp.ctypes.data, int(c['causal']),
                                           int(c['causal_id']), c['cull'], int(sep), ld, dA.data_ptr(), dW.data_ptr(),
                                           dYb.data_ptr(), g3.data_ptr(), None)
        assert rc == 0
        g = g3.cpu().numpy()
        assert np.all(np.isfinite(g)), g
        # reference: d/dtheta of sum over the live, unculled elements of (W + y Ybar) psi_Ahx
        wt = np.where(live, W, 0.0) + yy[None, :, None] * np.nan_to_num(Ybar[:, k_lo:k_lo + kwp])[:, None, :]
        wt = np.where(live & (E >= -cull), wt, 0.0)
        h = torch.tensor(c['hyp'], dtype=torch.float64, requires_grad=True)
        F = ahx_torch(t, th, tx, k_lo, kwp, nhp, nc, h, c['causal'], c['causal_id'])
        (torch.as_tensor(wt) * F).sum().backward()
        gr = h.grad.numpy()
        # bound: sum |w| |dA/dtheta| with the element derivative's parts taken in magnitude
        hb = torch.tensor(c['hyp'], dtype=torch.float64)
        mags = []
        for j in range(3):
            tang = torch.zeros(3, dtype=torch.float64)
            tang[j] = 1.0
            _, dF = torch.func.jvp(lambda hh: ahx_torch(t, th, tx, k_lo, kwp, nhp, nc, hh, c['causal'], c['causal_id']),
                                   (hb,), (tang,))
            mags.append(float((np.abs(wt) * np.abs(dF.numpy())).sum()))
        Eabs = np.abs(np.where(live & (E >= -cull), E, 0)).max()
        for j in range(3):
            assert abs(g[j] - gr[j]) <= 64 * EPS * (8 + Eabs) * mags[j] + 1e-300, (sep, j, g[j], gr[j], mags[j])
        print('%s sep=%d: |g - ref| / (eps sum|w||dA|) = %s' % (name, sep, [abs(g[j] - gr[j]) / (EPS * mags[j])
                                                                           for j in range(3)]))


# ---------------------------------------------------------------------------------------------------------- Axx sum
def axx_gpu(t, tx, hyp, causal, causal_id, cull, slices, sorted_, ld):
    nx = len(tx)
    out = torch.full((4, ld, ld), float('nan'), dtype=torch.float64, device='cuda')
    dt, dtx = _dev(t), _dev(tx)
    hp = np.ascontiguousarray(hyp, dtype=np.float64)
    rc = _lib.lib().cgpcm_axx_sum_test(dt.data_ptr(), len(t), int(sorted_), dtx.data_ptr(), nx, hp.ctypes.data,
                                       int(causal), int(causal_id), cull, slices, 1, ld, out.data_ptr(), None)
    assert rc == 0
    return out.cpu().numpy()


@functools.lru_cache(None)
def axx_ref(nx, rho_src, causal, causal_id, cull, seed):
    """sum_n psi_Axx (oracle) over the observations, its contraction with random weights R and the gradient of that
    contraction w.r.t. (alpha, gamma, omega) by torch autograd, chunked over observations; also sum_n |Axx|."""
    from oracle import model as om
    t, tx, hyp = axx_inputs(nx, rho_src)
    rng = np.random.default_rng(seed)
    R = np.tril(rng.standard_normal((nx, nx)))
    h = torch.tensor(hyp, dtype=torch.float64, requires_grad=True)
    S = torch.zeros(nx, nx, dtype=torch.float64)
    a, g, o = hyp
    A = a + g + o
    det = 4 * (A * A - g * g)
    S11, S12 = 2 * A / det, 2 * g / det
    g1, g2 = o * (1 - 2 * o * S11), 4 * o * o * S12
    for s in range(0, len(t), 64):
        tc = t[s:s + 64]
        d = tc[:, None] - tx[None, :]
        G = -g1 * (d[:, :, None] ** 2 + d[:, None, :] ** 2) + g2 * d[:, :, None] * d[:, None, :]
        X = om.psi_Axx(tc, tx, h[0], h[1], h[2], bool(causal), bool(causal_id))
        X = X * torch.as_tensor(G >= -(cull if cull > 0 else 746.0))
        S = S + X.sum(0)
    (S * torch.as_tensor(R)).sum().backward()
    return S.detach().numpy(), R, h.grad.numpy()


def axx_inputs(nx, rho_src):
    """Every 400th observation of the bench's series (250 over [0, 100]) and nx inducing inputs on the bench's grid
    spacing (the rest of the observations only add more of the same elements); rho_src = 'bench': the bench's
    hyper-parameters (rho = 0.968, hoisted BVN branch), 'low': omega 40 x larger (rho below 0.925)."""
    w = bench()
    t = np.ascontiguousarray(w['t'][::400])
    tx = w['tx'][100 - nx // 2:100 - nx // 2 + nx] if nx < 200 else w['tx']
    a, g, o = w['hyp']
    hyp = (a, g, o) if rho_src == 'bench' else (a, g, 40 * o)
    return t, np.ascontiguousarray(tx), np.array(hyp)


AXX_CASES = [  # nx, rho, causal, causal_id, cull, slices, sorted
    (16, 'bench', 1, 0, 746.0, 7, 1),
    (40, 'bench', 1, 0, 80.0, 1, 0),
    (40, 'low', 1, 0, 80.0, 64, 1),
    (40, 'low', 0, 0, 746.0, 7, 0),
    (40, 'bench', 1, 1, 80.0, 7, 1),
    (200, 'bench', 1, 0, 80.0, 64, 1),
    (200, 'bench', 1, 0, 746.0, 1, 0),
    (200, 'low', 1, 0, 746.0, 7, 0),
]


@pytest.mark.parametrize('case', AXX_CASES, ids=lambda c: '-'.join(map(str, c)))
def test_axx_sum_and_tangents_match_autograd(case):
    nx, rho_src, causal, causal_id, cull, slices, sorted_ = case
    t, tx, hyp = axx_inputs(nx, rho_src)
    if rho_src == 'bench':
        assert hyp[1] / hyp.sum() >= 0.925
    else:
        assert hyp[1] / hyp.sum() < 0.925
    ld = -(-nx // 8) * 8
    if not sorted_:
        t = np.ascontiguousarray(np.random.default_rng(2).permutation(t))
    out = axx_gpu(t, tx, hyp, causal, causal_id, cull, slices, sorted_, ld)
    S, R, gref = axx_ref(nx, rho_src, causal, causal_id, cull, 0)
    assert not np.isnan(out).any()
    assert np.all(out[:, nx:, :] == 0.0) and np.all(out[:, :, nx:] == 0.0)
    for m in range(4):
        np.testing.assert_array_equal(out[m, :nx, :nx], out[m, :nx, :nx].T)
    # values: the BVN of bvn.cuh (table Genz / Chebyshev-hoisted) and of the oracle are both within ~1e-15 absolute
    err = np.abs(out[0, :nx, :nx] - S)
    bar = 1e-13 * np.abs(S).max() + 64 * EPS * np.abs(S)
    assert np.all(err <= bar), (err / bar).max()
    # tangents: <R, dAxx/dtheta> against autograd; bound from the magnitudes the kernel sums
    for j in range(3):
        T = out[1 + j, :nx, :nx]
        got = float((np.tril(T) * R).sum())
        mag = float((np.abs(np.tril(T)) * np.abs(R)).sum())
        assert abs(got - gref[j]) <= 1e-12 * mag, (j, got, gref[j], abs(got - gref[j]) / (EPS * mag))
        print('tangent %d: |got - ref| / (eps sum|R||T|) = %.3g' % (j, abs(got - gref[j]) / (EPS * mag)))


# ---------------------------------------------------------------------------------------------------- window chol
def _spd(n, seed, cond=1e6):
    rng = np.random.default_rng(seed)
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    S = (Q * np.logspace(0, -math.log10(cond), n)) @ Q.T
    return (S + S.T) / 2


def window_chol_gpu(M, ld, sign, windows, tag):
    dM = _dev(M)
    total = sum(kw * kw for _, kw, _ in windows)
    out = torch.full((total,), float('nan'), dtype=torch.float64, device='cuda')
    win = np.ascontiguousarray(np.asarray(windows, dtype=np.int32).reshape(-1, 3))
    info = ctypes.c_int(-7)
    rc = _lib.lib().cgpcm_window_chol_test(dM.data_ptr(), ld, sign, len(windows), win.ctypes.data, tag, out.data_ptr(),
                                           ctypes.byref(info), None)
    assert rc == 0
    res, o = [], 0
    h = out.cpu().numpy()
    for _, kw, _ in windows:
        res.append(h[o:o + kw * kw].reshape(kw, kw))
        o += kw * kw
    return res, info.value


def _check_factor(S, M, sign, k_lo, kw, kv):
    """S = L^T of the identity-padded block: exactly upper triangular, identity rows / columns >= kv, backward error
    |L L^T - W| <= c eps |L| |L|^T."""
    assert not np.isnan(S).any()
    assert np.all(np.tril(S, -1) == 0.0)
    W = np.eye(kw)
    W[:kv, :kv] = sign * M[k_lo:k_lo + kv, k_lo:k_lo + kv]
    L = S.T
    err = np.abs(L @ L.T - W)
    assert np.all(err <= 4 * kw * EPS * (np.abs(L) @ np.abs(L).T) + 1e-300), (kw, kv)
    np.testing.assert_array_equal(S[kv:, kv:], np.eye(kw - kv))
    assert np.all(S[:kv, kv:] == 0.0)


@pytest.mark.parametrize('ld,sign', [(200, 1.0), (208, -1.0)])
def test_window_chol_all_widths_in_one_launch(ld, sign):
    n = ld
    M = sign * _spd(n, 3)
    widths = list(range(8, 105, 8)) + [120]
    rng = np.random.default_rng(4)
    windows = []
    for j, kw in enumerate(widths):
        kv = kw if j % 3 else max(0, kw - 2 * (j % 5) - 3)       # every third window: kv < kw (identity padding)
        k_lo = int(rng.integers(0, (n - kw) // 2 + 1)) * 2      # as in the sweep, k_lo + kw <= ld
        windows.append((k_lo, kw, kv))
    windows.append((n - 48, 48, 40))                            # the last window of a grid with nx = ld - 8
    res, info = window_chol_gpu(M, ld, sign, windows, 6)
    assert info == 0
    for (k_lo, kw, kv), S in zip(windows, res):
        _check_factor(S, M, sign, k_lo, kw, kv)


def test_window_chol_reports_the_failed_pivot():
    ld = 208
    M = _spd(ld, 5, cond=1e3)
    windows = [(0, 104, 104), (40, 64, 64), (100, 96, 96), (150, 56, 56)]
    j = 17
    bad_lo = 100
    M[bad_lo + j, bad_lo + j] = -1.0                             # only the third window contains it
    # keep the other windows away from row / column bad_lo + j = 117: window 0 covers 0..103, window 1 40..103
    res, info = window_chol_gpu(M, ld, 1.0, windows, 7)
    assert info == 7 * 100000 + bad_lo + j + 1
    for w in (0, 1, 3):
        _check_factor(res[w], M, 1.0, *windows[w])


# ------------------------------------------------------------------------------------------------- windowed products
def test_right_multiply_by_a_window_view():
    """Abar = T1 Wx as the sweep computes it: cgpcm_dgemm(1, 1, 1, kwp, nhp nc, kwp) with the resident operand a window
    of the ld x ld matrix (lds = ld > K), on the persistent small-left kernel."""
    ld, nhp = 208, 200
    Wm = _spd(ld, 6, cond=1e2)
    for kwp, nc, k_lo in [(16, 48, 10), (40, 64, 100), (104, 48, 104), (96, 56, 0)]:
        N = nhp * nc
        X = np.random.default_rng(kwp).standard_normal((N, kwp))
        dW, dX = _dev(Wm), _dev(X)
        out = torch.full((N, kwp), float('nan'), dtype=torch.float64, device='cuda')
        rc = _lib.lib().cgpcm_dgemm(1, 1, 1, kwp, N, kwp, 1.0, dW.data_ptr() + 8 * (k_lo * ld + k_lo), ld,
                                    dX.data_ptr(), kwp, 0.0, out.data_ptr(), kwp, 1, 0, 0, None)
        assert rc == 0
        got = out.cpu().numpy()
        blk = Wm[k_lo:k_lo + kwp, k_lo:k_lo + kwp]
        ref = X @ blk
        bound = np.abs(X) @ np.abs(blk)
        assert np.all(np.abs(got - ref) <= 4 * EPS * bound + 1e-300), (kwp, np.abs(got - ref).max())


def test_triangular_right_multiply_every_window_width():
    """V' = A L (cgpcm_dgemm_tri) at every width the sweep uses, N = nhp nc ragged against the 64-wide tile."""
    nhp, nc = 200, 52                                            # N = 10400 = 162.5 x 64
    N = nhp * nc
    rng = np.random.default_rng(7)
    X = rng.standard_normal((N, 104))
    for kwp in range(16, 105, 8):
        Xk = np.ascontiguousarray(X[:, :kwp])
        dX = _dev(Xk)
        S = np.triu(rng.standard_normal((kwp, kwp)))
        dS = _dev(S)
        out = torch.full((N, kwp), float('nan'), dtype=torch.float64, device='cuda')
        rc = _lib.lib().cgpcm_dgemm_tri(kwp, N, dS.data_ptr(), kwp, dX.data_ptr(), kwp, out.data_ptr(), kwp, None)
        assert rc == 0
        got = out.cpu().numpy()
        ref = Xk @ S.T
        bound = np.abs(Xk) @ np.abs(S.T)
        assert np.all(np.abs(got - ref) <= 4 * EPS * bound + 1e-300), (kwp, np.abs(got - ref).max())


def sym_accum_gpu(windows, A, B, n, ld):
    win = np.ascontiguousarray(np.asarray(windows, dtype=np.int64).reshape(-1, 6))
    out = torch.full((n, ld), float('nan'), dtype=torch.float64, device='cuda')
    rc = _lib.lib().cgpcm_sym_accum_test(len(windows), win.ctypes.data, A.data_ptr(), B.data_ptr(), n, ld,
                                         out.data_ptr(), None)
    assert rc == 0
    return out.cpu().numpy()[:, :n]


def _sym_ref(windows, A, B, n):
    ref, bound, cover = np.zeros((n, n)), np.zeros((n, n)), np.zeros((n, n), bool)
    for kc, k_lo, order, K, ao, bo in windows:
        if kc:
            a, b = A[ao:ao + order * K].reshape(order, K), B[bo:bo + order * K].reshape(order, K)
        else:
            a, b = A[ao:ao + K * order].reshape(K, order).T, B[bo:bo + K * order].reshape(K, order).T
        P = a @ b.T
        P = np.tril(P) + np.tril(P, -1).T                         # the kernels compute the lower triangle
        ref[k_lo:k_lo + order, k_lo:k_lo + order] += P
        bound[k_lo:k_lo + order, k_lo:k_lo + order] += np.abs(a) @ np.abs(b).T
        cover[k_lo:k_lo + order, k_lo:k_lo + order] = True
    return ref, np.maximum(bound, bound.T), cover


def test_symmetric_contractions_as_the_sweeps_accumulate_them():
    """C1-like: overlapping windows of orders 8..200 (both routes: the split-K tiled kernel up to order 40, dgemm_sym
    above) with k-contiguous operands as the forward sweep passes A and T1, K up to 200 x 2048 (148 K-slices), added
    into the slice buffers at (k_lo, k_lo); Q-like: order nhp with row-contiguous operands (a_kc = 1)."""
    n, ld = 200, 208
    rng = np.random.default_rng(8)
    c1 = [(0, 0, 104, 200 * 1024), (0, 96, 104, 200 * 512), (0, 48, 40, 200 * 2048), (0, 56, 8, 200 * 64),
          (0, 150, 48, 200 * 256), (0, 0, 200, 200 * 512), (0, 192, 8, 200 * 16)]
    q = [(1, 0, 200, 40 * 512), (1, 0, 200, 104 * 256)]
    for wl in (c1, q):
        total_a = sum(o * K for _, _, o, K in wl)
        A = rng.standard_normal(total_a)
        B = rng.standard_normal(total_a)                         # op(A) op(B)^T is not symmetric: the lower triangle counts
        wins, off = [], 0
        for kc, k_lo, order, K in wl:
            wins.append((kc, k_lo, order, K, off, off))
            off += order * K
        got = sym_accum_gpu(wins, _dev(A), _dev(B), n, ld)
        ref, bound, cover = _sym_ref(wins, A, B, n)
        assert not np.isnan(got).any()
        np.testing.assert_array_equal(got, got.T)
        assert np.all(got[~cover] == 0.0)
        err = np.abs(got - ref)
        print('sym accum: max err / (eps sum|A||B|) = %.3g' % (err / (EPS * bound + 1e-300)).max())
        assert np.all(err <= 4 * EPS * bound), (err / (EPS * bound + 1e-300)).max()


# ------------------------------------------------------------------------------------------------ routes vs oracle
ROUTES = [dict(tri=0), dict(sl=0), dict(sep=0), dict(axx_slices=1), dict(axx_slices=64)]


@functools.lru_cache(None)
def _oracle_m200(which):
    """96 observations in the middle of the series and the oracle's ELBO / gradient with their ulp noise; 'fixture':
    the M = 200 workload on [0, 4] (rho = 0.86), 'bench': the bench's own series and hyper-parameters (rho = 0.968)."""
    from oracle import model as om
    from tests.cases import ulp_noise
    w = sweep_workload(4000, 200, seed=3) if which == 'fixture' else bench()
    c = len(w['t']) // 2
    sl = slice(c - 48, c + 48)
    t, y = np.ascontiguousarray(w['t'][sl]), np.ascontiguousarray(w['y'][sl])
    om.PW_DISTS_EXACT = True
    try:
        (e0, t0, g0), (en, tn, gn) = ulp_noise(
            lambda p, th: om.elbo_and_grad(p, t, y, th, w['tx'], w['reg']), w['params'], w['th'], trials=1)
    finally:
        om.PW_DISTS_EXACT = False
    return w, t, y, (e0, t0, g0), (en, tn, gn)


@pytest.mark.parametrize('which', ['fixture', 'bench'])
@pytest.mark.parametrize('cull', [80.0, 746.0])
def test_every_route_matches_the_oracle_at_m200(which, cull):
    w, t, y, (e0, t0, g0), (en, tn, gn) = _oracle_m200(which)
    scale = max(abs(e0), np.abs(t0).max())
    for opts in [dict()] + ROUTES:
        e = cgpcm_b200.Engine(200, 200)
        e.set_option('cull', cull)
        e.set_option('chunk', 48)
        for k, v in opts.items():
            e.set_option(k, v)
        e.set_data(t, y, w['th'], w['tx'])
        e1, t1, g1 = e.elbo_grad(w['params'], reg=w['reg'])
        e.close()
        assert abs(e1 - e0) <= 1e-9 * scale + 3 * en, (opts, e1, e0)
        assert np.abs(t1 - t0).max() <= 1e-9 * scale + 3 * tn, opts
        assert np.abs(g1 - g0).max() <= 1e-9 * np.abs(g0).max() + 3 * gn, (opts, np.abs(g1 - g0).max())


def test_every_route_matches_the_default_at_full_size():
    """N = 1e5, M = 200: each option against the default route, within the bar of two summation orders of the same
    sums (tests/test_gpu_fullsize.py::test_dense_equals_culled_and_terms_sum)."""
    w = bench()
    e = cgpcm_b200.Engine(200, 200)
    e.set_data(w['t'], w['y'], w['th'], w['tx'])
    for cull in (80.0, 746.0):
        e.set_option('cull', cull)
        base = e.elbo_grad(w['params'], reg=w['reg'])
        for opts in ROUTES:
            for k, v in opts.items():
                e.set_option(k, v)
            got = e.elbo_grad(w['params'], reg=w['reg'])
            for k in opts:
                e.set_option(k, {'tri': 1, 'sl': 1, 'sep': 1, 'axx_slices': 0}[k])
            assert abs(got[0] - base[0]) <= 6e-10 * abs(base[0]), (cull, opts)
            assert np.abs(got[2] - base[2]).max() <= 1e-9 * np.abs(base[2]).max(), (cull, opts)
    e.close()

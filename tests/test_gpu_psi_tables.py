"""The table-driven routines of the separable Ahx kernel (csrc/cgmath.cuh: cg_erfcx_tab and cg_exp_neg with a
power-of-two bias) against mpmath over their whole range, through cgpcm_math_test_tab, and ahx_gen_sep_kernel<true>
against 40-digit values where f_i g_nk alone underflows: at the bench's hyper-parameters, the elements next to the
edges of an exact (cull 746) window, with ln(f_i g_nk) = E - z^2 below -708, must keep their relative accuracy."""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip('torch')

from cgpcm_b200 import _lib
from tests.test_gpu_sweep_kernels import EPS, _ahx_case, _ahx_terms, ahx_gen_gpu, ahx_mp, ahx_ref


def _tab(x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    oe, oc, prm = np.empty_like(x), np.empty_like(x), np.zeros(3)
    assert _lib.lib().cgpcm_math_test_tab(_lib.ptr(x), x.shape[0], _lib.ptr(oe), _lib.ptr(oc), _lib.ptr(prm)) == 0
    return oe, oc, prm


def test_erfcx_table_against_mpmath():
    """erfcx over the table's whole range [zlo, zhi]: <= 4.5 ulp against mpmath, both when four neighbouring arguments
    share one interval's coefficients (sorted, close) and when each takes its own (shuffled groups)."""
    import mpmath as mp
    mp.mp.dps = 40
    _, _, (zlo, zhi, _) = _tab(np.zeros(4))
    rng = np.random.default_rng(21)
    w = 1.0 / 32
    edges = zlo + w * np.arange(int(round((zhi - zlo) / w)) + 1)
    pts = np.concatenate([rng.uniform(zlo, zhi, 6000), edges, np.nextafter(edges, -np.inf), np.nextafter(edges, np.inf),
                          [0.0, -0.0, zlo, zhi]])
    pts = np.clip(pts, zlo, zhi)
    close = np.sort(pts)                                   # groups of 4 within one interval (or its margin)
    spread = rng.permutation(pts)                          # groups of 4 far apart: one interval each
    for name, x in (('close', close), ('spread', spread)):
        _, oc, _ = _tab(x)
        worst = 0.0
        for xi, got in zip(x, oc):
            want = mp.exp(mp.mpf(xi) ** 2) * mp.erfc(mp.mpf(xi))
            worst = max(worst, float(abs(mp.mpf(float(got)) - want) / mp.mpf(float(np.spacing(float(want))))))
        print('erfcx table, %s groups: worst %.3f ulp' % (name, worst))
        assert worst <= 4.5, (name, worst)


def test_biased_exp_against_mpmath():
    """exp(x) 2^B: the significand of the flushing exp (<= 2 ulp), normal down to about exp(-(1021 + B) ln 2), 0 from
    there on (flushed when the scaled power of two is below 2^-1021)."""
    import mpmath as mp
    mp.mp.dps = 40
    _, _, (_, _, bias) = _tab(np.zeros(4))
    bias = int(bias)
    lim = (1021 + bias) * math.log(2)
    rng = np.random.default_rng(22)
    x = np.concatenate([-rng.uniform(0, lim + 5, 3000), -10.0 ** rng.uniform(-12, 0, 200),
                        [0.0, -708.0, -745.5, -810.0, -lim + 0.01, -lim - 1.0, -2000.0]])
    oe, _, _ = _tab(x)
    worst = 0.0
    for xi, got in zip(x, oe):
        want = mp.exp(mp.mpf(float(xi))) * mp.mpf(2) ** bias
        if want < mp.mpf(2) ** -1021:
            assert got == 0.0 or got <= 2.0 ** -1021, (xi, got)
            continue
        worst = max(worst, float(abs(mp.mpf(float(got)) - want) / mp.mpf(float(np.spacing(float(want))))))
    assert worst <= 2.0, worst
    assert oe[x == -lim - 1.0] == 0.0 and oe[x == -2000.0] == 0.0 and oe[x == -lim + 0.01] > 0.0
    assert oe[x == 0.0] == 2.0 ** bias


@pytest.mark.parametrize('name', ['bench_746', 'bench_746_last'])
def test_ahx_gen_sep_where_the_gaussian_factor_underflows(name):
    """At the bench's exact windows, elements with E >= -cull and ln(f_i g_nk) = E - z^2 < -708 (f_i g_nk below the
    normal range): the separable kernel returns them to a relative bar in 40 digits, not 0 or a rounding residue."""
    c = _ahx_case(name)
    t, y, th, tx, nhp, nc, k_lo, kwp, ld = c['t'], c['y'], c['th'], c['tx'], c['nhp'], c['nc'], c['k_lo'], c['kwp'], c['ld']
    E, z, cc, S = _ahx_terms(t, th, tx, k_lo, kwp, nhp, nc, c['hyp'], c['causal_id'])
    ref = ahx_ref(t, th, tx, k_lo, kwp, nhp, nc, c['hyp'], c['causal'], c['causal_id'])[0]
    live = np.isfinite(E)
    assert z[live & (E >= -746.0)].min() > -8.0              # inside the erfcx table: the table path is the one taken
    A, _ = ahx_gen_gpu(t, y, th, tx, nhp, nc, k_lo, kwp, c['hyp'], c['causal'], c['causal_id'], c['cull'], True, ld)
    under = live & (E > -746.0 + 1e-6) & (cc < -708.0) & (E < -600.0)
    assert under.sum() > 0, 'the case must reach elements whose Gaussian factor underflows'
    rng = np.random.default_rng(3)
    idx = np.argwhere(under)
    idx = idx[rng.choice(len(idx), min(40, len(idx)), replace=False)]
    worst = 0.0
    for i, n, k in idx:
        v = ahx_mp(th[i], t[n] - tx[k_lo + k], c['hyp'], c['causal'], c['causal_id'])
        if v < 2.0 ** -1022:                                 # subnormal results: one rounding of the last scaling
            assert abs(A[i, n, k] - v) <= 2.0 ** -1074 + 16 * EPS * (8 + S[i, n, k]) * v, (i, n, k, A[i, n, k], v)
            continue
        rel = abs(A[i, n, k] - v) / v / (EPS * (8 + S[i, n, k]))
        worst = max(worst, rel)
    print('%s: %d elements with f g < 2^-1021, worst error %.3g eps (8 + S)' % (name, under.sum(), worst))
    assert worst <= 16.0, worst
    kept = live & (E > -746.0 + 1e-6)
    assert np.all(A[kept & (ref > 2.0 ** -1000)] > 0.0)

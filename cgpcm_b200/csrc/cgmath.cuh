// FP64 exp / erfc for the Psi kernels, U elements at a time (sm_100a).
//
// Why not the CUDA math library here: `ahx_gen_kernel` spends one exp() and one erfc() per element and is bound by
// instruction issue, not by the FP64 pipe (ncu, profiles/r01_ncu_psi_kernels_exact746.txt: FP64 pipe 54 % active,
// issue slots 77 %).  Its SASS shows why: ptxas materialises every polynomial coefficient of the inlined library
// routines with two 32-bit moves (UMOV / IMAD.MOV) right before the DFMA that uses it -- 105 of the 254 instructions of
// the per-element loop are constant moves, 89 are FP64.  The routines below evaluate U independent arguments in
// lock-step (arrays in registers, every step an unrolled loop over u), so one materialised coefficient feeds U DFMAs,
// and they are branch-free (no slow paths: the argument ranges of the Psi statistics are known).
//
//   cg_exp_neg<U>(x)   exp(x) for x <= 0 (arguments below -750 give 0): n = rint(x log2 e), r = x - n ln 2 (two FMAs),
//                      degree-12 polynomial (Chebyshev interpolant of exp on |r| <= ln2 / 2, error 3e-18), scaling by
//                      2^n in two exact steps so that subnormal results round once.
//   cg_erfc<U>(z)      erfc(z) for any finite z: with x = |z| (clamped at 27.3, where erfc underflows) and
//                      t = (x - 4) / (x + 4) in [-1, 1),  erfc(x) = exp(-x^2) g(t) / (1 + 2 x),  g(t) = (1 + 2x) erfcx(x)
//                      a degree-26 polynomial (Chebyshev interpolant, truncation 4e-17, sum |c_i| = 1.8 so Horner is
//                      well conditioned); exp(-x^2) from the rounded square and its exact residual (fma);
//                      one reciprocal (hardware approximation + 2 Newton steps) serves both divisions;
//                      erfc(z) = 2 - erfc(-z) for z < 0.
//   cg_erfcx_tab<U>(z) erfcx(z) for signed z in [-8, 3]: piecewise polynomial, 352 intervals of degree 10 (below).
// Coefficients: computed with mpmath at 60 digits (tools/fit_cgmath.py), rounded to double; accuracy against mpmath is
// tested in tests/test_gpu_kernels.py (cgpcm_math_test): <= 2 ulp (exp), <= 4 ulp (erfc) over the whole range, and in
// tests/test_gpu_psi_tables.py (cgpcm_math_test_tab): <= 4.5 ulp (cg_erfcx_tab).
#pragma once
#include <cuda_runtime.h>

namespace cg {

// descending order (Horner): c12 .. c0
#define CG_EXP_COEFS(X)                                                                                        \
  X(0x1.af785d433f066p-26) X(0x1.27e4cc1847a65p-22) X(0x1.71dde76ab2f81p-19) X(0x1.a01a01adc27e2p-16)          \
  X(0x1.a01a01b80226cp-13) X(0x1.6c16c16c14d77p-10) X(0x1.111111110db76p-7) X(0x1.5555555555559p-5)           \
  X(0x1.5555555555562p-3) X(0x1.0000000000000p-1) X(0x1.0000000000000p+0) X(0x1.0000000000000p+0)
#define CG_EXP_C12 0x1.1f8b43f2637adp-29

// descending order: c25 .. c0
#define CG_ERFC_COEFS(X)                                                                                       \
  X(-0x1.2dbbbb75b6682p-33) X(-0x1.2d277a41632e3p-31) X(0x1.ebb009434f4efp-30) X(0x1.117f492198859p-28)        \
  X(-0x1.f9443297365a1p-27) X(-0x1.78888d24fa8a1p-26) X(0x1.d8d5b12b4bdebp-24) X(0x1.5305495fa5317p-24)        \
  X(-0x1.badf24e872985p-21) X(0x1.385bb6c82456ap-22) X(0x1.7f235478fdcf6p-18) X(-0x1.788189c990557p-17)        \
  X(-0x1.9958a8c635c6bp-16) X(0x1.3be032de511d3p-13) X(-0x1.a1df2ad41dddep-13) X(-0x1.8d4a9990c5199p-11)       \
  X(0x1.49c6728db72cdp-8) X(-0x1.0962388548d8dp-6) X(0x1.3079edf668f38p-5) X(-0x1.0fb06dfe48b0ep-4)            \
  X(0x1.7fee004e13186p-4) X(-0x1.9ddb23c3e9106p-4) X(0x1.16ecefcfa533fp-4) X(0x1.f7f5df66fd7bep-7)             \
  X(-0x1.1df1ad154a28ep-3) X(0x1.3ba5916e9fd7fp+0)
#define CG_ERFC_C26 0x1.7d604a7f621f4p-35

// The erfc coefficients live in constant memory: ptxas then reads each with one uniform load (LDCU.64) instead of two
// UMOVs of a literal -- ahx_gen_kernel: 888 -> 832 instructions, 0.8 ms per evaluation at the bench shape.  The exp
// coefficients stay literals: the same change made ahx_dot_kernel (exp only, already short of registers) 0.9 ms slower.
#define CG_LIST(c) c,
__constant__ double cg_erfc_c[27] = {CG_ERFC_C26, CG_ERFC_COEFS(CG_LIST)};
#undef CG_LIST

// FLUSH = true: results below 2^-1021 (x < -708.05) are returned as 0 and the scaling is one integer add to the
// exponent field instead of two exact multiplications (bit-identical for every normal result).  The Psi kernels use
// it: an element below 5e-308 changes no bit of a sum whose terms are O(1).
// BIAS (FLUSH only): returns exp(x) 2^BIAS -- the same significand, BIAS added to the exponent -- so that factors down
// to exp(-(1021 + BIAS) ln 2) stay normal; results below 2^-1021 are still returned as 0.
template <int U, bool FLUSH = false, int BIAS = 0>
__device__ __forceinline__ void cg_exp_neg(const double (&x)[U], double (&out)[U]) {
  static_assert(BIAS == 0 || (FLUSH && BIAS > 0 && BIAS < 1000), "BIAS needs FLUSH");
  double r[U], p[U];
  int ni[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const double xc = fmax(x[u], -750.0 - 0.6931471805599453 * BIAS);
    const double t = fma(xc, 0x1.71547652b82fep+0, 6755399441055744.0);      // x log2(e) + 1.5 * 2^52
    ni[u] = __double2loint(t);
    const double n = t - 6755399441055744.0;
    double rr = fma(n, -0x1.62e42fefa39efp-1, xc);
    r[u] = fma(n, -0x1.abc9e3b39803fp-56, rr);
    p[u] = CG_EXP_C12;
  }
#define CG_STEP(c)                  \
  _Pragma("unroll") for (int u = 0; u < U; ++u) p[u] = fma(p[u], r[u], c);
  CG_EXP_COEFS(CG_STEP)
#undef CG_STEP
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (FLUSH) {
      // p in [0.70, 1.42]: exponent field 1022 or 1023, so p 2^n is normal for n >= -1021
      const int nb = ni[u] + BIAS;
      const double v = __hiloint2double(__double2hiint(p[u]) + (nb << 20), __double2loint(p[u]));
      out[u] = nb >= -1021 ? v : 0.0;
    } else {
      const int k1 = ni[u] >> 1, k2 = ni[u] - k1;                             // both >= -541: normal powers of two
      const double s1 = __hiloint2double((1023 + k1) << 20, 0), s2 = __hiloint2double((1023 + k2) << 20, 0);
      out[u] = (p[u] * s1) * s2;
    }
  }
}

// erfcx(|z|) = exp(z^2) erfc(|z|) = g(t) / (1 + 2|z|): the polynomial part of cg_erfc without its exp(-z^2).  The
// separable Psi kernels (psi_kernels.cuh: ahx_gen_sep_kernel) multiply it by exp(E - z^2), which factorises over the
// filter and the noise inducing inputs, so no exponential of the erfc is evaluated per element.
template <int U>
__device__ __forceinline__ void cg_erfcx_abs(const double (&z)[U], double (&out)[U]) {
  double t[U], inv[U], g[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const double x = fmin(fabs(z[u]), 27.3);
    const double a = x + 4.0, b = fma(2.0, x, 1.0);
    const double den = a * b;
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(den));
    double err = fma(-den, y, 1.0);
    y = fma(y, err, y);
    err = fma(-den, y, 1.0);
    y = fma(y, err, y);
    t[u] = (x - 4.0) * (b * y);
    inv[u] = a * y;
    g[u] = cg_erfc_c[0];
  }
#pragma unroll
  for (int k = 1; k < 27; ++k) {
#pragma unroll
    for (int u = 0; u < U; ++u) g[u] = fma(g[u], t[u], cg_erfc_c[k]);
  }
#pragma unroll
  for (int u = 0; u < U; ++u) out[u] = g[u] * inv[u];
}

// erfcx(z) = exp(z^2) erfc(z) for signed z in [CG_ERFCX_TAB_ZLO, CG_ERFCX_TAB_ZHI]: interval j = floor((z - ZLO) / W)
// of CG_ERFCX_TAB_NI, polynomial of degree CG_ERFCX_TAB_DEG in x = z - c_j (c_j the interval's centre, so x is exact).
// Each polynomial interpolates erfcx on its interval widened by W / 8 on both sides (tools/fit_cgmath.py, 60 digits):
// <= 2 ulp before rounding of the Horner steps; tested against mpmath in tests/test_gpu_psi_tables.py.  Width and
// degree: W = 1/32 keeps degree 10 within 2 ulp down to z = -8, where erfcx grows by e^{2|z| W} = 1.65 per interval
// (W = 1/16 needs degree 12 there).  The coefficients are read through the L1 cache, coefficient-major: the lanes of
// a warp step through consecutive intervals (ahx_gen_sep_kernel: 0.7 in z over a warp at the bench shape, 23
// intervals), so a coefficient load of a warp touches one or two 128-byte lines.
// The U arguments are evaluated in lock-step on the interval of the first one whose keep[u] is set, when every kept
// argument lies on its widened interval (ahx_gen_sep_kernel: the U arguments are U consecutive observations at one
// inducing input, so they nearly always share an interval): one load per coefficient for all U.  Otherwise each
// argument is evaluated on its own interval.  Arguments outside the range give the value of the nearest end interval's
// polynomial (finite or not): callers check the range, and results with keep[u] = false are to be discarded.
constexpr double CG_ERFCX_TAB_ZLO = -8.0, CG_ERFCX_TAB_W = 1.0 / 32;
constexpr int CG_ERFCX_TAB_NI = 352, CG_ERFCX_TAB_DEG = 10;
constexpr double CG_ERFCX_TAB_ZHI = CG_ERFCX_TAB_ZLO + CG_ERFCX_TAB_NI * CG_ERFCX_TAB_W;     // 3
__device__ double cg_erfcx_tab_c[(CG_ERFCX_TAB_DEG + 1) * CG_ERFCX_TAB_NI] = {
#include "cgmath_erfcx_tab.inc"
};

__device__ __forceinline__ int cg_erfcx_tab_index(double z) {
  const double s = fmin(fmax((z - CG_ERFCX_TAB_ZLO) * (1.0 / CG_ERFCX_TAB_W), 0.0), CG_ERFCX_TAB_NI - 1.0);
  return (int)s;
}

__device__ __forceinline__ double cg_erfcx_tab_centre(int j) {
  return fma((double)j, CG_ERFCX_TAB_W, CG_ERFCX_TAB_ZLO + 0.5 * CG_ERFCX_TAB_W);      // exact
}

template <int U>
__device__ __forceinline__ void cg_erfcx_tab(const double (&z)[U], const bool (&keep)[U], double (&out)[U]) {
  double zr = z[U - 1];
#pragma unroll
  for (int u = U - 2; u >= 0; --u) zr = keep[u] ? z[u] : zr;
  const int j = cg_erfcx_tab_index(zr);
  const double cj = cg_erfcx_tab_centre(j);
  double x[U];
  bool same = true;
#pragma unroll
  for (int u = 0; u < U; ++u) {
    x[u] = z[u] - cj;
    same = same && (!keep[u] || fabs(x[u]) <= (0.5 + 0.125) * CG_ERFCX_TAB_W);
  }
  if (same) {
    const double* c = cg_erfcx_tab_c + j;
    double p[U];
    const double cd = __ldg(c);
#pragma unroll
    for (int u = 0; u < U; ++u) p[u] = cd;
#pragma unroll
    for (int k = 1; k <= CG_ERFCX_TAB_DEG; ++k) {
      const double ck = __ldg(c + k * CG_ERFCX_TAB_NI);
#pragma unroll
      for (int u = 0; u < U; ++u) p[u] = fma(p[u], x[u], ck);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) out[u] = p[u];
  } else {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int ju = cg_erfcx_tab_index(z[u]);
      const double xu = z[u] - cg_erfcx_tab_centre(ju);
      const double* c = cg_erfcx_tab_c + ju;
      double p = __ldg(c);
#pragma unroll
      for (int k = 1; k <= CG_ERFCX_TAB_DEG; ++k) p = fma(p, xu, __ldg(c + k * CG_ERFCX_TAB_NI));
      out[u] = p;
    }
  }
}

template <int U>
__device__ __forceinline__ void cg_erfc(const double (&z)[U], double (&out)[U]) {
  double x[U], t[U], inv[U], g[U], mh[U], l[U], e[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    x[u] = fmin(fabs(z[u]), 27.3);
    const double a = x[u] + 4.0, b = fma(2.0, x[u], 1.0);
    const double den = a * b;
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(den));                   // ~2^-23 relative
    double err = fma(-den, y, 1.0);
    y = fma(y, err, y);
    err = fma(-den, y, 1.0);
    y = fma(y, err, y);                                                       // 1 / ((x + 4)(1 + 2x))
    t[u] = (x[u] - 4.0) * (b * y);
    inv[u] = a * y;                                                           // 1 / (1 + 2x)
    const double h = x[u] * x[u];
    l[u] = fma(x[u], x[u], -h);                                               // x^2 = h + l exactly
    mh[u] = -h;
    g[u] = cg_erfc_c[0];
  }
#pragma unroll
  for (int k = 1; k < 27; ++k) {
#pragma unroll
    for (int u = 0; u < U; ++u) g[u] = fma(g[u], t[u], cg_erfc_c[k]);
  }
  cg_exp_neg<U>(mh, e);
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const double ee = fma(-e[u], l[u], e[u]);                                 // exp(-(h + l)) = exp(-h) (1 - l)
    const double r = ee * (g[u] * inv[u]);
    out[u] = z[u] < 0.0 ? 2.0 - r : r;
  }
}

}  // namespace cg

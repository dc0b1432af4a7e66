// Interdomain expected-kernel ("Psi") statistics of the CGPCM on sm_100a, FP64.
//
// Replaces the reference's symbolic construction (src/core/exponentiated_quadratic.py:430-559 driven
// by src/core/cgpcm.py:111-203), which materialises N x nx x nx and N x nh x nx broadcast tensors,
// by closed forms (SURVEY.md App. A) evaluated in registers and reduced over observations on the fly:
//
//   axx_sum_kernel   sum_n Axx[n] (+ its three tangents d/d(alpha,gamma,omega), forward mode, App. E):
//                    one thread per (k,l) pair of the lower triangle, a register loop over the
//                    observations of its slice, in-register Genz BVN with per-launch tables.
//   ahx_gen_kernel   A[i][n][k] = Ahx[n,i,k] for a chunk of observations, written in the [i][n][k]
//                    layout that turns every contraction into a plain GEMM (DESIGN.md §3), fused with
//                    Y[i,k] += sum_n y_n A[i,n,k]  (cgpcm.py:243).
//   ahx_dot_kernel   sum_{i,n,k} Abar[i,n,k] * dA[i,n,k]/d(alpha,gamma,omega): the adjoint of the
//                    Ahx construction (replaces tf.gradients through exp/erf).
//   ahx_user_kernel  Ahx in the reference's [n][i][k] layout (cgpcm.py:239) for parity checks/predict.
//   ahh_kernel       Ahh[i,j] and tangents; prior kernels Kh, Kx (kernel.py:43-46).
#pragma once
#include "bvn.cuh"
#include "cgmath.cuh"

namespace cg {

struct PsiConst {
  double alpha, gamma, omega, A;
  int causal;
  // causal_id (src/core/cgpcm.py:168-180,194-203): upper integration limits min(t, tx) instead of t.  The Gaussian
  // envelopes exp(E), exp(G) are the unconstrained maxima of the integrands and do not depend on the limits; only the
  // arguments of erfc / Phi_2 move, by the distance max(t - tx, 0) from the limit to t in units of the conditional
  // standard deviation:  z += max(d, 0) sqrt(A);  x_i -= max(d_i, 0) / sqrt(Sigma_11).
  int causal_id;
  double sqrtA;        // Ahx:  z(d > 0) = z_default + d sqrt(A) = ((alpha + gamma) d - gamma th) / sqrt(A)
  double isq11;        // Axx:  1 / sqrt(Sigma_11)
  double disq11[3];    // its derivatives w.r.t. alpha, gamma, omega
  // Ahx
  double pref_hx;      // causal: 0.5 sqrt(pi/A)   acausal: sqrt(pi/A)
  double e_hh, e_dd, e_hd;
  double inv_sqrtA, inv_2A;
  // Axx
  double pref_xx;      // 2 pi / sqrt(det)
  double g1, g2, p, q;
  double dhalf_logdet[3], dg1[3], dg2[3], dp[3], dq[3], drho[3];
  // Ahh
  double pref_hh;      // causal: 0.5 sqrt(pi/2B)  acausal: sqrt(pi/2B),  B = alpha + gamma
  // culling: elements whose Gaussian envelope is below exp(-cull) are exactly 0
  double cull;
  double r_xx;         // |t - tx| beyond which every Axx element of that row / column is culled
};

inline void psi_make_const(double alpha, double gamma, double omega, int causal, double cull, PsiConst* c,
                           int causal_id = 0) {
  const double PI = 3.14159265358979323846;
  double A = alpha + gamma + omega;
  c->alpha = alpha; c->gamma = gamma; c->omega = omega; c->A = A; c->causal = causal;
  c->causal_id = (causal && causal_id) ? 1 : 0;
  c->sqrtA = sqrt(A);
  c->pref_hx = (causal ? 0.5 : 1.0) * sqrt(PI / A);
  c->e_hh = ((alpha + gamma) * A - gamma * gamma) / A;
  c->e_dd = omega * (alpha + gamma) / A;
  c->e_hd = 2.0 * gamma * omega / A;
  c->inv_sqrtA = 1.0 / sqrt(A);
  c->inv_2A = 0.5 / A;
  double det = 4.0 * (A * A - gamma * gamma);
  double ddet[3] = {8.0 * A, 8.0 * A - 8.0 * gamma, 8.0 * A};
  double S11 = 2.0 * A / det, S12 = 2.0 * gamma / det;
  double dgam[3] = {0.0, 1.0, 0.0}, dom[3] = {0.0, 0.0, 1.0};
  double sq = sqrt(S11);
  c->pref_xx = 2.0 * PI / sqrt(det);
  c->g1 = omega * (1.0 - 2.0 * omega * S11);
  c->g2 = 4.0 * omega * omega * S12;
  c->p = 2.0 * omega * sq;
  c->q = 2.0 * omega * S12 / sq;
  for (int i = 0; i < 3; ++i) {
    double dS11 = 2.0 / det - 2.0 * A * ddet[i] / (det * det);
    double dS12 = 2.0 * dgam[i] / det - 2.0 * gamma * ddet[i] / (det * det);
    c->dhalf_logdet[i] = ddet[i] / (2.0 * det);
    c->dg1[i] = dom[i] * (1.0 - 2.0 * omega * S11) + omega * (-2.0 * dom[i] * S11 - 2.0 * omega * dS11);
    c->dg2[i] = 8.0 * omega * dom[i] * S12 + 4.0 * omega * omega * dS12;
    c->dp[i] = 2.0 * dom[i] * sq + omega * dS11 / sq;
    c->dq[i] = 2.0 * dom[i] * S12 / sq + 2.0 * omega * dS12 / sq - omega * S12 * dS11 / (S11 * sq);
    c->drho[i] = dgam[i] / A - gamma / (A * A);
    c->disq11[i] = -0.5 * dS11 / (S11 * sq);
  }
  c->isq11 = 1.0 / sq;
  c->pref_hh = (causal ? 0.5 : 1.0) * sqrt(PI / (2.0 * (alpha + gamma)));
  // Element-wise threshold.  With culling off it is 746: exp(E) with E < -745.14 is exactly 0 in IEEE double (below
  // half the smallest subnormal), so such elements ARE 0 -- in the reference's TF arithmetic too -- and evaluating
  // erfc / the BVN for them cannot change a single bit of any sum.  (Windows of inducing inputs / GEMM tiles are
  // only dropped when the caller asks for culling: r_xx below and plan_chunks use `cull` itself.)
  c->cull = cull > 0.0 ? cull : 746.0;
  // g1 (dk^2 + dl^2) - g2 dk dl >= (g1 - |g2| / 2) (dk^2 + dl^2)
  double lam = c->g1 - 0.5 * fabs(c->g2);
  c->r_xx = (cull > 0.0 && lam > 0.0) ? sqrt(cull / lam) : INFINITY;
}

// Elements whose Gaussian envelope is below exp(-c.cull) (default 80: < 2e-35 of an O(1) prefactor)
// are set to exactly 0 without evaluating erfc / the BVN: far below one ulp of any sum they enter.

constexpr int AXX_TILE = 16;

// part layout: [slices][4][ld][ld]; slice blockIdx.y owns observations n_lo + blockIdx.y (+ gridDim.y ...)
// of each pair's own observation range and *stores* its lower-triangle partial sums (no zero-init needed).
// When t is sorted the range of a pair is the interval of observations whose envelope is not below exp(-cull)
// (closed form + binary search); everything outside is culled anyway.
template <bool TANGENTS, bool HOIST>
__global__ void __launch_bounds__(256, HOIST ? 2 : 3) axx_sum_kernel(const double* __restrict__ t, int n_obs, int sorted,
                                                      const double* __restrict__ tx, int nx,
                                                      double* __restrict__ part, long ld, const PsiConst c,
                                                      const BvnTab T, const double* __restrict__ cheb, int deg) {
  // HOIST: dynamic shared memory = B table [(deg + 1) * 20] followed by the per-thread Chebyshev coefficients
  extern __shared__ double axx_smem[];
  double* sB = axx_smem;
  double* sA = axx_smem + (HOIST ? (deg + 1) * 20 : 0);
  if (HOIST) {
    for (int e = threadIdx.x; e < (deg + 1) * 20; e += blockDim.x) sB[e] = cheb[e];
    __syncthreads();
  }
  // Thread <-> pair (k, l = k - s): a tile is 16 inducing inputs k x 16 separations s, and a warp holds two
  // separations.  The observations with a non-zero element of a pair are an interval whose length depends on the
  // separation only (below), so the lanes of a warp run (nearly) the same number of iterations, each over its own
  // interval.  (Round 1 mapped 16 x 16 tiles of the (k, l) triangle to one common observation range per tile: ncu
  // counted 23.4 active lanes per warp instruction -- the lanes whose pair was out of range idled through a full
  // element evaluation of the others -- and the diagonal tiles ran half empty.)
  const int nt = (nx + AXX_TILE - 1) / AXX_TILE;
  const int kb = blockIdx.x / nt, sb = blockIdx.x - kb * nt;
  const int k = kb * AXX_TILE + (threadIdx.x & 15);
  const int l = k - (sb * AXX_TILE + (threadIdx.x >> 4));
  if (k >= nx || l < 0) return;
  int n_lo = 0, n_hi = n_obs;
  if (sorted) {
    // G = -g1 (dk^2 + dl^2) + g2 dk dl = -(2 g1 - g2) u^2 - (2 g1 + g2) h^2 with u = t - (tx_k + tx_l) / 2 and
    // h = (tx_k - tx_l) / 2: G >= -cull on |u| <= U.  The interval is widened by a few ulp; the element-wise test below
    // still decides, so exactly the same elements are evaluated as with any other range.
    const double a = tx[k], b = tx[l];
    const double m = 0.5 * (a + b), hh = 0.5 * (a - b);
    const double den = 2.0 * c.g1 - c.g2;
    const double num = c.cull - (2.0 * c.g1 + c.g2) * hh * hh;
    if (den > 0.0) {
      if (num < 0.0) {
        n_hi = 0;
      } else {
        const double U = sqrt(num / den) * (1.0 + 1e-12) + 1e-300;
        const double lo = m - U - 1e-12 * fabs(m), hi = m + U + 1e-12 * fabs(m);
        int x = 0, y = n_obs;                       // first n with t[n] >= lo
        while (x < y) { int mid = (x + y) >> 1; if (__ldg(t + mid) < lo) x = mid + 1; else y = mid; }
        n_lo = x;
        y = n_obs;                                  // first n with t[n] > hi
        while (x < y) { int mid = (x + y) >> 1; if (__ldg(t + mid) <= hi) x = mid + 1; else y = mid; }
        n_hi = x;
      }
    }
  }
  const double txk = tx[k], txl = tx[l];
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  // HOIST (causal, rho >= 0.925): the pair constants of the Genz high-correlation branch (bvn.cuh) -- 20 exp and a
  // 20 x (deg + 1) table product per pair, skipped when this slice of the pair has no observation (most of them on a
  // shard of a multi-GPU run)
  BvnPair R;
  if (HOIST && n_lo + (int)blockIdx.y < n_hi) bvn_pair_init((c.p - c.q) * (txk - txl), T, R, sA, sB, deg);
  for (int n = n_lo + blockIdx.y; n < n_hi; n += gridDim.y) {
    const double tn = __ldg(t + n);
    const double dk = tn - txk, dl = tn - txl;
    const double q2 = dk * dk + dl * dl, pr = dk * dl;
    const double G = -c.g1 * q2 + c.g2 * pr;
    if (G < -c.cull) continue;
    if (HOIST && TANGENTS) {
      // every transcendental of the element in lock-step (bvn_pair_all); causal by construction of HOIST
      const double x1 = c.p * dk + c.q * dl, x2 = c.q * dk + c.p * dl;
      double eg, cdf, d1, d2, dr;
      if (!bvn_pair_all(G, x1, x2, T, R, sA, deg, eg, cdf, d1, d2, dr)) {
        eg = exp(G);
        bvn_cdf_grad_tab(x1, x2, T, cdf, d1, d2, dr);
      }
      const double env = c.pref_xx * eg;
      const double V = env * cdf;
      s0 += V;
      s1 += V * (-c.dg1[0] * q2 + c.dg2[0] * pr - c.dhalf_logdet[0]) +
            env * (d1 * (c.dp[0] * dk + c.dq[0] * dl) + d2 * (c.dq[0] * dk + c.dp[0] * dl) + dr * c.drho[0]);
      s2 += V * (-c.dg1[1] * q2 + c.dg2[1] * pr - c.dhalf_logdet[1]) +
            env * (d1 * (c.dp[1] * dk + c.dq[1] * dl) + d2 * (c.dq[1] * dk + c.dp[1] * dl) + dr * c.drho[1]);
      s3 += V * (-c.dg1[2] * q2 + c.dg2[2] * pr - c.dhalf_logdet[2]) +
            env * (d1 * (c.dp[2] * dk + c.dq[2] * dl) + d2 * (c.dq[2] * dk + c.dp[2] * dl) + dr * c.drho[2]);
      continue;
    }
    const double env = c.pref_xx * exp(G);
    if (!c.causal) {
      s0 += env;
      if (TANGENTS) {
        s1 += env * (-c.dg1[0] * q2 + c.dg2[0] * pr - c.dhalf_logdet[0]);
        s2 += env * (-c.dg1[1] * q2 + c.dg2[1] * pr - c.dhalf_logdet[1]);
        s3 += env * (-c.dg1[2] * q2 + c.dg2[2] * pr - c.dhalf_logdet[2]);
      }
      continue;
    }
    double x1 = c.p * dk + c.q * dl, x2 = c.q * dk + c.p * dl;
    const double ek = (!HOIST && c.causal_id) ? fmax(dk, 0.0) : 0.0, el = (!HOIST && c.causal_id) ? fmax(dl, 0.0) : 0.0;
    if (!HOIST && c.causal_id) { x1 -= ek * c.isq11; x2 -= el * c.isq11; }
    if (!TANGENTS) {
      s0 += env * (HOIST ? bvn_cdf_pair(x1, x2, T, R, sA, deg) : bvnd_tab(-x1, -x2, T));
    } else {
      double cdf, d1, d2, dr;
      if (HOIST) {
        cdf = bvn_cdf_pair(x1, x2, T, R, sA, deg);
        bvn_partials_tab(x1, x2, T, d1, d2, dr);
      } else {
        bvn_cdf_grad_tab(x1, x2, T, cdf, d1, d2, dr);
      }
      const double V = env * cdf;
      s0 += V;
      // causal_id: x_i also carries -e_i / sqrt(Sigma_11)  (ek = el = 0 otherwise)
      s1 += V * (-c.dg1[0] * q2 + c.dg2[0] * pr - c.dhalf_logdet[0]) +
            env * (d1 * (c.dp[0] * dk + c.dq[0] * dl - ek * c.disq11[0]) +
                   d2 * (c.dq[0] * dk + c.dp[0] * dl - el * c.disq11[0]) + dr * c.drho[0]);
      s2 += V * (-c.dg1[1] * q2 + c.dg2[1] * pr - c.dhalf_logdet[1]) +
            env * (d1 * (c.dp[1] * dk + c.dq[1] * dl - ek * c.disq11[1]) +
                   d2 * (c.dq[1] * dk + c.dp[1] * dl - el * c.disq11[1]) + dr * c.drho[1]);
      s3 += V * (-c.dg1[2] * q2 + c.dg2[2] * pr - c.dhalf_logdet[2]) +
            env * (d1 * (c.dp[2] * dk + c.dq[2] * dl - ek * c.disq11[2]) +
                   d2 * (c.dq[2] * dk + c.dp[2] * dl - el * c.disq11[2]) + dr * c.drho[2]);
    }
  }
  const long mat = ld * ld;
  double* o = part + (long)blockIdx.y * 4 * mat + (long)k * ld + l;
  o[0] = s0;
  if (TANGENTS) { o[mat] = s1; o[2 * mat] = s2; o[3 * mat] = s3; }
}

// Per-observation Axx in the reference's [n][k][l] layout (parity / predict use).
__global__ void axx_user_kernel(const double* __restrict__ t, int n_obs, const double* __restrict__ tx,
                                int nx, double* __restrict__ out, const PsiConst c, const BvnTab T) {
  long total = (long)n_obs * nx * nx;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    int l = (int)(idx % nx);
    int k = (int)((idx / nx) % nx);
    int n = (int)(idx / ((long)nx * nx));
    double dk = t[n] - tx[k], dl = t[n] - tx[l];
    double G = -c.g1 * (dk * dk + dl * dl) + c.g2 * dk * dl;
    double v = 0.0;
    if (G >= -c.cull) {
      v = c.pref_xx * exp(G);
      if (c.causal) {
        double x1 = c.p * dk + c.q * dl, x2 = c.q * dk + c.p * dl;
        if (c.causal_id) { x1 -= fmax(dk, 0.0) * c.isq11; x2 -= fmax(dl, 0.0) * c.isq11; }
        v *= bvnd_tab(-x1, -x2, T);
      }
    }
    out[idx] = v;
  }
}

// Ahx[n,i,k] for U values of d = t_n - tx_k at one th (App. A.3), in lock-step (cgmath.cuh): the envelope exp(E) and the
// causal factor erfc(z).  Elements whose envelope is below exp(-c.cull) are exactly 0; `live[u] = false` forces 0 as well
// (padding).  Every caller goes through this routine, so a given (th, d) gives the same bits everywhere.
template <int U>
__device__ __forceinline__ void ahx_values(double th, const double (&d)[U], const bool (&live)[U], const PsiConst& c,
                                           double (&v)[U]) {
  const double e0 = -c.e_hh * th * th, e1 = c.e_hd * th;
  const double z0 = -(c.gamma * th) * c.inv_sqrtA, z1 = -c.omega * c.inv_sqrtA;
  double E[U], z[U], ex[U], ec[U];
  bool any = false;
#pragma unroll
  for (int u = 0; u < U; ++u) {
    E[u] = fma(d[u], fma(-c.e_dd, d[u], e1), e0);            // -e_hh th^2 - e_dd d^2 + e_hd th d
    z[u] = fma(z1, d[u], z0);                                // -(gamma th + omega d) / sqrt(A)
    if (c.causal_id) z[u] = fma(fmax(d[u], 0.0), c.sqrtA, z[u]);   // limit min(t, tx): + max(d, 0) sqrt(A)
    any = any || (live[u] && E[u] >= -c.cull);
  }
  if (!any) {                                                // e.g. 80 % of the elements when no window is cut
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = 0.0;
    return;
  }
  cg_exp_neg<U>(E, ex);
  if (c.causal) cg_erfc<U>(z, ec);
#pragma unroll
  for (int u = 0; u < U; ++u) {
    double r = c.pref_hx * ex[u];
    if (c.causal) r *= ec[u];
    v[u] = (live[u] && E[u] >= -c.cull) ? r : 0.0;
  }
}

__device__ __forceinline__ double ahx_value(double th, double d, const PsiConst& c) {
  const double dd[1] = {d};
  const bool live[1] = {true};
  double v[1];
  ahx_values<1>(th, dd, live, c, v);
  return v[0];
}

constexpr int AHX_NSUB = 16;      // observations per CTA (many short CTAs: the tail of the last wave stays small)
constexpr int AHX_U = 4;          // observations a thread evaluates in lock-step

// A[(i*nc + n)*kwp + k] for i < nhp, n < nc, k < kwp (zero outside the valid nh x n_valid x nx box).
// Ypart[blockIdx.y][i][k_lo + k] += sum_n y_n A   (slice-private accumulation, reduced later).
__global__ void __launch_bounds__(256) ahx_gen_kernel(const double* __restrict__ t, const double* __restrict__ y,
                                                      int n_valid, int nc, const double* __restrict__ th, int nh,
                                                      const double* __restrict__ tx, int nx, int k_lo, int kwp,
                                                      double* __restrict__ A, double* __restrict__ Ypart,
                                                      long ldy, long ypart_stride, const PsiConst c) {
  const int i = blockIdx.x;
  const int n0 = blockIdx.y * AHX_NSUB;
  const int n1 = min(nc, n0 + AHX_NSUB);
  const bool row_ok = i < nh;
  const double thi = row_ok ? th[i] : 0.0;
  for (int k = threadIdx.x; k < kwp; k += blockDim.x) {
    const int kg = k_lo + k;
    const bool ok = row_ok && kg < nx;
    const double txk = ok ? tx[kg] : 0.0;
    double ysum = 0.0;
    double* dst = A + ((long)i * nc + n0) * kwp + k;
    for (int n = n0; n < n1; n += AHX_U, dst += (long)AHX_U * kwp) {
      double d[AHX_U], yv[AHX_U], v[AHX_U];
      bool live[AHX_U];
#pragma unroll
      for (int u = 0; u < AHX_U; ++u) {
        live[u] = ok && n + u < n_valid;
        d[u] = live[u] ? __ldg(t + n + u) - txk : 0.0;
        yv[u] = live[u] ? __ldg(y + n + u) : 0.0;
      }
      ahx_values<AHX_U>(thi, d, live, c, v);
#pragma unroll
      for (int u = 0; u < AHX_U; ++u) {
        ysum += yv[u] * v[u];                                // observations in increasing order, as before
        if (n + u < n1) dst[(long)u * kwp] = v[u];
      }
    }
    if (ok && Ypart) Ypart[(long)blockIdx.y * ypart_stride + (long)i * ldy + kg] += ysum;
  }
}

// ---- separable variants (default causal model, causal_id = false) -----------------------------------------------
// Ahx[n,i,k] = pref exp(E) erfc(z) with E = c + z^2 and c = -(alpha + gamma) th_i^2 - omega d_nk^2: the Gaussian factor
// of erfc(z) = exp(-z^2) erfcx(z) cancels the cross term of the envelope, and exp(c) = f_i g_nk with
//   f_i = exp(-(alpha + gamma) th_i^2)   (one per filter inducing point),   g_nk = exp(-omega d_nk^2)   (one per (n, k)).
// So   Ahx = pref f_i g_nk erfcx(z)   for either sign of z, and the Gaussian factor exp(E - z^2) of the erfc derivative in
// the adjoint is f_i g_nk itself.  A CTA covers AHX_IB filter rows of the same (n, k) block, so g_nk costs one exp per
// AHX_IB elements.  Padding (k >= nx, n >= n_valid) is expressed as d = 1e160, whose envelope is exactly 0.
//
// ahx_gen_sep_kernel<true> (the launch checks that every element with E >= -cull has z in the range of cg_erfcx_tab,
// psi_erfcx_tab_covers): one table-driven erfcx per element and no other transcendental.  f_i g_nk alone underflows
// where z^2 is large: an element with E >= -cull has ln(f_i g_nk) = E - z^2 >= -cull - z^2, down to -810 at cull 746
// and z = -8.  So f_i and g_nk are carried as f_i 2^480 and g_nk 2^480 (cg_exp_neg with BIAS: the same significands),
// which are normal down to e^-1040 each (the launch also checks cull + z^2 <= 1040), their product is at most
// pref 2^960, and the element is ((pref f_i 2^480) (g_nk 2^480)) erfcx(z) 2^-960: the same three roundings as the
// unscaled product, and the last scaling is exact unless the element is subnormal.
// ahx_gen_sep_kernel<false> (z outside the table): z >= 0: pref f_i g_nk erfcx(z); z < 0: pref (2 exp(E) -
// f_i g_nk erfcx(-z)), with erfcx(|z|) from cg_erfcx_abs and one exp(E) per element.
constexpr int AHX_IB = 8;
constexpr int AHX_US = 4;         // observations ahx_gen_sep_kernel evaluates in lock-step (8: 143 registers, 0.9 ms slower)
constexpr double AHX_FAR = 1e160;
constexpr int AHX_BIAS = 480;     // f_i and g_nk scaled by 2^AHX_BIAS each in ahx_gen_sep_kernel<true>

static_assert(2 * AHX_BIAS == 960, "ahx_gen_sep_kernel<true> scales by 2^-960");

struct AhxRow { double th, e0, e1, z0, pf, fx, pfs; };   // pf = pref f_i, fx = f_i / sqrt(A), pfs = pref f_i 2^AHX_BIAS

__device__ __forceinline__ void ahx_row_init(AhxRow* rows, int i0, const double* __restrict__ th, int nh, const PsiConst& c) {
  if (threadIdx.x < AHX_IB) {
    const int i = i0 + threadIdx.x;
    const double thi = i < nh ? th[i] : 0.0;
    AhxRow r;
    r.th = thi;
    r.e0 = -c.e_hh * thi * thi;
    r.e1 = c.e_hd * thi;
    r.z0 = -(c.gamma * thi) * c.inv_sqrtA;
    const double f = exp(-(c.alpha + c.gamma) * thi * thi);
    r.pf = c.pref_hx * f;
    r.fx = f * c.inv_sqrtA;
    const double lf[1] = {-(c.alpha + c.gamma) * thi * thi};
    double fs[1];
    cg_exp_neg<1, true, AHX_BIAS>(lf, fs);
    r.pfs = c.pref_hx * fs[0];
    rows[threadIdx.x] = r;
  }
  __syncthreads();
}

// z range of the elements with E >= -cull over filter inducing inputs th in [th_lo, th_hi] (host): for a fixed th those
// elements are an interval of d around e_hd th / (2 e_dd), and z is linear in d, so the largest z is a concave and the
// smallest a convex function of th on the th where the interval is not empty; golden-section search finds both.  The
// interval is taken at cull + 1 (covers the rounding of E in the kernel).  True when cg_erfcx_tab covers the range and
// the scaled factors of ahx_gen_sep_kernel<true> stay normal.
inline bool psi_erfcx_tab_covers(const PsiConst& c, double th_lo, double th_hi) {
  if (!c.causal || c.causal_id || !(th_lo <= th_hi)) return false;
  const double cl = c.cull + 1.0;
  const double k = c.e_hd / (2.0 * c.e_dd), m = c.e_hh - c.e_hd * k / 2.0;   // E = -e_dd (d - k th)^2 - m th^2
  if (!(m > 0.0) || !(c.e_dd > 0.0)) return false;
  const double tmax = sqrt(cl / m);                      // |th| beyond which no element is live
  const double lo = fmax(th_lo, -tmax), hi = fmin(th_hi, tmax);
  if (lo > hi) return true;                              // every element is culled
  auto zext = [&](double t, double sgn) {                // sgn * z at the end of the live d interval that maximises it
    const double r = sqrt(fmax(cl - m * t * t, 0.0) / c.e_dd);
    const double d = k * t - sgn * r;
    return sgn * (-(c.gamma * t + c.omega * d) * c.inv_sqrtA);
  };
  double zr[2];
  for (int s = 0; s < 2; ++s) {
    const double sgn = s ? -1.0 : 1.0, g = 0.6180339887498949;
    double a = lo, b = hi;
    for (int it = 0; it < 200 && b - a > 1e-15 * (fabs(a) + fabs(b)); ++it) {
      const double x1 = b - g * (b - a), x2 = a + g * (b - a);
      if (zext(x1, sgn) < zext(x2, sgn)) a = x1; else b = x2;
    }
    zr[s] = sgn * fmax(fmax(zext(a, sgn), zext(lo, sgn)), zext(hi, sgn));
  }
  const double zmax = zr[0], zmin = zr[1];
  return zmin >= CG_ERFCX_TAB_ZLO && zmax <= CG_ERFCX_TAB_ZHI &&
         c.cull + fmax(zmin * zmin, zmax * zmax) <= 1040.0;
}

template <bool TAB>
__global__ void __launch_bounds__(256) ahx_gen_sep_kernel(const double* __restrict__ t, const double* __restrict__ y,
                                                          int n_valid, int nc, const double* __restrict__ th, int nh, int nhp,
                                                          const double* __restrict__ tx, int nx, int k_lo, int kwp,
                                                          double* __restrict__ A, double* __restrict__ Ypart,
                                                          long ldy, long ypart_stride, const PsiConst c) {
  __shared__ AhxRow rows[AHX_IB];
  __shared__ double ys[AHX_IB][256];
  const int i0 = blockIdx.x * AHX_IB;
  const int n0 = blockIdx.y * AHX_NSUB;
  const int n1 = min(nc, n0 + AHX_NSUB);
  ahx_row_init(rows, i0, th, nh, c);
  const int ib = min(AHX_IB, nhp - i0);
  const double p2 = 2.0 * c.pref_hx, z1 = -c.omega * c.inv_sqrtA;
  for (int k = threadIdx.x; k < kwp; k += blockDim.x) {
    const int kg = k_lo + k;
    const bool kok = kg < nx;
    const double txk = kok ? tx[kg] : 0.0;
#pragma unroll
    for (int ii = 0; ii < AHX_IB; ++ii) ys[ii][threadIdx.x] = 0.0;
    for (int n = n0; n < n1; n += AHX_US) {
      double d[AHX_US], yv[AHX_US], w2[AHX_US], gk[AHX_US];
#pragma unroll
      for (int u = 0; u < AHX_US; ++u) {
        const bool live = kok && n + u < n_valid;
        d[u] = live ? __ldg(t + n + u) - txk : AHX_FAR;
        yv[u] = live ? __ldg(y + n + u) : 0.0;
        w2[u] = -c.omega * d[u] * d[u];
      }
      if (TAB) cg_exp_neg<AHX_US, true, AHX_BIAS>(w2, gk);
      else cg_exp_neg<AHX_US, true>(w2, gk);
      double* dst = A + ((long)i0 * nc + n) * kwp + k;
#pragma unroll 1
      for (int ii = 0; ii < ib; ++ii, dst += (long)nc * kwp) {
        const AhxRow r = rows[ii];
        double E[AHX_US], z[AHX_US], ex[AHX_US], q[AHX_US];
        bool any = false;
#pragma unroll
        for (int u = 0; u < AHX_US; ++u) {
          E[u] = fma(d[u], fma(-c.e_dd, d[u], r.e1), r.e0);
          z[u] = fma(z1, d[u], r.z0);
          any = any || E[u] >= -c.cull;
        }
        double ysum = 0.0;
        if (TAB && any && i0 + ii < nh) {
          bool keep[AHX_US];
#pragma unroll
          for (int u = 0; u < AHX_US; ++u) keep[u] = E[u] >= -c.cull;
          cg_erfcx_tab<AHX_US>(z, keep, q);
#pragma unroll
          for (int u = 0; u < AHX_US; ++u) {
            const double v = keep[u] ? ((r.pfs * gk[u]) * q[u]) * 0x1p-960 : 0.0;     // 2^-(2 AHX_BIAS)
            ysum = fma(yv[u], v, ysum);
            if (n + u < n1) dst[(long)u * kwp] = v;
          }
          ys[ii][threadIdx.x] += ysum;
        } else if (!TAB && any && i0 + ii < nh) {
          cg_exp_neg<AHX_US, true>(E, ex);
          cg_erfcx_abs<AHX_US>(z, q);
#pragma unroll
          for (int u = 0; u < AHX_US; ++u) {
            const double rr = (r.pf * gk[u]) * q[u];
            double v = z[u] < 0.0 ? fma(p2, ex[u], -rr) : rr;
            v = E[u] >= -c.cull ? v : 0.0;
            ysum = fma(yv[u], v, ysum);
            if (n + u < n1) dst[(long)u * kwp] = v;
          }
          ys[ii][threadIdx.x] += ysum;
        } else {
#pragma unroll
          for (int u = 0; u < AHX_US; ++u)
            if (n + u < n1) dst[(long)u * kwp] = 0.0;
        }
      }
    }
    if (kok && Ypart) {
      for (int ii = 0; ii < ib; ++ii)
        if (i0 + ii < nh) Ypart[(long)blockIdx.y * ypart_stride + (long)(i0 + ii) * ldy + kg] += ys[ii][threadIdx.x];
    }
  }
}

// gpart[(blockIdx.y * gridDim.x + blockIdx.x) * 3 + theta] += the block's part of sum (W + y Ybar) dA/dtheta (see ahx_dot_kernel)
__global__ void __launch_bounds__(256) ahx_dot_sep_kernel(const double* __restrict__ t, const double* __restrict__ y,
                                                          int n_valid, int nc, const double* __restrict__ th, int nh,
                                                          const double* __restrict__ tx, int nx, int k_lo, int kwp,
                                                          const double* __restrict__ A, const double* __restrict__ W,
                                                          const double* __restrict__ Ybar, long ldy,
                                                          double* __restrict__ gpart, const PsiConst c) {
  __shared__ AhxRow rows[AHX_IB];
  const int i0 = blockIdx.x * AHX_IB;
  const int n0 = blockIdx.y * AHX_NSUB;
  const int n1 = min(n_valid, n0 + AHX_NSUB);
  ahx_row_init(rows, i0, th, nh, c);
  const int ib = min(AHX_IB, nh - i0);
  const double inv_A = 2.0 * c.inv_2A;
  double g0 = 0.0, g1 = 0.0, g2 = 0.0;
  for (int k = threadIdx.x; k < kwp; k += blockDim.x) {
    const int kg = k_lo + k;
    if (kg >= nx) continue;
    const double txk = tx[kg];
    for (int nb = n0; nb < n1; nb += 4) {
      double d[4], yv[4], w2[4], gk[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const bool ok = nb + u < n1;
        d[u] = ok ? __ldg(t + nb + u) - txk : 0.0;            // padding: W = y = 0, every factor stays finite
        yv[u] = ok ? __ldg(y + nb + u) : 0.0;
        w2[u] = -c.omega * d[u] * d[u];
      }
      cg_exp_neg<4, true>(w2, gk);
      const long off = ((long)i0 * nc + nb) * kwp + k;
      const double* src = W + off;
      const double* asrc = A + off;
#pragma unroll 4
      for (int ii = 0; ii < ib; ++ii, src += (long)nc * kwp, asrc += (long)nc * kwp) {
        const AhxRow r = rows[ii];
        double wv[4], av[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool ok = nb + u < n1;
          wv[u] = ok ? src[(long)u * kwp] : 0.0;
          av[u] = ok ? asrc[(long)u * kwp] : 0.0;
        }
        const double yb = Ybar[(long)(i0 + ii) * ldy + kg];
        const double xf = r.fx;                                  // f_i / sqrt(A)
        const double ca = -fma(r.th, r.th, c.inv_2A);            // -th^2 - 1/(2A)
        const double gth = c.gamma * r.th, tis = r.th * c.inv_sqrtA;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const double E = fma(d[u], fma(-c.e_dd, d[u], r.e1), r.e0);
          const double w = E >= -c.cull ? fma(yv[u], yb, wv[u]) : 0.0;
          const double bh = -fma(c.omega, d[u], gth);            // b / 2 = -(gamma th + omega d)
          const double uu = bh * inv_A;                          // b / (2A)
          const double zc = (bh * c.inv_sqrtA) * c.inv_2A;       // z / (2A)
          const double F = av[u];
          const double X = xf * gk[u];                           // exp(E - z^2) / sqrt(A)
          const double su = r.th + uu, sd = d[u] + uu;
          const double da = fma(F, fma(-uu, uu, ca), X * zc);
          const double dg = fma(F, -fma(su, su, c.inv_2A), X * (tis + zc));
          const double dw = fma(F, -fma(sd, sd, c.inv_2A), X * fma(d[u], c.inv_sqrtA, zc));
          g0 = fma(w, da, g0); g1 = fma(w, dg, g1); g2 = fma(w, dw, g2);
        }
      }
    }
  }
  __shared__ double sh[3][8];
  for (int off = 16; off > 0; off >>= 1) {
    g0 += __shfl_down_sync(0xffffffffu, g0, off);
    g1 += __shfl_down_sync(0xffffffffu, g1, off);
    g2 += __shfl_down_sync(0xffffffffu, g2, off);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sh[0][warp] = g0; sh[1][warp] = g1; sh[2][warp] = g2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    double a0 = 0, a1 = 0, a2 = 0;
    for (int w = 0; w < nw; ++w) { a0 += sh[0][w]; a1 += sh[1][w]; a2 += sh[2][w]; }
    double* o = gpart + ((long)blockIdx.y * gridDim.x + blockIdx.x) * 3;
    o[0] += a0; o[1] += a1; o[2] += a2;
  }
}

// gpart[(blockIdx.y * gridDim.x + blockIdx.x) * 3 + theta] += sum over the block's elements of
//   (W[i][n][k] + y_n * Ybar[i][k_lo + k]) * dA[i,n,k]/dtheta,   A = the chunk's Ahx block (ahx_gen_kernel).
__global__ void __launch_bounds__(256) ahx_dot_kernel(const double* __restrict__ t, const double* __restrict__ y,
                                                      int n_valid, int nc, const double* __restrict__ th, int nh,
                                                      const double* __restrict__ tx, int nx, int k_lo, int kwp,
                                                      const double* __restrict__ A, const double* __restrict__ W,
                                                      const double* __restrict__ Ybar, long ldy,
                                                      double* __restrict__ gpart, const PsiConst c) {
  const int i = blockIdx.x;
  const int n0 = blockIdx.y * AHX_NSUB;
  const int n1 = min(n_valid, n0 + AHX_NSUB);
  double g0 = 0.0, g1 = 0.0, g2 = 0.0;
  if (i < nh) {
    const double thi = th[i];
    for (int k = threadIdx.x; k < kwp; k += blockDim.x) {
      const int kg = k_lo + k;
      if (kg >= nx) continue;
      const double txk = tx[kg];
      const double yb = Ybar[(long)i * ldy + kg];
      const long off = ((long)i * nc + n0) * kwp + k;
      const double* src = W + off;
      const double* asrc = A + off;
      // four observations per step: all eight loads are issued before the first exp() so that enough bytes
      // are in flight per SM (the kernel streams 16 B per element and is latency-bound otherwise)
      for (int nb = n0; nb < n1; nb += 4) {
        double wv[4], av[4], tv[4], yv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool ok = nb + u < n1;
          wv[u] = ok ? src[(long)u * kwp] : 0.0;
          av[u] = ok ? asrc[(long)u * kwp] : 0.0;
          tv[u] = ok ? __ldg(t + nb + u) : 0.0;
          yv[u] = ok ? __ldg(y + nb + u) : 0.0;
        }
        src += 4L * kwp;
        asrc += 4L * kwp;
        // F = Ahx[n,i,k] itself is still in the chunk's block (same bits as the forward value); only the Gaussian
        // factor exp(E - z^2) of the erfc derivative is evaluated here, four observations in lock-step (cgmath.cuh)
        double Ev[4], zv[4], ga[4], gx[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const double d = tv[u] - txk;
          Ev[u] = -c.e_hh * thi * thi - c.e_dd * d * d + c.e_hd * thi * d;
          zv[u] = -(c.gamma * thi + c.omega * d) * c.inv_sqrtA;
          if (c.causal_id) zv[u] = fma(fmax(d, 0.0), c.sqrtA, zv[u]);
          ga[u] = Ev[u] - zv[u] * zv[u];
        }
        if (c.causal) cg_exp_neg<4>(ga, gx);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (nb + u >= n1) break;
          const double d = tv[u] - txk;
          const double E = Ev[u];
          if (E < -c.cull) continue;
          const double w = wv[u] + yv[u] * yb;
          const double bh = -(c.gamma * thi + c.omega * d);    // b / 2
          const double uu = bh * 2.0 * c.inv_2A;               // b / (2A)
          const double z = zv[u];
          const double F = av[u];
          const double X = c.causal ? gx[u] * c.inv_sqrtA : 0.0;
          const double zc = z * c.inv_2A;
          // -X z_theta:  default z = -(gamma th + omega d) / sqrt(A);  causal_id, d > 0: z = ((alpha + gamma) d - gamma th) / sqrt(A)
          const bool idr = c.causal_id && d > 0.0;
          const double da = F * (-thi * thi - uu * uu - c.inv_2A) + X * ((idr ? -d * c.inv_sqrtA : 0.0) + zc);
          const double dg = F * (-(thi + uu) * (thi + uu) - c.inv_2A) + X * ((idr ? thi - d : thi) * c.inv_sqrtA + zc);
          const double dw = F * (-(d + uu) * (d + uu) - c.inv_2A) + X * ((idr ? 0.0 : d * c.inv_sqrtA) + zc);
          g0 += w * da; g1 += w * dg; g2 += w * dw;
        }
      }
    }
  }
  // block reduction (deterministic)
  __shared__ double sh[3][8];
  for (int off = 16; off > 0; off >>= 1) {
    g0 += __shfl_down_sync(0xffffffffu, g0, off);
    g1 += __shfl_down_sync(0xffffffffu, g1, off);
    g2 += __shfl_down_sync(0xffffffffu, g2, off);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sh[0][warp] = g0; sh[1][warp] = g1; sh[2][warp] = g2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    double a0 = 0, a1 = 0, a2 = 0;
    for (int w = 0; w < nw; ++w) { a0 += sh[0][w]; a1 += sh[1][w]; a2 += sh[2][w]; }
    double* o = gpart + ((long)blockIdx.y * gridDim.x + blockIdx.x) * 3;
    o[0] += a0; o[1] += a1; o[2] += a2;
  }
}

__global__ void ahx_user_kernel(const double* __restrict__ t, int n_obs, const double* __restrict__ th, int nh,
                                const double* __restrict__ tx, int nx, double* __restrict__ out, const PsiConst c) {
  long total = (long)n_obs * nh * nx;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    int k = (int)(idx % nx);
    int i = (int)((idx / nx) % nh);
    int n = (int)(idx / ((long)nx * nh));
    out[idx] = ahx_value(th[i], t[n] - tx[k], c);
  }
}

// Prior kernels and Ahh on padded ld x ld storage (zero padding).
// Kh0 = exp(-alpha (ti^2 + tj^2) - gamma (ti - tj)^2); Kx0 = sqrt(pi/2omega) exp(-omega/2 (tk - tl)^2).
__global__ void prior_kernels_kernel(const double* __restrict__ th, int nh, long ldh, const double* __restrict__ tx,
                                     int nx, long ldx, double reg, double* __restrict__ Kh0, double* __restrict__ Kh,
                                     double* __restrict__ Kx0, double* __restrict__ Kx, double* __restrict__ Ahh,
                                     double* __restrict__ dAhh_a, double* __restrict__ dAhh_g, const PsiConst c,
                                     const int pw_dists) {
  // pw_dists = 1: squared distances as the reference forms them, |x|^2 - 2 x y + |y|^2 (pw_dists2,
  // src/core/tf_util.py:24-31, used by DEQ._call, src/core/kernel.py:43-46), operation by operation and without FMA
  // contraction; default: (x - y)^2, the value that expression approximates (it loses ~eps x^2 gamma: 1e-7 relative at
  // the crude-oil time stamps t ~ 2010).
  const long nh2 = ldh * ldh, nx2 = ldx * ldx;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < nh2 + nx2; idx += (long)gridDim.x * blockDim.x) {
    if (idx < nh2) {
      int i = (int)(idx / ldh), j = (int)(idx % ldh);
      double k0 = 0.0, ahh = 0.0, da = 0.0, dg = 0.0;
      if (i < nh && j < nh) {
        double ti = th[i], tj = th[j];
        double q2 = ti * ti + tj * tj, s = ti + tj;
        if (pw_dists) {
          const double n2x = __dmul_rn(ti, ti), n2y = __dmul_rn(tj, tj);
          const double d2 = __dadd_rn(__dsub_rn(n2x, __dmul_rn(2.0, __dmul_rn(ti, tj))), n2y);
          k0 = exp(__dsub_rn(__dmul_rn(-c.alpha, __dadd_rn(n2x, n2y)), __dmul_rn(c.gamma, d2)));
        } else {
          k0 = exp(-c.alpha * q2 - c.gamma * (ti - tj) * (ti - tj));
        }
        // Ahh: D = 2B, b = -2 gamma s, cc = -B q2, E = cc + b^2/(4D), z = b / (2 sqrt D)
        double B = c.alpha + c.gamma, D = 2.0 * B;
        double b = -2.0 * c.gamma * s;
        double E = -B * q2 + b * b / (4.0 * D);
        double isd = 1.0 / sqrt(D);
        double z = 0.5 * b * isd;
        double u = b / (2.0 * D);
        double eE = exp(E);
        double F, X;
        if (c.causal) { F = c.pref_hh * eE * erfc(z); X = exp(E - z * z) * isd; }
        else { F = c.pref_hh * eE; X = 0.0; }
        ahh = F;
        // tangents: D_theta = 2; alpha: b_t = 0, c_t = -q2 ; gamma: b_t = -2 s, c_t = -q2
        double Ea = -q2 - 2.0 * u * u, Eg = -q2 - 2.0 * u * s - 2.0 * u * u;
        double za = -z / D, zg = -s * isd - z / D;
        da = F * (Ea - 1.0 / D) - X * za;
        dg = F * (Eg - 1.0 / D) - X * zg;
      }
      Kh0[idx] = k0;
      Kh[idx] = k0 + ((i == j && i < nh) ? reg : 0.0);
      Ahh[idx] = ahh;
      dAhh_a[idx] = da;
      dAhh_g[idx] = dg;
    } else {
      long id2 = idx - nh2;
      int k = (int)(id2 / ldx), l = (int)(id2 % ldx);
      double k0 = 0.0;
      if (k < nx && l < nx) {
        double d = tx[k] - tx[l];
        double d2 = d * d;
        if (pw_dists) {
          const double xk = tx[k], xl = tx[l];
          d2 = __dadd_rn(__dsub_rn(__dmul_rn(xk, xk), __dmul_rn(2.0, __dmul_rn(xk, xl))), __dmul_rn(xl, xl));
        }
        k0 = sqrt(1.5707963267948966 / c.omega) * exp(-(0.5 * c.omega) * d2);
      }
      Kx0[id2] = k0;
      Kx[id2] = k0 + ((k == l && k < nx) ? reg : 0.0);
    }
  }
}

}  // namespace cg

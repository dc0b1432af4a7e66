// Test-side kernels of VCGPCM.predict_f (src/core/cgpcm.py:781-846): per test input t*_n the reference builds
// Ahx*_n (nh x nx), Axx*_n (nx x nx) and, per filter sample h,
//     mu_n = sqrt(s2_f) h^T Ahx*_n x_mean
//     m2_n = s2_f (a + <Ahh, mh> + <Axx*_n, mx> + tr((mh Ahx*_n) o (Ahx*_n mx))),   mh = h h^T - iKh,  mx = x_m2 - iKx
// Here the sample-independent part of the last term is folded into the per-point matrix
//     Bxx*_n = Axx*_n - Ahx*_n^T iKh Ahx*_n        (the reference's mats['Bxx'], cgpcm.py:249-251)
// so that per sample and point only  v = Ahx*_n^T h,  v^T mx v  and  <Bxx*_n, mx>  remain:
//     m2_n = s2_f (a + h^T Ahh h - tr(Ahh iKh) + <Bxx*_n, mx> + v^T mx v).
#pragma once
#include <cfloat>
#include <cuda_runtime.h>

#include "dgemm_dmma.cuh"
#include "psi_kernels.cuh"

namespace cg {

// X[n][k][l] -= sum_i A[i][n][k] * T[i][n][l]   (A, T in the chunk layout [i][n][kw], X dense [n][nx][nx]).
// grid (tiles_l, tiles_k, n), block 16 x 16, each thread a 2 x 2 patch of a 32 x 32 tile.
__global__ void __launch_bounds__(256) bxx_star_kernel(const double* __restrict__ A, const double* __restrict__ T, int nh,
                                                      int nc, int kw, int nx, double* __restrict__ X) {
  __shared__ double sa[8][32], st[8][32];
  const int n = blockIdx.z;
  const int k0 = blockIdx.y * 32, l0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  double acc[2][2] = {{0, 0}, {0, 0}};
  for (int i0 = 0; i0 < nh; i0 += 8) {
    {
      const int r = threadIdx.x >> 5, c = threadIdx.x & 31;     // 8 rows (i) x 32 columns
      const int i = i0 + r;
      const long base = ((long)i * nc + n) * kw;
      sa[r][c] = (i < nh && k0 + c < nx) ? A[base + k0 + c] : 0.0;
      st[r][c] = (i < nh && l0 + c < nx) ? T[base + l0 + c] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const double a0 = sa[r][ty * 2], a1 = sa[r][ty * 2 + 1];
      const double t0 = st[r][tx * 2], t1 = st[r][tx * 2 + 1];
      acc[0][0] += a0 * t0; acc[0][1] += a0 * t1;
      acc[1][0] += a1 * t0; acc[1][1] += a1 * t1;
    }
    __syncthreads();
  }
#pragma unroll
  for (int u = 0; u < 2; ++u)
#pragma unroll
    for (int v = 0; v < 2; ++v) {
      const int k = k0 + ty * 2 + u, l = l0 + tx * 2 + v;
      if (k < nx && l < nx) X[((long)n * nx + k) * nx + l] -= acc[u][v];
    }
}

// One CTA per test point: accumulates this sample's mean and variance contribution (weight w = 1 / #samples).
//   A: chunk layout [i][n][kw];  hvec[nh];  xm[nx];  mx: nx x nx with leading dimension ld;  B: Bxx* dense [n][nx][nx]
//   q1 = a + h^T Ahh h - tr(Ahh iKh)
__global__ void __launch_bounds__(256) predict_point_kernel(const double* __restrict__ A, int nh, int nc, int kw, int nx,
                                                           const double* __restrict__ hvec, const double* __restrict__ xm,
                                                           const double* __restrict__ mx, long ld,
                                                           const double* __restrict__ B, const double* __restrict__ q1,
                                                           double sqrt_s2f, double s2f, double w,
                                                           double* __restrict__ acc_mu, double* __restrict__ acc_var) {
  extern __shared__ double pv[];          // v[nx]
  __shared__ double red[3][8];
  const int n = blockIdx.x;
  for (int k = threadIdx.x; k < nx; k += blockDim.x) {
    double s = 0.0;
    for (int i = 0; i < nh; ++i) s += hvec[i] * A[((long)i * nc + n) * kw + k];
    pv[k] = s;
  }
  __syncthreads();
  double mu = 0.0, qv = 0.0, qb = 0.0;
  for (int k = threadIdx.x; k < nx; k += blockDim.x) mu += pv[k] * xm[k];
  const double* Bn = B + (long)n * nx * nx;
  for (long e = threadIdx.x; e < (long)nx * nx; e += blockDim.x) {
    const int k = (int)(e / nx), l = (int)(e - (long)k * nx);
    const double m = mx[(long)k * ld + l];
    qv += pv[k] * m * pv[l];
    qb += Bn[e] * m;
  }
  for (int off = 16; off > 0; off >>= 1) {
    mu += __shfl_down_sync(0xffffffffu, mu, off);
    qv += __shfl_down_sync(0xffffffffu, qv, off);
    qb += __shfl_down_sync(0xffffffffu, qb, off);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][warp] = mu; red[1][warp] = qv; red[2][warp] = qb; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a0 = 0, a1 = 0, a2 = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a0 += red[0][i]; a1 += red[1][i]; a2 += red[2][i]; }
    const double m1 = sqrt_s2f * a0;
    const double m2 = s2f * (q1[0] + a2 + a1);
    acc_mu[n] += w * m1;
    acc_var[n] += w * (m2 - m1 * m1);
  }
}

// ---- Batched prediction (cgpcm_predict_f_batch): the test side for a batch of samples per launch.  Per chunk of test
// points, with V_b = H_B A* (one row v_nb = A*_n^T h_b per point, from the small-left GEMM):
//     Qb[n][b]   = <Bxx*_n, mx_b>            (predict_qb_kernel: points x samples x nx^2, Bxx* read once per batch)
//     quad[n][b] = v_nb^T mx_b v_nb,  lin[n][b] = v_nb . xm_b      (predict_quad_kernel)
//     mean_nb = sqrt(s2_f) lin,  var_nb = s2_f (q1_b + Qb + quad) - mean_nb^2      (predict_finish_kernel)
// Launch shapes are functions of the chunk and the internal batch size only, and every sum over k runs in an order
// fixed by nx, so a sample's moments are bitwise the same in any batch and at any position.
constexpr int PQ_T = 32;                 // rows (points) and columns of an output tile
constexpr int PQ_BK = 32;                // k per shared-memory stage
constexpr int PQ_LDS = PQ_BK + 4;        // == 4 (mod 8): conflict-free fragment loads
constexpr int PQ_SLICES = 8;             // fixed k slices of the Qb contraction (partials summed in order)

struct PredQbArgs {
  const double* X;      // Bxx*_n(k, l) at X[n * K + k * nx + l]  (K = nx^2)
  const double* mx;     // mx_b(k, l) at mx[b * mx_stride + k * nx + l]
  long mx_stride;
  long K;
  int nv, ncol;         // points of the chunk, valid sample columns
  double* q;            // partials: slice z at q[(z * nrow + n) * ldq + b]
  int nrow, ldq;
};

// grid (point tiles, sample tiles, PQ_SLICES), 128 threads: 4 warps own the 16 x 16 quadrants of a 32 x 32 tile
// (2 x 2 DMMA m8n8k4 tiles each).  Slice z contracts k-tiles [z per, (z + 1) per) in order.
__global__ void __launch_bounds__(128) predict_qb_kernel(const PredQbArgs g) {
  __shared__ __align__(16) double As[PQ_T * PQ_LDS];
  __shared__ __align__(16) double Bs[PQ_T * PQ_LDS];
  const int r0 = blockIdx.x * PQ_T, s0 = blockIdx.y * PQ_T, z = blockIdx.z;
  const long kt = (g.K + PQ_BK - 1) / PQ_BK, per = (kt + PQ_SLICES - 1) / PQ_SLICES;
  const long k_begin = z * per * PQ_BK, k_end = min(g.K, (z + 1) * per * PQ_BK);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wi = warp >> 1, wj = warp & 1, grp = lane >> 2, tig = lane & 3;
  double acc[2][2][2];
#pragma unroll
  for (int x = 0; x < 2; ++x)
#pragma unroll
    for (int y = 0; y < 2; ++y) acc[x][y][0] = acc[x][y][1] = 0.0;
  for (long k0 = k_begin; k0 < k_end; k0 += PQ_BK) {
#pragma unroll
    for (int q = 0; q < PQ_T * PQ_BK / 128; ++q) {
      const int e = q * 128 + tid, rr = e >> 5, cc = e & 31;
      const long k = k0 + cc;
      const bool kok = k < k_end;
      As[rr * PQ_LDS + cc] = (kok && r0 + rr < g.nv) ? g.X[(long)(r0 + rr) * g.K + k] : 0.0;
      Bs[rr * PQ_LDS + cc] = (kok && s0 + rr < g.ncol) ? g.mx[(long)(s0 + rr) * g.mx_stride + k] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k4 = 0; k4 < PQ_BK / 4; ++k4) {
      double fa[2], fb[2];
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        fa[x] = As[(wi * 16 + x * 8 + grp) * PQ_LDS + k4 * 4 + tig];
        fb[x] = Bs[(wj * 16 + x * 8 + grp) * PQ_LDS + k4 * 4 + tig];
      }
#pragma unroll
      for (int x = 0; x < 2; ++x)
#pragma unroll
        for (int y = 0; y < 2; ++y) dmma_8x8x4(acc[x][y][0], acc[x][y][1], fa[x], fb[y]);
    }
    __syncthreads();
  }
  double* Q = g.q + (long)z * g.nrow * g.ldq;
#pragma unroll
  for (int x = 0; x < 2; ++x) {
    const int row = r0 + wi * 16 + x * 8 + grp;
    if (row >= g.nv) continue;
#pragma unroll
    for (int y = 0; y < 2; ++y)
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int col = s0 + wj * 16 + y * 8 + tig * 2 + u;
        if (col < g.ncol) Q[(long)row * g.ldq + col] = acc[x][y][u];
      }
  }
}

struct PredQuadArgs {
  const double* V;      // v_nb(k) at V[b * v_stride + n * ldv + k]
  long v_stride;
  int ldv;
  const double* mx;     // mx_b(k, l) at mx[b * mx_stride + k * nx + l]  (stride 0: one q(z) for every sample)
  long mx_stride;
  const double* xm;     // xm_b at xm[b * xm_stride]
  long xm_stride;
  int nv, nx, nb;
  double* quad;         // [n][b] at n * ldo + b
  double* lin;
  int ldo;
};

// grid (point tiles, samples), 128 threads.  Per 32-column tile of Y = V_b mx_b (DMMA, warps on 16 x 16 quadrants as
// above), the epilogue multiplies Y element-wise with V_b and adds it into per-row partials; column tiles in order,
// then the four lanes of a row (fixed butterfly) and the two column-half warps in order.  Samples b >= nb return.
__global__ void __launch_bounds__(128) predict_quad_kernel(const PredQuadArgs g) {
  __shared__ __align__(16) double Vs[PQ_T * PQ_LDS];
  __shared__ __align__(16) double Ms[PQ_T * PQ_LDS];
  __shared__ double red[2][PQ_T];
  const int b = blockIdx.y;
  if (b >= g.nb) return;
  const int r0 = blockIdx.x * PQ_T, nx = g.nx;
  const double* Vb = g.V + (long)b * g.v_stride;
  const double* Mb = g.mx + (long)b * g.mx_stride;
  const double* Xb = g.xm + (long)b * g.xm_stride;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wi = warp >> 1, wj = warp & 1, grp = lane >> 2, tig = lane & 3;
  double rp[2] = {0.0, 0.0};
  for (int c0 = 0; c0 < nx; c0 += PQ_T) {
    double acc[2][2][2];
#pragma unroll
    for (int x = 0; x < 2; ++x)
#pragma unroll
      for (int y = 0; y < 2; ++y) acc[x][y][0] = acc[x][y][1] = 0.0;
    for (int k0 = 0; k0 < nx; k0 += PQ_BK) {
#pragma unroll
      for (int q = 0; q < PQ_T * PQ_BK / 128; ++q) {
        const int e = q * 128 + tid, hi = e >> 5, lo = e & 31;
        // Vs[row][k] = V(r0 + row, k0 + k);  Ms[col][k] = mx(k0 + k, c0 + col)
        Vs[hi * PQ_LDS + lo] = (r0 + hi < g.nv && k0 + lo < nx) ? Vb[(long)(r0 + hi) * g.ldv + k0 + lo] : 0.0;
        Ms[lo * PQ_LDS + hi] = (k0 + hi < nx && c0 + lo < nx) ? Mb[(long)(k0 + hi) * nx + c0 + lo] : 0.0;
      }
      __syncthreads();
#pragma unroll
      for (int k4 = 0; k4 < PQ_BK / 4; ++k4) {
        double fa[2], fb[2];
#pragma unroll
        for (int x = 0; x < 2; ++x) {
          fa[x] = Vs[(wi * 16 + x * 8 + grp) * PQ_LDS + k4 * 4 + tig];
          fb[x] = Ms[(wj * 16 + x * 8 + grp) * PQ_LDS + k4 * 4 + tig];
        }
#pragma unroll
        for (int x = 0; x < 2; ++x)
#pragma unroll
          for (int y = 0; y < 2; ++y) dmma_8x8x4(acc[x][y][0], acc[x][y][1], fa[x], fb[y]);
      }
      __syncthreads();
    }
#pragma unroll
    for (int x = 0; x < 2; ++x) {
      const int row = r0 + wi * 16 + x * 8 + grp;
      if (row >= g.nv) continue;
#pragma unroll
      for (int y = 0; y < 2; ++y)
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int col = c0 + wj * 16 + y * 8 + tig * 2 + u;
          if (col < nx) rp[x] += acc[x][y][u] * Vb[(long)row * g.ldv + col];
        }
    }
  }
#pragma unroll
  for (int x = 0; x < 2; ++x) {
    rp[x] += __shfl_xor_sync(0xffffffffu, rp[x], 1);
    rp[x] += __shfl_xor_sync(0xffffffffu, rp[x], 2);
    if (tig == 0) red[wj][wi * 16 + x * 8 + grp] = rp[x];
  }
  // lin: warp w takes rows w, w + 4, ..; lanes stride k, then a fixed shuffle tree
  for (int rr = warp; rr < PQ_T; rr += 4) {
    const int row = r0 + rr;
    if (row >= g.nv) continue;
    double s = 0.0;
    for (int k = lane; k < nx; k += 32) s += Vb[(long)row * g.ldv + k] * Xb[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
    if (lane == 0) g.lin[(long)row * g.ldo + b] = s;
  }
  __syncthreads();
  if (tid < PQ_T && r0 + tid < g.nv) g.quad[(long)(r0 + tid) * g.ldo + b] = red[0][tid] + red[1][tid];
}

// Launch shapes of the test-side kernels, shared by predict_batch_run and the C-ABI test hook.  The grids depend on the
// chunk's point count (nrow: its capacity, nv: valid points) and the batch's sample slots (nslots) only.
// q[z][n][b] (z < PQ_SLICES, n < nv, b < ncol) = partial <Bxx*_n, mx_b> over k slice z.
inline void predict_qb_launch(cudaStream_t st, const double* X, long K, const double* mx, long mx_stride, int ncol,
                              int nv, int nrow, int nslots, double* q, int ldq) {
  PredQbArgs g;
  g.X = X; g.K = K; g.mx = mx; g.mx_stride = mx_stride; g.nv = nv; g.ncol = ncol; g.q = q; g.nrow = nrow; g.ldq = ldq;
  predict_qb_kernel<<<dim3((nv + PQ_T - 1) / PQ_T, (nslots + PQ_T - 1) / PQ_T, PQ_SLICES), 128, 0, st>>>(g);
}

inline void predict_quad_launch(cudaStream_t st, const PredQuadArgs& g, int nslots) {
  predict_quad_kernel<<<dim3((g.nv + PQ_T - 1) / PQ_T, nslots), 128, 0, st>>>(g);
}

// One thread per point of the chunk: per-sample moments for b < nb in ascending b, and the running averages
//   mean_s[n][b] = m1 = sqrt(s2f) lin,  var_s[n][b] = m2 - m1^2,  m2 = s2f (q1_b + Qb + quad),
//   acc_mu[n] += w m1,  acc_var[n] += w (m2 - m1^2)          (the accumulation of predict_point_kernel)
// Qb = the PQ_SLICES partials of column b * q_col summed in order (q_col = 0: one q(z) for every sample).
__global__ void predict_finish_kernel(const double* __restrict__ qpart, int nrow, int ldq, int q_col,
                                      const double* __restrict__ quad, const double* __restrict__ lin, int ldo,
                                      const double* __restrict__ q1, int nv, int nb, double sqrt_s2f, double s2f,
                                      double w, double* __restrict__ mean_s, double* __restrict__ var_s, long lds,
                                      double* __restrict__ acc_mu, double* __restrict__ acc_var) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= nv) return;
  double am = acc_mu[n], av = acc_var[n];
  for (int b = 0; b < nb; ++b) {
    double qb = 0.0;
    for (int z = 0; z < PQ_SLICES; ++z) qb += qpart[((long)z * nrow + n) * ldq + b * q_col];
    const double m1 = sqrt_s2f * lin[(long)n * ldo + b];
    const double m2 = s2f * (q1[b] + qb + quad[(long)n * ldo + b]);
    const double v = m2 - m1 * m1;
    if (mean_s) mean_s[(long)n * lds + b] = m1;
    if (var_s) var_s[(long)n * lds + b] = v;
    am += w * m1;
    av += w * v;
  }
  acc_mu[n] = am;
  acc_var[n] = av;
}

// ---- Joint predictive covariance (cgpcm_predict_f_cov): the expectation of f_p f_q under sample b's q(z) is
//     E[f_p f_q | h_b] = s2_f (a_c(t_p - t_q) + <Ahh_c(t_p - t_q), h_b h_b^T - iKh> + <Bxx*(p, q), mx_b> + v_p^T mx_b v_q)
//     Bxx*(p, q) = Axx(t_p, t_q) - A*_p^T iKh A*_q,   v_p = A*_p^T h_b
// Axx(t_p, t_q) is the closed form of Axx with the two inputs on the two factors of the double integral: substituting
// s1 = t_p - tau1, s2 = t_q - tau2 leaves the quadratic form unchanged and only moves the linear terms, so it is
// axx_user_kernel's arithmetic with dk = t_p - tx_k and dl = t_q - tx_l (tests/pair_oracle.py).  The centre
// statistics a_c, Ahh_c at the lag are those of predict_k / the AKM sampler (ahh_center_kernel).  Work runs over tiles
// of P x Q point pairs, p >= q; pair e = i Q + j stands for (p0 + i, q0 + j).

// X[e][k][l] = Axx(tp[i], tq[j])[k][l] - G(i, k; j, l)   (e = i nq + j, dense [pair][nx][nx]; G optional:
// G(i, k; j, l) at G[(i gk + k) ldg + j gk + l], the fold A*_p^T iKh A*_q as one GEMM lays it out).  Evaluated densely
// (c.cull = 746: a skipped element is exactly 0).  Grid-stride, any grid.
__global__ void axx_pair_kernel(const double* __restrict__ tp, int np_, const double* __restrict__ tq, int nq,
                                const double* __restrict__ tx, int nx, const double* __restrict__ G, long ldg, int gk,
                                double* __restrict__ X, const PsiConst c, const BvnTab T) {
  const long per = (long)nx * nx;
  const long total = (long)np_ * nq * per;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const long e = idx / per;
    const int r = (int)(idx - e * per);
    const int k = r / nx, l = r - k * nx;
    const int i = (int)(e / nq), j = (int)(e - (long)i * nq);
    const double dk = tp[i] - tx[k], dl = tq[j] - tx[l];
    const double Gx = -c.g1 * (dk * dk + dl * dl) + c.g2 * dk * dl;
    double v = 0.0;
    if (Gx >= -c.cull) {
      v = c.pref_xx * exp(Gx);
      if (c.causal) {
        double x1 = c.p * dk + c.q * dl, x2 = c.q * dk + c.p * dl;
        if (c.causal_id) { x1 -= fmax(dk, 0.0) * c.isq11; x2 -= fmax(dl, 0.0) * c.isq11; }
        v *= bvnd_tab(-x1, -x2, T);
      }
    }
    if (G) v -= G[((long)i * gk + k) * ldg + (long)j * gk + l];
    X[idx] = v;
  }
}

inline void axx_pair_launch(cudaStream_t st, const double* tp, int np_, const double* tq, int nq, const double* tx,
                            int nx, const double* G, long ldg, int gk, double* X, const PsiConst& c, const BvnTab& T) {
  axx_pair_kernel<<<148 * 8, 256, 0, st>>>(tp, np_, tq, nq, tx, nx, G, ldg, gk, X, c, T);
}

// One thread per (pair, sample) of a tile with p >= q:
//   C_b[p][q] = C_b[q][p] = s2f (ac[e] + gf[e][b] + Qb + R) - m_p m_q
// with R = v_p^T mx_b v_q already in C_b[p][q] (the rank-one GEMMs), Qb the PQ_SLICES partials of column b * q_col
// summed in order, gf[e][b] = <Ahh_c, h_b h_b^T - iKh> and m the per-sample means at m[p * ldm + b].
__global__ void pcov_finish_kernel(const double* __restrict__ qpart, int nrow, int ldq, int q_col,
                                   const double* __restrict__ gf, int ldgf, const double* __restrict__ ac, int npairs,
                                   int nq, int p0, int q0, int nb, const double* __restrict__ m, long ldm, double s2f,
                                   double* __restrict__ C, long cstride, long ldc) {
  const long total = (long)npairs * nb;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int e = (int)(idx / nb), b = (int)(idx - (long)e * nb);
    const int p = p0 + e / nq, q = q0 + e % nq;
    if (p < q) continue;
    double qb = 0.0;
    for (int z = 0; z < PQ_SLICES; ++z) qb += qpart[((long)z * nrow + e) * ldq + b * q_col];
    double* Cb = C + (long)b * cstride;
    const double v = s2f * (ac[e] + gf[(long)e * ldgf + b] + qb + Cb[(long)p * ldc + q]) - m[(long)p * ldm + b] * m[(long)q * ldm + b];
    Cb[(long)p * ldc + q] = v;
    Cb[(long)q * ldc + p] = v;
  }
}

// ---- Held-out scoring (cgpcm_predict_logpdf): log N(y; m_b, S_b), S_b = C_b + d I, through one Cholesky factorisation
// of the bordered matrix
//     K_b = [[S_b, r_b], [r_b^T, c]],   r_b = y - m_b,   L_K = [[L_b, 0], [z_b^T, l]],   L_b L_b^T = S_b,  z_b = L_b^-1 r_b
// so that the factor's last row is the whitened residual and its first n diagonal entries give log det S_b.  c = DBL_MAX:
// the border pivot c - |z_b|^2 is positive for any finite z_b short of overflow, so the factorisation fails only where
// S_b does (a bound from d, such as c = 1 + 2 |r|^2 / d, needs d > 0, and d = reg = 0 is allowed), and nothing is ever
// read from that pivot (c - l^2 would cancel).  Rows and columns past n + 1 are the identity.

// K[b] (ldk x ldk, k2 apart) for samples b < nb of C (npad x npad, n2 apart) and the means m[p * ldm + b]; y == nullptr
// writes r = 0 and c = 1 (S_b with an identity border).  Grid-stride, any grid.
__global__ void pcov_border_kernel(const double* __restrict__ C, int npad, long n2, const double* __restrict__ m,
                                   long ldm, const double* __restrict__ y, int n, double d, int nb,
                                   double* __restrict__ K, int ldk, long k2) {
  const long total = (long)nb * k2;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int b = (int)(idx / k2);
    const long e = idx - (long)b * k2;
    const int i = (int)(e / ldk), j = (int)(e - (long)i * ldk);
    double v = (i == j) ? 1.0 : 0.0;
    if (i < n && j < n) v = C[(long)b * n2 + (long)i * npad + j] + (i == j ? d : 0.0);
    else if (i == n && j == n) v = y ? DBL_MAX : 1.0;
    else if (i == n && j < n) v = y ? y[j] - m[(long)j * ldm + b] : 0.0;
    else if (j == n && i < n) v = y ? y[i] - m[(long)i * ldm + b] : 0.0;
    K[idx] = v;
  }
}

// One CTA (256 threads) per sample b < gridDim.x of the factored K[b]: logdet = 2 sum log L_ii and q = sum z_i^2, each
// thread over i = tid, tid + 256, .. in order, then a fixed tree; lp[b] = -(n log 2 pi + logdet + q) / 2 and
// white[p * ldw + b] = z_p.
__global__ void __launch_bounds__(256) pcov_score_kernel(const double* __restrict__ K, int ldk, long k2, int n,
                                                         double* __restrict__ lp, double* __restrict__ white, long ldw) {
  __shared__ double sl[256], sq[256];
  const int b = blockIdx.x, tid = threadIdx.x;
  const double* Kb = K + (long)b * k2;
  const double* z = Kb + (long)n * ldk;
  double l = 0.0, q = 0.0;
  for (int i = tid; i < n; i += 256) {
    const double zi = z[i];
    l += log(Kb[(long)i * ldk + i]);
    q += zi * zi;
    if (white) white[(long)i * ldw + b] = zi;
  }
  sl[tid] = l;
  sq[tid] = q;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (tid < s) {
      sl[tid] += sl[tid + s];
      sq[tid] += sq[tid + s];
    }
    __syncthreads();
  }
  if (tid == 0) lp[b] = -0.5 * (n * 1.83787706640934548356 + 2.0 * sl[0] + sq[0]);    // log 2 pi
}

}  // namespace cg

namespace cg {

// Off-diagonal ("center") Psi statistics of predict_k (src/core/cgpcm.py:164-166,190-192): t2 = 0, upper limit
// min(t, 0) for the causal model.  Closed forms (oracle.model.psi_center_closed):
//   a_c(t)        = pref_a exp(-(alpha/2 + gamma) t^2) erfc(sqrt(2 alpha) |t| / 2)
//   Ahh_c(t)[i,j] = pref_h exp(c + b^2 / 8B) erfc(sqrt(2B) (b / 4B - min(t, 0))),   B = alpha + gamma,
//                   b = 2B t - 2 gamma (th_i + th_j),  c = -alpha (t^2 + th_i^2) - gamma (t - th_i)^2 - B th_j^2
// (acausal: no erfc, twice the prefactor).  AC: [n][nh * nhl] (row i at stride nhl, zero padded), ac: [n].
__global__ void ahh_center_kernel(const double* __restrict__ t, int n, const double* __restrict__ th, int nh, int nhl,
                                  double alpha, double gamma, int causal, double* __restrict__ AC,
                                  double* __restrict__ ac) {
  const double PI = 3.14159265358979323846;
  const double B = alpha + gamma;
  const double pref_a = (causal ? 0.5 : 1.0) * sqrt(PI / (2.0 * alpha));
  const double pref_h = (causal ? 0.5 : 1.0) * sqrt(PI / (2.0 * B));
  const long per = (long)nh * nhl;
  const long total = (long)n * per;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int p = (int)(idx / per);
    const int e = (int)(idx - (long)p * per);
    const int i = e / nhl, j = e - i * nhl;
    const double tt = t[p];
    if (e == 0) {
      double v = pref_a * exp(-(0.5 * alpha + gamma) * tt * tt);
      if (causal) v *= erfc(sqrt(2.0 * alpha) * fabs(tt) * 0.5);
      ac[p] = v;
    }
    double v = 0.0;
    if (j < nh) {
      const double ti = th[i], tj = th[j];
      const double b = 2.0 * B * tt - 2.0 * gamma * (ti + tj);
      const double c = -alpha * (tt * tt + ti * ti) - gamma * (tt - ti) * (tt - ti) - B * tj * tj;
      v = pref_h * exp(c + b * b / (8.0 * B));
      if (causal) v *= erfc(sqrt(2.0 * B) * (b / (4.0 * B) - fmin(tt, 0.0)));
    }
    AC[idx] = v;
  }
}

// HH[b][i * nhl + j] = h_b[i] h_b[j] - iKh[i][j]   (rows b >= nb and the padding are zero)
__global__ void hh_build_kernel(const double* __restrict__ hs, long ldh, int nb, int nbp, const double* __restrict__ iKh,
                                long ld, int nh, int nhl, double* __restrict__ HH) {
  const long per = (long)nh * nhl;
  const long total = (long)nbp * per;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int b = (int)(idx / per);
    const int e = (int)(idx - (long)b * per);
    const int i = e / nhl, j = e - i * nhl;
    double v = 0.0;
    if (b < nb && j < nh) v = hs[(long)b * ldh + i] * hs[(long)b * ldh + j] - iKh[(long)i * ld + j];
    HH[idx] = v;
  }
}

// out[p][b] = s2f (ac[p] + G[p][b])
__global__ void kernel_finish_kernel(const double* __restrict__ G, long ldg, const double* __restrict__ ac, int n, int nb,
                                     double s2f, double* __restrict__ out) {
  const long total = (long)n * nb;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const int p = (int)(idx / nb), b = (int)(idx - (long)p * nb);
    out[idx] = s2f * (ac[p] + G[(long)p * ldg + b]);
  }
}

}  // namespace cg

namespace cg {

// Filter-side kernel matrices of predict_h / predict_psd (src/core/cgpcm.py:685-688,738-741; DEQ kernel
// src/core/kernel.py:43-46):  Kuh[i][p] = k_h(th_i, t_p)  (nhp x ldn, zero padded),
// Ktt[p][q] = k_h(t_p, t_q) + reg [p == q]  (ldn x ldn; identity on the padding block so that its Cholesky exists).
__global__ void filter_kernels_kernel(const double* __restrict__ th, int nh, int nhp, const double* __restrict__ t, int n,
                                      int ldn, double alpha, double gamma, double reg, double* __restrict__ Kuh,
                                      double* __restrict__ Ktt) {
  const long n1 = (long)nhp * ldn, n2 = (long)ldn * ldn;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < n1 + n2; idx += (long)gridDim.x * blockDim.x) {
    if (idx < n1) {
      const int i = (int)(idx / ldn), p = (int)(idx - (long)i * ldn);
      double v = 0.0;
      if (i < nh && p < n) {
        const double a = th[i], b = t[p];
        v = exp(-alpha * (a * a + b * b) - gamma * (a - b) * (a - b));
      }
      Kuh[idx] = v;
    } else {
      const long e = idx - n1;
      const int p = (int)(e / ldn), q = (int)(e - (long)p * ldn);
      double v = (p == q) ? 1.0 : 0.0;
      if (p < n && q < n) {
        const double a = t[p], b = t[q];
        v = exp(-alpha * (a * a + b * b) - gamma * (a - b) * (a - b)) + (p == q ? reg : 0.0);
      } else if (p < n || q < n) {
        v = 0.0;
      }
      Ktt[e] = v;
    }
  }
}

}  // namespace cg

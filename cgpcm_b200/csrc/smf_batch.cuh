// Batched scoring of filter samples under the stochastic SMF bound (frozen regime), SURVEY.md §8f rank 2:
//
//   C1_b = sum_n A_n^T h_b h_b^T A_n = sum_n w_bn w_bn^T,   w_bn = A_n^T h_b   (rank one per observation)
//
// The caller forms W = H_B A per chunk with the small-left-operand GEMM (one row of W per sample); the kernels below
// add the windowed symmetric products W_b^T W_b into per-sample slabs and do the per-sample M x M algebra.  Every
// per-sample sum runs in an order that depends on the sample's own data and the chunk plan only -- never on how many
// samples share the launch or where the sample sits in the batch -- so a sample's result is bitwise the same in
// any batch.
#pragma once
#include "dgemm_dmma.cuh"

namespace cg {

constexpr int SMF_T = 32;               // output tile (rows = columns) of the windowed contraction
constexpr int SMF_BK = 32;              // observations per shared-memory stage
constexpr int SMF_LDS = SMF_T + 4;      // == 4 (mod 8): conflict-free fragment loads
constexpr int SMF_SLICES = 4;           // observation slices of a chunk (fixed: the sum order must not depend on B)
constexpr int SMF_ALG_THREADS = 512;

struct SmfC1Args {
  const double* W;     // W_b(n, k) at W[b * w_stride + n * kwp + k]
  long w_stride;
  int kwp, nc;         // window width, padded observations of the chunk
  double* part;        // slice z of sample b: part + (b * SMF_SLICES + z) * l2, window at offset `win`
  long l2, ld, win;
};

// grid (T (T + 1) / 2 lower tiles of the kwp x kwp window, SMF_SLICES, samples), 128 threads.  Each warp owns a 16 x 16
// quadrant of the 32 x 32 tile (2 x 2 DMMA m8n8k4 tiles).  part[b][z][window] += sum over the slice's observations of
// W_b(n, k) W_b(n, l): one CTA owns each (tile, slice, sample), and chunks are launched in order, so every element is
// accumulated in a fixed order.
__global__ void __launch_bounds__(128) smf_c1_kernel(const SmfC1Args g) {
  __shared__ __align__(16) double As[SMF_BK * SMF_LDS];
  __shared__ __align__(16) double Bs[SMF_BK * SMF_LDS];
  int ti = 0;
  while ((ti + 1) * (ti + 2) / 2 <= (int)blockIdx.x) ++ti;
  const int tj = (int)blockIdx.x - ti * (ti + 1) / 2;
  const int z = blockIdx.y, b = blockIdx.z;
  const int nb8 = (g.nc + 7) / 8, per = (nb8 + SMF_SLICES - 1) / SMF_SLICES;
  const int n0 = z * per * 8, n1 = min(g.nc, n0 + per * 8);
  if (n0 >= n1) return;
  const double* Wb = g.W + (long)b * g.w_stride;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wi = warp >> 1, wj = warp & 1, grp = lane >> 2, tig = lane & 3;
  const int ka0 = ti * SMF_T, kb0 = tj * SMF_T;
  double acc[2][2][2];
#pragma unroll
  for (int x = 0; x < 2; ++x)
#pragma unroll
    for (int y = 0; y < 2; ++y) acc[x][y][0] = acc[x][y][1] = 0.0;
  for (int nb = n0; nb < n1; nb += SMF_BK) {
#pragma unroll
    for (int q = 0; q < SMF_BK * SMF_T / 128; ++q) {
      const int e = q * 128 + tid, rr = e >> 5, cc = e & 31, n = nb + rr;
      const bool nok = n < n1;
      As[rr * SMF_LDS + cc] = (nok && ka0 + cc < g.kwp) ? Wb[(long)n * g.kwp + ka0 + cc] : 0.0;
      Bs[rr * SMF_LDS + cc] = (nok && kb0 + cc < g.kwp) ? Wb[(long)n * g.kwp + kb0 + cc] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int k4 = 0; k4 < SMF_BK / 4; ++k4) {
      const int kr = (k4 * 4 + tig) * SMF_LDS;
      double fa[2], fb[2];
#pragma unroll
      for (int x = 0; x < 2; ++x) {
        fa[x] = As[kr + wi * 16 + x * 8 + grp];
        fb[x] = Bs[kr + wj * 16 + x * 8 + grp];
      }
#pragma unroll
      for (int x = 0; x < 2; ++x)
#pragma unroll
        for (int y = 0; y < 2; ++y) dmma_8x8x4(acc[x][y][0], acc[x][y][1], fa[x], fb[y]);
    }
    __syncthreads();
  }
  double* C = g.part + ((long)b * SMF_SLICES + z) * g.l2 + g.win;
#pragma unroll
  for (int x = 0; x < 2; ++x) {
    const int row = ka0 + wi * 16 + x * 8 + grp;
    if (row >= g.kwp) continue;
#pragma unroll
    for (int y = 0; y < 2; ++y) {
      const int col = kb0 + wj * 16 + y * 8 + tig * 2;     // even; kwp is a multiple of 8
      if (col >= g.kwp) continue;
      double2* p = reinterpret_cast<double2*>(C + (long)row * g.ld + col);
      const double2 o = *p;
      *p = make_double2(o.x + acc[x][y][0], o.y + acc[x][y][1]);
    }
  }
}

// c1[b] (lower triangle, nx x nx; zero elsewhere) = sum of the SMF_SLICES slices in order 0, 1, ..
__global__ void smf_reduce_kernel(const double* __restrict__ part, long total, long l2, long ld, int nx,
                                  double* __restrict__ c1) {
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const long b = idx / l2, e = idx - b * l2;
    const int r = (int)(e / ld), c = (int)(e - (long)r * ld);
    double s = 0.0;
    if (r < nx && c <= r) {
      const double* p = part + b * SMF_SLICES * l2 + e;
#pragma unroll
      for (int z = 0; z < SMF_SLICES; ++z) s += p[z * l2];
    }
    c1[idx] = s;
  }
}

struct SmfAlgArgs {
  const double* kx;     // Kx (with its jitter), ld x ld
  const double* sxx;    // frozen sum_Bxx
  const double* c1;     // [b] slabs (lower triangle)
  const double* fy;     // frozen sum_Ahx_y, nh x nx at leading dimension ld
  const double* bhh;    // frozen sum_Bhh
  const double* hs;     // samples [b][ldh]
  double* work;         // [b][pass] ld x ld factor slabs
  double* out;          // [b][5]: logdet P, |L^-1 lam|^2, logdet P0, |L0^-1 lam|^2, h^T sum_Bhh h
  int* info;            // [b][2]: pivot + 1 of a failed factorisation of P / P0, else 0
  long ld, l2;
  int ldh, nh, nx;
  double r, c0, reg;
  int want_p, passes;   // blockIdx.y: pass 0 = P (when want_p), the other pass = P0
};

// One CTA per (sample, matrix): P_b = Kx + r S_b (+ reg I for P) with S_b = sum_Bxx + C1_b, its right-looking
// Cholesky factorisation in place in the sample's work slab, fused with the forward solve L z = lam_b,
// lam_b = c0 sum_Ahx_y^T h_b; log det P_b = sum_j log(pivot_j) and |z|^2 accumulate in column order.  The P0 pass
// also forms h_b^T sum_Bhh h_b.  Dynamic shared memory: 2 nx doubles.
__global__ void __launch_bounds__(SMF_ALG_THREADS) smf_algebra_kernel(const SmfAlgArgs g) {
  extern __shared__ double sh[];
  double* col = sh;           // column j of the factor below the diagonal
  double* zv = sh + g.nx;     // right-hand side / solution
  __shared__ double wsum[SMF_ALG_THREADS / 32];
  const int b = blockIdx.x;
  const int kind = g.want_p ? (int)blockIdx.y : 1;         // 0 = P, 1 = P0
  const double jit = kind == 0 ? g.reg : 0.0;
  const int n = g.nx, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = SMF_ALG_THREADS / 32;
  const long ld = g.ld;
  double* P = g.work + ((long)b * g.passes + blockIdx.y) * g.l2;
  const double* c1 = g.c1 + (long)b * g.l2;
  const double* hb = g.hs + (long)b * g.ldh;
  for (long idx = tid; idx < (long)n * n; idx += blockDim.x) {
    const int i = (int)(idx / n), j = (int)(idx - (long)i * n);
    if (j > i) continue;
    const long e = (long)i * ld + j;
    const double s = g.sxx[e] + c1[e];
    P[e] = g.kx[e] + g.r * s + (i == j ? jit : 0.0);
  }
  for (int k = tid; k < n; k += blockDim.x) {
    double s = 0.0;
    for (int i = 0; i < g.nh; ++i) s += g.fy[(long)i * ld + k] * hb[i];
    zv[k] = g.c0 * s;
  }
  __syncthreads();
  double logdet = 0.0, quad = 0.0;
  int fail = 0;
  for (int j = 0; j < n; ++j) {
    const double d = P[(long)j * ld + j];
    if (!(d > 0.0)) { fail = j + 1; break; }       // the same value in every thread: a uniform exit
    const double l = sqrt(d);
    for (int i = j + 1 + tid; i < n; i += blockDim.x) col[i] = P[(long)i * ld + j] / l;
    if (tid == 0) {
      const double zj = zv[j] / l;
      zv[j] = zj;
      logdet += log(d);
      quad += zj * zj;
    }
    __syncthreads();
    const double zj = zv[j];
    for (int i = j + 1 + warp; i < n; i += NW) {
      const double lij = col[i];
      double* row = P + (long)i * ld;
      for (int k = j + 1 + lane; k <= i; k += 32) row[k] -= lij * col[k];
      if (lane == 0) zv[i] -= lij * zj;
    }
    __syncthreads();
  }
  double* o = g.out + (long)b * 5;
  if (tid == 0) {
    g.info[b * 2 + kind] = fail;
    o[kind * 2] = logdet;
    o[kind * 2 + 1] = quad;
  }
  if (kind == 1) {
    // h^T sum_Bhh h: one warp per row (fixed shuffle tree), rows in a fixed order per warp, warps added in order
    double acc = 0.0;
    for (int i = warp; i < g.nh; i += NW) {
      double s = 0.0;
      for (int k = lane; k < g.nh; k += 32) s += g.bhh[(long)i * ld + k] * hb[k];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
      acc += hb[i] * s;
    }
    if (lane == 0) wsum[warp] = acc;
    __syncthreads();
    if (tid == 0) {
      double s = 0.0;
      for (int w = 0; w < NW; ++w) s += wsum[w];
      o[4] = s;
    }
  }
}

// h^T M h (M: nh x nh at leading dimension ld) for the whole block, valid in thread 0: one warp per row (fixed shuffle
// tree), rows in a fixed order per warp, warps added in order.  wsum: blockDim.x / 32 doubles of shared memory.
__device__ double block_quad_form(const double* M, long ld, const double* hb, int nh, double* wsum) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  double acc = 0.0;
  for (int i = warp; i < nh; i += nw) {
    double s = 0.0;
    for (int k = lane; k < nh; k += 32) s += M[(long)i * ld + k] * hb[k];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
    acc += hb[i] * s;
  }
  if (lane == 0) wsum[warp] = acc;
  __syncthreads();
  double s = 0.0;
  if (tid == 0)
    for (int w = 0; w < nw; ++w) s += wsum[w];
  return s;
}

struct SmfPostArgs {
  const double* kx;     // Kx (with its jitter), ld x ld
  const double* sxx;    // frozen sum_Bxx
  const double* c1;     // [b] slabs (lower triangle)
  const double* fy;     // frozen sum_Ahx_y, nh x nx at leading dimension ld
  const double* ahh;    // frozen Ahh, nh x nh at leading dimension ld
  const double* ikx;    // iKx, ld x ld
  const double* tr;     // device scalar tr(Ahh iKh)
  const double* hs;     // samples [b][ldh]
  double* work;         // [b][2] ld x ld slabs: Cholesky factor L of P_b, then L^-1
  double* mx;           // [b] at stride l2: mx_b = P_b^-1 + xm_b xm_b^T - iKx, full nx x nx at leading dimension nx
  double* xm;           // [b] at stride ld: xm_b = P_b^-1 lam_b
  double* q1;           // [b]: a + h_b^T Ahh h_b - tr(Ahh iKh)
  int* info;            // [b]: pivot + 1 of a failed factorisation of P_b, else 0
  long ld, l2;
  int ldh, nh, nx, nb;
  double r, c0, reg, a;
};

// The per-sample optimal q(z | h_b) of predict_f (SMF) and the scalar q1_b, one CTA per sample (b < nb):
// P_b = Kx + r (sum_Bxx + C1_b) + reg I, its right-looking Cholesky factorisation (stored as L in the first work slab)
// fused with the forward solve of lam_b = c0 sum_Ahx_y^T h_b, the backward solve for xm_b, Z = L^-1 by the same
// right-looking sweep (second slab), then mx_b[k][l] = sum_{i >= max(k, l)} Z[i][k] Z[i][l] + xm_k xm_l - iKx[k][l]
// (both triangles from the same value).  Every sum runs in an order fixed by nx alone.  Dynamic shared memory:
// 3 nx doubles.
__global__ void __launch_bounds__(SMF_ALG_THREADS) smf_posterior_kernel(const SmfPostArgs g) {
  extern __shared__ double sh[];
  double* col = sh;           // column j of the factor below the diagonal
  double* zv = sh + g.nx;     // right-hand side / solution
  double* dg = sh + 2 * g.nx; // diagonal of the factor
  __shared__ double wsum[SMF_ALG_THREADS / 32];
  const int b = blockIdx.x;
  if (b >= g.nb) return;
  const int n = g.nx, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = SMF_ALG_THREADS / 32;
  const long ld = g.ld;
  double* P = g.work + (long)b * 2 * g.l2;
  double* Z = P + g.l2;
  const double* c1 = g.c1 + (long)b * g.l2;
  const double* hb = g.hs + (long)b * g.ldh;
  for (long idx = tid; idx < (long)n * n; idx += blockDim.x) {
    const int i = (int)(idx / n), j = (int)(idx - (long)i * n);
    const long e = (long)i * ld + j;
    if (j <= i) {
      const double s = g.sxx[e] + c1[e];
      P[e] = g.kx[e] + g.r * s + (i == j ? g.reg : 0.0);
    }
    Z[e] = i == j ? 1.0 : 0.0;
  }
  for (int k = tid; k < n; k += blockDim.x) {
    double s = 0.0;
    for (int i = 0; i < g.nh; ++i) s += g.fy[(long)i * ld + k] * hb[i];
    zv[k] = g.c0 * s;
  }
  __syncthreads();
  int fail = 0;
  for (int j = 0; j < n; ++j) {
    const double d = P[(long)j * ld + j];
    if (!(d > 0.0)) { fail = j + 1; break; }       // the same value in every thread: a uniform exit
    const double l = sqrt(d);
    for (int i = j + 1 + tid; i < n; i += blockDim.x) {
      const double v = P[(long)i * ld + j] / l;
      col[i] = v;
      P[(long)i * ld + j] = v;
    }
    if (tid == 0) {
      zv[j] = zv[j] / l;
      dg[j] = l;
    }
    __syncthreads();
    const double zj = zv[j];
    for (int i = j + 1 + warp; i < n; i += NW) {
      const double lij = col[i];
      double* row = P + (long)i * ld;
      for (int k = j + 1 + lane; k <= i; k += 32) row[k] -= lij * col[k];
      if (lane == 0) zv[i] -= lij * zj;
    }
    __syncthreads();
  }
  if (fail) {
    if (tid == 0) g.info[b] = fail;
    return;
  }
  // backward solve L^T x = z (x overwrites zv)
  for (int j = n - 1; j >= 0; --j) {
    if (tid == 0) zv[j] = zv[j] / dg[j];
    __syncthreads();
    const double xj = zv[j];
    for (int i = tid; i < j; i += blockDim.x) zv[i] -= P[(long)j * ld + i] * xj;
    __syncthreads();
  }
  // Z = L^-1 (lower): row j is final once divided by L[j][j]; then it updates the rows below it
  for (int j = 0; j < n; ++j) {
    const double l = dg[j];
    for (int c = tid; c <= j; c += blockDim.x) Z[(long)j * ld + c] /= l;
    __syncthreads();
    const double* zj = Z + (long)j * ld;
    for (int i = j + 1 + warp; i < n; i += NW) {
      const double lij = P[(long)i * ld + j];
      double* row = Z + (long)i * ld;
      for (int c = lane; c <= j; c += 32) row[c] -= lij * zj[c];
    }
    __syncthreads();
  }
  double* mxb = g.mx + (long)b * g.l2;
  for (long idx = tid; idx < (long)n * n; idx += blockDim.x) {
    const int k = (int)(idx / n), l = (int)(idx - (long)k * n);
    if (l > k) continue;
    double s = 0.0;
    for (int i = k; i < n; ++i) s += Z[(long)i * ld + k] * Z[(long)i * ld + l];
    const double v = s + zv[k] * zv[l] - g.ikx[(long)k * ld + l];
    mxb[(long)k * n + l] = v;
    mxb[(long)l * n + k] = v;
  }
  for (int k = tid; k < n; k += blockDim.x) g.xm[(long)b * ld + k] = zv[k];
  const double q = block_quad_form(g.ahh, ld, hb, g.nh, wsum);
  if (tid == 0) {
    g.q1[b] = g.a + q - g.tr[0];
    g.info[b] = 0;
  }
}

// q1_b = a + h_b^T Ahh h_b - tr(Ahh iKh) for b < nb: the per-sample scalar of predict_f when q(z) is shared (smf = 0)
__global__ void __launch_bounds__(256) predict_q1_kernel(const double* __restrict__ ahh, long ld,
                                                         const double* __restrict__ hs, int ldh, int nh, int nb, double a,
                                                         const double* __restrict__ tr, double* __restrict__ q1) {
  __shared__ double wsum[8];
  const int b = blockIdx.x;
  if (b >= nb) return;
  const double q = block_quad_form(ahh, ld, hs + (long)b * ldh, nh, wsum);
  if (threadIdx.x == 0) q1[b] = a + q - tr[0];
}

// Launch shapes of the three kernels, shared by smf_batch_run and the C-ABI test hooks.
// part[b][z] += W_b^T W_b of one window (k_lo, kwp) over nc padded observations, for samples b < nb.
inline void smf_c1_launch(cudaStream_t st, const double* W, long w_stride, int kwp, int nc, int k_lo, double* part,
                          long ld, int nb) {
  SmfC1Args g;
  g.W = W; g.w_stride = w_stride; g.kwp = kwp; g.nc = nc;
  g.part = part; g.l2 = ld * ld; g.ld = ld; g.win = (long)k_lo * ld + k_lo;
  const int T = (kwp + SMF_T - 1) / SMF_T;
  smf_c1_kernel<<<dim3(T * (T + 1) / 2, SMF_SLICES, nb), 128, 0, st>>>(g);
}

inline void smf_reduce_launch(cudaStream_t st, const double* part, long ld, int nx, int nb, double* c1) {
  smf_reduce_kernel<<<148 * 4, 256, 0, st>>>(part, (long)nb * ld * ld, ld * ld, ld, nx, c1);
}

inline void smf_algebra_launch(cudaStream_t st, const SmfAlgArgs& a, int nb) {
  smf_algebra_kernel<<<dim3(nb, a.passes), SMF_ALG_THREADS, 2 * a.nx * sizeof(double), st>>>(a);
}

// one CTA per sample slot of the batch (samples b >= a.nb return at once)
inline void smf_posterior_launch(cudaStream_t st, const SmfPostArgs& a, int nslots) {
  smf_posterior_kernel<<<nslots, SMF_ALG_THREADS, 3 * a.nx * sizeof(double), st>>>(a);
}

}  // namespace cg

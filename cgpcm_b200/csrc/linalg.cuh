// Dense FP64 linear algebra on the device: the M x M part of the ELBO (M = nh, nx <= 4096), the replacements of
// tf.cholesky / tf.cholesky_solve / tf.matrix_triangular_solve / log_det (src/core/tf_util.py:98-105,134-138,271-278;
// used at src/core/cgpcm.py:214-229,535 and src/core/distribution.py:60-76), and the factorisations of the sampling
// and scoring paths: order <= 8192 (filter draws), <= 4096 (AKM draws, predictive draws) and <= 4104 (the bordered
// scoring matrix).  Everything runs on one stream, no host round trips; a failed factorisation is reported through a
// device-side info word, tag * 100000 + the first non-positive pivot + 1 (the first failing launch sets it; checked
// once per evaluation).
//
// All matrices are square row-major with leading dimension ld and a *padded* order np (multiple
// of 8, np <= ld): callers put the identity on the padding block so that factor / inverse / logdet of
// the padded matrix equal those of the logical one.
//
//   potrf_lower   blocked right-looking Cholesky, NB = 32: a panel kernel (diagonal block factored in
//                 shared memory by every CTA, row blocks solved one thread per row) + DMMA trailing
//                 update.  Leaves a clean lower-triangular factor (upper triangle zeroed).
//                 Every CTA of a panel launch reads the UNFACTORED diagonal block from A; CTA 0 therefore does not
//                 write the factored block into A (a late-scheduled CTA would read it half-written) but into a
//                 scratch slot, and the next panel launch copies it into place before doing anything else (the
//                 last panel has a single CTA and writes A directly).  No launch is added.
//   trtri_lower   inverse of the factor: diagonal blocks in shared memory, block rows by two DMMA GEMMs.
//   cholinv       A^{-1} = X^T X with X = L^{-1}.
#pragma once
#include "dgemm_dmma.cuh"

namespace cg {

constexpr int LA_NB = 32;
constexpr int LA_ROWS = 128;  // panel rows per CTA

// grid.x = 1 + ceil(rows_below / LA_ROWS); block = 256
__global__ void __launch_bounds__(256) potrf_panel_kernel(double* __restrict__ A, int np, long ld, int j0, int jb,
                                                          int* __restrict__ info, int info_tag,
                                                          double* __restrict__ scratch, int flush_j0, int flush_jb,
                                                          int defer) {
  __shared__ double D[LA_NB][LA_NB + 1];
  __shared__ double P[LA_ROWS][LA_NB + 1];
  __shared__ int bad;
  const int tid = threadIdx.x;
  if (tid == 0) bad = 0;
  if (blockIdx.x == 0 && flush_jb > 0) {
    // the previous panel's factored diagonal block: scratch -> A (nobody reads that block during this launch)
    for (int e = tid; e < flush_jb * flush_jb; e += blockDim.x) {
      int r = e / flush_jb, c = e % flush_jb;
      A[(long)(flush_j0 + r) * ld + flush_j0 + c] = scratch[r * LA_NB + c];
    }
  }
  for (int e = tid; e < LA_NB * LA_NB; e += blockDim.x) {
    int r = e / LA_NB, c = e % LA_NB;
    D[r][c] = (r < jb && c < jb && c <= r) ? A[(long)(j0 + r) * ld + j0 + c] : (r == c ? 1.0 : 0.0);
  }
  __syncthreads();
  // factor D in place (lower), column by column
  for (int j = 0; j < jb; ++j) {
    if (tid == 0) {
      double d = D[j][j];
      if (!(d > 0.0)) { if (!bad) bad = j + 1; d = 1.0; }
      D[j][j] = sqrt(d);
    }
    __syncthreads();
    const double djj = D[j][j];
    for (int r = j + 1 + tid; r < jb; r += blockDim.x) D[r][j] /= djj;
    __syncthreads();
    // trailing update of the block: thread (ty, tx) takes rows j + 1 + ty (+8 ..), column j + 1 + tx -- no index
    // divisions (ncu: the e / m, e % m form of this loop was 36 k of the kernel's 47 k warp instructions, 70 k cycles
    // per panel); every element still receives its updates in the order j = 0, 1, ..: the factor is bit-identical
    {
      const int tx = tid & 31, ty = tid >> 5;
      const int cc = j + 1 + tx;
      if (cc < jb) {
        const double lc = D[cc][j];
        for (int r = j + 1 + ty; r < jb; r += 8)
          if (cc <= r) D[r][cc] -= D[r][j] * lc;
      }
    }
    __syncthreads();
  }
  if (blockIdx.x == 0) {
    if (tid == 0 && bad && info) atomicCAS(info, 0, info_tag * 100000 + j0 + bad);
    for (int e = tid; e < jb * jb; e += blockDim.x) {
      int r = e / jb, c = e % jb;
      const double v = (c <= r) ? D[r][c] : 0.0;
      if (defer) scratch[r * LA_NB + c] = v;
      else A[(long)(j0 + r) * ld + j0 + c] = v;
    }
    return;
  }
  // rows below the diagonal block: X L^T = P
  const int r0 = j0 + jb + (blockIdx.x - 1) * LA_ROWS;
  const int nr = min(LA_ROWS, np - r0);
  if (nr <= 0) return;
  for (int e = tid; e < nr * jb; e += blockDim.x) {
    int r = e / jb, c = e % jb;
    P[r][c] = A[(long)(r0 + r) * ld + j0 + c];
  }
  __syncthreads();
  if (tid < nr) {
    for (int c = 0; c < jb; ++c) {
      double v = P[tid][c];
      for (int m = 0; m < c; ++m) v -= P[tid][m] * D[c][m];
      P[tid][c] = v / D[c][c];
    }
  }
  __syncthreads();
  for (int e = tid; e < nr * jb; e += blockDim.x) {
    int r = e / jb, c = e % jb;
    A[(long)(r0 + r) * ld + j0 + c] = P[r][c];
    A[(long)(j0 + c) * ld + r0 + r] = 0.0;   // clean upper triangle
  }
}

// scratch: LA_NB * LA_NB doubles (not aliased with A)
inline cudaError_t potrf_lower(cudaStream_t st, double* A, int np, long ld, int* info, int info_tag, double* scratch) {
  int flush_j0 = 0, flush_jb = 0;
  for (int j0 = 0; j0 < np; j0 += LA_NB) {
    int jb = np - j0 < LA_NB ? np - j0 : LA_NB;
    int below = np - j0 - jb;
    int nblk = 1 + (below + LA_ROWS - 1) / LA_ROWS;
    const int defer = nblk > 1;       // other CTAs of this launch read the unfactored block from A
    potrf_panel_kernel<<<nblk, 256, 0, st>>>(A, np, ld, j0, jb, info, info_tag, scratch, flush_j0, flush_jb, defer);
    flush_j0 = j0;
    flush_jb = defer ? jb : 0;
    if (below > 0) {
      const double* Pn = A + (long)(j0 + jb) * ld + j0;
      double* C = A + (long)(j0 + jb) * ld + (j0 + jb);
      cudaError_t e = dgemm(st, true, true, false, below, below, jb, -1.0, Pn, ld, Pn, ld, 1.0, C, ld, 1, 0, 1);
      if (e != cudaSuccess) return e;
    }
  }
  return cudaGetLastError();
}

// Batched Cholesky of window blocks of one symmetric matrix: CTA b factors  W_b = sign * M[k_lo : k_lo + kw, same]
// (rows / columns >= kv are padding: identity) in shared memory and writes the TRANSPOSED factor, the upper-triangular
// S_b[l][k] = L_b[k][l], dense kw x kw at out + off_b -- the resident operand of dgemm_sl_tri.  The windows are the
// chunks' windows of inducing inputs: W_b = iKx[window] (sign +1) or -C1bar[window] (sign -1), both positive definite.
struct WinDesc { int k_lo, kw, kv; long off; };

__global__ void __launch_bounds__(256) window_chol_kernel(const double* __restrict__ M, long ld, double sign,
                                                          const WinDesc* __restrict__ desc, double* __restrict__ out,
                                                          int* __restrict__ info, int info_tag) {
  extern __shared__ double Wsm[];
  __shared__ int bad;
  const WinDesc d = desc[blockIdx.x];
  const int n = d.kw, P = n + 1, tid = threadIdx.x;
  if (tid == 0) bad = 0;
  for (int e = tid; e < n * n; e += blockDim.x) {
    const int r = e / n, c = e - r * n;
    double v = r == c ? 1.0 : 0.0;
    if (r < d.kv && c < d.kv) v = sign * M[(long)(d.k_lo + r) * ld + d.k_lo + c];
    Wsm[r * P + c] = v;
  }
  __syncthreads();
  const int tx = tid & 31, ty = tid >> 5;
  for (int j = 0; j < n; ++j) {
    if (tid == 0) {
      double dj = Wsm[j * P + j];
      if (!(dj > 0.0)) { if (!bad) bad = j + 1; dj = 1.0; }
      Wsm[j * P + j] = sqrt(dj);
    }
    __syncthreads();
    const double djj = Wsm[j * P + j];
    for (int r = j + 1 + tid; r < n; r += blockDim.x) Wsm[r * P + j] /= djj;
    __syncthreads();
    for (int c = j + 1 + tx; c < n; c += 32) {
      const double lc = Wsm[c * P + j];
      for (int r = j + 1 + ty; r < n; r += 8)
        if (c <= r) Wsm[r * P + c] -= Wsm[r * P + j] * lc;
    }
    __syncthreads();
  }
  if (tid == 0 && bad && info) atomicCAS(info, 0, info_tag * 100000 + d.k_lo + bad);
  double* o = out + d.off;
  for (int e = tid; e < n * n; e += blockDim.x) {
    const int l = e / n, k = e - l * n;
    o[e] = k >= l ? Wsm[k * P + l] : 0.0;
  }
}

inline cudaError_t window_chol(cudaStream_t st, const double* M, long ld, double sign, const WinDesc* desc_d, int count,
                               int kw_max, double* out, int* info, int info_tag) {
  static DeviceOnce attr_once;
  unsigned long long attr_bit;
  if (attr_once.need(&attr_bit)) {
    cudaFuncSetAttribute((const void*)window_chol_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 121 * 8);
    attr_once.done(attr_bit);
  }
  if (count <= 0) return cudaSuccess;
  window_chol_kernel<<<count, 256, (size_t)kw_max * (kw_max + 1) * sizeof(double), st>>>(M, ld, sign, desc_d, out, info, info_tag);
  return cudaGetLastError();
}

// X diagonal blocks = inverse of the diagonal blocks of L; rest of X zeroed.  grid = number of blocks.
__global__ void __launch_bounds__(256) trtri_diag_kernel(const double* __restrict__ L, double* __restrict__ X, int np,
                                                         long ld) {
  __shared__ double D[LA_NB][LA_NB + 1];
  __shared__ double Xs[LA_NB][LA_NB + 1];
  const int j0 = blockIdx.x * LA_NB;
  const int jb = min(LA_NB, np - j0);
  const int tid = threadIdx.x;
  for (int e = tid; e < LA_NB * LA_NB; e += blockDim.x) {
    int r = e / LA_NB, c = e % LA_NB;
    D[r][c] = (r < jb && c < jb) ? L[(long)(j0 + r) * ld + j0 + c] : (r == c ? 1.0 : 0.0);
    Xs[r][c] = 0.0;
  }
  __syncthreads();
  if (tid < jb) {
    const int c = tid;   // solve L x = e_c
    for (int r = c; r < jb; ++r) {
      double v = (r == c) ? 1.0 : 0.0;
      for (int m = c; m < r; ++m) v -= D[r][m] * Xs[m][c];
      Xs[r][c] = v / D[r][r];
    }
  }
  __syncthreads();
  // zero this block row of X left/right of the diagonal block, then write the block
  for (int e = tid; e < jb * np; e += blockDim.x) {
    int r = e / np, c = e % np;
    double v = 0.0;
    if (c >= j0 && c < j0 + jb) v = Xs[r][c - j0];
    X[(long)(j0 + r) * ld + c] = v;
  }
}

// X = L^{-1} (lower).  W: workspace of at least LA_NB * ld doubles.
inline cudaError_t trtri_lower(cudaStream_t st, const double* L, double* X, double* W, int np, long ld) {
  int nb = (np + LA_NB - 1) / LA_NB;
  trtri_diag_kernel<<<nb, 256, 0, st>>>(L, X, np, ld);
  for (int i = 1; i < nb; ++i) {
    int i0 = i * LA_NB;
    int ib = np - i0 < LA_NB ? np - i0 : LA_NB;
    // W[ib x i0] = L[i, 0:i0] * X[0:i0, 0:i0]
    cudaError_t e = dgemm(st, true, false, false, ib, i0, i0, 1.0, L + (long)i0 * ld, ld, X, ld, 0.0, W, ld);
    if (e != cudaSuccess) return e;
    // X[i, 0:i0] = -X_ii * W
    e = dgemm(st, true, false, false, ib, i0, ib, -1.0, X + (long)i0 * ld + i0, ld, W, ld, 0.0, X + (long)i0 * ld, ld);
    if (e != cudaSuccess) return e;
  }
  return cudaGetLastError();
}

// out[0] = 2 * sum_i log L[i][i]   (single CTA, deterministic)
__global__ void logdet_kernel(const double* __restrict__ L, int n, long ld, double* __restrict__ out) {
  __shared__ double sh[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += log(L[(long)i * ld + i]);
  for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0;
    for (int w = 0; w < (int)((blockDim.x + 31) >> 5); ++w) a += sh[w];
    out[0] = 2.0 * a;
  }
}

// Identity on the padding block [n, np) (rows and columns cleared), or zero (after inversion).
__global__ void pad_block_kernel(double* __restrict__ A, int n, int np, long ld, double diag) {
  long total = (long)np * np;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    int r = (int)(idx / np), c = (int)(idx % np);
    if (r >= n || c >= n) A[(long)r * ld + c] = (r == c) ? diag : 0.0;
  }
}

// L (in place over A, padded identity), Ainv, optional logdet.  X, W: np x ld workspaces.
inline cudaError_t cholinv(cudaStream_t st, double* A, double* Ainv, double* X, double* W, int n, int np, long ld,
                           double* logdet_out, int* info, int info_tag) {
  int blocks = (int)(((long)np * np + 255) / 256);
  pad_block_kernel<<<blocks, 256, 0, st>>>(A, n, np, ld, 1.0);
  cudaError_t e = potrf_lower(st, A, np, ld, info, info_tag, X);
  if (e != cudaSuccess) return e;
  if (logdet_out) logdet_kernel<<<1, 256, 0, st>>>(A, n, ld, logdet_out);
  if (Ainv) {
    e = trtri_lower(st, A, X, W, np, ld);
    if (e != cudaSuccess) return e;
    e = dgemm(st, false, false, false, np, np, np, 1.0, X, ld, X, ld, 0.0, Ainv, ld);
    if (e != cudaSuccess) return e;
    pad_block_kernel<<<blocks, 256, 0, st>>>(Ainv, n, np, ld, 0.0);
  }
  return cudaGetLastError();
}

// ---- generic element-wise / reduction helpers (extended lambdas) ---------------------------------
template <class F>
__global__ void ew_kernel(long total, F f) {
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) f(idx);
}
template <class F>
inline void ew(cudaStream_t st, long total, F f) {
  if (total <= 0) return;
  long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  ew_kernel<<<(int)blocks, 256, 0, st>>>(total, f);
}
// out[0] = sum_{idx < total} f(idx): one CTA of 1024 threads, fixed order => deterministic.
template <class F>
__global__ void __launch_bounds__(1024) reduce_kernel(long total, F f, double* out) {
  __shared__ double sh[32];
  double s = 0.0;
  for (long idx = threadIdx.x; idx < total; idx += blockDim.x) s += f(idx);
  for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    double a = sh[threadIdx.x];
    for (int off = 16; off > 0; off >>= 1) a += __shfl_down_sync(0xffffffffu, a, off);
    if (threadIdx.x == 0) out[0] = a;
  }
}
template <class F>
inline void reduce_to(cudaStream_t st, long total, F f, double* out) {
  reduce_kernel<<<1, 1024, 0, st>>>(total, f, out);
}

}  // namespace cg

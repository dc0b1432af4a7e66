// FP64 tensor-core GEMM for sm_100a (DMMA.8x8x4 via mma.sync.m8n8k4.f64), the contraction engine
// of the VCGPCM hot path: the reference's batched `tf.matmul` contractions over observations
// (src/core/cgpcm.py:255-267, :473-475) become four plain GEMMs per chunk of observations
// (DESIGN.md §3).  tcgen05 has no f64 kind, so DMMA is the FP64 tensor path on B200; its measured
// peak (tools/fp64_peaks.cu) is 37.2 TFLOP/s = 64 FMA/clk/SM, fed comfortably by cp.async.
//
// C[M x N] = alpha * op(A)[M x K] * op(B)[K x N] + beta * C, all FP64.
//   A_KC : A(m,k) at A[m*lda + k]  (k contiguous)    else A[k*lda + m]  (m contiguous)
//   B_KC : B(k,n) at B[n*ldb + k]  (k contiguous)    else B[k*ldb + n]  (n contiguous)
//   C_TR : C(m,n) at C[n*ldc + m]                    else C[m*ldc + n]
// Requirements: M, N multiples of 8; K, lda, ldb, ldc even; 16-byte aligned pointers.
//
// Tiling: CTA tile = bm x 64 x 16 with bm = 32, 56 or 104 rows (pick_mb) chosen so that M splits
// evenly (M = 200 -> two tiles of 104/96 rows: 96 % useful instead of 78 % with 128-row tiles).
// 128 threads: 4 warps side by side along N; each warp owns all (<= 13) 8-row blocks x two 8-column
// blocks = 26 DMMA per k4 step with 52 FP64 accumulators, so every SM sub-partition carries the
// same tensor work.  Shared-memory strides are == 4 (mod 8) doubles: conflict-free fragment loads.
// 3-stage cp.async pipeline (zero-filled at every edge).  Split-K over blockIdx.z writes partial
// results C + z * c_split_stride (reduced by reduce_partials) so that sums stay deterministic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "device_once.cuh"

namespace cg {

constexpr int G_BM = 104;      // max rows per CTA tile
constexpr int G_MB = 13;       // max 8-row blocks per CTA tile
constexpr int G_BN = 64;       // 4 warps x 16 columns
constexpr int G_BK = 16;
constexpr int G_STAGES = 3;
constexpr int G_THREADS = 128;
constexpr int G_CTAS_PER_SM = 2;  // two co-resident CTAs: one's prologue / epilogue overlaps the other's DMMA loop
constexpr int G_AS = (G_BM * (G_BK + 4) > G_BK * (G_BM + 4)) ? G_BM * (G_BK + 4) : G_BK * (G_BM + 4);
constexpr int G_BS = (G_BN * (G_BK + 4) > G_BK * (G_BN + 4)) ? G_BN * (G_BK + 4) : G_BK * (G_BN + 4);
constexpr int G_SMEM_BYTES = G_STAGES * (G_AS + G_BS) * 8;

struct GemmArgs {
  const double* A;
  const double* B;
  double* C;
  int M, N, K;
  long lda, ldb, ldc;
  double alpha, beta;
  int splits;           // number of K splits (third tile-list dimension)
  int k_per_split;      // multiple of G_BK
  long c_split_stride;  // elements between split-K partial results
  int lower_only;       // skip CTA tiles that lie strictly above the diagonal (symmetric results)
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem, bool valid) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void dmma_8x8x4(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// One CTA = one (split, row tile, column tile).  Compile-time number MB of 8-row blocks per tile: every loop
// is fully unrolled and every shared-memory fragment address is `thread base + immediate`.  Rows / columns
// beyond the matrix edge are zero-filled in shared memory (cp.async src-size 0) and not stored.
// The operand fragments are double-buffered in registers (load k4+1 while the DMMAs of k4 issue): with a
// single buffer every LDS has to wait for the in-flight DMMA that still reads its destination register.
// The cp.async source pointers / shared offsets are computed once per CTA and only advanced per k-tile.
template <int MB, bool A_KC, bool B_KC, bool C_TR>
__device__ __forceinline__ void dgemm_body(const GemmArgs& g, double* smem, const int m0, const int tile_rows) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int grp = lane >> 2, tig = lane & 3;
  const int nw = warp * 16;
  constexpr int STAGE = G_AS + G_BS;
  constexpr int TROWS = MB * 8;
  const int n0 = blockIdx.x * G_BN;
  if (g.lower_only && n0 > m0 + tile_rows - 1) return;
  const int rows = g.M - m0, cols = g.N - n0;     // valid rows / columns from the tile origin (may exceed tile)
  const int kbeg = blockIdx.z * g.k_per_split;
  const int kend = min(g.K, kbeg + g.k_per_split);
  const int ktiles = kend > kbeg ? (kend - kbeg + G_BK - 1) / G_BK : 0;

  // ---- loader state: NA + NB 16-byte chunks per thread per k-tile
  constexpr int NCH_A = A_KC ? TROWS * (G_BK / 2) : G_BK * (TROWS / 2);
  constexpr int NA = (NCH_A + G_THREADS - 1) / G_THREADS;
  constexpr int NCH_B = G_BN * G_BK / 2;
  constexpr int NB = NCH_B / G_THREADS;
  const double* ga[NA];
  int sa[NA];        // shared offset (doubles) inside a stage, or -1 if this slot is unused
  int ka[NA];        // k offset of the chunk inside the k-tile
  const double* gb[NB];
  int sb[NB], kb[NB];
#pragma unroll
  for (int j = 0; j < NA; ++j) {
    const int ch = j * G_THREADS + tid;
    if (A_KC) {
      const int m = ch / (G_BK / 2), kc = (ch % (G_BK / 2)) * 2;
      const bool ok = ch < NCH_A && m < rows;
      sa[j] = ch < NCH_A ? m * (G_BK + 4) + kc : -1;
      ka[j] = ok ? kc : (1 << 28);
      ga[j] = g.A + (ok ? (long)(m0 + m) * g.lda + kbeg + kc : 0);
    } else {
      constexpr int HALF = TROWS / 2;
      const int kk = ch / HALF, mc = (ch - kk * HALF) * 2;
      const bool ok = ch < NCH_A && mc < rows;
      sa[j] = ch < NCH_A ? kk * (G_BM + 4) + mc : -1;
      ka[j] = ok ? kk : (1 << 28);
      ga[j] = g.A + (ok ? (long)(kbeg + kk) * g.lda + m0 + mc : 0);
    }
  }
#pragma unroll
  for (int j = 0; j < NB; ++j) {
    const int ch = j * G_THREADS + tid;
    if (B_KC) {
      const int n = ch / (G_BK / 2), kc = (ch % (G_BK / 2)) * 2;
      const bool ok = n < cols;
      sb[j] = G_AS + n * (G_BK + 4) + kc;
      kb[j] = ok ? kc : (1 << 28);
      gb[j] = g.B + (ok ? (long)(n0 + n) * g.ldb + kbeg + kc : 0);
    } else {
      constexpr int HALF = G_BN / 2;
      const int kk = ch / HALF, nc = (ch - kk * HALF) * 2;
      const bool ok = nc < cols;
      sb[j] = G_AS + kk * (G_BN + 4) + nc;
      kb[j] = ok ? kk : (1 << 28);
      gb[j] = g.B + (ok ? (long)(kbeg + kk) * g.ldb + n0 + nc : 0);
    }
  }
  const long a_step = A_KC ? G_BK : (long)G_BK * g.lda;
  const long b_step = B_KC ? G_BK : (long)G_BK * g.ldb;
  int kleft = kend - kbeg;       // k extent not yet issued
  auto issue = [&](int stage) {
    double* base = smem + stage * STAGE;
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      if (NCH_A % G_THREADS == 0 || sa[j] >= 0) {
        const bool ok = ka[j] < kleft;
        cp_async16(base + sa[j], ok ? ga[j] : g.A, ok);
        ga[j] += a_step;
      }
    }
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      const bool ok = kb[j] < kleft;
      cp_async16(base + sb[j], ok ? gb[j] : g.B, ok);
      gb[j] += b_step;
    }
    kleft -= G_BK;
  };

#pragma unroll
  for (int s0 = 0; s0 < G_STAGES - 1; ++s0) {
    if (s0 < ktiles) issue(s0);
    cp_async_commit();
  }

  const int a_off = A_KC ? grp * (G_BK + 4) + tig : tig * (G_BM + 4) + grp;
  const int b_off = G_AS + (B_KC ? (nw + grp) * (G_BK + 4) + tig : tig * (G_BN + 4) + nw + grp);
  const bool warp_live = nw < cols;

  double acc[MB][2][2];
#pragma unroll
  for (int i = 0; i < MB; ++i) { acc[i][0][0] = acc[i][0][1] = acc[i][1][0] = acc[i][1][1] = 0.0; }

  auto load_frags = [&](const double* Ap, const double* Bp, int k4, double (&a)[MB], double (&b)[2]) {
    b[0] = B_KC ? Bp[k4 * 4] : Bp[k4 * 4 * (G_BN + 4)];
    b[1] = B_KC ? Bp[8 * (G_BK + 4) + k4 * 4] : Bp[k4 * 4 * (G_BN + 4) + 8];
#pragma unroll
    for (int mb = 0; mb < MB; ++mb)
      a[mb] = A_KC ? Ap[mb * 8 * (G_BK + 4) + k4 * 4] : Ap[k4 * 4 * (G_BM + 4) + mb * 8];
  };

  int stage = 0;
  for (int kt = 0; kt < ktiles; ++kt) {
    cp_async_wait<G_STAGES - 2>();
    __syncthreads();
    {
      int st2 = stage + G_STAGES - 1;
      if (st2 >= G_STAGES) st2 -= G_STAGES;
      if (kt + G_STAGES - 1 < ktiles) issue(st2);
      cp_async_commit();
    }
    if (warp_live) {
      const double* Ap = smem + stage * STAGE + a_off;
      const double* Bp = smem + stage * STAGE + b_off;
      const int k4n = (kend - kbeg - kt * G_BK + 3) >> 2;      // k4 steps with data in this k-tile (last one may be short)
      double fa[2][MB], fb[2][2];
      load_frags(Ap, Bp, 0, fa[0], fb[0]);
#pragma unroll
      for (int k4 = 0; k4 < G_BK / 4; ++k4) {
        if (k4 + 1 < G_BK / 4) load_frags(Ap, Bp, k4 + 1, fa[(k4 + 1) & 1], fb[(k4 + 1) & 1]);
        if (k4 == 0 || k4 < k4n) {
#pragma unroll
          for (int mb = 0; mb < MB; ++mb) {
            dmma_8x8x4(acc[mb][0][0], acc[mb][0][1], fa[k4 & 1][mb], fb[k4 & 1][0]);
            dmma_8x8x4(acc[mb][1][0], acc[mb][1][1], fa[k4 & 1][mb], fb[k4 & 1][1]);
          }
        }
      }
    }
    if (++stage == G_STAGES) stage = 0;
  }
  cp_async_wait<0>();

  double* C = g.C + (long)blockIdx.z * g.c_split_stride;
  const bool nb_ok0 = nw < cols, nb_ok1 = nw + 8 < cols;
#pragma unroll
  for (int mb = 0; mb < MB; ++mb) {
    if (mb * 8 >= rows) continue;
    const int row = m0 + mb * 8 + grp;
#pragma unroll
    for (int nb = 0; nb < 2; ++nb) {
      if (nb == 0 ? !nb_ok0 : !nb_ok1) continue;
      const int col = n0 + nw + nb * 8 + tig * 2;
      double v0 = g.alpha * acc[mb][nb][0], v1 = g.alpha * acc[mb][nb][1];
      if (!C_TR) {
        double2* p = reinterpret_cast<double2*>(C + (long)row * g.ldc + col);
        if (g.beta != 0.0) {
          double2 o = *p;
          v0 += g.beta * o.x;
          v1 += g.beta * o.y;
        }
        *p = make_double2(v0, v1);
      } else {
        double* p0 = C + (long)col * g.ldc + row;
        double* p1 = p0 + g.ldc;
        if (g.beta != 0.0) {
          v0 += g.beta * *p0;
          v1 += g.beta * *p1;
        }
        *p0 = v0;
        *p1 = v1;
      }
    }
  }
}

// Row tiles are MB blocks high; the last row tile of the matrix may use the lower body MBL (M = 200: 13 + 12
// blocks, no padded rows).
template <int MB, int MBL, bool A_KC, bool B_KC, bool C_TR>
__global__ void __launch_bounds__(G_THREADS, G_CTAS_PER_SM) dgemm_dmma_kernel(const GemmArgs g) {
  extern __shared__ __align__(16) double smem[];
  const int m0 = blockIdx.y * (MB * 8);
  if (MBL != MB && m0 + MBL * 8 >= g.M) dgemm_body<MBL, A_KC, B_KC, C_TR>(g, smem, m0, MB * 8);
  else dgemm_body<MB, A_KC, B_KC, C_TR>(g, smem, m0, MB * 8);
}

// out[r][c] (+)= sum_s part[s][r][c]  (deterministic split-K reduction); optional mirroring of the
// lower triangle into the upper one for results computed with lower_only.
__global__ void reduce_partials_kernel(const double* __restrict__ part, long split_stride, int splits,
                                       double* __restrict__ out, int rows, int cols, long ld_part,
                                       long ld_out, double beta, int mirror_lower) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  long total = (long)rows * cols;
  if (idx >= total) return;
  int r = (int)(idx / cols), c = (int)(idx % cols);
  int rr = r, cc = c;
  if (mirror_lower && c > r) { rr = c; cc = r; }
  double s = 0.0;
  for (int k = 0; k < splits; ++k) s += part[(long)k * split_stride + (long)rr * ld_part + cc];
  double* o = out + (long)r * ld_out + c;
  *o = (beta != 0.0 ? beta * *o : 0.0) + s;
}

// Rows per CTA tile: the smallest supported block count (4 / 7 / 13 blocks of 8 rows) whose tiles cover M
// with the fewest padded rows.
inline int pick_mb(int M) {
  const int cand[3] = {4, 7, 13};
  int best = 13;
  long best_cost = -1;
  for (int i = 0; i < 3; ++i) {
    int rows = cand[i] * 8;
    long tiles = (M + rows - 1) / rows;
    long cost = tiles * rows;                     // rows of DMMA work issued
    if (best_cost < 0 || cost < best_cost || (cost == best_cost && cand[i] > best)) { best = cand[i]; best_cost = cost; }
  }
  return best;
}
inline int pick_bm(int M) { return pick_mb(M) * 8; }

// Launch.  Returns cudaError_t of the launch.
inline cudaError_t dgemm(cudaStream_t st, bool a_kc, bool b_kc, bool c_tr, int M, int N, int K, double alpha,
                         const double* A, long lda, const double* B, long ldb, double beta, double* C,
                         long ldc, int splits = 1, long c_split_stride = 0, int lower_only = 0) {
  if (M <= 0 || N <= 0) return cudaSuccess;
  GemmArgs g;
  g.A = A; g.B = B; g.C = C; g.M = M; g.N = N; g.K = K;
  g.lda = lda; g.ldb = ldb; g.ldc = ldc; g.alpha = alpha; g.beta = beta;
  const int mb = pick_mb(M);
  if (splits < 1) splits = 1;
  int kt = (K + G_BK - 1) / G_BK;
  int kt_per = (kt + splits - 1) / splits;
  if (kt_per < 1) kt_per = 1;
  g.splits = splits;
  g.k_per_split = kt_per * G_BK;
  g.c_split_stride = c_split_stride;
  g.lower_only = lower_only;
  const int rows = mb * 8;
  dim3 grid((N + G_BN - 1) / G_BN, (M + rows - 1) / rows, splits);
  // last row tile exactly 12 blocks high (M = 200, 408, ...): use the 13 / 12 pair
  const bool pair12 = mb == 13 && (M - (int)(grid.y - 1) * rows) == 96;
  static DeviceOnce attr_once;
  unsigned long long attr_bit;
#define CG_ATTR(MBV, MBLV, AK, BK, CT) \
  cudaFuncSetAttribute((const void*)dgemm_dmma_kernel<MBV, MBLV, AK, BK, CT>, cudaFuncAttributeMaxDynamicSharedMemorySize, G_SMEM_BYTES);
#define CG_ATTR4(MBV, MBLV) CG_ATTR(MBV, MBLV, true, true, false) CG_ATTR(MBV, MBLV, true, false, false) \
  CG_ATTR(MBV, MBLV, false, false, false) CG_ATTR(MBV, MBLV, true, true, true)
  if (attr_once.need(&attr_bit)) {
    CG_ATTR4(4, 4) CG_ATTR4(7, 7) CG_ATTR4(13, 13) CG_ATTR4(13, 12)
    CG_ATTR(13, 13, false, true, false) CG_ATTR(13, 13, true, false, true) CG_ATTR(13, 13, false, true, true)
    CG_ATTR(13, 13, false, false, true)
    attr_once.done(attr_bit);
  }
#undef CG_ATTR4
#undef CG_ATTR
#define CG_LAUNCH(MBV, MBLV, AK, BK, CT) dgemm_dmma_kernel<MBV, MBLV, AK, BK, CT><<<grid, G_THREADS, G_SMEM_BYTES, st>>>(g)
#define CG_PICK(AK, BK, CT)                              \
  do {                                                   \
    if (mb == 4) CG_LAUNCH(4, 4, AK, BK, CT);            \
    else if (mb == 7) CG_LAUNCH(7, 7, AK, BK, CT);       \
    else if (pair12) CG_LAUNCH(13, 12, AK, BK, CT);      \
    else CG_LAUNCH(13, 13, AK, BK, CT);                  \
  } while (0)
  // the four layouts the ELBO path uses come in every tile height; the others (C-ABI export only) in one
  if (!c_tr) {
    if (a_kc && b_kc) CG_PICK(true, true, false);
    else if (a_kc && !b_kc) CG_PICK(true, false, false);
    else if (!a_kc && !b_kc) CG_PICK(false, false, false);
    else { grid.y = (M + 103) / 104; CG_LAUNCH(13, 13, false, true, false); }
  } else {
    if (a_kc && b_kc) CG_PICK(true, true, true);
    else {
      grid.y = (M + 103) / 104;
      if (a_kc && !b_kc) CG_LAUNCH(13, 13, true, false, true);
      else if (!a_kc && b_kc) CG_LAUNCH(13, 13, false, true, true);
      else CG_LAUNCH(13, 13, false, false, true);
    }
  }
#undef CG_PICK
#undef CG_LAUNCH
  return cudaGetLastError();
}

}  // namespace cg

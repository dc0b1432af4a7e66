// libcgpcm_b200.so — host side of the C-ABI declared in include/cgpcm_b200.h.
//
// One handle = one GPU + one stream.  An evaluation (cgpcm_elbo_grad) is
//
//   1. M x M prologue      prior kernels, Choleskys / inverses, q(u) moments          (linalg.cuh)
//   2. forward sweep       sum_n Axx (+ tangents) in one launch; per chunk of observations the Ahx
//                          block A[i][n][k] is generated into HBM and contracted by four DMMA GEMMs
//                          into C1 = sum_n A_n^T H A_n, Q = sum_n A_n iKx A_n^T, Y = sum_n y_n A_n
//   3. all-reduce #1       one packed ncclAllReduce of the forward partials (multi-GPU only)
//   4. M x M algebra       P, its Cholesky / inverse, the 7 ELBO terms, the adjoints that seed the
//                          backward sweep (SURVEY.md App. D)
//   5. backward sweep      per chunk: regenerate A, Hbar = sum_n A_n C1bar A_n^T, Abar = H A_n Wx, and
//                          the contraction of Abar with dA/d(alpha, gamma, omega) on the fly
//   6. all-reduce #2       Hbar + 3 scalars
//   7. M x M epilogue      closing adjoint chain, gradient assembly.
//
// This replaces `sess.run([elbo, grad])` of the TF graph built by src/core/cgpcm.py:518-575 (ELBO),
// :458-477 (_optimal_q), :231-268 (model matrices), :214-229 (prior kernels) and
// src/core/distribution.py:60-76 (KL), differentiated by tf.gradients.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/cgpcm_b200.h"
#include "dgemm_sl.cuh"
#include "dgemm_sym.cuh"
#include "gram_kernels.cuh"
#include "linalg.cuh"
#include "predict_kernels.cuh"
#include "psi_kernels.cuh"
#include "smf_batch.cuh"

using namespace cg;

// ------------------------------------------------------------------------------------------------
// NCCL through dlopen: the library has no link-time dependency on NCCL; inside a torch process the
// already-loaded libnccl.so.2 is reused.
// ------------------------------------------------------------------------------------------------
namespace {

typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { NCCL_INT32 = 2, NCCL_DOUBLE = 8, NCCL_SUM = 0, NCCL_MAX = 2 };

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};

NcclApi& nccl() {
  static NcclApi api;
  static bool tried = false;
  if (tried) return api;
  tried = true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (api.lib) break;
  }
  if (!api.lib) return api;
  api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.lib, "ncclGetUniqueId");
  api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.lib, "ncclCommInitRank");
  api.AllReduce = (decltype(api.AllReduce))dlsym(api.lib, "ncclAllReduce");
  api.AllGather = (decltype(api.AllGather))dlsym(api.lib, "ncclAllGather");
  api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
  api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.lib, "ncclGetErrorString");
  api.ok = api.GetUniqueId && api.CommInitRank && api.AllReduce && api.AllGather && api.CommDestroy;
  return api;
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// matrix slots (each ld x ld doubles)
enum Mat {
  M_KH0, M_LH, M_IKH, M_KX0, M_KX, M_LX, M_IKX, M_AHH, M_DAHH_A, M_DAHH_G,
  M_AXX0, M_AXX1, M_AXX2, M_AXX3,          // sum_Axx and its tangents  } packed contiguously: the
  M_C1, M_Q, M_Y,                          //                            } forward all-reduce buffer
  M_HBAR,                                  // backward all-reduce buffer (+ 3 scalars behind it)
  M_LQ, M_VAR, M_LVAR, M_IVAR, M_M2, M_H, M_S, M_LP, M_PINV, M_PBAR, M_C1BAR, M_WX, M_YBAR,
  M_SO, M_ISO, M_BHH, M_M2BAR, M_T1, M_T2, M_T3, M_XW, M_WW, M_XW2, M_WW2, M_XW3, M_WW3,
  M_F_AXX, M_F_BHH, M_F_Y, M_F_IKH,        // frozen ("precomputed") Psi sums
  M_COUNT
};

// vector slots (each ld doubles)
enum Vec { V_MU, V_YTMU, V_LAM, V_LBAR, V_ISOMU, V_MUBAR, V_YLBAR, V_M2BMU, V_MUZ, V_SMP, V_COUNT };

// device scalars
enum Sc {
  S_LOGDET_KX, S_LOGDET_P, S_LOGDET_SO, S_LOGDET_VAR, S_TR_IKH_AHH, S_TR_IKX_AXX, S_TR_IKH_Q, S_TR_BHH_M2,
  S_TR_ISO_VAR, S_MU_ISO_MU, S_LAM_LBAR, S_PBAR_S, S_C0BAR, S_G_KH_A, S_G_KH_G, S_G_KX_O, S_G_AHH_A,
  S_G_AHH_G, S_G_AXX_A, S_G_AXX_G, S_G_AXX_O, S_LOGDET_P0, S_LAM_LBAR0, S_S_BHH_S, S_LOGDET_KH, S_COUNT
};

constexpr int AXX_MAX_SLICES = 64;    // slice-private partial sums: 64 x 4 x ld^2 doubles (82 MB at M = 200)

struct Chunk {
  long n0;      // first observation
  int nv;       // valid observations
  int nc;       // padded observation count (multiple of 8)
  int k_lo;     // first inducing input of the window (even)
  int kwp;      // padded window width (multiple of 8)
  long off;     // element offset of this chunk's block in the sweep stores (prefix sum of nhp * nc * kwp)
};

}  // namespace

struct cgpcm_handle {
  int device = 0;
  cudaStream_t st = nullptr;
  int nh = 0, nx = 0, nhp = 0, nxp = 0;
  long ld = 0;
  int causal = 1, causal_id = 0;
  // data
  double *t = nullptr, *y = nullptr, *th = nullptr, *tx = nullptr;
  long n_local = 0;
  std::vector<double> h_t, h_th, h_tx;
  bool t_sorted = false;
  double sum_y2_local = 0.0;
  // options
  int chunk = 512;          // observations per chunk at full window width
  double cull = 80.0;       // 0 = dense
  bool chunk_auto = true;   // option "chunk" <= 0 (default): plan_chunks picks 512 / 1024 / 2048 by its cost model
  int profile = 0;          // 1 = CUDA events around every GEMM launch (roofline measurement)
  int pw_dists = 0;         // 1 = prior kernels from |x|^2 - 2xy + |y|^2 as the reference forms them (psi_kernels.cuh)
  std::vector<cudaEvent_t> pev;
  size_t pev_used = 0;
  std::vector<char> pev_kind;  // per event pair: 0 = contraction GEMMs (a run of consecutive launches), 1 = Ahx generation
  bool prof_open = false;      // a GEMM run is being timed: its closing event is recorded before the next other kernel
  double gemm_flops = 0.0;  // algorithmic flops of the GEMM launches of the last evaluation (symmetric: M(M+1)K)
  double gemm_flops_exec = 0.0;   // flops of the CTA / warp tiles those launches computed
  long gemm_launches = 0;
  // memory
  double* mats = nullptr;
  double* vecs = nullptr;
  double* sc = nullptr;        // S_COUNT scalars
  double* fwd_tail = nullptr;  // [n, sum_y2] lives behind M_Y in the packed forward buffer
  int* info = nullptr;
  double* params_d = nullptr;
  double* gvar_d = nullptr;    // packed gradient of var_u
  // chunk workspaces
  long ws_elems = 0;
  double *wsA = nullptr, *wsT = nullptr, *wsV = nullptr;
  // sweep stores (option "store", default on when they fit): the Ahx blocks of all chunks (storeA) and
  // T1 = H A of the forward sweep (storeT) stay resident in HBM for the backward sweep instead of being
  // regenerated / recomputed -- 8 nhp N nx bytes each (32 GB at N = 1e5, M = 200; the B200 has 180 GB).
  int sep_opt = 1;             // 1: separable Ahx kernels for the default causal model (psi_kernels.cuh)
  int last_info_tag = 0;       // matrix of the last failed factorisation (evaluate)
  int tri_opt = 1;             // 1: Q / Hbar through the Cholesky factors of the window blocks (window_factors below)
  double* wfac = nullptr;      // transposed factors of the chunks' window blocks, kwp x kwp each, back to back
  long wfac_elems = 0;
  WinDesc* wdesc = nullptr;
  long wdesc_count = 0;
  int sl_opt = 1;              // 1: contractions with a small left operand run on the persistent kernel (dgemm_sl.cuh)
  int sms = 148;
  int store_opt = 1;
  double *storeA = nullptr, *storeT = nullptr;
  long storeA_elems = 0, storeT_elems = 0;
  bool use_store = false;      // decided per evaluation
  bool storeA_frozen_valid = false;   // storeA holds the frozen regime's Ahx blocks (constant between evaluations)
  // prior kernels of the precomputed regime: Kh, Kx, their factors and inverses only depend on (alpha, gamma, omega,
  // reg), which are constants between cgpcm_precompute and the next full-regime call -- MODE_FROZEN evaluations,
  // fixed-point rounds, SMF samples and predictions reuse them instead of refactoring (2 x ~40 launches) every time
  bool prior_valid = false;
  double prior_key[4] = {0, 0, 0, 0};
  // fourth-order Psi tensor of the frozen regime (gram_kernels.cuh), option "gram": 0 off (default), 1 when it pays,
  // 2 whenever it fits.  Opt-in: the contraction with m2 ~ iKh cancels AFTER the sum over observations instead of
  // before it, which costs ~sqrt(N) in rounding noise (gram_kernels.cuh).
  int gram_opt = 0;
  double* gram = nullptr;
  long gram_elems = 0;
  bool gram_valid = false;
  double* symacc[2] = {nullptr, nullptr};   // per-K-slice private accumulators of the symmetric contractions
  int sym_used[2] = {0, 0};                 // slices touched since sym_begin
  double* axx_part = nullptr;
  long axx_part_elems = 0;
  double* cheb_d = nullptr;    // Chebyshev table of the pair-hoisted BVN branch (bvn.cuh)
  // batched SMF scoring (cgpcm_elbo_smf_batch): one allocation for the samples, W = H_B A of a chunk, the slice partials
  // and C1 slabs, the factor slabs and the per-sample scalars; info words of the factorisations
  double* smf_buf = nullptr;
  long smf_elems = 0;
  int* smf_info = nullptr;
  int smf_info_count = 0;
  int axx_slices = 0;
  int axx_slices_opt = 0;      // option "axx_slices": 0 = automatic (axx_sweep)
  double* ypart = nullptr;     // [slices][nhp][ld] private Y accumulators
  int y_slices = 0;
  double* gpart = nullptr;     // partial sums of <Abar, dA/dtheta>
  long gpart_elems = 0;
  // frozen state
  bool frozen = false;
  PsiConst fc;
  double f_a = 0.0, f_sum_b = 0.0;
  // comm
  ncclComm_t comm = nullptr;
  bool own_comm = false;
  int rank = 0, world = 1;
  // bookkeeping
  std::string err;
  double timing[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  long launches = 0;
  cudaEvent_t ev[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // [7], [8]: before all-reduce #1 / #2
  // Side streams for the M x M factor / inverse chains that do not sit on the critical path of an evaluation: the
  // chains of Kh and Kx run beside each other (and beside the Axx sweep, which needs neither), those of the prior
  // covariance iKh + reg I and of the q(u) covariance beside the forward sweep.  Only the chain of P (which needs the
  // reduced sums) stays on the main stream.  Each chain has its own workspaces (M_XW*, M_WW*).
  cudaStream_t side[2] = {nullptr, nullptr};
  cudaEvent_t sev_fork[2] = {nullptr, nullptr};
  cudaEvent_t sev_join[2] = {nullptr, nullptr};
  bool prior_pending = false;                 // the prior chains have been forked and not yet joined

  double* M(int id) const { return mats + (long)id * ld * ld; }
  double* V(int id) const { return vecs + (long)id * ld; }
};

namespace {

#define CK(call)                                                                      \
  do {                                                                                \
    cudaError_t e_ = (call);                                                          \
    if (e_ != cudaSuccess) {                                                          \
      char buf_[512];                                                                 \
      snprintf(buf_, sizeof buf_, "CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_), __FILE__, __LINE__, #call); \
      h->err = buf_;                                                                  \
      return -2;                                                                      \
    }                                                                                 \
  } while (0)

bool is_device_ptr(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// ---- small kernels ------------------------------------------------------------------------------

// y[r] = alpha * sum_c op(A)[r][c] x[c]; one warp per row.
__global__ void matvec_kernel(const double* __restrict__ A, long ld, int rows, int cols, int trans,
                              const double* __restrict__ x, double alpha, double* __restrict__ y) {
  int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (r >= rows) return;
  double s = 0.0;
  for (int c = lane; c < cols; c += 32) s += (trans ? A[(long)c * ld + r] : A[(long)r * ld + c]) * x[c];
  for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
  if (lane == 0) y[r] = alpha * s;
}

void matvec(cgpcm_handle* h, const double* A, int rows, int cols, int trans, const double* x, double alpha,
            double* y) {
  matvec_kernel<<<(rows + 7) / 8, 256, 0, h->st>>>(A, h->ld, rows, cols, trans, x, alpha, y);
  h->launches++;
}

// Sum of the slice-private Axx partials into four full symmetric ld x ld matrices.
__global__ void axx_reduce_kernel(const double* __restrict__ part, int slices, int nmat, long ld, int nx,
                                  double* __restrict__ out) {
  long mat = ld * ld;
  long total = nmat * mat;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    int m = (int)(idx / mat);
    long e = idx % mat;
    int r = (int)(e / ld), c = (int)(e % ld);
    double s = 0.0;
    if (r < nx && c < nx) {
      int rr = r >= c ? r : c, cc = r >= c ? c : r;
      const double* p = part + (long)m * mat + (long)rr * ld + cc;
      for (int k = 0; k < slices; ++k) s += p[(long)k * 4 * mat];
    }
    out[idx] = s;
  }
}

// Y[i][k] = sum_s Ypart[s][i][k]
__global__ void ypart_reduce_kernel(const double* __restrict__ part, int slices, long stride, long total,
                                    double* __restrict__ out) {
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int k = 0; k < slices; ++k) s += part[(long)k * stride + idx];
    out[idx] = s;
  }
}

__global__ void sum3_kernel(const double* __restrict__ gpart, long n, double* __restrict__ out) {
  __shared__ double sh[3][32];
  double a0 = 0, a1 = 0, a2 = 0;
  for (long i = threadIdx.x; i < n; i += blockDim.x) {
    a0 += gpart[3 * i];
    a1 += gpart[3 * i + 1];
    a2 += gpart[3 * i + 2];
  }
  for (int off = 16; off > 0; off >>= 1) {
    a0 += __shfl_down_sync(0xffffffffu, a0, off);
    a1 += __shfl_down_sync(0xffffffffu, a1, off);
    a2 += __shfl_down_sync(0xffffffffu, a2, off);
  }
  int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { sh[0][w] = a0; sh[1][w] = a1; sh[2][w] = a2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double b0 = 0, b1 = 0, b2 = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { b0 += sh[0][i]; b1 += sh[1][i]; b2 += sh[2][i]; }
    out[0] = b0; out[1] = b1; out[2] = b2;
  }
}

__global__ void sumsq_kernel(const double* __restrict__ y, long n, double* __restrict__ out, int* __restrict__ bad,
                             const double* __restrict__ t) {
  __shared__ double sh[32];
  double s = 0.0;
  int nf = 0;
  for (long i = threadIdx.x; i < n; i += blockDim.x) {
    double v = y[i];
    s += v * v;
    if (!isfinite(v) || !isfinite(t[i])) nf = 1;
  }
  if (nf) atomicExch(bad, 1);
  for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) a += sh[i];
    out[0] = a;
  }
}

// ---- GEMM helper --------------------------------------------------------------------------------

int pick_splits(int Mr, int Nr, int K, bool lower) {
  // number of CTA tiles the launch computes per split
  const int bm = pick_bm(Mr);
  int tiles = 0;
  for (int m0 = 0; m0 < Mr; m0 += bm)
    for (int n0 = 0; n0 < Nr; n0 += G_BN)
      if (!(lower && n0 > m0 + bm - 1)) ++tiles;
  const int kt = (K + G_BK - 1) / G_BK;
  const int max_by_k = kt / 8 > 0 ? kt / 8 : 1;   // at least 8 k-tiles per split
  // two full waves of 148 CTAs (one CTA per SM) when K is long enough, else one
  int s = 296 / tiles;
  if (s < 1) s = 1;
  if (kt / s < 48) s = std::max(1, 148 / tiles);
  return std::min(s, max_by_k);
}

}  // namespace

// The lambdas below are extended __device__ lambdas: they must live in functions with external linkage.
namespace cgimpl {

using ::cgpcm_handle;

cudaEvent_t prof_event(cgpcm_handle* h, int kind);
// Option "profile": consecutive GEMM launches share one event pair (an event pair per launch cost 3.7 ms per
// evaluation at the bench shape).  prof_gemm_begin opens the run; prof_close ends it -- explicitly before the Psi
// kernels of the sweeps, and after any other (small) kernel through L().
inline void prof_gemm_begin(cgpcm_handle* h) {
  if (h->profile && !h->prof_open) { cudaEventRecord(prof_event(h, 0), h->st); h->prof_open = true; }
}
inline void prof_close(cgpcm_handle* h) {
  if (h->prof_open) { cudaEventRecord(prof_event(h, 0), h->st); h->prof_open = false; }
}
inline void L(cgpcm_handle* h, int n = 1) { prof_close(h); h->launches += n; }

// out[0] = sum_{r<rows, c<cols} A[r][c] * B[r][c]
void frob(cgpcm_handle* h, const double* A, const double* B, int rows, int cols, double* out) {
  const int ld = (int)h->ld;
  reduce_to(h->st, (long)rows * cols, [=] __device__(long idx) {
    const int r = (int)idx / cols, c = (int)idx - r * cols;      // rows * cols < 2^31: 32-bit division
    return A[r * ld + c] * B[r * ld + c];
  }, out);
  L(h);
}

void dot(cgpcm_handle* h, const double* a, const double* b, int n, double* out) {
  reduce_to(h->st, (long)n, [=] __device__(long i) { return a[i] * b[i]; }, out);
  L(h);
}

void zero(cgpcm_handle* h, double* p, long n) { cudaMemsetAsync(p, 0, n * sizeof(double), h->st); }

// ---- bookkeeping shared by the runs -------------------------------------------------------------

// Device scratch of one call: take(n) reserves a slice of n elements (aligned to 256 bytes, as cudaMalloc aligns; the
// DMMA paths need 16) and returns its byte offset, alloc() makes one cudaMalloc, and the destructor frees it.
struct Scratch {
  size_t bytes = 0;
  char* base = nullptr;
  Scratch() = default;
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;
  ~Scratch() { if (base) cudaFree(base); }
  size_t take(size_t n, size_t elem = sizeof(double)) {
    const size_t o = bytes;
    bytes += (n * elem + 255) / 256 * 256;
    return o;
  }
  cudaError_t alloc() { return bytes ? cudaMalloc(&base, bytes) : cudaSuccess; }
  template <class T = double> T* at(size_t off) const { return (T*)(base + off); }
};

// The hyper-parameters of params_host[0..4] (log s2, log s2_f, log alpha, log gamma, log omega) and the two ratios of
// the bound: r = s2_f / s2, c0 = sqrt(s2_f) / s2.
struct Hyp {
  double s2, s2f, alpha, gamma, omega, r, c0;
};
Hyp hyp_of(const double* p) {
  Hyp q;
  q.s2 = exp(p[0]); q.s2f = exp(p[1]);
  q.alpha = exp(p[2]); q.gamma = exp(p[3]); q.omega = exp(p[4]);
  q.r = q.s2f / q.s2; q.c0 = sqrt(q.s2f) / q.s2;
  return q;
}

// Start of a run: reset the launch, profile and GEMM counters, record ev[0] and clear the info word.
int begin_run(cgpcm_handle* h) {
  h->launches = 0;
  h->pev_used = 0;
  h->prof_open = false;
  h->gemm_flops = h->gemm_flops_exec = 0.0;
  h->gemm_launches = 0;
  CK(cudaEventRecord(h->ev[0], h->st));
  CK(cudaMemsetAsync(h->info, 0, 4 * sizeof(int), h->st));
  return 0;
}

// End of a run: close the profiled GEMM run, record ev[6], wait for the stream and fetch the info word.
int end_run(cgpcm_handle* h, int& info) {
  int w[4];
  CK(cudaMemcpyAsync(w, h->info, sizeof w, cudaMemcpyDeviceToHost, h->st));
  prof_close(h);
  CK(cudaEventRecord(h->ev[6], h->st));
  CK(cudaStreamSynchronize(h->st));
  CK(cudaGetLastError());
  info = w[0];
  return 0;
}

// cgpcm_last_timing of a run: [0] ev[0] -> ev[6] in ms, [6] launches, [7] GEMM flops, [8] GEMM launches, [9] executed
// GEMM flops; the rest 0.
void record_timing(cgpcm_handle* h) {
  float ms = 0;
  cudaEventElapsedTime(&ms, h->ev[0], h->ev[6]);
  memset(h->timing, 0, sizeof h->timing);
  h->timing[0] = ms;
  h->timing[6] = (double)h->launches;
  h->timing[7] = h->gemm_flops;
  h->timing[8] = (double)h->gemm_launches;
  h->timing[9] = h->gemm_flops_exec;
}

// A failed factorisation reported by the info word (tag * 100000 + pivot), named from the run's table: the prior
// kernels are refactored next time, and the run returns -3.
template <int N>
int pd_error(cgpcm_handle* h, int info, const char* const (&names)[N]) {
  if (!info) return 0;
  h->prior_valid = false;
  const int tag = info / 100000;
  char b[160];
  snprintf(b, sizeof b, "matrix %s is not positive definite (pivot %d)", tag >= 1 && tag < N ? names[tag] : "?",
           info % 100000);
  h->err = b;
  return -3;
}

// A failed per-sample factorisation (the prior is not involved).
int sample_pd_error(cgpcm_handle* h, const char* what, int sample, int pivot) {
  char b[160];
  snprintf(b, sizeof b, "matrix %s of sample %d is not positive definite (pivot %d)", what, sample, pivot);
  h->err = b;
  return -3;
}

// -4 with `msg` unless p[0..n) are all finite.
int check_finite(cgpcm_handle* h, const double* p, long n, const char* msg) {
  for (long i = 0; i < n; ++i)
    if (!std::isfinite(p[i])) { h->err = msg; return -4; }
  return 0;
}

// The same for B samples of nh values, naming the first sample with a non-finite value.
int check_samples(cgpcm_handle* h, const double* s, long B, int nh) {
  for (long i = 0; i < B * nh; ++i)
    if (!std::isfinite(s[i])) {
      char b[96];
      snprintf(b, sizeof b, "non-finite value in sample %ld", i / nh);
      h->err = b;
      return -4;
    }
  return 0;
}

// n values of a user buffer (host or device) into v.
int to_host(cgpcm_handle* h, const double* src, long n, std::vector<double>& v) {
  v.resize(n);
  if (is_device_ptr(src)) CK(cudaMemcpy(v.data(), src, n * sizeof(double), cudaMemcpyDeviceToHost));
  else memcpy(v.data(), src, n * sizeof(double));
  return 0;
}

// n host values into a user buffer (host or device; nothing when dst is NULL).
int put(cgpcm_handle* h, double* dst, const double* src, long n) {
  if (!dst || n == 0) return 0;
  if (is_device_ptr(dst)) CK(cudaMemcpy(dst, src, n * sizeof(double), cudaMemcpyHostToDevice));
  else memcpy(dst, src, n * sizeof(double));
  return 0;
}

// Shared argument checks of the entry points: the data (`data`: h->t, or h->th where only the inducing inputs are
// needed) has been set and reg is usable.
int check_call(cgpcm_handle* h, const double* data, double reg) {
  if (!data) { h->err = "cgpcm_set_data has not been called"; return -1; }
  if (!std::isfinite(reg) || reg < 0) { h->err = "reg must be finite and >= 0"; return -4; }
  return 0;
}

cudaEvent_t prof_event(cgpcm_handle* h, int kind) {
  if ((h->pev_used & 1) == 0) {
    if (h->pev_kind.size() <= h->pev_used / 2) h->pev_kind.resize(h->pev_used / 2 + 1);
    h->pev_kind[h->pev_used / 2] = (char)kind;
  }
  if (h->pev_used == h->pev.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    h->pev.push_back(e);
  }
  return h->pev[h->pev_used++];
}

// GEMM flop counters of one dgemm launch.  executed: the CTA tiles this launch computes (tiles strictly above the
// diagonal are skipped when lower); algorithmic: M x N cells, or the M (M + 1) / 2 cells of the lower triangle of a
// symmetric result
void gemm_count(cgpcm_handle* h, int Mr, int Nr, int K, int lower) {
  const int bm = pick_bm(Mr);
  double cells = 0.0;
  for (int m0 = 0; m0 < Mr; m0 += bm)
    for (int n0 = 0; n0 < Nr; n0 += G_BN) {
      if (lower && n0 > m0 + bm - 1) continue;
      cells += (double)std::min(bm, Mr - m0) * std::min(G_BN, Nr - n0);
    }
  h->gemm_flops_exec += 2.0 * cells * K;
  h->gemm_flops += 2.0 * K * ((lower && Mr == Nr) ? 0.5 * Mr * (Mr + 1.0) : (double)Mr * Nr);
}

int gemm(cgpcm_handle* h, bool a_kc, bool b_kc, bool c_tr, int Mr, int Nr, int K, double alpha, const double* A,
         long lda, const double* B, long ldb, double beta, double* C, long ldc, int splits = 1, long stride = 0,
         int lower = 0) {
  gemm_count(h, Mr, Nr, K, lower);
  h->gemm_launches++;
  prof_gemm_begin(h);
  cudaError_t e;
  if (h->sl_opt && a_kc && b_kc == c_tr && splits <= 1 && !lower && beta == 0.0 && dgemm_sl_supported(Mr, Nr, K))
    e = dgemm_sl(h->st, b_kc, Mr, Nr, K, alpha, A, lda, B, ldb, C, ldc, h->sms);
  else
    e = dgemm(h->st, a_kc, b_kc, c_tr, Mr, Nr, K, alpha, A, lda, B, ldb, beta, C, ldc, splits, stride, lower);
  h->launches++;
  if (e != cudaSuccess) {
    h->err = std::string("dgemm launch failed: ") + cudaGetErrorString(e);
    return -2;
  }
  return 0;
}

// square ld x ld product on padded sizes
int mm(cgpcm_handle* h, const double* A, bool ta, const double* B, bool tb, double* C, int Mr, int Nr, int K,
       double alpha = 1.0, double beta = 0.0) {
  // A(m,k): stored A[m*ld+k] (a_kc) unless transposed; B(k,n): stored B[k*ld+n] (!b_kc) unless transposed
  return gemm(h, !ta, tb, false, Mr, Nr, K, alpha, A, h->ld, B, h->ld, beta, C, h->ld);
}

// ws: 0 = main stream, 1 / 2 = side stream 0 / 1 (own workspaces)
int chol_inv_on(cgpcm_handle* h, int ws, double* A, double* Ainv, int n, int np, double* logdet, int tag) {
  cudaStream_t st = ws == 0 ? h->st : h->side[ws - 1];
  const int xw = ws == 0 ? M_XW : ws == 1 ? M_XW2 : M_XW3;
  cudaError_t e = cholinv(st, A, Ainv, h->M(xw), h->M(xw + 1), n, np, h->ld, logdet, h->info, tag);
  h->launches += 40;
  if (e != cudaSuccess) {
    h->err = std::string("cholinv launch failed: ") + cudaGetErrorString(e);
    return -2;
  }
  return 0;
}

// side stream k continues after everything issued to the main stream so far / the main stream after side stream k
int side_fork(cgpcm_handle* h, int k) {
  CK(cudaEventRecord(h->sev_fork[k], h->st));
  CK(cudaStreamWaitEvent(h->side[k], h->sev_fork[k], 0));
  return 0;
}
int side_join(cgpcm_handle* h, int k) {
  CK(cudaEventRecord(h->sev_join[k], h->side[k]));
  CK(cudaStreamWaitEvent(h->st, h->sev_join[k], 0));
  return 0;
}

int chol_inv(cgpcm_handle* h, double* A, double* Ainv, int n, int np, double* logdet, int tag) {
  cudaError_t e = cholinv(h->st, A, Ainv, h->M(M_XW), h->M(M_WW), n, np, h->ld, logdet, h->info, tag);
  L(h, 40);
  if (e != cudaSuccess) {
    h->err = std::string("cholinv launch failed: ") + cudaGetErrorString(e);
    return -2;
  }
  return 0;
}

// ---- chunk planning -----------------------------------------------------------------------------

double ahx_radius(const PsiConst& c, double cull) {
  // E(th, d) <= -(e_dd - e_hd^2 / (4 e_hh)) d^2 for every th
  double lam = c.e_dd - c.e_hd * c.e_hd / (4.0 * c.e_hh);
  if (!(lam > 0.0) || !(cull > 0.0)) return INFINITY;
  return sqrt(cull / lam);
}

void plan_chunks_fixed(cgpcm_handle* h, const PsiConst& c, int chunk, std::vector<Chunk>& out, bool snap = false) {
  out.clear();
  const long N = h->n_local;
  const double R = ahx_radius(c, h->cull);
  const long budget = (long)chunk * h->nxp;    // columns (n, k) per row i
  long n0 = 0;
  auto window = [&](long a, long b, int& k_lo, int& kwp) {
    if (!std::isfinite(R)) { k_lo = 0; kwp = h->nxp; return; }
    double tmin = INFINITY, tmax = -INFINITY;
    if (h->t_sorted) { tmin = h->h_t[a]; tmax = h->h_t[b - 1]; }
    else for (long n = a; n < b; ++n) { tmin = std::min(tmin, h->h_t[n]); tmax = std::max(tmax, h->h_t[n]); }
    int lo = h->nx, hi = -1;
    for (int k = 0; k < h->nx; ++k) {
      double x = h->h_tx[k];
      if (x >= tmin - R && x <= tmax + R) { lo = std::min(lo, k); hi = std::max(hi, k); }
    }
    if (hi < lo) { k_lo = 0; kwp = 8; return; }   // nothing in range: a token all-zero window
    // The window starts at an EVEN inducing input (every kernel needs 16-byte aligned rows of the window blocks, not
    // more) and is a multiple of 8 wide (DMMA row blocks).  Starting it at a multiple of 8 wasted up to 7 columns:
    // whether a chunk got a 96- or a 104-wide window then depended on where its shard happened to begin.
    k_lo = lo / 2 * 2;
    kwp = round_up(hi + 1 - k_lo, 8);
    if (kwp >= h->nxp) { k_lo = 0; kwp = h->nxp; }
    else if (k_lo + kwp > h->nxp) k_lo = h->nxp - kwp;
  };
  while (n0 < N) {
    long rem = N - n0;
    int nc = (int)std::min<long>(rem, chunk);
    int k_lo, kwp;
    window(n0, n0 + nc, k_lo, kwp);
    if (kwp < h->nxp && nc < rem) {
      // narrower window: take more observations for the same workspace
      for (int it = 0; it < 4; ++it) {
        long cand = std::min<long>(rem, budget / kwp / 32 * 32);
        if (cand < 32) cand = std::min<long>(rem, 32);
        int k2, w2;
        window(n0, n0 + cand, k2, w2);
        if (cand * w2 <= budget) { nc = (int)cand; k_lo = k2; kwp = w2; break; }
        kwp = w2;
      }
    }
    if (snap && std::isfinite(R) && kwp > 16 && nc >= 256 && nc < rem) {
      // windows come in steps of 8 inducing inputs: the largest chunk (>= 60 % of this one) whose window is one step
      // narrower costs ~8 / kwp fewer flops per observation for a few more chunks -- the planner's model decides
      long lo_n = (long)(0.6 * nc) / 32 * 32, hi_n = (nc - 1) / 32 * 32;
      int k2, w2;
      window(n0, n0 + std::max<long>(lo_n, 32), k2, w2);
      if (lo_n >= 32 && w2 <= kwp - 8) {
        long best_n = lo_n;
        int best_k = k2, best_w = w2;
        while (lo_n < hi_n) {                       // largest multiple of 32 in (lo_n, hi_n] that keeps the narrower window
          const long mid = ((lo_n + hi_n) / 2 + 31) / 32 * 32;
          window(n0, n0 + mid, k2, w2);
          if (w2 <= kwp - 8) { lo_n = mid; best_n = mid; best_k = k2; best_w = w2; }
          else hi_n = mid - 32;
        }
        nc = (int)best_n; k_lo = best_k; kwp = best_w;
      }
    }
    Chunk ch;
    ch.n0 = n0; ch.nv = nc; ch.nc = round_up(nc, 8); ch.k_lo = k_lo; ch.kwp = kwp;
    ch.off = out.empty() ? 0 : out.back().off + (long)h->nhp * out.back().nc * out.back().kwp;
    out.push_back(ch);
    n0 += nc;
  }
}

// Workspace budget of a chunk (columns = budget x nxp).  More observations per chunk mean fewer, longer launches (the
// persistent GEMM kernels lose ~0.2 ms per chunk to ragged tile counts, pipeline ramps and launch gaps) but a wider
// union window, i.e. more flops: measured at the bench shape, exact-zero windows, 127.6 / 126.3 / 120.0 / 131.1 / 140.0 ms
// for 512 / 1024 / 2048 / 3072 / 4096, while cull = 80 (narrow windows, which widen relatively more) is fastest at 512.
// With option "chunk" <= 0 (default) the planner evaluates the candidates with that cost model and keeps the cheapest;
// the model only depends on the plan, so the frozen regime plans the same chunks at every evaluation.
constexpr int CHUNK_AUTO_MAX = 2048;
inline int chunk_cap(const cgpcm_handle* h) { return h->chunk_auto ? CHUNK_AUTO_MAX : h->chunk; }

void plan_chunks(cgpcm_handle* h, const PsiConst& c, std::vector<Chunk>& out) {
  if (!h->chunk_auto) plan_chunks_fixed(h, c, h->chunk, out);
  double best = INFINITY;
  std::vector<Chunk> cand;
  for (int pass = 0; h->chunk_auto && pass < 6; ++pass) {
    const int chunk = pass / 2 == 0 ? 512 : pass / 2 == 1 ? 1024 : CHUNK_AUTO_MAX;
    plan_chunks_fixed(h, c, chunk, cand, (pass & 1) != 0);
    double cost = 0.0;
    for (const Chunk& ch : cand) {
      const double el = (double)ch.nc * h->nhp * ch.kwp;                       // Ahx elements of the chunk
      cost += el * (4.0 * h->nhp + 7.0 * ch.kwp) / 27e12 + el * 1.5e-11 + 0.21e-3;   // contractions + Psi kernels + per chunk
    }
    if (cost < best) { best = cost; out.swap(cand); h->chunk = chunk; }
  }
  if (getenv("CGPCM_DEBUG_PLAN")) {
    fprintf(stderr, "plan: n_local %ld, budget %d, %zu chunks:", (long)h->n_local, h->chunk, out.size());
    for (const Chunk& ch : out) fprintf(stderr, " (%d x %d @%d)", ch.nv, ch.kwp, ch.k_lo);
    fprintf(stderr, "\n");
  }
}

// Decide whether this evaluation keeps the Ahx blocks (and T1 when `need_t`) of all chunks resident, and
// size the stores.  Falls back to regenerate / recompute when the device does not have the room.
int plan_store(cgpcm_handle* h, const std::vector<Chunk>& chunks, bool need_t) {
  h->use_store = false;
  if (!h->store_opt || chunks.empty()) return 0;
  const Chunk& last = chunks.back();
  const long total = last.off + (long)h->nhp * last.nc * last.kwp;
  auto grow = [&](double*& buf, long& have) -> int {
    if (have >= total) return 0;
    if (buf) { cudaFree(buf); buf = nullptr; have = 0; h->storeA_frozen_valid = false; }
    size_t free_b = 0, tot_b = 0;
    if (cudaMemGetInfo(&free_b, &tot_b) != cudaSuccess) { cudaGetLastError(); return 1; }
    if ((double)total * sizeof(double) > 0.45 * (double)free_b) return 1;    // leave room for the other store + scratch
    if (cudaMalloc(&buf, total * sizeof(double)) != cudaSuccess) { cudaGetLastError(); buf = nullptr; return 1; }
    have = total;
    return 0;
  };
  if (grow(h->storeA, h->storeA_elems)) return 0;
  if (need_t && grow(h->storeT, h->storeT_elems)) return 0;
  h->use_store = true;
  return 0;
}

int ensure_ws(cgpcm_handle* h) {
  long need = (long)h->nhp * (round_up(chunk_cap(h), 32) + 32) * h->nxp;
  if (need > h->ws_elems) {
    if (h->wsA) { cudaFree(h->wsA); cudaFree(h->wsT); cudaFree(h->wsV); }
    h->wsA = h->wsT = h->wsV = nullptr;
    CK(cudaMalloc(&h->wsA, need * sizeof(double)));
    CK(cudaMalloc(&h->wsT, need * sizeof(double)));
    CK(cudaMalloc(&h->wsV, need * sizeof(double)));
    h->ws_elems = need;
  }
  return 0;
}

// ---- sweeps ---------------------------------------------------------------------------------------

// ---- launches of the sweeps' kernels (handle-free: the sweeps and the C-ABI test hooks share them) -----------------

// sum_n Axx (and tangents) of the n observations t -> out4 (1 or 4 ld x ld matrices): axx_sum_kernel into the slice
// partials part ([slices][4][ld][ld]), then axx_reduce_kernel.  cheb: device room for the Chebyshev table of the
// pair-hoisted branch.  Two launches.
cudaError_t axx_launch(cudaStream_t st, const double* t, int n, bool sorted, const double* tx, int nx, double* part,
                       long ld, int slices, const PsiConst& c, const BvnTab& T, double* cheb, bool tangents,
                       double* out4) {
  const int nt = (nx + AXX_TILE - 1) / AXX_TILE;
  const int ntiles = nt * nt;        // 16 inducing inputs x 16 separations per tile (psi_kernels.cuh)
  // pair-hoisted Genz branch: causal model, rho >= 0.925 (rho = gamma / A is always positive here)
  const bool hoist = c.causal && !c.causal_id && T.high && T.rho > 0.0 && T.as_ > 0.0 && T.ng == 20;
  dim3 grid(ntiles, slices);
  int deg = 0;
  size_t smem = 0;
  if (hoist) {
    double B[(BVN_CHEB_MAXDEG + 1) * 20];
    deg = bvn_make_cheb(T, B);
    cudaError_t e = cudaMemcpyAsync(cheb, B, (size_t)(deg + 1) * 20 * sizeof(double), cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    smem = (size_t)(deg + 1) * (20 + BVN_PAIR_THREADS) * sizeof(double);
    static DeviceOnce attr_once;
    unsigned long long attr_bit;
    if (attr_once.need(&attr_bit)) {
      const int mx = (BVN_CHEB_MAXDEG + 1) * (20 + BVN_PAIR_THREADS) * 8;
      cudaFuncSetAttribute((const void*)axx_sum_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
      cudaFuncSetAttribute((const void*)axx_sum_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx);
      attr_once.done(attr_bit);
    }
  }
#define CG_AXX(TG, HO) \
  axx_sum_kernel<TG, HO><<<grid, 256, smem, st>>>(t, n, sorted ? 1 : 0, tx, nx, part, ld, c, T, cheb, deg)
  if (tangents) { if (hoist) CG_AXX(true, true); else CG_AXX(true, false); }
  else { if (hoist) CG_AXX(false, true); else CG_AXX(false, false); }
#undef CG_AXX
  axx_reduce_kernel<<<148 * 4, 256, 0, st>>>(part, slices, tangents ? 4 : 1, ld, nx, out4);
  return cudaGetLastError();
}

// Whether ahx_gen_sep_kernel<true> (table-driven erfcx) covers every element for the filter inducing inputs th[0 .. nh)
// (host values) at the constants c.
bool ahx_gen_tab(const PsiConst& c, const double* th_host, int nh) {
  if (nh < 1) return false;
  double lo = th_host[0], hi = th_host[0];
  for (int i = 1; i < nh; ++i) { lo = std::min(lo, th_host[i]); hi = std::max(hi, th_host[i]); }
  return psi_erfcx_tab_covers(c, lo, hi);
}

// A[(i*nc + n)*kwp + k] = Ahx of the chunk's observations t[0 .. nv) at the window k_lo + k (ahx_gen_sep_kernel when
// `sep`: default causal model only; its table-driven erfcx when `tab`, see ahx_gen_tab), and when Ypart != NULL the
// slice partials of sum_n y_n A.  One launch.
void ahx_gen_launch(cudaStream_t st, bool sep, bool tab, const double* t, const double* y, int nv, int nc,
                    const double* th, int nh, int nhp, const double* tx, int nx, int k_lo, int kwp, double* A,
                    double* Ypart, long ldy, long ypart_stride, const PsiConst& c) {
  const int threads = std::min(256, round_up(kwp, 32));
  dim3 grid(nhp, (nc + AHX_NSUB - 1) / AHX_NSUB);
  if (sep) {
    // default causal model: separable form, AHX_IB filter rows per CTA (psi_kernels.cuh)
    grid.x = (nhp + AHX_IB - 1) / AHX_IB;
    if (tab)
      ahx_gen_sep_kernel<true><<<grid, threads, 0, st>>>(t, y, nv, nc, th, nh, nhp, tx, nx, k_lo, kwp, A, Ypart, ldy,
                                                         ypart_stride, c);
    else
      ahx_gen_sep_kernel<false><<<grid, threads, 0, st>>>(t, y, nv, nc, th, nh, nhp, tx, nx, k_lo, kwp, A, Ypart, ldy,
                                                          ypart_stride, c);
  } else {
    ahx_gen_kernel<<<grid, threads, 0, st>>>(t, y, nv, nc, th, nh, tx, nx, k_lo, kwp, A, Ypart, ldy, ypart_stride, c);
  }
}

// gpart[(slice * grid.x + cta) * 3 + theta] += sum (W + y Ybar) dA/dtheta over the chunk's block (ahx_dot_sep_kernel
// when `sep`).  One launch.
void ahx_dot_launch(cudaStream_t st, bool sep, const double* t, const double* y, int nv, int nc, const double* th, int nh,
                    int nhp, const double* tx, int nx, int k_lo, int kwp, const double* A, const double* W,
                    const double* Ybar, long ldy, double* gpart, const PsiConst& c) {
  const int threads = std::min(256, round_up(kwp, 32));
  dim3 grid(nhp, (nc + AHX_NSUB - 1) / AHX_NSUB);
  if (sep) {
    grid.x = (nhp + AHX_IB - 1) / AHX_IB;
    ahx_dot_sep_kernel<<<grid, threads, 0, st>>>(t, y, nv, nc, th, nh, tx, nx, k_lo, kwp, A, W, Ybar, ldy, gpart, c);
  } else {
    ahx_dot_kernel<<<grid, threads, 0, st>>>(t, y, nv, nc, th, nh, tx, nx, k_lo, kwp, A, W, Ybar, ldy, gpart, c);
  }
}

// The symmetric contractions' route: orders <= 40 (one warp block) stay on the tiled split-K kernel (154 us against
// 204 us at the bench shape's cull = 80 window).
inline bool sym_on_dgemm_sym(bool a_kc, bool b_kc, int Mr) {
  return a_kc == b_kc && dgemm_sym_supported(Mr) && Mr > SY_BLK;
}

// Adds the lower triangle of op(A) op(B)^T (Mr x Mr) slice by slice into the K-slice buffers acc (stride ld * ld) at
// element offset win; *splits = the slices the launch touched.  One launch.
cudaError_t sym_accum_launch(cudaStream_t st, bool a_kc, bool b_kc, int Mr, int K, const double* A, long lda,
                             const double* B, long ldb, double* acc, long ld, long win, int* splits) {
  const long l2 = ld * ld;
  double* C = acc + win;
  if (sym_on_dgemm_sym(a_kc, b_kc, Mr)) {
    *splits = dgemm_sym_splits(K);
    return dgemm_sym(st, a_kc, Mr, K, A, lda, B, ldb, C, ld, l2, 1);
  }
  int s = std::min(pick_splits(Mr, Mr, K, true), SY_MAX_SPLITS);
  // number of splits actually used by dgemm (it rounds the k range per split up to whole tiles)
  int kt = (K + G_BK - 1) / G_BK;
  int kt_per = (kt + s - 1) / s;
  s = (kt + kt_per - 1) / kt_per;
  *splits = s;
  return dgemm(st, a_kc, b_kc, false, Mr, Mr, K, 1.0, A, lda, B, ldb, 1.0, C, ld, s, l2, 1);
}

// out (n x n at ld) = sum over the first `slices` K-slice buffers, in slice order, mirrored.  One launch.
void sym_finish_launch(cudaStream_t st, const double* acc, long ld, int slices, int n, double* out) {
  const long total = (long)n * n;
  reduce_partials_kernel<<<(int)((total + 255) / 256), 256, 0, st>>>(acc, ld * ld, std::max(1, slices), out, n, n, ld,
                                                                    ld, 0.0, 1);
}

// sum_n Axx (and tangents) over this rank's observations -> M_AXX0..3
int axx_sweep(cgpcm_handle* h, const PsiConst& c, const BvnTab& T, bool tangents, double* out4) {
  // Observation slices (grid.y).  Fewer slices would amortise the per-pair set-up of the hoisted branch over more
  // observations, but measured slower (13 slices: 15.4 ms against 13.7 ms at the bench shape, 2.59 against 2.32 ms on an
  // 8-GPU shard): the per-CTA observation ranges are cut by the windows, and more, smaller CTAs balance better.
  int slices = h->axx_slices_opt > 0 ? h->axx_slices_opt : h->axx_slices;
  if (h->n_local > 0) {
    prof_close(h);
    CK(axx_launch(h->st, h->t, (int)h->n_local, h->t_sorted, h->tx, h->nx, h->axx_part, h->ld, slices, c, T, h->cheb_d,
                  tangents, out4));
    h->launches += 2;
  } else {
    zero(h, out4, 4 * h->ld * h->ld);
  }
  CK(cudaGetLastError());
  return 0;
}

// y-reduction slices (grid.y of ahx_gen_kernel) the chunks of a sweep touch: only these are zeroed and reduced
int y_slices_used(const std::vector<Chunk>& chunks) {
  int m = 1;
  for (const Chunk& ch : chunks) m = std::max(m, (ch.nc + AHX_NSUB - 1) / AHX_NSUB);
  return m;
}

// slice-private Y accumulators [slices][nhp][ld]: one slice per AHX_NSUB observations of the longest chunk of the plan
int ensure_ypart(cgpcm_handle* h, int slices) {
  if (slices > h->y_slices) {
    if (h->ypart) cudaFree(h->ypart);
    h->ypart = nullptr;
    h->y_slices = 0;
    CK(cudaMalloc(&h->ypart, (long)slices * h->nhp * h->ld * sizeof(double)));
    h->y_slices = slices;
  }
  return 0;
}

int gen_chunk(cgpcm_handle* h, const PsiConst& c, const Chunk& ch, bool with_y, double* dstA = nullptr) {
  if (!dstA) dstA = h->wsA;
  if ((ch.nc + AHX_NSUB - 1) / AHX_NSUB > h->y_slices) { h->err = "internal: y_slices too small"; return -1; }
  prof_close(h);
  if (h->profile) cudaEventRecord(prof_event(h, 1), h->st);
  const bool sep = c.causal && !c.causal_id && h->sep_opt;
  ahx_gen_launch(h->st, sep, sep && ahx_gen_tab(c, h->h_th.data(), h->nh), h->t + ch.n0, h->y + ch.n0, ch.nv, ch.nc,
                 h->th, h->nh, h->nhp, h->tx, h->nx, ch.k_lo, ch.kwp, dstA, with_y ? h->ypart : nullptr, h->ld,
                 (long)h->nhp * h->ld, c);
  if (h->profile) cudaEventRecord(prof_event(h, 1), h->st);
  L(h);
  return 0;
}

// Symmetric contractions, accumulated per K-slice over a whole sweep (dgemm_sym.cuh):
//   sym_begin(slot)            zero the slot's private slice buffers
//   gemm_splitk_sym(.., slot, win)   slice z of this launch adds its Mr x Mr lower triangle into buffer z at window
//                              offset win (= k_lo * ld + k_lo for a window of the full matrix)
//   sym_finish(slot, n, out)   out = sum over slices (fixed order), mirrored to the full symmetric n x n matrix
int sym_begin(cgpcm_handle* h, int slot) {
  CK(cudaMemsetAsync(h->symacc[slot], 0, (size_t)SY_MAX_SPLITS * h->ld * h->ld * sizeof(double), h->st));
  h->sym_used[slot] = 0;
  return 0;
}

int gemm_splitk_sym(cgpcm_handle* h, bool a_kc, bool b_kc, int Mr, int K, const double* A, long lda, const double* B,
                    long ldb, int slot, long win) {
  if (sym_on_dgemm_sym(a_kc, b_kc, Mr)) {
    h->gemm_flops_exec += 2.0 * K * dgemm_sym_cells(Mr);   // full + diagonal warp blocks of the launch's order
    h->gemm_flops += 2.0 * K * 0.5 * Mr * (Mr + 1.0);
  } else {
    gemm_count(h, Mr, Mr, K, 1);
  }
  h->gemm_launches++;
  prof_gemm_begin(h);
  int splits = 1;
  cudaError_t e = sym_accum_launch(h->st, a_kc, b_kc, Mr, K, A, lda, B, ldb, h->symacc[slot], h->ld, win, &splits);
  h->launches++;
  if (e != cudaSuccess) {
    h->err = std::string("symmetric contraction launch failed: ") + cudaGetErrorString(e);
    return -2;
  }
  h->sym_used[slot] = std::max(h->sym_used[slot], splits);
  return 0;
}

int sym_finish(cgpcm_handle* h, int slot, int n, double* out) {
  prof_close(h);
  sym_finish_launch(h->st, h->symacc[slot], h->ld, h->sym_used[slot], n, out);
  L(h);
  return 0;
}

// out[(i,n)][l] = sum_k X[(i,n)][k] W[k][l] for the chunk's window block of a *symmetric* ld x ld matrix W.
// Evaluated as out^T = W X^T with a transposed store, so that the 8-row-block dimension of the CTA tile is
// the window width (split evenly) and the long (i,n) dimension runs along the 128-wide tile columns.
int right_mul_sym(cgpcm_handle* h, const double* X, const double* W, const Chunk& ch, double* out) {
  return gemm(h, true, true, true, ch.kwp, h->nhp * ch.nc, ch.kwp, 1.0, W + (long)ch.k_lo * h->ld + ch.k_lo, h->ld, X,
              ch.kwp, 0.0, out, ch.kwp);
}

// ---- Q = sum_n A_n iKx A_n^T and Hbar = sum_n A_n C1bar A_n^T through Cholesky factors of the window blocks ----------
// Both middle matrices are definite on every window of inducing inputs: iKx[w] = L L^T, -C1bar[w] = r (Pinv / 2 +
// lbar lbar^T / 2)[w] = L L^T.  With V' = A[:, w] L the contraction is the symmetric product V' V'^T, and the
// right-multiply by a TRIANGULAR factor needs 54 % of the DMMAs of the product with the full block (dgemm_sl_tri).  The
// factors of all chunks of a sweep come from one launch of window_chol_kernel (linalg.cuh), one CTA per chunk.
bool tri_eligible(const cgpcm_handle* h, const std::vector<Chunk>& chunks) {
  if (!h->tri_opt || !h->sl_opt || chunks.empty()) return false;
  for (const Chunk& ch : chunks)
    if (!dgemm_sl_tri_supported(ch.kwp, h->nhp * ch.nc)) return false;
  return true;
}

// wfac[off_c ..] = transposed Cholesky factor of sign * M[window of chunk c]; offs[c] = off_c
int window_factors(cgpcm_handle* h, const double* M, double sign, const std::vector<Chunk>& chunks, int tag,
                   std::vector<long>& offs) {
  std::vector<WinDesc> desc(chunks.size());
  offs.resize(chunks.size());
  long off = 0;
  int kw_max = 8;
  for (size_t ci = 0; ci < chunks.size(); ++ci) {
    const Chunk& ch = chunks[ci];
    desc[ci].k_lo = ch.k_lo; desc[ci].kw = ch.kwp; desc[ci].kv = std::max(0, std::min(ch.kwp, h->nx - ch.k_lo));
    desc[ci].off = off;
    offs[ci] = off;
    off += (long)ch.kwp * ch.kwp;
    kw_max = std::max(kw_max, ch.kwp);
  }
  if (off > h->wfac_elems) {
    if (h->wfac) cudaFree(h->wfac);
    h->wfac = nullptr; h->wfac_elems = 0;
    CK(cudaMalloc(&h->wfac, off * sizeof(double)));
    h->wfac_elems = off;
  }
  if ((long)chunks.size() > h->wdesc_count) {
    if (h->wdesc) cudaFree(h->wdesc);
    h->wdesc = nullptr; h->wdesc_count = 0;
    CK(cudaMalloc(&h->wdesc, chunks.size() * sizeof(WinDesc)));
    h->wdesc_count = (long)chunks.size();
  }
  // (pageable source: the copy is staged before the call returns, `desc` may go out of scope)
  CK(cudaMemcpyAsync(h->wdesc, desc.data(), chunks.size() * sizeof(WinDesc), cudaMemcpyHostToDevice, h->st));
  prof_close(h);
  cudaError_t e = window_chol(h->st, M, h->ld, sign, h->wdesc, (int)chunks.size(), kw_max, h->wfac, h->info, tag);
  L(h);
  if (e != cudaSuccess) { h->err = std::string("window_chol launch failed: ") + cudaGetErrorString(e); return -2; }
  return 0;
}

// out[(i,n)][l] = sum_{k <= l ...} X[(i,n)][k] L[k][l]  with St = L^T (upper triangular, kwp x kwp, dense)
int right_mul_tri(cgpcm_handle* h, const double* X, const double* St, const Chunk& ch, double* out) {
  const double full = 2.0 * ch.kwp * ch.kwp * (double)h->nhp * ch.nc;
  h->gemm_flops_exec += full * dgemm_sl_tri_fraction(ch.kwp);
  h->gemm_flops += (double)ch.kwp * (ch.kwp + 1.0) * h->nhp * ch.nc;     // the triangular product
  h->gemm_launches++;
  prof_gemm_begin(h);
  cudaError_t e = dgemm_sl_tri(h->st, ch.kwp, h->nhp * ch.nc, St, ch.kwp, X, ch.kwp, out, ch.kwp, h->sms);
  h->launches++;
  if (e != cudaSuccess) { h->err = std::string("dgemm_sl_tri launch failed: ") + cudaGetErrorString(e); return -2; }
  return 0;
}

// Forward sweep over chunks: C1 += A^T (H A), and when `full`: Q += A iKx A^T, Y += sum y A.
int forward_sweep(cgpcm_handle* h, const PsiConst& c, const std::vector<Chunk>& chunks, const double* Hm,
                  const double* iKx, bool full, bool keep_t) {
  zero(h, h->M(M_C1), h->ld * h->ld);
  if (sym_begin(h, 0)) return -2;
  if (full) {
    zero(h, h->M(M_Q), h->ld * h->ld);
    if (sym_begin(h, 1)) return -2;
    if (ensure_ypart(h, y_slices_used(chunks))) return -2;
    zero(h, h->ypart, (long)y_slices_used(chunks) * h->nhp * h->ld);
  }
  // with the sweep stores the Ahx block (and T1 when the backward sweep will need it) go straight to their
  // resident slots; the frozen regime's blocks do not change between evaluations and are generated once
  const bool st = h->use_store;
  const bool have_a = st && !full && h->storeA_frozen_valid;
  const bool tri = full && tri_eligible(h, chunks);
  std::vector<long> woff;
  if (tri && window_factors(h, iKx, 1.0, chunks, 6, woff)) return -2;
  size_t ci = 0;
  for (const Chunk& ch : chunks) {
    const size_t cidx = ci++;
    double* Ab = st ? h->storeA + ch.off : h->wsA;
    double* Tb = (st && keep_t) ? h->storeT + ch.off : h->wsT;
    if (!have_a && gen_chunk(h, c, ch, full, Ab)) return -2;
    const long cols = (long)ch.nc * ch.kwp;
    // T1[i][(n,k)] = sum_j H[i][j] A[j][(n,k)]
    if (gemm(h, true, false, false, h->nhp, (int)cols, h->nhp, 1.0, Hm, h->ld, Ab, cols, 0.0, Tb, cols)) return -2;
    // C1[k][l] += sum_(i,n) A[(i,n)][k] T1[(i,n)][l]
    if (gemm_splitk_sym(h, false, false, ch.kwp, h->nhp * ch.nc, Ab, ch.kwp, Tb, ch.kwp, 0,
                        (long)ch.k_lo * h->ld + ch.k_lo)) return -2;
    if (full) {
      // V[(i,n)][l] = sum_k A[(i,n)][k] iKx[k][l]   (window block of iKx)
      // (computed as V^T = iKx A2^T with the transposed store: 200-row tiles split 104 + 96 instead of 128 + 72)
      if (tri) {
        // V' = A L with iKx[window] = L L^T;  Q += V' V'^T
        if (right_mul_tri(h, Ab, h->wfac + woff[cidx], ch, h->wsV)) return -2;
        if (gemm_splitk_sym(h, true, true, h->nhp, (int)cols, h->wsV, cols, h->wsV, cols, 1, 0)) return -2;
      } else {
        if (right_mul_sym(h, Ab, iKx, ch, h->wsV)) return -2;
        // Q[i][j] += sum_(n,k) A[i][(n,k)] V[j][(n,k)]
        if (gemm_splitk_sym(h, true, true, h->nhp, (int)cols, Ab, cols, h->wsV, cols, 1, 0)) return -2;
      }
    }
  }
  if (st && !full) h->storeA_frozen_valid = true;
  if (sym_finish(h, 0, h->nxp, h->M(M_C1))) return -2;
  if (full) {
    if (sym_finish(h, 1, h->nhp, h->M(M_Q))) return -2;
    long total = (long)h->nhp * h->ld;
    ypart_reduce_kernel<<<148, 256, 0, h->st>>>(h->ypart, y_slices_used(chunks), total, total,
                                                h->M(M_Y));
    L(h);
  }
  CK(cudaGetLastError());
  return 0;
}

// Backward sweep: Hbar = sum_n A_n C1bar A_n^T, and when `full`: g[3] = sum_n <H A_n Wx + y_n Ybar, dA_n/dtheta>.
int backward_sweep(cgpcm_handle* h, const PsiConst& c, const std::vector<Chunk>& chunks, const double* Hm,
                   bool full, double* g3) {
  zero(h, h->M(M_HBAR), h->ld * h->ld);
  if (sym_begin(h, 0)) return -2;
  long gneed = 0;
  for (const Chunk& ch : chunks) gneed = std::max<long>(gneed, (long)h->nhp * ((ch.nc + AHX_NSUB - 1) / AHX_NSUB));
  if (full) {
    if (gneed * 3 > h->gpart_elems) {
      if (h->gpart) cudaFree(h->gpart);
      h->gpart = nullptr;
      CK(cudaMalloc(&h->gpart, gneed * 3 * sizeof(double)));
      h->gpart_elems = gneed * 3;
    }
    zero(h, h->gpart, h->gpart_elems);
  }
  const bool st = h->use_store;
  // -C1bar = r (Pinv / 2 + lbar lbar^T / 2) is positive definite: Hbar = -sum_n (A_n L)(A_n L)^T with -C1bar[window] = L L^T
  const bool tri = tri_eligible(h, chunks);
  std::vector<long> woff;
  if (tri && window_factors(h, h->M(M_C1BAR), -1.0, chunks, 7, woff)) return -2;
  size_t ci = 0;
  for (const Chunk& ch : chunks) {
    const size_t cidx = ci++;
    const double* Ab = st ? h->storeA + ch.off : h->wsA;
    if (!st && gen_chunk(h, c, ch, false)) return -2;
    const long cols = (long)ch.nc * ch.kwp;
    if (tri) {
      if (right_mul_tri(h, Ab, h->wfac + woff[cidx], ch, h->wsV)) return -2;
      if (gemm_splitk_sym(h, true, true, h->nhp, (int)cols, h->wsV, cols, h->wsV, cols, 0, 0)) return -2;
    } else {
      // U1[(i,n)][l] = sum_k A[(i,n)][k] C1bar[k][l]
      if (right_mul_sym(h, Ab, h->M(M_C1BAR), ch, h->wsV)) return -2;
      // Hbar[i][j] += sum_(n,l) U1[i][(n,l)] A[j][(n,l)]
      if (gemm_splitk_sym(h, true, true, h->nhp, (int)cols, h->wsV, cols, Ab, cols, 0, 0)) return -2;
    }
    if (full) {
      // T1 = H A (kept from the forward sweep when stored) ;  Abar = T1 Wx  (window block)
      const double* Tb = st ? h->storeT + ch.off : h->wsT;
      if (!st && gemm(h, true, false, false, h->nhp, (int)cols, h->nhp, 1.0, Hm, h->ld, Ab, cols, 0.0, h->wsT, cols)) return -2;
      if (right_mul_sym(h, Tb, h->M(M_WX), ch, h->wsV)) return -2;
      prof_close(h);
      ahx_dot_launch(h->st, c.causal && !c.causal_id && h->sep_opt, h->t + ch.n0, h->y + ch.n0, ch.nv, ch.nc, h->th,
                     h->nh, h->nhp, h->tx, h->nx, ch.k_lo, ch.kwp, Ab, h->wsV, h->M(M_YBAR), h->ld, h->gpart, c);
      L(h);
    }
  }
  if (sym_finish(h, 0, h->nhp, h->M(M_HBAR))) return -2;
  if (tri) {
    double* hb = h->M(M_HBAR);
    ew(h->st, h->ld * h->ld, [=] __device__(long idx) { hb[idx] = -hb[idx]; });
    L(h);
  }
  if (full) {
    sum3_kernel<<<1, 1024, 0, h->st>>>(h->gpart, gneed, g3);
    L(h);
  }
  CK(cudaGetLastError());
  return 0;
}

// ---- fourth-order Psi tensor of the frozen regime (gram_kernels.cuh) --------------------------------------------
// Built at cgpcm_precompute when it pays: two streaming passes over G per evaluation (16 R^2 bytes, R = nxp nhp)
// against the contraction sweeps (4 nc nh kwp (nh + kwp) flops per chunk), and when it fits.
int gram_build(cgpcm_handle* h, const PsiConst& c, const std::vector<Chunk>& chunks) {
  h->gram_valid = false;
  if (!h->gram_opt || chunks.empty() || h->nhp > 512) return 0;
  const long R = (long)h->nxp * h->nhp;
  const double bytes = 8.0 * (double)R * R;
  double sweep_flops = 0.0;
  for (const Chunk& ch : chunks) sweep_flops += 4.0 * ch.nc * h->nhp * ch.kwp * (double)(h->nhp + ch.kwp);
  const double t_gram = 2.0 * bytes / 4e12, t_sweep = sweep_flops / 25e12 + 5e-6 * 6 * chunks.size();
  if (h->gram_opt == 1 && t_gram > 0.5 * t_sweep) return 0;
  if (h->gram_elems < R * R) {
    if (h->gram) { cudaFree(h->gram); h->gram = nullptr; h->gram_elems = 0; }
    size_t free_b = 0, tot_b = 0;
    if (cudaMemGetInfo(&free_b, &tot_b) != cudaSuccess) { cudaGetLastError(); return 0; }
    if (bytes > 0.35 * (double)free_b) return 0;
    if (cudaMalloc(&h->gram, (size_t)bytes) != cudaSuccess) { cudaGetLastError(); h->gram = nullptr; return 0; }
    h->gram_elems = R * R;
  }
  CK(cudaMemsetAsync(h->gram, 0, (size_t)bytes, h->st));
  for (const Chunk& ch : chunks) {
    const long row = (long)ch.kwp * h->nhp;
    ahx_gen_nki_kernel<<<148 * 8, 256, 0, h->st>>>(h->t + ch.n0, ch.nv, ch.nc, h->th, h->nh, h->nhp, h->tx, h->nx, ch.k_lo,
                                                   ch.kwp, h->wsT, c);
    L(h);
    double* Gwin = h->gram + (long)ch.k_lo * h->nhp * (R + 1);
    // G_window += Ac^T Ac (lower tiles)
    if (gemm(h, false, false, false, (int)row, (int)row, ch.nc, 1.0, h->wsT, row, h->wsT, row, 1.0, Gwin, R, 1, 0, 1))
      return -2;
  }
  dim3 grid((unsigned)((R + 31) / 32), (unsigned)((R + 31) / 32));
  gram_mirror_kernel<<<grid, 256, 0, h->st>>>(h->gram, R, (int)R);
  L(h);
  CK(cudaGetLastError());
  h->gram_valid = true;
  return 0;
}

// M_C1 = sum_n A_n^T Hm A_n over the frozen regime's blocks: from G when resident, else the forward sweep
int frozen_c1(cgpcm_handle* h, const std::vector<Chunk>& chunks, const double* Hm) {
  if (!h->gram_valid) return forward_sweep(h, h->fc, chunks, Hm, nullptr, false, false);
  const long R = (long)h->nxp * h->nhp;
  zero(h, h->M(M_C1), h->ld * h->ld);
  gram_c1_kernel<<<h->nx * (h->nx + 1) / 2, 256, 0, h->st>>>(h->gram, R, h->nx, h->nh, h->nhp, Hm, h->ld, h->M(M_C1), h->ld);
  L(h);
  CK(cudaGetLastError());
  return 0;
}

// out (ld x ld) = sum_n A_n W A_n^T from G
int gram_q(cgpcm_handle* h, const double* W, double* out) {
  const long R = (long)h->nxp * h->nhp;
  const int slices = 16;
  const int threads = std::min(256, round_up(h->nhp, 32));
  zero(h, out, h->ld * h->ld);
  dim3 grid(h->nh, slices);
  gram_q_kernel<<<grid, threads, h->nx * sizeof(double), h->st>>>(h->gram, R, h->nx, h->nh, h->nhp, W, h->ld, h->ypart,
                                                                  h->ld);
  L(h);
  const long total = (long)h->nhp * h->ld;
  ypart_reduce_kernel<<<148, 256, 0, h->st>>>(h->ypart, slices, total, total, out);
  L(h);
  CK(cudaGetLastError());
  return 0;
}

// Q-type sweep with an arbitrary symmetric ld x ld matrix W in place of iKx:  M_Q = sum_n A_n W A_n^T  over the
// frozen regime's Ahx blocks (the z = False contraction of _optimal_q, src/core/cgpcm.py:473-475).
int q_sweep(cgpcm_handle* h, const PsiConst& c, const std::vector<Chunk>& chunks, const double* W) {
  zero(h, h->M(M_Q), h->ld * h->ld);
  if (sym_begin(h, 1)) return -2;
  const bool st = h->use_store;
  const bool have_a = st && h->storeA_frozen_valid;
  for (const Chunk& ch : chunks) {
    double* Ab = st ? h->storeA + ch.off : h->wsA;
    if (!have_a && gen_chunk(h, c, ch, false, Ab)) return -2;
    const long cols = (long)ch.nc * ch.kwp;
    if (right_mul_sym(h, Ab, W, ch, h->wsV)) return -2;
    if (gemm_splitk_sym(h, true, true, h->nhp, (int)cols, Ab, cols, h->wsV, cols, 1, 0)) return -2;
  }
  if (st) h->storeA_frozen_valid = true;
  if (sym_finish(h, 1, h->nhp, h->M(M_Q))) return -2;
  CK(cudaGetLastError());
  return 0;
}

int allreduce(cgpcm_handle* h, void* buf, long count, int type = NCCL_DOUBLE, int op = NCCL_SUM) {
  if (h->world <= 1 || !h->comm) return 0;
  ncclResult_t r = nccl().AllReduce(buf, buf, (size_t)count, type, op, h->comm, h->st);
  if (r != 0) {
    h->err = std::string("ncclAllReduce failed: ") + (nccl().GetErrorString ? nccl().GetErrorString(r) : "?");
    return -2;
  }
  return 0;
}

// recv[r * count + i] = send_r[i] for every rank r (recv holds world * count doubles).
int allgather(cgpcm_handle* h, const double* send, double* recv, long count) {
  if (h->world <= 1 || !h->comm) return 0;
  ncclResult_t r = nccl().AllGather(send, recv, (size_t)count, NCCL_DOUBLE, h->comm, h->st);
  if (r != 0) {
    h->err = std::string("ncclAllGather failed: ") + (nccl().GetErrorString ? nccl().GetErrorString(r) : "?");
    return -2;
  }
  return 0;
}

// ---- M x M prologue: prior kernels, inverses (src/core/cgpcm.py:214-229) -----------------------------
// `defer_join`: the caller overlaps work that needs neither factorisation (the Axx sweep, the moments of q(u)) and calls
// prior_join itself; otherwise the main stream waits here.
int prior_join(cgpcm_handle* h) {
  if (!h->prior_pending) return 0;
  h->prior_pending = false;
  if (side_join(h, 0)) return -2;
  if (side_join(h, 1)) return -2;
  return 0;
}

int prior_stage(cgpcm_handle* h, const PsiConst& c, double reg, bool reuse = false, bool defer_join = false) {
  const long ld = h->ld;
  if (reuse && h->prior_valid && h->prior_key[0] == c.alpha && h->prior_key[1] == c.gamma && h->prior_key[2] == c.omega &&
      h->prior_key[3] == reg)
    return 0;
  h->prior_valid = false;
  // Kh0, Kh(+jitter) -> M_LH ; Kx0, Kx(+jitter) -> M_KX ; Ahh and tangents
  prior_kernels_kernel<<<148 * 2, 256, 0, h->st>>>(h->th, h->nh, ld, h->tx, h->nx, ld, reg, h->M(M_KH0), h->M(M_LH),
                                                    h->M(M_KX0), h->M(M_KX), h->M(M_AHH), h->M(M_DAHH_A),
                                                    h->M(M_DAHH_G), c, h->pw_dists);
  L(h);
  // the two factor / inverse chains run beside each other on the side streams
  if (side_fork(h, 0)) return -2;
  if (side_fork(h, 1)) return -2;
  if (chol_inv_on(h, 1, h->M(M_LH), h->M(M_IKH), h->nh, h->nhp, h->sc + S_LOGDET_KH, 1)) return -2;
  CK(cudaMemcpyAsync(h->M(M_LX), h->M(M_KX), ld * ld * sizeof(double), cudaMemcpyDeviceToDevice, h->side[1]));
  if (chol_inv_on(h, 2, h->M(M_LX), h->M(M_IKX), h->nx, h->nxp, h->sc + S_LOGDET_KX, 2)) return -2;
  h->prior_pending = true;
  if (!defer_join && prior_join(h)) return -2;
  h->prior_key[0] = c.alpha; h->prior_key[1] = c.gamma; h->prior_key[2] = c.omega; h->prior_key[3] = reg;
  h->prior_valid = true;      // withdrawn by the caller when the info word reports a failed factorisation
  return 0;
}

}  // namespace cgimpl

using namespace cgimpl;

// ------------------------------------------------------------------------------------------------
// C-ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int cgpcm_create(cgpcm_handle** out, int device, int nh, int nx, int causal, int causal_id, void* nccl_comm) {
  if (!out) return -1;
  *out = nullptr;
  if (nh < 1 || nx < 1 || nh > 4096 || nx > 4096) return -1;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0 || device < 0 || device >= count) {
    cudaGetLastError();
    return -2;   // no CPU fallback
  }
  cgpcm_handle* h = new cgpcm_handle();
  h->device = device;
  h->nh = nh; h->nx = nx;
  h->nhp = round_up(nh, 8); h->nxp = round_up(nx, 8);
  h->ld = std::max(h->nhp, h->nxp);
  h->causal = causal ? 1 : 0;
  h->causal_id = causal_id ? 1 : 0;
  auto fail = [&](int code) { cgpcm_destroy(h); return code; };
  if (cudaSetDevice(device) != cudaSuccess) return fail(-2);
  if (cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || h->sms < 2) h->sms = 148;
  if (cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking) != cudaSuccess) return fail(-2);
  for (int k = 0; k < 2; ++k) {
    if (cudaStreamCreateWithFlags(&h->side[k], cudaStreamNonBlocking) != cudaSuccess) return fail(-2);
    if (cudaEventCreateWithFlags(&h->sev_fork[k], cudaEventDisableTiming) != cudaSuccess) return fail(-2);
    if (cudaEventCreateWithFlags(&h->sev_join[k], cudaEventDisableTiming) != cudaSuccess) return fail(-2);
  }
  const long l2 = h->ld * h->ld;
  // forward all-reduce buffer: M_AXX0 .. M_Y contiguous + 2 scalars directly behind M_Y requires M_Y to
  // be followed by the tail: allocate mats with 8 spare doubles between slots M_Y and M_HBAR?  Simpler:
  // the tail lives in its own array and the forward reduction is two collectives fused by group size.
  if (cudaMalloc(&h->mats, (long)M_COUNT * l2 * sizeof(double)) != cudaSuccess) return fail(-2);
  if (cudaMemsetAsync(h->mats, 0, (long)M_COUNT * l2 * sizeof(double), h->st) != cudaSuccess) return fail(-2);
  if (cudaMalloc(&h->vecs, (long)V_COUNT * h->ld * sizeof(double)) != cudaSuccess) return fail(-2);
  cudaMemsetAsync(h->vecs, 0, (long)V_COUNT * h->ld * sizeof(double), h->st);
  if (cudaMalloc(&h->sc, (S_COUNT + 16) * sizeof(double)) != cudaSuccess) return fail(-2);
  cudaMemsetAsync(h->sc, 0, (S_COUNT + 16) * sizeof(double), h->st);
  h->fwd_tail = h->sc + S_COUNT;   // [n, sum_y2, g_alpha, g_gamma, g_omega]
  if (cudaMalloc(&h->info, 4 * sizeof(int)) != cudaSuccess) return fail(-2);
  cudaMemsetAsync(h->info, 0, 4 * sizeof(int), h->st);
  const long np = 5 + nh + (long)nh * (nh + 1) / 2;
  if (cudaMalloc(&h->params_d, np * sizeof(double)) != cudaSuccess) return fail(-2);
  // packed gradient of the variables; also the packed Cholesky factor of q(z) in cgpcm_fpi (nx (nx + 1) / 2)
  if (cudaMalloc(&h->gvar_d, std::max<long>(np, (long)nx * (nx + 1) / 2) * sizeof(double)) != cudaSuccess) return fail(-2);
  for (int k = 0; k < 2; ++k)
    if (cudaMalloc(&h->symacc[k], (size_t)SY_MAX_SPLITS * l2 * sizeof(double)) != cudaSuccess) return fail(-2);
  if (cudaMalloc(&h->cheb_d, (BVN_CHEB_MAXDEG + 1) * 20 * sizeof(double)) != cudaSuccess) return fail(-2);
  h->axx_slices = 64;      // tools/axx_probe.py: 10.88 / 10.45 / 10.37 ms at 32 / 64 / 96 (bench shape), 1.86 / 1.79 / 1.85 on an 8-way shard
  h->axx_part_elems = (long)AXX_MAX_SLICES * 4 * l2;
  if (cudaMalloc(&h->axx_part, h->axx_part_elems * sizeof(double)) != cudaSuccess) return fail(-2);
  for (auto& e : h->ev)
    if (cudaEventCreate(&e) != cudaSuccess) return fail(-2);
  if (nccl_comm) { h->comm = (ncclComm_t)nccl_comm; h->own_comm = false; }   // rank / world: cgpcm_comm_init(h, NULL, ..)
  if (cudaStreamSynchronize(h->st) != cudaSuccess) return fail(-2);
  *out = h;
  return 0;
}

int cgpcm_destroy(cgpcm_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  if (h->st) cudaStreamSynchronize(h->st);
  for (int k = 0; k < 2; ++k)
    if (h->side[k]) cudaStreamSynchronize(h->side[k]);
  if (h->comm && h->own_comm && nccl().ok) nccl().CommDestroy(h->comm);
  double* ptrs[] = {h->t, h->y, h->th, h->tx, h->mats, h->vecs, h->sc, h->params_d, h->gvar_d, h->wsA, h->wsT,
                    h->wsV, h->axx_part, h->ypart, h->gpart, h->symacc[0], h->symacc[1], h->storeA, h->storeT, h->cheb_d, h->gram};
  for (double* p : ptrs)
    if (p) cudaFree(p);
  if (h->wfac) cudaFree(h->wfac);
  if (h->wdesc) cudaFree(h->wdesc);
  if (h->smf_buf) cudaFree(h->smf_buf);
  if (h->smf_info) cudaFree(h->smf_info);
  if (h->info) cudaFree(h->info);
  for (auto& e : h->ev)
    if (e) cudaEventDestroy(e);
  for (auto& e : h->pev) cudaEventDestroy(e);
  for (int k = 0; k < 2; ++k) {
    if (h->sev_fork[k]) cudaEventDestroy(h->sev_fork[k]);
    if (h->sev_join[k]) cudaEventDestroy(h->sev_join[k]);
    if (h->side[k]) cudaStreamDestroy(h->side[k]);
  }
  if (h->st) cudaStreamDestroy(h->st);
  delete h;
  return 0;
}

const char* cgpcm_last_error(const cgpcm_handle* h) { return h ? h->err.c_str() : "null handle"; }

int cgpcm_device_count(int* out) {
  if (!out) return -1;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess) { cudaGetLastError(); *out = 0; return -2; }
  *out = count;
  return 0;
}

int cgpcm_comm_unique_id(void* id128) {
  if (!id128) return -1;
  if (!nccl().ok) return -2;
  ncclUniqueId id;
  if (nccl().GetUniqueId(&id) != 0) return -2;
  memcpy(id128, &id, sizeof id);
  return 0;
}

int cgpcm_comm_init(cgpcm_handle* h, const void* id128, int rank, int world) {
  if (!h || world < 1 || rank < 0 || rank >= world) return -1;
  CK(cudaSetDevice(h->device));
  h->rank = rank;
  h->world = world;
  if (world == 1) return 0;
  if (h->comm && !h->own_comm) return 0;   // communicator supplied at create time
  if (!id128) return -1;
  if (!nccl().ok) { h->err = "NCCL library not loadable"; return -2; }
  ncclUniqueId id;
  memcpy(&id, id128, sizeof id);
  ncclResult_t r = nccl().CommInitRank(&h->comm, world, id, rank);
  if (r != 0) {
    h->err = std::string("ncclCommInitRank failed: ") + (nccl().GetErrorString ? nccl().GetErrorString(r) : "?");
    h->comm = nullptr;
    return -2;
  }
  h->own_comm = true;
  return 0;
}

int cgpcm_set_option(cgpcm_handle* h, const char* key, double value) {
  if (!h || !key) return -1;
  cudaSetDevice(h->device);
  if (!strcmp(key, "chunk")) {
    if (value > (1 << 20) || (value > 0 && value < 8)) { h->err = "chunk out of range"; return -1; }
    h->chunk_auto = value <= 0;
    if (!h->chunk_auto) h->chunk = round_up((int)value, 32);
    h->storeA_frozen_valid = false;
    h->gram_valid = false;
    return 0;
  }
  if (!strcmp(key, "profile")) {
    h->profile = value != 0.0;
    return 0;
  }
  if (!strcmp(key, "cull")) {
    if (value < 0) { h->err = "cull must be >= 0"; return -1; }
    h->cull = value;
    h->storeA_frozen_valid = false;
    return 0;
  }
  if (!strcmp(key, "gram")) {
    h->gram_opt = (int)value;
    h->gram_valid = false;
    if (!h->gram_opt && h->gram) { cudaFree(h->gram); h->gram = nullptr; h->gram_elems = 0; }
    return 0;
  }
  if (!strcmp(key, "pw_dists")) {
    h->pw_dists = value != 0.0;
    h->prior_valid = false;
    return 0;
  }
  if (!strcmp(key, "sl")) {
    h->sl_opt = (int)value;
    return 0;
  }
  if (!strcmp(key, "axx_slices")) {
    if (value < 0 || value > AXX_MAX_SLICES) { h->err = "axx_slices out of range"; return -1; }
    h->axx_slices_opt = (int)value;      // 0 = automatic
    return 0;
  }
  if (!strcmp(key, "tri")) {
    h->tri_opt = (int)value;
    return 0;
  }
  if (!strcmp(key, "sep")) {
    h->sep_opt = (int)value;
    h->storeA_frozen_valid = false;
    return 0;
  }
  if (!strcmp(key, "store")) {
    h->store_opt = value != 0.0;
    h->storeA_frozen_valid = false;
    if (!h->store_opt) {
      if (h->storeA) cudaFree(h->storeA);
      if (h->storeT) cudaFree(h->storeT);
      h->storeA = h->storeT = nullptr;
      h->storeA_elems = h->storeT_elems = 0;
    }
    return 0;
  }
  h->err = std::string("unknown option ") + key;
  return -1;
}

int cgpcm_set_data(cgpcm_handle* h, const double* t, const double* y, int64_t n_local, const double* th,
                   const double* tx) {
  if (!h || n_local < 0 || !th || !tx || (n_local > 0 && (!t || !y))) return -1;
  if (n_local > 2000000000LL) { h->err = "n_local too large"; return -1; }
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->st));
  if (h->t) { cudaFree(h->t); h->t = nullptr; }
  if (h->y) { cudaFree(h->y); h->y = nullptr; }
  if (!h->th) CK(cudaMalloc(&h->th, h->ld * sizeof(double)));
  if (!h->tx) CK(cudaMalloc(&h->tx, h->ld * sizeof(double)));
  h->n_local = n_local;
  h->frozen = false;
  h->storeA_frozen_valid = false;
  h->gram_valid = false;
  h->prior_valid = false;
  const long na = std::max<long>(n_local, 1);
  CK(cudaMalloc(&h->t, na * sizeof(double)));
  CK(cudaMalloc(&h->y, na * sizeof(double)));
  if (n_local > 0) {
    CK(cudaMemcpyAsync(h->t, t, n_local * sizeof(double), cudaMemcpyDefault, h->st));
    CK(cudaMemcpyAsync(h->y, y, n_local * sizeof(double), cudaMemcpyDefault, h->st));
  }
  CK(cudaMemsetAsync(h->th, 0, h->ld * sizeof(double), h->st));
  CK(cudaMemsetAsync(h->tx, 0, h->ld * sizeof(double), h->st));
  CK(cudaMemcpyAsync(h->th, th, h->nh * sizeof(double), cudaMemcpyDefault, h->st));
  CK(cudaMemcpyAsync(h->tx, tx, h->nx * sizeof(double), cudaMemcpyDefault, h->st));
  h->h_t.resize(n_local);
  h->h_th.resize(h->nh);
  h->h_tx.resize(h->nx);
  if (n_local > 0) CK(cudaMemcpyAsync(h->h_t.data(), h->t, n_local * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CK(cudaMemcpyAsync(h->h_th.data(), h->th, h->nh * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CK(cudaMemcpyAsync(h->h_tx.data(), h->tx, h->nx * sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CK(cudaMemsetAsync(h->info, 0, 4 * sizeof(int), h->st));
  CK(cudaMemsetAsync(h->fwd_tail, 0, 2 * sizeof(double), h->st));
  if (n_local > 0) sumsq_kernel<<<1, 1024, 0, h->st>>>(h->y, n_local, h->fwd_tail + 1, h->info + 1, h->t);
  int bad = 0;
  CK(cudaMemcpyAsync(&bad, h->info + 1, sizeof(int), cudaMemcpyDeviceToHost, h->st));
  CK(cudaMemcpyAsync(&h->sum_y2_local, h->fwd_tail + 1, sizeof(double), cudaMemcpyDeviceToHost, h->st));
  CK(cudaStreamSynchronize(h->st));
  for (int i = 0; i < h->nh; ++i) if (!std::isfinite(h->h_th[i])) bad = 1;
  for (int i = 0; i < h->nx; ++i) if (!std::isfinite(h->h_tx[i])) bad = 1;
  if (bad) { h->err = "non-finite value in t, y, th or tx"; return -4; }
  h->t_sorted = true;
  for (long i = 1; i < n_local; ++i)
    if (h->h_t[i] < h->h_t[i - 1]) { h->t_sorted = false; break; }
  return 0;
}

}  // extern "C"

namespace cgimpl {

int ensure_sweep_buffers(cgpcm_handle* h) {
  if (ensure_ws(h)) return -2;
  return ensure_ypart(h, 16);   // the 16 slices of gram_q; the sweeps grow it to their plan (y_slices_used)
}

// copy an (r x c) block of a padded ld-matrix to a dense user buffer (host or device)
int export_mat(cgpcm_handle* h, const double* src, int r, int c, double* dst) {
  if (!dst) return 0;
  CK(cudaMemcpy2DAsync(dst, (size_t)c * sizeof(double), src, (size_t)h->ld * sizeof(double), (size_t)c * sizeof(double),
                       r, cudaMemcpyDefault, h->st));
  return 0;
}

}  // namespace cgimpl

extern "C" {

int cgpcm_psi(cgpcm_handle* h, const double hyp[3], double* sum_Axx, double* Ahh, double* a, double* sum_Ahx_y,
              double* Ahx, double* Axx) {
  if (!h || !hyp) return -1;
  if (!h->t) { h->err = "cgpcm_set_data has not been called"; return -1; }
  for (int i = 0; i < 3; ++i)
    if (!std::isfinite(hyp[i]) || hyp[i] <= 0) { h->err = "hyper-parameters must be positive and finite"; return -4; }
  CK(cudaSetDevice(h->device));
  if (ensure_sweep_buffers(h)) return -2;
  PsiConst c;
  psi_make_const(hyp[0], hyp[1], hyp[2], h->causal, h->cull, &c, h->causal_id);
  BvnTab T;
  bvn_make_tab(hyp[1] / (hyp[0] + hyp[1] + hyp[2]), &T);
  if (begin_run(h)) return -2;
  const long ld = h->ld;
  h->prior_valid = false;      // the slots of the prior kernels are overwritten below (without jitter)
  prior_kernels_kernel<<<148 * 2, 256, 0, h->st>>>(h->th, h->nh, ld, h->tx, h->nx, ld, 0.0, h->M(M_KH0), h->M(M_LH),
                                                    h->M(M_KX0), h->M(M_KX), h->M(M_AHH), h->M(M_DAHH_A),
                                                    h->M(M_DAHH_G), c, h->pw_dists);
  L(h);
  if (sum_Axx) {
    if (axx_sweep(h, c, T, false, h->M(M_AXX0))) return -2;
    if (allreduce(h, h->M(M_AXX0), ld * ld)) return -2;
    if (export_mat(h, h->M(M_AXX0), h->nx, h->nx, sum_Axx)) return -2;
  }
  if (export_mat(h, h->M(M_AHH), h->nh, h->nh, Ahh)) return -2;
  if (a) {
    double av = (h->causal ? 0.5 : 1.0) * sqrt(3.14159265358979323846 / (2.0 * hyp[0]));
    CK(cudaMemcpyAsync(h->sc, &av, sizeof(double), cudaMemcpyHostToDevice, h->st));
    CK(cudaMemcpyAsync(a, h->sc, sizeof(double), cudaMemcpyDefault, h->st));
  }
  if (sum_Ahx_y) {
    // Y only: generate chunks with the fused y-reduction, no GEMMs
    std::vector<Chunk> chunks;
    plan_chunks(h, c, chunks);
    const int ys = y_slices_used(chunks);
    if (ensure_ypart(h, ys)) return -2;
    zero(h, h->ypart, (long)ys * h->nhp * ld);
    for (const Chunk& ch : chunks)
      if (gen_chunk(h, c, ch, true)) return -2;
    long total = (long)h->nhp * ld;
    ypart_reduce_kernel<<<148, 256, 0, h->st>>>(h->ypart, ys, total, total, h->M(M_Y));
    L(h);
    if (allreduce(h, h->M(M_Y), ld * ld)) return -2;
    if (export_mat(h, h->M(M_Y), h->nh, h->nx, sum_Ahx_y)) return -2;
  }
  if (Ahx && h->n_local > 0) {
    double* dst = Ahx;
    Scratch tmp;                  // staging for a host destination
    long total = h->n_local * h->nh * h->nx;
    if (!is_device_ptr(Ahx)) { tmp.take(total); CK(tmp.alloc()); dst = tmp.at(0); }
    ahx_user_kernel<<<148 * 8, 256, 0, h->st>>>(h->t, (int)h->n_local, h->th, h->nh, h->tx, h->nx, dst, c);
    L(h);
    if (dst != Ahx) {
      CK(cudaMemcpyAsync(Ahx, dst, total * sizeof(double), cudaMemcpyDeviceToHost, h->st));
      CK(cudaStreamSynchronize(h->st));
    }
  }
  if (Axx && h->n_local > 0) {
    double* dst = Axx;
    Scratch tmp;
    long total = h->n_local * h->nx * h->nx;
    if (!is_device_ptr(Axx)) { tmp.take(total); CK(tmp.alloc()); dst = tmp.at(0); }
    axx_user_kernel<<<148 * 8, 256, 0, h->st>>>(h->t, (int)h->n_local, h->tx, h->nx, dst, c, T);
    L(h);
    if (dst != Axx) {
      CK(cudaMemcpyAsync(Axx, dst, total * sizeof(double), cudaMemcpyDeviceToHost, h->st));
      CK(cudaStreamSynchronize(h->st));
    }
  }
  int info;
  if (end_run(h, info)) return -2;
  record_timing(h);
  return 0;
}

}  // extern "C"

namespace cgimpl {

// q(u) from the packed parameters in params_d: L from var_u (np.tril_indices order, src/core/tf_util.py:419-447),
// var = L L^T + reg I (src/core/cgpcm.py:444-445, also into M_LVAR for its factorisation), m2 = var + mu mu^T
// (src/core/distribution.py:35-42)
int qu_moments(cgpcm_handle* h, double reg) {
  const int nh = h->nh, nhp = h->nhp;
  const long ld = h->ld, l2 = ld * ld;
  double* Lq = h->M(M_LQ);
  double* mu = h->V(V_MU);
  const double* pd = h->params_d;
  ew(h->st, l2, [=] __device__(long idx) {
    int i = (int)(idx / ld), j = (int)(idx % ld);
    Lq[idx] = (i < nh && j <= i) ? pd[5 + nh + (long)i * (i + 1) / 2 + j] : 0.0;
    if (idx < ld) mu[idx] = idx < nh ? pd[5 + idx] : 0.0;
  });
  L(h);
  if (mm(h, Lq, false, Lq, true, h->M(M_VAR), nhp, nhp, nhp)) return -2;
  double* var = h->M(M_VAR);
  double* lvar = h->M(M_LVAR);
  double* m2 = h->M(M_M2);
  ew(h->st, l2, [=] __device__(long idx) {
    int i = (int)(idx / ld), j = (int)(idx % ld);
    double v = var[idx] + ((i == j && i < nh) ? reg : 0.0);
    var[idx] = v;
    lvar[idx] = v;
    m2[idx] = v + mu[i] * mu[j];
  });
  L(h);
  return 0;
}

// The KL pieces (src/core/distribution.py:60-76) need the factor / inverse of So = iKh + reg I and of the q(u)
// covariance: two chains queued on the side streams (So behind the Kh chain, var behind the Kx chain); the caller joins
// both before kl_scalars.
int kl_fork(cgpcm_handle* h, double reg) {
  const int nh = h->nh, nhp = h->nhp;
  const long ld = h->ld, l2 = ld * ld;
  if (side_fork(h, 0)) return -2;
  if (side_fork(h, 1)) return -2;
  {
    double* so = h->M(M_SO);
    const double* ikh = h->M(M_IKH);
    ew(h->side[0], l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      so[idx] = ikh[idx] + ((i == j && i < nh) ? reg : 0.0);
    });
    h->launches++;
  }
  if (chol_inv_on(h, 1, h->M(M_SO), h->M(M_ISO), nh, nhp, h->sc + S_LOGDET_SO, 4)) return -2;
  if (chol_inv_on(h, 2, h->M(M_LVAR), h->M(M_IVAR), nh, nhp, h->sc + S_LOGDET_VAR, 5)) return -2;
  return 0;
}

void kl_scalars(cgpcm_handle* h) {
  const int nh = h->nh;
  frob(h, h->M(M_ISO), h->M(M_VAR), nh, nh, h->sc + S_TR_ISO_VAR);
  matvec(h, h->M(M_ISO), nh, nh, 0, h->V(V_MU), 1.0, h->V(V_ISOMU));
  dot(h, h->V(V_MU), h->V(V_ISOMU), nh, h->sc + S_MU_ISO_MU);
}

// The ELBO terms that do not depend on the optimal q(z): tm[0], tm[1], tm[4], tm[5], tm[6] (tm[2], tm[3] are left to
// the caller).  hs: the device scalars after the final all-reduce.
void fixed_terms(const cgpcm_handle* h, const double* hs, double s2, double r, double sum_b, double tr_bhh_m2,
                 double* tm) {
  const double Ng = hs[S_COUNT + 0], sum_y2 = hs[S_COUNT + 1];
  const double KL = 0.5 * (hs[S_TR_ISO_VAR] + hs[S_MU_ISO_MU] - h->nh + hs[S_LOGDET_SO] - hs[S_LOGDET_VAR]);
  tm[0] = -0.5 * Ng * log(2.0 * 3.14159265358979323846 * s2) - 0.5 * sum_y2 / s2;
  tm[1] = 0.5 * hs[S_LOGDET_KX];
  tm[2] = tm[3] = 0.0;
  tm[4] = -0.5 * r * sum_b;
  tm[5] = -0.5 * r * tr_bhh_m2;
  tm[6] = -KL;
}

// The whole evaluation.  mode FULL: hyper-parameters from params; mode FROZEN: Psi sums from the frozen
// state (precompute), prior kernels still from params (they stay symbolic in the reference too).
// `freeze`: run the forward Psi sums only and store them (cgpcm_precompute).
// `sample_host` (nh values, or NULL): the stochastic SMF bound elbo(smf=True, sample=...) (src/core/cgpcm.py:527-531):
// the optimal q(z) is built from (sample, sample sample^T) instead of the moments of q(u); value only.  `loglik`
// then also receives the pseudo-log-likelihood that VCGPCM.sample() hands to the slice sampler (cgpcm.py:857-866).
int evaluate_once(cgpcm_handle* h, const double* params_host, int mode, uint32_t grad_mask, double reg, bool freeze,
                  double* elbo, double* terms, double* grad, const double* sample_host, double* loglik);

int evaluate(cgpcm_handle* h, const double* params_host, int mode, uint32_t grad_mask, double reg, bool freeze,
             double* elbo, double* terms, double* grad, const double* sample_host = nullptr, double* loglik = nullptr) {
  h->last_info_tag = 0;
  int rc = evaluate_once(h, params_host, mode, grad_mask, reg, freeze, elbo, terms, grad, sample_host, loglik);
  if (rc == -3 && h->tri_opt && (h->last_info_tag == 6 || h->last_info_tag == 7) && h->world == 1) {
    // a window block lost definiteness in FP64: contract with the full blocks from now on (the reference's formulation).
    // (With several ranks the evaluation is NOT repeated here -- the other ranks may not have seen a failure and a
    // second pass would issue collectives they do not join; the caller gets the error and can set "tri" to 0 on every rank.)
    h->tri_opt = 0;
    rc = evaluate_once(h, params_host, mode, grad_mask, reg, freeze, elbo, terms, grad, sample_host, loglik);
  }
  return rc;
}

int evaluate_once(cgpcm_handle* h, const double* params_host, int mode, uint32_t grad_mask, double reg, bool freeze,
                  double* elbo, double* terms, double* grad, const double* sample_host, double* loglik) {
  const int nh = h->nh, nx = h->nx, nhp = h->nhp, nxp = h->nxp;
  const long ld = h->ld, l2 = ld * ld;
  const long nvar = (long)nh * (nh + 1) / 2;
  const long np = 5 + nh + nvar;
  if (check_finite(h, params_host, freeze ? 5 : np, "non-finite parameter")) return -4;
  const Hyp hp = hyp_of(params_host);
  const double s2 = hp.s2, alpha = hp.alpha, gamma = hp.gamma, omega = hp.omega, r = hp.r, c0 = hp.c0;
  const bool full = (mode == CGPCM_MODE_FULL) || freeze;
  if (!full && !h->frozen) { h->err = "MODE_FROZEN requires cgpcm_precompute"; return -1; }
  if (ensure_sweep_buffers(h)) return -2;

  PsiConst c;
  psi_make_const(alpha, gamma, omega, h->causal, h->cull, &c, h->causal_id);
  BvnTab T;
  bvn_make_tab(gamma / (alpha + gamma + omega), &T);
  const PsiConst& ca = full ? c : h->fc;       // constants that generate A
  std::vector<Chunk> chunks;
  plan_chunks(h, ca, chunks);

  cudaStream_t st = h->st;
  if (begin_run(h)) return -2;
  if (!freeze) CK(cudaMemcpyAsync(h->params_d, params_host, np * sizeof(double), cudaMemcpyHostToDevice, st));

  // ---- 1. prologue (a full-regime evaluation always rebuilds the prior kernels; the precomputed regime reuses them).
  // The factor / inverse chains of Kh and Kx run on the side streams; the main stream goes on with what needs neither
  // (the moments of q(u), the Axx sweep) and waits for them right before H = m2 - iKh.
  if (prior_stage(h, c, reg, !full, true)) return -2;
  double* Hm = h->M(M_H);
  const double* ikh_cur = h->M(M_IKH);
  const double* tl = h->fwd_tail;               // device: [N (all ranks), sum y^2 (all ranks)]
  const bool smf = sample_host != nullptr;
  if (!freeze) {
    if (smf) {
      double* smp = h->V(V_SMP);
      CK(cudaMemsetAsync(smp, 0, ld * sizeof(double), st));
      CK(cudaMemcpyAsync(smp, sample_host, nh * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    if (qu_moments(h, reg)) return -2;
  }
  CK(cudaEventRecord(h->ev[1], st));

  // ---- 2. forward sweep
  if (full) {
    if (axx_sweep(h, c, T, !freeze, h->M(M_AXX0))) return -2;
  }
  CK(cudaEventRecord(h->ev[2], st));
  // the KL pieces (src/core/distribution.py:60-76) need the factor / inverse of So = iKh + reg I and of the q(u)
  // covariance: two more chains that nothing in the forward sweep waits for.  So continues on side stream 0 behind the
  // Kh chain, var on side stream 1 behind the Kx chain and the moments above; the main stream picks them up in step 4.
  bool kl_pending = false;
  if (!freeze) {
    const bool had_prior = h->prior_pending;
    if (had_prior) {
      // the main stream's view of iKh / iKx: events recorded now, BEFORE the KL chains are queued behind them
      if (prior_join(h)) return -2;
    }
    if (kl_fork(h, reg)) return -2;
    kl_pending = true;
  } else {
    if (prior_join(h)) return -2;
  }
  if (!freeze) {
    const double* m2 = h->M(M_M2);
    const double* smp = h->V(V_SMP);
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      // the second moment that enters the optimal q(z): q(u)'s, or sample sample^T for the SMF bound
      const double mq = smf ? smp[i] * smp[j] : m2[idx];
      // FULL: H = m2 - iKh.  FROZEN: the frozen sum_Bxx already carries -sum A^T iKh A, so H = m2.
      Hm[idx] = full ? mq - ikh_cur[idx] : mq;
    });
    L(h);
  } else {
    // the frozen sums do not depend on q(u): H = -iKh gives C1 = -sum A^T iKh A (so that sum_Bxx = Axx + C1)
    const double* ik = h->M(M_IKH);
    ew(st, l2, [=] __device__(long idx) { Hm[idx] = -ik[idx]; });
    L(h);
  }
  const bool want_hyp = full && !freeze && grad && (grad_mask & (CGPCM_GRAD_ALPHA | CGPCM_GRAD_GAMMA | CGPCM_GRAD_OMEGA));
  // Precomputed regime: the reference freezes `mats` only (src/core/cgpcm.py:270-284); Kx, Lx and the prior of q(u)
  // (cgpcm.py:214-229) stay functions of the current (alpha, gamma, omega), so the value follows them (prior_stage
  // rebuilds them when they change) and tf.gradients returns the derivative through them: no sweep is involved.
  const bool want_hyp_prior = !full && grad && (grad_mask & (CGPCM_GRAD_ALPHA | CGPCM_GRAD_GAMMA | CGPCM_GRAD_OMEGA));
  if ((full || !h->gram_valid) && plan_store(h, chunks, want_hyp)) return -2;
  if (full) h->storeA_frozen_valid = false;      // a full-regime sweep overwrites the resident Ahx blocks
  if (!full && h->gram_valid) {
    if (frozen_c1(h, chunks, Hm)) return -2;     // two streaming passes over the resident Psi tensor instead of sweeps
  } else {
    if (forward_sweep(h, ca, chunks, Hm, h->M(M_IKX), full, want_hyp)) return -2;
  }
  // tail scalars [n, sum_y2]
  {
    double tail[2] = {(double)h->n_local, h->sum_y2_local};
    CK(cudaMemcpyAsync(h->fwd_tail, tail, sizeof tail, cudaMemcpyHostToDevice, st));
  }
  // ---- 3. all-reduce #1 (M_AXX0..M_Y are contiguous)
  CK(cudaEventRecord(h->ev[7], st));     // this rank's own forward work ends here (the collective waits for the slowest rank)
  if (h->world > 1) {
    if (full) { if (allreduce(h, h->M(M_AXX0), 7 * l2)) return -2; }
    else { if (allreduce(h, h->M(M_C1), l2)) return -2; }
    if (allreduce(h, h->fwd_tail, 2)) return -2;
  }
  CK(cudaEventRecord(h->ev[3], st));

  if (freeze) {
    // sum_Bhh = N Ahh - Q ; sum_b = N a - N tr(iKh Ahh) - tr(iKx sum_Axx) + tr(iKh Q)
    frob(h, h->M(M_IKH), h->M(M_AHH), nh, nh, h->sc + S_TR_IKH_AHH);
    frob(h, h->M(M_IKX), h->M(M_AXX0), nx, nx, h->sc + S_TR_IKX_AXX);
    frob(h, h->M(M_IKH), h->M(M_Q), nh, nh, h->sc + S_TR_IKH_Q);
    double hs[S_COUNT + 16];
    int info[4];
    CK(cudaMemcpyAsync(hs, h->sc, sizeof hs, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(info, h->info, sizeof info, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h->M(M_F_AXX), h->M(M_AXX0), l2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(h->M(M_F_Y), h->M(M_Y), l2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(h->M(M_F_IKH), h->M(M_IKH), l2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    // frozen sum_Bxx = sum_Axx + C1(-iKh): keep it in M_F_AXX's companion: store C1 into M_T3? -> fold:
    {
      double* fa = h->M(M_F_AXX);
      const double* c1 = h->M(M_C1);
      ew(st, l2, [=] __device__(long idx) { fa[idx] += c1[idx]; });   // M_F_AXX now holds sum_Bxx
      L(h);
    }
    CK(cudaStreamSynchronize(st));
    // the precomputation factorises Kh, Kx and (option "tri") the window blocks of iKx; a failed window block (tag 6)
    // makes evaluate() repeat the precomputation with the full blocks
    static const char* names[] = {"?", "Kh", "Kx", "?", "?", "?", "iKx (a window block)"};
    h->last_info_tag = info[0] / 100000;
    if (pd_error(h, info[0], names)) return -3;
    const double Ng = hs[S_COUNT + 0];
    const double a = (h->causal ? 0.5 : 1.0) * sqrt(3.14159265358979323846 / (2.0 * alpha));
    {
      double* fb = h->M(M_F_BHH);
      const double* ahh = h->M(M_AHH);
      const double* q = h->M(M_Q);
      ew(st, l2, [=] __device__(long idx) { fb[idx] = Ng * ahh[idx] - q[idx]; });
      L(h);
    }
    h->f_a = a;
    h->f_sum_b = Ng * a - Ng * hs[S_TR_IKH_AHH] - hs[S_TR_IKX_AXX] + hs[S_TR_IKH_Q];
    h->fc = c;
    h->frozen = true;
    h->storeA_frozen_valid = h->use_store;       // the blocks just generated are the frozen regime's
    if (gram_build(h, c, chunks)) return -2;
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    return 0;
  }

  // ---- 4. M x M algebra
  // S = sum_Bxx + sum A^T m2 A.  FULL: sum_Axx + C1 (C1 built with H = m2 - iKh).  FROZEN: frozen sum_Bxx + C1(m2).
  double* S = h->M(M_S);
  double* Pm = h->M(M_LP);
  {
    const double* axx = full ? h->M(M_AXX0) : h->M(M_F_AXX);
    const double* c1 = h->M(M_C1);
    const double* kx = h->M(M_KX);
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      double s = axx[idx] + c1[idx];
      S[idx] = s;
      Pm[idx] = kx[idx] + r * s + ((i == j && i < nx) ? reg : 0.0);
    });
    L(h);
  }
  if (chol_inv(h, Pm, h->M(M_PINV), nx, nxp, h->sc + S_LOGDET_P, 3)) return -2;
  const double* Ym = full ? h->M(M_Y) : h->M(M_F_Y);
  matvec(h, Ym, nx, nh, 1, sample_host ? h->V(V_SMP) : h->V(V_MU), 1.0, h->V(V_YTMU));   // Y^T mu (or Y^T sample)
  matvec(h, h->M(M_PINV), nx, nx, 0, h->V(V_YTMU), c0, h->V(V_LBAR));       // lbar = Pinv lam, lam = c0 Y^T mu
  {
    const double* ytmu = h->V(V_YTMU);
    const double* lbar = h->V(V_LBAR);
    reduce_to(st, (long)nx, [=] __device__(long i) { return c0 * ytmu[i] * lbar[i]; }, h->sc + S_LAM_LBAR);
    reduce_to(st, (long)nx, [=] __device__(long i) { return ytmu[i] * lbar[i]; }, h->sc + S_C0BAR);
    L(h, 2);
  }
  if (sample_host && loglik) {
    // sample(): L = chol(P) without jitter (cgpcm.py:856), log_lik = -1/2 logdet P + 1/2 |L^-1 lam|^2 - 1/2 r s^T sum_Bhh s
    double* P0 = h->M(M_T1);
    const double* kx = h->M(M_KX);
    ew(st, l2, [=] __device__(long idx) { P0[idx] = kx[idx] + r * S[idx]; });
    L(h);
    if (chol_inv(h, P0, h->M(M_T2), nx, nxp, h->sc + S_LOGDET_P0, 3)) return -2;
    matvec(h, h->M(M_T2), nx, nx, 0, h->V(V_YTMU), c0, h->V(V_LAM));
    const double* ytmu = h->V(V_YTMU);
    const double* l0 = h->V(V_LAM);
    reduce_to(st, (long)nx, [=] __device__(long i) { return c0 * ytmu[i] * l0[i]; }, h->sc + S_LAM_LBAR0);
    L(h);
  }
  // adjoint seeds: Pbar = -1/2 Pinv - 1/2 lbar lbar^T ; C1bar = r Pbar ; Wx = r (2 Pbar + iKx) ; Ybar = c0 mu lbar^T
  {
    const double* pinv = h->M(M_PINV);
    const double* lbar = h->V(V_LBAR);
    const double* mu = h->V(V_MU);
    const double* ikx = h->M(M_IKX);
    double* pbar = h->M(M_PBAR);
    double* c1bar = h->M(M_C1BAR);
    double* wx = h->M(M_WX);
    double* ybar = h->M(M_YBAR);
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      double pb = -0.5 * pinv[idx] - 0.5 * lbar[i] * lbar[j];
      pbar[idx] = pb;
      c1bar[idx] = r * pb;
      wx[idx] = r * (2.0 * pb + ikx[idx]);
      ybar[idx] = c0 * mu[i] * lbar[j];    // rows i < nhp (mu zero-padded), columns j
    });
    L(h);
  }
  frob(h, h->M(M_PBAR), S, nx, nx, h->sc + S_PBAR_S);
  // KL pieces (src/core/distribution.py:60-76): the chains of So = iKh + reg I and var were queued on the side streams
  // before the forward sweep
  if (kl_pending) {
    if (side_join(h, 0)) return -2;
    if (side_join(h, 1)) return -2;
  }
  kl_scalars(h);
  CK(cudaEventRecord(h->ev[4], st));

  // ---- 5. backward sweep
  const bool want_q = grad_mask & (CGPCM_GRAD_MU_U | CGPCM_GRAD_VAR_U);
  const bool want_grad = grad && grad_mask;
  if (want_grad && (want_hyp || want_q)) {
    if (!full && h->gram_valid) {
      if (gram_q(h, h->M(M_C1BAR), h->M(M_HBAR))) return -2;
    } else {
      if (backward_sweep(h, ca, chunks, Hm, want_hyp, h->fwd_tail + 2)) return -2;
    }
    // ---- 6. all-reduce #2
    CK(cudaEventRecord(h->ev[8], st));
    if (h->world > 1) {
      if (allreduce(h, h->M(M_HBAR), l2)) return -2;
      if (want_hyp && allreduce(h, h->fwd_tail + 2, 3)) return -2;
    }
  } else {
    CK(cudaEventRecord(h->ev[8], st));
  }
  CK(cudaEventRecord(h->ev[5], st));
  const double a = (h->causal ? 0.5 : 1.0) * sqrt(3.14159265358979323846 / (2.0 * alpha));

  // ---- 7. epilogue
  double* bhh = h->M(M_BHH);
  if (full) {
    const double* ahh = h->M(M_AHH);
    const double* q = h->M(M_Q);
    ew(st, l2, [=] __device__(long idx) { bhh[idx] = tl[0] * ahh[idx] - q[idx]; });
    L(h);
    frob(h, h->M(M_IKH), h->M(M_AHH), nh, nh, h->sc + S_TR_IKH_AHH);
    frob(h, h->M(M_IKX), h->M(M_AXX0), nx, nx, h->sc + S_TR_IKX_AXX);
    frob(h, h->M(M_IKH), h->M(M_Q), nh, nh, h->sc + S_TR_IKH_Q);
  } else {
    CK(cudaMemcpyAsync(bhh, h->M(M_F_BHH), l2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
  }
  frob(h, bhh, h->M(M_M2), nh, nh, h->sc + S_TR_BHH_M2);
  if (sample_host && loglik) {
    matvec(h, bhh, nh, nh, 0, h->V(V_SMP), 1.0, h->V(V_M2BMU));
    dot(h, h->V(V_SMP), h->V(V_M2BMU), nh, h->sc + S_S_BHH_S);
  }

  if (want_grad) {
    // m2bar = Hbar - 1/2 r sum_Bhh ; varbar = m2bar - 1/2 (iSo - ivar) ; Lbar = tril(2 varbar L)
    double* m2bar = h->M(M_M2BAR);
    double* varbar = h->M(M_T1);
    {
      const double* hbar = h->M(M_HBAR);
      const double* iso = h->M(M_ISO);
      const double* ivar = h->M(M_IVAR);
      ew(st, l2, [=] __device__(long idx) {
        double m = hbar[idx] - 0.5 * r * bhh[idx];
        m2bar[idx] = m;
        varbar[idx] = m - 0.5 * (iso[idx] - ivar[idx]);
      });
      L(h);
    }
    if (mm(h, varbar, false, h->M(M_LQ), false, h->M(M_T2), nhp, nhp, nhp, 2.0)) return -2;
    // mubar = 2 m2bar mu + c0 Y lbar - iSo mu
    matvec(h, m2bar, nh, nh, 0, h->V(V_MU), 2.0, h->V(V_M2BMU));
    matvec(h, Ym, nh, nx, 0, h->V(V_LBAR), c0, h->V(V_YLBAR));
    {
      const double* t2 = h->M(M_T2);
      const double* a1 = h->V(V_M2BMU);
      const double* a2 = h->V(V_YLBAR);
      const double* a3 = h->V(V_ISOMU);
      double* g = h->gvar_d;
      const bool wmu = grad_mask & CGPCM_GRAD_MU_U, wvar = grad_mask & CGPCM_GRAD_VAR_U;
      ew(st, np, [=] __device__(long idx) {
        double v = 0.0;
        if (idx >= 5 && idx < 5 + nh) {
          long i = idx - 5;
          if (wmu) v = a1[i] + a2[i] - a3[i];
        } else if (idx >= 5 + nh && wvar) {
          long e = idx - 5 - nh;
          long i = (long)((sqrt(8.0 * (double)e + 1.0) - 1.0) * 0.5);
          while ((i + 1) * (i + 2) / 2 <= e) ++i;
          while (i * (i + 1) / 2 > e) --i;
          long j = e - i * (i + 1) / 2;
          v = t2[i * ld + j];
        }
        g[idx] = v;
      });
      L(h);
    }
    if (want_hyp || want_hyp_prior) {
      // Sobar = 1/2 (iSo var iSo + (iSo mu)(iSo mu)^T - iSo)
      if (mm(h, h->M(M_ISO), false, h->M(M_VAR), false, h->M(M_T2), nhp, nhp, nhp)) return -2;
      if (mm(h, h->M(M_T2), false, h->M(M_ISO), false, h->M(M_T3), nhp, nhp, nhp)) return -2;
      // iKhbar = -Hbar + 1/2 r N Ahh - 1/2 r Q + Sobar  -> M_T2   (precomputed regime: Sobar alone, the sums are constants)
      {
        const double wsum = want_hyp ? 1.0 : 0.0;
        const double* t3 = h->M(M_T3);
        const double* iso = h->M(M_ISO);
        const double* ismu = h->V(V_ISOMU);
        const double* hbar = h->M(M_HBAR);
        double* out = h->M(M_T2);
        ew(st, l2, [=] __device__(long idx) {
          int i = (int)(idx / ld), j = (int)(idx % ld);
          double sobar = 0.5 * (t3[idx] + ismu[i] * ismu[j] - iso[idx]);
          out[idx] = wsum * (-hbar[idx] + 0.5 * r * bhh[idx]) + sobar;
        });
        L(h);
      }
      // Khbar = -iKh iKhbar iKh -> M_T1
      if (mm(h, h->M(M_IKH), false, h->M(M_T2), false, h->M(M_T3), nhp, nhp, nhp)) return -2;
      if (mm(h, h->M(M_T3), false, h->M(M_IKH), false, h->M(M_T1), nhp, nhp, nhp, -1.0)) return -2;
      {
        const double* khbar = h->M(M_T1);
        const double* kh0 = h->M(M_KH0);
        const double* thd = h->th;
        reduce_to(st, (long)nh * nh, [=] __device__(long idx) {
          const int i = (int)idx / nh, j = (int)idx - i * nh;   // 32-bit division (nh * nh < 2^31)
          double ti = thd[i], tj = thd[j];
          return -khbar[i * ld + j] * (ti * ti + tj * tj) * kh0[i * ld + j];
        }, h->sc + S_G_KH_A);
        reduce_to(st, (long)nh * nh, [=] __device__(long idx) {
          const int i = (int)idx / nh, j = (int)idx - i * nh;   // 32-bit division (nh * nh < 2^31)
          double d = thd[i] - thd[j];
          return -khbar[i * ld + j] * d * d * kh0[i * ld + j];
        }, h->sc + S_G_KH_G);
        L(h, 2);
      }
      // Kxbar = -iKx iKxbar iKx + Pbar + 1/2 iKx,  iKxbar = 1/2 r S   (precomputed regime: Pbar + 1/2 iKx)
      if (want_hyp) {
        if (mm(h, h->M(M_IKX), false, S, false, h->M(M_T3), nxp, nxp, nxp)) return -2;
        if (mm(h, h->M(M_T3), false, h->M(M_IKX), false, h->M(M_T2), nxp, nxp, nxp, -0.5 * r)) return -2;
      } else {
        zero(h, h->M(M_T2), l2);
      }
      {
        const double* t2 = h->M(M_T2);
        const double* pbar = h->M(M_PBAR);
        const double* ikx = h->M(M_IKX);
        const double* kx0 = h->M(M_KX0);
        const double* txd = h->tx;
        reduce_to(st, (long)nx * nx, [=] __device__(long idx) {
          const int k = (int)idx / nx, l = (int)idx - k * nx;
          double kxbar = t2[k * ld + l] + pbar[k * ld + l] + 0.5 * ikx[k * ld + l];
          double d = txd[k] - txd[l];
          return -kxbar * (0.5 / omega + 0.5 * d * d) * kx0[k * ld + l];
        }, h->sc + S_G_KX_O);
        L(h);
      }
      // <Ahhbar, dAhh>,  Ahhbar = 1/2 r N (iKh - m2)
      if (want_hyp) {
        const double* ikh = h->M(M_IKH);
        const double* m2 = h->M(M_M2);
        const double* da = h->M(M_DAHH_A);
        const double* dg = h->M(M_DAHH_G);
        reduce_to(st, (long)nh * nh, [=] __device__(long idx) {
          const int i = (int)idx / nh, j = (int)idx - i * nh;   // 32-bit division (nh * nh < 2^31)
          return 0.5 * r * tl[0] * (ikh[i * ld + j] - m2[i * ld + j]) * da[i * ld + j];
        }, h->sc + S_G_AHH_A);
        reduce_to(st, (long)nh * nh, [=] __device__(long idx) {
          const int i = (int)idx / nh, j = (int)idx - i * nh;   // 32-bit division (nh * nh < 2^31)
          return 0.5 * r * tl[0] * (ikh[i * ld + j] - m2[i * ld + j]) * dg[i * ld + j];
        }, h->sc + S_G_AHH_G);
        L(h, 2);
      }
      // <Axxbar, dAxx>,  Axxbar = r Pbar + 1/2 r iKx
      if (want_hyp) {
        const double* pbar = h->M(M_PBAR);
        const double* ikx = h->M(M_IKX);
        for (int k3 = 0; k3 < 3; ++k3) {
          const double* dm = h->M(M_AXX1 + k3);
          reduce_to(st, (long)nx * nx, [=] __device__(long idx) {
            const int k = (int)idx / nx, l = (int)idx - k * nx;
            return r * (pbar[k * ld + l] + 0.5 * ikx[k * ld + l]) * dm[k * ld + l];
          }, h->sc + S_G_AXX_A + k3);
        }
        L(h, 3);
      }
    }
  }

  // ---- collect
  double hs[S_COUNT + 16];
  int info;
  CK(cudaMemcpyAsync(hs, h->sc, sizeof hs, cudaMemcpyDeviceToHost, st));
  if (want_grad) CK(cudaMemcpyAsync(grad, h->gvar_d, np * sizeof(double), cudaMemcpyDefault, st));
  if (end_run(h, info)) return -2;
  const double Ng = hs[S_COUNT + 0], sum_y2 = hs[S_COUNT + 1];
  static const char* names[] = {"?", "Kh", "Kx", "P", "iKh + reg I (prior of q(u))", "q(u) covariance",
                                "iKx (a window block)", "-C1bar (a window block)"};
  h->last_info_tag = info / 100000;
  if (pd_error(h, info, names)) return -3;
  double sum_b, tr_bhh_m2 = hs[S_TR_BHH_M2];
  if (full) sum_b = Ng * a - Ng * hs[S_TR_IKH_AHH] - hs[S_TR_IKX_AXX] + hs[S_TR_IKH_Q];
  else sum_b = h->f_sum_b;
  double tm[7];
  fixed_terms(h, hs, s2, r, sum_b, tr_bhh_m2, tm);
  tm[2] = -0.5 * hs[S_LOGDET_P];
  tm[3] = 0.5 * hs[S_LAM_LBAR];
  double e = 0.0;
  for (int i = 0; i < 7; ++i) e += tm[i];
  if (terms) memcpy(terms, tm, sizeof tm);
  if (elbo) *elbo = e;
  if (sample_host && loglik) *loglik = -0.5 * hs[S_LOGDET_P0] + 0.5 * hs[S_LAM_LBAR0] - 0.5 * r * hs[S_S_BHH_S];
  if (want_grad) {
    const double rbar = hs[S_PBAR_S] - 0.5 * sum_b - 0.5 * tr_bhh_m2;
    const double c0bar = hs[S_C0BAR];
    double g5[5] = {0, 0, 0, 0, 0};
    if (grad_mask & CGPCM_GRAD_S2) g5[0] = -r * rbar - c0 * c0bar - 0.5 * Ng + 0.5 * sum_y2 / s2;
    if (grad_mask & CGPCM_GRAD_S2F) g5[1] = r * rbar + 0.5 * c0 * c0bar;
    if (want_hyp_prior) {
      if (grad_mask & CGPCM_GRAD_ALPHA) g5[2] = alpha * hs[S_G_KH_A];
      if (grad_mask & CGPCM_GRAD_GAMMA) g5[3] = gamma * hs[S_G_KH_G];
      if (grad_mask & CGPCM_GRAD_OMEGA) g5[4] = omega * hs[S_G_KX_O];
    }
    if (want_hyp) {
      const double abar = -0.5 * r * Ng;
      const double* gA = hs + S_COUNT + 2;
      double ga = hs[S_G_KH_A] + abar * (-a / (2.0 * alpha)) + hs[S_G_AHH_A] + hs[S_G_AXX_A] + gA[0];
      double gg = hs[S_G_KH_G] + hs[S_G_AHH_G] + hs[S_G_AXX_G] + gA[1];
      double go = hs[S_G_KX_O] + hs[S_G_AXX_O] + gA[2];
      if (grad_mask & CGPCM_GRAD_ALPHA) g5[2] = alpha * ga;
      if (grad_mask & CGPCM_GRAD_GAMMA) g5[3] = gamma * gg;
      if (grad_mask & CGPCM_GRAD_OMEGA) g5[4] = omega * go;
    }
    return put(h, grad, g5, 5);
  }
  return 0;
}

int predict_qz(cgpcm_handle* h, const std::vector<Chunk>& chunks, int smf, const double* mvec, const double* var,
               double r, double c0, double reg, double* xm);

// VCGPCM.fpi(num, z=True, high_reg) followed by convert(z=True) (src/core/cgpcm.py:479-516,577-592) on the frozen
// Psi statistics: num rounds of  q(u) -> optimal q(z) -> optimal q(u)  (Normal.from_natural,
// src/core/distribution.py:20-33), then the optimal q(z) of the final q(u).  Per round one C1-type sweep
// (sum_n A_n^T m2_u A_n) and one Q-type sweep (sum_n A_n m2_z A_n^T) over the resident Ahx blocks.
// `qz_mean` / `qz_chol` (host, nx and nx (nx + 1) / 2 values, or NULL): the z = False variants -- the iteration starts
// from the explicit q(z) = N(qz_mean, reg(Lz Lz^T)), every round is  q(z) -> optimal q(u) -> optimal q(z), and the
// closing half round is convert(z=False): the optimal q(u) of the final q(z)  (cgpcm.py:499,584-592).
int fpi_run(cgpcm_handle* h, const double* params_host, int num, int high_reg, double reg, double* mu_u, double* var_u,
            double* mu_z, double* var_z, const double* qz_mean = nullptr, const double* qz_chol = nullptr) {
  const int nh = h->nh, nx = h->nx, nhp = h->nhp, nxp = h->nxp;
  const long ld = h->ld, l2 = ld * ld;
  const long nvar = (long)nh * (nh + 1) / 2;
  const long np = 5 + nh + nvar;
  if (check_finite(h, params_host, np, "non-finite parameter")) return -4;
  if (!h->frozen) { h->err = "cgpcm_fpi requires cgpcm_precompute"; return -1; }
  const Hyp hp = hyp_of(params_host);
  const double r = hp.r, c0 = hp.c0;
  const double hr = high_reg ? 1e-4 : 0.0;
  if (ensure_sweep_buffers(h)) return -2;
  PsiConst c;
  psi_make_const(hp.alpha, hp.gamma, hp.omega, h->causal, h->cull, &c, h->causal_id);
  std::vector<Chunk> chunks;
  plan_chunks(h, h->fc, chunks);
  cudaStream_t st = h->st;
  if (begin_run(h)) return -2;
  CK(cudaMemcpyAsync(h->params_d, params_host, np * sizeof(double), cudaMemcpyHostToDevice, st));
  if (prior_stage(h, c, reg, true)) return -2;
  if (!h->gram_valid && plan_store(h, chunks, false)) return -2;
  double* mu = h->V(V_MU);
  double* muz = h->V(V_MUZ);
  double* var = h->M(M_VAR);
  // self.h = Normal(reg(L L^T), mu_u)  (cgpcm.py:444-445)
  if (qu_moments(h, reg)) return -2;
  const bool start_z = qz_mean != nullptr && qz_chol != nullptr;
  if (start_z) {
    // q(z) from the caller: mean, and covariance reg(Lz Lz^T) into M_PINV (the slot the q(z) covariance lives in)
    const long nvz = (long)nx * (nx + 1) / 2;
    if (check_finite(h, qz_mean, nx, "non-finite mu_z")) return -4;
    if (check_finite(h, qz_chol, nvz, "non-finite var_z")) return -4;
    CK(cudaMemsetAsync(muz, 0, ld * sizeof(double), st));
    CK(cudaMemcpyAsync(muz, qz_mean, nx * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->gvar_d, qz_chol, nvz * sizeof(double), cudaMemcpyHostToDevice, st));
    double* Lz = h->M(M_T1);
    const double* pz = h->gvar_d;
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      Lz[idx] = (i < nx && j <= i) ? pz[(long)i * (i + 1) / 2 + j] : 0.0;
    });
    L(h);
    if (mm(h, Lz, false, Lz, true, h->M(M_PINV), nxp, nxp, nxp)) return -2;
    double* vz = h->M(M_PINV);
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      if (i == j && i < nx) vz[idx] += reg;
    });
    L(h);
  }
  // one half round each: A = optimal q(z) given q(u) (z = True), B = optimal q(u) given q(z) (z = False)
  auto half_a = [&](double hrz) -> int { return predict_qz(h, chunks, 0, mu, var, r, c0, hrz + reg, muz); };
  auto half_b = [&](double hru) -> int {
    {
      double* W = h->M(M_WX);
      const double* vz = h->M(M_PINV);
      ew(st, l2, [=] __device__(long idx) {
        int i = (int)(idx / ld), j = (int)(idx % ld);
        W[idx] = vz[idx] + muz[i] * muz[j];
      });
      L(h);
    }
    if (h->gram_valid) { if (gram_q(h, h->M(M_WX), h->M(M_Q))) return -2; }
    else if (q_sweep(h, h->fc, chunks, h->M(M_WX))) return -2;
    if (allreduce(h, h->M(M_Q), l2)) return -2;
    {
      double* Pu = h->M(M_SO);
      const double* kh0 = h->M(M_KH0);
      const double* fb = h->M(M_F_BHH);
      const double* q = h->M(M_Q);
      ew(st, l2, [=] __device__(long idx) {
        int i = (int)(idx / ld), j = (int)(idx % ld);
        Pu[idx] = kh0[idx] + r * (fb[idx] + q[idx]) + ((i == j && i < nh) ? reg + hru + reg : 0.0);   // Kh = reg(Kh0)
      });
      L(h);
    }
    if (chol_inv(h, h->M(M_SO), var, nh, nhp, nullptr, 4)) return -2;
    matvec(h, h->M(M_F_Y), nh, nx, 0, muz, c0, h->V(V_LAM));                 // lam = c0 Y mean_z
    matvec(h, var, nh, nh, 0, h->V(V_LAM), 1.0, mu);                         // mean_u = var_u lam (padding stays 0)
    return 0;
  };
  for (int it = 0; it <= num; ++it) {
    const double hr_round = it < num ? hr : 0.0;      // convert() (the last half round) never uses high_reg
    if (!start_z) {
      if (half_a(hr_round)) return -2;
      if (it == num) break;
      if (half_b(hr)) return -2;
    } else {
      if (half_b(hr_round)) return -2;
      if (it == num) break;
      if (half_a(hr)) return -2;
    }
  }
  // outputs: means, and the Cholesky factors of the covariances in np.tril_indices order
  auto emit = [&](const double* mean, const double* cov, int n, int npad, double* mean_out, double* chol_out, int tag) -> int {
    if (mean_out) CK(cudaMemcpyAsync(mean_out, mean, n * sizeof(double), cudaMemcpyDefault, st));
    if (!chol_out) return 0;
    double* Lc = h->M(M_T1);
    CK(cudaMemcpyAsync(Lc, cov, l2 * sizeof(double), cudaMemcpyDeviceToDevice, st));
    if (chol_inv(h, Lc, nullptr, n, npad, nullptr, tag)) return -2;
    double* g = h->gvar_d;
    const long nv = (long)n * (n + 1) / 2;
    ew(st, nv, [=] __device__(long e) {
      long i = (long)((sqrt(8.0 * (double)e + 1.0) - 1.0) * 0.5);
      while ((i + 1) * (i + 2) / 2 <= e) ++i;
      while (i * (i + 1) / 2 > e) --i;
      g[e] = Lc[i * ld + (e - i * (i + 1) / 2)];
    });
    L(h);
    CK(cudaMemcpyAsync(chol_out, g, nv * sizeof(double), cudaMemcpyDefault, st));
    return 0;
  };
  if (emit(mu, var, nh, nhp, mu_u, var_u, 5)) return -2;
  if (emit(muz, h->M(M_PINV), nx, nxp, mu_z, var_z, 3)) return -2;
  int info;
  if (end_run(h, info)) return -2;
  static const char* names[] = {"?", "Kh", "Kx", "P of q(z)", "P of q(u)", "a q covariance"};
  if (pd_error(h, info, names)) return -3;
  record_timing(h);
  return 0;
}

// VCGPCM.elbo(z=False) (src/core/cgpcm.py:518-575 with the z = False branches :533-540,547-566 and _optimal_q(z=False)
// :470-477): the bound saturated for q(u), with q(z) = N(mu_z, reg(Lz Lz^T)) the explicit variational distribution.
// Value and the 7 terms, on the Psi statistics frozen by cgpcm_precompute (the prior kernels follow params, as in
// evaluate()).  The one sum over observations is the Q-type sweep  sum_n A_n m2_z A_n^T.
int qz_run(cgpcm_handle* h, const double* params_host, const double* qz_mean, const double* qz_chol, double reg,
           double* elbo, double* terms) {
  const int nh = h->nh, nx = h->nx, nhp = h->nhp, nxp = h->nxp;
  const long ld = h->ld, l2 = ld * ld;
  const long nvz = (long)nx * (nx + 1) / 2;
  if (check_finite(h, params_host, 5, "non-finite parameter")) return -4;
  if (check_finite(h, qz_mean, nx, "non-finite mu_z")) return -4;
  if (check_finite(h, qz_chol, nvz, "non-finite var_z")) return -4;
  if (!h->frozen) { h->err = "cgpcm_elbo_qz requires cgpcm_precompute"; return -1; }
  const Hyp hp = hyp_of(params_host);
  const double r = hp.r, c0 = hp.c0;
  if (ensure_sweep_buffers(h)) return -2;
  PsiConst c;
  psi_make_const(hp.alpha, hp.gamma, hp.omega, h->causal, h->cull, &c, h->causal_id);
  std::vector<Chunk> chunks;
  plan_chunks(h, h->fc, chunks);
  cudaStream_t st = h->st;
  if (begin_run(h)) return -2;
  if (prior_stage(h, c, reg, true)) return -2;
  if (!h->gram_valid && plan_store(h, chunks, false)) return -2;
  double* muz = h->V(V_MUZ);
  double* varz = h->M(M_VAR);          // covariance of q(z) (the q(u) slots are free in this evaluation)
  double* m2z = h->M(M_M2);
  {
    CK(cudaMemsetAsync(muz, 0, ld * sizeof(double), st));
    CK(cudaMemcpyAsync(muz, qz_mean, nx * sizeof(double), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(h->gvar_d, qz_chol, nvz * sizeof(double), cudaMemcpyHostToDevice, st));
    double* Lz = h->M(M_LQ);
    const double* pz = h->gvar_d;
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      Lz[idx] = (i < nx && j <= i) ? pz[(long)i * (i + 1) / 2 + j] : 0.0;
    });
    L(h);
    if (mm(h, Lz, false, Lz, true, varz, nxp, nxp, nxp)) return -2;
    double* lvar = h->M(M_LVAR);
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      const double v = varz[idx] + ((i == j && i < nx) ? reg : 0.0);
      varz[idx] = v;
      lvar[idx] = v;
      m2z[idx] = v + muz[i] * muz[j];
    });
    L(h);
  }
  // S = sum_Bhh + sum_n A_n m2_z A_n^T ;  P = Kh + r S
  if (h->gram_valid) { if (gram_q(h, m2z, h->M(M_Q))) return -2; }
  else if (q_sweep(h, h->fc, chunks, m2z)) return -2;
  if (allreduce(h, h->M(M_Q), l2)) return -2;
  {
    double* Pu = h->M(M_LP);
    const double* kh0 = h->M(M_KH0);
    const double* fb = h->M(M_F_BHH);
    const double* q = h->M(M_Q);
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      Pu[idx] = kh0[idx] + r * (fb[idx] + q[idx]) + ((i == j && i < nh) ? reg + reg : 0.0);   // reg(Kh) + reg(P)
    });
    L(h);
  }
  if (chol_inv(h, h->M(M_LP), h->M(M_PINV), nh, nhp, h->sc + S_LOGDET_P, 3)) return -2;
  matvec(h, h->M(M_F_Y), nh, nx, 0, muz, c0, h->V(V_LAM));                   // lam = c0 Y mean_z
  matvec(h, h->M(M_PINV), nh, nh, 0, h->V(V_LAM), 1.0, h->V(V_LBAR));
  dot(h, h->V(V_LAM), h->V(V_LBAR), nh, h->sc + S_LAM_LBAR);
  frob(h, h->M(M_F_AXX), m2z, nx, nx, h->sc + S_TR_BHH_M2);                  // tr(sum_Bxx m2_z)
  // -KL(q(z) || N(0, iKx + reg I))
  {
    double* so = h->M(M_SO);
    const double* ikx = h->M(M_IKX);
    ew(st, l2, [=] __device__(long idx) {
      int i = (int)(idx / ld), j = (int)(idx % ld);
      so[idx] = ikx[idx] + ((i == j && i < nx) ? reg : 0.0);
    });
    L(h);
  }
  if (chol_inv(h, h->M(M_SO), h->M(M_ISO), nx, nxp, h->sc + S_LOGDET_SO, 4)) return -2;
  if (chol_inv(h, h->M(M_LVAR), nullptr, nx, nxp, h->sc + S_LOGDET_VAR, 5)) return -2;
  frob(h, h->M(M_ISO), varz, nx, nx, h->sc + S_TR_ISO_VAR);
  matvec(h, h->M(M_ISO), nx, nx, 0, muz, 1.0, h->V(V_ISOMU));
  dot(h, muz, h->V(V_ISOMU), nx, h->sc + S_MU_ISO_MU);
  double hs[S_COUNT + 16];
  int info;
  CK(cudaMemcpyAsync(hs, h->sc, sizeof hs, cudaMemcpyDeviceToHost, st));
  if (end_run(h, info)) return -2;
  static const char* names[] = {"?", "Kh", "Kx", "P of q(u)", "iKx + reg I (prior of q(z))", "q(z) covariance"};
  if (pd_error(h, info, names)) return -3;
  // N and sum y^2 of all ranks
  double tail[2] = {(double)h->n_local, h->sum_y2_local};
  if (h->world > 1) {
    CK(cudaMemcpyAsync(h->fwd_tail, tail, sizeof tail, cudaMemcpyHostToDevice, st));
    if (allreduce(h, h->fwd_tail, 2)) return -2;
    CK(cudaMemcpyAsync(tail, h->fwd_tail, sizeof tail, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  const double KL = 0.5 * (hs[S_TR_ISO_VAR] + hs[S_MU_ISO_MU] - nx + hs[S_LOGDET_SO] - hs[S_LOGDET_VAR]);
  double tm[7];
  tm[0] = -0.5 * tail[0] * log(2.0 * 3.14159265358979323846 * hp.s2) - 0.5 * tail[1] / hp.s2;
  tm[1] = 0.5 * hs[S_LOGDET_KH];
  tm[2] = -0.5 * hs[S_LOGDET_P];
  tm[3] = 0.5 * hs[S_LAM_LBAR];
  tm[4] = -0.5 * r * h->f_sum_b;
  tm[5] = -0.5 * r * hs[S_TR_BHH_M2];
  tm[6] = -KL;
  double e = 0.0;
  for (int i = 0; i < 7; ++i) e += tm[i];
  if (terms) memcpy(terms, tm, sizeof tm);
  if (elbo) *elbo = e;
  record_timing(h);
  return 0;
}

// The moments of q(u) as predict_f uses them: mu (V_MU), var = L L^T + reg I (M_VAR), and tr(Ahh iKh) (S_TR_IKH_AHH).
int predict_qu(cgpcm_handle* h, double reg) {
  if (qu_moments(h, reg)) return -2;
  frob(h, h->M(M_AHH), h->M(M_IKH), h->nh, h->nh, h->sc + S_TR_IKH_AHH);
  return 0;
}

// One optimal q(z) of predict_f: Hm = m m^T (smf: m = a filter sample) or var + m m^T (m = mu of q(u)), C1 over the
// frozen statistics, P = Kx + r (sum_Bxx + C1) + reg I, P^-1 in M_PINV and xm = P^-1 c0 sum_Ahx_y^T m.
int predict_qz(cgpcm_handle* h, const std::vector<Chunk>& chunks, int smf, const double* mvec, const double* var,
               double r, double c0, double reg, double* xm) {
  const int nh = h->nh, nx = h->nx, nxp = h->nxp;
  const long ld = h->ld, l2 = ld * ld;
  cudaStream_t st = h->st;
  double* Hm = h->M(M_H);
  const int smf_ = smf;
  ew(st, l2, [=] __device__(long idx) {
    int i = (int)(idx / ld), j = (int)(idx % ld);
    Hm[idx] = smf_ ? mvec[i] * mvec[j] : var[idx] + mvec[i] * mvec[j];
  });
  L(h);
  if (frozen_c1(h, chunks, Hm)) return -2;
  if (allreduce(h, h->M(M_C1), l2)) return -2;
  double* Pm = h->M(M_LP);
  const double* kx = h->M(M_KX);
  const double* fb = h->M(M_F_AXX);
  const double* c1 = h->M(M_C1);
  ew(st, l2, [=] __device__(long idx) {
    int i = (int)(idx / ld), j = (int)(idx % ld);
    Pm[idx] = kx[idx] + r * (fb[idx] + c1[idx]) + ((i == j && i < nx) ? reg : 0.0);
  });
  L(h);
  if (chol_inv(h, Pm, h->M(M_PINV), nx, nxp, nullptr, 3)) return -2;
  matvec(h, h->M(M_F_Y), nx, nh, 1, mvec, c0, h->V(V_LAM));
  matvec(h, h->M(M_PINV), nx, nx, 0, h->V(V_LAM), 1.0, xm);
  return 0;
}

// Test-side blocks of a chunk of nv test points at tc: A* (h->wsA, [i][n][k] at kw = nxp), T = iKh A* (h->wsT) and
// Bxx*_n = Axx*_n - A*_n^T iKh A*_n (dense [n][nx][nx] in X).
int predict_chunk_blocks(cgpcm_handle* h, const PsiConst& cd, const BvnTab& T, const double* tc, int nv, double* X) {
  const int nh = h->nh, nx = h->nx, nhp = h->nhp, nxp = h->nxp;
  const long ld = h->ld;
  cudaStream_t st = h->st;
  const int nc = round_up(nv, 8);
  const long cols = (long)nc * nxp;
  {
    const int threads = std::min(256, round_up(nxp, 32));
    dim3 grid(nhp, (nc + AHX_NSUB - 1) / AHX_NSUB);
    ahx_gen_kernel<<<grid, threads, 0, st>>>(tc, tc, nv, nc, h->th, nh, h->tx, nx, 0, nxp, h->wsA, nullptr, ld,
                                             (long)nhp * ld, cd);
    L(h);
  }
  if (gemm(h, true, false, false, nhp, (int)cols, nhp, 1.0, h->M(M_IKH), ld, h->wsA, cols, 0.0, h->wsT, cols)) return -2;
  axx_user_kernel<<<148 * 8, 256, 0, st>>>(tc, nv, h->tx, nx, X, cd, T);
  L(h);
  {
    dim3 grid((nx + 31) / 32, (nx + 31) / 32, nv);
    bxx_star_kernel<<<grid, 256, 0, st>>>(h->wsA, h->wsT, nh, nc, nxp, nx, X);
    L(h);
  }
  return 0;
}

// VCGPCM.predict_f (src/core/cgpcm.py:781-846) for given filter samples: posterior mean and variance of the function
// at the test inputs, averaged over the samples.  smf = 0: one optimal q(z) from the moments of q(u); smf = 1: the
// optimal q(z | h) per sample.  Training side: the frozen regime's sweeps; test side: predict_kernels.cuh.
int predict_run(cgpcm_handle* h, const double* params_host, double reg, const double* tstar_host, long n_star,
                const double* samples_host, int B, int smf, double* mu_out, double* var_out) {
  const int nh = h->nh, nx = h->nx, nxp = h->nxp;
  const long ld = h->ld, l2 = ld * ld;
  const long np = 5 + nh + (long)nh * (nh + 1) / 2;
  if (check_finite(h, params_host, np, "non-finite parameter")) return -4;
  if (check_finite(h, tstar_host, n_star, "non-finite test input")) return -4;
  if (check_samples(h, samples_host, B, nh)) return -4;
  if (!h->frozen) { h->err = "cgpcm_predict_f requires cgpcm_precompute"; return -1; }
  const Hyp hp = hyp_of(params_host);
  const double r = hp.r, c0 = hp.c0, s2f = hp.s2f;
  if (ensure_sweep_buffers(h)) return -2;
  PsiConst c;
  psi_make_const(hp.alpha, hp.gamma, hp.omega, h->causal, h->cull, &c, h->causal_id);
  PsiConst cd = c;                       // test-side statistics are evaluated densely (no windows)
  cd.cull = 746.0;
  BvnTab T;
  bvn_make_tab(hp.gamma / (hp.alpha + hp.gamma + hp.omega), &T);
  std::vector<Chunk> chunks;
  plan_chunks(h, h->fc, chunks);
  cudaStream_t st = h->st;
  const int TC = std::min<long>(h->chunk, std::max<long>(n_star, 1));
  const int nq = smf ? B : 1;            // distinct q(z)
  Scratch s;
  const size_t o_t = s.take(std::max<long>(n_star, 1)), o_x = s.take((size_t)TC * nx * nx);
  const size_t o_mx = s.take((size_t)nq * l2), o_vec = s.take((size_t)(B + nq) * ld);   // samples h_b, then xm per q(z)
  const size_t o_q1 = s.take(B), o_acc = s.take(2 * std::max<long>(n_star, 1));
  CK(s.alloc());
  double *d_t = s.at(o_t), *d_x = s.at(o_x), *d_mx = s.at(o_mx), *d_vec = s.at(o_vec), *d_q1 = s.at(o_q1);
  double* d_acc = s.at(o_acc);
  double* d_h = d_vec;
  double* d_xm = d_vec + (long)B * ld;
  if (begin_run(h)) return -2;
  CK(cudaMemcpyAsync(h->params_d, params_host, np * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_t, tstar_host, n_star * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(d_vec, 0, (size_t)(B + nq) * ld * sizeof(double), st));
  CK(cudaMemcpy2DAsync(d_h, ld * sizeof(double), samples_host, nh * sizeof(double), nh * sizeof(double), B,
                       cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(d_acc, 0, (size_t)2 * std::max<long>(n_star, 1) * sizeof(double), st));
  if (prior_stage(h, c, reg, true)) return -2;
  if (!h->gram_valid && plan_store(h, chunks, false)) return -2;
  if (predict_qu(h, reg)) return -2;
  const double* mu = h->V(V_MU);
  const double* var = h->M(M_VAR);
  const double a_val = (h->causal ? 0.5 : 1.0) * sqrt(3.14159265358979323846 / (2.0 * hp.alpha));
  // ---- training side: q(z) (once, or per sample) and the per-sample scalar q1
  for (int b = 0; b < std::max(B, nq); ++b) {
    const double* hb = d_h + (long)b * ld;
    if (b < nq) {
      double* xm = d_xm + (long)b * ld;
      if (predict_qz(h, chunks, smf, smf ? hb : mu, var, r, c0, reg, xm)) return -2;
      double* mxb = d_mx + (long)b * l2;
      const double* xv = h->M(M_PINV);
      const double* ikx = h->M(M_IKX);
      ew(st, l2, [=] __device__(long idx) {
        int i = (int)(idx / ld), j = (int)(idx % ld);
        mxb[idx] = (i < nx && j < nx) ? xv[idx] + xm[i] * xm[j] - ikx[idx] : 0.0;
      });
      L(h);
    }
    if (b < B) {
      // q1 = a + h^T Ahh h - tr(Ahh iKh)
      matvec(h, h->M(M_AHH), nh, nh, 0, hb, 1.0, h->V(V_M2BMU));
      dot(h, hb, h->V(V_M2BMU), nh, h->sc + S_S_BHH_S);
      const double* scp = h->sc;
      double* q1 = d_q1 + b;
      ew(st, 1, [=] __device__(long) { q1[0] = a_val + scp[S_S_BHH_S] - scp[S_TR_IKH_AHH]; });
      L(h);
    }
  }
  // ---- test side, chunk by chunk
  for (long p0 = 0; p0 < n_star; p0 += TC) {
    const int nv = (int)std::min<long>(TC, n_star - p0);
    const int nc = round_up(nv, 8);
    if (predict_chunk_blocks(h, cd, T, d_t + p0, nv, d_x)) return -2;
    for (int b = 0; b < B; ++b) {
      const int qb = smf ? b : 0;
      predict_point_kernel<<<nv, 256, nx * sizeof(double), st>>>(h->wsA, nh, nc, nxp, nx, d_h + (long)b * ld,
                                                                 d_xm + (long)qb * ld, d_mx + (long)qb * l2, ld, d_x,
                                                                 d_q1 + b, sqrt(s2f), s2f, 1.0 / B, d_acc + p0,
                                                                 d_acc + n_star + p0);
      L(h);
    }
  }
  if (mu_out) CK(cudaMemcpyAsync(mu_out, d_acc, n_star * sizeof(double), cudaMemcpyDefault, st));
  if (var_out) CK(cudaMemcpyAsync(var_out, d_acc + n_star, n_star * sizeof(double), cudaMemcpyDefault, st));
  int info;
  if (end_run(h, info)) return -2;
  static const char* names[] = {"?", "Kh", "Kx", "P of q(z)"};
  if (pd_error(h, info, names)) return -3;
  record_timing(h);
  return 0;
}

// Monte-Carlo kernel samples of VCGPCM.predict_k (src/core/cgpcm.py:610-634), before normalisation:
//   out[p][b] = s2_f (a_c(t_p) + tr((h_b h_b^T - iKh) Ahh_c(t_p)))
// The n x nh^2 matrix of centre statistics times the nh^2 x B matrix of (h h^T - iKh) is one DMMA GEMM per chunk.
int kernel_run(cgpcm_handle* h, const double* params_host, double reg, const double* t_host, long n,
               const double* samples_host, int B, double* out) {
  const int nh = h->nh;
  const long ld = h->ld;
  if (check_finite(h, params_host, 5, "non-finite parameter")) return -4;
  if (check_finite(h, t_host, n, "non-finite input")) return -4;
  if (check_samples(h, samples_host, B, nh)) return -4;
  const Hyp hp = hyp_of(params_host);
  const double alpha = hp.alpha, gamma = hp.gamma;
  PsiConst c;
  psi_make_const(alpha, gamma, hp.omega, h->causal, h->cull, &c, h->causal_id);
  cudaStream_t st = h->st;
  const int nhl = round_up(nh, 2);
  const long K = (long)nh * nhl;
  const int Bp = round_up(B, 8);
  const int TC = (int)std::min<long>(round_up((int)std::min<long>(n, 1024), 8), 1024);
  Scratch s;
  const size_t o_t = s.take(n), o_hs = s.take((size_t)B * nh), o_ac = s.take(TC), o_AC = s.take((size_t)TC * K);
  const size_t o_HH = s.take((size_t)Bp * K), o_G = s.take((size_t)TC * Bp), o_out = s.take((size_t)n * B);
  CK(s.alloc());
  double *d_t = s.at(o_t), *d_hs = s.at(o_hs), *d_ac = s.at(o_ac), *d_AC = s.at(o_AC), *d_HH = s.at(o_HH);
  double *d_G = s.at(o_G), *d_out = s.at(o_out);
  if (begin_run(h)) return -2;
  CK(cudaMemcpyAsync(d_t, t_host, n * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_hs, samples_host, (size_t)B * nh * sizeof(double), cudaMemcpyHostToDevice, st));
  if (prior_stage(h, c, reg, true)) return -2;                // Kh -> iKh (M_IKH)
  hh_build_kernel<<<148 * 4, 256, 0, st>>>(d_hs, nh, B, Bp, h->M(M_IKH), ld, nh, nhl, d_HH);
  L(h);
  for (long p0 = 0; p0 < n; p0 += TC) {
    const int nv = (int)std::min<long>(TC, n - p0);
    const int nvp = round_up(nv, 8);
    if (nvp > nv) CK(cudaMemsetAsync(d_AC + (long)nv * K, 0, (size_t)(nvp - nv) * K * sizeof(double), st));
    ahh_center_kernel<<<148 * 8, 256, 0, st>>>(d_t + p0, nv, h->th, nh, nhl, alpha, gamma, h->causal, d_AC, d_ac);
    L(h);
    // G[p][b] = sum_e AC[p][e] HH[b][e]
    if (gemm(h, true, true, false, nvp, Bp, (int)K, 1.0, d_AC, K, d_HH, K, 0.0, d_G, Bp)) return -2;
    kernel_finish_kernel<<<148 * 2, 256, 0, st>>>(d_G, Bp, d_ac, nv, B, hp.s2f, d_out + p0 * B);
    L(h);
  }
  CK(cudaMemcpyAsync(out, d_out, (size_t)n * B * sizeof(double), cudaMemcpyDefault, st));
  int info;
  if (end_run(h, info)) return -2;
  static const char* names[] = {"?", "Kh", "Kx"};
  if (pd_error(h, info, names)) return -3;
  record_timing(h);
  return 0;
}

// Posterior draws of the filter for VCGPCM.predict_h / predict_psd (src/core/cgpcm.py:663-779):
//   out[p][b] = (Kuh^T h_b)[p] + (L eps_b)[p],   A = Lh^-1 Kuh,   L = chol(reg(k_h(t, t) - A^T A))
// noise_host: eps as [n][B] (row p, column b).  Four DMMA GEMMs, one triangular inverse, one Cholesky.
int filter_run(cgpcm_handle* h, const double* params_host, double reg, const double* t_host, long n,
               const double* samples_host, int B, const double* noise_host, double* out) {
  const int nh = h->nh, nhp = h->nhp;
  const long ld = h->ld;
  if (check_finite(h, params_host, 5, "non-finite parameter")) return -4;
  if (check_finite(h, t_host, n, "non-finite input")) return -4;
  if (check_samples(h, samples_host, B, nh)) return -4;
  if (check_finite(h, noise_host, n * B, "non-finite noise")) return -4;
  if (n > 8192) { h->err = "predict_h / predict_psd: at most 8192 inputs"; return -1; }
  const Hyp hp = hyp_of(params_host);
  PsiConst c;
  psi_make_const(hp.alpha, hp.gamma, hp.omega, h->causal, h->cull, &c, h->causal_id);
  cudaStream_t st = h->st;
  const int ldn = round_up((int)n, 8);
  const int Bp = round_up(B, 8);
  Scratch s;
  const size_t o_t = s.take(n), o_kuh = s.take((size_t)nhp * ldn), o_ktt = s.take((size_t)ldn * ldn);
  const size_t o_a = s.take((size_t)nhp * ldn), o_hs = s.take((size_t)nhp * Bp), o_e = s.take((size_t)ldn * Bp);
  const size_t o_o = s.take((size_t)ldn * Bp);
  CK(s.alloc());
  double *d_t = s.at(o_t), *d_kuh = s.at(o_kuh), *d_ktt = s.at(o_ktt), *d_a = s.at(o_a), *d_hs = s.at(o_hs);
  double *d_e = s.at(o_e), *d_o = s.at(o_o);
  if (begin_run(h)) return -2;
  CK(cudaMemcpyAsync(d_t, t_host, n * sizeof(double), cudaMemcpyHostToDevice, st));
  // Hs[i][b] = samples[b][i] (transposed on the host), E[p][b] = noise[p][b]; zero padding
  std::vector<double> hs((size_t)nhp * Bp, 0.0), ee((size_t)ldn * Bp, 0.0);
  for (int b = 0; b < B; ++b)
    for (int i = 0; i < nh; ++i) hs[(size_t)i * Bp + b] = samples_host[(size_t)b * nh + i];
  for (long p2 = 0; p2 < n; ++p2)
    for (int b = 0; b < B; ++b) ee[(size_t)p2 * Bp + b] = noise_host[(size_t)p2 * B + b];
  CK(cudaMemcpyAsync(d_hs, hs.data(), hs.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_e, ee.data(), ee.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  if (prior_stage(h, c, reg, true)) return -2;                        // M_LH = chol(reg(Kh)), padded with the identity
  filter_kernels_kernel<<<148 * 4, 256, 0, st>>>(h->th, nh, nhp, d_t, (int)n, ldn, hp.alpha, hp.gamma, reg, d_kuh,
                                                 d_ktt);
  L(h);
  // X = Lh^-1 ;  A = X Kuh ;  S = Ktt - A^T A ;  L = chol(S)
  {
    cudaError_t e = trtri_lower(st, h->M(M_LH), h->M(M_T1), h->M(M_T2), nhp, ld);
    L(h, 20);
    if (e != cudaSuccess) { h->err = "trtri launch failed"; return -2; }
  }
  if (gemm(h, true, false, false, nhp, ldn, nhp, 1.0, h->M(M_T1), ld, d_kuh, ldn, 0.0, d_a, ldn)) return -2;
  if (gemm(h, false, false, false, ldn, ldn, nhp, -1.0, d_a, ldn, d_a, ldn, 1.0, d_ktt, ldn)) return -2;
  {
    cudaError_t e = potrf_lower(st, d_ktt, ldn, ldn, h->info, 5, h->M(M_XW));
    L(h, 20);
    if (e != cudaSuccess) { h->err = "potrf launch failed"; return -2; }
  }
  // out = Kuh^T Hs + L E
  if (gemm(h, false, false, false, ldn, Bp, nhp, 1.0, d_kuh, ldn, d_hs, Bp, 0.0, d_o, Bp)) return -2;
  if (gemm(h, true, false, false, ldn, Bp, ldn, 1.0, d_ktt, ldn, d_e, Bp, 1.0, d_o, Bp)) return -2;
  CK(cudaMemcpy2DAsync(out, (size_t)B * sizeof(double), d_o, (size_t)Bp * sizeof(double), (size_t)B * sizeof(double), n,
                       cudaMemcpyDefault, st));
  int info;
  if (end_run(h, info)) return -2;
  static const char* names[] = {"?", "Kh", "Kx", "?", "?", "k_h(t, t) - A^T A + reg I"};
  if (pd_error(h, info, names)) return -3;
  record_timing(h);
  return 0;
}

// One draw of the Approximate Kernel Model, AKM.f() (src/core/cgpcm.py:382-392):
//   K[p][q] = a(t_p, t_q) + tr((h h^T - iKh) Ahh(t_p, t_q)),   f = sqrt(s2_f) chol(reg(K)) e.
// The pair statistics _a / _Ahh (cgpcm.py:156-158,182-184: upper limit min(t, t')) only depend on the lag:
// shifting tau by t' turns them into the centre statistics at t - t' (oracle.model.psi_pairs_generic checks this on
// the reference's integrands), so K is kernel_run at the n^2 lags with s2_f divided out again.
int akm_run(cgpcm_handle* h, const double* params_host, double reg, const double* t_host, long n,
            const double* h_host, const double* e_host, double* f_out, double* K_out) {
  for (long i = 0; i < n; ++i)
    if (!std::isfinite(t_host[i]) || !std::isfinite(e_host[i])) { h->err = "non-finite input"; return -4; }
  if (n > 4096) { h->err = "AKM sample: at most 4096 inputs"; return -1; }
  const double s2f = hyp_of(params_host).s2f;
  cudaStream_t st = h->st;
  const int ldn = round_up((int)n, 8);
  std::vector<double> lags((size_t)n * n);
  for (long p2 = 0; p2 < n; ++p2)
    for (long q = 0; q < n; ++q) lags[(size_t)p2 * n + q] = t_host[p2] - t_host[q];
  Scratch s;
  const size_t o_k = s.take((size_t)n * n), o_K = s.take((size_t)ldn * ldn), o_e = s.take(ldn), o_f = s.take(ldn);
  CK(s.alloc());
  double *d_k = s.at(o_k), *d_K = s.at(o_K), *d_e = s.at(o_e), *d_f = s.at(o_f);
  if (int rc = kernel_run(h, params_host, reg, lags.data(), n * n, h_host, 1, d_k)) return rc;   // s2_f (a + tr(..)) per lag
  // this run's own part: timed from a new ev[0] and added to the kernel_run part; the counters go on
  CK(cudaEventRecord(h->ev[0], st));
  CK(cudaMemsetAsync(h->info, 0, 4 * sizeof(int), st));
  CK(cudaMemsetAsync(d_e, 0, (size_t)ldn * sizeof(double), st));
  CK(cudaMemcpyAsync(d_e, e_host, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
  {
    const double* kk = d_k;
    double* Kp = d_K;
    const long nn = n;
    const double inv = 1.0 / s2f;
    ew(st, (long)ldn * ldn, [=] __device__(long idx) {
      const int r = (int)(idx / ldn), q = (int)(idx - (long)r * ldn);
      double v = (r == q) ? 1.0 : 0.0;                       // identity on the padding block
      if (r < nn && q < nn) v = kk[(long)r * nn + q] * inv + (r == q ? reg : 0.0);
      Kp[idx] = v;
    });
    L(h);
  }
  if (K_out)
    CK(cudaMemcpy2DAsync(K_out, (size_t)n * sizeof(double), d_K, (size_t)ldn * sizeof(double), (size_t)n * sizeof(double),
                         n, cudaMemcpyDefault, st));
  {
    cudaError_t e = potrf_lower(st, d_K, ldn, ldn, h->info, 6, h->M(M_XW));
    L(h, 2 * ((ldn + LA_NB - 1) / LA_NB));
    if (e != cudaSuccess) { h->err = "potrf launch failed"; return -2; }
  }
  matvec_kernel<<<(ldn + 7) / 8, 256, 0, st>>>(d_K, ldn, ldn, ldn, 0, d_e, sqrt(s2f), d_f);
  L(h);
  CK(cudaMemcpyAsync(f_out, d_f, (size_t)n * sizeof(double), cudaMemcpyDefault, st));
  int info;
  if (end_run(h, info)) return -2;
  if (info) h->prior_valid = false;
  if (info) { h->err = "AKM covariance a + tr((h h^T - iKh) Ahh) + reg I is not positive definite"; return -3; }
  const double kernel_ms = h->timing[0];
  record_timing(h);
  h->timing[0] += kernel_ms;
  return 0;
}

// Samples per internal batch of smf_batch_run: a function of the handle's shape only (the W GEMM always runs with this
// many rows, zero rows past the batch, so that its launch does not depend on the number of samples).  Seven ld x ld
// slabs per sample (SMF_SLICES partials, C1, the factors of P and P0) within ~1 GB.
int smf_bcap(const cgpcm_handle* h) {
  const double per = (SMF_SLICES + 3.0) * (double)h->ld * h->ld * sizeof(double);
  const int b = (int)std::min(64.0, 1e9 / per) / 8 * 8;
  return std::max(8, b);
}

// nb <= bcap samples (host, nb x nh) into d_hs (bcap x nhp, zero past each sample and past nb)
int stage_samples(cgpcm_handle* h, const double* samples_host, int nb, int bcap, double* d_hs) {
  const int nh = h->nh, nhp = h->nhp;
  std::vector<double> hsm((size_t)bcap * nhp, 0.0);
  for (int b = 0; b < nb; ++b)
    for (int i = 0; i < nh; ++i) hsm[(size_t)b * nhp + i] = samples_host[(size_t)b * nh + i];
  // (pageable source: staged before the call returns)
  CK(cudaMemcpyAsync(d_hs, hsm.data(), hsm.size() * sizeof(double), cudaMemcpyHostToDevice, h->st));
  return 0;
}

// The per-batch C1 stage of the batched SMF paths: stage nb <= bcap samples into d_hs (stage_samples), then per chunk
// W = H_B A (the small-left GEMM over the resident or regenerated Ahx block, always bcap rows) and part_b += W_b^T W_b
// (smf_c1_kernel), the slice sum into the C1 slabs and one all-reduce of them.
int smf_c1_stage(cgpcm_handle* h, const std::vector<Chunk>& chunks, const double* samples_host, int nb, int bcap,
                 double* d_hs, double* d_part, double* d_c1, double* d_w, long wstride) {
  const int nx = h->nx, nhp = h->nhp;
  const long ld = h->ld, l2 = ld * ld;
  cudaStream_t st = h->st;
  if (stage_samples(h, samples_host, nb, bcap, d_hs)) return -2;
  CK(cudaMemsetAsync(d_part, 0, (size_t)nb * SMF_SLICES * l2 * sizeof(double), st));
  const bool stor = h->use_store;
  const bool have_a = stor && h->storeA_frozen_valid;
  for (const Chunk& ch : chunks) {
    double* Ab = stor ? h->storeA + ch.off : h->wsA;
    if (!have_a && gen_chunk(h, h->fc, ch, false, Ab)) return -2;
    const long cols = (long)ch.nc * ch.kwp;
    // W[b][(n,k)] = sum_i h_b[i] A[i][(n,k)]
    if (gemm(h, true, false, false, bcap, (int)cols, nhp, 1.0, d_hs, nhp, Ab, cols, 0.0, d_w, wstride)) return -2;
    prof_close(h);
    smf_c1_launch(st, d_w, wstride, ch.kwp, ch.nc, ch.k_lo, d_part, ld, nb);
    h->gemm_flops += (double)nb * ch.nc * ch.kwp * (ch.kwp + 1.0);
    L(h);
  }
  if (stor) h->storeA_frozen_valid = true;
  smf_reduce_launch(st, d_part, ld, nx, nb, d_c1);
  L(h);
  return allreduce(h, d_c1, (long)nb * l2);
}

// The training side of the batched prediction paths with smf = 1, for the nb <= bcap samples from b0: the C1 stage,
// smf_posterior_kernel (P_b, xm_b, mx_b and q1_b with the constant term a) and the check of each P_b.
int smf_posterior_stage(cgpcm_handle* h, const std::vector<Chunk>& chunks, const double* samples_host, int b0, int nb,
                        int bcap, double* hs, double* part, double* c1, double* w, long wcols, double* work, int* info,
                        double* mx, double* xm, double* q1, double r, double c0, double reg, double a_val) {
  cudaStream_t st = h->st;
  if (smf_c1_stage(h, chunks, samples_host + (size_t)b0 * h->nh, nb, bcap, hs, part, c1, w, wcols)) return -2;
  SmfPostArgs a;
  a.kx = h->M(M_KX); a.sxx = h->M(M_F_AXX); a.c1 = c1; a.fy = h->M(M_F_Y); a.ahh = h->M(M_AHH);
  a.ikx = h->M(M_IKX); a.tr = h->sc + S_TR_IKH_AHH; a.hs = hs; a.work = work;
  a.mx = mx; a.xm = xm; a.q1 = q1; a.info = info;
  a.ld = h->ld; a.l2 = h->ld * h->ld; a.ldh = h->nhp; a.nh = h->nh; a.nx = h->nx; a.nb = nb;
  a.r = r; a.c0 = c0; a.reg = reg; a.a = a_val;
  CK(cudaMemsetAsync(info, 0, bcap * sizeof(int), st));
  smf_posterior_launch(st, a, bcap);
  L(h);
  CK(cudaGetLastError());
  std::vector<int> inf(bcap);
  CK(cudaMemcpyAsync(inf.data(), info, bcap * sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  for (int b = 0; b < nb; ++b)
    if (inf[b]) return sample_pd_error(h, "P", b0 + b, inf[b]);
  return 0;
}

// VCGPCM.elbo(smf=True, sample=h_b) and the slice sampler's log-likelihood (src/core/cgpcm.py:527-531,594-608,848-872)
// for B samples in the frozen regime.  Per call: the terms that do not depend on the sample (the prior, q(u) and
// its KL, the frozen sums), as evaluate_once forms them.  Per batch of <= smf_bcap samples: per chunk W = H_B A (the
// small-left GEMM over the resident or regenerated Ahx block) and C1_b += W_b^T W_b (smf_c1_kernel), one all-reduce
// of the C1 slabs, then the factorisations of P_b (want_p) and P0_b (want_p0) in one launch.
int smf_batch_run(cgpcm_handle* h, const double* params_host, double reg, const double* samples_host, int B,
                  bool want_p, bool want_p0, double* elbo_out, double* terms_out, double* loglik_out) {
  const int nh = h->nh, nx = h->nx, nhp = h->nhp;
  const long ld = h->ld, l2 = ld * ld;
  const long np = 5 + nh + (long)nh * (nh + 1) / 2;
  if (check_finite(h, params_host, np, "non-finite parameter")) return -4;
  if (check_samples(h, samples_host, B, nh)) return -4;
  if (!h->frozen) { h->err = "cgpcm_elbo_smf_batch requires cgpcm_precompute"; return -1; }
  if (!want_p && !want_p0) return 0;
  const Hyp hp = hyp_of(params_host);
  const double r = hp.r, c0 = hp.c0;
  if (ensure_sweep_buffers(h)) return -2;
  PsiConst c;
  psi_make_const(hp.alpha, hp.gamma, hp.omega, h->causal, h->cull, &c, h->causal_id);
  std::vector<Chunk> chunks;
  plan_chunks(h, h->fc, chunks);
  if (ensure_ypart(h, y_slices_used(chunks))) return -2;
  if (plan_store(h, chunks, false)) return -2;
  const int bcap = smf_bcap(h);
  const int passes = (want_p ? 1 : 0) + (want_p0 ? 1 : 0);
  long wcols = 0;
  for (const Chunk& ch : chunks) wcols = std::max<long>(wcols, (long)ch.nc * ch.kwp);
  // [hs: bcap x nhp][out: bcap x 5 (+ pad)][part: bcap x SMF_SLICES slabs][c1: bcap slabs][work: 2 bcap slabs][W]
  const long o_hs = 0, o_out = o_hs + (long)bcap * nhp, o_part = o_out + round_up(bcap * 5, 8);
  const long o_c1 = o_part + (long)bcap * SMF_SLICES * l2, o_work = o_c1 + (long)bcap * l2;
  const long o_w = o_work + 2L * bcap * l2, need = o_w + (long)bcap * wcols;
  if (need > h->smf_elems) {
    if (h->smf_buf) cudaFree(h->smf_buf);
    h->smf_buf = nullptr; h->smf_elems = 0;
    CK(cudaMalloc(&h->smf_buf, need * sizeof(double)));
    h->smf_elems = need;
  }
  if (2 * bcap > h->smf_info_count) {
    if (h->smf_info) cudaFree(h->smf_info);
    h->smf_info = nullptr; h->smf_info_count = 0;
    CK(cudaMalloc(&h->smf_info, 2 * bcap * sizeof(int)));
    h->smf_info_count = 2 * bcap;
  }
  double* d_hs = h->smf_buf + o_hs;
  double* d_out = h->smf_buf + o_out;
  double* d_part = h->smf_buf + o_part;
  double* d_c1 = h->smf_buf + o_c1;
  double* d_work = h->smf_buf + o_work;
  double* d_w = h->smf_buf + o_w;

  cudaStream_t st = h->st;
  if (begin_run(h)) return -2;
  CK(cudaMemcpyAsync(h->params_d, params_host, np * sizeof(double), cudaMemcpyHostToDevice, st));
  // ---- the terms that do not depend on the sample (evaluate_once, MODE_FROZEN)
  if (prior_stage(h, c, reg, true, true)) return -2;
  if (qu_moments(h, reg)) return -2;
  if (prior_join(h)) return -2;
  if (kl_fork(h, reg)) return -2;
  frob(h, h->M(M_F_BHH), h->M(M_M2), nh, nh, h->sc + S_TR_BHH_M2);
  {
    double tail[2] = {(double)h->n_local, h->sum_y2_local};
    CK(cudaMemcpyAsync(h->fwd_tail, tail, sizeof tail, cudaMemcpyHostToDevice, st));
  }
  if (allreduce(h, h->fwd_tail, 2)) return -2;
  if (side_join(h, 0)) return -2;
  if (side_join(h, 1)) return -2;
  kl_scalars(h);
  double hs[S_COUNT + 16];
  int info[4];
  CK(cudaMemcpyAsync(hs, h->sc, sizeof hs, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(info, h->info, sizeof info, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  static const char* names[] = {"?", "Kh", "Kx", "P", "iKh + reg I (prior of q(u))", "q(u) covariance"};
  if (pd_error(h, info[0], names)) return -3;
  double tm[7];
  fixed_terms(h, hs, hp.s2, r, h->f_sum_b, hs[S_TR_BHH_M2], tm);

  // ---- batches of samples
  std::vector<double> res((size_t)bcap * 5);
  std::vector<int> inf((size_t)2 * bcap);
  for (int b0 = 0; b0 < B; b0 += bcap) {
    const int nb = std::min(bcap, B - b0);
    if (smf_c1_stage(h, chunks, samples_host + (size_t)b0 * nh, nb, bcap, d_hs, d_part, d_c1, d_w, wcols)) return -2;
    SmfAlgArgs a;
    a.kx = h->M(M_KX); a.sxx = h->M(M_F_AXX); a.c1 = d_c1; a.fy = h->M(M_F_Y); a.bhh = h->M(M_F_BHH);
    a.hs = d_hs; a.work = d_work; a.out = d_out; a.info = h->smf_info;
    a.ld = ld; a.l2 = l2; a.ldh = nhp; a.nh = nh; a.nx = nx;
    a.r = r; a.c0 = c0; a.reg = reg; a.want_p = want_p; a.passes = passes;
    CK(cudaMemsetAsync(h->smf_info, 0, 2 * bcap * sizeof(int), st));
    smf_algebra_launch(st, a, nb);
    L(h);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(res.data(), d_out, (size_t)nb * 5 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(inf.data(), h->smf_info, (size_t)nb * 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int b = 0; b < nb; ++b)
      for (int k = 0; k < 2; ++k)
        if (inf[2 * b + k]) return sample_pd_error(h, k == 0 ? "P" : "P0 (no jitter)", b0 + b, inf[2 * b + k]);
    for (int b = 0; b < nb; ++b) {
      const double* o = &res[(size_t)b * 5];
      if (want_p) {
        double t[7];
        memcpy(t, tm, sizeof t);
        t[2] = -0.5 * o[0];
        t[3] = 0.5 * o[1];
        double e = 0.0;
        for (int i = 0; i < 7; ++i) e += t[i];
        if (elbo_out) elbo_out[b0 + b] = e;
        if (terms_out) memcpy(terms_out + (size_t)(b0 + b) * 7, t, sizeof t);
      }
      if (want_p0) loglik_out[b0 + b] = -0.5 * o[2] + 0.5 * o[3] - 0.5 * r * o[4];
    }
  }
  int info_end;      // the prior's, checked above
  if (end_run(h, info_end)) return -2;
  record_timing(h);
  return 0;
}

// Samples per internal batch of predict_batch_run: a function of the handle's shape and the test chunk budget only
// (every launch of the batch is shaped for this many samples).  Per sample: the C1 partials and slab and the two slabs
// of smf_posterior_kernel (SMF_SLICES + 3 ld x ld), and V_b of a test chunk (chunk x nxp), within ~1 GB.
int predict_bcap(const cgpcm_handle* h, int chunk) {
  const double per = ((SMF_SLICES + 3.0) * (double)h->ld * h->ld + (double)chunk * h->nxp) * sizeof(double);
  const int b = (int)std::min(64.0, 1e9 / per) / 8 * 8;
  return std::max(8, b);
}

// Budget of the test chunks and sample batches of the batched prediction paths: the chunk the planner chose for this
// rank's observations (plan_chunks).  With several ranks the largest over the ranks, so that every rank cuts the test
// inputs and sizes its batches alike: a rank plans from its own observations only, and one without any keeps 512.
int test_chunk(cgpcm_handle* h, int& chunk) {
  chunk = h->chunk;
  if (h->world <= 1) return 0;
  Scratch s;
  const size_t o = s.take(1, sizeof(int));
  CK(s.alloc());
  int* d = s.at<int>(o);
  CK(cudaMemcpyAsync(d, &chunk, sizeof(int), cudaMemcpyHostToDevice, h->st));
  if (allreduce(h, d, 1, NCCL_INT32, NCCL_MAX)) return -2;
  CK(cudaMemcpyAsync(&chunk, d, sizeof(int), cudaMemcpyDeviceToHost, h->st));
  CK(cudaStreamSynchronize(h->st));
  return 0;
}

// The training side shared by all samples of the batched prediction paths: with smf = 0 the one q(z) of q(u)
// (predict_qz) and mx = P^-1 + xm xm^T - iKx, dense nx x nx as the test-side kernels read it; then the check of the
// factorisations of the prior and of that q(z).
int shared_qz_stage(cgpcm_handle* h, const std::vector<Chunk>& chunks, int smf, double r, double c0, double reg,
                    double* xm, double* mx) {
  if (!smf) {
    if (predict_qz(h, chunks, 0, h->V(V_MU), h->M(M_VAR), r, c0, reg, xm)) return -2;
    const int nx = h->nx;
    const long ld = h->ld;
    const double* xv = h->M(M_PINV);
    const double* ikx = h->M(M_IKX);
    ew(h->st, (long)nx * nx, [=] __device__(long idx) {
      const int i = (int)(idx / nx), j = (int)(idx % nx);
      const long e = (long)i * ld + j;
      mx[idx] = xv[e] + xm[i] * xm[j] - ikx[e];
    });
    L(h);
  }
  int info[4];
  CK(cudaMemcpyAsync(info, h->info, sizeof info, cudaMemcpyDeviceToHost, h->st));
  CK(cudaStreamSynchronize(h->st));
  static const char* names[] = {"?", "Kh", "Kx", "P of q(z)"};
  return pd_error(h, info[0], names);
}

// nb dense nx x nx mx slabs (ld x ld apart) into the padded nxp x nxp layout of the rank-one GEMMs
void pad_mx(cgpcm_handle* h, const double* mx, int nb, double* mxp) {
  const int nx = h->nx, nxp = h->nxp;
  const long l2 = h->ld * h->ld, pp = (long)nxp * nxp;
  ew(h->st, (long)nb * pp, [=] __device__(long idx) {
    const int b = (int)(idx / pp);
    const long e = idx - (long)b * pp;
    const int i = (int)(e / nxp), j = (int)(e % nxp);
    mxp[idx] = (i < nx && j < nx) ? mx[(long)b * l2 + (long)i * nx + j] : 0.0;
  });
  L(h);
}

// predict_f's moments for each of B filter samples (and their average, as predict_run forms it) in the frozen regime.
// Training side: smf = 0, the one q(z) of q(u) (predict_qz, as predict_run); smf = 1, per batch of bcap samples the C1
// stage of smf_batch_run and smf_posterior_kernel (P_b, xm_b, mx_b, q1_b).  Test side, per chunk of test points: A* and
// Bxx* once (predict_chunk_blocks), then per batch V = H_B A* (small-left GEMM), Qb = <Bxx*, mx_b> (predict_qb_kernel),
// v^T mx_b v and v . xm_b (predict_quad_kernel) and predict_finish_kernel.  With smf = 1 the samples go in groups whose
// mx slabs fit ~1 GB; A* and Bxx* are rebuilt per group.  With several ranks every rank runs the training side (its
// sums are all-reduced), test chunk ci is computed by rank ci % world only, and the outputs, zero where another rank
// owns the chunk, are all-reduced once at the end: each element has one non-zero contributor, so the sum is exact.
int predict_batch_run(cgpcm_handle* h, const double* params_host, double reg, const double* tstar_host, long n_star,
                      const double* samples_host, int B, int smf, double* mu_out, double* var_out, double* mean_s_out,
                      double* var_s_out) {
  const int nh = h->nh, nx = h->nx, nhp = h->nhp, nxp = h->nxp;
  const long ld = h->ld, l2 = ld * ld;
  const long np = 5 + nh + (long)nh * (nh + 1) / 2;
  if (check_finite(h, params_host, np, "non-finite parameter")) return -4;
  if (check_finite(h, tstar_host, n_star, "non-finite test input")) return -4;
  if (check_samples(h, samples_host, B, nh)) return -4;
  if (!h->frozen) { h->err = "cgpcm_predict_f_batch requires cgpcm_precompute"; return -1; }
  const Hyp hp = hyp_of(params_host);
  const double r = hp.r, c0 = hp.c0, s2f = hp.s2f;
  if (ensure_sweep_buffers(h)) return -2;
  PsiConst c;
  psi_make_const(hp.alpha, hp.gamma, hp.omega, h->causal, h->cull, &c, h->causal_id);
  PsiConst cd = c;                       // test-side statistics are evaluated densely (no windows)
  cd.cull = 746.0;
  BvnTab T;
  bvn_make_tab(hp.gamma / (hp.alpha + hp.gamma + hp.omega), &T);
  std::vector<Chunk> chunks;
  plan_chunks(h, h->fc, chunks);
  if (ensure_ypart(h, y_slices_used(chunks))) return -2;
  cudaStream_t st = h->st;
  int tchunk;
  if (test_chunk(h, tchunk)) return -2;
  const int TC = std::min<long>(tchunk, n_star);
  const int TCP = round_up(TC, 8);
  const int bcap = predict_bcap(h, tchunk);
  const int gcap = smf ? std::max(bcap, std::min(round_up(B, bcap), (int)(1e9 / (l2 * 8.0)) / bcap * bcap))
                       : round_up(B, bcap);
  const int nq = smf ? gcap : 1;         // q(z) slabs held at a time
  long wcols = 0;
  for (const Chunk& ch : chunks) wcols = std::max<long>(wcols, (long)ch.nc * ch.kwp);
  const bool per_sample = mean_s_out || var_s_out;
  // [t][acc 2 n*][per-sample 2 n* B][X][hs][q1][xm][mx][part][c1][work][W][V][qpart][quad][lin][info]
  Scratch s;
  const size_t o_t = s.take(n_star), o_acc = s.take(2 * n_star), o_ps = s.take(per_sample ? 2 * n_star * B : 0);
  const size_t o_x = s.take((size_t)TC * nx * nx), o_hs = s.take((size_t)gcap * nhp), o_q1 = s.take(gcap);
  const size_t o_xm = s.take((size_t)nq * ld), o_mx = s.take((size_t)nq * l2);
  const size_t o_part = s.take(smf ? (size_t)bcap * SMF_SLICES * l2 : 0), o_c1 = s.take(smf ? (size_t)bcap * l2 : 0);
  const size_t o_work = s.take(smf ? 2 * (size_t)bcap * l2 : 0), o_w = s.take(smf ? (size_t)bcap * wcols : 0);
  const long vstride = (long)TCP * nxp;
  const size_t o_v = s.take((size_t)bcap * vstride), o_qp = s.take((size_t)PQ_SLICES * TC * bcap);
  const size_t o_quad = s.take((size_t)TC * bcap), o_lin = s.take((size_t)TC * bcap);
  const size_t o_info = s.take(bcap, sizeof(int));
  CK(s.alloc());
  double *d_t = s.at(o_t), *d_acc = s.at(o_acc), *d_ps = s.at(o_ps), *d_x = s.at(o_x), *d_hs = s.at(o_hs);
  double *d_q1 = s.at(o_q1), *d_xm = s.at(o_xm), *d_mx = s.at(o_mx), *d_part = s.at(o_part), *d_c1 = s.at(o_c1);
  double *d_work = s.at(o_work), *d_w = s.at(o_w), *d_v = s.at(o_v), *d_qp = s.at(o_qp), *d_quad = s.at(o_quad);
  double* d_lin = s.at(o_lin);
  int* d_info = s.at<int>(o_info);
  if (begin_run(h)) return -2;
  CK(cudaMemcpyAsync(h->params_d, params_host, np * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_t, tstar_host, n_star * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemsetAsync(d_acc, 0, (size_t)2 * n_star * sizeof(double), st));
  if (h->world > 1 && per_sample) CK(cudaMemsetAsync(d_ps, 0, (size_t)2 * n_star * B * sizeof(double), st));
  if (prior_stage(h, c, reg, true)) return -2;
  if ((smf || !h->gram_valid) && plan_store(h, chunks, false)) return -2;
  if (predict_qu(h, reg)) return -2;
  const double a_val = (h->causal ? 0.5 : 1.0) * sqrt(3.14159265358979323846 / (2.0 * hp.alpha));
  if (int rc = shared_qz_stage(h, chunks, smf, r, c0, reg, d_xm, d_mx)) return rc;
  const double w = 1.0 / B;
  for (int g0 = 0; g0 < B; g0 += gcap) {
    const int gn = std::min(gcap, B - g0);
    const int nbat = (gn + bcap - 1) / bcap;
    // ---- training side of the group
    for (int bi = 0; bi < nbat; ++bi) {
      const int b0 = g0 + bi * bcap, nb = std::min(bcap, B - b0);
      double* hs = d_hs + (long)bi * bcap * nhp;
      double* q1 = d_q1 + (long)bi * bcap;
      if (smf) {
        if (int rc = smf_posterior_stage(h, chunks, samples_host, b0, nb, bcap, hs, d_part, d_c1, d_w, wcols, d_work,
                                         d_info, d_mx + (long)bi * bcap * l2, d_xm + (long)bi * bcap * ld, q1, r, c0,
                                         reg, a_val))
          return rc;
      } else {
        if (stage_samples(h, samples_host + (size_t)b0 * nh, nb, bcap, hs)) return -2;
        predict_q1_kernel<<<bcap, 256, 0, st>>>(h->M(M_AHH), ld, hs, nhp, nh, nb, a_val, h->sc + S_TR_IKH_AHH, q1);
        L(h);
      }
    }
    // ---- test side of the group, chunk by chunk
    for (long p0 = 0; p0 < n_star; p0 += TC) {
      if ((p0 / TC) % h->world != h->rank) continue;
      const int nv = (int)std::min<long>(TC, n_star - p0);
      const long cols = (long)round_up(nv, 8) * nxp;
      if (predict_chunk_blocks(h, cd, T, d_t + p0, nv, d_x)) return -2;
      if (!smf) {
        predict_qb_launch(st, d_x, (long)nx * nx, d_mx, l2, 1, nv, TC, 1, d_qp, bcap);     // one column
        L(h);
      }
      for (int bi = 0; bi < nbat; ++bi) {
        const int b0 = g0 + bi * bcap, nb = std::min(bcap, B - b0);
        const double* hs = d_hs + (long)bi * bcap * nhp;
        // V[b][(n,k)] = sum_i h_b[i] A*[i][(n,k)]
        if (gemm(h, true, false, false, bcap, (int)cols, nhp, 1.0, hs, nhp, h->wsA, cols, 0.0, d_v, vstride)) return -2;
        prof_close(h);
        const double* mx = smf ? d_mx + (long)bi * bcap * l2 : d_mx;
        const double* xm = smf ? d_xm + (long)bi * bcap * ld : d_xm;
        if (smf) {
          predict_qb_launch(st, d_x, (long)nx * nx, mx, l2, nb, nv, TC, bcap, d_qp, bcap);
          L(h);
        }
        PredQuadArgs qa;
        qa.V = d_v; qa.v_stride = vstride; qa.ldv = nxp;
        qa.mx = mx; qa.mx_stride = smf ? l2 : 0; qa.xm = xm; qa.xm_stride = smf ? ld : 0;
        qa.nv = nv; qa.nx = nx; qa.nb = nb; qa.quad = d_quad; qa.lin = d_lin; qa.ldo = bcap;
        predict_quad_launch(st, qa, bcap);
        L(h);
        predict_finish_kernel<<<(nv + 127) / 128, 128, 0, st>>>(
            d_qp, TC, bcap, smf ? 1 : 0, d_quad, d_lin, bcap, d_q1 + (long)bi * bcap, nv, nb, sqrt(s2f), s2f, w,
            mean_s_out ? d_ps + p0 * B + b0 : nullptr, var_s_out ? d_ps + (n_star + p0) * B + b0 : nullptr, B,
            d_acc + p0, d_acc + n_star + p0);
        L(h);
      }
    }
    CK(cudaGetLastError());
  }
  if (allreduce(h, d_acc, 2 * n_star)) return -2;
  if (per_sample && allreduce(h, d_ps, 2 * n_star * B)) return -2;
  if (mu_out) CK(cudaMemcpyAsync(mu_out, d_acc, n_star * sizeof(double), cudaMemcpyDefault, st));
  if (var_out) CK(cudaMemcpyAsync(var_out, d_acc + n_star, n_star * sizeof(double), cudaMemcpyDefault, st));
  if (mean_s_out) CK(cudaMemcpyAsync(mean_s_out, d_ps, n_star * B * sizeof(double), cudaMemcpyDefault, st));
  if (var_s_out) CK(cudaMemcpyAsync(var_s_out, d_ps + n_star * B, n_star * B * sizeof(double), cudaMemcpyDefault, st));
  int info;          // the prior's and the shared q(z)'s, checked above
  if (end_run(h, info)) return -2;
  record_timing(h);
  return 0;
}

// Points per side of a pair tile of predict_cov_run: a function of nx only.  The tile's pair blocks (P^2 nx^2) and its
// fold (P nxp)^2 stay within ~1 GB.
int pcov_tile(const cgpcm_handle* h) {
  const int tp = (int)sqrt(6e7 / ((double)h->nxp * h->nxp)) / 8 * 8;
  return std::max(8, std::min(64, tp));
}

// The joint predictive covariance of f at n_star <= 4096 test inputs for each of B filter samples, and draws of f
// (cgpcm_predict_f_cov).  Training side as predict_batch_run: smf = 0 the one q(z) of q(u) (predict_qz); smf = 1 per
// batch of predict_bcap samples the C1 stage and smf_posterior_kernel.  Test side, once: A* and T = iKh A* for all test
// inputs.  Per group of samples (their covariance slabs within ~4 GB):
//   per batch   V = H_B A* (small-left GEMM), the means (predict_quad_kernel's v . xm_b), and per sample the rank-one
//               term R_b = (V_b mx_b) V_b^T into C_b (two GEMMs);
//   per tile    of P x Q points with p >= q: the fold A*_p^T T_q (one GEMM), the pair blocks Bxx* (axx_pair_kernel), the
//               centre statistics at the tile's lags (ahh_center_kernel) and, per batch, <Ahh_c, hh_b - iKh> (GEMM),
//               <Bxx*, mx_b> (predict_qb_kernel) and pcov_finish_kernel;
//   then        cov += C_b / B in ascending b, and per sample chol(C_b + reg I) (identity on the padding) and the draw;
//   scoring     (y_host given, cgpcm_predict_logpdf) per sample the bordered K_b = [[C_b + d I, y - m_b], [.., c]]
//               (pcov_border_kernel), its Cholesky factor, and per group pcov_score_kernel: lp_s[b] and the whitened
//               residuals; d = s2 with noise = 1 (observations), reg with noise = 0 (f itself).
// Every launch is shaped by the handle, n_star and the internal batch size, and no sum runs across samples except cov,
// so a sample's mean, C_b, draw, lp_s and whitened residuals are bitwise the same in any batch and at any position.
// Several ranks: every rank runs the training side, A*, T, V, the means and R_b.  Pair tile k is computed by rank
// k % world only and the tiles of the group's C_b are gathered (pcov_pack_kernel, ncclAllGather, pcov_unpack_kernel),
// so every rank holds every C_b and adds cov.  Sample b of a group is factorised (draw, score) by rank b % world only;
// draws, lp_s and whitened residuals, zero where another rank owns the sample, are all-reduced once at the end, and
// the info words per group before any rank decides, so that every rank returns the same code and message.  The
// tiles, groups and launch shapes do not depend on the world size (the batch size only on the test chunk budget,
// test_chunk), so no output changes a bit with it.
int predict_cov_run(cgpcm_handle* h, const double* params_host, double reg, const double* tstar_host, long n_star,
                    const double* samples_host, int B, int smf, const double* noise_host, double* mean_s_out,
                    double* cov_s_out, double* cov_out, double* draws_out, const double* y_host, int noise,
                    double* lp_s_out, double* white_out) {
  const int nh = h->nh, nx = h->nx, nhp = h->nhp, nxp = h->nxp;
  const long ld = h->ld, l2 = ld * ld;
  const long np = 5 + nh + (long)nh * (nh + 1) / 2;
  if (check_finite(h, params_host, np, "non-finite parameter")) return -4;
  if (check_finite(h, tstar_host, n_star, "non-finite test input")) return -4;
  if (check_samples(h, samples_host, B, nh)) return -4;
  if (noise_host && check_finite(h, noise_host, n_star * B, "non-finite noise")) return -4;
  if (y_host && check_finite(h, y_host, n_star, "non-finite y_star")) return -4;
  if (!h->frozen) {
    h->err = y_host ? "cgpcm_predict_logpdf requires cgpcm_precompute" : "cgpcm_predict_f_cov requires cgpcm_precompute";
    return -1;
  }
  const bool want_draws = draws_out && noise_host;
  const bool want_score = y_host != nullptr;
  const Hyp hp = hyp_of(params_host);
  const double r = hp.r, c0 = hp.c0, s2f = hp.s2f, alpha = hp.alpha, gamma = hp.gamma;
  if (ensure_sweep_buffers(h)) return -2;
  PsiConst c;
  psi_make_const(alpha, gamma, hp.omega, h->causal, h->cull, &c, h->causal_id);
  PsiConst cd = c;                       // test-side statistics are evaluated densely (no windows)
  cd.cull = 746.0;
  BvnTab T;
  bvn_make_tab(gamma / (alpha + gamma + hp.omega), &T);
  std::vector<Chunk> chunks;
  plan_chunks(h, h->fc, chunks);
  if (ensure_ypart(h, y_slices_used(chunks))) return -2;
  cudaStream_t st = h->st;
  const int n = (int)n_star, npad = round_up(n, 8);
  const long n2 = (long)npad * npad;
  const int TP = pcov_tile(h);
  const int TPP = TP * TP;               // pairs of a full tile (a multiple of 8)
  const int nhl = round_up(nh, 2);
  const long KH = (long)nh * nhl;
  int tchunk;
  if (test_chunk(h, tchunk)) return -2;
  const int bcap = predict_bcap(h, tchunk);
  const int ldk = round_up(n + 1, 8);    // the bordered matrix of the scoring stage
  const long k2 = (long)ldk * ldk;
  const double per = 8.0 * ((double)n2 + (double)KH + (double)nxp * nxp + (smf ? (double)l2 : 0.0) +
                            (want_score ? (double)k2 : 0.0));
  const int gcap = std::max(bcap, std::min(round_up(B, bcap), (int)std::min(1e6, 4e9 / per) / bcap * bcap));
  const int nq = smf ? gcap : 1;         // q(z) slabs held at a time
  long wcols = 0;
  for (const Chunk& ch : chunks) wcols = std::max<long>(wcols, (long)ch.nc * ch.kwp);
  const long acols = (long)npad * nxp;   // columns of A* / T: [i][p][k]
  const int ntile = (n + TP - 1) / TP;
  const long ntp = (long)ntile * (ntile + 1) / 2;            // pair tiles p >= q
  const int rank = h->rank, world = h->world;
  const long slots = world > 1 ? (ntp + world - 1) / world : 0;   // tiles per rank in the gather
  Scratch s;
  const size_t o_t = s.take(n), o_a = s.take((size_t)nhp * acols), o_ta = s.take((size_t)nhp * acols);
  const size_t o_mean = s.take((size_t)n * B), o_draw = s.take(want_draws ? (size_t)n * B : 0);
  const size_t o_noise = s.take(want_draws ? (size_t)B * npad : 0), o_cov = s.take(cov_out ? n2 : 0);
  const size_t o_x = s.take((size_t)TPP * nx * nx), o_g = s.take((size_t)TPP * nxp * nxp);
  const size_t o_ac = s.take(TPP), o_lag = s.take(TPP), o_AC = s.take((size_t)TPP * KH);
  const size_t o_gf = s.take((size_t)TPP * bcap), o_qp = s.take((size_t)PQ_SLICES * TPP * bcap);
  const size_t o_hs = s.take((size_t)gcap * nhp), o_q1 = s.take(gcap), o_xm = s.take((size_t)nq * ld);
  const size_t o_mx = s.take((size_t)nq * l2), o_mxp = s.take((size_t)nq * nxp * nxp);
  const size_t o_hh = s.take((size_t)gcap * KH), o_c = s.take((size_t)gcap * n2);
  const size_t o_part = s.take(smf ? (size_t)bcap * SMF_SLICES * l2 : 0), o_c1 = s.take(smf ? (size_t)bcap * l2 : 0);
  const size_t o_work = s.take(smf ? 2 * (size_t)bcap * l2 : 0), o_w = s.take(smf ? (size_t)bcap * wcols : 0);
  const size_t o_v = s.take((size_t)bcap * acols), o_y = s.take(acols);
  const size_t o_quad = s.take((size_t)npad * bcap), o_lin = s.take((size_t)npad * bcap);
  const size_t o_k = s.take(want_draws ? n2 : 0), o_f = s.take(want_draws ? npad : 0);
  const size_t o_ys = s.take(want_score ? n : 0), o_kb = s.take(want_score ? (size_t)gcap * k2 : 0);
  const size_t o_lps = s.take(want_score ? B : 0), o_white = s.take(want_score && white_out ? (size_t)n * B : 0);
  const size_t o_info = s.take(gcap + bcap, sizeof(int));
  const size_t o_pk = s.take((size_t)slots * gcap * TPP), o_pg = s.take((size_t)world * slots * gcap * TPP);
  CK(s.alloc());
  double *d_pk = s.at(o_pk), *d_pg = s.at(o_pg);
  double *d_ys = s.at(o_ys), *d_kb = s.at(o_kb), *d_lps = s.at(o_lps), *d_white = s.at(o_white);
  double *d_t = s.at(o_t), *d_A = s.at(o_a), *d_TA = s.at(o_ta), *d_mean = s.at(o_mean), *d_draw = s.at(o_draw);
  double *d_noise = s.at(o_noise), *d_cov = s.at(o_cov), *d_x = s.at(o_x), *d_g = s.at(o_g), *d_ac = s.at(o_ac);
  double *d_lag = s.at(o_lag), *d_AC = s.at(o_AC), *d_gf = s.at(o_gf), *d_qp = s.at(o_qp), *d_hs = s.at(o_hs);
  double *d_q1 = s.at(o_q1), *d_xm = s.at(o_xm), *d_mx = s.at(o_mx), *d_mxp = s.at(o_mxp), *d_hh = s.at(o_hh);
  double *d_c = s.at(o_c), *d_part = s.at(o_part), *d_c1 = s.at(o_c1), *d_work = s.at(o_work), *d_w = s.at(o_w);
  double *d_v = s.at(o_v), *d_y = s.at(o_y), *d_quad = s.at(o_quad), *d_lin = s.at(o_lin), *d_k = s.at(o_k);
  double* d_f = s.at(o_f);
  int* d_info = s.at<int>(o_info);
  int* d_pinfo = d_info + bcap;          // per sample of the group: the factorisation of C_b + reg I, or of K_b
  if (begin_run(h)) return -2;
  CK(cudaMemcpyAsync(h->params_d, params_host, np * sizeof(double), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_t, tstar_host, n * sizeof(double), cudaMemcpyHostToDevice, st));
  if (want_score) CK(cudaMemcpyAsync(d_ys, y_host, n * sizeof(double), cudaMemcpyHostToDevice, st));
  const double d_add = noise ? hp.s2 : reg;    // S_b = C_b + d_add I
  if (cov_out) CK(cudaMemsetAsync(d_cov, 0, (size_t)n2 * sizeof(double), st));
  if (world > 1) {                       // the per-sample outputs another rank owns stay 0 for the final all-reduce
    if (want_draws) CK(cudaMemsetAsync(d_draw, 0, (size_t)n * B * sizeof(double), st));
    if (want_score) CK(cudaMemsetAsync(d_lps, 0, (size_t)B * sizeof(double), st));
    if (want_score && white_out) CK(cudaMemsetAsync(d_white, 0, (size_t)n * B * sizeof(double), st));
  }
  std::vector<double> noise_t;
  if (want_draws) {
    // noise[p][b] -> one zero-padded column per sample
    noise_t.assign((size_t)B * npad, 0.0);
    for (int b = 0; b < B; ++b)
      for (int p = 0; p < n; ++p) noise_t[(size_t)b * npad + p] = noise_host[(size_t)p * B + b];
    CK(cudaMemcpyAsync(d_noise, noise_t.data(), noise_t.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  }
  if (prior_stage(h, c, reg, true)) return -2;
  if ((smf || !h->gram_valid) && plan_store(h, chunks, false)) return -2;
  if (predict_qu(h, reg)) return -2;
  if (int rc = shared_qz_stage(h, chunks, smf, r, c0, reg, d_xm, d_mx)) return rc;
  if (!smf) pad_mx(h, d_mx, 1, d_mxp);
  // ---- test side, once: A* and T = iKh A* for every test input
  {
    const int threads = std::min(256, round_up(nxp, 32));
    dim3 grid(nhp, (npad + AHX_NSUB - 1) / AHX_NSUB);
    ahx_gen_kernel<<<grid, threads, 0, st>>>(d_t, d_t, n, npad, h->th, nh, h->tx, nx, 0, nxp, d_A, nullptr, ld,
                                             (long)nhp * ld, cd);
    L(h);
  }
  if (gemm(h, true, false, false, nhp, (int)acols, nhp, 1.0, h->M(M_IKH), ld, d_A, acols, 0.0, d_TA, acols)) return -2;
  std::vector<int> inf(gcap);
  const double w = 1.0 / B;
  for (int g0 = 0; g0 < B; g0 += gcap) {
    const int gn = std::min(gcap, B - g0);
    const int nbat = (gn + bcap - 1) / bcap;
    // ---- training side of the group
    for (int bi = 0; bi < nbat; ++bi) {
      const int b0 = g0 + bi * bcap, nb = std::min(bcap, B - b0);
      double* hs = d_hs + (long)bi * bcap * nhp;
      if (smf) {
        if (int rc = smf_posterior_stage(h, chunks, samples_host, b0, nb, bcap, hs, d_part, d_c1, d_w, wcols, d_work,
                                         d_info, d_mx + (long)bi * bcap * l2, d_xm + (long)bi * bcap * ld,
                                         d_q1 + (long)bi * bcap, r, c0, reg, 0.0))
          return rc;
        pad_mx(h, d_mx + (long)bi * bcap * l2, nb, d_mxp + (long)bi * bcap * nxp * nxp);
      } else {
        if (stage_samples(h, samples_host + (size_t)b0 * nh, nb, bcap, hs)) return -2;
      }
    }
    // HH[b] = h_b h_b^T - iKh (rows past the group are zero)
    hh_build_kernel<<<148 * 4, 256, 0, st>>>(d_hs, nhp, gn, nbat * bcap, h->M(M_IKH), ld, nh, nhl, d_hh);
    L(h);
    // ---- per batch: V = H_B A*, the means, R_b = V_b mx_b V_b^T into C_b
    for (int bi = 0; bi < nbat; ++bi) {
      const int b0 = g0 + bi * bcap, nb = std::min(bcap, B - b0);
      const double* hs = d_hs + (long)bi * bcap * nhp;
      if (gemm(h, true, false, false, bcap, (int)acols, nhp, 1.0, hs, nhp, d_A, acols, 0.0, d_v, acols)) return -2;
      prof_close(h);
      PredQuadArgs qa;
      qa.V = d_v; qa.v_stride = acols; qa.ldv = nxp;
      qa.mx = smf ? d_mx + (long)bi * bcap * l2 : d_mx; qa.mx_stride = smf ? l2 : 0;
      qa.xm = smf ? d_xm + (long)bi * bcap * ld : d_xm; qa.xm_stride = smf ? ld : 0;
      qa.nv = n; qa.nx = nx; qa.nb = nb; qa.quad = d_quad; qa.lin = d_lin; qa.ldo = bcap;
      predict_quad_launch(st, qa, bcap);
      L(h);
      {
        const double* lin = d_lin;
        double* mean = d_mean + b0;
        const double sq = sqrt(s2f);
        const int nb_ = nb, Bn = B, bc = bcap;
        ew(st, (long)n * nb, [=] __device__(long idx) {
          const int p = (int)(idx / nb_), b = (int)(idx % nb_);
          mean[(long)p * Bn + b] = sq * lin[(long)p * bc + b];
        });
        L(h);
      }
      for (int b = 0; b < nb; ++b) {
        const double* Vb = d_v + (long)b * acols;
        const double* mxp = d_mxp + (smf ? (long)(bi * bcap + b) * nxp * nxp : 0);
        double* Cb = d_c + (long)(bi * bcap + b) * n2;
        if (gemm(h, true, false, false, npad, nxp, nxp, 1.0, Vb, nxp, mxp, nxp, 0.0, d_y, nxp)) return -2;
        if (gemm(h, true, true, false, npad, npad, nxp, 1.0, d_y, nxp, Vb, nxp, 0.0, Cb, npad)) return -2;
      }
    }
    // ---- pair tiles p >= q; tile k on rank k % world
    for (int pt = 0, k = 0; pt < ntile; ++pt)
      for (int qt = 0; qt <= pt; ++qt, ++k) {
        if (k % world != rank) continue;
        const int p0 = pt * TP, q0 = qt * TP;
        const int P = std::min(TP, n - p0), Q = std::min(TP, n - q0);
        const int npairs = P * Q, npp = round_up(npairs, 8);
        const long ldg = (long)TP * nxp;
        // G(i, k; j, l) = sum_m A*[m][(p0 + i, k)] T[m][(q0 + j, l)]
        if (gemm(h, false, false, false, P * nxp, Q * nxp, nhp, 1.0, d_A + (long)p0 * nxp, acols,
                 d_TA + (long)q0 * nxp, acols, 0.0, d_g, ldg)) return -2;
        prof_close(h);
        axx_pair_launch(st, d_t + p0, P, d_t + q0, Q, h->tx, nx, d_g, ldg, nxp, d_x, cd, T);
        L(h);
        {
          const double* tt = d_t;
          double* lag = d_lag;
          ew(st, npairs, [=] __device__(long e) { lag[e] = tt[p0 + e / Q] - tt[q0 + e % Q]; });
          L(h);
        }
        if (npp > npairs) CK(cudaMemsetAsync(d_AC + (long)npairs * KH, 0, (size_t)(npp - npairs) * KH * sizeof(double), st));
        ahh_center_kernel<<<148 * 8, 256, 0, st>>>(d_lag, npairs, h->th, nh, nhl, alpha, gamma, h->causal, d_AC, d_ac);
        L(h);
        if (!smf) {
          predict_qb_launch(st, d_x, (long)nx * nx, d_mx, l2, 1, npairs, TPP, 1, d_qp, bcap);     // one column
          L(h);
        }
        for (int bi = 0; bi < nbat; ++bi) {
          const int b0 = g0 + bi * bcap, nb = std::min(bcap, B - b0);
          // gf[e][b] = sum_(i,j) Ahh_c(lag_e)[i][j] HH_b[i][j]
          if (gemm(h, true, true, false, npp, bcap, (int)KH, 1.0, d_AC, KH, d_hh + (long)bi * bcap * KH, KH, 0.0, d_gf,
                   bcap)) return -2;
          prof_close(h);
          if (smf) {
            predict_qb_launch(st, d_x, (long)nx * nx, d_mx + (long)bi * bcap * l2, l2, nb, npairs, TPP, bcap, d_qp, bcap);
            L(h);
          }
          pcov_finish_kernel<<<(int)std::min<long>(((long)npairs * nb + 255) / 256, 148 * 16), 256, 0, st>>>(
              d_qp, TPP, bcap, smf ? 1 : 0, d_gf, bcap, d_ac, npairs, Q, p0, q0, nb, d_mean + b0, B, s2f,
              d_c + (long)bi * bcap * n2, n2, npad);
          L(h);
        }
      }
    CK(cudaGetLastError());
    if (world > 1) {
      pcov_pack_kernel<<<148 * 8, 256, 0, st>>>(d_c, n2, npad, gn, n, TP, ntp, rank, world, slots, d_pk);
      L(h);
      if (allgather(h, d_pk, d_pg, slots * gn * TPP)) return -2;
      pcov_unpack_kernel<<<148 * 8, 256, 0, st>>>(d_pg, world, slots, gn, n, TP, ntp, d_c, n2, npad);
      L(h);
    }
    // ---- cov += C_b / B in ascending b; the per-sample outputs
    if (cov_out) {
      const double* C = d_c;
      double* cv = d_cov;
      const int gn_ = gn;
      ew(st, n2, [=] __device__(long idx) {
        double s = cv[idx];
        for (int b = 0; b < gn_; ++b) s += w * C[(long)b * n2 + idx];
        cv[idx] = s;
      });
      L(h);
    }
    if (cov_s_out)
      for (int b = 0; b < gn; ++b)
        CK(cudaMemcpy2DAsync(cov_s_out + (size_t)(g0 + b) * n * n, (size_t)n * sizeof(double), d_c + (long)b * n2,
                              (size_t)npad * sizeof(double), (size_t)n * sizeof(double), n, cudaMemcpyDefault, st));
    if (want_draws) {
      CK(cudaMemsetAsync(d_pinfo, 0, (size_t)gn * sizeof(int), st));
      for (int b = 0; b < gn; ++b) {
        if (b % world != rank) continue;
        const double* Cb = d_c + (long)b * n2;
        double* Kp = d_k;
        const int nn = n, ldn = npad;
        ew(st, n2, [=] __device__(long idx) {
          const int rr = (int)(idx / ldn), qq = (int)(idx - (long)rr * ldn);
          double v = (rr == qq) ? 1.0 : 0.0;                  // identity on the padding block
          if (rr < nn && qq < nn) v = Cb[idx] + (rr == qq ? reg : 0.0);
          Kp[idx] = v;
        });
        L(h);
        cudaError_t e = potrf_lower(st, d_k, npad, npad, d_pinfo + b, 7, h->M(M_XW));
        L(h, 2 * ((npad + LA_NB - 1) / LA_NB));
        if (e != cudaSuccess) { h->err = "potrf launch failed"; return -2; }
        matvec_kernel<<<(npad + 7) / 8, 256, 0, st>>>(d_k, npad, npad, npad, 0, d_noise + (long)(g0 + b) * npad, 1.0, d_f);
        L(h);
        const double* fv = d_f;
        const double* mean = d_mean + g0 + b;
        double* dr = d_draw + g0 + b;
        const int Bn = B;
        ew(st, n, [=] __device__(long p) { dr[p * Bn] = mean[p * Bn] + fv[p]; });
        L(h);
      }
      if (allreduce(h, d_pinfo, gn, NCCL_INT32)) return -2;
      CK(cudaMemcpyAsync(inf.data(), d_pinfo, (size_t)gn * sizeof(int), cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      for (int b = 0; b < gn; ++b)
        if (inf[b]) return sample_pd_error(h, "C_b + reg I", g0 + b, inf[b] % 100000);
    }
    if (want_score) {
      CK(cudaMemsetAsync(d_pinfo, 0, (size_t)gn * sizeof(int), st));
      pcov_border_kernel<<<148 * 8, 256, 0, st>>>(d_c, npad, n2, d_mean + g0, B, d_ys, n, d_add, gn, d_kb, ldk, k2);
      L(h);
      for (int b = 0; b < gn; ++b) {
        if (b % world != rank) continue;
        cudaError_t e = potrf_lower(st, d_kb + (long)b * k2, ldk, ldk, d_pinfo + b, 8, h->M(M_XW));
        L(h, 2 * ((ldk + LA_NB - 1) / LA_NB));
        if (e != cudaSuccess) { h->err = "potrf launch failed"; return -2; }
      }
      pcov_score_kernel<<<gn, 256, 0, st>>>(d_kb, ldk, k2, n, d_lps + g0, white_out ? d_white + g0 : nullptr, B, rank,
                                            world);
      L(h);
      if (allreduce(h, d_pinfo, gn, NCCL_INT32)) return -2;
      CK(cudaMemcpyAsync(inf.data(), d_pinfo, (size_t)gn * sizeof(int), cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      for (int b = 0; b < gn; ++b) {
        if (!inf[b]) continue;
        int piv = inf[b] % 100000;
        if (piv == n + 1) {
          // The border pivot: potrf reports the first failed pivot, so every pivot of S_b passed and only the border
          // c - |z_b|^2 failed: |z_b|^2 overflows.  S_b is factorised alone with an identity border to confirm that
          // before the overflow message (a failure there would be named by its own pivot).  The owner of the sample
          // factorises; every rank receives its info word.
          CK(cudaMemsetAsync(d_pinfo + b, 0, sizeof(int), st));
          if (b % world == rank) {
            pcov_border_kernel<<<148 * 8, 256, 0, st>>>(d_c + (long)b * n2, npad, n2, d_mean + g0 + b, B, nullptr, n,
                                                        d_add, 1, d_kb + (long)b * k2, ldk, k2);
            L(h);
            cudaError_t e = potrf_lower(st, d_kb + (long)b * k2, ldk, ldk, d_pinfo + b, 8, h->M(M_XW));
            if (e != cudaSuccess) { h->err = "potrf launch failed"; return -2; }
          }
          if (allreduce(h, d_pinfo + b, 1, NCCL_INT32)) return -2;
          CK(cudaMemcpyAsync(&piv, d_pinfo + b, sizeof(int), cudaMemcpyDeviceToHost, st));
          CK(cudaStreamSynchronize(st));
          piv %= 100000;
          if (!piv) {           // S_b is positive definite and |z_b|^2 overflows
            char m[120];
            snprintf(m, sizeof m, "the whitened residual of sample %d overflows", g0 + b);
            h->err = m;
            return -3;
          }
        }
        return sample_pd_error(h, "C_b + d I", g0 + b, piv);
      }
    }
  }
  if (want_score && allreduce(h, d_lps, B)) return -2;
  if (want_score && white_out && allreduce(h, d_white, (long)n * B)) return -2;
  if (want_draws && allreduce(h, d_draw, (long)n * B)) return -2;
  if (want_score) {
    if (lp_s_out) CK(cudaMemcpyAsync(lp_s_out, d_lps, (size_t)B * sizeof(double), cudaMemcpyDefault, st));
    if (white_out) CK(cudaMemcpyAsync(white_out, d_white, (size_t)n * B * sizeof(double), cudaMemcpyDefault, st));
  }
  if (mean_s_out) CK(cudaMemcpyAsync(mean_s_out, d_mean, (size_t)n * B * sizeof(double), cudaMemcpyDefault, st));
  if (want_draws) CK(cudaMemcpyAsync(draws_out, d_draw, (size_t)n * B * sizeof(double), cudaMemcpyDefault, st));
  if (cov_out)
    CK(cudaMemcpy2DAsync(cov_out, (size_t)n * sizeof(double), d_cov, (size_t)npad * sizeof(double),
                         (size_t)n * sizeof(double), n, cudaMemcpyDefault, st));
  int info;          // the prior's and the shared q(z)'s, checked above
  if (end_run(h, info)) return -2;
  record_timing(h);
  return 0;
}

}  // namespace cgimpl

extern "C" {

int cgpcm_precompute(cgpcm_handle* h, const double hyp[3], double reg) {
  if (!h || !hyp) return -1;
  if (!h->t) { h->err = "cgpcm_set_data has not been called"; return -1; }
  for (int i = 0; i < 3; ++i)
    if (!std::isfinite(hyp[i]) || hyp[i] <= 0) { h->err = "hyper-parameters must be positive and finite"; return -4; }
  if (!std::isfinite(reg) || reg < 0) { h->err = "reg must be finite and >= 0"; return -4; }
  CK(cudaSetDevice(h->device));
  double p5[5] = {0.0, 0.0, log(hyp[0]), log(hyp[1]), log(hyp[2])};
  return evaluate(h, p5, CGPCM_MODE_FULL, 0, reg, true, nullptr, nullptr, nullptr);
}

int cgpcm_frozen_mats(cgpcm_handle* h, double* sum_Bxx, double* sum_Bhh, double* sum_b, double* sum_Ahx_y) {
  if (!h) return -1;
  if (!h->frozen) { h->err = "cgpcm_frozen_mats requires cgpcm_precompute"; return -1; }
  CK(cudaSetDevice(h->device));
  if (export_mat(h, h->M(M_F_AXX), h->nx, h->nx, sum_Bxx)) return -2;       // M_F_AXX holds sum_Axx + C1(-iKh) = sum_Bxx
  if (export_mat(h, h->M(M_F_BHH), h->nh, h->nh, sum_Bhh)) return -2;
  if (export_mat(h, h->M(M_F_Y), h->nh, h->nx, sum_Ahx_y)) return -2;
  CK(cudaStreamSynchronize(h->st));
  return put(h, sum_b, &h->f_sum_b, 1);
}

int cgpcm_elbo_smf(cgpcm_handle* h, const double* params, int32_t mode, double reg, const double* sample, double* elbo,
                   double* terms, double* loglik) {
  if (!h || !params || !sample || !elbo) return -1;
  if (mode != CGPCM_MODE_FROZEN && mode != CGPCM_MODE_FULL) { h->err = "bad mode"; return -1; }
  if (int rc = check_call(h, h->t, reg)) return rc;
  CK(cudaSetDevice(h->device));
  const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
  std::vector<double> host, smp;
  if (to_host(h, params, np, host) || to_host(h, sample, h->nh, smp)) return -2;
  if (check_samples(h, smp.data(), 1, h->nh)) return -4;
  double e = 0.0, tm[7], ll = 0.0;
  int rc = evaluate(h, host.data(), mode, 0u, reg, false, &e, tm, nullptr, smp.data(), &ll);
  if (rc) return rc;
  record_timing(h);
  if (put(h, elbo, &e, 1) || put(h, terms, tm, 7) || put(h, loglik, &ll, 1)) return -2;
  return 0;
}

int cgpcm_elbo_smf_batch(cgpcm_handle* h, const double* params, double reg, const double* samples, int32_t n_samples,
                         double* elbo, double* terms, double* loglik) {
  if (!h || !params || !samples) return -1;
  if (n_samples < 1) { h->err = "n_samples must be >= 1"; return -1; }
  if (int rc = check_call(h, h->t, reg)) return rc;
  CK(cudaSetDevice(h->device));
  const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
  std::vector<double> host, smp;
  if (to_host(h, params, np, host) || to_host(h, samples, (long)n_samples * h->nh, smp)) return -2;
  const bool want_p = elbo || terms;
  std::vector<double> e(want_p ? n_samples : 0), tm(want_p ? 7L * n_samples : 0), ll(loglik ? n_samples : 0);
  int rc = smf_batch_run(h, host.data(), reg, smp.data(), n_samples, want_p, loglik != nullptr,
                         want_p ? e.data() : nullptr, want_p ? tm.data() : nullptr, loglik ? ll.data() : nullptr);
  if (rc) return rc;
  if (put(h, elbo, e.data(), e.size()) || put(h, terms, tm.data(), tm.size()) || put(h, loglik, ll.data(), ll.size()))
    return -2;
  return 0;
}

int cgpcm_predict_f(cgpcm_handle* h, const double* params, double reg, const double* t_star, int64_t n_star,
                    const double* samples, int32_t n_samples, int32_t smf, double* mean, double* var) {
  if (!h || !params || n_star < 0 || n_samples < 1 || !samples || (n_star > 0 && !t_star)) return -1;
  if (int rc = check_call(h, h->t, reg)) return rc;
  if (n_star == 0) return 0;
  CK(cudaSetDevice(h->device));
  const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
  std::vector<double> host, ts, smp;
  if (to_host(h, params, np, host) || to_host(h, t_star, n_star, ts) || to_host(h, samples, (long)n_samples * h->nh, smp))
    return -2;
  return predict_run(h, host.data(), reg, ts.data(), n_star, smp.data(), n_samples, smf, mean, var);
}

int cgpcm_predict_f_batch(cgpcm_handle* h, const double* params, double reg, const double* t_star, int64_t n_star,
                          const double* samples, int32_t n_samples, int32_t smf, double* mean, double* var,
                          double* mean_s, double* var_s) {
  if (!h || !params || n_star < 0 || !samples || (n_star > 0 && !t_star)) return -1;
  if (n_samples < 1) { h->err = "n_samples must be >= 1"; return -1; }
  if (int rc = check_call(h, h->t, reg)) return rc;
  if (n_star == 0) return 0;
  CK(cudaSetDevice(h->device));
  const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
  std::vector<double> host, ts, smp;
  if (to_host(h, params, np, host) || to_host(h, t_star, n_star, ts) || to_host(h, samples, (long)n_samples * h->nh, smp))
    return -2;
  return predict_batch_run(h, host.data(), reg, ts.data(), n_star, smp.data(), n_samples, smf ? 1 : 0, mean, var,
                           mean_s, var_s);
}

int cgpcm_predict_f_cov(cgpcm_handle* h, const double* params, double reg, const double* t_star, int64_t n_star,
                        const double* samples, int32_t n_samples, int32_t smf, double* mean_s, double* cov_s,
                        double* cov, const double* noise, double* draws) {
  if (!h || !params || n_star < 0 || !samples || (n_star > 0 && !t_star)) return -1;
  if (n_samples < 1) { h->err = "n_samples must be >= 1"; return -1; }
  if (n_star > 4096) { h->err = "predict_f_cov: at most 4096 test inputs"; return -1; }
  if (draws && !noise) { h->err = "predict_f_cov: draws need noise"; return -1; }
  if (int rc = check_call(h, h->t, reg)) return rc;
  if (n_star == 0) return 0;
  CK(cudaSetDevice(h->device));
  const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
  std::vector<double> host, ts, smp, ns;
  if (to_host(h, params, np, host) || to_host(h, t_star, n_star, ts) || to_host(h, samples, (long)n_samples * h->nh, smp))
    return -2;
  if (draws && to_host(h, noise, (long)n_star * n_samples, ns)) return -2;
  return predict_cov_run(h, host.data(), reg, ts.data(), n_star, smp.data(), n_samples, smf ? 1 : 0,
                         draws ? ns.data() : nullptr, mean_s, cov_s, cov, draws, nullptr, 0, nullptr, nullptr);
}

int cgpcm_predict_logpdf(cgpcm_handle* h, const double* params, double reg, const double* t_star,
                         const double* y_star, int64_t n_star, const double* samples, int32_t n_samples, int32_t smf,
                         int32_t noise, double* lp, double* lp_s, double* white) {
  if (!h || !params || n_star < 0 || !samples || (n_star > 0 && (!t_star || !y_star))) return -1;
  if (n_samples < 1) { h->err = "n_samples must be >= 1"; return -1; }
  if (n_star > 4096) { h->err = "predict_logpdf: at most 4096 test inputs"; return -1; }
  if (noise != 0 && noise != 1) { h->err = "predict_logpdf: noise must be 0 or 1"; return -1; }
  if (int rc = check_call(h, h->t, reg)) return rc;
  if (!h->frozen) { h->err = "cgpcm_predict_logpdf requires cgpcm_precompute"; return -1; }
  CK(cudaSetDevice(h->device));
  std::vector<double> lps(n_samples, 0.0);
  if (n_star > 0) {
    const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
    std::vector<double> host, ts, ys, smp;
    if (to_host(h, params, np, host) || to_host(h, t_star, n_star, ts) || to_host(h, y_star, n_star, ys) ||
        to_host(h, samples, (long)n_samples * h->nh, smp))
      return -2;
    if (int rc = predict_cov_run(h, host.data(), reg, ts.data(), n_star, smp.data(), n_samples, smf ? 1 : 0, nullptr,
                                 nullptr, nullptr, nullptr, nullptr, ys.data(), noise, lps.data(), white))
      return rc;
  }
  // log (1 / B) sum_b exp(lp_s[b]), shifted by the largest term and added in ascending b
  double mx = lps[0];
  for (double v : lps) mx = std::max(mx, v);
  double acc = 0.0;
  for (double v : lps) acc += exp(v - mx);
  const double mix = mx + log(acc) - log((double)n_samples);
  if (put(h, lp, &mix, 1) || put(h, lp_s, lps.data(), n_samples)) return -2;
  return 0;
}

int cgpcm_kernel_samples(cgpcm_handle* h, const double* params, double reg, const double* t, int64_t n,
                         const double* samples, int32_t n_samples, double* out) {
  if (!h || !params || n < 0 || n_samples < 1 || !samples || !out || (n > 0 && !t)) return -1;
  if (int rc = check_call(h, h->th, reg)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(h->device));
  std::vector<double> host, ts, smp;
  if (to_host(h, params, 5, host) || to_host(h, t, n, ts) || to_host(h, samples, (long)n_samples * h->nh, smp)) return -2;
  return kernel_run(h, host.data(), reg, ts.data(), n, smp.data(), n_samples, out);
}

int cgpcm_filter_samples(cgpcm_handle* h, const double* params, double reg, const double* t, int64_t n,
                         const double* samples, int32_t n_samples, const double* noise, double* out) {
  if (!h || !params || n < 0 || n_samples < 1 || !samples || !noise || !out || (n > 0 && !t)) return -1;
  if (int rc = check_call(h, h->th, reg)) return rc;
  if (n == 0) return 0;
  CK(cudaSetDevice(h->device));
  std::vector<double> host, ts, smp, ns;
  if (to_host(h, params, 5, host) || to_host(h, t, n, ts) || to_host(h, samples, (long)n_samples * h->nh, smp) ||
      to_host(h, noise, n * n_samples, ns))
    return -2;
  return filter_run(h, host.data(), reg, ts.data(), n, smp.data(), n_samples, ns.data(), out);
}

int cgpcm_akm_sample(cgpcm_handle* h, const double* params, double reg, const double* t, int64_t n,
                     const double* sample_h, const double* e, double* f, double* K) {
  if (!h || !params || n < 1 || !t || !sample_h || !e || !f) return -1;
  if (int rc = check_call(h, h->th, reg)) return rc;
  CK(cudaSetDevice(h->device));
  std::vector<double> host, ts, hs, es;
  if (to_host(h, params, 5, host) || to_host(h, t, n, ts) || to_host(h, sample_h, h->nh, hs) || to_host(h, e, n, es))
    return -2;
  if (check_samples(h, hs.data(), 1, h->nh)) return -4;
  return akm_run(h, host.data(), reg, ts.data(), n, hs.data(), es.data(), f, K);
}

int cgpcm_fpi(cgpcm_handle* h, const double* params, int32_t num, int32_t high_reg, double reg, double* mu_u,
              double* var_u, double* mu_z, double* var_z) {
  if (!h || !params || num < 0) return -1;
  if (int rc = check_call(h, h->t, reg)) return rc;
  CK(cudaSetDevice(h->device));
  const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
  std::vector<double> host;
  if (to_host(h, params, np, host)) return -2;
  return fpi_run(h, host.data(), num, high_reg, reg, mu_u, var_u, mu_z, var_z);
}

int cgpcm_fpi_qz(cgpcm_handle* h, const double* params, const double* mu_z_in, const double* var_z_in, int32_t num,
                 int32_t high_reg, double reg, double* mu_u, double* var_u, double* mu_z, double* var_z) {
  if (!h || !params || !mu_z_in || !var_z_in || num < 0) return -1;
  if (int rc = check_call(h, h->t, reg)) return rc;
  CK(cudaSetDevice(h->device));
  const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
  std::vector<double> host, mz, vz;
  if (to_host(h, params, np, host) || to_host(h, mu_z_in, h->nx, mz) ||
      to_host(h, var_z_in, (long)h->nx * (h->nx + 1) / 2, vz))
    return -2;
  return fpi_run(h, host.data(), num, high_reg, reg, mu_u, var_u, mu_z, var_z, mz.data(), vz.data());
}

int cgpcm_elbo_qz(cgpcm_handle* h, const double* params, const double* mu_z, const double* var_z, double reg,
                  double* elbo, double* terms) {
  if (!h || !params || !mu_z || !var_z || !elbo) return -1;
  if (int rc = check_call(h, h->t, reg)) return rc;
  CK(cudaSetDevice(h->device));
  std::vector<double> host, mz, vz;
  if (to_host(h, params, 5, host) || to_host(h, mu_z, h->nx, mz) || to_host(h, var_z, (long)h->nx * (h->nx + 1) / 2, vz))
    return -2;
  double e = 0.0, tm[7];
  int rc = qz_run(h, host.data(), mz.data(), vz.data(), reg, &e, tm);
  if (rc) return rc;
  return put(h, elbo, &e, 1) || put(h, terms, tm, 7) ? -2 : 0;
}

int cgpcm_elbo_grad(cgpcm_handle* h, const double* params, int32_t mode, uint32_t grad_mask, double reg, double* elbo,
                    double* terms, double* grad) {
  if (!h || !params || !elbo) return -1;
  if (mode != CGPCM_MODE_FROZEN && mode != CGPCM_MODE_FULL) { h->err = "bad mode"; return -1; }
  if (int rc = check_call(h, h->t, reg)) return rc;
  CK(cudaSetDevice(h->device));
  const long np = 5 + h->nh + (long)h->nh * (h->nh + 1) / 2;
  std::vector<double> host;
  if (to_host(h, params, np, host)) return -2;
  double e = 0.0, tm[7];
  int rc = evaluate(h, host.data(), mode, grad ? grad_mask : 0u, reg, false, &e, tm, grad);
  if (rc) return rc;
  record_timing(h);
  float ms[5] = {0, 0, 0, 0, 0};
  cudaEventElapsedTime(&ms[1], h->ev[1], h->ev[3]);   // forward sweep (Axx + chunks + all-reduce)
  cudaEventElapsedTime(&ms[2], h->ev[4], h->ev[5]);   // backward sweep
  cudaEventElapsedTime(&ms[3], h->ev[3], h->ev[4]);   // M x M algebra between the sweeps
  cudaEventElapsedTime(&ms[4], h->ev[1], h->ev[2]);   // Axx kernels
  h->timing[1] = ms[1]; h->timing[2] = ms[2]; h->timing[3] = ms[3]; h->timing[4] = ms[4];
  h->timing[5] = ms[1] - ms[4] + ms[2];
  if (h->profile) {
    double tot = 0.0, tot_gen = 0.0;
    for (size_t i = 0; i + 1 < h->pev_used; i += 2) {
      float g = 0;
      cudaEventElapsedTime(&g, h->pev[i], h->pev[i + 1]);
      if (h->pev_kind[i / 2]) tot_gen += g; else tot += g;
    }
    h->timing[5] = tot;
    h->timing[10] = tot_gen;
  }
  {
    // this rank's own sweep time, without the waits inside the collectives: what a caller balances shards with
    float f = 0, b = 0;
    cudaEventElapsedTime(&f, h->ev[1], h->ev[7]);
    cudaEventElapsedTime(&b, h->ev[4], h->ev[8]);
    h->timing[11] = f + b;
  }
  return put(h, elbo, &e, 1) || put(h, terms, tm, 7) ? -2 : 0;
}

int cgpcm_last_timing(cgpcm_handle* h, double out[12]) {
  if (!h || !out) return -1;
  memcpy(out, h->timing, 12 * sizeof(double));
  return 0;
}

int cgpcm_bvn_cdf(const double* x1, const double* x2, const double* rho, double* out, size_t n, void* stream) {
  if (n == 0) return 0;
  if (!x1 || !x2 || !rho || !out) return -1;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) { cudaGetLastError(); return -2; }
  const bool dev = is_device_ptr(x1) && is_device_ptr(x2) && is_device_ptr(rho) && is_device_ptr(out);
  cudaStream_t st = (cudaStream_t)stream;
  size_t blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (dev) {
    bvn_cdf_kernel<<<(int)blocks, 256, 0, st>>>(x1, x2, rho, out, n);
    if (cudaGetLastError() != cudaSuccess) return -2;
    return cudaStreamSynchronize(st) == cudaSuccess ? 0 : -2;
  }
  double* d = nullptr;
  if (cudaMalloc(&d, 4 * n * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return -2; }
  int rc = 0;
  if (cudaMemcpyAsync(d, x1, n * sizeof(double), cudaMemcpyDefault, st) != cudaSuccess ||
      cudaMemcpyAsync(d + n, x2, n * sizeof(double), cudaMemcpyDefault, st) != cudaSuccess ||
      cudaMemcpyAsync(d + 2 * n, rho, n * sizeof(double), cudaMemcpyDefault, st) != cudaSuccess) rc = -2;
  if (!rc) {
    bvn_cdf_kernel<<<(int)blocks, 256, 0, st>>>(d, d + n, d + 2 * n, d + 3 * n, n);
    if (cudaGetLastError() != cudaSuccess) rc = -2;
  }
  if (!rc && cudaMemcpyAsync(out, d + 3 * n, n * sizeof(double), cudaMemcpyDefault, st) != cudaSuccess) rc = -2;
  if (cudaStreamSynchronize(st) != cudaSuccess) rc = -2;
  cudaFree(d);
  return rc;
}

int cgpcm_dgemm(int a_kc, int b_kc, int c_tr, int M, int N, int K, double alpha, const double* A, int64_t lda,
                const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int splits, int64_t c_split_stride,
                int lower_only, void* stream) {
  if (M < 0 || N < 0 || K < 0 || (M % 8) || (N % 8) || (K % 2) || (lda % 2) || (ldb % 2) || (ldc % 2)) return -1;
  if (!A || !B || !C) return -1;
  cudaError_t e;
  if (a_kc && (b_kc != 0) == (c_tr != 0) && splits <= 1 && !lower_only && beta == 0.0 && dgemm_sl_supported(M, N, K)) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 2) sms = 148;
    e = dgemm_sl((cudaStream_t)stream, b_kc != 0, M, N, K, alpha, A, lda, B, ldb, C, ldc, sms);
  } else {
    e = dgemm((cudaStream_t)stream, a_kc, b_kc, c_tr, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, splits,
              c_split_stride, lower_only);
  }
  if (e != cudaSuccess) return -2;
  return cudaStreamSynchronize((cudaStream_t)stream) == cudaSuccess ? 0 : -2;
}

int cgpcm_dgemm_tri(int M, int N, const double* S, int64_t lds, const double* B, int64_t ldb, double* C, int64_t ldc,
                    void* stream) {
  if (!S || !B || !C || (lds % 2) || (ldb % 2) || (ldc % 2)) return -1;
  if (!dgemm_sl_tri_supported(M, N)) return -1;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 2) sms = 148;
  if (dgemm_sl_tri((cudaStream_t)stream, M, N, S, lds, B, ldb, C, ldc, sms) != cudaSuccess) return -2;
  return cudaStreamSynchronize((cudaStream_t)stream) == cudaSuccess ? 0 : -2;
}

int cgpcm_dgemm_sym(int kc, int M, int K, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                    int64_t ldc, double* work, void* stream) {
  if (!A || !B || !C || K < 0 || (K % 2) || (lda % 2) || (ldb % 2) || ldc < M) return -1;
  if (!dgemm_sym_supported(M)) return -1;
  cudaStream_t st = (cudaStream_t)stream;
  const int splits = dgemm_sym_splits(K);
  double* acc = work;
  const long l2 = (long)M * M;
  if (!acc && cudaMalloc(&acc, (size_t)splits * l2 * sizeof(double)) != cudaSuccess) { cudaGetLastError(); return -2; }
  int rc = 0;
  if (dgemm_sym(st, kc != 0, M, K, A, lda, B, ldb, acc, M, l2, 0) != cudaSuccess) rc = -2;
  if (!rc) {
    reduce_partials_kernel<<<(int)((l2 + 255) / 256), 256, 0, st>>>(acc, l2, splits, C, M, M, M, ldc, 0.0, 1);
    if (cudaGetLastError() != cudaSuccess) rc = -2;
  }
  if (cudaStreamSynchronize(st) != cudaSuccess) rc = -2;
  if (!work) cudaFree(acc);
  return rc;
}

// cgmath.cuh under test: out_exp[i] = cg_exp_neg(min(x[i], 0)), out_erfc[i] = cg_erfc(x[i]), evaluated four at a time;
// *mismatch = number of elements whose one-at-a-time evaluation differs in any bit (must be 0).
__global__ void math_test_kernel(const double* __restrict__ x, long n, double* __restrict__ oe, double* __restrict__ oc,
                                 int* __restrict__ mismatch) {
  for (long i0 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i0 < n; i0 += (long)gridDim.x * blockDim.x * 4) {
    double xe[4], xc[4], e4[4], c4[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const double v = i0 + u < n ? x[i0 + u] : 0.0;
      xe[u] = fmin(v, 0.0);
      xc[u] = v;
    }
    cg_exp_neg<4>(xe, e4);
    cg_erfc<4>(xc, c4);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (i0 + u >= n) break;
      const double a1[1] = {xe[u]}, b1[1] = {xc[u]};
      double e1[1], c1[1];
      cg_exp_neg<1>(a1, e1);
      cg_erfc<1>(b1, c1);
      if (__double_as_longlong(e1[0]) != __double_as_longlong(e4[u]) ||
          __double_as_longlong(c1[0]) != __double_as_longlong(c4[u]))
        atomicAdd(mismatch, 1);
      oe[i0 + u] = e4[u];
      oc[i0 + u] = c4[u];
    }
  }
}

int cgpcm_math_test(const double* x, int64_t n, double* out_exp, double* out_erfc, int* mismatch_host) {
  if (!x || n < 1 || !out_exp || !out_erfc) return -1;
  double *dx = nullptr, *de = nullptr, *dc = nullptr;
  int* dm = nullptr;
  int rc = 0;
  if (cudaMalloc(&dx, n * sizeof(double)) != cudaSuccess || cudaMalloc(&de, n * sizeof(double)) != cudaSuccess ||
      cudaMalloc(&dc, n * sizeof(double)) != cudaSuccess || cudaMalloc(&dm, sizeof(int)) != cudaSuccess) rc = -2;
  if (!rc) {
    cudaMemcpy(dx, x, n * sizeof(double), cudaMemcpyDefault);
    cudaMemset(dm, 0, sizeof(int));
    math_test_kernel<<<148 * 4, 256>>>(dx, n, de, dc, dm);
    if (cudaDeviceSynchronize() != cudaSuccess) rc = -2;
    cudaMemcpy(out_exp, de, n * sizeof(double), cudaMemcpyDefault);
    cudaMemcpy(out_erfc, dc, n * sizeof(double), cudaMemcpyDefault);
    int m = 0;
    cudaMemcpy(&m, dm, sizeof(int), cudaMemcpyDeviceToHost);
    if (mismatch_host) *mismatch_host = m;
  }
  cudaGetLastError();
  if (dx) cudaFree(dx);
  if (de) cudaFree(de);
  if (dc) cudaFree(dc);
  if (dm) cudaFree(dm);
  return rc;
}

// out_exp[i] = cg_exp_neg<4, FLUSH>(min(x[i], 0)), out_erfcx[i] = cg_erfcx_abs<4>(x[i]) = erfcx(|x[i]|)
__global__ void math_test_fast_kernel(const double* __restrict__ x, long n, double* __restrict__ oe, double* __restrict__ oc) {
  for (long i0 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i0 < n; i0 += (long)gridDim.x * blockDim.x * 4) {
    double xe[4], xc[4], e4[4], c4[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const double v = i0 + u < n ? x[i0 + u] : 0.0;
      xe[u] = fmin(v, 0.0);
      xc[u] = v;
    }
    cg_exp_neg<4, true>(xe, e4);
    cg_erfcx_abs<4>(xc, c4);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (i0 + u >= n) break;
      oe[i0 + u] = e4[u];
      oc[i0 + u] = c4[u];
    }
  }
}

int cgpcm_math_test_fast(const double* x, int64_t n, double* out_exp, double* out_erfcx) {
  if (!x || n < 1 || !out_exp || !out_erfcx) return -1;
  double *dx = nullptr, *de = nullptr, *dc = nullptr;
  int rc = 0;
  if (cudaMalloc(&dx, n * sizeof(double)) != cudaSuccess || cudaMalloc(&de, n * sizeof(double)) != cudaSuccess ||
      cudaMalloc(&dc, n * sizeof(double)) != cudaSuccess) rc = -2;
  if (!rc) {
    cudaMemcpy(dx, x, n * sizeof(double), cudaMemcpyDefault);
    math_test_fast_kernel<<<148 * 4, 256>>>(dx, n, de, dc);
    if (cudaDeviceSynchronize() != cudaSuccess) rc = -2;
    cudaMemcpy(out_exp, de, n * sizeof(double), cudaMemcpyDefault);
    cudaMemcpy(out_erfcx, dc, n * sizeof(double), cudaMemcpyDefault);
  }
  cudaGetLastError();
  if (dx) cudaFree(dx);
  if (de) cudaFree(de);
  if (dc) cudaFree(dc);
  return rc;
}

// out_exp[i] = cg_exp_neg<4, true, AHX_BIAS>(min(x[i], 0)), out_erfcx[i] = cg_erfcx_tab<4>(x[i]) with x in groups of 4
// evaluated in lock-step as ahx_gen_sep_kernel<true> does (all kept)
__global__ void math_test_tab_kernel(const double* __restrict__ x, long n, double* __restrict__ oe, double* __restrict__ oc) {
  for (long i0 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * 4; i0 < n; i0 += (long)gridDim.x * blockDim.x * 4) {
    double xe[4], xc[4], e4[4], c4[4];
    bool keep[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      keep[u] = i0 + u < n;
      const double v = keep[u] ? x[i0 + u] : 0.0;
      xe[u] = fmin(v, 0.0);
      xc[u] = v;
    }
    cg_exp_neg<4, true, AHX_BIAS>(xe, e4);
    cg_erfcx_tab<4>(xc, keep, c4);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (i0 + u >= n) break;
      oe[i0 + u] = e4[u];
      oc[i0 + u] = c4[u];
    }
  }
}

int cgpcm_math_test_tab(const double* x, int64_t n, double* out_exp, double* out_erfcx, double* params) {
  if (!x || n < 1 || !out_exp || !out_erfcx || !params) return -1;
  params[0] = CG_ERFCX_TAB_ZLO;
  params[1] = CG_ERFCX_TAB_ZHI;
  params[2] = AHX_BIAS;
  double *dx = nullptr, *de = nullptr, *dc = nullptr;
  int rc = 0;
  if (cudaMalloc(&dx, n * sizeof(double)) != cudaSuccess || cudaMalloc(&de, n * sizeof(double)) != cudaSuccess ||
      cudaMalloc(&dc, n * sizeof(double)) != cudaSuccess) rc = -2;
  if (!rc) {
    cudaMemcpy(dx, x, n * sizeof(double), cudaMemcpyDefault);
    math_test_tab_kernel<<<148 * 4, 256>>>(dx, n, de, dc);
    if (cudaDeviceSynchronize() != cudaSuccess) rc = -2;
    cudaMemcpy(out_exp, de, n * sizeof(double), cudaMemcpyDefault);
    cudaMemcpy(out_erfcx, dc, n * sizeof(double), cudaMemcpyDefault);
  }
  cudaGetLastError();
  if (dx) cudaFree(dx);
  if (de) cudaFree(de);
  if (dc) cudaFree(dc);
  return rc;
}

int cgpcm_cholinv(double* A, double* Ainv, double* logdet, int n, int64_t ld, int* info_host) {
  if (!A || n < 1 || ld < n || (ld % 8)) return -1;
  int np = round_up(n, 8);
  if (np > ld) return -1;
  Scratch s;
  const size_t o_x = s.take(ld * ld), o_w = s.take(ld * ld), o_ld = s.take(1), o_info = s.take(1, sizeof(int));
  int rc = s.alloc() == cudaSuccess ? 0 : -2;
  double *X = s.at(o_x), *W = s.at(o_w), *ld_d = s.at(o_ld);
  int* info = s.at<int>(o_info);
  if (!rc) {
    cudaMemset(info, 0, sizeof(int));
    if (cholinv(nullptr, A, Ainv, X, W, n, np, ld, logdet ? ld_d : nullptr, info, 1) != cudaSuccess) rc = -2;
    if (cudaDeviceSynchronize() != cudaSuccess) rc = -2;
    int hi = 0;
    cudaMemcpy(&hi, info, sizeof(int), cudaMemcpyDeviceToHost);
    if (info_host) *info_host = hi % 100000;
    if (logdet) cudaMemcpy(logdet, ld_d, sizeof(double), cudaMemcpyDefault);
    if (!rc && hi) rc = -3;
  }
  return rc;
}

int cgpcm_smf_c1_test(const double* W, int64_t w_stride, int B, int nwin, const int64_t* windows, int nx, int64_t ld,
                      double* c1, void* stream) {
  if (!W || !windows || !c1 || B < 1 || nwin < 1 || nx < 1 || (ld % 8) || round_up(nx, 8) > ld) return -1;
  for (int w = 0; w < nwin; ++w) {
    const int64_t k_lo = windows[4 * w], kwp = windows[4 * w + 1], nc = windows[4 * w + 2], off = windows[4 * w + 3];
    if (kwp < 8 || kwp % 8 || nc < 8 || nc % 8 || k_lo < 0 || k_lo % 2 || k_lo + kwp > round_up(nx, 8) || off < 0 ||
        off + nc * kwp > w_stride)
      return -1;
  }
  cudaStream_t st = (cudaStream_t)stream;
  Scratch s;
  const size_t bytes = (size_t)B * SMF_SLICES * ld * ld * sizeof(double);
  s.take(bytes, 1);
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  double* part = s.at(0);
  int rc = cudaMemsetAsync(part, 0, bytes, st) == cudaSuccess ? 0 : -2;
  for (int w = 0; w < nwin && !rc; ++w) {
    const int64_t* win = windows + 4 * w;
    smf_c1_launch(st, W + win[3], w_stride, (int)win[1], (int)win[2], (int)win[0], part, ld, B);
    if (cudaGetLastError() != cudaSuccess) rc = -2;
  }
  if (!rc) {
    smf_reduce_launch(st, part, ld, nx, B, c1);
    if (cudaGetLastError() != cudaSuccess) rc = -2;
  }
  if (cudaStreamSynchronize(st) != cudaSuccess) rc = -2;
  return rc;
}

int cgpcm_smf_algebra_test(const double* kx, const double* sum_Bxx, const double* c1, const double* sum_Ahx_y,
                           const double* sum_Bhh, const double* samples, int B, int nx, int nh, int64_t ld, int ldh,
                           double r, double c0, double reg, int want_p, int want_p0, double* out, int* info,
                           void* stream) {
  if (!kx || !sum_Bxx || !c1 || !sum_Ahx_y || !sum_Bhh || !samples || !out || !info || B < 1 || nx < 1 || nh < 1 ||
      ld < nx || ld < nh || ldh < nh || (!want_p && !want_p0) || 2L * nx * sizeof(double) > 48 * 1024)
    return -1;
  cudaStream_t st = (cudaStream_t)stream;
  const int passes = (want_p ? 1 : 0) + (want_p0 ? 1 : 0);
  Scratch s;
  s.take((size_t)B * passes * ld * ld);
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  double* work = s.at(0);
  SmfAlgArgs a;
  a.kx = kx; a.sxx = sum_Bxx; a.c1 = c1; a.fy = sum_Ahx_y; a.bhh = sum_Bhh;
  a.hs = samples; a.work = work; a.out = out; a.info = info;
  a.ld = ld; a.l2 = ld * ld; a.ldh = ldh; a.nh = nh; a.nx = nx;
  a.r = r; a.c0 = c0; a.reg = reg; a.want_p = want_p != 0; a.passes = passes;
  int rc = cudaMemsetAsync(info, 0, 2 * (size_t)B * sizeof(int), st) == cudaSuccess ? 0 : -2;
  if (!rc) {
    smf_algebra_launch(st, a, B);
    if (cudaGetLastError() != cudaSuccess) rc = -2;
  }
  if (cudaStreamSynchronize(st) != cudaSuccess) rc = -2;
  return rc;
}

int cgpcm_smf_posterior_test(const double* kx, const double* sum_Bxx, const double* c1, const double* sum_Ahx_y,
                             const double* Ahh, const double* iKx, const double* tr_ahh_ikh, const double* samples,
                             int B, int nslots, int nx, int nh, int64_t ld, int ldh, double r, double c0, double reg,
                             double a, double* mx, double* xm, double* q1, int* info, void* stream) {
  if (!kx || !sum_Bxx || !c1 || !sum_Ahx_y || !Ahh || !iKx || !tr_ahh_ikh || !samples || !mx || !xm || !q1 || !info ||
      B < 1 || nslots < B || nx < 1 || nh < 1 || ld < nx || ld < nh || ldh < nh || 3L * nx * sizeof(double) > 48 * 1024)
    return -1;
  cudaStream_t st = (cudaStream_t)stream;
  const long l2 = ld * ld;
  Scratch s;
  s.take((size_t)B * 2 * l2);
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  double* work = s.at(0);
  SmfPostArgs g;
  g.kx = kx; g.sxx = sum_Bxx; g.c1 = c1; g.fy = sum_Ahx_y; g.ahh = Ahh; g.ikx = iKx; g.tr = tr_ahh_ikh; g.hs = samples;
  g.work = work; g.mx = mx; g.xm = xm; g.q1 = q1; g.info = info;
  g.ld = ld; g.l2 = l2; g.ldh = ldh; g.nh = nh; g.nx = nx; g.nb = B;
  g.r = r; g.c0 = c0; g.reg = reg; g.a = a;
  int rc = cudaMemsetAsync(info, 0, (size_t)B * sizeof(int), st) == cudaSuccess ? 0 : -2;
  if (!rc) {
    smf_posterior_launch(st, g, nslots);
    if (cudaGetLastError() != cudaSuccess) rc = -2;
  }
  if (cudaStreamSynchronize(st) != cudaSuccess) rc = -2;
  return rc;
}

int cgpcm_predict_quad_test(const double* V, int64_t v_stride, int ldv, const double* mx, int64_t mx_stride,
                            const double* xm, int64_t xm_stride, const double* bxx, int nv, int nx, int B, int nslots,
                            double* quad, double* lin, double* qb, void* stream) {
  if (!V || !mx || !xm || !quad || !lin || (qb && !bxx) || nv < 1 || nx < 1 || B < 1 || nslots < B || ldv < nx ||
      (B > 1 && v_stride < (int64_t)(nv - 1) * ldv + nx) || mx_stride < 0 || (mx_stride > 0 && mx_stride < (int64_t)nx * nx) ||
      xm_stride < 0 || (xm_stride > 0 && xm_stride < nx))
    return -1;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = 0;
  PredQuadArgs g;
  g.V = V; g.v_stride = v_stride; g.ldv = ldv; g.mx = mx; g.mx_stride = mx_stride; g.xm = xm; g.xm_stride = xm_stride;
  g.nv = nv; g.nx = nx; g.nb = B; g.quad = quad; g.lin = lin; g.ldo = B;
  predict_quad_launch(st, g, nslots);
  if (cudaGetLastError() != cudaSuccess) rc = -2;
  Scratch s;
  if (!rc && qb) {
    // Qb = the PQ_SLICES partials summed in order, as predict_finish_kernel sums them
    s.take((size_t)PQ_SLICES * nv * B);
    if (s.alloc() != cudaSuccess) { cudaGetLastError(); rc = -2; }
    double* part = s.at(0);
    if (!rc) {
      predict_qb_launch(st, bxx, (long)nx * nx, mx, mx_stride, B, nv, nv, nslots, part, B);
      if (cudaGetLastError() != cudaSuccess) rc = -2;
    }
    if (!rc) {
      const int zs = PQ_SLICES;
      ew(st, (long)nv * B, [=] __device__(long idx) {
        double s = 0.0;
        for (int z = 0; z < zs; ++z) s += part[(long)z * nv * B + idx];
        qb[idx] = s;
      });
      if (cudaGetLastError() != cudaSuccess) rc = -2;
    }
  }
  if (cudaStreamSynchronize(st) != cudaSuccess) rc = -2;
  return rc;
}

int cgpcm_predict_pair_test(const double* tp, int np_, const double* tq, int nq, const double* tx, int nx,
                            const double hyp[3], int causal, int causal_id, const double* G, int64_t ldg, int gk,
                            double* X, void* stream) {
  if (!tp || !tq || !tx || !hyp || !X || np_ < 1 || nq < 1 || nx < 1 || (G && (gk < nx || ldg < (int64_t)nq * gk)))
    return -1;
  for (int i = 0; i < 3; ++i)
    if (!std::isfinite(hyp[i]) || hyp[i] <= 0) return -4;
  cudaStream_t st = (cudaStream_t)stream;
  PsiConst c;
  psi_make_const(hyp[0], hyp[1], hyp[2], causal ? 1 : 0, 0.0, &c, causal_id);      // cull 0: dense (746)
  BvnTab T;
  bvn_make_tab(hyp[1] / (hyp[0] + hyp[1] + hyp[2]), &T);
  axx_pair_launch(st, tp, np_, tq, nq, tx, nx, G, (long)ldg, gk, X, c, T);
  int rc = cudaGetLastError() == cudaSuccess ? 0 : -2;
  if (cudaStreamSynchronize(st) != cudaSuccess) rc = -2;
  return rc;
}


}  // extern "C"

// ---- the sweeps' kernels under test (see the header) ----------------------------------------------------------------

namespace {

int psi_args(const double hyp[3], int causal, int causal_id, double cull, PsiConst* c) {
  for (int i = 0; i < 3; ++i)
    if (!std::isfinite(hyp[i]) || hyp[i] <= 0) return -4;
  if (!std::isfinite(cull) || cull < 0) return -1;
  psi_make_const(hyp[0], hyp[1], hyp[2], causal ? 1 : 0, cull, c, causal_id);
  return 0;
}

bool chunk_ok(int n_valid, int nc, int nh, int nhp, int nx, int k_lo, int kwp, int64_t ld, int causal, int causal_id,
              int sep) {
  return n_valid >= 0 && n_valid <= nc && nc >= 8 && nc % 8 == 0 && nh >= 1 && nhp >= nh && nhp % 8 == 0 && nx >= 1 &&
         kwp >= 8 && kwp % 8 == 0 && k_lo >= 0 && k_lo % 2 == 0 && ld % 8 == 0 && k_lo + kwp <= ld && nx <= ld &&
         nhp <= ld && (!sep || (causal && !causal_id));
}

int drain(cudaStream_t st, int rc) {
  if (cudaGetLastError() != cudaSuccess) rc = -2;
  if (cudaStreamSynchronize(st) != cudaSuccess) rc = -2;
  return rc;
}

}  // namespace

extern "C" {

int cgpcm_ahx_gen_test(const double* t, const double* y, int n_valid, int nc, const double* th, int nh, int nhp,
                       const double* tx, int nx, int k_lo, int kwp, const double hyp[3], int causal, int causal_id,
                       double cull, int sep, int64_t ld, double* A, double* ypart, void* stream) {
  if (!t || !y || !th || !tx || !hyp || !A || !chunk_ok(n_valid, nc, nh, nhp, nx, k_lo, kwp, ld, causal, causal_id, sep))
    return -1;
  PsiConst c;
  if (int rc = psi_args(hyp, causal, causal_id, cull, &c)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long ystride = (long)nhp * ld;
  int rc = 0;
  if (ypart && cudaMemsetAsync(ypart, 0, (size_t)((nc + AHX_NSUB - 1) / AHX_NSUB) * ystride * sizeof(double), st) !=
                   cudaSuccess)
    rc = -2;
  std::vector<double> th_host(nh);
  if (!rc && cudaMemcpy(th_host.data(), th, nh * sizeof(double), cudaMemcpyDefault) != cudaSuccess) rc = -2;
  if (!rc)
    ahx_gen_launch(st, sep != 0, sep != 0 && ahx_gen_tab(c, th_host.data(), nh), t, y, n_valid, nc, th, nh, nhp, tx,
                   nx, k_lo, kwp, A, ypart, ld, ystride, c);
  return drain(st, rc);
}

int cgpcm_ahx_dot_test(const double* t, const double* y, int n_valid, int nc, const double* th, int nh, int nhp,
                       const double* tx, int nx, int k_lo, int kwp, const double hyp[3], int causal, int causal_id,
                       double cull, int sep, int64_t ld, const double* A, const double* W, const double* Ybar,
                       double* g3, void* stream) {
  if (!t || !y || !th || !tx || !hyp || !A || !W || !Ybar || !g3 ||
      !chunk_ok(n_valid, nc, nh, nhp, nx, k_lo, kwp, ld, causal, causal_id, sep))
    return -1;
  PsiConst c;
  if (int rc = psi_args(hyp, causal, causal_id, cull, &c)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  // CTA partials as the backward sweep sizes them: nhp x slices entries of 3
  const long gneed = (long)nhp * ((nc + AHX_NSUB - 1) / AHX_NSUB);
  Scratch s;
  s.take(3 * gneed);
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  double* gpart = s.at(0);
  int rc = cudaMemsetAsync(gpart, 0, 3 * gneed * sizeof(double), st) == cudaSuccess ? 0 : -2;
  if (!rc) {
    ahx_dot_launch(st, sep != 0, t, y, n_valid, nc, th, nh, nhp, tx, nx, k_lo, kwp, A, W, Ybar, ld, gpart, c);
    sum3_kernel<<<1, 1024, 0, st>>>(gpart, gneed, g3);
  }
  return drain(st, rc);
}

int cgpcm_axx_sum_test(const double* t, int n, int sorted, const double* tx, int nx, const double hyp[3], int causal,
                       int causal_id, double cull, int slices, int tangents, int64_t ld, double* out4, void* stream) {
  if (!t || !tx || !hyp || !out4 || n < 1 || nx < 1 || ld < nx || slices < 1 || slices > AXX_MAX_SLICES) return -1;
  PsiConst c;
  if (int rc = psi_args(hyp, causal, causal_id, cull, &c)) return rc;
  BvnTab T;
  bvn_make_tab(hyp[1] / (hyp[0] + hyp[1] + hyp[2]), &T);
  cudaStream_t st = (cudaStream_t)stream;
  Scratch s;
  const size_t o_part = s.take((size_t)slices * 4 * ld * ld), o_cheb = s.take((BVN_CHEB_MAXDEG + 1) * 20);
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  int rc = axx_launch(st, t, n, sorted != 0, tx, nx, s.at(o_part), ld, slices, c, T, s.at(o_cheb), tangents != 0,
                      out4) == cudaSuccess ? 0 : -2;
  return drain(st, rc);
}

int cgpcm_window_chol_test(const double* M, int64_t ld, double sign, int nwin, const int32_t* windows, int tag,
                           double* out, int* info_host, void* stream) {
  if (!M || !windows || !out || !info_host || nwin < 1 || ld < 1 || tag < 0 || tag > 20000) return -1;
  std::vector<WinDesc> desc(nwin);
  long off = 0;
  int kw_max = 8;
  for (int w = 0; w < nwin; ++w) {
    const int k_lo = windows[3 * w], kw = windows[3 * w + 1], kv = windows[3 * w + 2];
    if (kw < 8 || kw > 120 || kw % 8 || kv < 0 || kv > kw || k_lo < 0 || k_lo + kv > ld) return -1;
    desc[w].k_lo = k_lo; desc[w].kw = kw; desc[w].kv = kv; desc[w].off = off;
    off += (long)kw * kw;
    kw_max = std::max(kw_max, kw);
  }
  cudaStream_t st = (cudaStream_t)stream;
  Scratch s;
  const size_t o_desc = s.take(nwin * sizeof(WinDesc), 1), o_info = s.take(1, sizeof(int));
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  int* info = s.at<int>(o_info);
  int rc = 0;
  if (cudaMemcpyAsync(s.at<WinDesc>(o_desc), desc.data(), nwin * sizeof(WinDesc), cudaMemcpyHostToDevice, st) !=
          cudaSuccess || cudaMemsetAsync(info, 0, sizeof(int), st) != cudaSuccess)
    rc = -2;
  if (!rc && window_chol(st, M, ld, sign, s.at<WinDesc>(o_desc), nwin, kw_max, out, info, tag) != cudaSuccess) rc = -2;
  if (!rc && cudaMemcpyAsync(info_host, info, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -2;
  return drain(st, rc);
}

int cgpcm_potrf_test(double* A, int np, int64_t ld, int tag, int* info_host, void* stream) {
  if (!A || !info_host || np < 8 || np % 8 || ld < np || ld % 2 || tag < 0 || tag > 20000) return -1;
  cudaStream_t st = (cudaStream_t)stream;
  Scratch s;
  const size_t o_scr = s.take(LA_NB * LA_NB), o_info = s.take(1, sizeof(int));
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  int* info = s.at<int>(o_info);
  int rc = cudaMemsetAsync(info, 0, sizeof(int), st) == cudaSuccess ? 0 : -2;
  if (!rc && potrf_lower(st, A, np, ld, info, tag, s.at(o_scr)) != cudaSuccess) rc = -2;
  if (!rc && cudaMemcpyAsync(info_host, info, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = -2;
  return drain(st, rc);
}

int cgpcm_trtri_test(const double* L, double* X, int np, int64_t ld, void* stream) {
  if (!L || !X || np < 8 || np % 8 || ld < np || ld % 2) return -1;
  cudaStream_t st = (cudaStream_t)stream;
  Scratch s;
  s.take((size_t)LA_NB * ld);
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  const int rc = trtri_lower(st, L, X, s.at(0), np, ld) == cudaSuccess ? 0 : -2;
  return drain(st, rc);
}

int cgpcm_sym_accum_test(int nwin, const int64_t* windows, const double* A, const double* B, int n, int64_t ld,
                         double* out, void* stream) {
  if (!windows || !A || !B || !out || nwin < 1 || n < 1 || ld < n || ld % 8) return -1;
  for (int w = 0; w < nwin; ++w) {
    const int64_t* v = windows + 6 * w;
    const int64_t k_lo = v[1], order = v[2], K = v[3];
    if (order < 8 || order % 8 || order > SY_MP || K < 2 || K % 2 || K > (1 << 30) || k_lo < 0 || k_lo + order > n ||
        v[4] < 0 || v[5] < 0 || v[4] % 2 || v[5] % 2)
      return -1;
  }
  cudaStream_t st = (cudaStream_t)stream;
  Scratch s;
  s.take((size_t)SY_MAX_SPLITS * ld * ld);
  if (s.alloc() != cudaSuccess) { cudaGetLastError(); return -2; }
  double* acc = s.at(0);
  int rc = cudaMemsetAsync(acc, 0, (size_t)SY_MAX_SPLITS * ld * ld * sizeof(double), st) == cudaSuccess ? 0 : -2;
  int used = 0;
  for (int w = 0; w < nwin && !rc; ++w) {
    const int64_t* v = windows + 6 * w;
    const bool kc = v[0] != 0;
    const int order = (int)v[2], K = (int)v[3];
    const long lda = kc ? K : order;
    int splits = 1;
    if (sym_accum_launch(st, kc, kc, order, K, A + v[4], lda, B + v[5], lda, acc, ld, v[1] * ld + v[1], &splits) !=
        cudaSuccess)
      rc = -2;
    used = std::max(used, splits);
  }
  if (!rc) sym_finish_launch(st, acc, ld, used, n, out);
  return drain(st, rc);
}

}  // extern "C"

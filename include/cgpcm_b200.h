/* cgpcm_b200 — C-ABI of the B200-native VCGPCM hot path (libcgpcm_b200.so).
 *
 * Drop-in boundary for ONE path of wesselb/cgpcm: evaluating the saturated VCGPCM evidence lower
 * bound and its gradient (SURVEY.md §8).  The reference is pure Python + TensorFlow; its only native
 * FFI on this path is the external custom op `bvn_cdf` (loaded at src/core/tf_util.py:9-13, called at
 * src/core/exponentiated_quadratic.py:552).  Everything else this header exposes replaces a
 * `sess.run(...)` of a TF sub-graph; each entry point cites the reference code it stands in for.
 *
 * Conventions
 *   - Plain C types only.  All floating point data is IEEE double.
 *   - Return value: 0 = success, -1 = bad argument, -2 = CUDA / NCCL error, -3 = a matrix was not
 *     positive definite (which one: cgpcm_last_error), -4 = non-finite input.  No exceptions.
 *   - Every pointer argument may be a CUDA device pointer or a host pointer unless stated otherwise
 *     (resolved with cudaPointerGetAttributes); host buffers are copied inside the call.
 *   - Calls are host-synchronous: they return after the handle's stream has drained.
 *   - A handle owns one device, one stream and all scratch memory; it is not thread-safe; different
 *     handles are independent (one per GPU / per restart).
 *   - There is no CPU fallback: without a CUDA device cgpcm_create fails with -2.
 *
 * Parameter vector (all unconstrained, exactly the reference's TF variables:
 * var_pos logs src/core/tf_util.py:323-332, mu_u / var_u src/core/cgpcm.py:435-445, packing of
 * var_u = np.tril_indices order src/core/tf_util.py:419-447):
 *     params = [log s2, log s2_f, log alpha, log gamma, log omega, mu_u[nh], var_u[nh(nh+1)/2]]
 * Gradients are with respect to this vector (so d/dlog theta for the five positives).
 */
#ifndef CGPCM_B200_H
#define CGPCM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cgpcm_handle cgpcm_handle;

/* grad_mask bits: which entries of the gradient are wanted (others are returned as 0). */
#define CGPCM_GRAD_S2     (1u << 0)
#define CGPCM_GRAD_S2F    (1u << 1)
#define CGPCM_GRAD_ALPHA  (1u << 2)
#define CGPCM_GRAD_GAMMA  (1u << 3)
#define CGPCM_GRAD_OMEGA  (1u << 4)
#define CGPCM_GRAD_MU_U   (1u << 5)
#define CGPCM_GRAD_VAR_U  (1u << 6)
#define CGPCM_GRAD_ALL    0x7fu

/* Evaluation regimes (src/core/cgpcm.py:270-292, src/core/experiment.py:217-250). */
#define CGPCM_MODE_FROZEN 0  /* "precomputed": Psi statistics frozen by cgpcm_precompute            */
#define CGPCM_MODE_FULL   1  /* Psi statistics rebuilt and differentiated every evaluation            */

/* Model construction: the state VCGPCM.__init__ builds (src/core/cgpcm.py:24-30,430-433).
 * nccl_comm: an existing ncclComm_t to reduce over, or NULL (single GPU, or use cgpcm_comm_init). */
int cgpcm_create(cgpcm_handle** out, int device, int nh, int nx, int causal, int causal_id, void* nccl_comm);
int cgpcm_destroy(cgpcm_handle* h);
const char* cgpcm_last_error(const cgpcm_handle* h);

/* Number of CUDA devices visible to the process: the multi-restart driver (cgpcm_b200/batch.py; the reference's unit
 * is one controller.py process per resample index, src/experiment_toy.sh:7-11) opens one handle per device.
 * Handles on different devices are independent and may be driven from different host threads. */
int cgpcm_device_count(int* out);

/* Multi-GPU: rank 0 makes a 128-byte NCCL unique id, every rank joins with it (one process per GPU).
 * After this, the sums over observations (src/core/cgpcm.py:240-267,473-475) are all-reduced. */
int cgpcm_comm_unique_id(void* id128);
int cgpcm_comm_init(cgpcm_handle* h, const void* id128, int rank, int world);

/* This rank's slice of the observations e.x, e.y (src/core/cgpcm.py:208-212) and the inducing inputs
 * th, tx (src/core/cgpcm.py:72-95). */
int cgpcm_set_data(cgpcm_handle* h, const double* t, const double* y, int64_t n_local, const double* th,
                   const double* tx);

/* Tuning knobs: "chunk" (workspace budget of a contraction chunk in observations x nx columns; 0 = default: the
 * planner picks 512 / 1024 / 2048 per evaluation by its cost model), "cull" (0 = dense; e > 0 = Psi entries whose
 * Gaussian envelope is below exp(-e) are exactly 0 and whole windows of them are skipped; default 80),
 * "profile" (1 = CUDA events around every run of consecutive GEMM launches so that cgpcm_last_timing reports their sum),
 * "store" (1 = default: keep the Ahx blocks and H*Ahx of the forward sweep resident in HBM for the backward sweep
 * when they fit -- 2 x 8 nh N nx bytes; 0 = always regenerate / recompute per chunk),
 * "sl" (1 = default: products with a small left operand run on the persistent bulk-copy kernel; 0 = tiled kernel),
 * "pw_dists" (0 = default: the prior kernels Kh, Kx use (x - y)^2; 1 = they use |x|^2 - 2xy + |y|^2 exactly as the
 * reference's pw_dists2 forms it, src/core/tf_util.py:24-31 -- for bit-level comparisons with the reference at inputs with a
 * large offset, where that expression loses ~eps x^2 gamma, e.g. 1e-7 relative at decimal-year time stamps),
 * "gram" (0 = default: off; 1: cgpcm_precompute also builds the fourth-order tensor G = sum_n Ahx_n (x) Ahx_n, 8 (nh nx)^2
 * bytes, when it fits and pays, and MODE_FROZEN evaluations / fpi / SMF / predict_f contract with it instead of
 * sweeping over the observations; 2 = whenever it fits.  Opt-in because it is noisier: the cancellation against
 * m2 ~ iKh then happens after the sum over observations, ~sqrt(N) more rounding noise than the sweeps),
 * "sep" (1 = default: the Ahx construction / adjoint kernels of the default causal model use the separable form
 * exp(E - z^2) = f_i g_nk, csrc/psi_kernels.cuh; 0 = the generic kernels, which causal_id = 1 and the acausal model
 * always use), "axx_slices" (0 = default 64; observation slices of the Axx kernel's grid, <= 64),
 * "tri" (1 = default: when every chunk has a window of <= 104 inducing inputs, Q = sum A iKx A^T and Hbar = sum A C1bar A^T
 * are contracted as V' V'^T with V' = A L and L L^T = iKx[window] / -C1bar[window] -- the triangular right-multiply needs
 * 54 % of the DMMAs; if a window block is not positive definite in FP64 the handle falls back to 0 = the products with
 * the full blocks, the reference's formulation, and repeats the evaluation). */
int cgpcm_set_option(cgpcm_handle* h, const char* key, double value);

/* Psi statistics at hyper-parameters hyp = {alpha, gamma, omega}: what `sess.run(mats[...])` returns
 * for 'sum_Axx' [nx*nx], 'Ahh' [nh*nh], 'a' [1], 'sum_Ahx_y' [nh*nx] and optionally 'Ahx'
 * [n_local*nh*nx] and 'Axx' [n_local*nx*nx] (src/core/cgpcm.py:235-243).  Any output may be NULL.
 * sum_* are summed over all ranks. */
int cgpcm_psi(cgpcm_handle* h, const double hyp[3], double* sum_Axx, double* Ahh, double* a, double* sum_Ahx_y,
              double* Ahx, double* Axx);

/* mod.precompute() (src/core/cgpcm.py:270-284): freeze the Psi statistics at hyp for MODE_FROZEN.
 * As in the reference, only `mats` (the sums over observations, evaluated at hyp) are frozen: the prior kernels Kh, Kx,
 * their factors and the prior of q(u) (src/core/cgpcm.py:214-229) stay functions of the CURRENT alpha, gamma, omega
 * of every later MODE_FROZEN call.  The value of such a call follows them, and its gradient entries for
 * CGPCM_GRAD_ALPHA / GAMMA / OMEGA are the derivatives through those kernels (what tf.gradients returns on the
 * precomputed graph) -- not zero, and consistent with the value. */
int cgpcm_precompute(cgpcm_handle* h, const double hyp[3], double reg);

/* The derived sums of `mats` that mod.precompute() freezes (src/core/cgpcm.py:255-267): 'sum_Bxx' [nx*nx], 'sum_Bhh'
 * [nh*nh], 'sum_b' [1] and 'sum_Ahx_y' [nh*nx], summed over all ranks, at the hyper-parameters of cgpcm_precompute.
 * Any output may be NULL. */
int cgpcm_frozen_mats(cgpcm_handle* h, double* sum_Bxx, double* sum_Bhh, double* sum_b, double* sum_Ahx_y);

/* One `sess.run([elbo, grad] + terms)` (src/core/cgpcm.py:518-575 through
 * src/core/learn.py:102-133): ELBO, its 7 terms and the gradient w.r.t. params.
 * reg = config.reg (src/config.py:3).  elbo[1], terms[7], grad[5 + nh + nh(nh+1)/2]; grad may be NULL. */
int cgpcm_elbo_grad(cgpcm_handle* h, const double* params, int32_t mode, uint32_t grad_mask, double reg,
                    double* elbo, double* terms, double* grad);

/* The stochastic SMF bound `mod.elbo(smf=True, sample=h)` (src/core/cgpcm.py:527-531, used by elbo_smf :594-608): the
 * optimal q(z) is built from (h, h h^T) instead of the moments of q(u).  sample[nh]; value only (elbo[1], terms[7]).
 * loglik (may be NULL) receives the pseudo-log-likelihood of h that VCGPCM.sample() gives to the elliptical slice
 * sampler (src/core/cgpcm.py:848-872; Cholesky of P without jitter, as there). */
int cgpcm_elbo_smf(cgpcm_handle* h, const double* params, int32_t mode, double reg, const double* sample, double* elbo,
                   double* terms, double* loglik);

/* cgpcm_elbo_smf in MODE_FROZEN for many filter samples in one call (src/core/cgpcm.py:527-531,594-608,848-872):
 * samples[n_samples][nh] -> elbo[n_samples], terms[n_samples][7], loglik[n_samples].  The optimal q(z) of every sample
 * comes from C1_b = sum_n w_bn w_bn^T with w_bn = A_n^T h_b (H = h_b h_b^T has rank one), contracted for a batch of
 * samples at a time over the frozen regime's Ahx blocks.  elbo and terms may both be NULL (then P_b, the jittered
 * matrix, is not factorised), loglik may be NULL; any n_samples >= 1 (split internally into batches).  A sample's
 * results are bitwise the same whatever batch it is scored in and at whatever position; they agree with
 * cgpcm_elbo_smf(MODE_FROZEN) up to the rounding of the other summation order.  Requires cgpcm_precompute (-1
 * otherwise); -4 for a non-finite parameter or sample; -3 when P_b or P0_b is not positive definite
 * (cgpcm_last_error names the sample). */
int cgpcm_elbo_smf_batch(cgpcm_handle* h, const double* params, double reg, const double* samples, int32_t n_samples,
                         double* elbo, double* terms, double* loglik);

/* mod.predict_f(t, samples_h) (src/core/cgpcm.py:781-846): posterior mean[n_star] and variance[n_star] of the function
 * at the test inputs t_star, averaged over the filter samples samples[n_samples][nh].  smf = 0: the optimal q(z) of
 * q(u) (the reference's numeric samples_h: draws from q(u)); smf = 1: the optimal q(z | h) of every sample (the
 * reference's list samples_h, e.g. from mod.sample()).  Uses the Psi statistics frozen by cgpcm_precompute. */
int cgpcm_predict_f(cgpcm_handle* h, const double* params, double reg, const double* t_star, int64_t n_star,
                    const double* samples, int32_t n_samples, int32_t smf, double* mean, double* var);

/* predict_f's moments per filter sample: for every test input n and sample b, the predictive mean and variance of the
 * function under that sample's q(z) (smf = 1: q(z | h_b); smf = 0: the one q(z) of q(u)):
 * mean_s[n * n_samples + b], var_s[n * n_samples + b] (the layout of cgpcm_kernel_samples), and their averages over
 * the samples mean[n_star], var[n_star] -- what cgpcm_predict_f returns for the same arguments, added per sample in
 * ascending b with weight 1 / n_samples.  The law of total variance gives the mixture variance of the samples as
 * mean_b(var_s) + var_b(mean_s).  Any output may be NULL; host or device pointers.  The samples are processed in
 * internal batches whose size depends on the handle's shape only, and no sum runs across samples except the average:
 * a sample's mean_s / var_s are bitwise the same whatever other samples share the call and in any position.  Uses the
 * statistics frozen by cgpcm_precompute (-1 otherwise); -1 when n_samples < 1; -4 for a non-finite parameter, sample or
 * test input; -3 when some P_b is not positive definite (cgpcm_last_error names the sample and the pivot); n_star = 0
 * returns 0 and writes nothing. */
int cgpcm_predict_f_batch(cgpcm_handle* h, const double* params, double reg, const double* t_star, int64_t n_star,
                          const double* samples, int32_t n_samples, int32_t smf, double* mean, double* var,
                          double* mean_s, double* var_s);

/* The joint predictive covariance of the function at n_star <= 4096 test inputs, per filter sample, and posterior
 * draws of f.  For sample b, under the q(z) of cgpcm_predict_f_batch (smf = 1: q(z | h_b); smf = 0: the one q(z) of
 * q(u)):
 *   mean_s[p * n_samples + b]       the predictive mean, as cgpcm_predict_f_batch;
 *   cov_s[(b * n_star + p) * n_star + q] = C_b[p][q] = E[f_p f_q | h_b] - mean_s[p][b] mean_s[q][b], full and exactly
 *                                   symmetric; diag(C_b) is cgpcm_predict_f_batch's var_s[:, b];
 *   cov[p * n_star + q]             (1 / n_samples) sum_b C_b, added in ascending b; its diagonal is cgpcm_predict_f's
 *                                   var.  By the law of total covariance the covariance of the mixture of the samples'
 *                                   predictive distributions is cov + Cov_b(mean_s);
 *   draws[p * n_samples + b]        mean_s[:, b] + chol(C_b + reg I) noise[:, b] for the caller's standard normal
 *                                   noise[p * n_samples + b] (so that draws follow the host generator).
 * With E[f_p f_q | h] = s2_f (a_c(t_p - t_q) + <Ahh_c(t_p - t_q), h h^T - iKh> + <Axx(t_p, t_q), mx>
 *                             + <(h h^T - iKh) Ahx_q mx, Ahx_p>),  mx = x_m2 - iKx,
 * a_c / Ahh_c the centre statistics of cgpcm_kernel_samples at the lag and Axx(t_p, t_q) the Axx statistic with the two
 * inputs on its two factors.  Every output may be NULL (draws then needs no noise; draws without noise is -1); host or
 * device pointers.  C_b + reg I is only factorised when draws is requested.  Internal batch sizes depend on the
 * handle's shape and n_star only and no sum runs across samples except cov: a sample's mean_s, C_b and draw are bitwise
 * the same in any batch and at any position.  Uses the statistics frozen by cgpcm_precompute (-1 otherwise); -1 when
 * n_samples < 1 or n_star > 4096; -4 for a non-finite parameter, sample, test input or noise; -3 when some P_b or some
 * C_b + reg I is not positive definite (cgpcm_last_error names the sample and the pivot); n_star = 0 returns 0 and
 * writes nothing. */
int cgpcm_predict_f_cov(cgpcm_handle* h, const double* params, double reg, const double* t_star, int64_t n_star,
                        const double* samples, int32_t n_samples, int32_t smf, double* mean_s, double* cov_s,
                        double* cov, const double* noise, double* draws);

/* Held-out scoring: the log predictive density of a block y_star[n_star] at the test inputs t_star, n_star <= 4096,
 * per filter sample and for the mixture of the samples.  For sample b, with m_b and C_b the mean and covariance of f of
 * cgpcm_predict_f_cov (smf as there) and S_b = C_b + d I, d = s2 = exp(params[0]) when noise = 1 (y_star are
 * observations) and d = reg when noise = 0 (y_star is f itself):
 *   lp_s[b]                      log N(y_star; m_b, S_b) = -(n log 2 pi + log det S_b + |z_b|^2) / 2,
 *                                z_b = L_b^-1 (y_star - m_b), L_b L_b^T = S_b;
 *   lp[0]                        log ((1 / n_samples) sum_b exp(lp_s[b])), a log-sum-exp shifted by the largest lp_s
 *                                and added in ascending b (finite however negative the lp_s are);
 *   white[p * n_samples + b]     z_b[p], the whitened residuals (standard normal when y_star is drawn from the
 *                                sample's predictive distribution).
 * One Cholesky factorisation per sample of the bordered matrix [[S_b, y - m_b], [(y - m_b)^T, c]] gives log det S_b and
 * z_b together.  Every output may be NULL; host or device pointers.  Internal batch sizes depend on the handle's shape
 * and n_star only and no sum runs across samples except lp: a sample's lp_s and whitened residuals are bitwise the same
 * in any batch and at any position.  Uses the statistics frozen by cgpcm_precompute (-1 otherwise); -1 when n_samples
 * < 1, n_star > 4096 or noise is not 0 or 1; -4 for a non-finite parameter, sample, test input or y_star; -3 when some
 * P_b or some C_b + d I is not positive definite (cgpcm_last_error names the sample and the pivot); n_star = 0 writes
 * lp = 0 and lp_s = 0 (the empty block has density 1). */
int cgpcm_predict_logpdf(cgpcm_handle* h, const double* params, double reg, const double* t_star,
                         const double* y_star, int64_t n_star, const double* samples, int32_t n_samples, int32_t smf,
                         int32_t noise, double* lp, double* lp_s, double* white);

/* The Monte-Carlo kernel samples of mod.predict_k(t, samples_h) (src/core/cgpcm.py:610-634; centre statistics
 * _a_center / _Ahh_center :164-166,190-192), before normalisation / FFT / percentiles (host post-processing):
 * out[p * n_samples + b] = s2_f (a_c(t_p) + tr((h_b h_b^T - iKh) Ahh_c(t_p))) for lags t[n] and filter samples
 * samples[n_samples][nh].  Needs only the inducing inputs (cgpcm_set_data) and the hyper-parameters in params[0..4]. */
int cgpcm_kernel_samples(cgpcm_handle* h, const double* params, double reg, const double* t, int64_t n,
                         const double* samples, int32_t n_samples, double* out);

/* The posterior draws of the filter that mod.predict_h / mod.predict_psd post-process (src/core/cgpcm.py:663-779):
 * out[p * n_samples + b] = (Kuh^T h_b + L eps_b)[p] at inputs t[n] with Kuh = k_h(th, t), A = Lh^-1 Kuh,
 * L = chol(reg(k_h(t, t) - A^T A)); samples[n_samples][nh] are the filter samples h_b, noise[n][n_samples] the
 * standard normal draws eps (the reference draws them inside the graph).  n <= 8192. */
int cgpcm_filter_samples(cgpcm_handle* h, const double* params, double reg, const double* t, int64_t n,
                         const double* samples, int32_t n_samples, const double* noise, double* out);

/* One draw of the Approximate Kernel Model, AKM.f() (src/core/cgpcm.py:295-422, f: 382-392; the sampler behind
 * data.load_akm, src/core/data.py:594-641, i.e. the toy experiment's series): f = sqrt(s2_f) chol(reg(K)) e at inputs
 * t[n] with K[p][q] = a(t_p, t_q) + tr((h h^T - iKh) Ahh(t_p, t_q)) (pair statistics _a / _Ahh, cgpcm.py:156-158,
 * 182-184), for the filter draw sample_h[nh] and the standard normal draw e[n] (the reference draws both inside the
 * graph).  f[n] and the optional K[n][n] (before the Cholesky, reg included) may be host or device.  n <= 4096. */
int cgpcm_akm_sample(cgpcm_handle* h, const double* params, double reg, const double* t, int64_t n,
                     const double* sample_h, const double* e, double* f, double* K);

/* mod.fpi(num, z=True, high_reg) followed by mod.convert(z=True) (src/core/cgpcm.py:479-516,577-592): num rounds of
 * the fixed-point iteration q(u) -> optimal q(z) -> optimal q(u) on the Psi statistics frozen by cgpcm_precompute
 * (Normal.from_natural, src/core/distribution.py:20-33; high_reg adds 1e-4 to both precisions), starting from the
 * q(u) in params.  Outputs (each may be NULL; host or device): mu_u[nh], var_u[nh(nh+1)/2] = tril_to_vec(chol(cov))
 * as the reference assigns them, and the optimal q(z) of the final q(u): mu_z[nx], var_z[nx(nx+1)/2].
 * num = 0 is convert(z=True) alone. */
int cgpcm_fpi(cgpcm_handle* h, const double* params, int32_t num, int32_t high_reg, double reg, double* mu_u,
              double* var_u, double* mu_z, double* var_z);

/* Timing of the last cgpcm_elbo_grad / cgpcm_psi on the handle's stream (CUDA events, ms):
 * out[0] total device time, out[1] forward sweep, out[2] backward sweep, out[3] M x M algebra,
 * out[4] Axx kernel, out[5] contraction GEMM kernels (exact sum with option "profile", else the sweeps
 * minus the Axx kernel), out[6] number of kernel launches, out[7] algorithmic FP64 flops of those GEMM
 * launches (2 K M N; symmetric results K M (M + 1)), out[8] number of GEMM launches, out[9] flops of the CTA /
 * warp tiles the launches actually computed, out[10] Ahx generation kernels (option "profile" only);
 * out[11] reserved. */
/* The z = False variants (src/core/cgpcm.py:472-476,499,537-540,584-592): q(z) = N(mu_z, reg(Lz Lz^T)) is the explicit
 * variational distribution (mu_z[nx], var_z[nx(nx+1)/2] = Lz in np.tril_indices order) and q(u) is the optimal one.
 * Both use the Psi statistics frozen by cgpcm_precompute; params supplies s2, s2_f and the hyper-parameters of the prior
 * kernels (its q(u) part is not read).
 *   cgpcm_fpi_qz   mod.fpi(num, z=False, high_reg) followed by mod.convert(z=False): num rounds of
 *                  q(z) -> optimal q(u) -> optimal q(z), then the optimal q(u) of the final q(z).  Outputs as cgpcm_fpi.
 *   cgpcm_elbo_qz  mod.elbo(z=False): the bound saturated for q(u); value and the 7 terms ('p(u) complexity',
 *                  'q*(u) complexity', 'q*(u) fit', ..., -KL[q(z)||p(z)]).  No gradient: no task of the reference
 *                  optimises q(z) directly (src/core/experiment.py:209-250 trains q(u) with z = True throughout). */
int cgpcm_fpi_qz(cgpcm_handle* h, const double* params, const double* mu_z_in, const double* var_z_in, int32_t num,
                 int32_t high_reg, double reg, double* mu_u, double* var_u, double* mu_z, double* var_z);
int cgpcm_elbo_qz(cgpcm_handle* h, const double* params, const double* mu_z, const double* var_z, double reg,
                  double* elbo, double* terms);

/* Device times (ms) and counters of the last cgpcm_elbo_grad: [0] whole call, [1] forward sweep (incl. all-reduce #1),
 * [2] backward sweep (incl. #2), [3] M x M algebra between them, [4] Axx kernel, [5] GEMM launches (option "profile"),
 * [6] kernel launches, [7] algorithmic / [9] executed GEMM flops, [8] GEMM launches, [10] Ahx generation ("profile"),
 * [11] this rank's own sweep time WITHOUT the waits inside the collectives (what a caller balances shards with:
 * cgpcm_b200.rebalance_costs). */
int cgpcm_last_timing(cgpcm_handle* h, double out[12]);

/* The reference's native op: Phi_2(x1, x2; rho) element-wise on three FP64 vectors of length n
 * (src/core/exponentiated_quadratic.py:547-552).  stream: a cudaStream_t or NULL. */
int cgpcm_bvn_cdf(const double* x1, const double* x2, const double* rho, double* out, size_t n, void* stream);

/* Building blocks exported for tests and micro-benchmarks (device pointers only).
 * cgpcm_dgemm: C = alpha op(A) op(B) + beta C on the DMMA kernels; a_kc/b_kc/c_tr as in dgemm_dmma.cuh
 * (shapes with a small k-contiguous left operand, 16 <= M <= 208, 16 <= K <= 200, N >= 9472, go to dgemm_sl.cuh).
 * cgpcm_cholinv: A (n x n, ld) -> L in place, Ainv, logdet (each may be NULL). */
int cgpcm_dgemm(int a_kc, int b_kc, int c_tr, int M, int N, int K, double alpha, const double* A, int64_t lda,
                const double* B, int64_t ldb, double beta, double* C, int64_t ldc, int splits,
                int64_t c_split_stride, int lower_only, void* stream);
/* cgpcm_dgemm_sym: the symmetric-output split-K contraction of dgemm_sym.cuh, C = op(A) op(B)^T (M x M, full
 * symmetric matrix written; 8 <= M <= 200, M % 8 == 0).  kc = 1: A[m*lda + k], B[n*ldb + k]; kc = 0: A[k*lda + m],
 * B[k*ldb + n].  The result is only meaningful when the product is symmetric (the lower triangle is mirrored).
 * work: NULL or a device buffer of 148 * M * M doubles for the K-slice partial results. */
int cgpcm_dgemm_sym(int kc, int M, int K, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                    int64_t ldc, double* work, void* stream);
/* cgpcm_dgemm_tri: C[n*ldc + m] = sum_{k >= m} S[m*lds + k] B[n*ldb + k] for an upper-triangular M x M operand S
 * (16 <= M <= 104, M % 8 == 0, N >= 9472): the right-multiply by the transposed Cholesky factor of a window block;
 * DMMA blocks below the diagonal are not issued. */
int cgpcm_dgemm_tri(int M, int N, const double* S, int64_t lds, const double* B, int64_t ldb, double* C, int64_t ldc,
                    void* stream);
int cgpcm_cholinv(double* A, double* Ainv, double* logdet, int n, int64_t ld, int* info_host);
/* cgpcm_math_test: the in-register exp / erfc of the Psi kernels (csrc/cgmath.cuh) on n arguments (host or device):
 * out_exp[i] = exp(min(x[i], 0)), out_erfc[i] = erfc(x[i]), evaluated four at a time; *mismatch = elements whose
 * one-at-a-time evaluation differs in any bit (0 when the lock-step evaluation is faithful). */
int cgpcm_math_test(const double* x, int64_t n, double* out_exp, double* out_erfc, int* mismatch_host);
/* cgpcm_math_test_fast: the variants the separable Psi kernels use: out_exp[i] = exp(min(x[i], 0)) with results below
 * 2^-1021 flushed to 0 (one integer add scales by 2^n), out_erfcx[i] = erfcx(|x[i]|) = exp(x^2) erfc(|x|). */
int cgpcm_math_test_fast(const double* x, int64_t n, double* out_exp, double* out_erfcx);
/* cgpcm_math_test_tab: the routines of the table-driven separable Ahx kernel: out_exp[i] = exp(min(x[i], 0)) 2^B
 * (results below 2^-1021 flushed to 0) and out_erfcx[i] = erfcx(x[i]) from the piecewise table, x in groups of 4
 * evaluated in lock-step (4 neighbours share one interval's coefficients when they fit on it).  params receives
 * {table range low, table range high, B}; erfcx outside the range is not meaningful. */
int cgpcm_math_test_tab(const double* x, int64_t n, double* out_exp, double* out_erfcx, double* params);
/* The kernels of cgpcm_elbo_smf_batch (csrc/smf_batch.cuh) with the launch shapes that call uses.  Device pointers only,
 * except `windows`; stream: a cudaStream_t or NULL; both return after the stream has drained.
 * cgpcm_smf_c1_test: c1[b] (B slabs of ld x ld) = sum over the windows of W_w,b^T W_w,b placed at (k_lo, k_lo), lower
 * triangle of the leading nx x nx block, 0 elsewhere.  windows: host int64 [nwin][4] = (k_lo, kwp, nc, w_offset);
 * window w reads W_w,b(n, k) = W[w_offset + b * w_stride + n * kwp + k] for n < nc, k < kwp.  The windows are added into
 * zeroed per-slice partials in list order, then the slices are summed.  -1 unless kwp and nc are positive multiples of 8,
 * k_lo is even, k_lo + kwp <= round_up(nx, 8) <= ld, ld % 8 == 0 and w_offset + nc * kwp <= w_stride.
 * cgpcm_smf_algebra_test: per sample b (samples[b * ldh + i], i < nh), with S_b = sum_Bxx + C1_b (lower triangles of
 * the nx x nx blocks at leading dimension ld are read) and lam_b = c0 sum_Ahx_y^T h_b (sum_Ahx_y: nh x nx at ld):
 * out[b][0..1] = log det P_b, |L^-1 lam_b|^2 of P_b = Kx + r S_b + reg I (want_p), out[b][2..3] the same for
 * P0_b = Kx + r S_b and out[b][4] = h_b^T sum_Bhh h_b (want_p0); entries of a pass not run are not written.
 * info[b][0 / 1] (int, device) = pivot + 1 of a failed factorisation of P_b / P0_b, else 0.  nx <= 3072. */
int cgpcm_smf_c1_test(const double* W, int64_t w_stride, int B, int nwin, const int64_t* windows, int nx, int64_t ld,
                      double* c1, void* stream);
int cgpcm_smf_algebra_test(const double* kx, const double* sum_Bxx, const double* c1, const double* sum_Ahx_y,
                           const double* sum_Bhh, const double* samples, int B, int nx, int nh, int64_t ld, int ldh,
                           double r, double c0, double reg, int want_p, int want_p0, double* out, int* info,
                           void* stream);
/* The kernels of cgpcm_predict_f_batch (csrc/smf_batch.cuh, csrc/predict_kernels.cuh) with its launch shapes; device
 * pointers only; they return after the stream has drained.  nslots >= B: the sample slots the grid is shaped for (the
 * internal batch size; slots b >= B do nothing).
 * cgpcm_smf_posterior_test: per sample b, P_b = Kx + r (sum_Bxx + C1_b) + reg I (lower triangles read, ld x ld),
 * lam_b = c0 sum_Ahx_y^T h_b, xm[b * ld + k] = (P_b^-1 lam_b)[k], mx[b * ld * ld + k * nx + l] =
 * (P_b^-1 + xm xm^T - iKx)[k][l] (full nx x nx), q1[b] = a + h_b^T Ahh h_b - tr_ahh_ikh[0] (a device scalar).
 * info[b] = pivot + 1 of a failed factorisation of P_b (its other outputs are not written), else 0.  nx <= 2048.
 * cgpcm_predict_quad_test: per point n < nv and sample b < B, with v = V[b * v_stride + n * ldv + k],
 * M_b = mx[b * mx_stride + k * nx + l] and x_b = xm[b * xm_stride + k] (stride 0: one matrix for every sample):
 * quad[n * B + b] = v^T M_b v, lin[n * B + b] = v . x_b and, when qb is not NULL, qb[n * B + b] = <Bxx_n, M_b> with
 * Bxx_n = bxx[n * nx * nx + k * nx + l]. */
int cgpcm_smf_posterior_test(const double* kx, const double* sum_Bxx, const double* c1, const double* sum_Ahx_y,
                             const double* Ahh, const double* iKx, const double* tr_ahh_ikh, const double* samples,
                             int B, int nslots, int nx, int nh, int64_t ld, int ldh, double r, double c0, double reg,
                             double a, double* mx, double* xm, double* q1, int* info, void* stream);
int cgpcm_predict_quad_test(const double* V, int64_t v_stride, int ldv, const double* mx, int64_t mx_stride,
                            const double* xm, int64_t xm_stride, const double* bxx, int nv, int nx, int B, int nslots,
                            double* quad, double* lin, double* qb, void* stream);
/* The pair-block kernel of cgpcm_predict_f_cov (axx_pair_kernel, csrc/predict_kernels.cuh) with its launch shape; device
 * pointers only; returns after the stream has drained.  For i < np, j < nq, k, l < nx, with hyp = (alpha, gamma, omega)
 * on the host and the model's causal / causal_id flags:
 *   X[((i * nq + j) * nx + k) * nx + l] = Axx(tp[i], tq[j])[k][l] - G[(i * gk + k) * ldg + j * gk + l]
 * (G may be NULL: no fold; ldg >= nq gk, gk >= nx), Axx(t1, t2) the Axx statistic with dk = t1 - tx_k, dl = t2 - tx_l,
 * evaluated densely.  -1 for bad shapes, -4 for a non-positive or non-finite hyper-parameter. */
int cgpcm_predict_pair_test(const double* tp, int np, const double* tq, int nq, const double* tx, int nx,
                            const double hyp[3], int causal, int causal_id, const double* G, int64_t ldg, int gk,
                            double* X, void* stream);
/* The kernels of the ELBO sweeps (csrc/psi_kernels.cuh, csrc/linalg.cuh, csrc/dgemm_sym.cuh) through the launch code the
 * sweeps use, and the dense factorisation under every entry point.  Device pointers, except the descriptor arrays and hyp = (alpha, gamma, omega), which are on the host;
 * stream: a cudaStream_t or NULL; each returns after the stream has drained.  -1 for bad shapes, -4 for a non-positive
 * or non-finite hyper-parameter.  sep = 1 selects the separable kernels (default causal model only: causal = 1,
 * causal_id = 0); cull = 0 evaluates every element (threshold 746).
 * cgpcm_ahx_gen_test: one chunk of observations t[0 .. n_valid), n_valid <= nc, nc % 8 == 0, over the window of
 * inducing inputs k_lo .. k_lo + kwp (k_lo even, kwp % 8 == 0, k_lo + kwp <= ld): A[(i * nc + n) * kwp + k] = Ahx for
 * i < nhp (nhp % 8 == 0, nhp >= nh), 0 outside the valid nh x n_valid x nx box; when ypart is not NULL,
 * ypart[s * nhp * ld + i * ld + k_lo + k] = sum over the observations n of slice s (16 per slice) of y_n A, the slices
 * zeroed first ((nc + 15) / 16 slices of nhp x ld).
 * cgpcm_ahx_dot_test: g3[theta] = sum over i < nh, n < n_valid, k_lo + k < nx, elements not culled, of
 * (W[(i * nc + n) * kwp + k] + y_n Ybar[i * ld + k_lo + k]) dA/dtheta, theta = (alpha, gamma, omega), with A the block of
 * cgpcm_ahx_gen_test; the same CTA partials and final sum as the backward sweep.
 * cgpcm_axx_sum_test: out4[m * ld * ld + k * ld + l] = sum_n Axx[n] (m = 0) and its derivatives w.r.t. alpha, gamma,
 * omega (m = 1..3, when tangents), k, l < nx, 0 elsewhere; `slices` observation slices (1..64); sorted = 1 declares t
 * non-decreasing (each pair then visits only its own observation interval).  The pair-hoisted BVN branch is taken as
 * the sweep takes it (causal model, rho = gamma / (alpha + gamma + omega) >= 0.925).
 * cgpcm_window_chol_test: for window w of `windows` (host int32 [nwin][3] = k_lo, kw, kv; kw % 8 == 0, 8 <= kw <= 120,
 * 0 <= kv <= kw, k_lo + kv <= ld), the upper-triangular S_w = L_w^T of sign * M[k_lo .. k_lo + kv, same] padded with
 * the identity to kw x kw, dense at out + sum of kw^2 of the windows before it; all windows in one launch.
 * *info_host = tag * 100000 + k_lo + j + 1 for the first pivot j that was not positive within a window (the window
 * is any of those that have one), else 0.
 * cgpcm_sym_accum_test: out (n x n at ld) = the sum of the windows' products op(A_w) op(B_w)^T, each order_w x order_w at
 * (k_lo_w, k_lo_w), symmetric.  windows: host int64 [nwin][6] = (kc, k_lo, order, K, a_off, b_off); kc = 1:
 * A_w[m][k] = A[a_off + m * K + k], kc = 0: A_w[m][k] = A[a_off + k * order + m], B_w likewise from B at b_off.  The
 * windows are added into the sweep's zeroed K-slice buffers in list order, then summed and mirrored.
 * cgpcm_potrf_test: the blocked Cholesky factorisation (potrf_lower, csrc/linalg.cuh) as the sampling and scoring
 * paths call it: A (np x np at ld, lower triangle read) -> L in place, upper triangle of the np x np block zeroed,
 * nothing outside it touched; a 32 x 32 scratch slot of its own.  A non-positive pivot is replaced by 1 and the
 * factorisation goes on; *info_host = tag * 100000 + j + 1 for the first such pivot j, else 0.  -1 unless
 * np % 8 == 0, np <= ld and ld is even.
 * cgpcm_trtri_test: X = L^-1 (trtri_lower) for the lower-triangular L (np x np at ld), X exactly lower triangular,
 * nothing outside its np x np block touched; a workspace of 32 x ld of its own.  Shapes as cgpcm_potrf_test. */
int cgpcm_ahx_gen_test(const double* t, const double* y, int n_valid, int nc, const double* th, int nh, int nhp,
                       const double* tx, int nx, int k_lo, int kwp, const double hyp[3], int causal, int causal_id,
                       double cull, int sep, int64_t ld, double* A, double* ypart, void* stream);
int cgpcm_ahx_dot_test(const double* t, const double* y, int n_valid, int nc, const double* th, int nh, int nhp,
                       const double* tx, int nx, int k_lo, int kwp, const double hyp[3], int causal, int causal_id,
                       double cull, int sep, int64_t ld, const double* A, const double* W, const double* Ybar,
                       double* g3, void* stream);
int cgpcm_axx_sum_test(const double* t, int n, int sorted, const double* tx, int nx, const double hyp[3], int causal,
                       int causal_id, double cull, int slices, int tangents, int64_t ld, double* out4, void* stream);
int cgpcm_window_chol_test(const double* M, int64_t ld, double sign, int nwin, const int32_t* windows, int tag,
                           double* out, int* info_host, void* stream);
int cgpcm_sym_accum_test(int nwin, const int64_t* windows, const double* A, const double* B, int n, int64_t ld,
                         double* out, void* stream);
int cgpcm_potrf_test(double* A, int np, int64_t ld, int tag, int* info_host, void* stream);
int cgpcm_trtri_test(const double* L, double* X, int np, int64_t ld, void* stream);

#ifdef __cplusplus
}
#endif
#endif

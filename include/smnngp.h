/* libsmnngp - C-ABI of the B200 (sm_100a) NNGP exact-GP hot path.
 *
 * Drop-in boundary for the reference's spax kernel / model / likelihood API
 * (Hyungi-Lee/Scale-Mixtures-of-Neural-Network-Gaussian-Processes).  Every entry point below replaces work the
 * reference delegates to neural_tangents / jax.lax.linalg behind the cited call site.  Conventions:
 *   - all matrices row-major FP64; every pointer is a DEVICE pointer unless the function name ends in _host_f64;
 *   - `stream` is a cudaStream_t passed as void*; functions only enqueue (no host sync, no allocation), so they
 *     are CUDA-graph capturable; the *_host_f64 variants allocate / copy / synchronise themselves;
 *   - `hp_dev` is a device array of 6 doubles {w_std, b_std, last_w_std, eps, alpha, beta} - the softplus'ed
 *     "safe values" of the six trainable scalars (spax/kernels.py:19-21, spax/models.py:91,
 *     spax/likelihoods.py:42-43).  They are runtime operands (traced in the reference), never baked in;
 *   - return value: 0 = ok, non-zero = invalid argument / CUDA error (text via smnngp_last_error()).  A
 *     non-positive-definite matrix is NOT an error: outputs are NaN and *info_dev = 1 + index of the first bad
 *     pivot, mirroring jax's lax.linalg.cholesky NaN semantics that regression/train.py:211 relies on;
 *   - workspaces are caller-owned (so the framework allocator accounts for them): ask *_workspace_bytes first.
 */
#ifndef SMNNGP_H_
#define SMNNGP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMNNGP_ABI_VERSION 1

enum { SMNNGP_OK = 0, SMNNGP_EINVAL = 1, SMNNGP_ECUDA = 2, SMNNGP_EWORKSPACE = 3 };
/* experiments/nt_kernels.py:12-18 get_act_class */
enum { SMNNGP_ACT_RELU = 0, SMNNGP_ACT_ERF = 1 };
/* experiments/nt_kernels.py:21 get_mlp_kernel, :83 get_dense_resnet_kernel */
enum { SMNNGP_ARCH_MLP = 0, SMNNGP_ARCH_RESNET = 1 };
/* spax/likelihoods.py:22 GaussianLikelihood, :37 StudentTLikelihood */
enum { SMNNGP_KIND_GAUSS = 0, SMNNGP_KIND_STUDENT_T = 1 };
/* diagonal regulariser folded into the Gram epilogue:
 *   EPS_ABS  K + eps I                (spax/models.py:96 + spax/utils.py:26-27 jitter)
 *   EPS_REL  K + eps tr(K)/N I        (neural_tangents predict diag_reg, spax/kernels.py:30)
 *   LIK      K + 1e-6 (alpha/beta) I  (spax/likelihoods.py:60, after factoring out beta/alpha) */
enum { SMNNGP_SHIFT_NONE = 0, SMNNGP_SHIFT_EPS_ABS = 1, SMNNGP_SHIFT_EPS_REL = 2, SMNNGP_SHIFT_LIK = 3 };
enum { SMNNGP_OUT_FULL = 0, SMNNGP_OUT_LOWER = 1 };

int smnngp_abi_version(void);
const char* smnngp_last_error(void);

/* ---- Gram: replaces kernel_fn(x1, x2, get="nngp") of spax/kernels.py:23-27 with the layer stacks of
 * experiments/nt_kernels.py:21-31 / :83-103.  X2 == NULL (or == X) selects the symmetric path: only tiles on or
 * below the diagonal are computed; out_mode FULL mirrors them, LOWER leaves the strict upper part untouched.
 * `shift` is only honoured on the symmetric path. */
size_t smnngp_gram_workspace_bytes(int64_t N, int64_t M, int n_hidden, int arch);
int smnngp_gram_f64(void* stream, const double* X, const double* X2, int64_t N, int64_t M, int64_t D,
                    int n_hidden, int act, int arch, const double* hp_dev, int shift, int out_mode,
                    double* K_out, int64_t ld, void* workspace, size_t workspace_bytes);
/* marginal variances k(x_i, x_i) of the same stack (the diagonal NT carries as cov1) */
int smnngp_nngp_diag_f64(void* stream, const double* X, int64_t N, int64_t D, int n_hidden, int act, int arch,
                         const double* hp_dev, double* q_out, void* workspace, size_t workspace_bytes);

/* ---- Cholesky: replaces lax.linalg.cholesky (spax/utils.py:179).  In place on the lower triangle of the
 * row-major A; the strict upper triangle is neither read nor written.  The trapezoid form factors the leading
 * N x N of A [M, N] (M >= N) and turns the extra rows R into R L^-T, i.e. it also performs the triangular
 * solves of spax/utils.py:180 / cho_solve for right-hand sides appended as rows.
 * *logdet_dev receives sum_i log L_ii. */
size_t smnngp_potrf_workspace_bytes(int64_t N);
int smnngp_potrf_f64(void* stream, double* A, int64_t N, int64_t ld, int* info_dev, void* workspace,
                     size_t workspace_bytes);
int smnngp_potrf_trapezoid_f64(void* stream, double* A, int64_t M, int64_t N, int64_t ld, double* logdet_dev,
                               int* info_dev, void* workspace, size_t workspace_bytes);

/* ---- generic covariance solve: factors (scale * cov + shift I) in workspace (cov is not modified) and returns
 * out_dev[2] = { sum_i log L_ii, ||L^-1 y||^2 }.  Backs Likelihood.prior_logpdf(y, cov)
 * (spax/likelihoods.py:25-28, :45-50) and the `d` term of StudentTLikelihood.logpdf (:60-61) when the caller
 * passes an explicit covariance instead of using the fused entry points.  N < 65535. */
size_t smnngp_cov_solve_workspace_bytes(int64_t N);
int smnngp_cov_solve_f64(void* stream, const double* cov, int64_t N, int64_t ld, const double* y, double scale,
                         double shift, void* workspace, size_t workspace_bytes, double* out_dev, int* info_dev);

/* ---- fused log marginal likelihood: replaces SPR.loss (spax/models.py:93-98) =
 * Gram + jitter + prior_logpdf (spax/likelihoods.py:25-28 / :45-50 -> spax/utils.py:160-183).
 * out_dev[4] = { log p(y), -log p(y)/N (the loss), sum_i log L_ii of chol(K + eps I), ||L^-1 y||^2 }.
 * The N x N matrix lives only in `workspace`. */
size_t smnngp_lml_workspace_bytes(int64_t N, int64_t D, int n_hidden, int arch);
int smnngp_lml_f64(void* stream, const double* X, const double* y, int64_t N, int64_t D, int n_hidden, int act,
                   int arch, const double* hp_dev, int kind, void* workspace, size_t workspace_bytes,
                   double* out_dev, int* info_dev);

/* ---- loss AND its gradient w.r.t. the six scalars: what objax.GradValues(model.loss, model.vars()) evaluates at
 * every step of the reference's training loop (experiments/regression/train.py:62-66, :178-179) by reverse-mode
 * AD through spax/models.py:93-98.  out_dev[4] as smnngp_lml_f64; grad_dev[6] = d loss / d {w_std, b_std,
 * last_w_std, eps, alpha, beta} (loss = -log p / N; derivatives w.r.t. the constrained "safe" values - the caller
 * applies the softplus chain rule, spax/bijectors.py:51-53).  A^-1 is formed explicitly from the factor (identity
 * rows carried through the factorisation, one SYRK) and dK/dtheta is contracted inside a second Gram pass in dual
 * arithmetic; ~3x the work of the value alone, workspace 16 N^2 bytes.  Bit-reproducible. */
size_t smnngp_lml_grad_workspace_bytes(int64_t N, int64_t D, int n_hidden, int arch);
int smnngp_lml_grad_f64(void* stream, const double* X, const double* y, int64_t N, int64_t D, int n_hidden, int act,
                        int arch, const double* hp_dev, int kind, void* workspace, size_t workspace_bytes,
                        double* out_dev, double* grad_dev, int* info_dev);

/* ---- predictive: replaces NNGPKernel.predict (spax/kernels.py:29-32 -> neural_tangents
 * gradient_descent_mse_ensemble, get="nngp", compute_cov=True) with `shift` = EPS_REL.  Y is [N, C];
 * mean_out [T, C]; var_out [T] = diag(cov) - the only part of cov the reference consumes
 * (spax/likelihoods.py:31, :62). */
size_t smnngp_predict_workspace_bytes(int64_t N, int64_t T, int64_t C, int64_t D, int n_hidden, int arch);
int smnngp_predict_f64(void* stream, const double* X, const double* Y, const double* Xt, int64_t N, int64_t T,
                       int64_t C, int64_t D, int n_hidden, int act, int arch, const double* hp_dev, int shift,
                       void* workspace, size_t workspace_bytes, double* mean_out, double* var_out,
                       int* info_dev);

/* same, plus the FULL posterior covariance cov_out [T, ld_cov] = K_tt - K_td A^-1 K_dt that neural_tangents
 * returns with compute_cov=True (spax/kernels.py:31; consumed whole only by the SVSP path, spax/models.py:43) */
int smnngp_predict_cov_f64(void* stream, const double* X, const double* Y, const double* Xt, int64_t N, int64_t T,
                           int64_t C, int64_t D, int n_hidden, int act, int arch, const double* hp_dev, int shift,
                           void* workspace, size_t workspace_bytes, double* mean_out, double* var_out,
                           double* cov_out, int64_t ld_cov, int* info_dev);

/* ---- SPR.test_nll (spax/models.py:100-120) incl. Likelihood.logpdf (spax/likelihoods.py:30-33 / :52-65):
 * predictive (relative jitter) + second factorisation of K + 1e-6 (alpha/beta) I for the Student-t scale +
 * de-standardisation + mean negative log density.  nll_out_dev[1]; mean_out / var_out / logp_out are [T] and
 * may be NULL.  workspace: smnngp_predict_workspace_bytes(N, T, 1, D, ...). */
int smnngp_test_nll_f64(void* stream, const double* X, const double* y, const double* Xt, const double* yt,
                        int64_t N, int64_t T, int64_t D, int n_hidden, int act, int arch, const double* hp_dev,
                        int kind, double y_mean, double y_std, void* workspace, size_t workspace_bytes,
                        double* nll_out_dev, double* mean_out, double* var_out, double* logp_out,
                        int* info_dev);

/* ---- hyper-parameter grid search with a cached base Gram (SURVEY section 8f row N3): the reference's
 * experiments/regression/find.py:134-199 evaluates, for every (w_std, b_std) x eps of a grid, the kernel matrix
 * (find.py:64-70), the predictive with the relative regulariser (find.py:73-78) and the log-determinant / quadratic
 * form of K + eps I (find.py:149-156) on the SAME inputs.  X.X'^T does not depend on the scalars:
 *   grid_base   K0dd [N, ld0] (lower) = X X^T / D, K0td [T, ld0t] = Xt X^T / D, q_d [N], q_t [T] = ||x||^2 / D   (once)
 *   grid_point  one grid point from the bases: recursion-only passes (8 B read + 8 B written per entry) + the two
 *               factorisations.  mean_out [T], var_out [T] (predict(eps), relative regulariser);
 *               out_dev[2] = { sum log L_ii of chol(K + eps I)  (= 1/2 log det),  y^T (K + eps I)^-1 y }.
 * The (alpha, beta) importance-sampling table that follows (find.py:163-186) is host arithmetic on these outputs. */
int smnngp_grid_base_f64(void* stream, const double* X, const double* Xt, int64_t N, int64_t T, int64_t D,
                         double* K0dd, int64_t ld0, double* K0td, int64_t ld0t, double* q_d, double* q_t);
size_t smnngp_grid_workspace_bytes(int64_t N, int64_t T, int n_hidden, int arch);
int smnngp_grid_point_f64(void* stream, const double* K0dd, int64_t ld0, const double* K0td, int64_t ld0t,
                          const double* q_d, const double* q_t, const double* y, int64_t N, int64_t T, int n_hidden,
                          int act, int arch, const double* hp_dev, void* workspace, size_t workspace_bytes,
                          double* mean_out, double* var_out, double* out_dev, int* info_dev);
/* grid_batch  G points in ONE launch for N <= 4096 (the reference's UCI sizes), where a single point leaves the GPU
 *             nearly idle: a CTA evaluates a whole point in its own slot of the workspace and walks the points with a
 *             static stride.  Inputs as grid_point; hp_dev [G][6]; mean_out [G][T], var_out [G][T], out_dev [G][2] and
 *             info_dev [G]: row g is what grid_point returns for hp_dev + 6 g (NaN outputs when a factorisation fails),
 *             and no point affects another: a point's outputs are the same bits in any batch, order or slot count.
 *             The slot count (points in flight) is workspace_bytes / smnngp_grid_batch_workspace_bytes(.., 1); each
 *             slot holds the (N + T + 1) x N trapezoid and the layer tables.  Fewer than one slot: SMNNGP_EWORKSPACE;
 *             N > 4096, T < 1, G < 1, a null pointer, ld0 or ld0t < N or an invalid stack: SMNNGP_EINVAL, both before
 *             anything is enqueued.  Enqueue-only (one kernel launch), no allocation, graph-capturable. */
size_t smnngp_grid_batch_workspace_bytes(int64_t N, int64_t T, int n_hidden, int arch, int64_t slots);
int smnngp_grid_batch_f64(void* stream, const double* K0dd, int64_t ld0, const double* K0td, int64_t ld0t,
                          const double* q_d, const double* q_t, const double* y, int64_t N, int64_t T, int64_t G,
                          int n_hidden, int act, int arch, const double* hp_dev, void* workspace,
                          size_t workspace_bytes, double* mean_out, double* var_out, double* out_dev, int* info_dev);
/* lml_grad_batch  SPR.loss and its gradient at G points in ONE launch for N <= 4096 (multi-start training, gradient
 *             refinement of a grid search).  K0dd / ld0 / q_d are the bases of grid_base with T = 0, y [N] the targets;
 *             hp_dev [G][6]; kind as smnngp_lml_grad_f64 (absolute regulariser K + eps I).  out_dev [G][4], grad_dev
 *             [G][6] and info_dev [G]: row g is what smnngp_lml_grad_f64 returns for hp_dev + 6 g, up to rounding
 *             (same matrix, different blocking).  When a factorisation fails all of out_dev[g] and grad_dev[g] are
 *             NaN and info_dev[g] = 1 + the first bad pivot.  No point affects another: a point's outputs are the
 *             same bits in any batch, order or slot count.  The slot count is workspace_bytes /
 *             smnngp_lml_grad_batch_workspace_bytes(.., 1); each slot holds the (2N + 1) x N trapezoid A | y^T | I,
 *             the dual layer tables and A^-1 y.  Fewer than one slot: SMNNGP_EWORKSPACE; N < 1, N > 4096, G < 1, a
 *             null pointer, ld0 < N, an invalid stack or kind: SMNNGP_EINVAL, both before anything is enqueued.
 *             Enqueue-only (one kernel launch), no allocation, graph-capturable. */
size_t smnngp_lml_grad_batch_workspace_bytes(int64_t N, int n_hidden, int arch, int64_t slots);
int smnngp_lml_grad_batch_f64(void* stream, const double* K0dd, int64_t ld0, const double* q_d, const double* y,
                              int64_t N, int64_t G, int n_hidden, int act, int arch, const double* hp_dev, int kind,
                              void* workspace, size_t workspace_bytes, double* out_dev, double* grad_dev,
                              int* info_dev);
/* test_nll_batch  SPR.test_nll at G points in ONE launch for N <= 4096 (the validation / test NLL of multi-start
 *             training, selection of grid points by held-out NLL).  K0dd / K0td / q_d / q_t are the bases of grid_base,
 *             y [N] the training targets, yt [T] the standardised test targets; hp_dev [G][6]; kind, y_mean and
 *             y_std as smnngp_test_nll_f64.  nll_out [G] and info_dev [G]; mean_out, var_out and logp_out are [G][T]
 *             each and may be NULL.  Row g is what smnngp_test_nll_f64 returns for hp_dev + 6 g, up to rounding (same
 *             matrices, different blocking).  mean / var of a point are NaN when its predictive factorisation
 *             (K + eps tr(K)/N I) fails; nll and logp are NaN when it or the Student-t one (K + 1e-6 (alpha/beta) I)
 *             fails; info_dev[g] is the first bad pivot (1-based) of the predictive factorisation, else of the
 *             Student-t one, else 0.  No point affects another, and nll does not depend on which optional outputs
 *             are asked for: a point's outputs are the same bits in any batch, order or slot count.  The slot count
 *             is workspace_bytes / smnngp_test_nll_batch_workspace_bytes(.., 1); each slot holds the (N + T + 1) x N
 *             trapezoid, the layer tables and 2T doubles of mean / var.  Fewer than one slot: SMNNGP_EWORKSPACE;
 *             N < 1, N > 4096, T < 1, G < 1, a null required pointer, ld0 or ld0t < N, an invalid stack or kind:
 *             SMNNGP_EINVAL, both before anything is enqueued.  Enqueue-only (one kernel launch), no allocation,
 *             graph-capturable. */
size_t smnngp_test_nll_batch_workspace_bytes(int64_t N, int64_t T, int n_hidden, int arch, int64_t slots);
int smnngp_test_nll_batch_f64(void* stream, const double* K0dd, int64_t ld0, const double* K0td, int64_t ld0t,
                              const double* q_d, const double* q_t, const double* y, const double* yt,
                              int64_t N, int64_t T, int64_t G, int n_hidden, int act, int arch,
                              const double* hp_dev, int kind, double y_mean, double y_std,
                              void* workspace, size_t workspace_bytes,
                              double* nll_out, double* mean_out, double* var_out, double* logp_out, int* info_dev);

/* ---- posterior draw stage of the classification / ensemble configuration (SURVEY section 8f, row N2).
 * mean [T, C]; var [T] (shared by the classes, var_per_class = 0) or [C, T] (var_per_class = 1); kind STUDENT_T:
 * InverseGammaPrior.sample_f_iid (spax/priors.py:60-68), f = mean + sqrt((b/a) var) t_{2a}; kind GAUSS:
 * GaussianPrior.sample_f_iid (spax/priors.py:30-36).  Counter-based Philox stream keyed by `seed`.
 *   sample_f_iid : materialises out [C, T, S]
 *   draw_metrics : the same draws, never written: per-point log-likelihood of the true label
 *                  logsumexp_s(log_softmax_c f)[label] - log S  (spax/utils.py:61-66), predicted class
 *                  argmax_c logsumexp_s log_softmax (spax/utils.py:69-74); out_dev[2] = { nll, correct count }.
 *                  A label outside [0, C) gives ll_per_test = NaN (so nll = NaN) and never counts as correct.
 * Both draw the same value for the same (seed, s, t, c) and launch on the device of `stream`.  T, C or S < 1,
 * T or S > INT32_MAX, for sample_f_iid C > INT32_MAX or C * T * S > INT64_MAX, for draw_metrics C > 16, an invalid
 * kind or a null pointer: SMNNGP_EINVAL before anything is enqueued, with smnngp_last_error() naming the call. */
int smnngp_sample_f_iid_f64(void* stream, const double* mean, const double* var, int var_per_class, int64_t T,
                            int64_t C, int64_t S, const double* hp_dev, int kind, uint64_t seed, double* out);
int smnngp_draw_metrics_f64(void* stream, const double* mean, const double* var, int var_per_class,
                            const int* label, int64_t T, int64_t C, int64_t S, const double* hp_dev, int kind,
                            uint64_t seed, double* ll_per_test, int* pred, double* out_dev);

/* ---- stage-level entry points (multi-GPU driver: one process per GPU interleaves these with NCCL collectives;
 * same kernels as the fused calls).  Layout and algorithm: DESIGN.md section 7.
 *   qtable      per-row layer tables (+ optional scalar block: tr(K)/N and the shift values)
 *   gram        one block of the Gram matrix (symmetric_lower: X1 == X2 rows, lower part + diagonal shift)
 *   factor_diag Cholesky of a diagonal block, keeps inv(L) of every 128-block (linv_blocks [ceil(w/128)][128*128])
 *   trsm        panel rows <- rows * L^-T by 128-block substitution
 *   update      C -= A B^T with the (block-row-cyclic) lower mask: local row r of the region belongs to local
 *               block r / cyc_db; its largest active column is r + base_shift + (r / cyc_db) (cyc_p - 1) cyc_db;
 *               sm_reserve SMs are left free for look-ahead work running on another stream
 *   sumsq, lml_finalize   reductions / closed form on (all-reduced) scalars */
int smnngp_stage_qtable_f64(void* stream, const double* X, int64_t N, int64_t D, int n_hidden, int act, int arch,
                            const double* hp_dev, double* tab, int64_t tab_ld, double* q, double* scal);
int smnngp_stage_gram_f64(void* stream, const double* X1, int64_t n1, const double* X2, int64_t n2, int64_t D,
                          int n_hidden, int act, int arch, const double* hp_dev, const double* tab1,
                          int64_t tab_ld1, const double* tab2, int64_t tab_ld2, const double* scal, int shift,
                          int symmetric_lower, double* K, int64_t ldk);
int smnngp_stage_factor_diag_f64(void* stream, double* A, int64_t lda, int64_t w, double* linv_blocks,
                                 double* logdet_dev, int* info_dev, int64_t gcol0);
int smnngp_stage_trsm_f64(void* stream, double* R, int64_t ldr, int64_t m, int64_t w, const double* L, int64_t ldl,
                          const double* linv_blocks);
int smnngp_stage_update_f64(void* stream, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                            int64_t ldc, int64_t M, int64_t N, int64_t K, int lower, int64_t cyc_db, int64_t cyc_p,
                            int64_t base_shift, int sm_reserve);
int smnngp_stage_sumsq_f64(void* stream, const double* z, int64_t n, double* out_dev);
/* predictive tail on rows carried through the (distributed) factorisation: V [T, ldv] = K_td L^-T, Z [C, ldz] =
 * (L^-1 Y)^T, ktt [T] -> mean [T, C] = V Z^T, var [T] = ktt - ||v||^2 (spax/kernels.py:29-32; NaN when *info_dev != 0) */
/* SPR.test_nll tail (spax/models.py:114-119 with Likelihood.logpdf, spax/likelihoods.py:30-33 / :52-65) on predictive
 * moments: de-standardisation, per-point log density (logp [T], may be NULL) and nll_out_dev[1] = -mean.  quad2_dev =
 * ||L2^-1 y||^2 of the factorisation of K + 1e-6 (alpha/beta) I (Student-t; NULL allowed for gauss) */
int smnngp_stage_test_nll_finalize_f64(void* stream, const double* mean, const double* var, const double* ytest,
                                       int64_t T, int64_t N, double y_mean, double y_std, const double* hp_dev, int kind,
                                       const double* quad2_dev, const int* info_dev, double* logp, double* nll_out_dev);
int smnngp_stage_predict_finalize_f64(void* stream, const double* V, int64_t ldv, const double* Z, int64_t ldz,
                                      const double* ktt, int64_t T, int64_t C, int64_t N, const int* info_dev,
                                      double* mean, double* var);
int smnngp_stage_lml_finalize_f64(void* stream, const double* sums_dev, const double* hp_dev, int kind, int64_t N,
                                  const int* info_dev, double* out_dev);

/* ---- multi-GPU panel exchange by peer stores over NVLink (csrc/exchange.cu; replaces one ncclBroadcast + one
 * ncclAllGather per panel).  Pointer arrays are HOST arrays of P device pointers (index = rank), read at call time.
 *   factor_diag_inv : factor the diagonal block inside the scratch T [2w, w] with identity rows carried along:
 *                     T rows 0..w-1 = L, rows w..2w-1 = L^-T (A is only read)
 *   scatter_inverse : W = inv(L) = (L^-T)^T, lower triangular row-major, stored into every rank's buffer, then the
 *                     flag word `flag_index` of every rank is set to seq
 *   trsm_scatter    : Ploc = R W^T (tensor pipe, one launch) and the same rows stored at (global row - c1) of every
 *                     rank's panel buffer; the last CTA sets flag word `flag_index` on every rank to seq
 *   signal / wait_flags : raise a flag on every rank / one-thread spin until flags[first .. first+count) >= seq;
 *                     after timeout_s the wait gives up and sets *info_dev = INT_MAX (results become NaN) so a dead
 *                     peer cannot hang the device */
int smnngp_stage_factor_diag_inv_f64(void* stream, const double* A, int64_t lda, int64_t w, double* T,
                                     double* linv_ws, double* logdet_dev, int* info_dev, int64_t gcol0);
int smnngp_stage_scatter_inverse_f64(void* stream, const double* Ut, int64_t ldu, int64_t w, void* const* dst_ptrs,
                                     int P, int64_t ldw, void* const* flag_ptrs, int64_t flag_index, uint64_t seq,
                                     unsigned int* counter);
int smnngp_stage_signal_f64(void* stream, void* const* flag_ptrs, int P, int64_t flag_index, uint64_t seq);
int smnngp_stage_wait_flags_f64(void* stream, const void* flags_local, int64_t first, int count, uint64_t seq,
                                double timeout_s, int* info_dev);
/* copy-engine flavour of the all-gather: trsm_scatter is called with P = 1 (own buffers only), then push_panel copies
 * the solved rows (whole distribution blocks, w == db) to every other rank's panel buffer with cudaMemcpy2DAsync over
 * NVLink and raises this rank's flag everywhere */
int smnngp_stage_push_panel_f64(void* stream, const double* Ploc, int64_t m, int64_t w, int64_t db, int P, int rank,
                                int64_t local_row0, int64_t c1, int64_t n, void* const* peer_ptrs,
                                void* const* flag_ptrs, int64_t flag_index, uint64_t seq);
/* how wait_flags waits: 0 (default) = cuStreamWaitValue64 on the stream (no SM occupied, no timeout), 1 = one-thread
 * spin kernel with the timeout described above */
void smnngp_set_peer_wait_mode(int mode);
/* variants for the snake (boustrophedon) block distributions of csrc/multigpu.cu: cyc_alt = extra column shift of the
 * rows of odd local blocks in the update mask; even_off / odd_off: the global block of this rank's local block lb is
 * lb * P + (lb odd ? odd_off : even_off)  (plain cyclic: both = rank) */
int smnngp_stage_update2_f64(void* stream, const double* A, int64_t lda, const double* B, int64_t ldb, double* C,
                             int64_t ldc, int64_t M, int64_t N, int64_t K, int lower, int64_t cyc_db, int64_t cyc_p,
                             int64_t base_shift, int64_t cyc_alt, int sm_reserve);
int smnngp_stage_trsm_scatter2_f64(void* stream, const double* R, int64_t ldr, int64_t m, int64_t w, const double* W,
                                   int64_t ldw, double* Ploc, int64_t ldp, void* const* peer_ptrs, int P, int rank,
                                   int64_t db, int64_t local_row0, int64_t c1, int64_t n, int64_t ld_peer,
                                   void* const* flag_ptrs, int64_t flag_index, uint64_t seq, unsigned int* counter,
                                   int64_t even_off, int64_t odd_off);
int smnngp_stage_trsm_scatter_f64(void* stream, const double* R, int64_t ldr, int64_t m, int64_t w, const double* W,
                                  int64_t ldw, double* Ploc, int64_t ldp, void* const* peer_ptrs, int P, int rank,
                                  int64_t db, int64_t local_row0, int64_t c1, int64_t n, int64_t ld_peer,
                                  void* const* flag_ptrs, int64_t flag_index, uint64_t seq, unsigned int* counter);

/* W = inv(L) of a factored panel diagonal block (w <= 512) assembled from L and the inverses of its 128 x 128
 * diagonal blocks (what smnngp_stage_factor_diag_f64 leaves behind), stored into the W buffer of every rank; when
 * flag_ptrs / counter are given the last CTA sets flag word `flag_index` on every rank to seq */
int smnngp_stage_assemble_inverse_f64(void* stream, const double* L, int64_t ldl, int64_t w, const double* linv_blocks,
                                      void* const* dst_ptrs, int P, int64_t ldw, void* const* flag_ptrs,
                                      int64_t flag_index, uint64_t seq, unsigned int* counter);

/* ---- multi-GPU in ONE call per rank (csrc/multigpu.cu; SURVEY.md section 8b "multi-GPU variants", 8e) ------------
 * Replaces, for the sharded case, the same reference lines as smnngp_lml_f64 (spax/models.py:93-98 under objax.Jit,
 * experiments/regression/train.py:61-67).  One handle per rank owns everything the distributed factorisation needs
 * (row shard of K, NVLink-visible panel / W / flag / reduce buffers, side stream, watchdog); the library needs no
 * communicator: the caller moves the 64-byte IPC handles between the processes once (any transport), or connects
 * several devices of one process by pointer.
 *   smnngp_mg_create         on the rank's device (current device); block = distribution block = outer panel width
 *                            (multiple of 128, <= 512)
 *   smnngp_mg_ipc_handle     64-byte CUDA IPC handle of the rank's peer-visible region
 *   smnngp_mg_connect_ipc    handles = world x 64 bytes, rank-major (one process per GPU)
 *   smnngp_mg_connect_ptrs   regions[r] = smnngp_mg_region() of rank r (same process, peer access enabled inside)
 *   smnngp_mg_connect_emulated  timing dry-run of one rank on one device (all peers alias the local region)
 *   smnngp_lml_mg_f64        enqueue-only on `stream` (same device as the handle); every rank passes the same X, y, hp
 *                            (device pointers on ITS device); out_dev[4] as smnngp_lml_f64, identical on every rank;
 *                            shift = SMNNGP_SHIFT_* added to the Gram diagonal (SMNNGP_SHIFT_EPS_ABS for SPR.loss)
 *   a peer that dies cannot hang the GPU: a host watchdog releases the stream waits after the time-out (default 20 s)
 *   and poisons info (all results NaN); the handle is unusable afterwards */
typedef struct smnngp_mg smnngp_mg;
int smnngp_mg_create(smnngp_mg** out, int rank, int world, int64_t n, int64_t block);
int smnngp_mg_destroy(smnngp_mg* g);
int smnngp_mg_ipc_handle(smnngp_mg* g, unsigned char* handle_out64);
void* smnngp_mg_region(smnngp_mg* g);
int smnngp_mg_connect_ipc(smnngp_mg* g, const unsigned char* handles);
int smnngp_mg_connect_ptrs(smnngp_mg* g, void* const* regions, const int* peer_devices);
int smnngp_mg_connect_emulated(smnngp_mg* g);
void smnngp_mg_set_timeout(smnngp_mg* g, double seconds);
void smnngp_mg_set_sm_reserve(smnngp_mg* g, int sms);         /* < 0: automatic (default) */
void smnngp_mg_set_reserve_margin(smnngp_mg* g, double margin); /* automatic reserve = margin * 82.5 w / ncols + 3 (4.5) */
void smnngp_mg_timeline(smnngp_mg* g, int enable);            /* profiling: CUDA events at the stage boundaries */
int smnngp_mg_timeline_read(smnngp_mg* g, int cap, int* panel_out, int* label_out, double* ms_out);
const char* smnngp_mg_last_error(void);
/* pure host function: the block -> rank map of a handle (layout: 0 cyclic, 1 snake, 2 snake_end, 3 auto = default;
 * env SMNNGP_MG_LAYOUT overrides the default of smnngp_mg_create); owner_out [nblocks], load_out [world] (optional,
 * modelled update work per rank); returns the number of distribution blocks */
int64_t smnngp_mg_layout(int world, int64_t n, int64_t extra_rows, int64_t block, int layout, int* owner_out,
                         double* load_out);
int smnngp_lml_mg_f64(smnngp_mg* g, void* stream, const double* X, const double* y, int64_t D, int n_hidden, int act,
                      int arch, const double* hp_dev, int kind, int shift, double* out_dev, int* info_dev);
/* NNGPKernel.predict (spax/kernels.py:29-32) / SPR.test_nll (spax/models.py:100-120, spax/likelihoods.py:30-33, :52-65)
 * on the handle group.  smnngp_mg_create_predict: T test points and C right-hand sides ride through the distributed
 * factorisation as extra global rows.  predict: Y [N, C] row-major, Xt [T, D] -> mean_out [T, C], var_out [T] (diag of
 * the posterior covariance), identical on every rank; shift = SMNNGP_SHIFT_EPS_REL for the reference semantics.
 * test_nll: g_pred built with c = 1, g_lik a plain smnngp_mg_create handle of the same n / block / group (second
 * factorisation K + 1e-6 (a/b) I of the Student-t likelihood; may be NULL for kind = gauss) -> nll_out_dev [1]. */
int smnngp_mg_create_predict(smnngp_mg** out, int rank, int world, int64_t n, int64_t t, int64_t c, int64_t block);
/* SPR.loss AND d loss / d {w_std, b_std, last_w_std, eps, alpha, beta} on the handle group - the value / gradient pair
 * objax.GradValues(model.loss, model.vars()) produces in the reference's train step (experiments/regression/train.py:
 * 62-66; the softplus chain rule is the caller's, as for smnngp_lml_grad_f64).  smnngp_mg_create_grad: the N identity
 * rows ride through the distributed factorisation (-> U = L^-T), U is all-gathered over NVLink (every rank needs
 * 8 N^2 bytes for it), every rank contracts one row strip of A^-1 = U U^T with dK/dtheta.  out_dev[4] as
 * smnngp_lml_mg_f64, grad_dev[6], identical on every rank. */
int smnngp_mg_create_grad(smnngp_mg** out, int rank, int world, int64_t n, int64_t block);
int smnngp_lml_grad_mg_f64(smnngp_mg* g, void* stream, const double* X, const double* y, int64_t D, int n_hidden,
                           int act, int arch, const double* hp_dev, int kind, double* out_dev, double* grad_dev,
                           int* info_dev);
int smnngp_predict_mg_f64(smnngp_mg* g, void* stream, const double* X, const double* Y, const double* Xt, int64_t D,
                          int n_hidden, int act, int arch, const double* hp_dev, int shift, double* mean_out,
                          double* var_out, int* info_dev);
int smnngp_test_nll_mg_f64(smnngp_mg* g_pred, smnngp_mg* g_lik, void* stream, const double* X, const double* y,
                           const double* Xt, const double* yt, int64_t D, int n_hidden, int act, int arch,
                           const double* hp_dev, int kind, double y_mean, double y_std, double* nll_out_dev,
                           double* mean_out, double* var_out, int* info_dev);

/* ---- peer memory (multi-GPU, one process per GPU): cudaMalloc'ed buffers exported / imported as 64-byte CUDA IPC
 * handles so that every rank can store into every other rank's panel buffer over NVLink (no reference
 * counterpart: the reference is single-device). */
int smnngp_peer_alloc(size_t bytes, void** ptr_out, unsigned char* handle_out64);
int smnngp_peer_open(const unsigned char* handle64, void** ptr_out);
int smnngp_peer_close(void* ptr);
int smnngp_peer_free(void* ptr);

/* ---- host-buffer entry points (what a ctypes / cgo / JNI caller without device arrays binds): inputs and
 * outputs are HOST pointers; device staging comes from a grow-only arena released by smnngp_host_release(). */
int smnngp_lml_host_f64(const double* X, const double* y, int64_t N, int64_t D, int n_hidden, int act, int arch,
                        const double* hp, int kind, double* out, int* info);
int smnngp_lml_grad_host_f64(const double* X, const double* y, int64_t N, int64_t D, int n_hidden, int act, int arch,
                             const double* hp, int kind, double* out, double* grad, int* info);
int smnngp_predict_host_f64(const double* X, const double* Y, const double* Xt, int64_t N, int64_t T, int64_t C,
                            int64_t D, int n_hidden, int act, int arch, const double* hp, int shift,
                            double* mean_out, double* var_out, int* info);
int smnngp_test_nll_host_f64(const double* X, const double* y, const double* Xt, const double* yt, int64_t N,
                             int64_t T, int64_t D, int n_hidden, int act, int arch, const double* hp, int kind,
                             double y_mean, double y_std, double* nll_out, double* mean_out, double* var_out,
                             int* info);
void smnngp_host_release(void);

/* tuning knob: outer panel width of the Cholesky (multiple of 128; 0 = automatic) */
void smnngp_set_panel_width(int nb);
/* tuning knob: GEMM core. 0 = TMA-fed persistent ping-pong kernel (default; cp.async 128x64 for unaligned
 * operands); 1 = cp.async 128x128, one CTA per SM; 2 = cp.async 128x64, two CTAs per SM */
void smnngp_set_tile_variant(int v);
/* tuning knob: 1 (default) = the fused Cholesky factors the next panel's diagonal block on an internal
 * high-priority side stream while the bulk of the trailing update runs (fork / join with events: still
 * enqueue-only and graph-capturable); 0 = single stream */
void smnngp_set_lookahead(int on);
/* 1 (default): per outer panel the rows below the diagonal block are solved by ONE launch (full inverse of the block,
 * out of place); 0: 128-block substitution in place (round-1 path).  Applies to the current device. */
void smnngp_set_fused_panel(int on);
/* tuning knob: the look-ahead factorisation (N >= 8192, 512-wide panels) hands its last <= cols columns to the
 * single-stream 128-column path, whose per-step chain is shorter than a 512-wide panel's once the trailing update is
 * small.  Default 2048 (measured: 10.07 -> 9.81 ms at N = 8192; 4096 is slower); 0 = never.  Applies to the current device. */
void smnngp_set_tail_cols(int64_t cols);
/* tuning knob: L2-aware tile walk of the Gram kernel - tiles are visited in square super-tiles of `sr` x 2 sr tiles
 * (128 sr elements a side) so that the operand rows of the tiles in flight stay L2 resident; 0 = row-major walk.
 * Used when the column operand (M x D doubles) is at least min_operand_bytes (default 40 MB; < 0 restores it).
 * Default sr = 8.  Applies to the current device. */
void smnngp_set_gram_super_rows(int sr, int64_t min_operand_bytes);
/* tuning knob: SMs the bulk trailing update leaves free for the look-ahead chain (the persistent update kernel
 * would otherwise hold every SM until it ends): trailing matrix narrower than 24000 columns / wider.  Default 8, 0
 * (measured at C3: reserving even 1 SM costs more than the exposed diagonal-block chain, 2234 vs 2224 ms) */
void smnngp_set_lookahead_reserve(int small_trailing, int large_trailing);
/* diagnostic: device buffer (>= 64 int64) receiving clock64() at the phase boundaries of the diagonal-block
 * kernel; NULL switches it off */
void smnngp_debug_potf2_clocks(long long* dev_buf);
/* resident CTAs per SM of the update kernel for a tile variant (diagnostic) */
int smnngp_debug_occupancy(int variant);

/* ---- instrumentation (bench.py; no reference counterpart): kernel-launch counter, CUDA-event timing of the
 * Cholesky trailing updates (the dominant kernel) and a register-resident DMMA.8x8x4 issue-rate probe that
 * measures the FP64 tensor peak of the device the roofline fraction is quoted against. */
void smnngp_instr_reset(int time_updates);
long long smnngp_instr_launches(void);
int smnngp_instr_updates(double* total_ms, double* alg_flops);
double smnngp_dmma_peak_tflops(void);

#ifdef __cplusplus
}
#endif
#endif /* SMNNGP_H_ */

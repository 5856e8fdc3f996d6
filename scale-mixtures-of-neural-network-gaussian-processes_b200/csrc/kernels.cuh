// Internal (C++) launch interface of libsmnngp: every function only enqueues work on `stream`.
#pragma once
#include "common.cuh"

namespace smnngp {

constexpr int HP_W = 0, HP_B = 1, HP_V = 2, HP_EPS = 3, HP_ALPHA = 4, HP_BETA = 5, HP_COUNT = 6;
constexpr int PB = 128;  // diagonal block / inner panel width of the Cholesky
constexpr int LINV_BLOCKS = 4;   // inverse diagonal blocks kept per outer panel (NB <= 512)

// 0 = TilePair (128x64, two CTAs per SM; default), 1 = TileBig (128x128, one CTA per SM)
int& tile_variant();
int debug_gemm_occupancy(int variant);
// 1 (default): the fused factorisation runs the next panel's diagonal block on a side stream (look-ahead)
int& lookahead_mode();
// super-tile height (in 128-row tiles) of the Gram kernel's L2-aware tile walk; 0 = plain row-major walk
int& gram_super_rows();
int* lookahead_reserve();
// diagnostic: when non-null, thread 0 of the diagonal-block kernel stores clock64() at its phase boundaries
long long*& potf2_clock_buffer();

__host__ __device__ inline int n_act_applications(int n_hidden, int arch) { return arch == ARCH_RESNET ? n_hidden + 1 : n_hidden; }

struct GramParams {
  const double* X1;   // [N, D] rows of the output
  const double* X2;   // [M, D] cols of the output (== X1 for the symmetric case)
  long long ld1, ld2;
  int N, M, D;
  const double* tab1; // [n_act, tab_ld1] per-layer encoded marginal variances of X1 rows
  const double* tab2;
  long long tab_ld1, tab_ld2;
  int n_hidden, act, arch;
  const double* hp;   // device: w_std, b_std, last_w_std, ...
  const double* scal; // device scalar block (diagonal shift values)
  int shift;          // enum Shift, applied where global row == global col (symmetric only)
  int symmetric;      // 1: only tiles tj <= ti are computed
  int out_full;       // symmetric only: also store the mirrored element
  double* K;
  long long ldk;
};

struct GemmParams {
  const double* A;    // [M, K] rows
  const double* B;    // [N, K] rows
  double* C;          // [M, N]
  long long lda, ldb, ldc;
  int M, N, K;
  int lower;          // 1: only elements col <= diag_limit(row) are touched (C(0,0) on the diagonal by default)
  // block-row-cyclic generalisation (multi-GPU local update): local row r lives in local block r / cyc_db whose
  // global rows are shifted by (cyc_p - 1) * cyc_db per block; cyc_db == 0 -> plain lower triangle
  int cyc_db, cyc_p, base_shift;
  int sm_reserve;     // persistent kernel leaves this many SMs free (look-ahead work on another stream)
  int k_from_row;     // 1: contraction of the tile whose first row is r0 starts at k = r0 (operands upper triangular)
  int k_upto_col;     // 1: B is lower triangular - the contraction of the tile whose first column is c0 stops at c0 + 64
  // snake (boustrophedon) block distribution: consecutive local blocks are alternately (P - 1 - 2 rank) blocks
  // closer / further apart than P; rows of ODD local blocks (counted from the first row of C) get this extra shift
  int cyc_alt;
  int k_row0;         // with k_from_row: global index of C's first row when C is a row strip of a larger product
};

// largest active column of local row r (rows are non-decreasing in this limit)
__host__ __device__ __forceinline__ long long diag_limit(const GemmParams& p, int r) {
  if (!p.lower) return (1ll << 40);
  if (p.cyc_db == 0) return r;
  const int lb = r / p.cyc_db;
  return (long long)r + p.base_shift + (long long)lb * (p.cyc_p - 1) * p.cyc_db + ((lb & 1) ? p.cyc_alt : 0);
}

// ---- NNGP Gram -------------------------------------------------------------------------------------------
// per-row layer table + final marginal variance (nngp diag) for X [N, D]
cudaError_t launch_qtable(cudaStream_t s, const double* X, long long ldx, int N, int D, int n_hidden, int act,
                          int arch, const double* hp, double* tab, long long tab_ld, double* qfin);
// the same tables from cached input variances q0 [N] (hp == nullptr anywhere in this group: unit scalars)
cudaError_t launch_qtable_from_q(cudaStream_t s, const double* q0, int N, int n_hidden, int act, int arch,
                                 const double* hp, double* tab, long long tab_ld, double* qfin);
// recursion-only pass over a cached base Gram (X.X'^T / D); p describes the output, X1 / X2 / D are ignored
cudaError_t launch_gram_from_base(cudaStream_t s, GramParams p, const double* base, long long ldb);
// scal[SC_TRMEAN], shift table; zeroes the log-det / quad accumulators
cudaError_t launch_scalars(cudaStream_t s, const double* qfin, int N, const double* hp, double* scal);
cudaError_t launch_gram(cudaStream_t s, const GramParams& p);

// ---- Cholesky --------------------------------------------------------------------------------------------
// Factor the w x w (w <= 128) diagonal block at A (row-major, lower) in place, write inv(L) (128x128, ld 128,
// zero above the diagonal, identity padded) to Linv, add sum(log L_ii) to *logdet, record first bad pivot.
cudaError_t launch_potf2_trtri(cudaStream_t s, double* A, long long lda, int w, double* Linv, double* logdet,
                               int* info, int global_col0);
// C = A * B^T (store) or C -= A * B^T (lower-masked when p.lower)
cudaError_t launch_gemm_store(cudaStream_t s, const GemmParams& p);
cudaError_t launch_gemm_sub(cudaStream_t s, const GemmParams& p);
// Blocked right-looking Cholesky of the leading N x N of the row-major trapezoid A [Mtot, N] (lower part);
// rows N..Mtot-1 are carried along and end up as (rows) * L^-T.  NB = outer panel (multiple of 128).
// linv_stride = 0: Linv_ws (128x128) is reused by every inner step; otherwise step k writes Linv_ws + k*linv_stride
// ident_row0 >= 0: rows ident_row0 .. ident_row0 + N - 1 of A start as the identity (the caller wrote it) and end up
// as U = L^-T (upper triangular).  Identity row i stays e_i until the panel that contains column i, so while
// factoring panel [c0, c1) only carried rows below ident_row0 + c1 are touched (N^3/3 flop instead of N^3).
// fused_ws (optional, fused_ws_doubles(Mtot) doubles): enables the single-launch panel solve.  Per outer panel the rows below the diagonal block are then solved OUT OF PLACE into the
// panel buffer (one TMA GEMM with the block's full inverse) and the trailing updates read the panel buffer; carried
// rows (>= N) are copied back into A, the square rows of L only when want_L is set - the fused LML / predictive
// paths never read them.
cudaError_t potrf_trapezoid(cudaStream_t s, double* A, long long lda, long long Mtot, long long N, int NB,
                            double* Linv_ws, double* logdet, int* info, long long linv_stride = 0,
                            long long ident_row0 = -1, double* fused_ws = nullptr, bool want_L = true);
// C = A B^T, lower part only, C does not alias the operands (TMA-fed persistent kernel when the operands allow)
cudaError_t launch_gemm_store_lower(cudaStream_t s, const GemmParams& p);
// C = A B^T out of place on the TMA core (p.lower / p.k_upto_col honoured); cudaErrorInvalidValue if an operand is
// not TMA-addressable (16-byte aligned base, even pitch)
cudaError_t launch_gemm_store_tma(cudaStream_t s, const GemmParams& p);

// ---- full inverse of a panel's diagonal block (trtri.cu) -----------------------------------------------------
struct PeerSignal;
bool assemble_inverse_ok(const double* L, long long ldl, int w, long long ldw);
// W [w, ldw] = inv(L) (lower, zero above the diagonal inside the diagonal blocks) from the factored block L and the
// inverses of its 128 x 128 diagonal blocks; stored to out_ptrs[0 .. P) (peer buffers); sig != nullptr: the last CTA
// raises the flags it describes
cudaError_t launch_assemble_inverse(cudaStream_t s, const double* L, long long ldl, int w, const double* linv_blocks,
                                    double* const* out_ptrs, int P, long long ldw, const PeerSignal* sig);

// doubles of the extra workspace of potrf_trapezoid's single-launch panel solve for a trapezoid of Mtot rows:
// W (512 x 512) + the out-of-place panel buffer (Mtot x 512)
constexpr int FUSED_LD = LINV_BLOCKS * PB;
inline size_t fused_ws_doubles(long long Mtot) { return (size_t)FUSED_LD * FUSED_LD + (size_t)Mtot * FUSED_LD; }

// ---- reductions / closed forms ---------------------------------------------------------------------------
cudaError_t launch_sumsq(cudaStream_t s, const double* z, long long n, double* out);
// out[0] = lml, out[1] = -lml/N (SPR.loss), out[2] = sum log L_ii (of K + shift I), out[3] = ||L^-1 y||^2
cudaError_t launch_lml_finalize(cudaStream_t s, const double* scal, const double* hp, int kind, long long N,
                                const int* info, double* out);
// V [T, ldv] = K_td L^-T rows, Z [C, ldz] = (L^-1 Y)^T rows, ktt [T] prior variances
cudaError_t launch_predict_finalize(cudaStream_t s, const double* V, long long ldv, const double* Z,
                                    long long ldz, const double* ktt, int T, int C, long long N,
                                    const int* info, double* mean, double* var);
// SPR.test_nll tail: per-test log-density and its mean.  scal2 holds ||L2^-1 y||^2 for the Student-t d term.
cudaError_t launch_test_nll_finalize(cudaStream_t s, const double* mean, const double* var, const double* ytest,
                                     int T, long long N, double y_mean, double y_std, const double* hp,
                                     int kind, const double* quad2, const int* info, double* logp,
                                     double* nll_out);
cudaError_t launch_fill_nan_if_bad(cudaStream_t s, const int* info, double* buf, long long n);

// ---- batched grid search (grid_batch.cu) ---------------------------------------------------------------------
constexpr int GRID_BATCH_MAX_N = 4096;
struct GridBatchParams {
  const double *K0dd, *K0td, *q_d, *q_t, *y;   // cached bases (smnngp_grid_base_f64) and the targets
  const double* hp;                            // [G][HP_COUNT]
  long long ld0, ld0t;
  int N, T, G, n_hidden, arch;
  char* ws;                                    // slot k at ws + k * slot_bytes
  long long slot_bytes, lda;                   // lda: row stride of a slot's (N + T + 1)-row trapezoid
  long long off_tab, off_q, off_tab_t, off_q_t;   // layer tables inside a slot (doubles from its start)
  double *mean, *var, *out;                    // [G][T], [G][T], [G][2]
  int* info;                                   // [G]
};
// one persistent launch: min(slots, G) CTAs, each owns one slot and evaluates points blockIdx.x, + gridDim.x, ...
cudaError_t launch_grid_batch(cudaStream_t s, const GridBatchParams& p, int act, long long slots);

// ---- batched loss + gradient (grad_batch.cu) ----------------------------------------------------------------
struct GradBatchParams {
  const double *K0dd, *q_d, *y;                // cached base (smnngp_grid_base_f64, T = 0) and the targets
  const double* hp;                            // [G][HP_COUNT]
  long long ld0;
  int N, G, n_hidden, arch, kind;
  char* ws;                                    // slot k at ws + k * slot_bytes
  long long slot_bytes, lda;                   // lda: row stride of a slot's (2N + 1)-row trapezoid
  long long off_tab3, off_alpha;               // dual tables [3][n_act][N] and A^-1 y inside a slot (doubles)
  double *out, *grad;                          // [G][4], [G][6]
  int* info;                                   // [G]
};
// one persistent launch: min(slots, G) CTAs, each owns one slot and evaluates points blockIdx.x, + gridDim.x, ...
cudaError_t launch_lml_grad_batch(cudaStream_t s, const GradBatchParams& p, int act, long long slots);

// ---- batched test NLL (test_nll_batch.cu) --------------------------------------------------------------------
struct TestNllBatchParams {
  const double *K0dd, *K0td, *q_d, *q_t, *y;   // cached bases (smnngp_grid_base_f64) and the targets
  const double* yt;                            // [T] standardised test targets
  const double* hp;                            // [G][HP_COUNT]
  long long ld0, ld0t;
  int N, T, G, n_hidden, arch, kind;
  double y_mean, y_std;
  char* ws;                                    // slot k at ws + k * slot_bytes
  long long slot_bytes, lda;                   // lda: row stride of a slot's (N + T + 1)-row trapezoid
  long long off_tab, off_q, off_tab_t, off_q_t, off_mv;   // layer tables, [2][T] mean / var inside a slot (doubles)
  double* nll;                                 // [G]
  double *mean, *var, *logp;                   // [G][T] each, may be null
  int* info;                                   // [G]
};
// one persistent launch: min(slots, G) CTAs, each owns one slot and evaluates points blockIdx.x, + gridDim.x, ...
cudaError_t launch_test_nll_batch(cudaStream_t s, const TestNllBatchParams& p, int act, long long slots);

// ---- posterior draw stage (draws.cu) -------------------------------------------------------------------------
constexpr int DRAW_MAXC = 16;   // classes draw_metrics keeps in registers
// out [C, T, S] <- mean [T, C] + sigma [C, T] * variate, one counter-based Philox stream per (s, t, c)
cudaError_t launch_sample_f_iid(cudaStream_t s, const double* mean, const double* var, int var_per_class, int T, int C,
                                int S, const double* hp, int kind, uint64_t seed, double* out);
// the same draws, reduced to ll_per_test [T], pred [T] and out [2] = { nll, correct count }; C <= DRAW_MAXC
cudaError_t launch_draw_metrics(cudaStream_t s, const double* mean, const double* var, int var_per_class,
                                const int* label, int T, int C, int S, const double* hp, int kind, uint64_t seed,
                                double* ll_per_test, int* pred, double* out);

// ---- scale mixture by importance sampling (mixture.cu) --------------------------------------------------------
enum ScaleFamily { SCALE_INVGAMMA = 0, SCALE_BURR12 = 1 };
// draws [P][S] of the scale prior of row p (params [P][2]: (a, b) or (c, k)); counter (j, p, 0xFFFFFFFF, n)
cudaError_t launch_scale_draws(cudaStream_t s, int family, const double* params, long long P, long long S,
                               uint64_t seed, double* out);
struct MixtureParams {
  const double* scal;                          // [G][2] {sum log L_ii, y^T A^-1 y}
  const double *mean, *var;                    // [G][ld] predictive (standardised units); null when T = 0
  const double* yt;                            // [T] standardised test targets
  const double* draws;                         // [P][S]
  long long N, T, G, P, S, ld;
  double y_mean, y_std;
  double *nll, *lml, *ess;                     // [G][P]; nll may be null when T = 0
  double* logp;                                // [G][P][T] or null
};
// one launch, a warp per (g, p) pair; a pair's outputs depend only on its rows and the scalars
cudaError_t launch_mixture_nll(cudaStream_t s, const MixtureParams& p);

// ---- gradient of the log marginal likelihood (grad.cu) -------------------------------------------------------
// tab3 [3][n_act][tab_ld]: encoded marginal variances + the two dual planes the gradient epilogue needs
cudaError_t launch_qtable_dual(cudaStream_t s, const double* X, long long ldx, int N, int D, int n_hidden, int act,
                               int arch, const double* hp, double* tab3, long long tab_ld);
// A [N, lda] <- identity (zero fill + ones)
cudaError_t launch_set_identity(cudaStream_t s, double* A, long long lda, long long N);
// A[i, i] = 1 for i < N (no zero fill)
cudaError_t launch_set_ones_diag(cudaStream_t s, double* A, long long lda, long long N);
// out_i = sum_{k >= i} U[i,k] z[k]
cudaError_t launch_upper_gemv(cudaStream_t s, const double* U, long long ldu, const double* z, long long N,
                              double* out);
long long grad_partial_slots(long long N);
// partial[slots][4] = per-warp sums of G_ij dK_ij/d(w_std, b_std, last_w_std) and tr G over the lower triangle
cudaError_t launch_grad_gram(cudaStream_t s, const double* X, long long N, long long D, int n_hidden, int act,
                             int arch, const double* hp, const double* tab3, long long tab_ld, const double* Winv,
                             long long ldw, const double* alpha, const double* quad, int kind, double* partial,
                             long long slots);
// the same contraction restricted to the row strip [row0, row0 + rows) x [0, row0 + rows) of the lower triangle
// (multi-GPU gradient: every rank takes one strip): Winv [rows, ldw] = that strip of A^-1, everything else global
cudaError_t launch_grad_gram_strip(cudaStream_t s, const double* X, long long N, long long D, long long row0,
                                   long long rows, int n_hidden, int act, int arch, const double* hp, const double* tab3,
                                   long long tab_ld, const double* Winv_strip, long long ldw, const double* alpha,
                                   const double* quad, int kind, double* partial, long long slots);
// out4 = fixed-order sum of partial [slots][4]
cudaError_t launch_sum_slots(cudaStream_t s, const double* partial, long long slots, double* out4);
cudaError_t launch_grad_finalize(cudaStream_t s, const double* partial, long long slots, const double* hp,
                                 const double* quad, int kind, long long N, const int* info, double* grad);

// ---- instrumentation (bench.py): kernel-launch counter and CUDA-event timing of the trailing updates -------
struct Instrumentation {
  long long launches = 0;          // kernels of this library enqueued since the last reset
  bool time_updates = false;       // record an event pair around every outer trailing update
  double update_flops = 0.0;       // algorithmic flops of the timed trailing updates (executed lower tiles)
  double update_alg_flops = 0.0;   // m*(n)*k style algorithmic count (lower triangle only, 2 flop / MAC)
};
Instrumentation& instr();
void instr_begin_update(cudaStream_t s, double alg_flops);
void instr_end_update(cudaStream_t s);
// returns total milliseconds of the recorded trailing updates (synchronises on the events), count via n_out
double instr_collect_update_ms(int* n_out);
void instr_reset();
// register-resident DMMA.8x8x4 issue-rate probe: returns TFLOP/s (synchronous; measurement tool)
double dmma_peak_tflops(int device_sms);

}  // namespace smnngp

// extern "C" boundary of libsmnngp (declared in include/smnngp.h).  Host-side orchestration only: carve the
// caller's workspace, enqueue the kernels of gram.cu / chol.cu / reduce.cu on the caller's stream.
#include "../../include/smnngp.h"

#include <cstdio>
#include <cstring>
#include <string>

#include "context.cuh"
#include "kernels.cuh"

using namespace smnngp;

namespace {

thread_local std::string g_err;

int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
  char buf[512];
  if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
  else snprintf(buf, sizeof buf, "%s", what);
  g_err = buf;
  return code;
}
#define CU(call)                                                       \
  do {                                                                 \
    cudaError_t e__ = (call);                                          \
    if (e__ != cudaSuccess) return fail(SMNNGP_ECUDA, #call, e__);     \
  } while (0)

// bump allocator over the caller's workspace; base == nullptr only measures
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<char*>(b)) {}
  template <typename T>
  T* take(size_t count) {
    off = (off + 255) & ~size_t(255);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
  size_t total() const { return (off + 255) & ~size_t(255); }
};

inline long long round_up(long long x, long long m) { return (x + m - 1) / m * m; }

int pick_nb(long long N) {
  const int pw = dctx().panel_width;
  if (pw > 0) return pw;
  if (N >= 8192) return 512;
  if (N >= 2048) return 256;
  return 128;
}

bool valid_stack(int n_hidden, int act, int arch) {
  return n_hidden >= 0 && n_hidden <= 64 && (act == ACT_RELU || act == ACT_ERF) &&
         (arch == ARCH_MLP || arch == ARCH_RESNET);
}

__global__ void transpose_rows_kernel(const double* __restrict__ Y, long long N, int C, double* __restrict__ out,
                                      long long ldo) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * C) return;
  long long n = i / C;
  int c = (int)(i % C);
  out[(long long)c * ldo + n] = Y[i];
}

// ---- workspace layouts ----------------------------------------------------------------------------------
struct GramWs { double *tab1, *tab2, *q1, *q2, *scal; };
size_t carve_gram(Carver& c, GramWs& w, long long N, long long M, int n_act, bool cross) {
  w.scal = c.take<double>(SC_COUNT);
  w.tab1 = c.take<double>((size_t)(n_act > 0 ? n_act : 1) * N);
  w.q1 = c.take<double>(N);
  w.tab2 = cross ? c.take<double>((size_t)(n_act > 0 ? n_act : 1) * M) : w.tab1;
  w.q2 = cross ? c.take<double>(M) : w.q1;
  return c.total();
}

struct SolveWs {
  double *scal, *scal2, *tab, *q, *tab_t, *q_t, *linv, *A, *mean, *var, *fws;
  long long lda, rows;
};
// A holds N train rows + T cross-Gram rows + C right-hand-side rows
size_t carve_solve(Carver& c, SolveWs& w, long long N, long long T, long long C, int n_act) {
  const size_t na = (size_t)(n_act > 0 ? n_act : 1);
  w.scal = c.take<double>(SC_COUNT);
  w.scal2 = c.take<double>(SC_COUNT);
  w.tab = c.take<double>(na * N);
  w.q = c.take<double>(N);
  w.tab_t = c.take<double>(na * (T > 0 ? T : 1));
  w.q_t = c.take<double>(T > 0 ? T : 1);
  w.linv = c.take<double>(LINV_BLOCKS * PB * PB);
  w.mean = c.take<double>((size_t)(T > 0 ? T : 1) * (C > 0 ? C : 1));
  w.var = c.take<double>(T > 0 ? T : 1);
  w.lda = round_up(N, 16);
  w.rows = N + T + C;
  w.A = c.take<double>((size_t)w.rows * w.lda);
  w.fws = c.take<double>(fused_ws_doubles(w.rows));          // W + panel buffer of the single-launch panel solve
  return c.total();
}

cudaError_t enqueue_sym_gram(cudaStream_t s, const double* X, long long N, long long D, int n_hidden, int act,
                             int arch, const double* hp, const double* tab, const double* scal, int shift,
                             int out_full, double* K, long long ldk) {
  GramParams g{};
  g.X1 = X; g.X2 = X; g.ld1 = D; g.ld2 = D; g.N = (int)N; g.M = (int)N; g.D = (int)D;
  g.tab1 = tab; g.tab2 = tab; g.tab_ld1 = N; g.tab_ld2 = N;
  g.n_hidden = n_hidden; g.act = act; g.arch = arch; g.hp = hp; g.scal = scal; g.shift = shift;
  g.symmetric = 1; g.out_full = out_full; g.K = K; g.ldk = ldk;
  return launch_gram(s, g);
}

cudaError_t enqueue_cross_gram(cudaStream_t s, const double* X1, long long N, const double* X2, long long M,
                               long long D, int n_hidden, int act, int arch, const double* hp, const double* tab1,
                               const double* tab2, const double* scal, double* K, long long ldk) {
  GramParams g{};
  g.X1 = X1; g.X2 = X2; g.ld1 = D; g.ld2 = D; g.N = (int)N; g.M = (int)M; g.D = (int)D;
  g.tab1 = tab1; g.tab2 = tab2; g.tab_ld1 = N; g.tab_ld2 = M;
  g.n_hidden = n_hidden; g.act = act; g.arch = arch; g.hp = hp; g.scal = scal; g.shift = SHIFT_NONE;
  g.symmetric = 0; g.out_full = 1; g.K = K; g.ldk = ldk;
  return launch_gram(s, g);
}

// grow-only device arena of the *_host_f64 entry points: owned by the device context (context.cuh)
int arena_reserve(DeviceCtx& c, size_t bytes) {
  if (!c.arena_stream) CU(cudaStreamCreateWithFlags(&c.arena_stream, cudaStreamNonBlocking));
  if (bytes <= c.arena_bytes) return SMNNGP_OK;
  if (c.arena) CU(cudaFree(c.arena));
  c.arena = nullptr;
  c.arena_bytes = 0;
  CU(cudaMalloc(&c.arena, bytes));
  c.arena_bytes = bytes;
  return SMNNGP_OK;
}

}  // namespace

extern "C" {

int smnngp_abi_version(void) { return SMNNGP_ABI_VERSION; }
const char* smnngp_last_error(void) { return g_err.c_str(); }
void smnngp_set_panel_width(int nb) { dctx().panel_width = nb > 0 ? (nb + PB - 1) / PB * PB : 0; }

void smnngp_set_tile_variant(int v) { tile_variant() = (v >= 0 && v <= 2) ? v : 0; }
int smnngp_debug_occupancy(int variant) { return debug_gemm_occupancy(variant); }
void smnngp_set_lookahead(int on) { lookahead_mode() = on ? 1 : 0; }
// 1 (default): single-launch panel solve with the diagonal block's full inverse; 0: 128-block substitution in place
void smnngp_set_fused_panel(int on) { dctx().fused_panel = on ? 1 : 0; }
// the look-ahead factorisation (N >= 8192) hands its last <= cols columns to the single-stream 128-column path; 0: never
void smnngp_set_tail_cols(int64_t cols) { dctx().tail_cols = cols < 0 ? 0 : cols; }
// super-tile height (128-row tiles) of the Gram kernel's L2-aware tile walk; 0 = row-major walk (round-1 behaviour)
void smnngp_set_gram_super_rows(int sr, int64_t min_operand_bytes) {
  dctx().gram_super = sr < 0 ? 0 : (sr > 64 ? 64 : sr);
  dctx().gram_super_min_bytes = min_operand_bytes < 0 ? 40000000 : min_operand_bytes;
}
void smnngp_set_lookahead_reserve(int small_trailing, int large_trailing) {
  lookahead_reserve()[0] = small_trailing < 0 ? 0 : small_trailing;
  lookahead_reserve()[1] = large_trailing < 0 ? 0 : large_trailing;
}
void smnngp_debug_potf2_clocks(long long* dev_buf) { potf2_clock_buffer() = dev_buf; }

// ---- instrumentation for bench.py ------------------------------------------------------------------------
void smnngp_instr_reset(int time_updates) {
  instr_reset();
  instr().time_updates = time_updates != 0;
}
long long smnngp_instr_launches(void) { return instr().launches; }
int smnngp_instr_updates(double* total_ms, double* alg_flops) {
  int n = 0;
  double ms = instr_collect_update_ms(&n);
  if (total_ms) *total_ms = ms;
  if (alg_flops) *alg_flops = instr().update_alg_flops;
  return n;
}
double smnngp_dmma_peak_tflops(void) {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1.0;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1.0;
  return dmma_peak_tflops(sms);
}

// ---------------------------------------------------------------------------------------------------------
size_t smnngp_gram_workspace_bytes(int64_t N, int64_t M, int n_hidden, int arch) {
  Carver c(nullptr);
  GramWs w;
  return carve_gram(c, w, N, M, n_act_applications(n_hidden, arch), true);
}

int smnngp_gram_f64(void* stream, const double* X, const double* X2, int64_t N, int64_t M, int64_t D,
                    int n_hidden, int act, int arch, const double* hp_dev, int shift, int out_mode,
                    double* K_out, int64_t ld, void* workspace, size_t workspace_bytes) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  const bool sym = (X2 == nullptr || X2 == X);
  if (sym) M = N;
  if (!X || !K_out || !hp_dev || N < 0 || M < 0 || D <= 0 || ld < M || !valid_stack(n_hidden, act, arch) ||
      shift < 0 || shift > 3 || N > INT32_MAX || M > INT32_MAX || D > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_gram_f64: invalid argument");
  if (N == 0 || M == 0) return SMNNGP_OK;
  const int n_act = n_act_applications(n_hidden, arch);
  Carver c(workspace);
  GramWs w;
  if (carve_gram(c, w, N, M, n_act, !sym) > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_gram_f64: workspace too small");
  CU(launch_qtable(s, X, D, (int)N, (int)D, n_hidden, act, arch, hp_dev, w.tab1, N, w.q1));
  CU(launch_scalars(s, w.q1, (int)N, hp_dev, w.scal));
  if (sym) {
    CU(enqueue_sym_gram(s, X, N, D, n_hidden, act, arch, hp_dev, w.tab1, w.scal, shift,
                        out_mode == SMNNGP_OUT_FULL, K_out, ld));
  } else {
    CU(launch_qtable(s, X2, D, (int)M, (int)D, n_hidden, act, arch, hp_dev, w.tab2, M, w.q2));
    CU(enqueue_cross_gram(s, X, N, X2, M, D, n_hidden, act, arch, hp_dev, w.tab1, w.tab2, w.scal, K_out, ld));
  }
  return SMNNGP_OK;
}

int smnngp_nngp_diag_f64(void* stream, const double* X, int64_t N, int64_t D, int n_hidden, int act, int arch,
                         const double* hp_dev, double* q_out, void* workspace, size_t workspace_bytes) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!X || !q_out || !hp_dev || N < 0 || D <= 0 || !valid_stack(n_hidden, act, arch) || N > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_nngp_diag_f64: invalid argument");
  if (N == 0) return SMNNGP_OK;
  const int n_act = n_act_applications(n_hidden, arch);
  Carver c(workspace);
  GramWs w;
  if (carve_gram(c, w, N, N, n_act, false) > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_nngp_diag_f64: workspace too small");
  CU(launch_qtable(s, X, D, (int)N, (int)D, n_hidden, act, arch, hp_dev, w.tab1, N, q_out));
  return SMNNGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
size_t smnngp_potrf_workspace_bytes(int64_t N) {
  // sized for the square case; a trapezoid with M > N rows falls back to the in-place panel solve when the panel
  // buffer does not fit (see smnngp_potrf_trapezoid_f64)
  Carver c(nullptr);
  c.take<double>(SC_COUNT);
  c.take<double>(LINV_BLOCKS * PB * PB);
  c.take<double>(fused_ws_doubles(N > 0 ? N : 0));
  return c.total();
}

int smnngp_potrf_trapezoid_f64(void* stream, double* A, int64_t M, int64_t N, int64_t ld, double* logdet_dev,
                               int* info_dev, void* workspace, size_t workspace_bytes) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!A || N < 0 || M < N || ld < N || !info_dev || M > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_potrf_trapezoid_f64: invalid argument");
  Carver c(workspace);
  double* scal = c.take<double>(SC_COUNT);
  double* linv = c.take<double>(LINV_BLOCKS * PB * PB);
  if (c.total() > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_potrf_trapezoid_f64: workspace too small");
  double* fws = c.take<double>(fused_ws_doubles(M));           // optional: enables the single-launch panel solve
  if (c.total() > workspace_bytes) fws = nullptr;
  CU(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
  CU(cudaMemsetAsync(scal, 0, SC_COUNT * sizeof(double), s));
  if (N == 0) return SMNNGP_OK;
  CU(potrf_trapezoid(s, A, ld, M, N, pick_nb(N), linv, scal + SC_LOGDET, info_dev, 0, -1, fws, true));
  if (logdet_dev) CU(cudaMemcpyAsync(logdet_dev, scal + SC_LOGDET, sizeof(double), cudaMemcpyDeviceToDevice, s));
  return SMNNGP_OK;
}

int smnngp_potrf_f64(void* stream, double* A, int64_t N, int64_t ld, int* info_dev, void* workspace,
                     size_t workspace_bytes) {
  return smnngp_potrf_trapezoid_f64(stream, A, N, N, ld, nullptr, info_dev, workspace, workspace_bytes);
}


// ---------------------------------------------------------------------------------------------------------
// generic covariance solve: factor (scale * cov + shift I) without touching `cov`, return
// out_dev[2] = { sum_i log L_ii, ||L^-1 y||^2 }.  Backs Likelihood.prior_logpdf(y, cov)
// (spax/likelihoods.py:25-28, :45-50) and the d term of StudentTLikelihood.logpdf (:60-61) when the caller
// hands over an explicit covariance matrix instead of using the fused entry points.
size_t smnngp_cov_solve_workspace_bytes(int64_t N) {
  Carver c(nullptr);
  c.take<double>(SC_COUNT);
  c.take<double>(LINV_BLOCKS * PB * PB);
  c.take<double>((size_t)(N + 1) * round_up(N, 16));
  c.take<double>(fused_ws_doubles(N + 1));
  return c.total();
}

__global__ void scale_shift_copy_kernel(const double* __restrict__ src, long long lds, double* __restrict__ dst,
                                        long long ldd, long long N, double scale, double shift) {
  long long r = blockIdx.y;
  for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c <= r; c += (long long)gridDim.x * blockDim.x) {
    double v = scale * src[r * lds + c];
    if (c == r) v += shift;
    dst[r * ldd + c] = v;
  }
}

int smnngp_cov_solve_f64(void* stream, const double* cov, int64_t N, int64_t ld, const double* y, double scale,
                         double shift, void* workspace, size_t workspace_bytes, double* out_dev, int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!cov || !y || !out_dev || !info_dev || N <= 0 || ld < N || N + 1 > 65535)
    return fail(SMNNGP_EINVAL, "smnngp_cov_solve_f64: invalid argument (N must be < 65535 on this entry point)");
  Carver c(workspace);
  double* scal = c.take<double>(SC_COUNT);
  double* linv = c.take<double>(LINV_BLOCKS * PB * PB);
  const long long lda = round_up(N, 16);
  double* A = c.take<double>((size_t)(N + 1) * lda);
  double* fws = c.take<double>(fused_ws_doubles(N + 1));
  if (c.total() > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_cov_solve_f64: workspace too small");
  CU(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
  CU(cudaMemsetAsync(scal, 0, SC_COUNT * sizeof(double), s));
  dim3 grid((unsigned)((N + 255) / 256 < 64 ? (N + 255) / 256 : 64), (unsigned)N);
  scale_shift_copy_kernel<<<grid, 256, 0, s>>>(cov, ld, A, lda, N, scale, shift);
  instr().launches++;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(A + N * lda, y, N * sizeof(double), cudaMemcpyDeviceToDevice, s));
  CU(potrf_trapezoid(s, A, lda, N + 1, N, pick_nb(N), linv, scal + SC_LOGDET, info_dev, 0, -1, fws, false));
  CU(launch_sumsq(s, A + N * lda, N, scal + SC_QUAD));
  CU(cudaMemcpyAsync(out_dev, scal + SC_LOGDET, 2 * sizeof(double), cudaMemcpyDeviceToDevice, s));
  CU(launch_fill_nan_if_bad(s, info_dev, out_dev, 2));
  return SMNNGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
size_t smnngp_lml_workspace_bytes(int64_t N, int64_t D, int n_hidden, int arch) {
  (void)D;
  Carver c(nullptr);
  SolveWs w;
  return carve_solve(c, w, N, 0, 1, n_act_applications(n_hidden, arch));
}

int smnngp_lml_f64(void* stream, const double* X, const double* y, int64_t N, int64_t D, int n_hidden, int act,
                   int arch, const double* hp_dev, int kind, void* workspace, size_t workspace_bytes,
                   double* out_dev, int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!X || !y || !hp_dev || !out_dev || !info_dev || N <= 0 || D <= 0 || !valid_stack(n_hidden, act, arch) ||
      (kind != KIND_GAUSS && kind != KIND_STUDENT_T) || N + 1 > INT32_MAX || D > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_lml_f64: invalid argument");
  const int n_act = n_act_applications(n_hidden, arch);
  Carver c(workspace);
  SolveWs w;
  if (carve_solve(c, w, N, 0, 1, n_act) > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_lml_f64: workspace too small");
  CU(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
  CU(launch_qtable(s, X, D, (int)N, (int)D, n_hidden, act, arch, hp_dev, w.tab, N, w.q));
  CU(launch_scalars(s, w.q, (int)N, hp_dev, w.scal));
  // K + eps I, lower triangle only, straight into the factorisation buffer (spax/models.py:96)
  CU(enqueue_sym_gram(s, X, N, D, n_hidden, act, arch, hp_dev, w.tab, w.scal, SHIFT_EPS_ABS, 0, w.A, w.lda));
  // y^T appended as row N: the factorisation turns it into (L^-1 y)^T (spax/utils.py:180)
  CU(cudaMemcpyAsync(w.A + N * w.lda, y, N * sizeof(double), cudaMemcpyDeviceToDevice, s));
  CU(potrf_trapezoid(s, w.A, w.lda, N + 1, N, pick_nb(N), w.linv, w.scal + SC_LOGDET, info_dev, 0, -1, w.fws, false));
  CU(launch_sumsq(s, w.A + N * w.lda, N, w.scal + SC_QUAD));
  CU(launch_lml_finalize(s, w.scal, hp_dev, kind, N, info_dev, out_dev));
  return SMNNGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// loss and its gradient w.r.t. the six scalars (SURVEY section 8f, row N1)
namespace {
struct GradWs {
  double *scal, *tab, *q, *tab3, *linv, *alpha, *partial, *A, *fws;
  long long lda, slots;
};
size_t carve_grad(Carver& c, GradWs& w, long long N, int n_act) {
  const size_t na = (size_t)(n_act > 0 ? n_act : 1);
  w.scal = c.take<double>(SC_COUNT);
  w.tab = c.take<double>(na * N);
  w.q = c.take<double>(N);
  w.tab3 = c.take<double>(3 * na * N);
  w.linv = c.take<double>(LINV_BLOCKS * PB * PB);
  w.alpha = c.take<double>(N);
  w.slots = grad_partial_slots(N);
  w.partial = c.take<double>((size_t)w.slots * 4);
  w.lda = round_up(N, 16);
  w.A = c.take<double>((size_t)(2 * N + 1) * w.lda);   // K -> L -> A^-1 | y^T -> z^T | I -> U = L^-T
  w.fws = c.take<double>(fused_ws_doubles(2 * N + 1));
  return c.total();
}
}  // namespace

size_t smnngp_lml_grad_workspace_bytes(int64_t N, int64_t D, int n_hidden, int arch) {
  (void)D;
  Carver c(nullptr);
  GradWs w;
  return carve_grad(c, w, N, n_act_applications(n_hidden, arch));
}

int smnngp_lml_grad_f64(void* stream, const double* X, const double* y, int64_t N, int64_t D, int n_hidden, int act,
                        int arch, const double* hp_dev, int kind, void* workspace, size_t workspace_bytes,
                        double* out_dev, double* grad_dev, int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!X || !y || !hp_dev || !out_dev || !grad_dev || !info_dev || N <= 0 || D <= 0 ||
      !valid_stack(n_hidden, act, arch) || (kind != KIND_GAUSS && kind != KIND_STUDENT_T) ||
      2 * N + 1 > INT32_MAX || D > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_lml_grad_f64: invalid argument");
  const int n_act = n_act_applications(n_hidden, arch);
  Carver c(workspace);
  GradWs w;
  if (carve_grad(c, w, N, n_act) > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_lml_grad_f64: workspace too small");
  double* zrow = w.A + N * w.lda;
  double* U = w.A + (N + 1) * w.lda;
  CU(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
  CU(launch_qtable(s, X, D, (int)N, (int)D, n_hidden, act, arch, hp_dev, w.tab, N, w.q));
  CU(launch_scalars(s, w.q, (int)N, hp_dev, w.scal));
  CU(launch_qtable_dual(s, X, D, (int)N, (int)D, n_hidden, act, arch, hp_dev, w.tab3, N));
  CU(enqueue_sym_gram(s, X, N, D, n_hidden, act, arch, hp_dev, w.tab, w.scal, SHIFT_EPS_ABS, 0, w.A, w.lda));
  CU(cudaMemcpyAsync(zrow, y, N * sizeof(double), cudaMemcpyDeviceToDevice, s));
  CU(launch_set_identity(s, U, w.lda, N));
  // forward value exactly as smnngp_lml_f64; the identity rows come out as U = L^-T
  CU(potrf_trapezoid(s, w.A, w.lda, 2 * N + 1, N, pick_nb(N), w.linv, w.scal + SC_LOGDET, info_dev, 0, N + 1, w.fws, false));
  CU(launch_sumsq(s, zrow, N, w.scal + SC_QUAD));
  CU(launch_lml_finalize(s, w.scal, hp_dev, kind, N, info_dev, out_dev));
  // a = A^-1 y = U z;  A^-1 = U U^T over the (now free) lower triangle of the factor
  CU(launch_upper_gemv(s, U, w.lda, zrow, N, w.alpha));
  {
    GemmParams g{};
    g.A = U; g.lda = w.lda;
    g.B = U; g.ldb = w.lda;
    g.C = w.A; g.ldc = w.lda;
    g.M = (int)N; g.N = (int)N; g.K = (int)N; g.lower = 1; g.k_from_row = 1;
    CU(launch_gemm_store_lower(s, g));
  }
  CU(launch_grad_gram(s, X, N, D, n_hidden, act, arch, hp_dev, w.tab3, N, w.A, w.lda, w.alpha, w.scal + SC_QUAD,
                      kind, w.partial, w.slots));
  CU(launch_grad_finalize(s, w.partial, w.slots, hp_dev, w.scal + SC_QUAD, kind, N, info_dev, grad_dev));
  return SMNNGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
size_t smnngp_predict_workspace_bytes(int64_t N, int64_t T, int64_t C, int64_t D, int n_hidden, int arch) {
  (void)D;
  Carver c(nullptr);
  SolveWs w;
  return carve_solve(c, w, N, T, C < 1 ? 1 : C, n_act_applications(n_hidden, arch));
}

static int predict_enqueue(cudaStream_t s, const double* X, const double* Y, const double* Xt, int64_t N,
                           int64_t T, int64_t C, int64_t D, int n_hidden, int act, int arch,
                           const double* hp_dev, int shift, SolveWs& w, double* mean_out, double* var_out,
                           int* info_dev, double* cov_out = nullptr, int64_t ld_cov = 0) {
  CU(launch_qtable(s, X, D, (int)N, (int)D, n_hidden, act, arch, hp_dev, w.tab, N, w.q));
  CU(launch_scalars(s, w.q, (int)N, hp_dev, w.scal));
  CU(launch_qtable(s, Xt, D, (int)T, (int)D, n_hidden, act, arch, hp_dev, w.tab_t, T, w.q_t));
  CU(enqueue_sym_gram(s, X, N, D, n_hidden, act, arch, hp_dev, w.tab, w.scal, shift, 0, w.A, w.lda));
  CU(enqueue_cross_gram(s, Xt, T, X, N, D, n_hidden, act, arch, hp_dev, w.tab_t, w.tab, w.scal,
                        w.A + N * w.lda, w.lda));
  {
    long long total = N * C;
    transpose_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(Y, N, (int)C, w.A + (N + T) * w.lda,
                                                                           w.lda);
    instr().launches++;
    CU(cudaGetLastError());
  }
  CU(potrf_trapezoid(s, w.A, w.lda, N + T + C, N, pick_nb(N), w.linv, w.scal + SC_LOGDET, info_dev, 0, -1, w.fws, false));
  CU(launch_predict_finalize(s, w.A + N * w.lda, w.lda, w.A + (N + T) * w.lda, w.lda, w.q_t, (int)T, (int)C, N,
                             info_dev, mean_out, var_out));
  if (cov_out) {
    // full posterior covariance K_tt - V V^T (what neural_tangents returns with compute_cov=True): Gram of the
    // test points, then one rank-N update with the carried rows V = K_td L^-T on the same GEMM core
    CU(enqueue_sym_gram(s, Xt, T, D, n_hidden, act, arch, hp_dev, w.tab_t, w.scal, SHIFT_NONE, 1, cov_out, ld_cov));
    GemmParams u{};
    u.A = w.A + N * w.lda; u.lda = w.lda;
    u.B = w.A + N * w.lda; u.ldb = w.lda;
    u.C = cov_out; u.ldc = ld_cov;
    u.M = (int)T; u.N = (int)T; u.K = (int)N; u.lower = 0;
    CU(launch_gemm_sub(s, u));
    CU(launch_fill_nan_if_bad(s, info_dev, cov_out, T * ld_cov));
  }
  return SMNNGP_OK;
}

int smnngp_predict_f64(void* stream, const double* X, const double* Y, const double* Xt, int64_t N, int64_t T,
                       int64_t C, int64_t D, int n_hidden, int act, int arch, const double* hp_dev, int shift,
                       void* workspace, size_t workspace_bytes, double* mean_out, double* var_out,
                       int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!X || !Y || !Xt || !hp_dev || !mean_out || !var_out || !info_dev || N <= 0 || T <= 0 || C <= 0 || D <= 0 ||
      !valid_stack(n_hidden, act, arch) || shift < 0 || shift > 3 || N + T + C > INT32_MAX || D > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_predict_f64: invalid argument");
  Carver c(workspace);
  SolveWs w;
  if (carve_solve(c, w, N, T, C, n_act_applications(n_hidden, arch)) > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_predict_f64: workspace too small");
  CU(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
  return predict_enqueue(s, X, Y, Xt, N, T, C, D, n_hidden, act, arch, hp_dev, shift, w, mean_out, var_out,
                         info_dev);
}

int smnngp_predict_cov_f64(void* stream, const double* X, const double* Y, const double* Xt, int64_t N, int64_t T,
                           int64_t C, int64_t D, int n_hidden, int act, int arch, const double* hp_dev, int shift,
                           void* workspace, size_t workspace_bytes, double* mean_out, double* var_out,
                           double* cov_out, int64_t ld_cov, int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!X || !Y || !Xt || !hp_dev || !mean_out || !var_out || !cov_out || !info_dev || N <= 0 || T <= 0 || C <= 0 ||
      D <= 0 || ld_cov < T || !valid_stack(n_hidden, act, arch) || shift < 0 || shift > 3 ||
      N + T + C > INT32_MAX || D > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_predict_cov_f64: invalid argument");
  Carver c(workspace);
  SolveWs w;
  if (carve_solve(c, w, N, T, C, n_act_applications(n_hidden, arch)) > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_predict_cov_f64: workspace too small");
  CU(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
  return predict_enqueue(s, X, Y, Xt, N, T, C, D, n_hidden, act, arch, hp_dev, shift, w, mean_out, var_out,
                         info_dev, cov_out, ld_cov);
}

int smnngp_test_nll_f64(void* stream, const double* X, const double* y, const double* Xt, const double* yt,
                        int64_t N, int64_t T, int64_t D, int n_hidden, int act, int arch, const double* hp_dev,
                        int kind, double y_mean, double y_std, void* workspace, size_t workspace_bytes,
                        double* nll_out_dev, double* mean_out, double* var_out, double* logp_out,
                        int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!X || !y || !Xt || !yt || !hp_dev || !nll_out_dev || !info_dev || N <= 0 || T <= 0 || D <= 0 ||
      !valid_stack(n_hidden, act, arch) || (kind != KIND_GAUSS && kind != KIND_STUDENT_T) ||
      N + T + 1 > INT32_MAX || D > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_test_nll_f64: invalid argument");
  Carver c(workspace);
  SolveWs w;
  if (carve_solve(c, w, N, T, 1, n_act_applications(n_hidden, arch)) > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_test_nll_f64: workspace too small");
  double* mean = mean_out ? mean_out : w.mean;
  double* var = var_out ? var_out : w.var;
  CU(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
  // (1) kernel.predict with the RELATIVE regulariser eps tr(K)/N  (spax/models.py:103)
  int rc = predict_enqueue(s, X, y, Xt, N, T, 1, D, n_hidden, act, arch, hp_dev, SHIFT_EPS_REL, w, mean, var,
                           info_dev);
  if (rc != SMNNGP_OK) return rc;
  // (2) Student-t scale d = 2a + y^T ((b/a) K + 1e-6 I)^-1 y  (spax/likelihoods.py:60-61): second
  //     factorisation with the absolute shift 1e-6 a/b, re-using the same buffer (stream ordered)
  if (kind == KIND_STUDENT_T) {
    CU(enqueue_sym_gram(s, X, N, D, n_hidden, act, arch, hp_dev, w.tab, w.scal, SHIFT_LIK, 0, w.A, w.lda));
    CU(cudaMemcpyAsync(w.A + N * w.lda, y, N * sizeof(double), cudaMemcpyDeviceToDevice, s));
    CU(cudaMemsetAsync(w.scal2, 0, SC_COUNT * sizeof(double), s));
    CU(potrf_trapezoid(s, w.A, w.lda, N + 1, N, pick_nb(N), w.linv, w.scal2 + SC_LOGDET, info_dev, 0, -1, w.fws, false));
    CU(launch_sumsq(s, w.A + N * w.lda, N, w.scal2 + SC_QUAD));
  }
  CU(launch_test_nll_finalize(s, mean, var, yt, (int)T, N, y_mean, y_std, hp_dev, kind, w.scal2 + SC_QUAD,
                              info_dev, logp_out, nll_out_dev));
  return SMNNGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// hyper-parameter grid search with a cached base Gram (SURVEY section 8f, row N3; experiments/regression/find.py)
// ---------------------------------------------------------------------------------------------------------
int smnngp_grid_base_f64(void* stream, const double* X, const double* Xt, int64_t N, int64_t T, int64_t D,
                         double* K0dd, int64_t ld0, double* K0td, int64_t ld0t, double* q_d, double* q_t) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!X || !K0dd || !q_d || N <= 0 || D <= 0 || ld0 < N || T < 0 || (T > 0 && (!Xt || !K0td || !q_t || ld0t < N)) ||
      N > INT32_MAX || T > INT32_MAX || D > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_grid_base_f64: invalid argument");
  // unit scalars (hp = nullptr), no hidden layer: K0 = X X'^T / D and q0 = ||x||^2 / D
  CU(launch_qtable(s, X, D, (int)N, (int)D, 0, ACT_RELU, ARCH_MLP, nullptr, nullptr, N, q_d));
  CU(enqueue_sym_gram(s, X, N, D, 0, ACT_RELU, ARCH_MLP, nullptr, nullptr, nullptr, SHIFT_NONE, 0, K0dd, ld0));
  if (T > 0) {
    CU(launch_qtable(s, Xt, D, (int)T, (int)D, 0, ACT_RELU, ARCH_MLP, nullptr, nullptr, T, q_t));
    CU(enqueue_cross_gram(s, Xt, T, X, N, D, 0, ACT_RELU, ARCH_MLP, nullptr, nullptr, nullptr, nullptr, K0td, ld0t));
  }
  return SMNNGP_OK;
}

size_t smnngp_grid_workspace_bytes(int64_t N, int64_t T, int n_hidden, int arch) {
  Carver c(nullptr);
  SolveWs w;
  return carve_solve(c, w, N, T, 1, n_act_applications(n_hidden, arch));
}

int smnngp_grid_point_f64(void* stream, const double* K0dd, int64_t ld0, const double* K0td, int64_t ld0t,
                          const double* q_d, const double* q_t, const double* y, int64_t N, int64_t T, int n_hidden,
                          int act, int arch, const double* hp_dev, void* workspace, size_t workspace_bytes,
                          double* mean_out, double* var_out, double* out_dev, int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!K0dd || !K0td || !q_d || !q_t || !y || !hp_dev || !mean_out || !var_out || !out_dev || !info_dev || N <= 0 ||
      T <= 0 || ld0 < N || ld0t < N || !valid_stack(n_hidden, act, arch) || N + T + 1 > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_grid_point_f64: invalid argument");
  Carver c(workspace);
  SolveWs w;
  if (carve_solve(c, w, N, T, 1, n_act_applications(n_hidden, arch)) > workspace_bytes || !workspace)
    return fail(SMNNGP_EWORKSPACE, "smnngp_grid_point_f64: workspace too small");
  CU(cudaMemsetAsync(info_dev, 0, sizeof(int), s));
  CU(launch_qtable_from_q(s, q_d, (int)N, n_hidden, act, arch, hp_dev, w.tab, N, w.q));
  CU(launch_scalars(s, w.q, (int)N, hp_dev, w.scal));
  CU(launch_qtable_from_q(s, q_t, (int)T, n_hidden, act, arch, hp_dev, w.tab_t, T, w.q_t));
  GramParams g{};
  g.N = (int)N; g.M = (int)N; g.tab1 = w.tab; g.tab2 = w.tab; g.tab_ld1 = N; g.tab_ld2 = N;
  g.n_hidden = n_hidden; g.act = act; g.arch = arch; g.hp = hp_dev; g.scal = w.scal;
  g.symmetric = 1; g.out_full = 0; g.K = w.A; g.ldk = w.lda;
  // (1) predict(eps): K + eps tr(K)/N I, K_td rows and y^T carried through the factorisation (find.py:75-77, :139)
  g.shift = SHIFT_EPS_REL;
  CU(launch_gram_from_base(s, g, K0dd, ld0));
  {
    GramParams x = g;
    x.N = (int)T; x.M = (int)N; x.tab1 = w.tab_t; x.tab_ld1 = T; x.shift = SHIFT_NONE; x.symmetric = 0; x.out_full = 1;
    x.K = w.A + N * w.lda;
    CU(launch_gram_from_base(s, x, K0td, ld0t));
  }
  CU(cudaMemcpyAsync(w.A + (N + T) * w.lda, y, N * sizeof(double), cudaMemcpyDeviceToDevice, s));
  CU(potrf_trapezoid(s, w.A, w.lda, N + T + 1, N, pick_nb(N), w.linv, w.scal + SC_LOGDET, info_dev, 0, -1, w.fws, false));
  CU(launch_predict_finalize(s, w.A + N * w.lda, w.lda, w.A + (N + T) * w.lda, w.lda, w.q_t, (int)T, 1, N, info_dev,
                             mean_out, var_out));
  // (2) log det(K + eps I) and y^T (K + eps I)^-1 y with the ABSOLUTE jitter (find.py:149-156)
  g.shift = SHIFT_EPS_ABS;
  CU(launch_gram_from_base(s, g, K0dd, ld0));
  CU(cudaMemcpyAsync(w.A + N * w.lda, y, N * sizeof(double), cudaMemcpyDeviceToDevice, s));
  CU(cudaMemsetAsync(w.scal2, 0, SC_COUNT * sizeof(double), s));
  CU(potrf_trapezoid(s, w.A, w.lda, N + 1, N, pick_nb(N), w.linv, w.scal2 + SC_LOGDET, info_dev, 0, -1, w.fws, false));
  CU(launch_sumsq(s, w.A + N * w.lda, N, w.scal2 + SC_QUAD));
  CU(cudaMemcpyAsync(out_dev, w.scal2 + SC_LOGDET, 2 * sizeof(double), cudaMemcpyDeviceToDevice, s));
  CU(launch_fill_nan_if_bad(s, info_dev, out_dev, 2));
  return SMNNGP_OK;
}

// the whole grid in one launch (grid_batch.cu): one slot per point in flight, the trapezoid first, then the tables
namespace {
size_t carve_grid_slot(GridBatchParams& p, long long N, long long T, int n_act) {
  const size_t na = (size_t)(n_act > 0 ? n_act : 1);
  Carver c(nullptr);
  p.lda = round_up(N, 16);
  c.take<double>((size_t)(N + T + 1) * p.lda);
  p.off_tab = (long long)(c.total() / 8);
  c.take<double>(na * N);
  p.off_q = (long long)(c.total() / 8);
  c.take<double>(N);
  p.off_tab_t = (long long)(c.total() / 8);
  c.take<double>(na * T);
  p.off_q_t = (long long)(c.total() / 8);
  c.take<double>(T);
  p.slot_bytes = (long long)c.total();
  return c.total();
}
}  // namespace

size_t smnngp_grid_batch_workspace_bytes(int64_t N, int64_t T, int n_hidden, int arch, int64_t slots) {
  GridBatchParams p{};
  return (size_t)(slots > 0 ? slots : 0) * carve_grid_slot(p, N, T, n_act_applications(n_hidden, arch));
}

int smnngp_grid_batch_f64(void* stream, const double* K0dd, int64_t ld0, const double* K0td, int64_t ld0t,
                          const double* q_d, const double* q_t, const double* y, int64_t N, int64_t T, int64_t G,
                          int n_hidden, int act, int arch, const double* hp_dev, void* workspace,
                          size_t workspace_bytes, double* mean_out, double* var_out, double* out_dev, int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!K0dd || !K0td || !q_d || !q_t || !y || !hp_dev || !mean_out || !var_out || !out_dev || !info_dev || N < 1 ||
      N > GRID_BATCH_MAX_N || T < 1 || G < 1 || ld0 < N || ld0t < N || !valid_stack(n_hidden, act, arch) ||
      N + T + 1 > INT32_MAX || G > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_grid_batch_f64: invalid argument");
  GridBatchParams p{};
  const size_t slot_bytes = carve_grid_slot(p, N, T, n_act_applications(n_hidden, arch));
  const long long slots = workspace ? (long long)(workspace_bytes / slot_bytes) : 0;
  if (slots < 1) return fail(SMNNGP_EWORKSPACE, "smnngp_grid_batch_f64: workspace holds no slot");
  p.K0dd = K0dd; p.K0td = K0td; p.q_d = q_d; p.q_t = q_t; p.y = y; p.hp = hp_dev;
  p.ld0 = ld0; p.ld0t = ld0t;
  p.N = (int)N; p.T = (int)T; p.G = (int)G; p.n_hidden = n_hidden; p.arch = arch;
  p.ws = static_cast<char*>(workspace);
  p.mean = mean_out; p.var = var_out; p.out = out_dev; p.info = info_dev;
  CU(launch_grid_batch(s, p, act, slots));
  return SMNNGP_OK;
}

// loss and gradient at every point in one launch (grad_batch.cu): the trapezoid A | y^T | I, then the tables and A^-1 y
namespace {
size_t carve_grad_slot(GradBatchParams& p, long long N, int n_act) {
  const size_t na = (size_t)(n_act > 0 ? n_act : 1);
  Carver c(nullptr);
  p.lda = round_up(N, 16);
  c.take<double>((size_t)(2 * N + 1) * p.lda);
  p.off_tab3 = (long long)(c.total() / 8);
  c.take<double>(3 * na * N);
  p.off_alpha = (long long)(c.total() / 8);
  c.take<double>(N);
  p.slot_bytes = (long long)c.total();
  return c.total();
}
}  // namespace

size_t smnngp_lml_grad_batch_workspace_bytes(int64_t N, int n_hidden, int arch, int64_t slots) {
  GradBatchParams p{};
  return (size_t)(slots > 0 ? slots : 0) * carve_grad_slot(p, N, n_act_applications(n_hidden, arch));
}

int smnngp_lml_grad_batch_f64(void* stream, const double* K0dd, int64_t ld0, const double* q_d, const double* y,
                              int64_t N, int64_t G, int n_hidden, int act, int arch, const double* hp_dev, int kind,
                              void* workspace, size_t workspace_bytes, double* out_dev, double* grad_dev,
                              int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!K0dd || !q_d || !y || !hp_dev || !out_dev || !grad_dev || !info_dev || N < 1 || N > GRID_BATCH_MAX_N || G < 1 ||
      ld0 < N || !valid_stack(n_hidden, act, arch) || (kind != KIND_GAUSS && kind != KIND_STUDENT_T) ||
      G > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_lml_grad_batch_f64: invalid argument");
  GradBatchParams p{};
  const size_t slot_bytes = carve_grad_slot(p, N, n_act_applications(n_hidden, arch));
  const long long slots = workspace ? (long long)(workspace_bytes / slot_bytes) : 0;
  if (slots < 1) return fail(SMNNGP_EWORKSPACE, "smnngp_lml_grad_batch_f64: workspace holds no slot");
  p.K0dd = K0dd; p.q_d = q_d; p.y = y; p.hp = hp_dev; p.ld0 = ld0;
  p.N = (int)N; p.G = (int)G; p.n_hidden = n_hidden; p.arch = arch; p.kind = kind;
  p.ws = static_cast<char*>(workspace);
  p.out = out_dev; p.grad = grad_dev; p.info = info_dev;
  CU(launch_lml_grad_batch(s, p, act, slots));
  return SMNNGP_OK;
}

// SPR.test_nll at every point in one launch (test_nll_batch.cu): the trapezoid, the tables, then the mean / var scratch
namespace {
size_t carve_test_nll_slot(TestNllBatchParams& p, long long N, long long T, int n_act) {
  const size_t na = (size_t)(n_act > 0 ? n_act : 1);
  Carver c(nullptr);
  p.lda = round_up(N, 16);
  c.take<double>((size_t)(N + T + 1) * p.lda);
  p.off_tab = (long long)(c.total() / 8);
  c.take<double>(na * N);
  p.off_q = (long long)(c.total() / 8);
  c.take<double>(N);
  p.off_tab_t = (long long)(c.total() / 8);
  c.take<double>(na * T);
  p.off_q_t = (long long)(c.total() / 8);
  c.take<double>(T);
  p.off_mv = (long long)(c.total() / 8);
  c.take<double>(2 * (size_t)T);
  p.slot_bytes = (long long)c.total();
  return c.total();
}
}  // namespace

size_t smnngp_test_nll_batch_workspace_bytes(int64_t N, int64_t T, int n_hidden, int arch, int64_t slots) {
  TestNllBatchParams p{};
  return (size_t)(slots > 0 ? slots : 0) * carve_test_nll_slot(p, N, T, n_act_applications(n_hidden, arch));
}

int smnngp_test_nll_batch_f64(void* stream, const double* K0dd, int64_t ld0, const double* K0td, int64_t ld0t,
                              const double* q_d, const double* q_t, const double* y, const double* yt, int64_t N,
                              int64_t T, int64_t G, int n_hidden, int act, int arch, const double* hp_dev, int kind,
                              double y_mean, double y_std, void* workspace, size_t workspace_bytes, double* nll_out,
                              double* mean_out, double* var_out, double* logp_out, int* info_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!K0dd || !K0td || !q_d || !q_t || !y || !yt || !hp_dev || !nll_out || !info_dev || N < 1 ||
      N > GRID_BATCH_MAX_N || T < 1 || G < 1 || ld0 < N || ld0t < N || !valid_stack(n_hidden, act, arch) ||
      (kind != KIND_GAUSS && kind != KIND_STUDENT_T) || N + T + 1 > INT32_MAX || G > INT32_MAX)
    return fail(SMNNGP_EINVAL, "smnngp_test_nll_batch_f64: invalid argument");
  TestNllBatchParams p{};
  const size_t slot_bytes = carve_test_nll_slot(p, N, T, n_act_applications(n_hidden, arch));
  const long long slots = workspace ? (long long)(workspace_bytes / slot_bytes) : 0;
  if (slots < 1) return fail(SMNNGP_EWORKSPACE, "smnngp_test_nll_batch_f64: workspace holds no slot");
  p.K0dd = K0dd; p.K0td = K0td; p.q_d = q_d; p.q_t = q_t; p.y = y; p.yt = yt; p.hp = hp_dev;
  p.ld0 = ld0; p.ld0t = ld0t;
  p.N = (int)N; p.T = (int)T; p.G = (int)G; p.n_hidden = n_hidden; p.arch = arch; p.kind = kind;
  p.y_mean = y_mean; p.y_std = y_std;
  p.ws = static_cast<char*>(workspace);
  p.nll = nll_out; p.mean = mean_out; p.var = var_out; p.logp = logp_out; p.info = info_dev;
  CU(launch_test_nll_batch(s, p, act, slots));
  return SMNNGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// posterior draw stage (draws.cu)
// ---------------------------------------------------------------------------------------------------------
int smnngp_sample_f_iid_f64(void* stream, const double* mean, const double* var, int var_per_class, int64_t T,
                            int64_t C, int64_t S, const double* hp_dev, int kind, uint64_t seed, double* out) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!mean || !var || !hp_dev || !out || T <= 0 || C <= 0 || S <= 0 || T > INT32_MAX || C > INT32_MAX ||
      S > INT32_MAX || C * T > INT64_MAX / S || (kind != KIND_GAUSS && kind != KIND_STUDENT_T))
    return fail(SMNNGP_EINVAL, "smnngp_sample_f_iid_f64: invalid argument");
  CU(launch_sample_f_iid(s, mean, var, var_per_class, (int)T, (int)C, (int)S, hp_dev, kind, seed, out));
  return SMNNGP_OK;
}

int smnngp_draw_metrics_f64(void* stream, const double* mean, const double* var, int var_per_class,
                            const int* label, int64_t T, int64_t C, int64_t S, const double* hp_dev, int kind,
                            uint64_t seed, double* ll_per_test, int* pred, double* out_dev) {
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Enter scope(s);
  if (!mean || !var || !label || !hp_dev || !ll_per_test || !pred || !out_dev || T <= 0 || C <= 0 || C > DRAW_MAXC ||
      S <= 0 || T > INT32_MAX || S > INT32_MAX || (kind != KIND_GAUSS && kind != KIND_STUDENT_T))
    return fail(SMNNGP_EINVAL, "smnngp_draw_metrics_f64: invalid argument");
  CU(launch_draw_metrics(s, mean, var, var_per_class, label, (int)T, (int)C, (int)S, hp_dev, kind, seed, ll_per_test,
                         pred, out_dev));
  return SMNNGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// host-buffer entry points
// ---------------------------------------------------------------------------------------------------------
void smnngp_host_release(void) {
  DeviceCtx& c = dctx();
  std::lock_guard<std::recursive_mutex> lk(c.mu);
  if (c.arena) cudaFree(c.arena);
  c.arena = nullptr;
  c.arena_bytes = 0;
  if (c.arena_stream) cudaStreamDestroy(c.arena_stream);
  c.arena_stream = nullptr;
}

int smnngp_lml_host_f64(const double* X, const double* y, int64_t N, int64_t D, int n_hidden, int act, int arch,
                        const double* hp, int kind, double* out, int* info) {
  if (!X || !y || !hp || !out || N <= 0 || D <= 0) return fail(SMNNGP_EINVAL, "smnngp_lml_host_f64: invalid argument");
  const size_t ws_bytes = smnngp_lml_workspace_bytes(N, D, n_hidden, arch);
  Carver c(nullptr);
  c.take<double>((size_t)N * D); c.take<double>(N); c.take<double>(HP_COUNT); c.take<double>(4); c.take<int>(1);
  const size_t io_bytes = c.total();
  Enter scope(nullptr);                       // host entry points run on the calling thread's current device
  DeviceCtx& dc = *scope.ctx;
  int rc = arena_reserve(dc, io_bytes + ws_bytes);
  if (rc != SMNNGP_OK) return rc;
  Carver a(dc.arena);
  double* dX = a.take<double>((size_t)N * D);
  double* dy = a.take<double>(N);
  double* dhp = a.take<double>(HP_COUNT);
  double* dout = a.take<double>(4);
  int* dinfo = a.take<int>(1);
  void* ws = static_cast<char*>(dc.arena) + io_bytes;
  cudaStream_t s = dc.arena_stream;
  CU(cudaMemcpyAsync(dX, X, (size_t)N * D * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dy, y, (size_t)N * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dhp, hp, HP_COUNT * 8, cudaMemcpyHostToDevice, s));
  rc = smnngp_lml_f64(s, dX, dy, N, D, n_hidden, act, arch, dhp, kind, ws, ws_bytes, dout, dinfo);
  if (rc != SMNNGP_OK) return rc;
  int hinfo = 0;
  CU(cudaMemcpyAsync(out, dout, 4 * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (info) *info = hinfo;
  return SMNNGP_OK;
}

int smnngp_lml_grad_host_f64(const double* X, const double* y, int64_t N, int64_t D, int n_hidden, int act, int arch,
                             const double* hp, int kind, double* out, double* grad, int* info) {
  if (!X || !y || !hp || !out || !grad || N <= 0 || D <= 0)
    return fail(SMNNGP_EINVAL, "smnngp_lml_grad_host_f64: invalid argument");
  const size_t ws_bytes = smnngp_lml_grad_workspace_bytes(N, D, n_hidden, arch);
  Carver c(nullptr);
  c.take<double>((size_t)N * D); c.take<double>(N); c.take<double>(HP_COUNT); c.take<double>(4);
  c.take<double>(HP_COUNT); c.take<int>(1);
  const size_t io_bytes = c.total();
  Enter scope(nullptr);                       // host entry points run on the calling thread's current device
  DeviceCtx& dc = *scope.ctx;
  int rc = arena_reserve(dc, io_bytes + ws_bytes);
  if (rc != SMNNGP_OK) return rc;
  Carver a(dc.arena);
  double* dX = a.take<double>((size_t)N * D);
  double* dy = a.take<double>(N);
  double* dhp = a.take<double>(HP_COUNT);
  double* dout = a.take<double>(4);
  double* dgrad = a.take<double>(HP_COUNT);
  int* dinfo = a.take<int>(1);
  void* ws = static_cast<char*>(dc.arena) + io_bytes;
  cudaStream_t s = dc.arena_stream;
  CU(cudaMemcpyAsync(dX, X, (size_t)N * D * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dy, y, (size_t)N * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dhp, hp, HP_COUNT * 8, cudaMemcpyHostToDevice, s));
  rc = smnngp_lml_grad_f64(s, dX, dy, N, D, n_hidden, act, arch, dhp, kind, ws, ws_bytes, dout, dgrad, dinfo);
  if (rc != SMNNGP_OK) return rc;
  int hinfo = 0;
  CU(cudaMemcpyAsync(out, dout, 4 * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(grad, dgrad, HP_COUNT * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (info) *info = hinfo;
  return SMNNGP_OK;
}

int smnngp_predict_host_f64(const double* X, const double* Y, const double* Xt, int64_t N, int64_t T, int64_t C,
                            int64_t D, int n_hidden, int act, int arch, const double* hp, int shift,
                            double* mean_out, double* var_out, int* info) {
  if (!X || !Y || !Xt || !hp || !mean_out || !var_out || N <= 0 || T <= 0 || C <= 0 || D <= 0)
    return fail(SMNNGP_EINVAL, "smnngp_predict_host_f64: invalid argument");
  const size_t ws_bytes = smnngp_predict_workspace_bytes(N, T, C, D, n_hidden, arch);
  Carver c(nullptr);
  c.take<double>((size_t)N * D); c.take<double>((size_t)N * C); c.take<double>((size_t)T * D);
  c.take<double>(HP_COUNT); c.take<double>((size_t)T * C); c.take<double>(T); c.take<int>(1);
  const size_t io_bytes = c.total();
  Enter scope(nullptr);                       // host entry points run on the calling thread's current device
  DeviceCtx& dc = *scope.ctx;
  int rc = arena_reserve(dc, io_bytes + ws_bytes);
  if (rc != SMNNGP_OK) return rc;
  Carver a(dc.arena);
  double* dX = a.take<double>((size_t)N * D);
  double* dY = a.take<double>((size_t)N * C);
  double* dXt = a.take<double>((size_t)T * D);
  double* dhp = a.take<double>(HP_COUNT);
  double* dmean = a.take<double>((size_t)T * C);
  double* dvar = a.take<double>(T);
  int* dinfo = a.take<int>(1);
  void* ws = static_cast<char*>(dc.arena) + io_bytes;
  cudaStream_t s = dc.arena_stream;
  CU(cudaMemcpyAsync(dX, X, (size_t)N * D * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dY, Y, (size_t)N * C * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dXt, Xt, (size_t)T * D * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dhp, hp, HP_COUNT * 8, cudaMemcpyHostToDevice, s));
  rc = smnngp_predict_f64(s, dX, dY, dXt, N, T, C, D, n_hidden, act, arch, dhp, shift, ws, ws_bytes, dmean, dvar,
                          dinfo);
  if (rc != SMNNGP_OK) return rc;
  int hinfo = 0;
  CU(cudaMemcpyAsync(mean_out, dmean, (size_t)T * C * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(var_out, dvar, (size_t)T * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (info) *info = hinfo;
  return SMNNGP_OK;
}

int smnngp_test_nll_host_f64(const double* X, const double* y, const double* Xt, const double* yt, int64_t N,
                             int64_t T, int64_t D, int n_hidden, int act, int arch, const double* hp, int kind,
                             double y_mean, double y_std, double* nll_out, double* mean_out, double* var_out,
                             int* info) {
  if (!X || !y || !Xt || !yt || !hp || !nll_out || N <= 0 || T <= 0 || D <= 0)
    return fail(SMNNGP_EINVAL, "smnngp_test_nll_host_f64: invalid argument");
  const size_t ws_bytes = smnngp_predict_workspace_bytes(N, T, 1, D, n_hidden, arch);
  Carver c(nullptr);
  c.take<double>((size_t)N * D); c.take<double>(N); c.take<double>((size_t)T * D); c.take<double>(T);
  c.take<double>(HP_COUNT); c.take<double>(T); c.take<double>(T); c.take<double>(1); c.take<int>(1);
  const size_t io_bytes = c.total();
  Enter scope(nullptr);                       // host entry points run on the calling thread's current device
  DeviceCtx& dc = *scope.ctx;
  int rc = arena_reserve(dc, io_bytes + ws_bytes);
  if (rc != SMNNGP_OK) return rc;
  Carver a(dc.arena);
  double* dX = a.take<double>((size_t)N * D);
  double* dy = a.take<double>(N);
  double* dXt = a.take<double>((size_t)T * D);
  double* dyt = a.take<double>(T);
  double* dhp = a.take<double>(HP_COUNT);
  double* dmean = a.take<double>(T);
  double* dvar = a.take<double>(T);
  double* dnll = a.take<double>(1);
  int* dinfo = a.take<int>(1);
  void* ws = static_cast<char*>(dc.arena) + io_bytes;
  cudaStream_t s = dc.arena_stream;
  CU(cudaMemcpyAsync(dX, X, (size_t)N * D * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dy, y, (size_t)N * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dXt, Xt, (size_t)T * D * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dyt, yt, (size_t)T * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(dhp, hp, HP_COUNT * 8, cudaMemcpyHostToDevice, s));
  rc = smnngp_test_nll_f64(s, dX, dy, dXt, dyt, N, T, D, n_hidden, act, arch, dhp, kind, y_mean, y_std, ws,
                           ws_bytes, dnll, dmean, dvar, nullptr, dinfo);
  if (rc != SMNNGP_OK) return rc;
  int hinfo = 0;
  CU(cudaMemcpyAsync(nll_out, dnll, 8, cudaMemcpyDeviceToHost, s));
  if (mean_out) CU(cudaMemcpyAsync(mean_out, dmean, (size_t)T * 8, cudaMemcpyDeviceToHost, s));
  if (var_out) CU(cudaMemcpyAsync(var_out, dvar, (size_t)T * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof(int), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (info) *info = hinfo;
  return SMNNGP_OK;
}

}  // extern "C"

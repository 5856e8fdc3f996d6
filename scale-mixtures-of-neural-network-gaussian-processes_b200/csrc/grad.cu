// Gradient of the log marginal likelihood w.r.t. the six positive scalars {w_std, b_std, last_w_std, eps, alpha,
// beta} - what objax.GradValues(model.loss, model.vars()) obtains by reverse-mode AD through SPR.loss in the
// reference's training loop (experiments/regression/train.py:62-66, :178-179; spax/models.py:93-98).
//
//   d log p / d A = G = 1/2 (gamma a a^T - A^-1),   A = K + eps I,  a = A^-1 y,
//   gamma = (2 alpha + N) / ((2 alpha + quad alpha / beta) beta / alpha)  (Student-t),  1 (Gaussian)
//   d log p / d theta = sum_ij G_ij dK_ij / d theta        (theta = w_std, b_std, last_w_std),   d / d eps = tr G
//
// A^-1 comes from the factorisation itself: identity rows carried through potrf_trapezoid become U = L^-T
// (chol.cu, ident_row0), A^-1 = U U^T is one lower-triangular SYRK on the same GEMM core (k >= row only).
// dK/dtheta is never materialised: this file's Gram pass recomputes the X.X^T tile on the tensor pipe, runs the
// layer recursion in forward-mode dual arithmetic on the accumulators (3 values per entry) and contracts with the
// G tile in registers.  Partial sums go to one slot per warp (fixed tile order per warp, fixed-order final
// reduction): bit-reproducible.
#include "closed_forms.cuh"
#include "gemm_core.cuh"
#include "kernels.cuh"
#include "nngp_math.cuh"
#include "tma_core.cuh"

namespace smnngp {

namespace {

__global__ void qtable_dual_kernel(const double* __restrict__ X, long long ldx, int N, int D, int n_hidden, int act,
                                   int arch, const double* __restrict__ hp, double* __restrict__ tab3,
                                   long long tab_ld, int n_act) {
  int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  int lane = threadIdx.x & 31;
  if (row >= N) return;
  const double* x = X + (long long)row * ldx;
  double s = 0.0;
  for (int k = lane; k < D; k += 32) s = fma(x[k], x[k], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane != 0) return;
  fill_row_dual_tables(s, D, row, n_hidden, act, arch, hp, tab3, tab_ld, n_act);
}

struct GradParams {
  GramParams g;           // symmetric Gram description (X1 == X2, tab1 = plane 0 of tab3)
  const double* tab3;     // [3][n_act][tab_ld]
  long long plane;
  const double* Winv;     // A^-1, lower triangle valid
  long long ldw;
  const double* alpha;    // A^-1 y
  const double* quad;     // device: y^T A^-1 y
  int kind;
  double* partial;        // [slots][4]: sum G dK/dw, sum G dK/db, sum G K, tr G
  // row strip (multi-GPU): tile rows are local to the strip, g.N = rows of the strip, Winv = the strip of A^-1;
  // global row = row0 + local row; n_total = order of the whole matrix (0: not a strip, g.N)
  int row0, n_total;
};

__device__ __forceinline__ double grad_gamma(const GradParams& p) {
  if (p.kind != KIND_STUDENT_T) return 1.0;
  const double a = p.g.hp[HP_ALPHA], b = p.g.hp[HP_BETA];
  const double n = (double)(p.n_total > 0 ? p.n_total : p.g.N);
  return (2.0 * a + n) / ((2.0 * a + (*p.quad) * a / b) * (b / a));
}

// one warp's 64 x 32 part of a tile: returns the four partial sums of this THREAD in sums[]
template <int ACT>
__device__ __forceinline__ void grad_epilogue(const GradParams& p, double (&acc)[MI][NI][2], int rbase, int cbase,
                                              double (&sums)[4]) {
  const int N = p.g.N;
  const double w = p.g.hp[HP_W], b = p.g.hp[HP_B], v = p.g.hp[HP_V];
  const double w2 = w * w, b2 = b * b, v2 = v * v;
  const double inv_d = 1.0 / (double)p.g.D;
  const bool resnet = p.g.arch == ARCH_RESNET;
  const int n_act = resnet ? p.g.n_hidden + 1 : p.g.n_hidden;
  const double gamma = grad_gamma(p);
  const double* __restrict__ t0 = p.tab3;
  const double* __restrict__ t1 = p.tab3 + p.plane;
  const double* __restrict__ t2 = p.tab3 + 2 * p.plane;
  const long long tl = p.g.tab_ld1;
  sums[0] = sums[1] = sums[2] = sums[3] = 0.0;
  const int row0 = p.row0;                                       // global row of the strip's first row (0: whole matrix)
  if (cbase > row0 + rbase + (MI - 1) * 8 || rbase >= N) return; // nothing of this thread lies in the lower triangle
  const int ncols = p.g.M;

  int cc[NI][2];
  double al_c[NI][2];
#pragma unroll
  for (int ni = 0; ni < NI; ni++)
#pragma unroll
    for (int e = 0; e < 2; e++) {
      cc[ni][e] = min(cbase + ni * 8 + e, ncols - 1);
      al_c[ni][e] = p.alpha[cc[ni][e]];
    }

  // ROLLED over the 8 row groups (see gram_epilogue): each trip works on accumulator row 0 and rotates the rows
  // through the registers - the fully unrolled version was ~29k instructions and ran at the instruction-fetch rate.
#pragma unroll 1
  for (int it = 0; it < MI; it++) {
    const int rl = rbase + it * 8;                               // row inside the strip
    const int r = row0 + rl;                                       // global row
    if (rl < N && cbase <= r) {
      double k[NI][2], dw[NI][2], db[NI][2];
#pragma unroll
      for (int ni = 0; ni < NI; ni++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const double k0 = acc[0][ni][e] * inv_d;
          // dense-resnet: leading Dense(512)
          k[ni][e] = resnet ? fma(w2, k0, b2) : k0;
          dw[ni][e] = resnet ? 2.0 * w * k0 : 0.0;
          db[ni][e] = resnet ? 2.0 * b : 0.0;
        }
      for (int a = 0; a < n_act; a++) {
        const double e1 = t0[a * tl + r], fw1 = t1[a * tl + r], fb1 = t2[a * tl + r];
        const bool plain = !resnet || (a == n_act - 1);
#pragma unroll
        for (int ni = 0; ni < NI; ni++)
#pragma unroll
          for (int e = 0; e < 2; e++) {
            const long long ci = a * tl + cc[ni][e];
            layer_step_dual<ACT>(k[ni][e], dw[ni][e], db[ni][e], e1, t0[ci], fw1 + t1[ci], fb1 + t2[ci], w, b, w2, b2,
                                 resnet, plain);
          }
      }
      const double al_r = p.alpha[r];
      const double* __restrict__ wrow = p.Winv + (long long)rl * p.ldw;
#pragma unroll
      for (int ni = 0; ni < NI; ni++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int c = cbase + ni * 8 + e;
          if (c > r) continue;                                     // c <= r < N
          double g = 0.5 * fma(gamma * al_r, al_c[ni][e], -wrow[c]);
          if (c == r) sums[3] += g;
          else g += g;                                             // the mirrored entry
          sums[0] = fma(g, v2 * dw[ni][e], sums[0]);
          sums[1] = fma(g, v2 * db[ni][e], sums[1]);
          sums[2] = fma(g, k[ni][e], sums[2]);                     // d K / d last_w_std = 2 v k
        }
    }
#pragma unroll
    for (int mi = 0; mi < MI - 1; mi++)
#pragma unroll
      for (int ni = 0; ni < NI; ni++) {
        acc[mi][ni][0] = acc[mi + 1][ni][0];
        acc[mi][ni][1] = acc[mi + 1][ni][1];
      }
  }
  sums[2] *= 2.0 * v;
}

__device__ __forceinline__ void warp_reduce4(double (&sums)[4]) {
#pragma unroll
  for (int q = 0; q < 4; q++)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sums[q] += __shfl_xor_sync(0xffffffffu, sums[q], o);
}

// TMA-fed persistent variant: slot = (CTA, math warp); a warp visits its tiles in a fixed order
template <int ACT>
struct EpiGradTma {
  using Params = GradParams;
  static __device__ __forceinline__ void apply(const Params& p, double (&acc)[MI][NI][2], int r0, int c0, int wm,
                                               int wn, int lane) {
    double sums[4];
    grad_epilogue<ACT>(p, acc, r0 + wm * 64 + (lane >> 2), c0 + wn * 32 + (lane & 3) * 2, sums);
    warp_reduce4(sums);
    if (lane == 0) {
      double* slot = p.partial + ((long long)blockIdx.x * 8 + ((threadIdx.x >> 5) - 4)) * 4;
#pragma unroll
      for (int q = 0; q < 4; q++) slot[q] += sums[q];
    }
  }
};

template <typename Cfg, bool ALIGN16, int ACT>
__global__ void __launch_bounds__(Cfg::THREADS, Cfg::MIN_BLOCKS) grad_gram_kernel(const GradParams p) {
  extern __shared__ __align__(16) double smem[];
  const int ntn = (p.g.M + Cfg::BN - 1) / Cfg::BN;
  int ti, tj;
  decode_tile<Cfg::Q>(blockIdx.x, ntn, 1, ti, tj);
  const int r0 = ti * Cfg::BM, c0 = tj * Cfg::BN;
  double acc[MI][NI][2];
  gemm_mainloop<Cfg, ALIGN16>(acc, p.g.X1 + (long long)r0 * p.g.ld1, p.g.ld1, min(Cfg::BM, p.g.N - r0),
                              p.g.X2 + (long long)c0 * p.g.ld2, p.g.ld2, min(Cfg::BN, p.g.M - c0), p.g.D, smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double sums[4];
  grad_epilogue<ACT>(p, acc, r0 + (warp / Cfg::WARPS_N) * 64 + (lane >> 2),
                     c0 + (warp % Cfg::WARPS_N) * 32 + (lane & 3) * 2, sums);
  warp_reduce4(sums);
  if (lane == 0) {
    double* slot = p.partial + ((long long)blockIdx.x * (Cfg::THREADS / 32) + warp) * 4;
#pragma unroll
    for (int q = 0; q < 4; q++) slot[q] = sums[q];
  }
}

template <bool ALIGN16>
cudaError_t launch_grad_fallback(cudaStream_t s, const GradParams& p) {
  using Cfg = TilePair;
  long long tiles = count_tiles<Cfg>(p.g.N, p.g.M, 1);
  auto kern = p.g.act == ACT_RELU ? grad_gram_kernel<Cfg, ALIGN16, ACT_RELU> : grad_gram_kernel<Cfg, ALIGN16, ACT_ERF>;
  cudaError_t e = configure_kernel_once(reinterpret_cast<const void*>(kern), Cfg::SMEM_BYTES, true);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)tiles, Cfg::THREADS, Cfg::SMEM_BYTES, s>>>(p);
  instr().launches++;
  return cudaGetLastError();
}

// one block: fixed-order sum of the slots, then the closed forms.  grad[6] = d loss / d hp, loss = -log p / N.
__global__ void __launch_bounds__(1024) grad_finalize_kernel(const double* __restrict__ partial, long long slots,
                                                             const double* __restrict__ hp,
                                                             const double* __restrict__ quad_p, int kind,
                                                             long long N, const int* __restrict__ info,
                                                             double* __restrict__ grad) {
  __shared__ double red[4][1024];
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  for (long long i = threadIdx.x; i < slots; i += 1024)
#pragma unroll
    for (int q = 0; q < 4; q++) s[q] += partial[i * 4 + q];
#pragma unroll
  for (int q = 0; q < 4; q++) red[q][threadIdx.x] = s[q];
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o)
#pragma unroll
      for (int q = 0; q < 4; q++) red[q][threadIdx.x] += red[q][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  grad_closed_form(red[0][0], red[1][0], red[2][0], red[3][0], hp, quad_p, kind, N, info, grad);
}

// alpha_i = sum_{k >= i} U[i,k] z[k]   (U = L^-T upper triangular, row-major): one block per row
__global__ void __launch_bounds__(128) upper_gemv_kernel(const double* __restrict__ U, long long ldu,
                                                         const double* __restrict__ z, long long N,
                                                         double* __restrict__ out) {
  __shared__ double red[4];
  const long long i = blockIdx.x;
  const double* u = U + i * ldu;
  double a0 = 0.0, a1 = 0.0;
  long long k = (i & ~1ll) + 2ll * threadIdx.x;                  // even start: 16-byte loads (ldu is even)
  for (; k + 1 < N; k += 256) {
    const double2 uv = *reinterpret_cast<const double2*>(u + k);
    const double2 zv = *reinterpret_cast<const double2*>(z + k);
    if (k >= i) a0 = fma(uv.x, zv.x, a0);
    a1 = fma(uv.y, zv.y, a1);
  }
  if (k < N && k >= i) a0 = fma(u[k], z[k], a0);
  double v = a0 + a1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) out[i] = (red[0] + red[1]) + (red[2] + red[3]);
}

__global__ void set_identity_kernel(double* __restrict__ A, long long lda, long long N) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) A[i * lda + i] = 1.0;
}

}  // namespace

long long grad_partial_slots(long long N) {
  const long long tma = (long long)device_sm_count() * 8;
  const long long fb = count_tiles<TilePair>(N, N, 1) * (TilePair::THREADS / 32);
  return tma > fb ? tma : fb;
}

cudaError_t launch_qtable_dual(cudaStream_t s, const double* X, long long ldx, int N, int D, int n_hidden, int act,
                               int arch, const double* hp, double* tab3, long long tab_ld) {
  if (N <= 0) return cudaSuccess;
  const int warps_per_block = 8;
  const unsigned blocks = (unsigned)((N + warps_per_block - 1) / warps_per_block);
  qtable_dual_kernel<<<blocks, warps_per_block * 32, 0, s>>>(X, ldx, N, D, n_hidden, act, arch, hp, tab3, tab_ld,
                                                             n_act_applications(n_hidden, arch));
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_set_identity(cudaStream_t s, double* A, long long lda, long long N) {
  cudaError_t e = cudaMemsetAsync(A, 0, (size_t)N * lda * sizeof(double), s);
  if (e != cudaSuccess) return e;
  set_identity_kernel<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(A, lda, N);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_set_ones_diag(cudaStream_t s, double* A, long long lda, long long N) {
  if (N <= 0) return cudaSuccess;
  set_identity_kernel<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(A, lda, N);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_upper_gemv(cudaStream_t s, const double* U, long long ldu, const double* z, long long N,
                              double* out) {
  if (N <= 0) return cudaSuccess;
  upper_gemv_kernel<<<(unsigned)N, 128, 0, s>>>(U, ldu, z, N, out);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_grad_gram(cudaStream_t s, const double* X, long long N, long long D, int n_hidden, int act,
                             int arch, const double* hp, const double* tab3, long long tab_ld, const double* Winv,
                             long long ldw, const double* alpha, const double* quad, int kind, double* partial,
                             long long slots) {
  if (N <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(partial, 0, (size_t)slots * 4 * sizeof(double), s);
  if (e != cudaSuccess) return e;
  GradParams p{};
  p.g.X1 = X; p.g.X2 = X; p.g.ld1 = D; p.g.ld2 = D; p.g.N = (int)N; p.g.M = (int)N; p.g.D = (int)D;
  p.g.tab1 = tab3; p.g.tab2 = tab3; p.g.tab_ld1 = tab_ld; p.g.tab_ld2 = tab_ld;
  p.g.n_hidden = n_hidden; p.g.act = act; p.g.arch = arch; p.g.hp = hp; p.g.symmetric = 1;
  p.tab3 = tab3;
  const int n_act = n_act_applications(n_hidden, arch);
  p.plane = (long long)(n_act > 0 ? n_act : 1) * tab_ld;
  p.Winv = Winv; p.ldw = ldw; p.alpha = alpha; p.quad = quad; p.kind = kind; p.partial = partial;
  if (tile_variant() == 0 && tma_operand_ok(X, D)) {
    CUtensorMap ma, mb;
    if (!make_tmap(&ma, X, N, D, D, TM_BM) || !make_tmap(&mb, X, N, D, D, TM_BN)) return cudaErrorInvalidValue;
    TmaShape sh{(int)N, (int)N, (int)D, 1, count_tiles<TileTma>(N, N, 1), 0, 1, 0, 0};
    e = act == ACT_RELU ? launch_tma_gemm<EpiGradTma<ACT_RELU>>(s, ma, mb, sh, p, device_sm_count())
                        : launch_tma_gemm<EpiGradTma<ACT_ERF>>(s, ma, mb, sh, p, device_sm_count());
    instr().launches++;
    return e;
  }
  const bool a16 = (D % 2 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
  return a16 ? launch_grad_fallback<true>(s, p) : launch_grad_fallback<false>(s, p);
}

cudaError_t launch_grad_gram_strip(cudaStream_t s, const double* X, long long N, long long D, long long row0,
                                   long long rows, int n_hidden, int act, int arch, const double* hp, const double* tab3,
                                   long long tab_ld, const double* Winv_strip, long long ldw, const double* alpha,
                                   const double* quad, int kind, double* partial, long long slots) {
  cudaError_t e = cudaMemsetAsync(partial, 0, (size_t)slots * 4 * sizeof(double), s);
  if (e != cudaSuccess || rows <= 0) return e;
  if (!(tile_variant() == 0 && tma_operand_ok(X, D)) || (row0 % TM_BM) != 0) return cudaErrorInvalidValue;
  const long long ncols = row0 + rows;
  GradParams p{};
  p.g.X1 = X + row0 * D; p.g.X2 = X; p.g.ld1 = D; p.g.ld2 = D; p.g.N = (int)rows; p.g.M = (int)ncols; p.g.D = (int)D;
  p.g.tab1 = tab3; p.g.tab2 = tab3; p.g.tab_ld1 = tab_ld; p.g.tab_ld2 = tab_ld;
  p.g.n_hidden = n_hidden; p.g.act = act; p.g.arch = arch; p.g.hp = hp; p.g.symmetric = 1;
  p.tab3 = tab3;
  const int n_act = n_act_applications(n_hidden, arch);
  p.plane = (long long)(n_act > 0 ? n_act : 1) * tab_ld;
  p.Winv = Winv_strip; p.ldw = ldw; p.alpha = alpha; p.quad = quad; p.kind = kind; p.partial = partial;
  p.row0 = (int)row0; p.n_total = (int)N;
  CUtensorMap ma, mb;
  if (!make_tmap(&ma, X + row0 * D, rows, D, D, TM_BM) || !make_tmap(&mb, X, ncols, D, D, TM_BN))
    return cudaErrorInvalidValue;
  // lower part of the strip: local row r may touch columns <= row0 + r (the shifted-diagonal mask of the update kernel)
  TmaShape sh{(int)rows, (int)ncols, (int)D, 0, 0, 1 << 30, 1, (int)row0, 0};
  sh.tiles = tma_cyc_count_tiles(sh);
  e = act == ACT_RELU ? launch_tma_gemm<EpiGradTma<ACT_RELU>>(s, ma, mb, sh, p, device_sm_count())
                      : launch_tma_gemm<EpiGradTma<ACT_ERF>>(s, ma, mb, sh, p, device_sm_count());
  instr().launches++;
  return e;
}

namespace {
__global__ void __launch_bounds__(1024) sum_slots_kernel(const double* __restrict__ partial, long long slots,
                                                         double* __restrict__ out4) {
  __shared__ double red[4][1024];
  double s[4] = {0.0, 0.0, 0.0, 0.0};
  for (long long i = threadIdx.x; i < slots; i += 1024)
#pragma unroll
    for (int q = 0; q < 4; q++) s[q] += partial[i * 4 + q];
#pragma unroll
  for (int q = 0; q < 4; q++) red[q][threadIdx.x] = s[q];
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o)
#pragma unroll
      for (int q = 0; q < 4; q++) red[q][threadIdx.x] += red[q][threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x < 4) out4[threadIdx.x] = red[threadIdx.x][0];
}
}  // namespace

cudaError_t launch_sum_slots(cudaStream_t s, const double* partial, long long slots, double* out4) {
  sum_slots_kernel<<<1, 1024, 0, s>>>(partial, slots, out4);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_grad_finalize(cudaStream_t s, const double* partial, long long slots, const double* hp,
                                 const double* quad, int kind, long long N, const int* info, double* grad) {
  grad_finalize_kernel<<<1, 1024, 0, s>>>(partial, slots, hp, quad, kind, N, info, grad);
  instr().launches++;
  return cudaGetLastError();
}

}  // namespace smnngp

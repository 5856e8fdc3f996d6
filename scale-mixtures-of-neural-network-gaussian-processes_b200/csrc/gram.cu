// NNGP Gram matrix for the MLP / dense-resnet stacks of the reference (experiments/nt_kernels.py:21-31,
// :83-103, called through spax/kernels.py:23-27): one FP64 tensor-core X.X'^T contraction whose epilogue
// applies the whole L-layer ReLU arc-cosine / erf recursion in registers, so every kernel entry is written to
// HBM exactly once.  Symmetric case: only tiles on or below the diagonal are computed (optionally mirrored).
#include "gemm_core.cuh"
#include "context.cuh"
#include "kernels.cuh"
#include "nngp_math.cuh"
#include "tma_core.cuh"

namespace smnngp {

namespace {

__global__ void qtable_kernel(const double* __restrict__ X, long long ldx, int N, int D, int n_hidden, int act,
                              int arch, const double* __restrict__ hp, double* __restrict__ tab,
                              long long tab_ld, double* __restrict__ qfin) {
  int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  int lane = threadIdx.x & 31;
  if (row >= N) return;
  const double* x = X + (long long)row * ldx;
  double s = 0.0;
  for (int k = lane; k < D; k += 32) s = fma(x[k], x[k], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane != 0) return;
  fill_row_tables(s / (double)D, row, n_hidden, act, arch, hp, tab, tab_ld, qfin);
}

// the same tables from a cached q0 (grid search: X is not touched again)
__global__ void qtable_from_q_kernel(const double* __restrict__ q0, int N, int n_hidden, int act, int arch,
                                     const double* __restrict__ hp, double* __restrict__ tab, long long tab_ld,
                                     double* __restrict__ qfin) {
  const int row = blockIdx.x * blockDim.x + threadIdx.x;
  if (row < N) fill_row_tables(q0[row], row, n_hidden, act, arch, hp, tab, tab_ld, qfin);
}

// single block, fixed reduction order (deterministic)
__global__ void scalars_kernel(const double* __restrict__ qfin, int N, const double* __restrict__ hp,
                               double* __restrict__ scal) {
  __shared__ double red[1024];
  double s = 0.0;
  for (int i = threadIdx.x; i < N; i += blockDim.x) s += qfin[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    double trmean = red[0] / (double)N;
    double eps = hp[HP_EPS];
    scal[SC_TRMEAN] = trmean;
    scal[SC_SHIFT0 + SHIFT_NONE] = 0.0;
    scal[SC_SHIFT0 + SHIFT_EPS_ABS] = eps;
    scal[SC_SHIFT0 + SHIFT_EPS_REL] = eps * trmean;
    scal[SC_SHIFT0 + SHIFT_LIK] = 1e-6 * hp[HP_ALPHA] / hp[HP_BETA];
    scal[SC_LOGDET] = 0.0;
    scal[SC_QUAD] = 0.0;
  }
}

#ifndef SMNNGP_GRAM_RU
#define SMNNGP_GRAM_RU 1
#endif
constexpr int RU = SMNNGP_GRAM_RU;   // accumulator rows (of 8 entries) evaluated per trip of the rolled epilogue loop

// L-layer recursion + final Dense + diagonal shift + store for one warp's 64 x 32 part of a tile
template <int ACT>
__device__ __forceinline__ void gram_epilogue(const GramParams& p, double (&acc)[MI][NI][2], int rbase, int cbase) {
  // hp == nullptr: unit scalars - the base Gram K0 = X.X'^T / D of the grid search (n_hidden = 0)
  const double w2 = p.hp ? p.hp[HP_W] * p.hp[HP_W] : 1.0, b2 = p.hp ? p.hp[HP_B] * p.hp[HP_B] : 0.0,
               v2 = p.hp ? p.hp[HP_V] * p.hp[HP_V] : 1.0;
  const double inv_d = 1.0 / (double)p.D;
  const bool resnet = p.arch == ARCH_RESNET;

  // which of this thread's 64 entries are real output (edge tiles, strict upper part on the symmetric path)
  unsigned long long live = 0ull;
#pragma unroll
  for (int mi = 0; mi < MI; mi++)
#pragma unroll
    for (int ni = 0; ni < NI; ni++)
#pragma unroll
      for (int e = 0; e < 2; e++) {
        int r = rbase + mi * 8, c = cbase + ni * 8 + e;
        bool ok = r < p.N && c < p.M && (!p.symmetric || c <= r);
        if (ok) live |= 1ull << (mi * 8 + ni * 2 + e);
        double k = acc[mi][ni][e] * inv_d;              // kernel_fn normalises X.X'^T by the feature count
        acc[mi][ni][e] = resnet ? (w2 * k + b2) : k;    // dense-resnet: leading Dense(512)
      }

  const int n_act = resnet ? p.n_hidden + 1 : p.n_hidden;
  for (int a = 0; a < n_act; a++) {
    double tr[MI], tc[NI][2];
#pragma unroll
    for (int mi = 0; mi < MI; mi++) {
      int r = rbase + mi * 8;
      tr[mi] = r < p.N ? p.tab1[a * p.tab_ld1 + r] : 1.0;
    }
#pragma unroll
    for (int ni = 0; ni < NI; ni++)
#pragma unroll
      for (int e = 0; e < 2; e++) {
        int c = cbase + ni * 8 + e;
        tc[ni][e] = c < p.M ? p.tab2[a * p.tab_ld2 + c] : 1.0;
      }
    const bool plain = !resnet || (a == n_act - 1);     // MLP layer, or the trailing activation of the resnet
    {
      // Entries that are not real output (edge tiles: zero accumulators and table value 1; strict upper part on the
      // symmetric path) are evaluated like the others and simply never stored.
      // The loop over the 8 row groups is ROLLED: each trip evaluates the 8 entries of accumulator
      // row 0 (8 independent chains) and then rotates the rows through the registers, so the body is ~1/8 of the
      // fully unrolled code.  Unrolled, the 64 inlined evaluations were ~90 KB of SASS per pass - more than the
      // instruction cache holds next to the other math group - and the epilogue ran at the instruction-fetch rate
      // (first layer of a tile ~4x slower than the FP64 pipe allows).
#pragma unroll 1
      for (int it = 0; it < MI / RU; it++) {
        double res[RU][NI][2];
#pragma unroll
        for (int u = 0; u < RU; u++)
#pragma unroll
          for (int ni = 0; ni < NI; ni++)
#pragma unroll
            for (int e = 0; e < 2; e++) {
              res[u][ni][e] = layer_step<ACT>(acc[u][ni][e], tr[u], tc[ni][e], w2, b2, resnet, plain);
            }
#pragma unroll
        for (int mi = 0; mi < MI - RU; mi++) {
          tr[mi] = tr[mi + RU];
#pragma unroll
          for (int ni = 0; ni < NI; ni++) {
            acc[mi][ni][0] = acc[mi + RU][ni][0];
            acc[mi][ni][1] = acc[mi + RU][ni][1];
          }
        }
#pragma unroll
        for (int u = 0; u < RU; u++)
#pragma unroll
          for (int ni = 0; ni < NI; ni++) {
            acc[MI - RU + u][ni][0] = res[u][ni][0];
            acc[MI - RU + u][ni][1] = res[u][ni][1];
          }
      }
    }
  }

  const double sh = (p.symmetric && p.shift != SHIFT_NONE) ? p.scal[SC_SHIFT0 + p.shift] : 0.0;
  const bool vec_ok = ((p.ldk & 1) == 0) && ((reinterpret_cast<uintptr_t>(p.K) & 15) == 0);
  const bool mirror = p.symmetric && p.out_full;
#pragma unroll
  for (int mi = 0; mi < MI; mi++) {
    const int r = rbase + mi * 8;
    if (r >= p.N) continue;
#pragma unroll
    for (int ni = 0; ni < NI; ni++) {
      const int c = cbase + ni * 8;
      double k0 = v2 * acc[mi][ni][0], k1 = v2 * acc[mi][ni][1];   // final Dense(num_class, W_std=last_w_std)
      if (p.symmetric) {
        if (r == c) k0 += sh;
        if (r == c + 1) k1 += sh;
      }
      const bool ok0 = (live >> (mi * 8 + ni * 2)) & 1ull, ok1 = (live >> (mi * 8 + ni * 2 + 1)) & 1ull;
      double* dst = p.K + (long long)r * p.ldk + c;
      if (ok0 && ok1 && vec_ok) {
        *reinterpret_cast<double2*>(dst) = make_double2(k0, k1);
      } else {
        if (ok0) dst[0] = k0;
        if (ok1) dst[1] = k1;
      }
      if (mirror) {
        if (ok0 && c != r) p.K[(long long)c * p.ldk + r] = k0;
        if (ok1 && c + 1 != r) p.K[(long long)(c + 1) * p.ldk + r] = k1;
      }
    }
  }
}

template <typename Cfg, bool ALIGN16, int ACT>
__global__ void __launch_bounds__(Cfg::THREADS, Cfg::MIN_BLOCKS) gram_kernel(const GramParams p) {
  extern __shared__ __align__(16) double smem[];
  const int ntn = (p.M + Cfg::BN - 1) / Cfg::BN;
  int ti, tj;
  decode_tile<Cfg::Q>(blockIdx.x, ntn, p.symmetric, ti, tj);
  const int r0 = ti * Cfg::BM, c0 = tj * Cfg::BN;
  double acc[MI][NI][2];
  gemm_mainloop<Cfg, ALIGN16>(acc, p.X1 + (long long)r0 * p.ld1, p.ld1, min(Cfg::BM, p.N - r0),
                              p.X2 + (long long)c0 * p.ld2, p.ld2, min(Cfg::BN, p.M - c0), p.D, smem);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  gram_epilogue<ACT>(p, acc, r0 + (warp / Cfg::WARPS_N) * 64 + (lane >> 2),
                     c0 + (warp % Cfg::WARPS_N) * 32 + (lane & 3) * 2);
}

// Recursion-only pass over a cached base Gram K0 (= X.X'^T / D): the hyper-parameter grid search of
// experiments/regression/find.py:134-199 evaluates many (w_std, b_std) on the same inputs, so the contraction is done
// once and every grid point is one HBM pass (8 B read + 8 B written per entry).  A 128 x 64 tile per CTA, the K0
// values are loaded straight into the accumulator layout of the GEMM core and handed to the same epilogue.
template <int ACT>
__global__ void __launch_bounds__(128) gram_from_base_kernel(const GramParams p, const double* __restrict__ base,
                                                             long long ldb) {
  const int ntn = (p.M + 63) / 64;
  int ti, tj;
  decode_tile<2>(blockIdx.x, ntn, p.symmetric, ti, tj);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rbase = ti * 128 + (warp >> 1) * 64 + (lane >> 2), cbase = tj * 64 + (warp & 1) * 32 + (lane & 3) * 2;
  const bool vec_ok = ((ldb & 1) == 0) && ((reinterpret_cast<uintptr_t>(base) & 15) == 0);
  double acc[MI][NI][2];
#pragma unroll
  for (int mi = 0; mi < MI; mi++) {
    const int r = rbase + mi * 8;
#pragma unroll
    for (int ni = 0; ni < NI; ni++) {
      const int c = cbase + ni * 8;
      double2 v = make_double2(0.0, 0.0);
      if (r < p.N && (!p.symmetric || c <= r)) {        // the strict upper part of a lower-only base is never read
        const double* src = base + (long long)r * ldb + c;
        if (c + 1 < p.M && vec_ok && (!p.symmetric || c + 1 <= r)) v = *reinterpret_cast<const double2*>(src);
        else {
          if (c < p.M) v.x = src[0];
          if (c + 1 < p.M && (!p.symmetric || c + 1 <= r)) v.y = src[1];
        }
      }
      acc[mi][ni][0] = v.x;
      acc[mi][ni][1] = v.y;
    }
  }
  gram_epilogue<ACT>(p, acc, rbase, cbase);
}

// TMA-fed persistent variant (tma_core.cuh)
template <int ACT>
struct EpiGramTma {
  using Params = GramParams;
  static __device__ __forceinline__ void apply(const Params& p, double (&acc)[MI][NI][2], int r0, int c0, int wm,
                                               int wn, int lane) {
    gram_epilogue<ACT>(p, acc, r0 + wm * 64 + (lane >> 2), c0 + wn * 32 + (lane & 3) * 2);
  }
};

cudaError_t launch_gram_tma(cudaStream_t s, const GramParams& p) {
  CUtensorMap ma, mb;
  if (!make_tmap(&ma, p.X1, p.N, p.D, p.ld1, TM_BM) || !make_tmap(&mb, p.X2, p.M, p.D, p.ld2, TM_BN))
    return cudaErrorInvalidValue;
  TmaShape sh{p.N, p.M, p.D, p.symmetric, count_tiles<TileTma>(p.N, p.M, p.symmetric), 0, 1, 0};
  // L2-aware rasterisation once a tile row's B operand no longer fits the L2 next to everything else (~40 MB)
  const int sr = gram_super_rows();
  if (sr > 0 && (double)p.M * (double)p.D * 8.0 >= (double)dctx().gram_super_min_bytes) {
    sh.super_rows = sr;
    sh.tiles = tma_super_count_tiles(p.N, p.M, p.symmetric, sr);
  }
  cudaError_t e = p.act == ACT_RELU ? launch_tma_gemm<EpiGramTma<ACT_RELU>>(s, ma, mb, sh, p, device_sm_count())
                                    : launch_tma_gemm<EpiGramTma<ACT_ERF>>(s, ma, mb, sh, p, device_sm_count());
  instr().launches++;
  return e;
}

template <typename Cfg, bool ALIGN16>
cudaError_t launch_gram_t(cudaStream_t s, const GramParams& p) {
  long long tiles = count_tiles<Cfg>(p.N, p.M, p.symmetric);
  auto kern = p.act == ACT_RELU ? gram_kernel<Cfg, ALIGN16, ACT_RELU> : gram_kernel<Cfg, ALIGN16, ACT_ERF>;
  cudaError_t e = configure_kernel_once(reinterpret_cast<const void*>(kern), Cfg::SMEM_BYTES, true);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)tiles, Cfg::THREADS, Cfg::SMEM_BYTES, s>>>(p);
  instr().launches++;
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_qtable(cudaStream_t s, const double* X, long long ldx, int N, int D, int n_hidden, int act,
                          int arch, const double* hp, double* tab, long long tab_ld, double* qfin) {
  if (N <= 0) return cudaSuccess;
  int warps_per_block = 8;
  unsigned blocks = (unsigned)((N + warps_per_block - 1) / warps_per_block);
  qtable_kernel<<<blocks, warps_per_block * 32, 0, s>>>(X, ldx, N, D, n_hidden, act, arch, hp, tab, tab_ld, qfin);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_qtable_from_q(cudaStream_t s, const double* q0, int N, int n_hidden, int act, int arch,
                                 const double* hp, double* tab, long long tab_ld, double* qfin) {
  if (N <= 0) return cudaSuccess;
  qtable_from_q_kernel<<<(unsigned)((N + 255) / 256), 256, 0, s>>>(q0, N, n_hidden, act, arch, hp, tab, tab_ld, qfin);
  instr().launches++;
  return cudaGetLastError();
}

// p describes the OUTPUT (tables, hp, shift, symmetric, out_full, K, ldk; X1 / X2 / D are ignored)
cudaError_t launch_gram_from_base(cudaStream_t s, GramParams p, const double* base, long long ldb) {
  if (p.N <= 0 || p.M <= 0) return cudaSuccess;
  p.D = 1;
  const long long tiles = count_tiles<TilePair>(p.N, p.M, p.symmetric);
  if (p.act == ACT_RELU) gram_from_base_kernel<ACT_RELU><<<(unsigned)tiles, 128, 0, s>>>(p, base, ldb);
  else gram_from_base_kernel<ACT_ERF><<<(unsigned)tiles, 128, 0, s>>>(p, base, ldb);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_scalars(cudaStream_t s, const double* qfin, int N, const double* hp, double* scal) {
  scalars_kernel<<<1, 1024, 0, s>>>(qfin, N, hp, scal);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_gram(cudaStream_t s, const GramParams& p) {
  if (p.N <= 0 || p.M <= 0) return cudaSuccess;
  bool a16 = (p.ld1 % 2 == 0) && (p.ld2 % 2 == 0) && ((reinterpret_cast<uintptr_t>(p.X1) & 15) == 0) &&
             ((reinterpret_cast<uintptr_t>(p.X2) & 15) == 0);
  if (tile_variant() == 1) return a16 ? launch_gram_t<TileBig, true>(s, p) : launch_gram_t<TileBig, false>(s, p);
  if (tile_variant() == 0 && tma_operand_ok(p.X1, p.ld1) && tma_operand_ok(p.X2, p.ld2)) return launch_gram_tma(s, p);
  return a16 ? launch_gram_t<TilePair, true>(s, p) : launch_gram_t<TilePair, false>(s, p);
}

}  // namespace smnngp

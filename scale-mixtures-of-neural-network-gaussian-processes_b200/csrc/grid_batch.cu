// Batched grid search (experiments/regression/find.py:134-199 for a whole grid at once, N <= 4096): one persistent
// launch in which every CTA owns a private slot of the workspace and evaluates whole grid points, one after the other,
// with a static stride.  A point never leaves its CTA, so its outputs depend on nothing but its own inputs: they are
// the same bits alone, inside any batch, in any order and with any slot count.
//
// Per point (the outputs of smnngp_grid_point_f64, DESIGN section 3):
//   1. layer tables of the train and test rows for this point's scalars, tr(K)/N by a fixed-order block reduction;
//   2. trapezoid in the slot: rows 0..N-1 = K + eps tr(K)/N I (lower part), rows N..N+T-1 = K_td, row N+T = y^T;
//   3. in-CTA blocked right-looking Cholesky (below) - the carried rows come out as K_td L^-T and (L^-1 y)^T - then
//      mean = K_td L^-T . L^-1 y and var = k_tt - ||K_td L^-T||^2 (NaN when the factorisation failed);
//   4. rows 0..N-1 = K + eps I and row N = y^T again, factor again: sum log L_ii and ||L^-1 y||^2.
//
// Cholesky of a slot (A row-major, lda, rows 0..N-1 lower = the matrix, rows N..M-1 carried), 64-column outer panels:
//   per 16 columns:  the 16 x 16 diagonal block is staged to shared memory and factored + inverted by one warp
//                    (diag_factor_invert, the routine of the blocked factorisation's diagonal kernel); the rows below
//                    are solved in place against inv(L_jj) and the rest of the outer panel is updated, both on DMMA
//                    with 8-row strips per warp straight from global memory (L2);
//   trailing update: rows >= c1 x cols [c1, N), lower part, C -= P P^T with K = 64: 64 x 64 tiles whose two panel
//                    operands are staged by cp.async into shared memory (row stride 68: conflict-free fragments).
#include "chol_core.cuh"
#include "context.cuh"
#include "kernels.cuh"
#include "nngp_math.cuh"

namespace smnngp {

namespace {

constexpr int GB_THREADS = 256;
constexpr int GB_WARPS = GB_THREADS / 32;
constexpr int GB_NB = 64;                  // outer panel width = K of the trailing update
constexpr int GB_TLD = GB_NB + 4;          // 68: row stride of the staged panel tiles
constexpr int GB_SMEM_DOUBLES = DB * GLD + DB * MLD + 2 * GB_NB * GB_TLD + GB_WARPS;
constexpr int GB_SMEM_BYTES = GB_SMEM_DOUBLES * 8 + 16;

__device__ __forceinline__ double qnan_d() { return __longlong_as_double(0x7ff8000000000000ll); }

// K entry from its base value: the recursion of gram_epilogue (gram.cu) on one element, then the final Dense
template <int ACT>
__device__ __forceinline__ double nngp_entry(double k, const double* __restrict__ tab_r, long long ld_r, int r,
                                             const double* __restrict__ tab_c, long long ld_c, int c, int n_act,
                                             bool resnet, double w2, double b2, double v2) {
  if (resnet) k = w2 * k + b2;
  for (int a = 0; a < n_act; a++)
    k = layer_step<ACT>(k, tab_r[a * ld_r + r], tab_c[a * ld_c + c], w2, b2, resnet, !resnet || a == n_act - 1);
  return v2 * k;
}

// rows 0..N-1 (lower) of the slot = K + shift I
template <int ACT>
__device__ void build_gram(const GridBatchParams& p, const double* __restrict__ hp, const double* __restrict__ tab,
                           double* __restrict__ A, double shift) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool resnet = p.arch == ARCH_RESNET;
  const int n_act = n_act_applications(p.n_hidden, p.arch);
  const double w2 = hp[HP_W] * hp[HP_W], b2 = hp[HP_B] * hp[HP_B], v2 = hp[HP_V] * hp[HP_V];
  for (int r = warp; r < p.N; r += GB_WARPS) {
    const double* src = p.K0dd + (long long)r * p.ld0;
    double* dst = A + (long long)r * p.lda;
    for (int c = lane; c <= r; c += 32) {
      double v = nngp_entry<ACT>(src[c], tab, p.N, r, tab, p.N, c, n_act, resnet, w2, b2, v2);
      if (c == r) v += shift;
      dst[c] = v;
    }
  }
}

// rows N..N+T-1 of the slot = K_td
template <int ACT>
__device__ void build_cross(const GridBatchParams& p, const double* __restrict__ hp, const double* __restrict__ tab,
                            const double* __restrict__ tab_t, double* __restrict__ A) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool resnet = p.arch == ARCH_RESNET;
  const int n_act = n_act_applications(p.n_hidden, p.arch);
  const double w2 = hp[HP_W] * hp[HP_W], b2 = hp[HP_B] * hp[HP_B], v2 = hp[HP_V] * hp[HP_V];
  for (int t = warp; t < p.T; t += GB_WARPS) {
    const double* src = p.K0td + (long long)t * p.ld0t;
    double* dst = A + (long long)(p.N + t) * p.lda;
    for (int c = lane; c < p.N; c += 32)
      dst[c] = nngp_entry<ACT>(src[c], tab_t, p.T, t, tab, p.N, c, n_act, resnet, w2, b2, v2);
  }
}

__device__ void copy_row(const double* __restrict__ src, double* __restrict__ dst, int n) {
  for (int i = threadIdx.x; i < n; i += GB_THREADS) dst[i] = src[i];
}

// 8-row strip r0.. of the 16 columns at j0 (w valid) <- strip * inv(L_jj)^T, in place (rows < M)
__device__ __forceinline__ void panel_solve_strip(double* __restrict__ A, long long lda, int M, int r0, int j0, int w,
                                                  const double* __restrict__ Mi, int lane) {
  const int r = r0 + (lane >> 2);
  double* row = A + (long long)r * lda + j0;
  double af[KS];
#pragma unroll
  for (int ks = 0; ks < KS; ks++) {
    const int c = ks * 4 + (lane & 3);
    af[ks] = (r < M && c < w) ? row[c] : 0.0;
  }
  double acc[NT][2];
#pragma unroll
  for (int nt = 0; nt < NT; nt++) {
    acc[nt][0] = acc[nt][1] = 0.0;
    const double* bp = Mi + (nt * 8 + (lane >> 2)) * MLD + (lane & 3);
#pragma unroll
    for (int ks = 0; ks < KS; ks++)
      if (ks <= 2 * nt + 1) dmma8x8x4(acc[nt], af[ks], bp[ks * 4]);   // inv(L) is lower triangular
  }
  __syncwarp();
  if (r < M) {
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
      const int c = nt * 8 + (lane & 3) * 2;
      if (c < w) row[c] = acc[nt][0];
      if (c + 1 < w) row[c + 1] = acc[nt][1];
    }
  }
}

// Cholesky of the slot's leading N x N (lower) with rows N..M-1 carried; returns through *bad_s the 1-based column of
// the first pivot that is not > 0 (0: none) and adds log L_ii of this thread's diagonal entries to lsum
__device__ void factor_slot(double* __restrict__ A, long long lda, int M, int N, double* __restrict__ smem,
                            int* bad_s, double& lsum) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double* Gd = smem;                       // [DB][GLD] staged diagonal block
  double* Mi = Gd + DB * GLD;              // [DB][MLD] its inverse
  double* Pa = Mi + DB * MLD;              // [64][68] panel rows of the output row block
  double* Pb = Pa + GB_NB * GB_TLD;        // [64][68] panel rows of the output column block
  if (tid == 0) *bad_s = 0;
  for (int c0 = 0; c0 < N; c0 += GB_NB) {
    const int c1 = min(c0 + GB_NB, N);
    for (int j0 = c0; j0 < c1; j0 += DB) {
      const int j1 = min(j0 + DB, N), w = j1 - j0;
      for (int i = tid; i < DB * DB; i += GB_THREADS) {
        const int r = i / DB, c = i % DB;
        double v;
        if (r < w) v = c <= r ? A[(long long)(j0 + r) * lda + j0 + c] : 0.0;
        else v = (c == r) ? 1.0 : 0.0;                   // identity padding of a short last block
        Gd[r * GLD + c] = v;
      }
      __syncthreads();
      if (warp == 0) diag_factor_invert(Gd, Mi, lane, j0, bad_s);
      __syncthreads();
      if (tid < w) lsum += log(Gd[tid * GLD + tid]);
      // rows below: solve against inv(L_jj)
      const int nstrips = (M - j1 + 7) / 8;
      for (int s = warp; s < nstrips; s += GB_WARPS) panel_solve_strip(A, lda, M, j1 + s * 8, j0, w, Mi, lane);
      __syncthreads();
      // the rest of the outer panel: C[r][c] -= P[r] . P[c] for j1 <= c < c1, c <= r
      if (j1 < c1) {
        for (int s = warp; s < nstrips; s += GB_WARPS) {
          const int r0 = j1 + s * 8, r = r0 + (lane >> 2);
          double af[KS];
#pragma unroll
          for (int ks = 0; ks < KS; ks++) {
            const int c = ks * 4 + (lane & 3);
            af[ks] = (r < M && c < w) ? A[(long long)r * lda + j0 + c] : 0.0;
          }
          for (int ct = j1; ct < c1 && ct <= r0 + 7; ct += 8) {
            const int rc = ct + (lane >> 2);                // B fragment: panel row of output column rc
            double acc[2] = {0.0, 0.0};
#pragma unroll
            for (int ks = 0; ks < KS; ks++) {
              const int c = ks * 4 + (lane & 3);
              const double b = (rc < c1 && c < w) ? A[(long long)rc * lda + j0 + c] : 0.0;
              dmma8x8x4(acc, af[ks], b);
            }
            const int cc = ct + (lane & 3) * 2;
            if (r < M) {
              double* dst = A + (long long)r * lda + cc;
              if (cc < c1 && cc <= r) dst[0] -= acc[0];
              if (cc + 1 < c1 && cc + 1 <= r) dst[1] -= acc[1];
            }
          }
        }
        __syncthreads();
      }
    }
    if (c1 >= N) break;
    // trailing update with the whole outer panel (K = 64 exactly: only the last panel is narrower, and it has none)
    const int wm = warp >> 2, wn = warp & 3;       // warp tile: rows wm*32 .. +32, cols wn*16 .. +16
    for (int rb = c1; rb < M; rb += GB_NB) {
      for (int i = tid; i < GB_NB * (GB_NB / 2); i += GB_THREADS) {
        const int r = i / (GB_NB / 2), c = (i % (GB_NB / 2)) * 2;
        const bool ok = rb + r < M;
        cp_async16(Pa + r * GB_TLD + c, A + (long long)(ok ? rb + r : c0) * lda + c0 + c, ok ? 16 : 0);
      }
      for (int cb = c1; cb < N && cb <= rb + GB_NB - 1; cb += GB_NB) {
        for (int i = tid; i < GB_NB * (GB_NB / 2); i += GB_THREADS) {
          const int r = i / (GB_NB / 2), c = (i % (GB_NB / 2)) * 2;
          const bool ok = cb + r < N;
          cp_async16(Pb + r * GB_TLD + c, A + (long long)(ok ? cb + r : c0) * lda + c0 + c, ok ? 16 : 0);
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        const int r_lo = rb + wm * 32, c_lo = cb + wn * 16;
        if (c_lo <= r_lo + 31 && r_lo < M && c_lo < N) {   // warp tile not entirely above the diagonal / outside
          double acc[4][2][2];
#pragma unroll
          for (int mi = 0; mi < 4; mi++)
#pragma unroll
            for (int ni = 0; ni < 2; ni++) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
          const double* ap = Pa + (wm * 32 + (lane >> 2)) * GB_TLD + (lane & 3);
          const double* bp = Pb + (wn * 16 + (lane >> 2)) * GB_TLD + (lane & 3);
#pragma unroll 4
          for (int ks = 0; ks < GB_NB / 4; ks++) {
            double a[4], b[2];
#pragma unroll
            for (int mi = 0; mi < 4; mi++) a[mi] = ap[mi * 8 * GB_TLD + ks * 4];
#pragma unroll
            for (int ni = 0; ni < 2; ni++) b[ni] = bp[ni * 8 * GB_TLD + ks * 4];
#pragma unroll
            for (int mi = 0; mi < 4; mi++)
#pragma unroll
              for (int ni = 0; ni < 2; ni++) dmma8x8x4(acc[mi][ni], a[mi], b[ni]);
          }
#pragma unroll
          for (int mi = 0; mi < 4; mi++) {
            const int r = r_lo + mi * 8 + (lane >> 2);
            if (r >= M) continue;
#pragma unroll
            for (int ni = 0; ni < 2; ni++) {
              const int c = c_lo + ni * 8 + (lane & 3) * 2;
              double* dst = A + (long long)r * lda + c;
              if (c < N && c <= r) dst[0] -= acc[mi][ni][0];
              if (c + 1 < N && c + 1 <= r) dst[1] -= acc[mi][ni][1];
            }
          }
        }
        __syncthreads();                               // Pb (and, after the last column block, Pa) is free again
      }
    }
  }
}

template <int ACT>
__global__ void __launch_bounds__(GB_THREADS, 2) grid_batch_kernel(const GridBatchParams p) {
  extern __shared__ __align__(16) double smem[];
  double* red = smem + GB_SMEM_DOUBLES - GB_WARPS;
  int* bad_s = reinterpret_cast<int*>(smem + GB_SMEM_DOUBLES);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  char* slot = p.ws + (long long)blockIdx.x * p.slot_bytes;
  double* A = reinterpret_cast<double*>(slot);
  double* tab = reinterpret_cast<double*>(slot) + p.off_tab;
  double* q = reinterpret_cast<double*>(slot) + p.off_q;
  double* tab_t = reinterpret_cast<double*>(slot) + p.off_tab_t;
  double* q_t = reinterpret_cast<double*>(slot) + p.off_q_t;
  const int N = p.N, T = p.T;

  for (int g = blockIdx.x; g < p.G; g += gridDim.x) {
    const double* hp = p.hp + (long long)g * HP_COUNT;
    // 1. layer tables and tr(K)/N
    double qs = 0.0;
    for (int r = tid; r < N; r += GB_THREADS) {
      fill_row_tables(p.q_d[r], r, p.n_hidden, ACT, p.arch, hp, tab, N, q);
      qs += q[r];
    }
    for (int t = tid; t < T; t += GB_THREADS) fill_row_tables(p.q_t[t], t, p.n_hidden, ACT, p.arch, hp, tab_t, T, q_t);
    const double trmean = block_sum<GB_THREADS>(qs, red) / (double)N;   // its __syncthreads also publishes the tables
    const double eps = hp[HP_EPS];

    // 2. + 3. predictive with the relative regulariser
    build_gram<ACT>(p, hp, tab, A, eps * trmean);
    build_cross<ACT>(p, hp, tab, tab_t, A);
    copy_row(p.y, A + (long long)(N + T) * p.lda, N);
    __syncthreads();
    double lsum = 0.0;
    factor_slot(A, p.lda, N + T + 1, N, smem, bad_s, lsum);
    __syncthreads();
    const int bad1 = *bad_s;
    const double* z = A + (long long)(N + T) * p.lda;
    for (int t = warp; t < T; t += GB_WARPS) {
      const double* v = A + (long long)(N + t) * p.lda;
      double vv = 0.0, vz = 0.0;
      for (int n = lane; n < N; n += 32) {
        const double x = v[n];
        vv = fma(x, x, vv);
        vz = fma(x, z[n], vz);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        vv += __shfl_xor_sync(0xffffffffu, vv, o);
        vz += __shfl_xor_sync(0xffffffffu, vz, o);
      }
      if (lane == 0) {
        p.var[(long long)g * T + t] = bad1 ? qnan_d() : q_t[t] - vv;
        p.mean[(long long)g * T + t] = bad1 ? qnan_d() : vz;
      }
    }
    __syncthreads();

    // 4. log det(K + eps I) and y^T (K + eps I)^-1 y with the absolute regulariser
    build_gram<ACT>(p, hp, tab, A, eps);
    copy_row(p.y, A + (long long)N * p.lda, N);
    __syncthreads();
    lsum = 0.0;
    factor_slot(A, p.lda, N + 1, N, smem, bad_s, lsum);
    __syncthreads();
    const int bad2 = *bad_s;
    const double logdet = block_sum<GB_THREADS>(lsum, red);
    double zz = 0.0;
    for (int n = tid; n < N; n += GB_THREADS) {
      const double x = A[(long long)N * p.lda + n];
      zz = fma(x, x, zz);
    }
    const double quad = block_sum<GB_THREADS>(zz, red);
    if (tid == 0) {
      const bool bad = bad1 != 0 || bad2 != 0;
      p.out[2ll * g] = bad ? qnan_d() : logdet;
      p.out[2ll * g + 1] = bad ? qnan_d() : quad;
      p.info[g] = bad1 ? bad1 : bad2;
    }
    __syncthreads();                                   // the slot and bad_s are reused by the next point
  }
}

}  // namespace

cudaError_t launch_grid_batch(cudaStream_t s, const GridBatchParams& p, int act, long long slots) {
  auto kern = act == ACT_RELU ? grid_batch_kernel<ACT_RELU> : grid_batch_kernel<ACT_ERF>;
  cudaError_t e = configure_kernel_once(reinterpret_cast<const void*>(kern), GB_SMEM_BYTES, false);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)(slots < p.G ? slots : p.G), GB_THREADS, GB_SMEM_BYTES, s>>>(p);
  instr().launches++;
  return cudaGetLastError();
}

}  // namespace smnngp

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
//   Both factorisations are factor_slot (slot_chol.cuh).
#include "context.cuh"
#include "slot_chol.cuh"

namespace smnngp {

namespace {

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
    factor_slot<false>(A, p.lda, N + T + 1, N, smem, bad_s, lsum);
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
    factor_slot<false>(A, p.lda, N + 1, N, smem, bad_s, lsum);
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

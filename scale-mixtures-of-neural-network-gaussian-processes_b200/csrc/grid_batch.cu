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
//   Steps 1 - 3 are predictive_slot, both factorisations factor_slot (slot_chol.cuh).
#include "context.cuh"
#include "slot_chol.cuh"

namespace smnngp {

namespace {

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
    // 1. - 3. layer tables, tr(K)/N and the predictive with the relative regulariser
    double eps;
    const int bad1 = predictive_slot<ACT>(p, hp, A, tab, q, tab_t, q_t, smem, red, bad_s, tid, lane, warp, N, T, eps,
                                          [&](int t, double vv, double vz, int bad) {
                                            p.var[(long long)g * T + t] = bad ? qnan_d() : q_t[t] - vv;
                                            p.mean[(long long)g * T + t] = bad ? qnan_d() : vz;
                                          });

    // 4. log det(K + eps I) and y^T (K + eps I)^-1 y with the absolute regulariser
    build_gram<ACT>(p, hp, tab, A, eps);
    copy_row(p.y, A + (long long)N * p.lda, N);
    __syncthreads();
    double lsum = 0.0;
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

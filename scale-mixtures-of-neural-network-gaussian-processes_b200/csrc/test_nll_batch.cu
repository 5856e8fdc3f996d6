// Batched test NLL (N <= 4096): SPR.test_nll (what smnngp_test_nll_f64 returns) at G hyper-parameter points in one
// persistent launch - the validation and test evaluations of multi-start training (experiments/regression/train.py:
// 194-212 for every restart) and the selection of grid points by held-out NLL, at the sizes where one
// smnngp_test_nll_f64 call leaves the GPU nearly idle.  Every CTA owns a private slot of the workspace and evaluates
// whole points, one after the other, with a static stride.  A point never leaves its CTA and every reduction has a
// fixed order, so its outputs are the same bits alone, inside any batch, in any order and with any slot count.
//
// Per point (DESIGN section 3, spax/models.py:100-120):
//   1. + 2. predictive_slot (slot_chol.cuh): layer tables, tr(K)/N, K + eps tr(K)/N I | K_td | y^T factorised, and per
//      test row mean = v . z and var = k_tt - ||v||^2 into the slot's [2][T] scratch (and the optional outputs);
//   3. Student-t only: rows 0..N-1 = K + 1e-6 (alpha/beta) I, row N = y^T, factor_slot, quad2 = ||L2^-1 y||^2;
//   4. per test row the log density of test_nll_finalize (closed_forms.cuh), nll = -(sum_t lp_t) / T.
//   The scratch makes nll the same bits whether or not mean, var and logp are asked for.
#include "closed_forms.cuh"
#include "context.cuh"
#include "slot_chol.cuh"

namespace smnngp {

namespace {

template <int ACT>
__global__ void __launch_bounds__(GB_THREADS, 2) test_nll_batch_kernel(const TestNllBatchParams p) {
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
  double* mv = reinterpret_cast<double*>(slot) + p.off_mv;   // [0, T): mean, [T, 2T): var
  const int N = p.N, T = p.T;

  for (int g = blockIdx.x; g < p.G; g += gridDim.x) {
    const double* hp = p.hp + (long long)g * HP_COUNT;
    // 1. + 2. the predictive with the relative regulariser
    double eps;
    const int bad1 = predictive_slot<ACT>(p, hp, A, tab, q, tab_t, q_t, smem, red, bad_s, tid, lane, warp, N, T, eps,
                                          [&](int t, double vv, double vz, int bad) {
                                            const double var = q_t[t] - vv;
                                            mv[t] = vz;
                                            mv[T + t] = var;
                                            const long long o = (long long)g * T + t;
                                            if (p.mean) p.mean[o] = bad ? qnan_d() : vz;
                                            if (p.var) p.var[o] = bad ? qnan_d() : var;
                                          });

    // 3. Student-t scale: y^T (K + 1e-6 (a/b) I)^-1 y (the shift of scalars_kernel, SHIFT_LIK)
    int bad2 = 0;
    double quad2 = 0.0;
    if (p.kind == KIND_STUDENT_T) {
      build_gram<ACT>(p, hp, tab, A, 1e-6 * hp[HP_ALPHA] / hp[HP_BETA]);
      copy_row(p.y, A + (long long)N * p.lda, N);
      __syncthreads();
      double lsum = 0.0;
      factor_slot<false>(A, p.lda, N + 1, N, smem, bad_s, lsum);
      __syncthreads();
      bad2 = *bad_s;
      double zz = 0.0;
      for (int n = tid; n < N; n += GB_THREADS) {
        const double x = A[(long long)N * p.lda + n];
        zz = fma(x, x, zz);
      }
      quad2 = block_sum<GB_THREADS>(zz, red);
    }

    // 4. log density per test row (de-standardised), nll = -mean
    const bool bad = bad1 != 0 || bad2 != 0;
    double acc = 0.0;
    for (int t = tid; t < T; t += GB_THREADS) {
      const double x = p.yt[t] * p.y_std + p.y_mean;
      const double m = mv[t] * p.y_std + p.y_mean;
      const double cv = mv[T + t] * (p.y_std * p.y_std);
      double lp = test_logpdf(x, m, cv, hp, p.kind, N, &quad2);
      if (bad) lp = qnan_d();
      if (p.logp) p.logp[(long long)g * T + t] = lp;
      acc += lp;
    }
    const double s = block_sum<GB_THREADS>(acc, red);
    if (tid == 0) {
      p.nll[g] = -s / (double)T;
      p.info[g] = bad1 ? bad1 : bad2;
    }
    __syncthreads();                                   // the slot, its scratch and bad_s are reused by the next point
  }
}

}  // namespace

cudaError_t launch_test_nll_batch(cudaStream_t s, const TestNllBatchParams& p, int act, long long slots) {
  auto kern = act == ACT_RELU ? test_nll_batch_kernel<ACT_RELU> : test_nll_batch_kernel<ACT_ERF>;
  cudaError_t e = configure_kernel_once(reinterpret_cast<const void*>(kern), GB_SMEM_BYTES, false);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)(slots < p.G ? slots : p.G), GB_THREADS, GB_SMEM_BYTES, s>>>(p);
  instr().launches++;
  return cudaGetLastError();
}

}  // namespace smnngp

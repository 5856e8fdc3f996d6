// Scalar tails of the hot path: ||L^-1 y||^2, the closed-form Student-t / Gaussian log marginal likelihood
// (spax/utils.py:181-183, spax/likelihoods.py:25-28, :45-50, spax/models.py:98), the predictive mean /
// variance (neural_tangents predict as used at spax/kernels.py:29-32; only diag(cov) is consumed downstream,
// spax/likelihoods.py:31,62) and the per-test-point log density (spax/likelihoods.py:52-65, :30-33).
// All reductions run in a fixed order (deterministic).
#include "closed_forms.cuh"
#include "kernels.cuh"

namespace smnngp {

namespace {

__device__ __forceinline__ double qnan() { return __longlong_as_double(0x7ff8000000000000ll); }

__global__ void sumsq_kernel(const double* __restrict__ z, long long n, double* __restrict__ out) {
  __shared__ double red[32];
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
  long long i = threadIdx.x;
  for (; i + 3 * 1024 < n; i += 4 * 1024) {
    double x0 = z[i], x1 = z[i + 1024], x2 = z[i + 2048], x3 = z[i + 3072];
    a0 = fma(x0, x0, a0); a1 = fma(x1, x1, a1); a2 = fma(x2, x2, a2); a3 = fma(x3, x3, a3);
  }
  for (; i < n; i += 1024) { double x = z[i]; a0 = fma(x, x, a0); }
  double s = block_sum<1024>((a0 + a1) + (a2 + a3), red);
  if (threadIdx.x == 0) *out = s;
}

__global__ void lml_finalize_kernel(const double* __restrict__ scal, const double* __restrict__ hp, int kind,
                                    long long N, const int* __restrict__ info, double* __restrict__ out) {
  lml_closed_form(scal[SC_LOGDET], scal[SC_QUAD], hp, kind, N, info, out);
}

constexpr int PRED_MAXC = 16;
// one CTA per test row: var = k_tt - ||v||^2, mean_c = v . z_c
__global__ void __launch_bounds__(256) predict_finalize_kernel(const double* __restrict__ V, long long ldv,
                                                               const double* __restrict__ Z, long long ldz,
                                                               const double* __restrict__ ktt, int C,
                                                               long long N, const int* __restrict__ info,
                                                               double* __restrict__ mean,
                                                               double* __restrict__ var) {
  __shared__ double red[32];
  const int t = blockIdx.x;
  const double* v = V + (long long)t * ldv;
  const bool bad = *info != 0;
  for (int cb = 0; cb < C || cb == 0; cb += PRED_MAXC) {
    const int nc = min(PRED_MAXC, C - cb);
    double vv = 0.0, vz[PRED_MAXC];
#pragma unroll
    for (int c = 0; c < PRED_MAXC; c++) vz[c] = 0.0;
    for (long long n = threadIdx.x; n < N; n += 256) {
      const double x = v[n];
      vv = fma(x, x, vv);
#pragma unroll
      for (int c = 0; c < PRED_MAXC; c++)
        if (c < nc) vz[c] = fma(x, Z[(long long)(cb + c) * ldz + n], vz[c]);
    }
    if (cb == 0) {
      double s = block_sum<256>(vv, red);
      if (threadIdx.x == 0) var[t] = bad ? qnan() : ktt[t] - s;
    }
    for (int c = 0; c < nc; c++) {
      double s = block_sum<256>(vz[c], red);
      if (threadIdx.x == 0) mean[(long long)t * C + cb + c] = bad ? qnan() : s;
    }
    if (C == 0) break;
  }
}

__global__ void __launch_bounds__(1024) test_nll_finalize_kernel(
    const double* __restrict__ mean, const double* __restrict__ var, const double* __restrict__ ytest, int T,
    long long N, double y_mean, double y_std, const double* __restrict__ hp, int kind,
    const double* __restrict__ quad2, const int* __restrict__ info, double* __restrict__ logp,
    double* __restrict__ nll_out) {
  __shared__ double red[32];
  const bool bad = *info != 0;
  double acc = 0.0;
  for (int t = threadIdx.x; t < T; t += 1024) {
    const double x = ytest[t] * y_std + y_mean;
    const double m = mean[t] * y_std + y_mean;
    const double cv = var[t] * (y_std * y_std);
    double lp = test_logpdf(x, m, cv, hp, kind, N, quad2);
    if (bad) lp = qnan();
    if (logp) logp[t] = lp;
    acc += lp;
  }
  double s = block_sum<1024>(acc, red);
  if (threadIdx.x == 0) *nll_out = -s / (double)T;
}

__global__ void fill_nan_if_bad_kernel(const int* __restrict__ info, double* __restrict__ buf, long long n) {
  if (*info == 0) return;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    buf[i] = qnan();
}

}  // namespace

cudaError_t launch_sumsq(cudaStream_t s, const double* z, long long n, double* out) {
  sumsq_kernel<<<1, 1024, 0, s>>>(z, n, out);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_lml_finalize(cudaStream_t s, const double* scal, const double* hp, int kind, long long N,
                                const int* info, double* out) {
  lml_finalize_kernel<<<1, 1, 0, s>>>(scal, hp, kind, N, info, out);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_predict_finalize(cudaStream_t s, const double* V, long long ldv, const double* Z,
                                    long long ldz, const double* ktt, int T, int C, long long N,
                                    const int* info, double* mean, double* var) {
  if (T <= 0) return cudaSuccess;
  predict_finalize_kernel<<<T, 256, 0, s>>>(V, ldv, Z, ldz, ktt, C, N, info, mean, var);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_test_nll_finalize(cudaStream_t s, const double* mean, const double* var, const double* ytest,
                                     int T, long long N, double y_mean, double y_std, const double* hp,
                                     int kind, const double* quad2, const int* info, double* logp,
                                     double* nll_out) {
  test_nll_finalize_kernel<<<1, 1024, 0, s>>>(mean, var, ytest, T, N, y_mean, y_std, hp, kind, quad2, info, logp,
                                              nll_out);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_fill_nan_if_bad(cudaStream_t s, const int* info, double* buf, long long n) {
  if (n <= 0) return cudaSuccess;
  long long blocks = (n + 255) / 256;
  if (blocks > 1184) blocks = 1184;
  fill_nan_if_bad_kernel<<<(unsigned)blocks, 256, 0, s>>>(info, buf, n);
  instr().launches++;
  return cudaGetLastError();
}


// ---- instrumentation ---------------------------------------------------------------------------------------
namespace {
template <int NACC>
__global__ void dmma_peak_kernel(double* out, int iters, double seed) {
  double c[NACC][2];
#pragma unroll
  for (int i = 0; i < NACC; i++) c[i][0] = c[i][1] = 0.0;
  double a = seed + threadIdx.x * 1e-9, b = seed - threadIdx.x * 1e-9;
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int i = 0; i < NACC; i++)
      asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+d"(c[i][0]), "+d"(c[i][1]) : "d"(a), "d"(b));
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < NACC; i++) s += c[i][0] + c[i][1];
  if (s == 123.456) out[0] = s;
}
}  // namespace

double dmma_peak_tflops(int sms) {
  double* d = nullptr;
  if (cudaMalloc(&d, 64) != cudaSuccess) return -1.0;
  const int iters = 20000, threads = 256;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  float best = 1e30f;
  for (int r = 0; r < 4; r++) {
    cudaEventRecord(e0);
    dmma_peak_kernel<16><<<sms, threads>>>(d, iters, 1.0);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms;
    cudaEventElapsedTime(&ms, e0, e1);
    if (r > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  const double flop = 2.0 * 8 * 8 * 4 * 16.0 * iters * (threads / 32) * sms;
  return flop / best * 1e-9;
}

}  // namespace smnngp

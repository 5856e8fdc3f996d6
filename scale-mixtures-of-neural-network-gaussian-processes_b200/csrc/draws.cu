// Posterior draw stage of the classification / ensemble configuration (SURVEY.md section 8f, row N2):
//   InverseGammaPrior.sample_f_iid (spax/priors.py:60-68):  f[c,t,s] = mean[c,t] + sqrt((b/a) var[c,t]) * T_{2a}
//   GaussianPrior.sample_f_iid     (spax/priors.py:30-36):  f[c,t,s] = mean[c,t] + sqrt(var[c,t]) * N(0,1)
//   test_log_likelihood (spax/utils.py:61-66), get_correct_count (spax/utils.py:69-74)
// Two kernels share ONE counter-based generator (Philox4x32-10 keyed by seed, counter = (sample, test point,
// class)): `sample_f_iid` materialises the draws, `draw_metrics` fuses draw -> log-softmax -> online log-sum-exp
// so that for S = 10^4 draws x T = 10^4 points x C = 10 classes nothing but the T results ever touches HBM.
// Because the generator is counter based the fused kernel sees exactly the draws the materialising one writes,
// which is what the parity test relies on.  (Bit parity with JAX's threefry stream is not a goal.)
#include "kernels.cuh"
#include "philox.cuh"

namespace smnngp {

namespace {

// sigma of the draw for (class c, point t): student -> sqrt((b/a) var), gaussian -> sqrt(var)
__device__ __forceinline__ double draw_value(CellRng& rng, double mean, double sigma, int kind, double df) {
  const double e = (kind == KIND_STUDENT_T) ? rng.student_t(df) : rng.normal();
  return fma(e, sigma, mean);
}

__global__ void sample_f_iid_kernel(const double* __restrict__ mean, const double* __restrict__ var, int var_per_class,
                                    int T, int C, int S, const double* __restrict__ hp, int kind, uint32_t k0,
                                    uint32_t k1, double* __restrict__ out) {
  const long long total = (long long)C * T * S;
  const double a = hp[HP_ALPHA], b = hp[HP_BETA];
  const double scale = (kind == KIND_STUDENT_T) ? b / a : 1.0, df = 2.0 * a;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int s = (int)(i % S);
    const int t = (int)((i / S) % T);
    const int c = (int)(i / ((long long)S * T));
    const double v = var_per_class ? var[(long long)c * T + t] : var[t];
    CellRng rng(k0, k1, (uint32_t)s, (uint32_t)t, (uint32_t)c);
    out[i] = draw_value(rng, mean[(long long)t * C + c], sqrt(scale * v), kind, df);   // out [C, T, S]
  }
}

// one CTA per test point; threads stride over the S samples; C+... online LSEs per thread, merged in a fixed order
__global__ void __launch_bounds__(256)
draw_metrics_kernel(const double* __restrict__ mean, const double* __restrict__ var, int var_per_class,
                    const int* __restrict__ label, int T, int C, int S, const double* __restrict__ hp, int kind,
                    uint32_t k0, uint32_t k1, double* __restrict__ ll_per_test, int* __restrict__ pred) {
  __shared__ double sm_m[256], sm_s[256];
  const int t = blockIdx.x;
  const double a = hp[HP_ALPHA], b = hp[HP_BETA];
  const double scale = (kind == KIND_STUDENT_T) ? b / a : 1.0, df = 2.0 * a;
  double mu[DRAW_MAXC], sg[DRAW_MAXC];
#pragma unroll
  for (int c = 0; c < DRAW_MAXC; c++) {
    mu[c] = c < C ? mean[(long long)t * C + c] : 0.0;
    sg[c] = c < C ? sqrt(scale * (var_per_class ? var[(long long)c * T + t] : var[t])) : 0.0;
  }
  const int y = label[t];
  Lse acc[DRAW_MAXC];
#pragma unroll
  for (int c = 0; c < DRAW_MAXC; c++) acc[c].init();
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    double f[DRAW_MAXC];
    double fmaxv = -INFINITY;
#pragma unroll
    for (int c = 0; c < DRAW_MAXC; c++) {
      if (c < C) {
        CellRng rng(k0, k1, (uint32_t)s, (uint32_t)t, (uint32_t)c);
        f[c] = draw_value(rng, mu[c], sg[c], kind, df);
        fmaxv = fmax(fmaxv, f[c]);
      }
    }
    double se = 0.0;
#pragma unroll
    for (int c = 0; c < DRAW_MAXC; c++)
      if (c < C) se += exp(f[c] - fmaxv);
    const double lse = fmaxv + log(se);                 // log_softmax over classes (axis 0 in the reference)
#pragma unroll
    for (int c = 0; c < DRAW_MAXC; c++)
      if (c < C) acc[c].add(f[c] - lse);
  }
  // fixed-order merge over the block, one class at a time
  double best = -INFINITY, ll_true = __longlong_as_double(0x7ff8000000000000ll);   // stays NaN if y is not in [0, C)
  int best_c = 0;
  for (int c = 0; c < C; c++) {
    double m = -INFINITY, s = 0.0;
#pragma unroll
    for (int cc = 0; cc < DRAW_MAXC; cc++)
      if (cc == c) { m = acc[cc].m; s = acc[cc].s; }
    sm_m[threadIdx.x] = m;
    sm_s[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      Lse tot;
      tot.init();
      for (int k = 0; k < (int)blockDim.x; k++) tot.merge(sm_m[k], sm_s[k]);
      const double v = tot.value();                    // logsumexp over samples of log_softmax[c, t, :]
      if (v > best) { best = v; best_c = c; }          // argmax over classes, first maximum (jnp.argmax)
      if (c == y) ll_true = v - log((double)S);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    ll_per_test[t] = ll_true;
    pred[t] = best_c;
  }
}

__global__ void draw_finalize_kernel(const double* __restrict__ ll_per_test, const int* __restrict__ pred,
                                     const int* __restrict__ label, int T, double* __restrict__ out) {
  __shared__ double red[1024];
  __shared__ int redc[1024];
  double s = 0.0;
  int c = 0;
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    s += ll_per_test[t];
    c += (pred[t] == label[t]) ? 1 : 0;
  }
  red[threadIdx.x] = s;
  redc[threadIdx.x] = c;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { red[threadIdx.x] += red[threadIdx.x + o]; redc[threadIdx.x] += redc[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[0] = -red[0] / (double)T;      // nll = -mean_t( logsumexp_s - log S )
    out[1] = (double)redc[0];          // correct count
  }
}

}  // namespace

cudaError_t launch_sample_f_iid(cudaStream_t s, const double* mean, const double* var, int var_per_class, int T, int C,
                                int S, const double* hp, int kind, uint64_t seed, double* out) {
  const long long total = (long long)C * T * S;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  sample_f_iid_kernel<<<(unsigned)blocks, 256, 0, s>>>(mean, var, var_per_class, T, C, S, hp, kind, (uint32_t)seed,
                                                       (uint32_t)(seed >> 32), out);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_draw_metrics(cudaStream_t s, const double* mean, const double* var, int var_per_class,
                                const int* label, int T, int C, int S, const double* hp, int kind, uint64_t seed,
                                double* ll_per_test, int* pred, double* out) {
  draw_metrics_kernel<<<(unsigned)T, 256, 0, s>>>(mean, var, var_per_class, label, T, C, S, hp, kind, (uint32_t)seed,
                                                  (uint32_t)(seed >> 32), ll_per_test, pred);
  instr().launches++;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  draw_finalize_kernel<<<1, 1024, 0, s>>>(ll_per_test, pred, label, T, out);
  instr().launches++;
  return cudaGetLastError();
}

}  // namespace smnngp

// Scale mixture of NNGPs under a prior without a conjugate form (the reference's find.py:163-191 importance-sampling
// table): a scale s > 0 multiplies the whole covariance, y | s ~ N(0, s A), f_t | y, s ~ N(m_t, s v_t), and the
// posterior over s is represented by S draws s_j from the prior, weighted by their likelihood
//   l_j = -(N/2) log s_j - quad / (2 s_j)                    (quad = y^T A^-1 y; l_j = -inf for s_j = 0 or +inf)
//   lml = logsumexp_j l_j - log S - sum log L_ii - (N/2) log 2 pi
//   logp_t = logsumexp_j [l_j + log N(y~_t; m~_t, s_j v~_t)] - logsumexp_j l_j          (de-standardised as test_nll)
//   ess = (sum_j w_j)^2 / sum_j w_j^2,  w_j = exp(l_j - max l)
// `scale_draws` fills the draws from the same counter-based Philox stream as the posterior draw stage (draws.cu), with
// the counter (j, p, 0xFFFFFFFF, n) that sample_f_iid never uses; `mixture_nll` evaluates every (grid point g, prior
// row p) pair of the table in one launch.
#include "kernels.cuh"
#include "philox.cuh"

namespace smnngp {

namespace {

constexpr int MIX_WARPS = 8;   // warps per CTA; a warp evaluates one (g, p) pair at a time
constexpr int MIX_TPL = 4;     // test points per lane in one pass over the draws
constexpr double kLog2Pi = 1.8378770664093454836;

__global__ void scale_draws_kernel(int family, const double* __restrict__ params, long long P, long long S,
                                   uint32_t k0, uint32_t k1, double* __restrict__ out) {
  const long long total = P * S;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long p = i / S, j = i % S;
    const double a = params[2 * p], b = params[2 * p + 1];
    double s = __longlong_as_double(0x7ff8000000000000ll);            // NaN for a row that is not a valid prior
    if (a > 0.0 && b > 0.0 && a < INFINITY && b < INFINITY) {
      CellRng rng(k0, k1, (uint32_t)j, (uint32_t)p, 0xFFFFFFFFu);
      if (family == SCALE_INVGAMMA) s = b / rng.gamma(a);                 // IG(a, b): b / Gamma(a, 1)
      else s = exp(log(expm1(-log(rng.uniform()) / b)) / a);             // Burr XII (c, k) by inversion of its CDF
    }
    out[i] = s;
  }
}

// log-sum-exp steps that keep exactly what they must: a term of -inf adds nothing (Lse::add would turn it into NaN
// while the accumulator is empty), a NaN is never dropped (Lse::merge would drop one held with m = -inf)
__device__ __forceinline__ void lse_add(Lse& acc, double x) {
  if (x != -INFINITY) acc.add(x);
}
__device__ __forceinline__ void lse_merge(Lse& acc, double m2, double s2) {
  const bool nan = isnan(acc.s) || isnan(s2);
  acc.merge(m2, s2);
  if (nan) acc.s = __longlong_as_double(0x7ff8000000000000ll);
}
// fixed-order tree over the 32 lanes of a warp; the result is in lane 0
__device__ __forceinline__ void lse_warp_merge(Lse& acc) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const double m2 = __shfl_down_sync(0xffffffffu, acc.m, d), s2 = __shfl_down_sync(0xffffffffu, acc.s, d);
    lse_merge(acc, m2, s2);
  }
}

// the per-draw quantities of pair (g, p): l_j and the log-density offset a_j = l_j - max_l - log(s_j) / 2, with
// 1 / (2 s_j); for s_j in {0, +inf} the draw has zero weight (l = a = -inf, 1 / (2 s) = 0 keeps the FMA finite)
__device__ __forceinline__ double draw_ell(double s, double hN, double quad, double& ls, double& i2s) {
  if (s == 0.0 || s == INFINITY) { ls = 0.0; i2s = 0.0; return -INFINITY; }
  ls = log(s);
  i2s = 0.5 / s;
  return fma(-hN, ls, -(quad * i2s));
}

__global__ void __launch_bounds__(32 * MIX_WARPS)
mixture_nll_kernel(MixtureParams p) {
  __shared__ double2 hoisted[MIX_WARPS][32];                          // (a_j, 1 / (2 s_j)) of 32 consecutive draws
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const double hN = 0.5 * (double)p.N, nan = __longlong_as_double(0x7ff8000000000000ll);
  const long long pairs = p.G * p.P;
  for (long long pr = (long long)blockIdx.x * MIX_WARPS + w; pr < pairs; pr += (long long)gridDim.x * MIX_WARPS) {
    const long long g = pr / p.P, q = pr % p.P;
    const double logdet = p.scal[2 * g], quad = p.scal[2 * g + 1];
    const bool bad = isnan(logdet) || isnan(quad);
    const double* __restrict__ d = p.draws + q * p.S;
    // evidence: lane k takes the draws j = k (mod 32) in order, then the fixed-order tree; the two accumulators see
    // the same comparisons, so ev2.m = 2 ev.m and ess = ev.s^2 / ev2.s is (sum w)^2 / sum w^2 with w = exp(l - max l)
    Lse ev, ev2;
    ev.init();
    ev2.init();
    for (long long j = lane; j < p.S; j += 32) {
      double ls, i2s;
      const double l = draw_ell(d[j], hN, quad, ls, i2s);
      lse_add(ev, l);
      lse_add(ev2, 2.0 * l);
    }
    lse_warp_merge(ev);
    lse_warp_merge(ev2);
    // (when every weight is zero mmax = -inf and each a_j is NaN: logp and nll come out NaN, as they must)
    const double mmax = __shfl_sync(0xffffffffu, ev.m, 0);
    const double log_s1 = __shfl_sync(0xffffffffu, log(ev.s), 0);    // log sum_j exp(l_j - max l)
    if (lane == 0) {
      const bool empty = (ev.m == -INFINITY && ev.s == 0.0);
      p.lml[pr] = bad ? nan : ev.value() - log((double)p.S) - logdet - hN * kLog2Pi;
      p.ess[pr] = bad ? nan : (empty ? 0.0 : ev.s * ev.s / ev2.s);
    }
    // test points: lane k holds t = t0 + k + 32 i (i < MIX_TPL) and runs through all draws in order, 32 at a time,
    // each chunk's a_j and 1 / (2 s_j) computed once by the warp; then logp_t and a fixed-order sum for the nll
    double nsum = 0.0;
    for (long long t0 = 0; t0 < p.T; t0 += 32 * MIX_TPL) {
      double r[MIX_TPL], c[MIX_TPL];
      Lse acc[MIX_TPL];
#pragma unroll
      for (int i = 0; i < MIX_TPL; i++) {
        const long long t = t0 + lane + 32 * i;
        acc[i].init();
        r[i] = 0.0;
        c[i] = 0.0;
        if (t < p.T) {
          const double ys = p.y_std;
          const double yt = p.yt[t] * ys + p.y_mean, m = p.mean[g * p.ld + t] * ys + p.y_mean;
          const double v = p.var[g * p.ld + t] * (ys * ys);
          const double e = yt - m;
          r[i] = e * e / v;
          c[i] = -0.5 * kLog2Pi - 0.5 * log(v);
        }
      }
      for (long long j0 = 0; j0 < p.S; j0 += 32) {
        const long long j = j0 + lane;
        double2 h = make_double2(-INFINITY, 0.0);
        if (j < p.S) {
          double ls, i2s;
          const double l = draw_ell(d[j], hN, quad, ls, i2s);
          h = make_double2(fma(-0.5, ls, l - mmax), i2s);
        }
        __syncwarp();
        hoisted[w][lane] = h;
        __syncwarp();
        const int n = (int)min(32ll, p.S - j0);
        for (int k = 0; k < n; k++) {
          const double2 hk = hoisted[w][k];
#pragma unroll
          for (int i = 0; i < MIX_TPL; i++)
            if (t0 + lane + 32 * i < p.T) lse_add(acc[i], fma(-r[i], hk.y, hk.x));
        }
      }
      double part = 0.0;
#pragma unroll
      for (int i = 0; i < MIX_TPL; i++) {
        const long long t = t0 + lane + 32 * i;
        if (t < p.T) {
          const double lp = bad ? nan : acc[i].value() + c[i] - log_s1;
          if (p.logp) p.logp[pr * p.T + t] = lp;
          part += lp;
        }
      }
#pragma unroll
      for (int dd = 16; dd > 0; dd >>= 1) part += __shfl_down_sync(0xffffffffu, part, dd);
      nsum += part;
    }
    if (lane == 0 && p.nll) p.nll[pr] = (p.T > 0 && !bad) ? -nsum / (double)p.T : nan;
  }
}

}  // namespace

cudaError_t launch_scale_draws(cudaStream_t s, int family, const double* params, long long P, long long S,
                               uint64_t seed, double* out) {
  long long blocks = (P * S + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  scale_draws_kernel<<<(unsigned)blocks, 256, 0, s>>>(family, params, P, S, (uint32_t)seed, (uint32_t)(seed >> 32),
                                                      out);
  instr().launches++;
  return cudaGetLastError();
}

cudaError_t launch_mixture_nll(cudaStream_t s, const MixtureParams& p) {
  long long blocks = (p.G * p.P + MIX_WARPS - 1) / MIX_WARPS;
  if (blocks > 148 * 8) blocks = 148 * 8;
  mixture_nll_kernel<<<(unsigned)blocks, 32 * MIX_WARPS, 0, s>>>(p);
  instr().launches++;
  return cudaGetLastError();
}

}  // namespace smnngp

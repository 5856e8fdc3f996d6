// Scalar closed forms of SPR.loss, of its gradient and of the log density of SPR.test_nll, shared by the per-call
// finalize kernels (reduce.cu, grad.cu) and the batched kernels (grad_batch.cu, test_nll_batch.cu).
#pragma once
#include "nngp_math.cuh"

namespace smnngp {

// out[0] = log p(y), out[1] = -log p / N (SPR.loss), out[2] = sum log L_ii, out[3] = ||L^-1 y||^2
// (spax/utils.py:181-183, spax/likelihoods.py:25-28, :45-50, spax/models.py:98); log p is NaN when *info != 0
__device__ __forceinline__ void lml_closed_form(double logdet, double zz, const double* __restrict__ hp, int kind,
                                                long long N, const int* __restrict__ info, double* __restrict__ out) {
  const double n = (double)N;
  double lml;
  if (kind == KIND_STUDENT_T) {
    // Sigma = (b/a)(K + eps I): chol(c S) = sqrt(c) chol(S)  =>  log-det += N/2 log c, quadratic form /= c
    const double a = hp[HP_ALPHA], b = hp[HP_BETA];
    const double c = b / a, df = 2.0 * a, t = 0.5 * (df + n);
    const double half_logdet = logdet + 0.5 * n * log(c);
    const double quad = zz / c;
    lml = -t * log(1.0 + quad / df) - 0.5 * n * log(df * kPi) + lgamma(t) - lgamma(0.5 * df) - half_logdet;
  } else {
    lml = -0.5 * zz - 0.5 * n * log(2.0 * kPi) - logdet;
  }
  if (*info != 0) lml = __longlong_as_double(0x7ff8000000000000ll);
  out[0] = lml;
  out[1] = -lml / n;
  out[2] = logdet;
  out[3] = zz;
}

// jax.scipy.stats.t.logpdf (spax/likelihoods.py:64)
__device__ __forceinline__ double t_logpdf(double x, double df, double loc, double scale) {
  const double z = (x - loc) / scale;
  const double norm = lgamma(0.5 * df) + 0.5 * log(df) + 0.5 * log(scale * scale * kPi) - lgamma(0.5 * (df + 1.0));
  return -(norm + 0.5 * (df + 1.0) * log1p(z * z / df));
}

// log density of one de-standardised test target x under the predictive of SPR.test_nll with mean m and variance cv
// (spax/likelihoods.py:52-65 Student-t, :30-33 Gaussian); *quad2 = ||L2^-1 y||^2 with L2 = chol(K + 1e-6 (a/b) I) is
// read under Student-t only
__device__ __forceinline__ double test_logpdf(double x, double m, double cv, const double* __restrict__ hp, int kind,
                                              long long N, const double* __restrict__ quad2) {
  double lp;
  if (kind == KIND_STUDENT_T) {
    const double a = hp[HP_ALPHA], b = hp[HP_BETA];
    const double df = 2.0 * a, cond_df = df + (double)N;
    // y^T ((b/a) K + 1e-6 I)^-1 y = (a/b) ||L2^-1 y||^2
    const double d = df + (a / b) * (*quad2);
    const double sigma = sqrt(d / cond_df * b / a * cv);
    lp = t_logpdf(x, cond_df, m, sigma);
  } else {
    const double sigma = sqrt(cv);
    const double z = (x - m) / sigma;
    lp = -0.5 * log(2.0 * kPi) - log(sigma) - 0.5 * z * z;
  }
  return lp;
}

namespace {
// digamma for x > 0: recurrence up to x >= 10, then the asymptotic series (error < 1e-17)
__device__ double digamma_pos(double x) {
  double r = 0.0;
  while (x < 10.0) { r -= 1.0 / x; x += 1.0; }
  const double f = 1.0 / (x * x);
  const double t = f * (-1.0 / 12.0 + f * (1.0 / 120.0 + f * (-1.0 / 252.0 + f * (1.0 / 240.0 + f * (-1.0 / 132.0 +
                   f * (691.0 / 32760.0 + f * (-1.0 / 12.0)))))));
  return r + log(x) - 0.5 / x + t;
}
}  // namespace

// grad[6] = d loss / d hp (loss = -log p / N) from the four contractions of G = d log p / d A = 1/2 (gamma a a^T - A^-1)
// with the derivatives of K: s_w = sum G dK/dw_std, s_b = sum G dK/db_std, s_v = sum G dK/dlast_w_std, s_e = tr G
// (= d log p / d eps); the alpha / beta entries are closed forms in quad = y^T A^-1 y (zero under Gaussian).  NaN when
// *info != 0.
__device__ __forceinline__ void grad_closed_form(double s_w, double s_b, double s_v, double s_e,
                                                 const double* __restrict__ hp, const double* __restrict__ quad_p,
                                                 int kind, long long N, const int* __restrict__ info,
                                                 double* __restrict__ grad) {
  const double n = (double)N, quad = *quad_p;
  double dlp[6] = {s_w, s_b, s_v, s_e, 0.0, 0.0};
  if (kind == KIND_STUDENT_T) {
    const double a = hp[HP_ALPHA], b = hp[HP_BETA], t = a + 0.5 * n;
    // quad / nu = quad / (2 b) does not depend on a; the N/2 log terms in a cancel
    dlp[4] = -log1p(quad / (2.0 * b)) + digamma_pos(t) - digamma_pos(a);
    dlp[5] = t * quad / (b * (2.0 * b + quad)) - 0.5 * n / b;
  }
  const bool bad = *info != 0;
  for (int q = 0; q < 6; q++) grad[q] = bad ? __longlong_as_double(0x7ff8000000000000ll) : -dlp[q] / n;
}

}  // namespace smnngp

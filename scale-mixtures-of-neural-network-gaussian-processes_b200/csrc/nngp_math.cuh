// Device math of the NNGP layer recursion (experiments/nt_kernels.py:12-31, :83-103 with neural_tangents
// semantics): diagonal maps, the branch-free ReLU arc-cosine step and the erf step, plus their partial
// derivatives (used by the gradient passes, grad.cu and grad_batch.cu).
#pragma once
#include "kernels.cuh"

namespace smnngp {

constexpr double kPi = 3.14159265358979323846;
constexpr double kInv2Pi = 0.15915494309189533577;
constexpr double kTwoOverPi = 0.63661977236758134308;

__device__ __forceinline__ double act_diag(double u, int act) {
  if (act == ACT_RELU) return 0.5 * u;
  return kTwoOverPi * asin(2.0 * u / (1.0 + 2.0 * u));
}
// what the Gram epilogue needs per row and layer: relu -> u itself, erf -> 1/sqrt(1+2u)
__device__ __forceinline__ double encode_var(double u, int act) {
  return act == ACT_RELU ? u : 1.0 / sqrt(1.0 + 2.0 * u);
}

// ---- branch-free ReLU arc-cosine step ---------------------------------------------------------------------
// phi(k; u1, u2) = ( s + k * (pi - atan2(s, k)) ) / (2 pi),  s = sqrt(max(u1 u2 - k^2, 0))
//                = ( s + k * atan2(s, -k) ) / (2 pi)
// The library sqrt / atan2 carry special-case branches that keep the compiler from interleaving the 64
// independent evaluations a thread owns, and with 4-8 resident math warps the epilogue was latency bound
// (50 Geval/s vs 197 Geval/s of FP64-pipe capacity).  This version is straight-line code: MUFU seeds
// (rsqrt.approx / rcp.approx on the double directly) + Newton steps, one division, an 11-term minimax
// polynomial for atan on |z| <= tan(pi/8) (fitted in 60-digit arithmetic, relative error 2.2e-16).
// Accuracy of phi: <= 2.5e-16 * sqrt(u1 u2) absolute (checked against 50-digit mpmath), i.e. the same as the
// libm formulation, for layer variances with 1e-260 <= u1 u2 <= 1e300.  u is a layer variance, not an input: a deep
// ReLU stack halves it at every layer, small weights or inputs in small units shrink it further, and the radicand
// u1 u2 - k^2 is of the order of u^2.  The seeds are floored at 1e-300, where rsqrt / rcp still return normal
// doubles; a radicand below the floor belongs to a pair with s < 1e-150, which phi ~ sqrt(u1 u2) cannot resolve.
__device__ __forceinline__ double rsqrt_seed(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  return y;
}
__device__ __forceinline__ double rcp_seed(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  return y;
}
__device__ __forceinline__ double sqrt_nobranch(double x) {          // x >= 0
  const double y = rsqrt_seed(fmax(x, 1e-300));
  double g = x * y, h = 0.5 * y;
  double r = fma(-g, h, 0.5);
  g = fma(g, r, g); h = fma(h, r, h);
  r = fma(-g, h, 0.5);
  g = fma(g, r, g); h = fma(h, r, h);
  return fma(fma(-g, g, x), h, g);
}
__device__ __forceinline__ double div_nobranch(double n, double d) {  // d >= 1e-300
  double y = rcp_seed(d);
  double e = fma(-d, y, 1.0);
  y = fma(y, e, y);
  e = fma(-d, y, 1.0);
  y = fma(y, e, y);
  const double q = n * y;
  return fma(y, fma(-q, d, n), q);
}
// returns phi; s_out = s, a_out = atan2(s, -k) = pi - theta  (d phi / d k = a / (2 pi), d phi / d u_i = s / (4 pi u_i))
__device__ __forceinline__ double phi_relu_parts(double k, double t1, double t2, double& s_out, double& a_out) {
  const double s = sqrt_nobranch(fmax(__dsub_rn(__dmul_rn(t1, t2), __dmul_rn(k, k)), 0.0));
  // a = atan2(s, -k) in [0, pi]
  const double ax = fabs(k);
  const bool swap = s > ax;
  const double num = swap ? ax : s;
  const double den = fmax(swap ? s : ax, 1e-300);
  const bool hi = num > 0.41421356237309503 * den;                   // tan(pi/8): atan(r) = pi/4 + atan((r-1)/(r+1))
  const double z = div_nobranch(hi ? num - den : num, hi ? num + den : den);
  const double w = z * z;
  double p = -0.017805397205419446;
  p = fma(p, w, 0.03796525745386593);
  p = fma(p, w, -0.05035102456601552);
  p = fma(p, w, 0.05846878297330872);
  p = fma(p, w, -0.06662951813629191);
  p = fma(p, w, 0.07692045330902225);
  p = fma(p, w, -0.09090896809064027);
  p = fma(p, w, 0.11111110744919658);
  p = fma(p, w, -0.14285714279250245);
  p = fma(p, w, 0.19999999999940893);
  p = fma(p, w, -0.3333333333333312);
  p = fma(p, w, 1.0);
  double a = fma(z, p, hi ? 0.78539816339744831 : 0.0);
  a = swap ? 1.5707963267948966 - a : a;
  a = (k > 0.0) ? kPi - a : a;                                        // x = -k < 0
  s_out = s;
  a_out = a;
  return fma(k, a, s) * kInv2Pi;
}
__device__ __forceinline__ double phi_relu_fast(double k, double t1, double t2) {
  double s, a;
  return phi_relu_parts(k, t1, t2, s, a);
}

// one nonlinearity on a cross-covariance k given the encoded marginals of its row and column
template <int ACT>
__device__ __forceinline__ double phi(double k, double t1, double t2) {
  if (ACT == ACT_RELU) {
    return phi_relu_fast(k, t1, t2);
  } else {
    double x = 2.0 * k * t1 * t2;
    x = fmin(fmax(x, -1.0), 1.0);
    return kTwoOverPi * asin(x);
  }
}

// per-row layer tables from the input variance q0 = ||x||^2 / D.  hp == nullptr: unit scalars (w = v = 1, b = 0)
__device__ __forceinline__ void fill_row_tables(double q, int row, int n_hidden, int act, int arch,
                                                const double* __restrict__ hp, double* __restrict__ tab,
                                                long long tab_ld, double* __restrict__ qfin) {
  const double w2 = hp ? hp[HP_W] * hp[HP_W] : 1.0, b2 = hp ? hp[HP_B] * hp[HP_B] : 0.0,
               v2 = hp ? hp[HP_V] * hp[HP_V] : 1.0;
  if (arch == ARCH_MLP) {
    for (int a = 0; a < n_hidden; a++) {
      double u = w2 * q + b2;
      tab[a * tab_ld + row] = encode_var(u, act);
      q = act_diag(u, act);
    }
  } else {
    double u = w2 * q + b2;
    for (int a = 0; a < n_hidden; a++) {
      tab[a * tab_ld + row] = encode_var(u, act);
      u = u + (w2 * act_diag(u, act) + b2);
    }
    tab[(long long)n_hidden * tab_ld + row] = encode_var(u, act);
    q = act_diag(u, act);
  }
  qfin[row] = v2 * q;
}

// One layer of the recursion on one kernel entry k given the encoded marginals of its row and column: an MLP layer
// (Dense then the nonlinearity), a dense-resnet block (k + Dense(phi(k))), or the resnet's trailing activation (plain).
template <int ACT>
__device__ __forceinline__ double layer_step(double k, double tr, double tc, double w2, double b2, bool resnet,
                                             bool plain) {
  if (!resnet) k = w2 * k + b2;
  const double ph = phi<ACT>(k, tr, tc);
  return plain ? ph : k + (w2 * ph + b2);
}

// K entry from its base value (X.X'^T / D): the recursion of gram_epilogue (gram.cu) on one element, then the final
// Dense
template <int ACT>
__device__ __forceinline__ double nngp_entry(double k, const double* __restrict__ tab_r, long long ld_r, int r,
                                             const double* __restrict__ tab_c, long long ld_c, int c, int n_act,
                                             bool resnet, double w2, double b2, double v2) {
  if (resnet) k = w2 * k + b2;
  for (int a = 0; a < n_act; a++)
    k = layer_step<ACT>(k, tab_r[a * ld_r + r], tab_c[a * ld_c + c], w2, b2, resnet, !resnet || a == n_act - 1);
  return v2 * k;
}

// ---- forward-mode duals of the recursion (gradient w.r.t. w_std and b_std) -------------------------------------
constexpr double kInv4Pi = 0.079577471545947667884;
constexpr double kFourOverPi = 1.27323954473516268615;

// per-row dual tables tab3 = [3][n_act][tab_ld]:
//   plane 0: encoded marginal variance (relu: u, erf: 1/sqrt(1+2u))  (as fill_row_tables)
//   plane 1: f(u) du/dw_std,  plane 2: f(u) du/db_std
// with f(u) = 1/(4 pi u) (relu: d phi / d u_i = s f(u_i)),  1/(1+2u) (erf: d phi / d u_i = -g x f(u_i))
__device__ __forceinline__ void store_dual(double* tab3, long long plane, long long idx, double u, double duw,
                                           double dub, int act) {
  const double f = act == ACT_RELU ? (u > 0.0 ? kInv4Pi / u : 0.0) : 1.0 / (1.0 + 2.0 * u);
  tab3[idx] = encode_var(u, act);
  tab3[plane + idx] = f * duw;
  tab3[2 * plane + idx] = f * dub;
}
// act_diag'(u)
__device__ __forceinline__ double act_diag_deriv(double u, int act) {
  if (act == ACT_RELU) return 0.5;
  return kFourOverPi / ((1.0 + 2.0 * u) * sqrt(1.0 + 4.0 * u));
}

// the dual tables of one row from its input variance q = ss / D (ss = ||x||^2; a cached q is passed with D = 1, exact)
// n_act = n_act_applications(n_hidden, arch)
__device__ __forceinline__ void fill_row_dual_tables(double ss, int D, int row, int n_hidden, int act, int arch,
                                                     const double* __restrict__ hp, double* __restrict__ tab3,
                                                     long long tab_ld, int n_act) {
  const double w = hp[HP_W], b = hp[HP_B];
  const double w2 = w * w, b2 = b * b;
  const long long plane = (long long)(n_act > 0 ? n_act : 1) * tab_ld;
  double q = ss / (double)D, dqw = 0.0, dqb = 0.0;
  if (arch == ARCH_MLP) {
    for (int a = 0; a < n_hidden; a++) {
      const double u = w2 * q + b2, duw = 2.0 * w * q + w2 * dqw, dub = w2 * dqb + 2.0 * b;
      store_dual(tab3, plane, a * tab_ld + row, u, duw, dub, act);
      const double d = act_diag_deriv(u, act);
      q = act_diag(u, act);
      dqw = d * duw;
      dqb = d * dub;
    }
  } else {
    double u = w2 * q + b2, duw = 2.0 * w * q, dub = 2.0 * b;
    for (int a = 0; a < n_hidden; a++) {
      store_dual(tab3, plane, a * tab_ld + row, u, duw, dub, act);
      const double ph = act_diag(u, act), d = act_diag_deriv(u, act);
      u = u + (w2 * ph + b2);
      const double nw = duw + (2.0 * w * ph + w2 * d * duw), nb = dub + (w2 * d * dub + 2.0 * b);
      duw = nw;
      dub = nb;
    }
    store_dual(tab3, plane, (long long)n_hidden * tab_ld + row, u, duw, dub, act);
  }
}

// dual layer step.  in: k, dw, db (value and d/dw_std, d/db_std of the pre-activation cross-covariance), row / column
// table entries; out: phi and its duals
template <int ACT>
__device__ __forceinline__ void phi_dual(double k, double dw, double db, double e1, double e2, double fw, double fb,
                                         double& ph, double& phw, double& phb) {
  if (ACT == ACT_RELU) {
    double s, a;
    ph = phi_relu_parts(k, e1, e2, s, a);
    const double pk = a * kInv2Pi;                 // (pi - theta) / (2 pi)
    phw = fma(pk, dw, s * fw);                     // fw = f(u1) du1/dw + f(u2) du2/dw
    phb = fma(pk, db, s * fb);
  } else {
    double x = 2.0 * k * e1 * e2;
    x = fmin(fmax(x, -1.0), 1.0);
    ph = kTwoOverPi * asin(x);
    const double g = kTwoOverPi * rsqrt(fmax(1.0 - x * x, 1e-300));
    const double pk = 2.0 * g * e1 * e2;
    phw = fma(pk, dw, -g * x * fw);
    phb = fma(pk, db, -g * x * fb);
  }
}

// One layer of the dual recursion on one entry (k, dw, db) in place: MLP layer, resnet block or trailing activation
// (plain), as layer_step.  e1 / e2: plane 0 of the row / column; fw / fb: sums of the row's and column's planes 1 / 2.
template <int ACT>
__device__ __forceinline__ void layer_step_dual(double& k, double& dw, double& db, double e1, double e2, double fw,
                                                double fb, double w, double b, double w2, double b2, bool resnet,
                                                bool plain) {
  double kin = k, dwin = dw, dbin = db;
  if (!resnet) {                                         // Dense(512, W_std, b_std)
    dwin = fma(w2, dwin, 2.0 * w * kin);
    dbin = fma(w2, dbin, 2.0 * b);
    kin = fma(w2, kin, b2);
  }
  double ph, phw, phb;
  phi_dual<ACT>(kin, dwin, dbin, e1, e2, fw, fb, ph, phw, phb);
  if (plain) {
    k = ph; dw = phw; db = phb;
  } else {                                               // ResBlock: z + Dense(act(z))
    k = kin + fma(w2, ph, b2);
    dw = dwin + fma(w2, phw, 2.0 * w * ph);
    db = dbin + fma(w2, phb, 2.0 * b);
  }
}

}  // namespace smnngp

// Counter-based random numbers and the online log-sum-exp shared by the draw stage (draws.cu) and the scale mixture
// (mixture.cu).  A stream is a pure function of (key, counter), so a kernel that redraws a cell sees exactly the
// variates another kernel wrote, and a CPU replica (oracle/draws_ref.py; tests/mixture_ref.py for the scale draws)
// can recompute any cell.
#pragma once
#include <cstdint>

namespace smnngp {

struct Philox {
  uint32_t k0, k1;
  __device__ __forceinline__ uint4 operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
    uint32_t a = k0, b = k1;
#pragma unroll
    for (int r = 0; r < 10; r++) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      c0 = hi1 ^ c1 ^ a; c1 = lo1; c2 = hi0 ^ c3 ^ b; c3 = lo0;
      a += 0x9E3779B9u; b += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};

__device__ __forceinline__ double u01(uint32_t hi, uint32_t lo) {     // (0, 1], 53 bits
  const unsigned long long v = ((unsigned long long)hi << 21) ^ (lo >> 11);
  return ((double)(v & ((1ull << 53) - 1)) + 1.0) * (1.0 / 9007199254740992.0);
}

// stream of uniforms for one (sample, test point, class) cell
struct CellRng {
  Philox ph;
  uint32_t s, t, c, n;
  uint4 buf;
  int have;
  __device__ __forceinline__ CellRng(uint32_t k0, uint32_t k1, uint32_t s_, uint32_t t_, uint32_t c_)
      : ph{k0, k1}, s(s_), t(t_), c(c_), n(0), have(0) {}
  __device__ __forceinline__ double uniform() {
    if (have == 0) { buf = ph(s, t, c, n++); have = 2; }
    double u = (have == 2) ? u01(buf.x, buf.y) : u01(buf.z, buf.w);
    have--;
    return u;
  }
  __device__ __forceinline__ double normal() {                         // Box-Muller (one of the pair)
    const double u1 = uniform(), u2 = uniform();
    return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
  }
  __device__ __forceinline__ double gamma(double alpha) {              // Marsaglia & Tsang (2000), shape alpha
    double boost = 1.0;
    if (alpha < 1.0) { boost = pow(uniform(), 1.0 / alpha); alpha += 1.0; }
    const double d = alpha - 1.0 / 3.0, cc = 1.0 / sqrt(9.0 * d);
    for (int it = 0; it < 64; it++) {
      const double x = normal();
      double v = 1.0 + cc * x;
      if (v <= 0.0) continue;
      v = v * v * v;
      const double u = uniform();
      if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) return boost * d * v;
    }
    return boost * d;
  }
  // standard Student-t with df degrees of freedom (jax.random.t: normal / sqrt(gamma(df/2) / (df/2)))
  __device__ __forceinline__ double student_t(double df) {
    const double z = normal();
    const double g = gamma(0.5 * df);
    return z / sqrt(g / (0.5 * df));
  }
};

// online log-sum-exp accumulator
struct Lse {
  double m, s;
  __device__ __forceinline__ void init() { m = -INFINITY; s = 0.0; }
  __device__ __forceinline__ void add(double x) {
    if (x > m) { s = s * exp(m - x) + 1.0; m = x; }
    else s += exp(x - m);
  }
  __device__ __forceinline__ void merge(double m2, double s2) {
    if (m2 == -INFINITY) return;
    if (m == -INFINITY) { m = m2; s = s2; return; }
    if (m2 > m) { s = s * exp(m - m2) + s2; m = m2; }
    else s += s2 * exp(m2 - m);
  }
  __device__ __forceinline__ double value() const { return m + log(s); }
};

}  // namespace smnngp

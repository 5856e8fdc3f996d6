// Device building blocks of the in-CTA Cholesky, shared by the diagonal-block kernel of the blocked factorisation
// (chol.cu) and the batched grid search (grid_batch.cu): a branch-free 1/sqrt, the register-resident factor + inverse
// of a DB x DB diagonal block, and an 8x8 DMMA tile product out of shared memory.
#pragma once
#include "kernels.cuh"

namespace smnngp {

namespace {

#ifndef SMNNGP_DB
#define SMNNGP_DB 16
#endif
constexpr int DB = SMNNGP_DB;          // register-resident diagonal block (16: ~400 instructions, stays in the
                                       // instruction cache; the 32-wide version was instruction-fetch bound)
constexpr int KS = DB / 4;             // k4-steps per block
constexpr int NT = DB / 8;             // 8-wide tiles per block
constexpr int GLD = PB + 4;            // 132: (4 * row + k) mod 16 distinct over a half-warp's 4 rows x 4 k
constexpr int MLD = DB + 4;            // 20 / 36: same property

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// 1/sqrt(d) without the library's special-case branches: MUFU.RSQ64H seed + two coupled Newton steps + one
// correction (<= 1 ulp for normal d > 0).  The library rsqrt() / division cost ~300 dependent cycles each and
// sat on the critical path of every pivot: they were 60 % of the whole diagonal-block kernel.
__device__ __forceinline__ double rsqrt_fast(double d) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
  double g = d * y, h = 0.5 * y;
  double r = fma(-g, h, 0.5);
  g = fma(g, r, g); h = fma(h, r, h);
  r = fma(-g, h, 0.5);
  h = fma(h, r, h);                       // h ~ 0.5 / sqrt(d)
  double y2 = h + h;
  return fma(y2, fma(-d * y2, y2, 1.0) * 0.5, y2);   // one more Newton step on y = 1/sqrt(d)
}

// warp 0: factor the DB x DB block at Gbb (row stride GLD, lower part valid) in place and write inv(L) to M (row
// stride MLD).  *bad, if still 0, receives col_base + 1 + the first pivot that is not > 0.
//   lanes 0 .. DB-1   hold row `lane` of the block,
//   lanes DB .. 2DB-1 hold row `lane - DB` of the IDENTITY: carried through the same column operations they come out
//                     as rows of L^-T, i.e. the columns of inv(L) - the inverse costs nothing extra (it used to be a
//                     separate 16-step forward substitution: ~40 % of this routine's time and half of its code).
// The pivot loop stays fully unrolled (ptxas interleaves pivot j's remaining column updates with pivot j+1's
// rsqrt chain; a rolled loop with a rotating register window measured 580 cycles per pivot against ~200 unrolled:
// profiles/r02_potf2_phases.txt) but the routine is a single out-of-line copy (~800 instructions) instead of two inlined
// ~2000-instruction ones: this kernel runs every instruction about once per launch, so its first diagonal block was
// bound by cold instruction fetch (64 k cycles, the following blocks 6 k).
__device__ __noinline__ void diag_factor_invert(double* __restrict__ Gbb, double* __restrict__ M, int lane,
                                                int col_base, int* bad) {
  static_assert(2 * DB <= 32, "block rows + carried identity rows must fit one warp");
  const bool is_row = lane < DB;
  const int r = is_row ? lane : lane - DB;               // block row, or the identity row this lane carries
  double a[DB];
#pragma unroll
  for (int c = 0; c < DB; c++) a[c] = is_row ? Gbb[r * GLD + c] : (c == r ? 1.0 : 0.0);
  int first_bad = 0;
#pragma unroll
  for (int j = 0; j < DB; j++) {
    double d = shfl_d(a[j], j);                          // pivot: row j, column j
    if (!(d > 0.0)) {                                    // non-PD (or NaN input): mirror lax.linalg.cholesky -> NaN
      if (first_bad == 0) first_bad = col_base + j + 1;
      d = __longlong_as_double(0x7ff8000000000000ll);
    }
    const double rinv = rsqrt_fast(d);                   // = 1 / L_jj (same value in every lane)
    const double l = (lane == j) ? d * rinv : a[j] * rinv;     // column j of L (rows >= j) / of the carried rows
    a[j] = l;
#pragma unroll
    for (int c = j + 1; c < DB; c++) a[c] = fma(-l, shfl_d(l, c), a[c]);
  }
  if (first_bad != 0 && *bad == 0) *bad = first_bad;
  if (is_row) {
#pragma unroll
    for (int c = 0; c < DB; c++)
      if (c <= r) Gbb[r * GLD + c] = a[c];
  } else {
    // inv(L)[c][r] = (L^-T)[r][c], zero above the diagonal
#pragma unroll
    for (int c = 0; c < DB; c++) M[c * MLD + r] = (c >= r) ? a[c] : 0.0;
  }
}

// acc(8x8) += sum over nks k4-steps of A[row, k] * B[k, col]; A K-contiguous, B k-major (element (k, col) at
// B[k*ldb + col])
__device__ __forceinline__ void tile_nn(double (&acc)[2], const double* __restrict__ A, int lda,
                                        const double* __restrict__ B, int ldb, int nks, int lane) {
  const double* ap = A + (lane >> 2) * lda + (lane & 3);
  const double* bp = B + (lane & 3) * ldb + (lane >> 2);
  for (int ks = 0; ks < nks; ks++) dmma8x8x4(acc, ap[ks * 4], bp[ks * 4 * ldb]);
}

}  // namespace

}  // namespace smnngp

// In-CTA building blocks of the batched kernels (grid_batch.cu, grad_batch.cu, test_nll_batch.cu): one CTA of
// GB_THREADS threads owns a workspace slot and works on one point at a time - the Gram rebuilt from its cached base, a
// blocked Cholesky of the slot, and the predictive of a point.
//
// Cholesky of a slot (A row-major, lda, rows 0..N-1 lower = the matrix, rows N..M-1 carried), 64-column outer panels:
//   per 16 columns:  the 16 x 16 diagonal block is staged to shared memory and factored + inverted by one warp
//                    (diag_factor_invert, the routine of the blocked factorisation's diagonal kernel); the rows below
//                    are solved in place against inv(L_jj) and the rest of the outer panel is updated, both on DMMA
//                    with 8-row strips per warp straight from global memory (L2);
//   trailing update: rows >= c1 x cols [c1, N), lower part, C -= P P^T with K = 64: 64 x 64 tiles whose two panel
//                    operands are staged by cp.async into shared memory (row stride 68: conflict-free fragments).
#pragma once
#include "chol_core.cuh"
#include "kernels.cuh"
#include "nngp_math.cuh"

namespace smnngp {

namespace {

constexpr int GB_THREADS = 256;
constexpr int GB_WARPS = GB_THREADS / 32;
constexpr int GB_NB = 64;                  // outer panel width = K of the trailing update
constexpr int GB_TLD = GB_NB + 4;          // 68: row stride of the staged panel tiles
constexpr int GB_SMEM_DOUBLES = DB * GLD + DB * MLD + 2 * GB_NB * GB_TLD + GB_WARPS;
constexpr int GB_SMEM_BYTES = GB_SMEM_DOUBLES * 8 + 16;

__device__ __forceinline__ double qnan_d() { return __longlong_as_double(0x7ff8000000000000ll); }

// rows 0..N-1 (lower) of the slot = K + shift I
template <int ACT, class P>
__device__ void build_gram(const P& p, const double* __restrict__ hp, const double* __restrict__ tab,
                           double* __restrict__ A, double shift) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool resnet = p.arch == ARCH_RESNET;
  const int n_act = n_act_applications(p.n_hidden, p.arch);
  const double w2 = hp[HP_W] * hp[HP_W], b2 = hp[HP_B] * hp[HP_B], v2 = hp[HP_V] * hp[HP_V];
  for (int r = warp; r < p.N; r += GB_WARPS) {
    const double* src = p.K0dd + (long long)r * p.ld0;
    double* dst = A + (long long)r * p.lda;
    for (int c = lane; c <= r; c += 32) {
      double v = nngp_entry<ACT>(src[c], tab, p.N, r, tab, p.N, c, n_act, resnet, w2, b2, v2);
      if (c == r) v += shift;
      dst[c] = v;
    }
  }
}

__device__ void copy_row(const double* __restrict__ src, double* __restrict__ dst, int n) {
  for (int i = threadIdx.x; i < n; i += GB_THREADS) dst[i] = src[i];
}

// rows N..N+T-1 of the slot = K_td
template <int ACT, class P>
__device__ void build_cross(const P& p, const double* __restrict__ hp, const double* __restrict__ tab,
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

// 8-row strip r0.. of the 16 columns at j0 (w valid) <- strip * inv(L_jj)^T, in place (rows < M)
__device__ __forceinline__ void panel_solve_strip(double* __restrict__ A, long long lda, int M, int r0, int j0, int w,
                                                  const double* __restrict__ Mi, int lane) {
  const int r = r0 + (lane >> 2);
  double* row = A + (long long)r * lda + j0;
  double af[KS];
#pragma unroll
  for (int ks = 0; ks < KS; ks++) {
    const int c = ks * 4 + (lane & 3);
    af[ks] = (r < M && c < w) ? row[c] : 0.0;
  }
  double acc[NT][2];
#pragma unroll
  for (int nt = 0; nt < NT; nt++) {
    acc[nt][0] = acc[nt][1] = 0.0;
    const double* bp = Mi + (nt * 8 + (lane >> 2)) * MLD + (lane & 3);
#pragma unroll
    for (int ks = 0; ks < KS; ks++)
      if (ks <= 2 * nt + 1) dmma8x8x4(acc[nt], af[ks], bp[ks * 4]);   // inv(L) is lower triangular
  }
  __syncwarp();
  if (r < M) {
#pragma unroll
    for (int nt = 0; nt < NT; nt++) {
      const int c = nt * 8 + (lane & 3) * 2;
      if (c < w) row[c] = acc[nt][0];
      if (c + 1 < w) row[c + 1] = acc[nt][1];
    }
  }
}

// this warp's 32 x 16 part (rows wm*32.., cols wn*16..) of a 64 x 64 tile: acc += Pa Pb^T over the 64 staged columns
// (Pa, Pb: [64][GB_TLD] in shared memory)
__device__ __forceinline__ void tile64_mma(double (&acc)[4][2][2], const double* __restrict__ Pa,
                                           const double* __restrict__ Pb, int wm, int wn, int lane) {
  const double* ap = Pa + (wm * 32 + (lane >> 2)) * GB_TLD + (lane & 3);
  const double* bp = Pb + (wn * 16 + (lane >> 2)) * GB_TLD + (lane & 3);
#pragma unroll 4
  for (int ks = 0; ks < GB_NB / 4; ks++) {
    double a[4], b[2];
#pragma unroll
    for (int mi = 0; mi < 4; mi++) a[mi] = ap[mi * 8 * GB_TLD + ks * 4];
#pragma unroll
    for (int ni = 0; ni < 2; ni++) b[ni] = bp[ni * 8 * GB_TLD + ks * 4];
#pragma unroll
    for (int mi = 0; mi < 4; mi++)
#pragma unroll
      for (int ni = 0; ni < 2; ni++) dmma8x8x4(acc[mi][ni], a[mi], b[ni]);
  }
}

// Cholesky of the slot's leading N x N (lower) with rows N..Mtot-1 carried; returns through *bad_s the 1-based column of
// the first pivot that is not > 0 (0: none) and adds log L_ii of this thread's diagonal entries to lsum
// IDENT: rows N+1 .. 2N start as the identity and come out as U = L^-T.  Identity row N+1+i is still e_i until the
// panel that holds column i, so panel [c0, c1) only touches the rows below N+1+c1 (the carried work is N^3/3, not N^3:
// the skip of ident_row0 in potrf_trapezoid).
template <bool IDENT>
__device__ void factor_slot(double* __restrict__ A, long long lda, int Mtot, int N, double* __restrict__ smem,
                            int* bad_s, double& lsum) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double* Gd = smem;                       // [DB][GLD] staged diagonal block
  double* Mi = Gd + DB * GLD;              // [DB][MLD] its inverse
  double* Pa = Mi + DB * MLD;              // [64][68] panel rows of the output row block
  double* Pb = Pa + GB_NB * GB_TLD;        // [64][68] panel rows of the output column block
  if (tid == 0) *bad_s = 0;
  for (int c0 = 0; c0 < N; c0 += GB_NB) {
    const int c1 = min(c0 + GB_NB, N);
    const int M = IDENT ? min(Mtot, N + 1 + c1) : Mtot;   // rows that take part in this panel
    for (int j0 = c0; j0 < c1; j0 += DB) {
      const int j1 = min(j0 + DB, N), w = j1 - j0;
      for (int i = tid; i < DB * DB; i += GB_THREADS) {
        const int r = i / DB, c = i % DB;
        double v;
        if (r < w) v = c <= r ? A[(long long)(j0 + r) * lda + j0 + c] : 0.0;
        else v = (c == r) ? 1.0 : 0.0;                   // identity padding of a short last block
        Gd[r * GLD + c] = v;
      }
      __syncthreads();
      if (warp == 0) diag_factor_invert(Gd, Mi, lane, j0, bad_s);
      __syncthreads();
      if (tid < w) lsum += log(Gd[tid * GLD + tid]);
      // rows below: solve against inv(L_jj)
      const int nstrips = (M - j1 + 7) / 8;
      for (int s = warp; s < nstrips; s += GB_WARPS) panel_solve_strip(A, lda, M, j1 + s * 8, j0, w, Mi, lane);
      __syncthreads();
      // the rest of the outer panel: C[r][c] -= P[r] . P[c] for j1 <= c < c1, c <= r
      if (j1 < c1) {
        for (int s = warp; s < nstrips; s += GB_WARPS) {
          const int r0 = j1 + s * 8, r = r0 + (lane >> 2);
          double af[KS];
#pragma unroll
          for (int ks = 0; ks < KS; ks++) {
            const int c = ks * 4 + (lane & 3);
            af[ks] = (r < M && c < w) ? A[(long long)r * lda + j0 + c] : 0.0;
          }
          for (int ct = j1; ct < c1 && ct <= r0 + 7; ct += 8) {
            const int rc = ct + (lane >> 2);                // B fragment: panel row of output column rc
            double acc[2] = {0.0, 0.0};
#pragma unroll
            for (int ks = 0; ks < KS; ks++) {
              const int c = ks * 4 + (lane & 3);
              const double b = (rc < c1 && c < w) ? A[(long long)rc * lda + j0 + c] : 0.0;
              dmma8x8x4(acc, af[ks], b);
            }
            const int cc = ct + (lane & 3) * 2;
            if (r < M) {
              double* dst = A + (long long)r * lda + cc;
              if (cc < c1 && cc <= r) dst[0] -= acc[0];
              if (cc + 1 < c1 && cc + 1 <= r) dst[1] -= acc[1];
            }
          }
        }
        __syncthreads();
      }
    }
    if (c1 >= N) break;
    // trailing update with the whole outer panel (K = 64 exactly: only the last panel is narrower, and it has none)
    const int wm = warp >> 2, wn = warp & 3;       // warp tile: rows wm*32 .. +32, cols wn*16 .. +16
    for (int rb = c1; rb < M; rb += GB_NB) {
      for (int i = tid; i < GB_NB * (GB_NB / 2); i += GB_THREADS) {
        const int r = i / (GB_NB / 2), c = (i % (GB_NB / 2)) * 2;
        const bool ok = rb + r < M;
        cp_async16(Pa + r * GB_TLD + c, A + (long long)(ok ? rb + r : c0) * lda + c0 + c, ok ? 16 : 0);
      }
      for (int cb = c1; cb < N && cb <= rb + GB_NB - 1; cb += GB_NB) {
        for (int i = tid; i < GB_NB * (GB_NB / 2); i += GB_THREADS) {
          const int r = i / (GB_NB / 2), c = (i % (GB_NB / 2)) * 2;
          const bool ok = cb + r < N;
          cp_async16(Pb + r * GB_TLD + c, A + (long long)(ok ? cb + r : c0) * lda + c0 + c, ok ? 16 : 0);
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        const int r_lo = rb + wm * 32, c_lo = cb + wn * 16;
        if (c_lo <= r_lo + 31 && r_lo < M && c_lo < N) {   // warp tile not entirely above the diagonal / outside
          double acc[4][2][2];
#pragma unroll
          for (int mi = 0; mi < 4; mi++)
#pragma unroll
            for (int ni = 0; ni < 2; ni++) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
          const double* ap = Pa + (wm * 32 + (lane >> 2)) * GB_TLD + (lane & 3);
          const double* bp = Pb + (wn * 16 + (lane >> 2)) * GB_TLD + (lane & 3);
#pragma unroll 4
          for (int ks = 0; ks < GB_NB / 4; ks++) {
            double a[4], b[2];
#pragma unroll
            for (int mi = 0; mi < 4; mi++) a[mi] = ap[mi * 8 * GB_TLD + ks * 4];
#pragma unroll
            for (int ni = 0; ni < 2; ni++) b[ni] = bp[ni * 8 * GB_TLD + ks * 4];
#pragma unroll
            for (int mi = 0; mi < 4; mi++)
#pragma unroll
              for (int ni = 0; ni < 2; ni++) dmma8x8x4(acc[mi][ni], a[mi], b[ni]);
          }
#pragma unroll
          for (int mi = 0; mi < 4; mi++) {
            const int r = r_lo + mi * 8 + (lane >> 2);
            if (r >= M) continue;
#pragma unroll
            for (int ni = 0; ni < 2; ni++) {
              const int c = c_lo + ni * 8 + (lane & 3) * 2;
              double* dst = A + (long long)r * lda + c;
              if (c < N && c <= r) dst[0] -= acc[mi][ni][0];
              if (c + 1 < N && c + 1 <= r) dst[1] -= acc[mi][ni][1];
            }
          }
        }
        __syncthreads();                               // Pb (and, after the last column block, Pa) is free again
      }
    }
  }
}


// W (rows 0..N-1, lower part) = U U^T for the upper triangular U [N][ldu] (A^-1 from U = L^-T).  64 x 64 output tiles
// through the staged tile loop of factor_slot's trailing update; the contraction of a tile whose first row is rb runs
// over k >= rb only (U[r][k] = 0 for k < r).  U's columns N .. ldu-1 must be zero; W must not overlap U.
__device__ void syrk_upper_slot(const double* __restrict__ U, long long ldu, int N, double* __restrict__ W,
                                long long ldw, double* __restrict__ smem) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double* Pa = smem + DB * GLD + DB * MLD;   // the panel buffers of factor_slot
  double* Pb = Pa + GB_NB * GB_TLD;
  const int wm = warp >> 2, wn = warp & 3;
  for (int rb = 0; rb < N; rb += GB_NB) {
    for (int cb = 0; cb <= rb; cb += GB_NB) {
      const int r_lo = rb + wm * 32, c_lo = cb + wn * 16;
      const bool active = c_lo <= r_lo + 31 && r_lo < N;
      double acc[4][2][2];
#pragma unroll
      for (int mi = 0; mi < 4; mi++)
#pragma unroll
        for (int ni = 0; ni < 2; ni++) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
      for (int k0 = rb; k0 < N; k0 += GB_NB) {
        for (int i = tid; i < GB_NB * (GB_NB / 2); i += GB_THREADS) {
          const int r = i / (GB_NB / 2), c = (i % (GB_NB / 2)) * 2;
          const bool ka = k0 + c < N;              // k0 + c even and < N <= ldu: the pair stays inside the row
          const bool oka = ka && rb + r < N, okb = ka && cb + r < N;
          cp_async16(Pa + r * GB_TLD + c, U + (oka ? (long long)(rb + r) * ldu + k0 + c : 0), oka ? 16 : 0);
          cp_async16(Pb + r * GB_TLD + c, U + (okb ? (long long)(cb + r) * ldu + k0 + c : 0), okb ? 16 : 0);
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        if (active) tile64_mma(acc, Pa, Pb, wm, wn, lane);
        __syncthreads();                           // Pa / Pb are free again
      }
      if (active) {
#pragma unroll
        for (int mi = 0; mi < 4; mi++) {
          const int r = r_lo + mi * 8 + (lane >> 2);
          if (r >= N) continue;
#pragma unroll
          for (int ni = 0; ni < 2; ni++) {
            const int c = c_lo + ni * 8 + (lane & 3) * 2;
            double* dst = W + (long long)r * ldw + c;
            if (c <= r) dst[0] = acc[mi][ni][0];
            if (c + 1 <= r) dst[1] = acc[mi][ni][1];
          }
        }
      }
    }
  }
}

// The predictive of one point with the relative regulariser (what smnngp_grid_point_f64 and the first half of
// smnngp_test_nll_f64 compute), for the point's scalars hp:
//   1. layer tables of the train rows (tab, q) and the test rows (tab_t, q_t), tr(K)/N by a fixed-order block sum;
//   2. the trapezoid K + eps tr(K)/N I (lower) | K_td | y^T in the slot A, factor_slot - the carried rows come out as
//      v_t = K_td L^-T and z = (L^-1 y)^T - then, per test row t, lane 0 of one warp calls
//      emit(t, ||v_t||^2, v_t . z, bad) with bad = the factorisation's *bad_s: mean_t = v_t . z and
//      var_t = q_t[t] - ||v_t||^2 (emit forms var_t itself, so that it reads q_t only for a good point).
// tid, lane, warp, N and T are the caller's; eps is set to hp[HP_EPS].  Returns bad; ends on a __syncthreads (the
// slot is free again, emit's stores are visible to the CTA).
template <int ACT, class P, class Emit>
__device__ __forceinline__ int predictive_slot(const P& p, const double* __restrict__ hp, double* __restrict__ A,
                                               double* __restrict__ tab, double* __restrict__ q,
                                               double* __restrict__ tab_t, double* __restrict__ q_t,
                                               double* __restrict__ smem, double* __restrict__ red, int* bad_s,
                                               int tid, int lane, int warp, int N, int T, double& eps, Emit&& emit) {
  double qs = 0.0;
  for (int r = tid; r < N; r += GB_THREADS) {
    fill_row_tables(p.q_d[r], r, p.n_hidden, ACT, p.arch, hp, tab, N, q);
    qs += q[r];
  }
  for (int t = tid; t < T; t += GB_THREADS) fill_row_tables(p.q_t[t], t, p.n_hidden, ACT, p.arch, hp, tab_t, T, q_t);
  const double trmean = block_sum<GB_THREADS>(qs, red) / (double)N;   // its __syncthreads also publishes the tables
  eps = hp[HP_EPS];

  build_gram<ACT>(p, hp, tab, A, eps * trmean);
  build_cross<ACT>(p, hp, tab, tab_t, A);
  copy_row(p.y, A + (long long)(N + T) * p.lda, N);
  __syncthreads();
  double lsum = 0.0;
  factor_slot<false>(A, p.lda, N + T + 1, N, smem, bad_s, lsum);
  __syncthreads();
  const int bad = *bad_s;
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
    if (lane == 0) emit(t, vv, vz, bad);
  }
  __syncthreads();
  return bad;
}

}  // namespace

}  // namespace smnngp

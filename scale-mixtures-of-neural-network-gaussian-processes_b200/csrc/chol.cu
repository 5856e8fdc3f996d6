// Blocked right-looking FP64 Cholesky on the row-major lower triangle (replaces lax.linalg.cholesky at
// spax/utils.py:179 and the cho_factor inside neural_tangents' predict, spax/kernels.py:29-32).
//   diagonal block : one-CTA fused potf2 + triangular inverse in shared memory
//   TRSM           : panel <- panel * inv(L_kk)^T on the DMMA GEMM core (in place, one column tile)
//   trailing update: C -= P * P^T on the DMMA GEMM core, lower tiles only
// Rows below the square part (the trapezoid) are carried through TRSM + update, so appended rows y^T and K_td
// come out as (L^-1 y)^T and (L^-1 K_dt)^T: the triangular solves of spax/utils.py:180 and of cho_solve are
// fused into the factorisation and run on the tensor pipe.
#include "context.cuh"
#include "gemm_core.cuh"
#include "chol_core.cuh"
#include "kernels.cuh"
#include "tma_core.cuh"

namespace smnngp {

namespace {

constexpr int EPI_STORE = 0, EPI_SUB = 1;

// C (op)= acc for one warp's 64 x 32 part of a tile whose origin is (r0, c0) and size tile_bm x tile_bn.
template <int EPI>
__device__ __forceinline__ void gemm_epilogue(const GemmParams& p, double (&acc)[MI][NI][2], int r0, int c0,
                                              int tile_bm, int tile_bn, int rbase, int cbase) {
  double* __restrict__ Cg = p.C;
  const bool vec_ok = ((p.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
  // tile fully inside the matrix and (if masked) fully below the diagonal: batched 16-byte read-modify-write
  const bool interior = vec_ok && (r0 + tile_bm <= p.M) && (c0 + tile_bn <= p.N) &&
                        (c0 + tile_bn - 1 <= diag_limit(p, r0));
  if (interior) {
#pragma unroll
    for (int half = 0; half < 2; half++) {
      double2 cv[MI / 2][NI];
      if (EPI == EPI_SUB) {
#pragma unroll
        for (int m = 0; m < MI / 2; m++)
#pragma unroll
          for (int ni = 0; ni < NI; ni++)
            cv[m][ni] = *reinterpret_cast<const double2*>(
                Cg + (long long)(rbase + (half * (MI / 2) + m) * 8) * p.ldc + cbase + ni * 8);
      }
#pragma unroll
      for (int m = 0; m < MI / 2; m++)
#pragma unroll
        for (int ni = 0; ni < NI; ni++) {
          const int mi = half * (MI / 2) + m;
          double2 v;
          if (EPI == EPI_SUB) {
            v.x = cv[m][ni].x - acc[mi][ni][0];
            v.y = cv[m][ni].y - acc[mi][ni][1];
          } else {
            v = make_double2(acc[mi][ni][0], acc[mi][ni][1]);
          }
          *reinterpret_cast<double2*>(Cg + (long long)(rbase + mi * 8) * p.ldc + cbase + ni * 8) = v;
        }
    }
    return;
  }
#pragma unroll
  for (int mi = 0; mi < MI; mi++) {
    const int r = rbase + mi * 8;
    if (r >= p.M) continue;
    const long long lim = diag_limit(p, r);
#pragma unroll
    for (int ni = 0; ni < NI; ni++) {
      const int c = cbase + ni * 8;
      const bool ok0 = c < p.N && c <= lim;
      const bool ok1 = (c + 1) < p.N && (c + 1) <= lim;
      double* dst = Cg + (long long)r * p.ldc + c;
      if (ok0 && ok1 && vec_ok) {
        double2* d2 = reinterpret_cast<double2*>(dst);
        if (EPI == EPI_STORE) {
          *d2 = make_double2(acc[mi][ni][0], acc[mi][ni][1]);
        } else {
          double2 v = *d2;
          v.x -= acc[mi][ni][0];
          v.y -= acc[mi][ni][1];
          *d2 = v;
        }
      } else {
        if (ok0) dst[0] = (EPI == EPI_STORE) ? acc[mi][ni][0] : dst[0] - acc[mi][ni][0];
        if (ok1) dst[1] = (EPI == EPI_STORE) ? acc[mi][ni][1] : dst[1] - acc[mi][ni][1];
      }
    }
  }
}

template <typename Cfg, bool ALIGN16, int EPI>
__global__ void __launch_bounds__(Cfg::THREADS, Cfg::MIN_BLOCKS) gemm_kernel(const GemmParams p) {
  extern __shared__ __align__(16) double smem[];
  const int ntn = (p.N + Cfg::BN - 1) / Cfg::BN;
  int ti, tj;
  decode_tile<Cfg::Q>(blockIdx.x, ntn, p.lower && p.cyc_db == 0, ti, tj);
  const int r0 = ti * Cfg::BM, c0 = tj * Cfg::BN;
  if (p.cyc_db != 0 && c0 > diag_limit(p, min(r0 + Cfg::BM, p.M) - 1)) return;   // tile above the diagonal
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rbase = r0 + (warp / Cfg::WARPS_N) * 64 + (lane >> 2);
  const int cbase = c0 + (warp % Cfg::WARPS_N) * 32 + (lane & 3) * 2;
  if (EPI == EPI_SUB) {
    // pull this thread's part of the C tile towards L2 while the contraction runs (no registers held)
#pragma unroll
    for (int mi = 0; mi < MI; mi++) {
      const int r = rbase + mi * 8;
      if (r < p.M && cbase < p.N && (lane & 3) == 0)
        asm volatile("prefetch.global.L2 [%0];" ::"l"(p.C + (long long)r * p.ldc + cbase));
    }
  }
  double acc[MI][NI][2];
  const int k0 = p.k_from_row ? p.k_row0 + r0 : 0;   // multiples of 64: alignment of the operands is kept
  gemm_mainloop<Cfg, ALIGN16>(acc, p.A + (long long)r0 * p.lda + k0, p.lda, min(Cfg::BM, p.M - r0),
                              p.B + (long long)c0 * p.ldb + k0, p.ldb, min(Cfg::BN, p.N - c0), p.K - k0, smem);
  gemm_epilogue<EPI>(p, acc, r0, c0, Cfg::BM, Cfg::BN, rbase, cbase);
}

// TMA-fed persistent variant (tma_core.cuh): trailing / inner updates C -= A B^T
struct EpiSubTma {
  using Params = GemmParams;
  static __device__ __forceinline__ void apply(const Params& p, double (&acc)[MI][NI][2], int r0, int c0, int wm,
                                               int wn, int lane) {
    gemm_epilogue<EPI_SUB>(p, acc, r0, c0, TM_BM, TM_BN, r0 + wm * 64 + (lane >> 2), c0 + wn * 32 + (lane & 3) * 2);
  }
};

// out-of-place C = A B^T (lower-masked when p.lower)
struct EpiStoreTma {
  using Params = GemmParams;
  static __device__ __forceinline__ void apply(const Params& p, double (&acc)[MI][NI][2], int r0, int c0, int wm,
                                               int wn, int lane) {
    gemm_epilogue<EPI_STORE>(p, acc, r0, c0, TM_BM, TM_BN, r0 + wm * 64 + (lane >> 2), c0 + wn * 32 + (lane & 3) * 2);
  }
};

template <class Epi>
cudaError_t launch_gemm_tma(cudaStream_t s, const GemmParams& p) {
  CUtensorMap ma, mb;
  if (!make_tmap(&ma, p.A, p.M, p.K, p.lda, TM_BM) || !make_tmap(&mb, p.B, p.N, p.K, p.ldb, TM_BN))
    return cudaErrorInvalidValue;
  const int tri = p.lower && p.cyc_db == 0;
  TmaShape sh{p.M, p.N, p.K, tri, count_tiles<TileTma>(p.M, p.N, tri), p.lower ? p.cyc_db : 0, p.cyc_p, p.base_shift,
              p.k_from_row, p.k_upto_col};
  sh.cyc_alt = p.lower ? p.cyc_alt : 0;
  sh.k_row0 = p.k_row0;
  if (sh.cyc_db != 0) sh.tiles = tma_cyc_count_tiles(sh);       // active tiles only
  int sms = device_sm_count() - p.sm_reserve;
  if (sms < 8) sms = 8;
  cudaError_t e = launch_tma_gemm<Epi>(s, ma, mb, sh, p, sms);
  instr().launches++;
  return e;
}
cudaError_t launch_gemm_sub_tma(cudaStream_t s, const GemmParams& p) { return launch_gemm_tma<EpiSubTma>(s, p); }

template <typename Cfg, int EPI>
cudaError_t launch_gemm_cfg(cudaStream_t s, const GemmParams& p) {
  long long tiles = count_tiles<Cfg>(p.M, p.N, p.lower && p.cyc_db == 0);
  bool a16 = (p.lda % 2 == 0) && (p.ldb % 2 == 0) && ((reinterpret_cast<uintptr_t>(p.A) & 15) == 0) &&
             ((reinterpret_cast<uintptr_t>(p.B) & 15) == 0);
  auto kern = a16 ? gemm_kernel<Cfg, true, EPI> : gemm_kernel<Cfg, false, EPI>;
  cudaError_t e = configure_kernel_once(reinterpret_cast<const void*>(kern), Cfg::SMEM_BYTES, true);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)tiles, Cfg::THREADS, Cfg::SMEM_BYTES, s>>>(p);
  instr().launches++;
  return cudaGetLastError();
}

template <int EPI>
cudaError_t launch_gemm_t(cudaStream_t s, const GemmParams& p) {
  if (p.M <= 0 || p.N <= 0) return cudaSuccess;
  // The TRSM runs IN PLACE (C aliases A): a CTA must own whole rows of the <= 128-column panel, otherwise one
  // column tile could overwrite rows a sibling tile is still reading -> always the 128 x 128 tile for EPI_STORE.
  if (EPI == EPI_STORE && p.M <= 1024 && tile_variant() == 0) return launch_gemm_cfg<TileSmallWide, EPI>(s, p);
  if (EPI == EPI_STORE || tile_variant() == 1) return launch_gemm_cfg<TileBig, EPI>(s, p);
  // fewer 128 x 64 tiles than the persistent kernel has math groups on ~1/3 of the GPU: 64 x 64 tiles, one per CTA
  if (tile_variant() == 0 && p.cyc_db == 0 && !p.k_from_row && !p.k_upto_col &&
      count_tiles<TileTma>(p.M, p.N, p.lower) < 96)
    return launch_gemm_cfg<TileSmall, EPI>(s, p);
  if (tile_variant() == 0 && tma_operand_ok(p.A, p.lda) && tma_operand_ok(p.B, p.ldb)) return launch_gemm_sub_tma(s, p);
  return launch_gemm_cfg<TilePair, EPI>(s, p);
}

// ---------------------------------------------------------------------------------------------------------
// Diagonal block (w <= 128): Cholesky factor AND its inverse in one CTA, blocked by 32 columns.
//   per 32-block b:  warp 0 factors the 32x32 diagonal block in registers (lane = row, pivots and column
//                    entries exchanged with warp shuffles) and inverts the factor (lane = column, forward
//                    substitution with broadcast shared-memory reads);
//                    all warps: panel below = S_ib * inv(L_bb)^T and trailing update S -= P P^T, both as
//                    8x8x4 DMMA tiles straight out of shared memory (row strips of 8, conflict-free ld 132);
//   afterwards inv(L) is assembled block-wise:  X_ii = inv(L_ii),  X_ik = -X_ii * sum_{m=k}^{i-1} L_im X_mk,
//   the off-diagonal X blocks living in the otherwise unused upper triangle of the shared-memory matrix.
// ---------------------------------------------------------------------------------------------------------
constexpr int PF_THREADS = 256;
constexpr int PF_WARPS = PF_THREADS / 32;
constexpr int NBLK = PB / DB;
constexpr int PF_SMEM_BYTES = (PB * GLD + NBLK * DB * MLD + 64) * 8;

__global__ void __launch_bounds__(PF_THREADS, 1)
potf2_trtri_kernel(double* __restrict__ A, long long lda, int w, double* __restrict__ Linv,
                   double* __restrict__ logdet, int* __restrict__ info, int gcol0, long long* __restrict__ clk) {
  int nclk = 0;
#define PF_CLK() do { if (clk != nullptr && threadIdx.x == 0) clk[nclk++] = clock64(); } while (0)
  PF_CLK();
  extern __shared__ __align__(16) double sm[];
  double* G = sm;                          // [128][132]
  double* Mi = G + PB * GLD;               // NBLK x [DB][MLD] inverse diagonal blocks
  double* red = Mi + NBLK * DB * MLD;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nblk = (w + DB - 1) / DB;
  const int wp = nblk * DB;                // padded size (identity padding)

  // stage the lower triangle (the upper part of G is scratch for the inverse assembly and must start at zero);
  // 8 independent 16-byte slots per thread and batch so the global loads overlap
  for (int base = 0; base < wp * (PB / 2); base += PF_THREADS * 8) {
    double2 g[8];
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const int idx = base + u * PF_THREADS + tid;
      const int i = idx >> 6, c = (idx & 63) * 2;
      g[u] = make_double2(0.0, 0.0);
      if (idx < wp * (PB / 2) && i < w && c <= i) {
        const double* src = A + (long long)i * lda + c;
        g[u].x = src[0];
        if (c + 1 <= i) g[u].y = src[1];
      }
    }
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const int idx = base + u * PF_THREADS + tid;
      if (idx >= wp * (PB / 2)) continue;
      const int i = idx >> 6, c = (idx & 63) * 2;
      if (i >= w) {
        if (c == i) g[u].x = 1.0;
        if (c + 1 == i) g[u].y = 1.0;
      }
      G[i * GLD + c] = g[u].x;
      G[i * GLD + c + 1] = g[u].y;
    }
  }
  __syncthreads();
  PF_CLK();   // 1: staged

  // In-CTA look-ahead: the serial part (warp 0 factoring + inverting a 16 x 16 diagonal block in registers, ~2.8 us)
  // used to alternate with the panel / trailing-update phases of the other warps.  Now, once block b's panel is solved,
  // warp 0 updates ONLY the next diagonal block and factors it while warps 1..7 apply the rest of block b's trailing
  // update - the update hides under the pivot chain instead of adding to it.
  int bad = 0;
  if (warp == 0) diag_factor_invert(G, Mi, lane, 0, &bad);
  __syncthreads();
  PF_CLK();   // diag 0
  for (int b = 0; b < nblk; b++) {
    const int b0 = b * DB;
    const int r_first = b0 + DB;
    const int nstrips = (wp - r_first) / 8;
    // panel: rows below, P = S_ib * inv(L_bb)^T   (a warp owns whole 8-row strips -> in place)
    for (int s = warp; s < nstrips; s += PF_WARPS) {
      const int r0 = r_first + s * 8;
      double af[KS];
      const double* ap = G + (r0 + (lane >> 2)) * GLD + b0 + (lane & 3);
#pragma unroll
      for (int ks = 0; ks < KS; ks++) af[ks] = ap[ks * 4];
      double acc[NT][2];
#pragma unroll
      for (int nt = 0; nt < NT; nt++) {
        acc[nt][0] = acc[nt][1] = 0.0;
        const double* bp = Mi + b * DB * MLD + (nt * 8 + (lane >> 2)) * MLD + (lane & 3);
#pragma unroll
        for (int ks = 0; ks < KS; ks++)
          if (ks <= 2 * nt + 1) dmma8x8x4(acc[nt], af[ks], bp[ks * 4]);   // inv(L) is lower triangular
      }
      __syncwarp();
      double* op = G + (r0 + (lane >> 2)) * GLD + b0 + (lane & 3) * 2;
#pragma unroll
      for (int nt = 0; nt < NT; nt++) { op[nt * 8] = acc[nt][0]; op[nt * 8 + 1] = acc[nt][1]; }
    }
    __syncthreads();
    PF_CLK();   // panel
    // trailing update S_ic -= P_i P_c^T for r_first <= c-tile <= row strip.  Strips 0 .. NT-1 only touch the next
    // diagonal block: warp 0 takes them and goes on to factor that block; the other warps share the remaining strips.
    if (warp == 0) {
      for (int s = 0; s < NT && s < nstrips; s++) {
        const int r0 = r_first + s * 8;
        double af[KS];
        const double* ap = G + (r0 + (lane >> 2)) * GLD + b0 + (lane & 3);
#pragma unroll
        for (int ks = 0; ks < KS; ks++) af[ks] = ap[ks * 4];
        for (int c0 = r_first; c0 <= r0; c0 += 8) {
          double acc[2] = {0.0, 0.0};
          const double* bp = G + (c0 + (lane >> 2)) * GLD + b0 + (lane & 3);
#pragma unroll
          for (int ks = 0; ks < KS; ks++) dmma8x8x4(acc, af[ks], bp[ks * 4]);
          double* cp = G + (r0 + (lane >> 2)) * GLD + c0 + (lane & 3) * 2;
          cp[0] -= acc[0];
          cp[1] -= acc[1];
        }
      }
      __syncwarp();
      if (b + 1 < nblk) diag_factor_invert(G + r_first * GLD + r_first, Mi + (b + 1) * DB * MLD, lane, r_first, &bad);
    } else {
      for (int s = NT + (warp - 1); s < nstrips; s += PF_WARPS - 1) {
        const int r0 = r_first + s * 8;
        double af[KS];
        const double* ap = G + (r0 + (lane >> 2)) * GLD + b0 + (lane & 3);
#pragma unroll
        for (int ks = 0; ks < KS; ks++) af[ks] = ap[ks * 4];
        for (int c0 = r_first; c0 <= r0; c0 += 8) {
          double acc[2] = {0.0, 0.0};
          const double* bp = G + (c0 + (lane >> 2)) * GLD + b0 + (lane & 3);
#pragma unroll
          for (int ks = 0; ks < KS; ks++) dmma8x8x4(acc, af[ks], bp[ks * 4]);
          double* cp = G + (r0 + (lane >> 2)) * GLD + c0 + (lane & 3) * 2;
          cp[0] -= acc[0];
          cp[1] -= acc[1];
        }
      }
    }
    __syncthreads();
    PF_CLK();   // update + next diag
  }

  // ---- inverse assembly: X_ik (i > k) is kept at block position (k, i) of G (upper triangle, untransposed)
  for (int dist = 1; dist < nblk; dist++) {
    const int npairs = nblk - dist;
    // phase A: T_ik = sum_{m=k}^{i-1} L_im X_mk ; NT*NT output tiles per pair
    for (int u = warp; u < npairs * NT * NT; u += PF_WARPS) {
      const int k = u / (NT * NT), t = u % (NT * NT), i = k + dist;
      const int tr = (t / NT) * 8, tc = (t % NT) * 8;
      double acc[2] = {0.0, 0.0};
      for (int m = k; m < i; m++) {
        const double* Lim = G + (i * DB + tr) * GLD + m * DB;
        if (m == k) tile_nn(acc, Lim, GLD, Mi + k * DB * MLD + tc, MLD, KS, lane);
        else tile_nn(acc, Lim, GLD, G + (k * DB) * GLD + m * DB + tc, GLD, KS, lane);
      }
      // T is written to its final place (k, i); nobody reads that block in this phase
      double* tp = G + (k * DB + tr + (lane >> 2)) * GLD + i * DB + tc + (lane & 3) * 2;
      tp[0] = acc[0];
      tp[1] = acc[1];
    }
    __syncthreads();
    // phase B: X_ik = -inv(L_ii) T_ik in place; a warp owns an 8-column strip of one block
    for (int u = warp; u < npairs * NT; u += PF_WARPS) {
      const int k = u / NT, tc = (u % NT) * 8, i = k + dist;
      double* T = G + (k * DB) * GLD + i * DB + tc;
      double bf[KS];
#pragma unroll
      for (int ks = 0; ks < KS; ks++) bf[ks] = T[(ks * 4 + (lane & 3)) * GLD + (lane >> 2)];
      double acc[NT][2];
#pragma unroll
      for (int rt = 0; rt < NT; rt++) {
        acc[rt][0] = acc[rt][1] = 0.0;
        const double* ap = Mi + i * DB * MLD + (rt * 8 + (lane >> 2)) * MLD + (lane & 3);
#pragma unroll
        for (int ks = 0; ks < KS; ks++)
          if (ks <= 2 * rt + 1) dmma8x8x4(acc[rt], ap[ks * 4], bf[ks]);
      }
      __syncwarp();
#pragma unroll
      for (int rt = 0; rt < NT; rt++) {
        double* op = T + (rt * 8 + (lane >> 2)) * GLD + (lane & 3) * 2;
        op[0] = -acc[rt][0];
        op[1] = -acc[rt][1];
      }
    }
    __syncthreads();
  }
  PF_CLK();   // inverse assembled

  // write back: L and inv(L), lower parts only (the strict upper triangle of A is never touched; the part of
  // the inverse above the diagonal is zero and the workspace block was zero-filled when the factorisation began)
#pragma unroll 4
  for (int idx = tid; idx < wp * (PB / 2); idx += PF_THREADS) {
    const int i = idx >> 6, c = (idx & 63) * 2;
    if (c > i) continue;
    if (i < w) {
      double* dst = A + (long long)i * lda + c;
      dst[0] = G[i * GLD + c];
      if (c + 1 <= i) dst[1] = G[i * GLD + c + 1];
    }
    double2 v = make_double2(0.0, 0.0);
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int cc = c + e;
      double x = 0.0;
      if (cc <= i) {
        const int bi = i / DB, bc = cc / DB;
        x = (bi == bc) ? Mi[bi * DB * MLD + (i - bi * DB) * MLD + (cc - bc * DB)]
                       : G[(bc * DB + (i - bi * DB)) * GLD + bi * DB + (cc - bc * DB)];
      }
      if (e == 0) v.x = x; else v.y = x;
    }
    *reinterpret_cast<double2*>(Linv + (long long)i * PB + c) = v;
  }
  // sum of log L_ii in a fixed order
  double lg = (tid < w) ? log(G[tid * GLD + tid]) : 0.0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lg += __shfl_xor_sync(0xffffffffu, lg, o);
  if (lane == 0) red[warp] = lg;
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int k = 0; k < PB / 32; k++) s += red[k];
    atomicAdd(logdet, s);                       // kernels on one stream: still a fixed order, no load latency
    if (bad != 0) atomicCAS(info, 0, gcol0 + bad);
  }
  PF_CLK();   // written back
#undef PF_CLK
}

}  // namespace

int debug_gemm_occupancy(int variant) {
  int nb = -1;
  if (variant == 1) {
    auto k = gemm_kernel<TileBig, true, EPI_SUB>;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, TileBig::SMEM_BYTES);
    cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k, TileBig::THREADS, TileBig::SMEM_BYTES);
  } else {
    auto k = gemm_kernel<TilePair, true, EPI_SUB>;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, TilePair::SMEM_BYTES);
    cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k, TilePair::THREADS, TilePair::SMEM_BYTES);
  }
  return nb;
}

cudaError_t launch_gemm_store(cudaStream_t s, const GemmParams& p) { return launch_gemm_t<EPI_STORE>(s, p); }
cudaError_t launch_gemm_sub(cudaStream_t s, const GemmParams& p) { return launch_gemm_t<EPI_SUB>(s, p); }
cudaError_t launch_gemm_store_tma(cudaStream_t s, const GemmParams& p) {
  if (p.M <= 0 || p.N <= 0) return cudaSuccess;
  if (!tma_operand_ok(p.A, p.lda) || !tma_operand_ok(p.B, p.ldb)) return cudaErrorInvalidValue;
  return launch_gemm_tma<EpiStoreTma>(s, p);
}
cudaError_t launch_gemm_store_lower(cudaStream_t s, const GemmParams& p) {
  if (p.M <= 0 || p.N <= 0) return cudaSuccess;
  if (tile_variant() == 0 && tma_operand_ok(p.A, p.lda) && tma_operand_ok(p.B, p.ldb))
    return launch_gemm_tma<EpiStoreTma>(s, p);
  return launch_gemm_cfg<TilePair, EPI_STORE>(s, p);
}

cudaError_t launch_potf2_trtri(cudaStream_t s, double* A, long long lda, int w, double* Linv, double* logdet,
                               int* info, int global_col0) {
  cudaError_t e = configure_kernel_once(reinterpret_cast<const void*>(potf2_trtri_kernel), PF_SMEM_BYTES, false);
  if (e != cudaSuccess) return e;
  potf2_trtri_kernel<<<1, PF_THREADS, PF_SMEM_BYTES, s>>>(A, lda, w, Linv, logdet, info, global_col0, potf2_clock_buffer());
  instr().launches++;
  return cudaGetLastError();
}

// Plain right-looking two-level factorisation on ONE stream (also the building block of the look-ahead variant,
// where it factors the NB x NB diagonal blocks).
// rows touched while factoring the outer panel that ends at column c1 (see potrf_trapezoid: identity-carried rows)
static inline long long active_rows(long long Mtot, long long ident_row0, long long c1) {
  if (ident_row0 < 0) return Mtot;
  return (ident_row0 + c1 < Mtot) ? ident_row0 + c1 : Mtot;
}

static cudaError_t potrf_serial(cudaStream_t s, double* A, long long lda, long long Mfull, long long N, int NB,
                                double* Linv_base, double* logdet, int* info, long long linv_stride, int gcol_base,
                                bool zero_linv = true, long long ident_row0 = -1) {
  cudaError_t e;
  if (zero_linv) {     // the diagonal kernel only writes the lower part of each inverse block
    const long long blocks = linv_stride == 0 ? 1 : (N + PB - 1) / PB;
    e = cudaMemsetAsync(Linv_base, 0, (size_t)blocks * PB * PB * sizeof(double), s);
    if (e != cudaSuccess) return e;
  }
  for (long long c0 = 0; c0 < N; c0 += NB) {
    const long long c1 = (c0 + NB < N) ? c0 + NB : N;
    const long long Mtot = active_rows(Mfull, ident_row0, c1);
    for (long long j0 = c0; j0 < c1; j0 += PB) {
      const long long j1 = (j0 + PB < N) ? j0 + PB : N;
      const int w = (int)(j1 - j0);
      double* Linv_ws = Linv_base + (j0 / PB) * linv_stride;
      e = launch_potf2_trtri(s, A + j0 * lda + j0, lda, w, Linv_ws, logdet, info, gcol_base + (int)j0);
      if (e != cudaSuccess) return e;
      // identity-carried rows below ident_row0 + j1 are the only ones with entries in this 128-block so far
      const long long Mj = active_rows(Mfull, ident_row0, j1);
      if (Mj > j1) {
        GemmParams t{};   // panel rows <- panel rows * inv(L_jj)^T   (in place: one CTA owns whole rows)
        t.A = A + j1 * lda + j0; t.lda = lda;
        t.B = Linv_ws;           t.ldb = PB;
        t.C = A + j1 * lda + j0; t.ldc = lda;
        t.M = (int)(Mj - j1); t.N = w; t.K = w; t.lower = 0;
        e = launch_gemm_store(s, t);
        if (e != cudaSuccess) return e;
        if (j1 < c1) {    // remaining columns of the outer panel
          GemmParams u{};
          u.A = A + j1 * lda + j0; u.lda = lda;
          u.B = A + j1 * lda + j0; u.ldb = lda;
          u.C = A + j1 * lda + j1; u.ldc = lda;
          u.M = (int)(Mj - j1); u.N = (int)(c1 - j1); u.K = w; u.lower = 1;
          e = launch_gemm_sub(s, u);
          if (e != cudaSuccess) return e;
        }
      }
    }
    if (c1 < N) {         // trailing update with the whole outer panel, K = NB
      GemmParams u{};
      u.A = A + c1 * lda + c0; u.lda = lda;
      u.B = A + c1 * lda + c0; u.ldb = lda;
      u.C = A + c1 * lda + c1; u.ldc = lda;
      u.M = (int)(Mtot - c1); u.N = (int)(N - c1); u.K = (int)(c1 - c0); u.lower = 1;
      if (instr().time_updates) {
        // algorithmic flops: lower triangle of the square part + the carried rows, 2 flop per MAC
        const double nsq = (double)(N - c1), extra = (double)(Mtot - N);
        instr_begin_update(s, (nsq * (nsq + 1.0) + 2.0 * extra * nsq) * (double)u.K);
      }
      e = launch_gemm_sub(s, u);
      if (instr().time_updates) instr_end_update(s);
      if (e != cudaSuccess) return e;
    }
  }
  return cudaSuccess;
}

// ---- look-ahead ---------------------------------------------------------------------------------------------
// Per outer panel p:   side stream : factor the NB x NB diagonal block (latency-bound chain of small kernels)
//                      main stream : TRSM of the rows below, update of the NEXT panel's block column (update_a),
//                                    then the bulk of the trailing matrix (update_b).
// The diagonal block of panel p+1 only needs update_a(p), so its chain runs under update_b(p).  The persistent
// update kernel would otherwise hold every SM, so for trailing matrices small enough that the chain matters
// update_b leaves a few SMs free.
namespace {
// side stream + events of the current device's context (context.cuh), created on first use
DeviceCtx* lookahead_ctx() {
  DeviceCtx& c = dctx();
  if (!c.la_ok) {
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (cudaStreamCreateWithPriority(&c.side, cudaStreamNonBlocking, hi) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&c.ev_fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&c.ev_diag, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&c.ev_a, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    c.la_ok = true;
  }
  return &c;
}
}  // namespace

cudaError_t potrf_trapezoid(cudaStream_t s, double* A, long long lda, long long Mfull, long long N, int NB,
                            double* Linv_base, double* logdet, int* info, long long linv_stride,
                            long long ident_row0, double* fused_ws, bool want_L) {
  if (NB < PB) NB = PB;
  NB = (NB / PB) * PB;
  if (NB > LINV_BLOCKS * PB) NB = LINV_BLOCKS * PB;
  DeviceCtx* la = (lookahead_mode() != 0 && linv_stride == 0 && N > NB) ? lookahead_ctx() : nullptr;
  if (la == nullptr)
    return potrf_serial(s, A, lda, Mfull, N, NB, Linv_base, logdet, info, linv_stride, 0, true, ident_row0);

#define LA_CK(call)                 \
  do {                              \
    cudaError_t e__ = (call);       \
    if (e__ != cudaSuccess) return e__; \
  } while (0)
  const long long ls = (long long)PB * PB;          // one inverse block per 128 columns of the current panel
  // single-launch panel solve (see kernels.cuh): needs the extra workspace and TMA-addressable operands
  const bool fused = fused_ws != nullptr && la->fused_panel != 0 && tile_variant() == 0 && tma_operand_ok(A, lda);
  double* const W = fused_ws;
  double* const Pb = fused ? fused_ws + (size_t)FUSED_LD * FUSED_LD : nullptr;
  const long long ldp = FUSED_LD;
  LA_CK(cudaEventRecord(la->ev_fork, s));
  LA_CK(cudaStreamWaitEvent(la->side, la->ev_fork, 0));
  const long long tail = NB >= 4 * PB ? la->tail_cols : 0;
  for (long long c0 = 0; c0 < N; c0 += NB) {
    if (c0 > 0 && N - c0 <= tail) {
      // Tail: once the trailing matrix is this small every 512-wide panel costs ~0.5 ms of chain (diagonal block,
      // inverse, one-wave panel solve) against < 0.1 ms of update.  The plain single-stream 128-column factorisation
      // (diagonal kernel + one TRSM + one update per step, ~75-95 us per 128 columns) is faster from here on.
      LA_CK(cudaEventRecord(la->ev_diag, la->side));          // the side stream's last update_a
      LA_CK(cudaStreamWaitEvent(s, la->ev_diag, 0));
      return potrf_serial(s, A + c0 * lda + c0, lda, Mfull - c0, N - c0, PB, Linv_base, logdet, info, 0, (int)c0, false,
                          ident_row0);
    }
    const long long c1 = (c0 + NB < N) ? c0 + NB : N;
    const int w = (int)(c1 - c0);
    const long long Mtot = active_rows(Mfull, ident_row0, c1);
    const long long m = Mtot - c1;
    // side: diagonal block (w x w) with its block inverses, then (fused) its full inverse W
    LA_CK(potrf_serial(la->side, A + c0 * lda + c0, lda, w, w, NB, Linv_base, logdet, info, ls, (int)c0, c0 == 0));
    if (fused && m > 0) {
      double* outs[1] = {W};
      LA_CK(launch_assemble_inverse(la->side, A + c0 * lda + c0, lda, w, Linv_base, outs, 1, FUSED_LD, nullptr));
    }
    LA_CK(cudaEventRecord(la->ev_diag, la->side));
    LA_CK(cudaStreamWaitEvent(s, la->ev_diag, 0));
    // main: rows below the diagonal block <- rows * L_pp^-T
    if (m > 0 && fused) {
      GemmParams t{};     // P = R W^T, contraction cut at W's diagonal, out of place (column tiles of one row block
      t.A = A + c1 * lda + c0; t.lda = lda;     // read each other's input columns: in place would race)
      t.B = W;                 t.ldb = FUSED_LD;
      t.C = Pb;                t.ldc = ldp;
      t.M = (int)m; t.N = w; t.K = w; t.lower = 0; t.k_upto_col = 1;
      LA_CK(launch_gemm_store_tma(s, t));
    } else if (m > 0) {
      double* R = A + c1 * lda + c0;            // 128-block substitution, in place
      for (long long j0 = 0; j0 < w; j0 += PB) {
        const long long j1 = (j0 + PB < w) ? j0 + PB : w;
        GemmParams t{};
        t.A = R + j0; t.lda = lda;
        t.B = Linv_base + (j0 / PB) * ls; t.ldb = PB;
        t.C = R + j0; t.ldc = lda;
        t.M = (int)m; t.N = (int)(j1 - j0); t.K = (int)(j1 - j0); t.lower = 0;
        LA_CK(launch_gemm_store(s, t));
        if (j1 < w) {
          GemmParams u{};
          u.A = R + j0; u.lda = lda;
          u.B = A + (c0 + j1) * lda + c0 + j0; u.ldb = lda;
          u.C = R + j1; u.ldc = lda;
          u.M = (int)m; u.N = (int)(w - j1); u.K = (int)(j1 - j0); u.lower = 0;
          LA_CK(launch_gemm_sub(s, u));
        }
      }
    }
    LA_CK(cudaEventRecord(la->ev_a, s));                    // panel p solved
    if (m > 0 && fused) {
      // copy back what somebody reads later: carried rows (>= N) always, the square rows of L only on request
      const long long r_first = want_L ? c1 : (N > c1 ? N : c1);
      if (r_first < Mtot)
        LA_CK(cudaMemcpy2DAsync(A + r_first * lda + c0, (size_t)lda * 8, Pb + (r_first - c1) * ldp, (size_t)ldp * 8,
                                (size_t)w * 8, (size_t)(Mtot - r_first), cudaMemcpyDeviceToDevice, s));
    }
    if (c1 >= N) break;
    // panel operands of the trailing updates: the panel buffer (fused) or the solved columns of A
    const double* Pop = fused ? Pb : A + c1 * lda + c0;     // row 0 = global row c1
    const long long ldo = fused ? ldp : lda;
    // Look-ahead split: the NEXT diagonal block (na x na, lower) is updated first, on the side stream, so that its
    // factorisation chain can start at once; everything else - including the rest of the next block column - is one
    // well-filled launch on the main stream that leaves a few SMs to the chain when the trailing matrix is small.
    const long long na = (c1 + NB < N) ? NB : N - c1;
    LA_CK(cudaStreamWaitEvent(la->side, la->ev_a, 0));
    {
      GemmParams u{};
      u.A = Pop; u.lda = ldo;
      u.B = Pop; u.ldb = ldo;
      u.C = A + c1 * lda + c1; u.ldc = lda;
      u.M = (int)na; u.N = (int)na; u.K = w; u.lower = 1;
      LA_CK(launch_gemm_sub(la->side, u));
    }
    const long long cb = c1 + na;
    if (cb < Mtot) {
      // rows [cb, Mtot) x cols [c1, N): local row r may touch columns <= r + na (plain shifted diagonal = the
      // block-row-cyclic mask with one huge block)
      GemmParams u{};
      u.A = Pop + (cb - c1) * ldo; u.lda = ldo;
      u.B = Pop; u.ldb = ldo;
      u.C = A + cb * lda + c1; u.ldc = lda;
      u.M = (int)(Mtot - cb); u.N = (int)(N - c1); u.K = w; u.lower = 1;
      u.cyc_db = 1 << 30; u.cyc_p = 1; u.base_shift = (int)na;
      u.sm_reserve = lookahead_reserve()[(N - cb < 24000) ? 0 : 1];
      if (instr().time_updates) {
        const double nb = (double)(N > cb ? N - cb : 0), extra = (double)(Mtot - (N > cb ? N : cb));
        const double pairs = 0.5 * nb * (nb + 1.0) + nb * (double)na + extra * (double)(N - c1);
        instr_begin_update(s, 2.0 * pairs * (double)w);
      }
      LA_CK(launch_gemm_sub(s, u));
      if (instr().time_updates) instr_end_update(s);
    }
  }
  // the side stream's last work (diagonal block of the last panel) was joined through ev_diag
#undef LA_CK
  return cudaSuccess;
}

}  // namespace smnngp

// Shared device helpers for the sm_100a FP64 path: DMMA.8x8x4 wrapper, cp.async staging, tile decode.
// FP64 has no tcgen05 kind on Blackwell; the FP64 tensor path is mma.sync.m8n8k4 (SASS DMMA.8x8x4),
// measured at 37.1 TFLOP/s register-resident on B200 (profiles/r01_fp64_peak.txt).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

namespace smnngp {

constexpr int BK = 16;           // k-slab per pipeline stage
constexpr int LDK = BK + 4;      // padded smem row (doubles): 160 B rows -> conflict-free 8-row x 4-k fragment loads
constexpr int MI = 8;            // m8 blocks per warp tile (warp tile = 64 x 32)
constexpr int NI = 4;            // n8 blocks per warp tile

// CTA tile configuration of the GEMM core.  Warp tile is fixed at 64 x 32 (64 FP64 accumulators per thread).
//   TilePair: 128 x 64, 4 warps, 90 KB ring -> TWO CTAs per SM: while one CTA is in its prologue / epilogue the
//             other one owns the FP64 pipe (ping-pong), which is what keeps DMMA issue saturated;
//   TileBig : 128 x 128, 8 warps, 160 KB ring, one CTA per SM (round-1 first version, kept for comparison).
template <int BM_, int BN_, int STAGES_, int MINB_>
struct TileCfg {
  static constexpr int BM = BM_, BN = BN_, STAGES = STAGES_, MIN_BLOCKS = MINB_;
  static constexpr int WARPS_M = BM / 64, WARPS_N = BN / 32;
  static constexpr int THREADS = WARPS_M * WARPS_N * 32;
  static constexpr int STAGE_DOUBLES = (BM + BN) * LDK;
  static constexpr int SMEM_BYTES = STAGES * STAGE_DOUBLES * 8;
  static constexpr int Q = BM / BN;    // column tiles per row tile on the diagonal
};
using TilePair = TileCfg<128, 64, 3, 2>;   // 3 x 30 KB (padded) = 90 KB -> two CTAs fit in 228 KB
using TileBig = TileCfg<128, 128, 4, 1>;
// Small problems (the TRSM / inner updates INSIDE a 512-wide diagonal block: <= 384 rows): with 128-row tiles they ran
// on 3-12 CTAs and were bound by the FP64 rate of those few SMs (~17 us each, on the critical path of every panel).
// Half-size tiles spread the same flops over 2-4x as many SMs.
using TileSmall = TileCfg<64, 64, 3, 2>;        // 2 warps, updates C -= A B^T
using TileSmallWide = TileCfg<64, 128, 3, 1>;   // 4 warps, in-place TRSM (a CTA owns whole rows of the <= 128-col panel)

enum Act { ACT_RELU = 0, ACT_ERF = 1 };
enum Arch { ARCH_MLP = 0, ARCH_RESNET = 1 };
enum Kind { KIND_GAUSS = 0, KIND_STUDENT_T = 1 };
// which diagonal shift the Gram epilogue adds (values live in the device scalar block, see scal layout)
enum Shift { SHIFT_NONE = 0, SHIFT_EPS_ABS = 1, SHIFT_EPS_REL = 2, SHIFT_LIK = 3 };
enum GramOut { OUT_FULL = 0, OUT_LOWER = 1 };

// device scalar block ("scal"), doubles
constexpr int SC_TRMEAN = 0;     // tr(K)/N of the un-shifted Gram
constexpr int SC_SHIFT0 = 1;     // scal[SC_SHIFT0 + shift] = shift value: [0, eps, eps*tr/N, 1e-6*a/b]
constexpr int SC_LOGDET = 5;     // running sum of log L_ii
constexpr int SC_QUAD = 6;       // ||L^-1 y||^2
constexpr int SC_COUNT = 16;

__device__ __forceinline__ void dmma8x8x4(double (&c)[2], double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c[0]), "+d"(c[1])
      : "d"(a), "d"(b));
}

__device__ __forceinline__ void cp_async16(double* smem_dst, const double* gmem_src, int src_bytes) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async8(double* smem_dst, const double* gmem_src, int src_bytes) {
  uint32_t s = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(s), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// fixed-order sum over a CTA of NT threads (red: NT / 32 doubles of shared memory); every thread gets the result
template <int NT>
__device__ __forceinline__ double block_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  for (int k = 0; k < NT / 32; k++) s += red[k];
  return s;
}

// Linear tile id -> (ti, tj).  lower != 0: only tiles that contain an element with col <= row (the region
// starts on the diagonal; rows may extend past the column count = trapezoid).  With BM = Q*BN row tile r owns
// min(ntn, Q*r + Q) column tiles.  ntn = number of column tiles.
template <int Q>
__device__ __forceinline__ void decode_tile(long long t, int ntn, int lower, int& ti, int& tj) {
  if (!lower) {
    ti = (int)(t / ntn);
    tj = (int)(t % ntn);
    return;
  }
  const long long r0 = ntn / Q;                   // rows 0..r0-1 are strictly triangular
  const long long tri = Q * r0 * (r0 + 1) / 2;
  if (t < tri) {
    long long r = (long long)((sqrt(8.0 * (double)t / (double)Q + 1.0) - 1.0) * 0.5);
    while (Q * r * (r + 1) / 2 > t) --r;
    while (Q * (r + 1) * (r + 2) / 2 <= t) ++r;
    ti = (int)r;
    tj = (int)(t - Q * r * (r + 1) / 2);
  } else {
    long long u = t - tri;
    ti = (int)(r0 + u / ntn);
    tj = (int)(u % ntn);
  }
}

template <typename Cfg>
static inline long long count_tiles(long long M, long long N, int lower) {
  const long long ntm = (M + Cfg::BM - 1) / Cfg::BM, ntn = (N + Cfg::BN - 1) / Cfg::BN;
  if (!lower) return ntm * ntn;
  const long long r0 = ntn / Cfg::Q;
  if (ntm <= r0) return Cfg::Q * ntm * (ntm + 1) / 2;
  return Cfg::Q * r0 * (r0 + 1) / 2 + (ntm - r0) * ntn;
}

}  // namespace smnngp

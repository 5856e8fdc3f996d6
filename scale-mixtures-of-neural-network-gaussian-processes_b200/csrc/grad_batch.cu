// Batched loss and gradient (N <= 4096): SPR.loss and its six-scalar gradient (what smnngp_lml_grad_f64 returns) at
// G hyper-parameter points in one persistent launch - multi-start training and gradient refinement of a grid search
// at the sizes the reference trains on (experiments/regression/train.py:178), where one smnngp_lml_grad_f64 call
// leaves the GPU nearly idle.  Every CTA owns a private slot of the workspace and evaluates whole points, one after
// the other, with a static stride.  A point never leaves its CTA and every reduction has a fixed order, so its outputs
// are the same bits alone, inside any batch, in any order and with any slot count.
//
// Per point, A = K + eps I (the absolute regulariser of SPR.loss):
//   1. the value / dual layer tables of every row for this point's scalars (fill_row_dual_tables);
//   2. trapezoid in the slot: rows 0..N-1 = A (lower part) from the cached base, row N = y^T, rows N+1..2N = I;
//   3. factor_slot<true>: row N comes out as z = L^-1 y, rows N+1..2N as U = L^-T (identity-prefix skip);
//   4. alpha = U z (in-CTA GEMV), quad = ||z||^2, A^-1 = U U^T over rows 0..N-1 (in-CTA DMMA SYRK);
//   5. one pass over the lower triangle of the base: (k, dk/dw, dk/db) by the dual recursion, contracted with
//      G = 1/2 (gamma alpha alpha^T - A^-1) into the four sums of grad_epilogue (grad.cu), fixed-order block sums;
//   6. the closed forms of lml_finalize / grad_finalize (closed_forms.cuh); all-NaN outputs when a pivot failed.
#include "closed_forms.cuh"
#include "context.cuh"
#include "slot_chol.cuh"

namespace smnngp {

namespace {

// rows N+1 .. 2N of the slot = I, whole rows (the SYRK reads the padding columns of U as zeros)
__device__ void set_identity_rows(double* __restrict__ U, long long lda, int N) {
  const long long n = (long long)N * lda;
  for (long long i = threadIdx.x; i < n; i += GB_THREADS) U[i] = (i / lda == i % lda) ? 1.0 : 0.0;
}

// alpha_i = sum_{k >= i} U[i][k] z[k], one warp per row
__device__ void upper_gemv_slot(const double* __restrict__ U, long long ldu, const double* __restrict__ z, int N,
                                double* __restrict__ alpha) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = warp; i < N; i += GB_WARPS) {
    const double* u = U + (long long)i * ldu;
    double s = 0.0;
    for (int k = i + lane; k < N; k += 32) s = fma(u[k], z[k], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) alpha[i] = s;
  }
}

template <int ACT>
__global__ void __launch_bounds__(GB_THREADS, 2) lml_grad_batch_kernel(const GradBatchParams p) {
  extern __shared__ __align__(16) double smem[];
  double* red = smem + GB_SMEM_DOUBLES - GB_WARPS;
  int* bad_s = reinterpret_cast<int*>(smem + GB_SMEM_DOUBLES);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  char* slot = p.ws + (long long)blockIdx.x * p.slot_bytes;
  double* A = reinterpret_cast<double*>(slot);
  double* tab3 = reinterpret_cast<double*>(slot) + p.off_tab3;
  double* alpha = reinterpret_cast<double*>(slot) + p.off_alpha;
  const int N = p.N;
  const long long lda = p.lda;
  double* z = A + (long long)N * lda;
  double* U = A + (long long)(N + 1) * lda;
  const bool resnet = p.arch == ARCH_RESNET;
  const int n_act = n_act_applications(p.n_hidden, p.arch);
  const long long plane = (long long)(n_act > 0 ? n_act : 1) * N;
  const double* t0 = tab3;
  const double* t1 = tab3 + plane;
  const double* t2 = tab3 + 2 * plane;

  for (int g = blockIdx.x; g < p.G; g += gridDim.x) {
    const double* hp = p.hp + (long long)g * HP_COUNT;
    // 1. tables
    for (int r = tid; r < N; r += GB_THREADS)
      fill_row_dual_tables(p.q_d[r], 1, r, p.n_hidden, ACT, p.arch, hp, tab3, N, n_act);
    __syncthreads();

    // 2. + 3. A + eps I | y^T | I, factorised
    build_gram<ACT>(p, hp, t0, A, hp[HP_EPS]);
    copy_row(p.y, z, N);
    set_identity_rows(U, lda, N);
    __syncthreads();
    double lsum = 0.0;
    factor_slot<true>(A, lda, 2 * N + 1, N, smem, bad_s, lsum);
    __syncthreads();
    const int bad = *bad_s;
    const double logdet = block_sum<GB_THREADS>(lsum, red);
    double zz = 0.0;
    for (int n = tid; n < N; n += GB_THREADS) zz = fma(z[n], z[n], zz);
    const double quad = block_sum<GB_THREADS>(zz, red);

    // 4. alpha = U z and A^-1 = U U^T over the rows of L (no longer needed)
    upper_gemv_slot(U, lda, z, N, alpha);
    syrk_upper_slot(U, lda, N, A, lda, smem);
    __syncthreads();

    // 5. sum over the lower triangle of G_rc dK_rc / d{w_std, b_std, last_w_std} and tr G (grad_epilogue, grad.cu)
    const double w = hp[HP_W], b = hp[HP_B], v = hp[HP_V];
    const double w2 = w * w, b2 = b * b, v2 = v * v;
    double gamma = 1.0;
    if (p.kind == KIND_STUDENT_T) {
      const double a = hp[HP_ALPHA], be = hp[HP_BETA];
      gamma = (2.0 * a + (double)N) / ((2.0 * a + quad * a / be) * (be / a));
    }
    double sums[4] = {0.0, 0.0, 0.0, 0.0};
    for (int r = warp; r < N; r += GB_WARPS) {
      const double* src = p.K0dd + (long long)r * p.ld0;
      const double* wrow = A + (long long)r * lda;
      const double al_r = alpha[r];
      for (int c = lane; c <= r; c += 32) {
        const double k0 = src[c];
        double k = resnet ? fma(w2, k0, b2) : k0;      // dense-resnet: leading Dense(512)
        double dw = resnet ? 2.0 * w * k0 : 0.0;
        double db = resnet ? 2.0 * b : 0.0;
        for (int a = 0; a < n_act; a++) {
          const long long ir = a * (long long)N + r, ic = a * (long long)N + c;
          layer_step_dual<ACT>(k, dw, db, t0[ir], t0[ic], t1[ir] + t1[ic], t2[ir] + t2[ic], w, b, w2, b2, resnet,
                               !resnet || a == n_act - 1);
        }
        double gv = 0.5 * fma(gamma * al_r, alpha[c], -wrow[c]);
        if (c == r) sums[3] += gv;
        else gv += gv;                                 // the mirrored entry
        sums[0] = fma(gv, v2 * dw, sums[0]);
        sums[1] = fma(gv, v2 * db, sums[1]);
        sums[2] = fma(gv, k, sums[2]);                 // d K / d last_w_std = 2 v k
      }
    }
    const double s_w = block_sum<GB_THREADS>(sums[0], red);
    const double s_b = block_sum<GB_THREADS>(sums[1], red);
    const double s_v = block_sum<GB_THREADS>(sums[2] * (2.0 * v), red);
    const double s_e = block_sum<GB_THREADS>(sums[3], red);

    // 6. closed forms
    if (tid == 0) {
      double* out = p.out + 4ll * g;
      double* grad = p.grad + 6ll * g;
      lml_closed_form(logdet, quad, hp, p.kind, N, &bad, out);
      grad_closed_form(s_w, s_b, s_v, s_e, hp, &quad, p.kind, N, &bad, grad);
      if (bad) out[0] = out[1] = out[2] = out[3] = qnan_d();
      p.info[g] = bad;
    }
    __syncthreads();                                   // the slot and bad_s are reused by the next point
  }
}

}  // namespace

cudaError_t launch_lml_grad_batch(cudaStream_t s, const GradBatchParams& p, int act, long long slots) {
  auto kern = act == ACT_RELU ? lml_grad_batch_kernel<ACT_RELU> : lml_grad_batch_kernel<ACT_ERF>;
  cudaError_t e = configure_kernel_once(reinterpret_cast<const void*>(kern), GB_SMEM_BYTES, false);
  if (e != cudaSuccess) return e;
  kern<<<(unsigned)(slots < p.G ? slots : p.G), GB_THREADS, GB_SMEM_BYTES, s>>>(p);
  instr().launches++;
  return cudaGetLastError();
}

}  // namespace smnngp

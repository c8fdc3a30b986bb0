// Covariance builders (kernel #1): K(X,X) (+ noise/jitter on the diagonal) and K(X*,X) tiles,
// ARD squared-exponential and Matern-5/2.
//
// Replaces the kernel evaluation inside gpTorch7's gp_regressor (external; called through
// model:predict at reference scores/expected_improvement.lua:63).  The only in-tree witness of
// that arithmetic is utils.math.pdist (utils/math.lua:65-111), which forms distances in the
// cancellation-prone expanded form |x|^2+|z|^2-2xz through a GEMM and clamps at 0.  Here the
// distance is accumulated directly, r2 = sum_d ((a_d - b_d) w_d)^2 (oracle/SPEC.md), in registers:
// the pass writes 8 B per matrix entry and reads nothing but the (cache-resident) inputs.
//
// Layout: out is rows_pad x Np row-major (k contiguous).  One thread owns one column k (one
// observation) and keeps its d coordinates in registers; the block walks over a chunk of rows
// (candidates) whose coordinates sit in shared memory and are read as warp broadcasts; every
// store instruction writes 32 consecutive doubles.
#include "b7_internal.h"
#include "cov_entry.cuh"

namespace {

constexpr int kRowsPerBlock = 32;

template <int DT, int KERNEL>
__global__ void __launch_bounds__(256)
cov_kernel(const double* __restrict__ A, long long rows, long long rows_pad, int d, const double* __restrict__ Xt,
           int N, int Np, const double* __restrict__ par_base, long long par_stride, double* __restrict__ out_base,
           long long out_stride, int is_kxx, int tiled) {
  __shared__ double s_a[kRowsPerBlock][DT];
  __shared__ double s_w[DT];
  __shared__ double s_tab[64];
  if (threadIdx.x < 64) s_tab[threadIdx.x] = c_exp_tab[threadIdx.x];
  const double* par = par_base + (long long)blockIdx.z * par_stride;
  double* out = out_base + (long long)blockIdx.z * out_stride;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  const long long r0 = (long long)blockIdx.y * kRowsPerBlock;
  // K(X,X): only 128x128 blocks at or below the diagonal are ever read (lower Cholesky)
  if (is_kxx && (long long)(blockIdx.x * blockDim.x) > (r0 | 127)) return;
  for (int e = threadIdx.x; e < kRowsPerBlock * DT; e += blockDim.x) {
    int r = e / DT, i = e % DT;
    long long row = r0 + r;
    s_a[r][i] = (row < rows && i < d) ? A[row * d + i] : 0.0;
  }
  if (threadIdx.x < DT) s_w[threadIdx.x] = threadIdx.x < d ? par[threadIdx.x] : 0.0;
  __syncthreads();
  if (k >= Np) return;
  const double sf2 = par[B7_MAX_DIMS], diag_add = par[B7_MAX_DIMS + 1];
  double b[DT];
#pragma unroll
  for (int i = 0; i < DT; ++i) b[i] = (i < d && k < N) ? Xt[(long long)i * Np + k] : 0.0;
  const int r_end = (int)((rows_pad - r0) < kRowsPerBlock ? (rows_pad - r0) : kRowsPerBlock);
  for (int r = 0; r < r_end; ++r) {
    const long long row = r0 + r;
    double val;
    if (row >= rows || k >= N) {
      val = (is_kxx && row == k) ? 1.0 : 0.0;   // identity padding keeps the padded factor trivial
    } else {
      double r2 = 0.0;
#pragma unroll
      for (int i = 0; i < DT; ++i) {
        double t = (s_a[r][i] - b[i]) * s_w[i];
        r2 = fma(t, t, r2);
      }
      val = cov_value<KERNEL>(r2, sf2, s_tab);
      if (is_kxx && row == k) val += diag_add;
    }
    if (tiled) {
      // fragment order of gemm_tile.cuh: [row tile][k tile 16][k group 4][row 128][4]
      const long long off = ((row >> 7) * (long long)(Np >> 4) + (k >> 4)) * 2048 + ((k >> 2) & 3) * 512 + (row & 127) * 4 + (k & 3);
      out[off] = val;
    } else {
      out[row * Np + k] = val;
    }
  }
}

template <int DT>
int launch_dt(b7_ctx* ctx, int kernel, const double* A, long long rows, long long rows_pad, int d, const double* Xt,
              int N, int Np, const double* par, long long par_stride, double* out, long long out_stride, int batch,
              bool is_kxx, bool tiled) {
  dim3 grid((Np + 255) / 256, (unsigned)((rows_pad + kRowsPerBlock - 1) / kRowsPerBlock), batch);
  if (kernel == B7_KERNEL_ARDSE)
    cov_kernel<DT, B7_KERNEL_ARDSE><<<grid, 256, 0, ctx->stream>>>(A, rows, rows_pad, d, Xt, N, Np, par, par_stride, out,
                                                                 out_stride, is_kxx, tiled);
  else
    cov_kernel<DT, B7_KERNEL_MATERN52><<<grid, 256, 0, ctx->stream>>>(A, rows, rows_pad, d, Xt, N, Np, par, par_stride,
                                                                    out, out_stride, is_kxx, tiled);
  b7_count(ctx);
  B7_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

int b7_launch_cov_batched(b7_ctx* ctx, int kernel, const double* A, int64_t rows, int64_t rows_pad, int d,
                          const double* Xt, int N, int Np, const double* par, int64_t par_stride, double* out,
                          int64_t out_stride, int batch, bool is_kxx, bool tiled) {
  if (rows_pad <= 0) return 0;
  if (rows_pad / kRowsPerBlock + 1 > 65535) { b7_set_error("cov: too many rows per launch"); return B7_ERR_ARG; }
  if (d <= 2) return launch_dt<2>(ctx, kernel, A, rows, rows_pad, d, Xt, N, Np, par, par_stride, out, out_stride, batch, is_kxx, tiled);
  if (d <= 4) return launch_dt<4>(ctx, kernel, A, rows, rows_pad, d, Xt, N, Np, par, par_stride, out, out_stride, batch, is_kxx, tiled);
  if (d <= 6) return launch_dt<6>(ctx, kernel, A, rows, rows_pad, d, Xt, N, Np, par, par_stride, out, out_stride, batch, is_kxx, tiled);
  if (d <= 8) return launch_dt<8>(ctx, kernel, A, rows, rows_pad, d, Xt, N, Np, par, par_stride, out, out_stride, batch, is_kxx, tiled);
  if (d <= 16) return launch_dt<16>(ctx, kernel, A, rows, rows_pad, d, Xt, N, Np, par, par_stride, out, out_stride, batch, is_kxx, tiled);
  if (d <= 24) return launch_dt<24>(ctx, kernel, A, rows, rows_pad, d, Xt, N, Np, par, par_stride, out, out_stride, batch, is_kxx, tiled);
  return launch_dt<40>(ctx, kernel, A, rows, rows_pad, d, Xt, N, Np, par, par_stride, out, out_stride, batch, is_kxx, tiled);
}


// DNGO Bayesian-linear-regression head (kernel #5): feature Gram, D x D Cholesky, predictive
// mean / variance over the candidate features.
//
// Replaces gpTorch7's bayes_linear:predict as called from reference models/dngo.lua:174
// (Z0: N x D basis features of the observations, Z1: M x D of the candidates, models/dngo.lua:121-122).
// Declared arithmetic (oracle/SPEC.md; gpTorch7 itself is not available):
//   A = beta Z0^T Z0 + alpha_p I,  L = chol(A),  w = beta A^-1 Z0^T (y - m),
//   mean* = m + phi^T w,  var* = |L^-1 phi|^2 + 1/beta.
//
// fit:   gram_kernel accumulates per-block partial sums of Z0^T Z0, Z0^T y, Z0^T 1 in registers
//        (fixed row partition, partials added in block order => deterministic), blr_finish_kernel
//        factors and inverts the D x D system in shared memory, one CTA per (alpha_p, beta) draw.
// refit: the partials, Z0 and y stay on the device; new rows give the log evidence (blr_evidence_kernel +
//        blr_residual_kernel, the slice sampler's density) and, on request, a new predictor through blr_finish_kernel.
// score: one thread per candidate keeps its D features in registers (instantiated for D rounded up
//        to a multiple of 8, D <= 64), L^-1 sits in shared memory and is read as warp broadcasts;
//        the pass reads 8D bytes per candidate once (tile staged through shared memory so the
//        global reads are coalesced) and does D^2/2 FMAs: on B200 (5.8 flop per HBM byte) that is
//        balanced between the FP64 pipe and HBM for D = 50.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "b7_internal.h"

int b7_score_grid_size(b7_ctx* ctx, int64_t M);
// blr_dmma.cu: MLP basis + BLR head on DMMA tiles; returns 1 when the shapes do not fit (use the kernels below)
int b7_launch_dngo_tiles(b7_ctx* ctx, const double* in, int64_t M, int n_layers, const int* dims, const double* const* W_dev,
                         const double* const* b_dev, const int* act, const double* Linv, const double* w, const double* par, int D, int S,
                         int64_t ld_out, double* mean, double* var, double* feat_out);

namespace {

constexpr int kMaxD = 64;
constexpr int kGramBlocks = 296;

// partial[b] = [ G (D*D) | Z^T y (D) | Z^T 1 (D) ]
__global__ void __launch_bounds__(256)
gram_kernel(const double* __restrict__ Z, const double* __restrict__ y, int N, int D, double* __restrict__ partial) {
  extern __shared__ double sh[];   // [32][D+1] rows, then y[32]
  const int ldz = D + 1;
  double* ys = sh + 32 * ldz;
  const int rows_per = (N + gridDim.x - 1) / gridDim.x;
  const int r0 = blockIdx.x * rows_per, r1 = min(N, r0 + rows_per);
  const int n_out = D * D + 2 * D;
  double acc[18];   // ceil((64*64 + 128) / 256) = 17
#pragma unroll
  for (int t = 0; t < 18; ++t) acc[t] = 0.0;
  for (int rb = r0; rb < r1; rb += 32) {
    const int nr = min(32, r1 - rb);
    __syncthreads();
    for (int e = threadIdx.x; e < nr * D; e += blockDim.x) sh[(e / D) * ldz + e % D] = Z[(long long)(rb + e / D) * D + e % D];
    if (threadIdx.x < nr) ys[threadIdx.x] = y[rb + threadIdx.x];
    __syncthreads();
#pragma unroll
    for (int t = 0; t < 18; ++t) {
      const int o = threadIdx.x + t * 256;
      if (o >= n_out) break;
      double a = acc[t];
      if (o < D * D) {
        const int i = o / D, j = o % D;
        for (int r = 0; r < nr; ++r) a = fma(sh[r * ldz + i], sh[r * ldz + j], a);
      } else if (o < D * D + D) {
        const int i = o - D * D;
        for (int r = 0; r < nr; ++r) a = fma(sh[r * ldz + i], ys[r], a);
      } else {
        const int i = o - D * D - D;
        for (int r = 0; r < nr; ++r) a += sh[r * ldz + i];
      }
      acc[t] = a;
    }
  }
#pragma unroll
  for (int t = 0; t < 18; ++t) {
    const int o = threadIdx.x + t * 256;
    if (o < n_out) partial[(long long)blockIdx.x * n_out + o] = acc[t];
  }
}

// par[s] = alpha_p, beta, m, 1/beta.  Outputs Linv[s] (D x D lower, row-major), w[s] (D), info[s].
__global__ void __launch_bounds__(256)
blr_finish_kernel(const double* __restrict__ partial, int n_blocks, int D, const double* __restrict__ par,
                  double* __restrict__ Linv, double* __restrict__ w, int* __restrict__ info) {
  extern __shared__ double sh[];
  const int ld = D + 1, s = blockIdx.x, tid = threadIdx.x, n_out = D * D + 2 * D;
  double* A = sh;                 // D x ld : lower = L
  double* X = A + D * ld;         // D x ld : inverse
  double* b = X + D * ld;         // D
  double* t1 = b + D;             // D
  const double alpha_p = par[s * 4 + 0], beta = par[s * 4 + 1], m = par[s * 4 + 2];
  for (int o = tid; o < n_out; o += blockDim.x) {
    double a = 0.0;
    for (int p = 0; p < n_blocks; ++p) a += partial[(long long)p * n_out + o];   // block order: deterministic
    if (o < D * D) {
      const int i = o / D, j = o % D;
      A[i * ld + j] = beta * a + (i == j ? alpha_p : 0.0);
      X[i * ld + j] = (i == j) ? 1.0 : 0.0;
    } else if (o < D * D + D) b[o - D * D] = a;
    else t1[o - D * D - D] = a;
  }
  __syncthreads();
  if (tid < D) b[tid] = beta * (b[tid] - m * t1[tid]);   // beta Z^T (y - m)
  int my_info = 0;
  __syncthreads();
  for (int q = 0; q < D; ++q) {
    const double piv = A[q * ld + q];
    const double lq = sqrt(piv), inv = 1.0 / lq;
    if (tid == 0 && !(piv > 0.0) && my_info == 0) my_info = q + 1;
    __syncthreads();
    if (tid < D) {
      if (tid > q) A[tid * ld + q] *= inv;
      else X[q * ld + tid] *= inv;
      if (tid == q) A[q * ld + q] = lq;
    }
    __syncthreads();
    for (int e = tid; e < (D - 1 - q) * D; e += blockDim.x) {
      const int i = q + 1 + e / D, k = e % D;
      const double liq = A[i * ld + q];
      if (k > q && k <= i) A[i * ld + k] -= liq * A[k * ld + q];
      if (k <= q) X[i * ld + k] -= liq * X[q * ld + k];
    }
    __syncthreads();
  }
  // w = Linv^T (Linv b)
  if (tid < D) {
    double v = 0.0;
    for (int k = 0; k <= tid; ++k) v = fma(X[tid * ld + k], b[k], v);
    t1[tid] = v;
  }
  __syncthreads();
  if (tid < D) {
    double v = 0.0;
    for (int i = tid; i < D; ++i) v = fma(X[i * ld + tid], t1[i], v);
    w[(long long)s * D + tid] = v;
  }
  for (int e = tid; e < D * D; e += blockDim.x) {
    const int i = e / D, k = e % D;
    Linv[(long long)s * D * D + e] = (k <= i) ? X[i * ld + k] : 0.0;
  }
  if (tid == 0) info[s] = my_info;
}

// ---- log evidence of the BLR head for S rows (b7_blr_refit) --------------------------------------------------
//   log p(y | h) = D/2 log alpha_p + N/2 log beta - E - sum_i log (L_A)_ii - N/2 log 2 pi,
//   E = beta/2 |r - Z0 w|^2 + alpha_p/2 |w|^2,  r = y - m.
// E is evaluated as written, by a residual pass over the resident Z0 (blr_residual_kernel): E is the minimum over w of
// that quadratic, so an error in w enters E at second order only.  The shortcut E = (beta r^T r - |L_A^-1 beta Z0^T r|^2) / 2
// subtracts two numbers of size beta r^T r and loses their common digits (at beta = 1e4, N = 20 000 that is 1e-8 relative
// to the result when the features explain y well).  Every draw is computed by its own CTA / its own registers, so a draw's
// result does not depend on the other rows of the launch.

// gram[o] = sum_p partial[p][o], in block order: the sums blr_finish_kernel forms, so A below has the same bits
__global__ void blr_gram_reduce_kernel(const double* __restrict__ partial, int n_blocks, int n_out, double* __restrict__ gram) {
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= n_out) return;
  double a = 0.0;
  for (int p = 0; p < n_blocks; ++p) a += partial[(long long)p * n_out + o];
  gram[o] = a;
}

// One CTA per draw: A = beta G + alpha_p I, L_A = chol(A) in shared memory (no inverse), u = L_A^-1 beta Z0^T r by
// forward substitution, w = L_A^-T u by back substitution.  Writes w[s], stat[s] = (sum log (L_A)_ii, |w|^2), info[s]
// (first failing pivot; a non-finite pivot fails too).
__global__ void __launch_bounds__(256)
blr_evidence_kernel(const double* __restrict__ gram, int D, const double* __restrict__ par, double* __restrict__ w_out,
                    double* __restrict__ stat, int* __restrict__ info) {
  extern __shared__ double sh[];
  const int ld = D + 1, s = blockIdx.x, tid = threadIdx.x, n_out = D * D + 2 * D;
  double* A = sh;                 // D x ld : lower = L_A
  double* b = A + D * ld;         // D
  double* t1 = b + D;             // D
  const double alpha_p = par[s * 4 + 0], beta = par[s * 4 + 1], m = par[s * 4 + 2];
  for (int o = tid; o < n_out; o += blockDim.x) {
    const double a = gram[o];
    if (o < D * D) {
      const int i = o / D, j = o % D;
      A[i * ld + j] = beta * a + (i == j ? alpha_p : 0.0);
    } else if (o < D * D + D) b[o - D * D] = a;
    else t1[o - D * D - D] = a;
  }
  __syncthreads();
  if (tid < D) b[tid] = beta * (b[tid] - m * t1[tid]);   // beta Z^T (y - m)
  int my_info = 0;
  __syncthreads();
  for (int q = 0; q < D; ++q) {
    const double piv = A[q * ld + q];
    const double lq = sqrt(piv), inv = 1.0 / lq;
    if (tid == 0 && !(piv > 0.0 && piv < INFINITY) && my_info == 0) my_info = q + 1;
    __syncthreads();
    if (tid < D) {
      if (tid > q) A[tid * ld + q] *= inv;
      if (tid == q) A[q * ld + q] = lq;
    }
    __syncthreads();
    const int n = D - 1 - q;
    for (int e = tid; e < n * n; e += blockDim.x) {
      const int i = q + 1 + e / n, k = q + 1 + e % n;
      if (k <= i) A[i * ld + k] -= A[i * ld + q] * A[k * ld + q];
    }
    __syncthreads();
  }
  if (tid >= 32) return;
  // warp 0: lane l owns rows l and l + 32 of the right-hand side; each step broadcasts the solved entry
  const int lane = tid;
  double r0 = lane < D ? b[lane] : 0.0, r1 = lane + 32 < D ? b[lane + 32] : 0.0;
  for (int i = 0; i < D; ++i) {                                   // u = L_A^-1 b
    const double own = i < 32 ? r0 : r1;
    const double ui = __shfl_sync(0xffffffffu, own, i & 31) / A[i * ld + i];
    if (lane == (i & 31)) { if (i < 32) r0 = ui; else r1 = ui; }
    if (lane > i && lane < D) r0 -= A[lane * ld + i] * ui;
    if (lane + 32 > i && lane + 32 < D) r1 -= A[(lane + 32) * ld + i] * ui;
  }
  for (int i = D - 1; i >= 0; --i) {                              // w = L_A^-T u
    const double own = i < 32 ? r0 : r1;
    const double wi = __shfl_sync(0xffffffffu, own, i & 31) / A[i * ld + i];
    if (lane == (i & 31)) { if (i < 32) r0 = wi; else r1 = wi; }
    if (lane < i) r0 -= A[i * ld + lane] * wi;
    if (lane + 32 < i) r1 -= A[i * ld + lane + 32] * wi;
  }
  double ld_sum = (lane < D ? log(A[lane * ld + lane]) : 0.0) + (lane + 32 < D ? log(A[(lane + 32) * ld + lane + 32]) : 0.0);
  double ww = (lane < D ? r0 * r0 : 0.0) + (lane + 32 < D ? r1 * r1 : 0.0);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ld_sum += __shfl_xor_sync(0xffffffffu, ld_sum, o);
    ww += __shfl_xor_sync(0xffffffffu, ww, o);
  }
  if (lane < D) w_out[(long long)s * D + lane] = r0;
  if (lane + 32 < D) w_out[(long long)s * D + lane + 32] = r1;
  if (lane == 0) {
    stat[s * 2 + 0] = ld_sum;
    stat[s * 2 + 1] = ww;
    info[s] = my_info;
  }
}

// res[s][block] = sum over the block's rows of (y_i - m_s - z_i^T w_s)^2.  A fixed row partition (it depends on N only), one warp
// per row (lane l holds z_il and z_i,l+32), eight draws per pass over the rows, warp sums added in warp order.
constexpr int kResBlocks = 296;
constexpr int kResDraws = 8;

__global__ void __launch_bounds__(256)
blr_residual_kernel(const double* __restrict__ Z, const double* __restrict__ y, int N, int D, const double* __restrict__ w,
                    const double* __restrict__ par, int S, double* __restrict__ res) {
  __shared__ double wsum[8][kResDraws];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rows_per = (N + gridDim.x - 1) / gridDim.x;
  const int r0 = blockIdx.x * rows_per, r1 = min(N, r0 + rows_per);
  for (int s0 = 0; s0 < S; s0 += kResDraws) {
    double wa[kResDraws], wb[kResDraws], m[kResDraws], acc[kResDraws];
#pragma unroll
    for (int j = 0; j < kResDraws; ++j) {
      const bool on = s0 + j < S;
      wa[j] = on && lane < D ? w[(long long)(s0 + j) * D + lane] : 0.0;
      wb[j] = on && lane + 32 < D ? w[(long long)(s0 + j) * D + lane + 32] : 0.0;
      m[j] = on ? par[(s0 + j) * 4 + 2] : 0.0;
      acc[j] = 0.0;
    }
    for (int i = r0 + warp; i < r1; i += 8) {
      const double za = lane < D ? Z[(long long)i * D + lane] : 0.0;
      const double zb = lane + 32 < D ? Z[(long long)i * D + lane + 32] : 0.0;
      const double yi = y[i];
#pragma unroll
      for (int j = 0; j < kResDraws; ++j) {
        double d = fma(zb, wb[j], za * wa[j]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        const double r = (yi - m[j]) - d;
        acc[j] = fma(r, r, acc[j]);
      }
    }
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < kResDraws; ++j) wsum[warp][j] = acc[j];
    }
    __syncthreads();
    if (threadIdx.x < kResDraws && s0 + (int)threadIdx.x < S) {
      double a = 0.0;
      for (int k = 0; k < 8; ++k) a += wsum[k][threadIdx.x];
      res[(long long)(s0 + threadIdx.x) * gridDim.x + blockIdx.x] = a;
    }
    __syncthreads();
  }
}

// one thread per draw: the residual partials in block order, then log p(y | row s); -inf for a failed factor or a
// non-finite value
__global__ void blr_evidence_finish_kernel(const double* __restrict__ res, int n_blocks, const double* __restrict__ stat,
                                           const double* __restrict__ hyp, const double* __restrict__ par, const int* __restrict__ info,
                                           int N, int D, int S, double* __restrict__ logev) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  double e = 0.0;
  for (int p = 0; p < n_blocks; ++p) e += res[(long long)s * n_blocks + p];
  const double alpha_p = par[s * 4 + 0], beta = par[s * 4 + 1];
  const double E = 0.5 * beta * e + 0.5 * alpha_p * stat[s * 2 + 1];
  const double lp = 0.5 * D * hyp[s * 3 + 0] + 0.5 * N * hyp[s * 3 + 1] - E - stat[s * 2 + 0] - 0.5 * N * 1.83787706640934548356;
  logev[s] = (info[s] == 0 && isfinite(lp)) ? lp : -INFINITY;
}

// moments of draws [0, S) for a tile of 128 candidates per block
template <int DP>
__global__ void __launch_bounds__(128)
blr_moments_kernel(const double* __restrict__ Z, long long M, int D, const double* __restrict__ Linv,
                   const double* __restrict__ w, const double* __restrict__ par, int S, long long ld_out,
                   double* __restrict__ mean, double* __restrict__ var) {
  extern __shared__ __align__(16) double sh[];
  // the staged candidate tile is only needed until the features sit in registers; L^-1 then reuses the space
  double* zt = sh;                    // 128 x (D | 1) staged tile
  double* Ls = sh;                    // DP x DP (transposed, zero padded)
  double* ws = Ls + DP * DP;          // DP
  const int ldz = D | 1;              // odd stride: conflict-free row reads
  const int tid = threadIdx.x;
  const long long c0 = (long long)blockIdx.x * 128;
  const int nc = (int)min((long long)128, M - c0);
  for (int e = tid; e < nc * D; e += 128) zt[(e / D) * ldz + e % D] = Z[c0 * D + e];
  __syncthreads();
  double phi[DP];
#pragma unroll
  for (int k = 0; k < DP; ++k) phi[k] = (k < D && tid < nc) ? zt[tid * ldz + k] : 0.0;
  for (int s = 0; s < S; ++s) {
    __syncthreads();
    for (int e = tid; e < DP * DP; e += 128) {
      const int k = e / DP, i = e % DP;          // stored transposed: Ls[k][i] = Linv[i][k]
      Ls[e] = (i < D && k < D) ? Linv[(long long)s * D * D + i * D + k] : 0.0;
    }
    if (tid < DP) ws[tid] = tid < D ? w[(long long)s * D + tid] : 0.0;
    __syncthreads();
    double s2 = 0.0, mu = 0.0;
#pragma unroll
    for (int k = 0; k < DP; ++k) mu = fma(ws[k], phi[k], mu);
    // four rows of v = Linv phi at a time: four independent FMA chains, and for a fixed k the four
    // matrix entries Linv[i..i+3][k] are 32 contiguous bytes of the transposed copy (two LDS.128 broadcasts)
#pragma unroll
    for (int i = 0; i < DP; i += 4) {
      double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;
#pragma unroll
      for (int k = 0; k < i + 4; ++k) {
        const double2 l01 = *reinterpret_cast<const double2*>(Ls + k * DP + i);
        const double2 l23 = *reinterpret_cast<const double2*>(Ls + k * DP + i + 2);
        const double p = phi[k];
        v0 = fma(l01.x, p, v0);   // entries above the diagonal are zero in the padded copy
        v1 = fma(l01.y, p, v1);
        v2 = fma(l23.x, p, v2);
        v3 = fma(l23.y, p, v3);
      }
      s2 = fma(v0, v0, s2);
      s2 = fma(v1, v1, s2);
      s2 = fma(v2, v2, s2);
      s2 = fma(v3, v3, s2);
    }
    if (tid < nc) {
      mean[(long long)s * ld_out + c0 + tid] = par[s * 4 + 2] + mu;
      var[(long long)s * ld_out + c0 + tid] = s2 + par[s * 4 + 3];
    }
  }
}

template <int DP>
int launch_moments_dp(b7_ctx* ctx, const double* Z, int64_t M, int D, const b7_blr* blr, int s0, int S, int64_t ld_out,
                      double* mean, double* var) {
  const size_t a = ((size_t)DP * DP + DP) * 8, b = 128 * (size_t)(D | 1) * 8;
  const size_t smem = a > b ? a : b;
  static bool done[16] = {false};   // function attributes are per device
  if (!done[ctx->device & 15]) {
    B7_CUDA(cudaFuncSetAttribute(blr_moments_kernel<DP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    done[ctx->device & 15] = true;
  }
  blr_moments_kernel<DP><<<(unsigned)((M + 127) / 128), 128, smem, ctx->stream>>>(
      Z, M, D, blr->Linv + (size_t)s0 * D * D, blr->w + (size_t)s0 * D, blr->par + (size_t)s0 * 4, S, ld_out, mean, var);
  b7_count(ctx);
  B7_CUDA(cudaGetLastError());
  return 0;
}

int launch_moments(b7_ctx* ctx, const double* Z, int64_t M, const b7_blr* blr, int s0, int S, int64_t ld_out, double* mean,
                   double* var) {
  if (M <= 0) return 0;
  const int D = blr->D, dp = (D + 7) / 8 * 8;
  static const bool tiles = !(getenv("B7_BLR_DMMA") && getenv("B7_BLR_DMMA")[0] == '0');
  if (tiles) {
    // DMMA tiles (blr_dmma.cu); the draws are staged in shared memory in chunks (4, 2 or 1 draws, whatever fits)
    int rc = 0, chunk = 4;
    for (int c0 = 0; c0 < S && rc == 0;) {
      const int sc = std::min(chunk, S - c0);
      rc = b7_launch_dngo_tiles(ctx, Z, M, 0, &D, nullptr, nullptr, 0, blr->Linv + (size_t)(s0 + c0) * D * D, blr->w + (size_t)(s0 + c0) * D,
                                blr->par + (size_t)(s0 + c0) * 4, D, sc, ld_out, mean + (size_t)c0 * ld_out, var + (size_t)c0 * ld_out, nullptr);
      if (rc == 1 && chunk > 1 && c0 == 0) { chunk /= 2; rc = 0; continue; }
      c0 += sc;
    }
    if (rc <= 0) return rc;
  }
  switch (dp) {
    case 8: return launch_moments_dp<8>(ctx, Z, M, D, blr, s0, S, ld_out, mean, var);
    case 16: return launch_moments_dp<16>(ctx, Z, M, D, blr, s0, S, ld_out, mean, var);
    case 24: return launch_moments_dp<24>(ctx, Z, M, D, blr, s0, S, ld_out, mean, var);
    case 32: return launch_moments_dp<32>(ctx, Z, M, D, blr, s0, S, ld_out, mean, var);
    case 40: return launch_moments_dp<40>(ctx, Z, M, D, blr, s0, S, ld_out, mean, var);
    case 48: return launch_moments_dp<48>(ctx, Z, M, D, blr, s0, S, ld_out, mean, var);
    case 56: return launch_moments_dp<56>(ctx, Z, M, D, blr, s0, S, ld_out, mean, var);
    default: return launch_moments_dp<64>(ctx, Z, M, D, blr, s0, S, ld_out, mean, var);
  }
}

// ---- DNGO basis: X -> features through the trained MLP (models/dngo.lua:155-171) ---------------------------
// One dense layer: out[c][j] = act(b[j] + sum_k W[j][k] in[c][k]).  One thread per candidate keeps its input row in
// registers (width rounded up to a multiple of 8, <= 64); the weights sit transposed in shared memory so that the
// four outputs computed together read 32 contiguous bytes per k (two LDS.128 warp broadcasts per 4 FMAs); input and
// output tiles are staged through shared memory so that global accesses are coalesced.
template <int HP, bool TANH>      // TANH: act may be B7_ACT_TANH (tanh kept out of the other instantiation, as in blr_dmma.cu)
__global__ void __launch_bounds__(128)
mlp_layer_kernel(const double* __restrict__ in, long long M, int h_in, int h_out, const double* __restrict__ W,
                 const double* __restrict__ bias, int act, double* __restrict__ out) {
  extern __shared__ __align__(16) double sh[];
  const int ho4 = (h_out + 3) & ~3;
  double* Wt = sh;                          // [HP][ho4]  (Wt[k][j] = W[j][k], zero padded)
  double* bs = Wt + HP * ho4;               // [ho4]
  double* tile = bs + ho4;                  // 128 x max(h_in | 1, h_out | 1)
  const int ldi = h_in | 1, ldo = h_out | 1, tid = threadIdx.x;
  const long long c0 = (long long)blockIdx.x * 128;
  const int nc = (int)min((long long)128, M - c0);
  for (int e = tid; e < HP * ho4; e += 128) {
    const int k = e / ho4, j = e % ho4;
    Wt[e] = (k < h_in && j < h_out) ? W[(long long)j * h_in + k] : 0.0;
  }
  for (int e = tid; e < ho4; e += 128) bs[e] = e < h_out ? bias[e] : 0.0;
  for (int e = tid; e < nc * h_in; e += 128) tile[(e / h_in) * ldi + e % h_in] = in[c0 * h_in + e];
  __syncthreads();
  double x[HP];
#pragma unroll
  for (int k = 0; k < HP; ++k) x[k] = (k < h_in && tid < nc) ? tile[tid * ldi + k] : 0.0;
  __syncthreads();   // the tile is reused for the outputs
  for (int j = 0; j < ho4; j += 4) {
    double a0 = bs[j], a1 = bs[j + 1], a2 = bs[j + 2], a3 = bs[j + 3];
#pragma unroll
    for (int k = 0; k < HP; ++k) {
      const double2 w01 = *reinterpret_cast<const double2*>(Wt + k * ho4 + j);
      const double2 w23 = *reinterpret_cast<const double2*>(Wt + k * ho4 + j + 2);
      a0 = fma(w01.x, x[k], a0);
      a1 = fma(w01.y, x[k], a1);
      a2 = fma(w23.x, x[k], a2);
      a3 = fma(w23.y, x[k], a3);
    }
    if (act == B7_ACT_RELU) { a0 = a0 > 0.0 ? a0 : 0.0; a1 = a1 > 0.0 ? a1 : 0.0; a2 = a2 > 0.0 ? a2 : 0.0; a3 = a3 > 0.0 ? a3 : 0.0; }
    else if (TANH && act == B7_ACT_TANH) { a0 = tanh(a0); a1 = tanh(a1); a2 = tanh(a2); a3 = tanh(a3); }
    if (j < h_out) tile[tid * ldo + j] = a0;
    if (j + 1 < h_out) tile[tid * ldo + j + 1] = a1;
    if (j + 2 < h_out) tile[tid * ldo + j + 2] = a2;
    if (j + 3 < h_out) tile[tid * ldo + j + 3] = a3;
  }
  __syncthreads();
  for (int e = tid; e < nc * h_out; e += 128) out[c0 * h_out + e] = tile[(e / h_out) * ldo + e % h_out];
}

template <int HP>
int launch_mlp_layer(b7_ctx* ctx, const double* in, int64_t M, int h_in, int h_out, const double* W, const double* b, int act,
                     double* out) {
  const int ho4 = (h_out + 3) & ~3, wmax = (h_in | 1) > (h_out | 1) ? (h_in | 1) : (h_out | 1);
  const size_t smem = ((size_t)HP * ho4 + ho4 + 128 * (size_t)wmax) * 8;
  static bool done[16] = {false};
  if (!done[ctx->device & 15]) {
    B7_CUDA(cudaFuncSetAttribute(mlp_layer_kernel<HP, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B7_CUDA(cudaFuncSetAttribute(mlp_layer_kernel<HP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    done[ctx->device & 15] = true;
  }
  const unsigned blocks = (unsigned)((M + 127) / 128);
  if (act == B7_ACT_TANH) mlp_layer_kernel<HP, true><<<blocks, 128, smem, ctx->stream>>>(in, M, h_in, h_out, W, b, act, out);
  else mlp_layer_kernel<HP, false><<<blocks, 128, smem, ctx->stream>>>(in, M, h_in, h_out, W, b, act, out);
  b7_count(ctx);
  B7_CUDA(cudaGetLastError());
  return 0;
}

template <typename T>
int dalloc(b7_ctx* ctx, T** p, size_t n) {
  void* q = nullptr;
  int rc = b7_pool_alloc(ctx, &q, std::max<size_t>(n, 1) * sizeof(T));
  *p = static_cast<T*>(q);
  return rc;
}

struct Part {
  b7_ctx* ctx;
  double* best = nullptr; int64_t* idx = nullptr; int64_t* nan = nullptr;
  explicit Part(b7_ctx* c) : ctx(c) {}
  ~Part() { b7_pool_free(ctx, best); b7_pool_free(ctx, idx); b7_pool_free(ctx, nan); }
};

// device copies of the layer weights for one call (freed when the call returns)
struct DevWeights {
  b7_ctx* ctx;
  std::vector<const double*> W, b;
  std::vector<double*> owned;
  explicit DevWeights(b7_ctx* c) : ctx(c) {}
  ~DevWeights() { for (double* p : owned) b7_pool_free(ctx, p); }
  int upload(int n_layers, const int* dims, const double* const* Wh, const double* const* bh) {
    for (int l = 0; l < n_layers; ++l) {
      double *dW = nullptr, *db = nullptr;
      B7_CHECK(dalloc(ctx, &dW, (size_t)dims[l] * dims[l + 1]));
      owned.push_back(dW);
      B7_CHECK(dalloc(ctx, &db, (size_t)dims[l + 1]));
      owned.push_back(db);
      B7_CUDA(cudaMemcpyAsync(dW, Wh[l], (size_t)dims[l] * dims[l + 1] * 8, cudaMemcpyHostToDevice, ctx->stream));
      B7_CUDA(cudaMemcpyAsync(db, bh[l], (size_t)dims[l + 1] * 8, cudaMemcpyHostToDevice, ctx->stream));
      W.push_back(dW);
      b.push_back(db);
    }
    B7_CUDA(cudaStreamSynchronize(ctx->stream));     // the host arrays are borrowed for the duration of the call only
    return 0;
  }
};

bool mlp_tiles_enabled() {
  static const bool on = !(getenv("B7_BLR_DMMA") && getenv("B7_BLR_DMMA")[0] == '0');
  return on;
}

}  // namespace

int b7_check_act(const char* what, int n_layers, const int* act) {
  if (!act) { b7_set_error("%s: null activation codes", what); return B7_ERR_ARG; }
  for (int l = 0; l < n_layers; ++l)
    if (act[l] != B7_ACT_NONE && act[l] != B7_ACT_RELU && act[l] != B7_ACT_TANH) {
      b7_set_error("%s: unknown activation code %d after layer %d (B7_ACT_NONE, B7_ACT_RELU or B7_ACT_TANH)", what, act[l], l);
      return B7_ERR_ARG;
    }
  return 0;
}

extern "C" {

int b7_mlp_features(b7_ctx* ctx, b7_grid* in, int n_layers, const int* dims, const double* const* W, const double* const* b,
                    int relu_last, b7_grid** out) {
  return b7_mlp_features_act(ctx, in, n_layers, dims, W, b, b7_relu_codes(n_layers, relu_last).data(), out);
}

int b7_mlp_features_act(b7_ctx* ctx, b7_grid* in, int n_layers, const int* dims, const double* const* W, const double* const* b,
                        const int* act, b7_grid** out) {
  if (!ctx || !in || !out || n_layers < 1 || !dims || !W || !b || dims[0] != in->d) {
    b7_set_error("mlp_features: bad arguments (dims[0] must equal the grid's dims)");
    return B7_ERR_ARG;
  }
  *out = nullptr;
  if (in->ctx != ctx) { b7_set_error("mlp_features: the grid lives on another context / device"); return B7_ERR_ARG; }
  for (int l = 0; l <= n_layers; ++l)
    if (dims[l] < 1 || dims[l] > 64) { b7_set_error("mlp_features: layer widths must be in [1, 64] (got %d)", dims[l]); return B7_ERR_ARG; }
  B7_CHECK(b7_check_act("mlp_features", n_layers, act));
  B7_CUDA(cudaSetDevice(ctx->device));
  const int64_t M = in->rows;
  double* feat = nullptr;
  {
    // all layers in one pass over the grid on DMMA tiles (blr_dmma.cu): the intermediate activations stay in shared memory
    DevWeights dw(ctx);
    B7_CHECK(dw.upload(n_layers, dims, W, b));
    B7_CHECK(dalloc(ctx, &feat, (size_t)std::max<int64_t>(M, 1) * dims[n_layers]));
    StageTimer t(ctx, ST_BLR);
    int rc_t = mlp_tiles_enabled() ? b7_launch_dngo_tiles(ctx, in->X, M, n_layers, dims, dw.W.data(), dw.b.data(), act, nullptr, nullptr, nullptr,
                                                          0, 0, 0, nullptr, nullptr, feat)
                                   : 1;
    t.stop(1);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (rc_t == 0 && e != cudaSuccess) { b7_set_error("mlp_features: %s", cudaGetErrorString(e)); rc_t = B7_ERR_CUDA; }
    if (rc_t < 0) { b7_pool_free(ctx, feat); return rc_t; }
    if (rc_t == 0) {
      b7_grid* g = new b7_grid();
      g->ctx = ctx; g->rows = M; g->d = dims[n_layers]; g->X = feat;
      g->removed = in->removed;            // the feature grid inherits the candidate bookkeeping
      g->removed_dirty = !g->removed.empty();
      *out = g;
      return 0;
    }
    b7_pool_free(ctx, feat);
  }
  const double* cur = in->X;
  double* bufs[2] = {nullptr, nullptr};
  int rc = 0;
  StageTimer t(ctx, ST_BLR);
  for (int l = 0; l < n_layers && rc == 0; ++l) {
    const int hi = dims[l], ho = dims[l + 1];
    double *dW = nullptr, *db = nullptr, *dst = nullptr;
    if ((rc = dalloc(ctx, &dW, (size_t)hi * ho)) || (rc = dalloc(ctx, &db, (size_t)ho)) || (rc = dalloc(ctx, &dst, (size_t)std::max<int64_t>(M, 1) * ho))) break;
    cudaMemcpyAsync(dW, W[l], (size_t)hi * ho * 8, cudaMemcpyHostToDevice, ctx->stream);
    cudaMemcpyAsync(db, b[l], (size_t)ho * 8, cudaMemcpyHostToDevice, ctx->stream);
    if (M > 0) {
      switch ((hi + 7) / 8) {
        case 1: rc = launch_mlp_layer<8>(ctx, cur, M, hi, ho, dW, db, act[l], dst); break;
        case 2: rc = launch_mlp_layer<16>(ctx, cur, M, hi, ho, dW, db, act[l], dst); break;
        case 3: rc = launch_mlp_layer<24>(ctx, cur, M, hi, ho, dW, db, act[l], dst); break;
        case 4: rc = launch_mlp_layer<32>(ctx, cur, M, hi, ho, dW, db, act[l], dst); break;
        case 5: rc = launch_mlp_layer<40>(ctx, cur, M, hi, ho, dW, db, act[l], dst); break;
        case 6: rc = launch_mlp_layer<48>(ctx, cur, M, hi, ho, dW, db, act[l], dst); break;
        case 7: rc = launch_mlp_layer<56>(ctx, cur, M, hi, ho, dW, db, act[l], dst); break;
        default: rc = launch_mlp_layer<64>(ctx, cur, M, hi, ho, dW, db, act[l], dst); break;
      }
    }
    cudaStreamSynchronize(ctx->stream);
    b7_pool_free(ctx, dW); b7_pool_free(ctx, db);
    if (bufs[l & 1]) b7_pool_free(ctx, bufs[l & 1]);
    bufs[l & 1] = dst;
    cur = dst;
  }
  t.stop(n_layers);
  const int last = (n_layers - 1) & 1;
  if (bufs[last ^ 1]) b7_pool_free(ctx, bufs[last ^ 1]);
  if (rc < 0) { if (bufs[last]) b7_pool_free(ctx, bufs[last]); return rc; }
  b7_grid* g = new b7_grid();
  g->ctx = ctx; g->rows = M; g->d = dims[n_layers]; g->X = bufs[last];
  g->removed = in->removed;            // the feature grid inherits the candidate bookkeeping
  g->removed_dirty = !g->removed.empty();
  *out = g;
  return 0;
}

void b7_blr_free(b7_blr* blr) {
  if (!blr) return;
  cudaSetDevice(blr->ctx->device);
  cudaStreamSynchronize(blr->ctx->stream);
  b7_pool_free(blr->ctx, blr->Linv);
  b7_pool_free(blr->ctx, blr->w);
  b7_pool_free(blr->ctx, blr->par);
  for (double* p : {blr->Z, blr->y, blr->partial, blr->gram, blr->hyp, blr->ev_w, blr->ev_stat, blr->ev_res, blr->ev_out})
    b7_pool_free(blr->ctx, p);
  b7_pool_free(blr->ctx, blr->ev_info);
  delete blr;
}

int b7_blr_fit(b7_ctx* ctx, const double* Z0, const double* y, int N, int D, const double* hyp, int S, b7_blr** out,
               int* info) {
  if (!ctx || !out || !Z0 || !y || !hyp || N < 1 || D < 1 || D > kMaxD || S < 1) {
    b7_set_error("blr_fit: bad arguments (N=%d D=%d S=%d; D <= %d)", N, D, S, kMaxD);
    return B7_ERR_ARG;
  }
  *out = nullptr;
  B7_CUDA(cudaSetDevice(ctx->device));
  b7_blr* blr = new b7_blr();
  blr->ctx = ctx; blr->N = N; blr->D = D; blr->S = S;
  double *dZ = nullptr, *dy = nullptr, *partial = nullptr;
  int* dinfo = nullptr;
  const int n_out = D * D + 2 * D;
  const int blocks = std::min(kGramBlocks, (N + 31) / 32);
  int rc = 0;
  if ((rc = dalloc(ctx, &dZ, (size_t)N * D)) || (rc = dalloc(ctx, &dy, (size_t)N)) || (rc = dalloc(ctx, &partial, (size_t)blocks * n_out)) ||
      (rc = dalloc(ctx, &dinfo, (size_t)S)) || (rc = dalloc(ctx, &blr->Linv, (size_t)S * D * D)) || (rc = dalloc(ctx, &blr->w, (size_t)S * D)) ||
      (rc = dalloc(ctx, &blr->par, (size_t)S * 4))) {
    b7_blr_free(blr); b7_pool_free(ctx, dZ); b7_pool_free(ctx, dy); b7_pool_free(ctx, partial); b7_pool_free(ctx, dinfo);
    return rc;
  }
  blr->par_host.resize((size_t)S * 4);
  for (int s = 0; s < S; ++s) {
    const double ap = exp(hyp[s * 3 + 0]), be = exp(hyp[s * 3 + 1]);
    blr->par_host[s * 4 + 0] = ap; blr->par_host[s * 4 + 1] = be; blr->par_host[s * 4 + 2] = hyp[s * 3 + 2];
    blr->par_host[s * 4 + 3] = 1.0 / be;
  }
  cudaStream_t st = ctx->stream;
  cudaMemcpyAsync(dZ, Z0, (size_t)N * D * 8, cudaMemcpyHostToDevice, st);
  cudaMemcpyAsync(dy, y, (size_t)N * 8, cudaMemcpyHostToDevice, st);
  cudaMemcpyAsync(blr->par, blr->par_host.data(), (size_t)S * 4 * 8, cudaMemcpyHostToDevice, st);
  static bool attr_done_dev[16] = {false};
  bool& attr_done = attr_done_dev[ctx->device & 15];
  if (!attr_done) {
    cudaFuncSetAttribute(blr_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (2 * kMaxD * (kMaxD + 1) + 2 * kMaxD) * 8);
    attr_done = true;
  }
  StageTimer t(ctx, ST_BLR);
  gram_kernel<<<blocks, 256, (32 * (D + 1) + 32) * 8, st>>>(dZ, dy, N, D, partial);
  blr_finish_kernel<<<S, 256, (2 * D * (D + 1) + 2 * D) * 8, st>>>(partial, blocks, D, blr->par, blr->Linv, blr->w, dinfo);
  b7_count(ctx, 2);
  t.stop(2);
  std::vector<int> hi((size_t)S);
  cudaMemcpyAsync(hi.data(), dinfo, S * sizeof(int), cudaMemcpyDeviceToHost, st);
  cudaError_t e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = cudaGetLastError();
  b7_pool_free(ctx, dinfo);
  // observations and Gram partials stay on the device for b7_blr_refit
  blr->Z = dZ; blr->y = dy; blr->partial = partial; blr->gram_blocks = blocks;
  if (e != cudaSuccess) { b7_set_error("blr_fit: %s", cudaGetErrorString(e)); b7_blr_free(blr); return B7_ERR_CUDA; }
  int worst = 0;
  for (int s = 0; s < S; ++s) { if (info) info[s] = hi[s]; if (hi[s] && !worst) worst = hi[s]; }
  *out = blr;
  return worst;   // LAPACK-style: >0 = first failing pivot of the first failing draw
}

int b7_blr_refit(b7_blr* blr, const double* hyp, int flags, int* info, double* logev) {
  if (!blr || !hyp || (flags != B7_FIT_PREDICT && flags != B7_FIT_LOGML_ONLY)) {
    b7_set_error("blr_refit: bad arguments (flags must be B7_FIT_PREDICT or B7_FIT_LOGML_ONLY)");
    return B7_ERR_ARG;
  }
  b7_ctx* ctx = blr->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  const int N = blr->N, D = blr->D, S = blr->S, n_out = D * D + 2 * D;
  const int res_blocks = std::min(kResBlocks, (N + 63) / 64);
  cudaStream_t st = ctx->stream;
  if (!blr->gram) {
    B7_CHECK(dalloc(ctx, &blr->gram, (size_t)n_out));
    B7_CHECK(dalloc(ctx, &blr->hyp, (size_t)S * 3));
    B7_CHECK(dalloc(ctx, &blr->ev_w, (size_t)S * D));
    B7_CHECK(dalloc(ctx, &blr->ev_stat, (size_t)S * 2));
    B7_CHECK(dalloc(ctx, &blr->ev_res, (size_t)S * res_blocks));
    B7_CHECK(dalloc(ctx, &blr->ev_out, (size_t)S));
    B7_CHECK(dalloc(ctx, &blr->ev_info, (size_t)2 * S));
    blr_gram_reduce_kernel<<<(n_out + 255) / 256, 256, 0, st>>>(blr->partial, blr->gram_blocks, n_out, blr->gram);
    b7_count(ctx);
  }
  for (int s = 0; s < S; ++s) {                       // same conversion as b7_blr_fit
    const double ap = exp(hyp[s * 3 + 0]), be = exp(hyp[s * 3 + 1]);
    blr->par_host[s * 4 + 0] = ap; blr->par_host[s * 4 + 1] = be; blr->par_host[s * 4 + 2] = hyp[s * 3 + 2];
    blr->par_host[s * 4 + 3] = 1.0 / be;
  }
  cudaMemcpyAsync(blr->par, blr->par_host.data(), (size_t)S * 4 * 8, cudaMemcpyHostToDevice, st);
  cudaMemcpyAsync(blr->hyp, hyp, (size_t)S * 3 * 8, cudaMemcpyHostToDevice, st);
  const bool predict = flags == B7_FIT_PREDICT;
  StageTimer t(ctx, ST_BLR);
  blr_evidence_kernel<<<S, 256, ((size_t)D * (D + 1) + 2 * D) * 8, st>>>(blr->gram, D, blr->par, blr->ev_w, blr->ev_stat, blr->ev_info);
  blr_residual_kernel<<<res_blocks, 256, 0, st>>>(blr->Z, blr->y, N, D, blr->ev_w, blr->par, S, blr->ev_res);
  blr_evidence_finish_kernel<<<(S + 127) / 128, 128, 0, st>>>(blr->ev_res, res_blocks, blr->ev_stat, blr->hyp, blr->par, blr->ev_info, N, D, S,
                                                              blr->ev_out);
  // the predictor: the kept partials through blr_finish_kernel, exactly as b7_blr_fit reduces them
  if (predict)
    blr_finish_kernel<<<S, 256, (2 * D * (D + 1) + 2 * D) * 8, st>>>(blr->partial, blr->gram_blocks, D, blr->par, blr->Linv, blr->w,
                                                                      blr->ev_info + S);
  b7_count(ctx, predict ? 4 : 3);
  t.stop(predict ? 4 : 3);
  std::vector<int> hi((size_t)2 * S);
  std::vector<double> hl((size_t)S);
  cudaMemcpyAsync(hi.data(), blr->ev_info, (size_t)(predict ? 2 : 1) * S * sizeof(int), cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(hl.data(), blr->ev_out, (size_t)S * 8, cudaMemcpyDeviceToHost, st);
  cudaError_t e = cudaStreamSynchronize(st);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) { b7_set_error("blr_refit: %s", cudaGetErrorString(e)); blr->ready = false; return B7_ERR_CUDA; }
  blr->ready = predict;
  int worst = 0;
  for (int s = 0; s < S; ++s) {
    const int f = hi[s] ? hi[s] : (predict ? hi[S + s] : 0);
    if (info) info[s] = f;
    if (logev) logev[s] = f ? -INFINITY : hl[s];
    if (f && !worst) worst = f;
  }
  return worst;
}

int b7_blr_num_draws(b7_blr* blr) {
  if (!blr) { b7_set_error("blr_num_draws: null handle"); return B7_ERR_ARG; }
  return blr->S;
}

int b7_blr_predict(b7_blr* blr, int s, const double* Z1, int64_t M, double* mean, double* var) {
  if (!blr || s < 0 || s >= blr->S || M < 0 || (M > 0 && (!Z1 || !mean || !var))) { b7_set_error("blr_predict: bad arguments"); return B7_ERR_ARG; }
  if (!blr->ready) { b7_set_error("blr_predict: the last refit was B7_FIT_LOGML_ONLY; refit with B7_FIT_PREDICT first"); return B7_ERR_STATE; }
  b7_ctx* ctx = blr->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  const int64_t chunk = 1 << 20;
  double *dz = nullptr, *dm = nullptr;
  B7_CHECK(dalloc(ctx, &dz, (size_t)std::min(chunk, std::max<int64_t>(M, 1)) * blr->D));
  B7_CHECK(dalloc(ctx, &dm, (size_t)2 * std::min(chunk, std::max<int64_t>(M, 1))));
  int rc = 0;
  for (int64_t c0 = 0; c0 < M && rc == 0; c0 += chunk) {
    const int64_t n = std::min(chunk, M - c0);
    cudaMemcpyAsync(dz, Z1 + c0 * blr->D, (size_t)n * blr->D * 8, cudaMemcpyHostToDevice, ctx->stream);
    StageTimer t(ctx, ST_BLR);
    rc = launch_moments(ctx, dz, n, blr, s, 1, n, dm, dm + n);
    t.stop(1);
    cudaMemcpyAsync(mean + c0, dm, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(var + c0, dm + n, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (rc == 0 && e != cudaSuccess) { b7_set_error("blr_predict: %s", cudaGetErrorString(e)); rc = B7_ERR_CUDA; }
  }
  b7_pool_free(ctx, dz); b7_pool_free(ctx, dm);
  return rc;
}

// shared body of b7_blr_score (n_layers = 0: `features` already holds the basis) and b7_dngo_score (the basis is
// evaluated tile by tile in front of the head and never stored)
static int blr_score_impl(b7_blr* blr, b7_grid* features, int n_layers, const int* dims, const double* const* W, const double* const* b,
                          const int* act, int kind, double tradeoff, int bound, double sign, double fmin, double* score_host, int64_t* argmax,
                          int64_t* argmax_original, double* best, int64_t* nan_count) {
  if (!blr || !features || (kind != B7_SCORE_EI && kind != B7_SCORE_CB) || (n_layers == 0 && features->d != blr->D)) {
    b7_set_error("blr_score: bad arguments (feature dims %d vs D %d)", features ? features->d : -1, blr ? blr->D : -1);
    return B7_ERR_ARG;
  }
  if (features->ctx != blr->ctx) { b7_set_error("blr_score: the feature grid and the model live on different contexts / devices"); return B7_ERR_ARG; }
  if (!blr->ready) { b7_set_error("blr_score: the last refit was B7_FIT_LOGML_ONLY; refit with B7_FIT_PREDICT first"); return B7_ERR_STATE; }
  b7_ctx* ctx = blr->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  const int64_t M = features->rows;
  const int S = blr->S;
  double *mom = nullptr, *sc = nullptr;
  B7_CHECK(dalloc(ctx, &mom, (size_t)2 * S * std::max<int64_t>(M, 1)));
  B7_CHECK(dalloc(ctx, &sc, (size_t)std::max<int64_t>(M, 1)));
  Part pb(ctx);
  const int cap = b7_score_grid_size(ctx, M) + 1;
  B7_CHECK(dalloc(ctx, &pb.best, (size_t)cap)); B7_CHECK(dalloc(ctx, &pb.idx, (size_t)cap)); B7_CHECK(dalloc(ctx, &pb.nan, (size_t)cap));
  if (features->removed_dirty || features->removed.size()) {
    int64_t n = (int64_t)features->removed.size();
    if (n > features->removed_cap) {
      b7_pool_free(ctx, features->removed_dev);
      features->removed_cap = std::max<int64_t>(256, 2 * n);
      B7_CHECK(dalloc(ctx, &features->removed_dev, (size_t)features->removed_cap));
    }
    if (n) cudaMemcpyAsync(features->removed_dev, features->removed.data(), n * 8, cudaMemcpyHostToDevice, ctx->stream);
    features->removed_dirty = false;
  }
  int rc = 0, parts = 0;
  if (n_layers == 0) {
    StageTimer t(ctx, ST_BLR);
    rc = launch_moments(ctx, features->X, M, blr, 0, S, M, mom, mom + (size_t)S * M);
    t.stop(1);
  } else {
    DevWeights dw(ctx);
    if ((rc = dw.upload(n_layers, dims, W, b)) == 0) {
      StageTimer t(ctx, ST_BLR);
      const int D = blr->D;
      int chunk = 4;
      for (int c0 = 0; c0 < S && rc == 0;) {
        const int sc_ = std::min(chunk, S - c0);
        rc = b7_launch_dngo_tiles(ctx, features->X, M, n_layers, dims, dw.W.data(), dw.b.data(), act, blr->Linv + (size_t)c0 * D * D,
                                  blr->w + (size_t)c0 * D, blr->par + (size_t)c0 * 4, D, sc_, M, mom + (size_t)c0 * M,
                                  mom + (size_t)(S + c0) * M, nullptr);
        if (rc == 1 && chunk > 1 && c0 == 0) { chunk /= 2; rc = 0; continue; }
        c0 += sc_;
      }
      t.stop(1);
      cudaStreamSynchronize(ctx->stream);              // dw's buffers are released when this scope ends
      if (rc == 1) { b7_set_error("dngo_score: layer shapes do not fit the tile kernel (widths <= 63, at most 4 layers)"); rc = B7_ERR_ARG; }
    }
  }
  if (rc == 0 && M > 0) {
    StageTimer t(ctx, ST_SCORE);
    rc = b7_launch_score(ctx, kind, mom, mom + (size_t)S * M, S, M, M, tradeoff, bound, sign, fmin, features->removed_dev,
                         (int64_t)features->removed.size(), 0, sc, pb.best, pb.idx, pb.nan, &parts);
    t.stop(1);
  }
  std::vector<double> hb((size_t)parts); std::vector<int64_t> hi((size_t)parts), hn((size_t)parts);
  if (rc == 0 && parts) {
    cudaMemcpyAsync(hb.data(), pb.best, parts * 8, cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(hi.data(), pb.idx, parts * 8, cudaMemcpyDeviceToHost, ctx->stream);
    cudaMemcpyAsync(hn.data(), pb.nan, parts * 8, cudaMemcpyDeviceToHost, ctx->stream);
  }
  if (rc == 0 && score_host && M > 0) cudaMemcpyAsync(score_host, sc, (size_t)M * 8, cudaMemcpyDeviceToHost, ctx->stream);
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  b7_pool_free(ctx, mom); b7_pool_free(ctx, sc);
  if (rc == 0 && e != cudaSuccess) { b7_set_error("blr_score: %s", cudaGetErrorString(e)); rc = B7_ERR_CUDA; }
  if (rc < 0) return rc;
  double bv = -INFINITY; int64_t bi = INT64_MAX, nn = 0;
  for (int p = 0; p < parts; ++p) {
    nn += hn[p];
    if (hi[p] == INT64_MAX) continue;
    if (hb[p] > bv || (hb[p] == bv && hi[p] < bi)) { bv = hb[p]; bi = hi[p]; }
  }
  const int64_t orig = bi == INT64_MAX ? 0 : bi + 1;
  if (argmax_original) *argmax_original = orig;
  if (argmax) {
    if (!orig) *argmax = 0;
    else *argmax = (orig - 1) - (std::lower_bound(features->removed.begin(), features->removed.end(), orig - 1) - features->removed.begin()) + 1;
  }
  if (best) *best = orig ? bv : NAN;
  if (nan_count) *nan_count = nn;
  return 0;
}

int b7_blr_score(b7_blr* blr, b7_grid* features, int kind, double tradeoff, int bound, double sign, double fmin,
                 double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count) {
  return blr_score_impl(blr, features, 0, nullptr, nullptr, nullptr, nullptr, kind, tradeoff, bound, sign, fmin, score_host, argmax, argmax_original,
                        best, nan_count);
}

int b7_dngo_score(b7_blr* blr, b7_grid* grid, int n_layers, const int* dims, const double* const* W, const double* const* b, int relu_last,
                  int kind, double tradeoff, int bound, double sign, double fmin, double* score_host, int64_t* argmax,
                  int64_t* argmax_original, double* best, int64_t* nan_count) {
  return b7_dngo_score_act(blr, grid, n_layers, dims, W, b, b7_relu_codes(n_layers, relu_last).data(), kind, tradeoff, bound, sign, fmin,
                           score_host, argmax, argmax_original, best, nan_count);
}

int b7_dngo_score_act(b7_blr* blr, b7_grid* grid, int n_layers, const int* dims, const double* const* W, const double* const* b,
                      const int* act, int kind, double tradeoff, int bound, double sign, double fmin, double* score_host, int64_t* argmax,
                      int64_t* argmax_original, double* best, int64_t* nan_count) {
  if (!grid || n_layers < 1 || !dims || !W || !b || dims[0] != grid->d || !blr || dims[n_layers] != blr->D) {
    b7_set_error("dngo_score: bad arguments (dims[0] must equal the grid's dims, dims[n_layers] the head's D)");
    return B7_ERR_ARG;
  }
  B7_CHECK(b7_check_act("dngo_score", n_layers, act));
  return blr_score_impl(blr, grid, n_layers, dims, W, b, act, kind, tradeoff, bound, sign, fmin, score_host, argmax, argmax_original, best,
                        nan_count);
}

}  // extern "C"

// One step of the directed slice sampler (reference samplers/slice.lua:92-168; bot7_b200/samplers.py: slice.directed_slice)
// on GP hyper-parameters in one launch, for fits of up to 128 observations (one 128 x 128 block).
//
// One CTA of DIAG_THREADS threads.  Every density evaluation -- kernel parameters, K(X, X), Cholesky, beta = L^-1 (y - m),
// log-determinant, the jitter retry of utils.math.chol and the N(0, prior_std^2) prior -- runs in shared memory, and the
// step-out / shrink control flow runs between them.  The host pre-draws the step's random numbers (the direction, log U of
// the level, the bracket and K shrink uniforms) and gets back the new point and how many shrink uniforms it used.
//
// A density must carry the bits of b7_gp_refit(B7_FIT_LOGML_ONLY) + the host's prior term, because the samplers compare it
// with the level Y.  So it is made of the same operations as that path:
//   * kernel parameters: exp(-log l), exp(2 log sigma) with the host libm's arithmetic (host_exp.cuh), as set_hypers_host;
//   * K: the entry expression of the covariance builder (cov_entry.cuh), identity padding to 128;
//   * the diagonal-block factorisation of potrf.cu (potrf_diag.cuh): info, x = inv(L_00) r, the log-determinant;
//   * the jitter retry of api.cu:gp_retry_draw: ||K||_F by frob_rows_kernel's reduction tree, eps *= 1.1 until the
//     factorisation succeeds or eps > ||K||_F, in which case the density is -inf like the host's guard;
//   * log ml = -1/2 beta^T beta - log det - N/2 log 2 pi and the prior in the host's order of operations, every one an
//     explicitly rounded intrinsic (the host code has no fused multiply-add).
#include <math.h>

#include "b7_internal.h"
#include "cov_entry.cuh"
#include "host_exp.cuh"
#include "potrf_diag.cuh"

namespace {

constexpr int kHP = 48;                        // padded length of the hyper-parameter vectors in shared memory
constexpr double kLog2Pi = 1.83787706640934548356;
// shared memory after the diagonal-block region: y, w, point, x0, dir, left, right, dx, beta, frobenius rows, exp table
constexpr int kExtraDoubles = NBK + kHP + 6 * kHP + NBK + NBK + 64 + 8;
constexpr int kSmem = DIAG_SMEM + kExtraDoubles * 8;
static_assert(kSmem <= 227 * 1024, "slice step: shared memory");
static_assert((8 * SB * DSLD + 64 * TLD) >= NBK * (B7_MAX_DIMS - 1), "slice step: X staging area");

struct Smem {
  double *M, *X, *rj, *lg, *y, *w, *h, *x0, *dir, *left, *right, *dx, *beta, *frob, *tab, *sc;
  int* info;
  __device__ void init(double* sm, int* s_info) {
    M = sm;
    X = M + NBK * DLD;                         // DS and T: free while K is built
    rj = X + 8 * SB * DSLD + 64 * TLD + 2 * NBK;
    lg = rj + NBK;
    y = sm + DIAG_SMEM / 8;
    w = y + NBK;
    h = w + kHP;
    x0 = h + kHP;
    dir = x0 + kHP;
    left = dir + kHP;
    right = left + kHP;
    dx = right + kHP;
    beta = dx + kHP;
    frob = beta + NBK;
    tab = frob + NBK;
    sc = tab + 64;                             // scalars: sf2, diag0, density
    info = s_info;
  }
};

struct Args {
  const double* X;        // device N x d
  int N, d, noiseless, prior_order, K;
  double log_u, width, max_step, prior_std;
};

// K(X, X) with `diag` on the diagonal into M (lower triangle, zeros above, identity padding), as cov_kernel + the load of
// diag_kernel produce it; X is staged first (the area is the factorisation's scratch)
template <int KERNEL>
__device__ void build_k(const Smem& S, const Args& a, double diag) {
  const int tid = threadIdx.x, N = a.N, d = a.d;
  for (int e = tid; e < N * d; e += blockDim.x) S.X[e] = a.X[e];
  __syncthreads();
  const double sf2 = S.sc[0];
  for (int e = tid; e < NBK * NBK; e += blockDim.x) {
    const int i = e >> 7, k = e & (NBK - 1);
    double val = 0.0;
    if (k <= i) {
      if (i < N) {
        double r2 = 0.0;
        for (int c = 0; c < d; ++c) {
          const double t = __dmul_rn(__dsub_rn(S.X[i * d + c], S.X[k * d + c]), S.w[c]);
          r2 = __fma_rn(t, t, r2);
        }
        val = cov_value<KERNEL>(r2, sf2, S.tab);
        if (i == k) val = __dadd_rn(val, diag);
      } else {
        val = (i == k) ? 1.0 : 0.0;
      }
    }
    S.M[i * DLD + k] = val;
  }
  if (tid == 0) *S.info = 0;
  __syncthreads();
}

// the kernel parameters of the point in S.h (api.cu: set_hypers_host): w, sf2, the nominal diagonal addend; and r = y - m
__device__ void set_params(const Smem& S, const Args& a) {
  const int tid = threadIdx.x, d = a.d;
  if (tid < d) S.w[tid] = host_exp(-S.h[tid]);
  if (tid == 32) {
    const double sf2 = host_exp(__dmul_rn(2.0, S.h[d])), sn2 = host_exp(__dmul_rn(2.0, S.h[d + 1]));
    S.sc[0] = sf2;
    S.sc[1] = __dadd_rn(sn2, a.noiseless ? __dmul_rn(1e-8, sf2) : 0.0);
  }
  if (tid >= 64 && tid < 64 + NBK) {
    const int i = tid - 64;
    S.rj[i] = i < a.N ? __dsub_rn(S.y[i], S.h[d + 2]) : 0.0;
  }
  __syncthreads();
}

// factor M; returns info (all threads) and leaves beta = L^-1 r in S.beta
__device__ int factor(const Smem& S) {
  diag_factor_invert<false>(S.M, S.info, nullptr, 0);
  const double xv = diag_solve(S.M, S.rj, threadIdx.x);
  if ((threadIdx.x & 3) == 0) S.beta[threadIdx.x >> 2] = xv;
  __syncthreads();
  return *S.info;
}

// ||K||_F from the lower triangle in M, in the order of frob_rows_kernel (a 256-thread tree per row: entries k <= row < 128
// sit in the first half, so its first level adds zeros) and of gp_retry_draw's host sum over the rows
__device__ double frobenius(const Smem& S, int N) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int row = warp; row < N; row += DIAG_WARPS) {
    double v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int k = lane + 32 * q;
      const double m = S.M[row * DLD + k];
      v[q] = k <= row ? __dmul_rn(__dmul_rn(k < row ? 2.0 : 1.0, m), m) : 0.0;
    }
    double t = __dadd_rn(__dadd_rn(v[0], v[2]), __dadd_rn(v[1], v[3]));   // levels 64 and 32
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t = __dadd_rn(t, __shfl_down_sync(0xffffffffu, t, o));
    if (lane == 0) S.frob[row] = t;
  }
  __syncthreads();
  double ss = 0.0;
  for (int i = 0; i < N; ++i) ss = __dadd_rn(ss, S.frob[i]);
  return __dsqrt_rn(ss);
}

// log p(y | h) of the point in S.h, as b7_gp_refit(B7_FIT_LOGML_ONLY) and the host guard make it (-inf unless info == 0
// and the value is finite)
template <int KERNEL>
__device__ double log_lik(const Smem& S, const Args& a) {
  set_params(S, a);
  const double diag0 = S.sc[1];
  build_k<KERNEL>(S, a, diag0);
  int info = factor(S);
  if (info != 0) {                               // utils.math.chol's retry (api.cu: gp_retry_draw)
    build_k<KERNEL>(S, a, diag0);
    const double max_eps = frobenius(S, a.N);
    double eps = 1e-8;
    while (true) {
      if (eps > max_eps || !isfinite(max_eps)) return -INFINITY;   // chol(I): info stays that of the plain attempt
      eps = __dmul_rn(eps, 1.1);
      build_k<KERNEL>(S, a, __dadd_rn(diag0, eps));
      info = factor(S);
      if (info == 0) break;
    }
  }
  double q = 0.0;
  for (int k = 0; k < a.N; ++k) q = __dadd_rn(q, __dmul_rn(S.beta[k], S.beta[k]));
  const double ld = __dadd_rn(0.0, diag_logdet(S.lg));
  const double lml = __dsub_rn(__dsub_rn(__dmul_rn(-0.5, q), ld), __dmul_rn(__dmul_rn(0.5, (double)a.N), kLog2Pi));
  return isfinite(lml) ? lml : -INFINITY;
}

// -1/2 sum (h_i / prior_std)^2 subtracted from lp in the caller's order: 0 sequential (Torch7's sum), 1 numpy's pairwise
// sum (eight partial sums from eight terms on, then the rest one by one)
__device__ double add_prior(const double* h, int H, double sd, int order, double lp) {
  auto sq = [&](int i) { const double t = __ddiv_rn(h[i], sd); return __dmul_rn(t, t); };
  double sum = 0.0;
  if (order == 0 || H < 8) {
    for (int i = 0; i < H; ++i) sum = __dadd_rn(sum, sq(i));
  } else {
    double r[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = sq(j);
    int i = 8;
    for (; i < H - (H % 8); i += 8)
#pragma unroll
      for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], sq(i + j));
    double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])), __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
    for (; i < H; ++i) res = __dadd_rn(res, sq(i));
    sum = __dadd_rn(0.0, res);
  }
  return __dsub_rn(lp, __dmul_rn(0.5, sum));
}

// the density at x0 + dir * dx (dx in S.dx), broadcast to every thread
template <int KERNEL>
__device__ double density(const Smem& S, const Args& a) {
  const int H = a.d + 3;
  if (threadIdx.x < H) S.h[threadIdx.x] = __dadd_rn(S.x0[threadIdx.x], __dmul_rn(S.dir[threadIdx.x], S.dx[threadIdx.x]));
  __syncthreads();
  const double lp = log_lik<KERNEL>(S, a);
  if (threadIdx.x == 0) S.sc[2] = add_prior(S.h, H, a.prior_std, a.prior_order, lp);
  __syncthreads();
  const double v = S.sc[2];
  __syncthreads();
  return v;
}

// io: [x0 | dir | u_right] (H each) | u_shrink (K) | out: x1 (H), log p(x1), shrink uniforms used, evaluations, status
template <int KERNEL>
__global__ void __launch_bounds__(DIAG_THREADS, 1)
slice_step_kernel(const double* __restrict__ gX, const double* __restrict__ gy, double* __restrict__ io, Args a) {
  extern __shared__ __align__(16) double sm[];
  __shared__ int s_info;
  Smem S;
  S.init(sm, &s_info);
  const int tid = threadIdx.x, H = a.d + 3;
  a.X = gX;
  const double* u_right = io + 2 * H;
  const double* u_shrink = io + 3 * H;
  double* out = io + 3 * H + a.K;
  if (tid < NBK) S.y[tid] = tid < a.N ? gy[tid] : 0.0;
  if (tid < 64) S.tab[tid] = c_exp_tab[tid];
  if (tid < H) {
    S.x0[tid] = io[tid];
    S.dir[tid] = io[H + tid];
    S.dx[tid] = 0.0;
  }
  __syncthreads();
  int evals = 1;
  const double Y = __dadd_rn(density<KERNEL>(S, a), a.log_u);      // samplers/slice.lua:106-108
  if (tid < H) {                                                     // :114-115
    S.right[tid] = __dmul_rn(u_right[tid], a.width);
    S.left[tid] = __dsub_rn(S.right[tid], a.width);
  }
  __syncthreads();
  for (int side = 0; side < 2; ++side) {                             // :118-130, the right end first
    double* end = side == 0 ? S.right : S.left;
    double itr = 0.0;
    while (true) {
      if (tid < H) S.dx[tid] = end[tid];
      __syncthreads();
      const double f = density<KERNEL>(S, a);
      ++evals;
      if (!(f > Y && itr < a.max_step)) break;
      itr += 1.0;
      if (tid < H) end[tid] = side == 0 ? __dadd_rn(end[tid], a.width) : __dsub_rn(end[tid], a.width);
    }
  }
  int used = 0, status = 0;
  double y = 0.0;
  while (true) {                                                     // :134-164
    if (used == a.K) { status = 1; break; }
    const double u = u_shrink[used++];
    if (tid < H) S.dx[tid] = __dadd_rn(S.left[tid], __dmul_rn(__dsub_rn(S.right[tid], S.left[tid]), u));
    __syncthreads();
    y = density<KERNEL>(S, a);
    ++evals;
    if (y != y) break;
    if (y > Y) break;
    if (__syncthreads_or(tid < H && S.dx[tid] == 0.0)) break;
    if (tid < H) {
      const double v = S.dx[tid];
      if (v > 0.0) S.right[tid] = v;
      if (v < 0.0) S.left[tid] = v;
    }
  }
  if (tid < H) out[tid] = S.h[tid];                                  // x0 + dir * dx of the last proposal
  if (tid == 0) {
    out[H] = y;
    out[H + 1] = used;
    out[H + 2] = evals;
    out[H + 3] = status;
  }
}

}  // namespace

int b7_launch_slice_step(b7_gp* gp, double* io, int K, double log_u, double width, double max_step, double prior_std,
                         int prior_order) {
  b7_ctx* ctx = gp->ctx;
  static bool attr[16] = {false};
  if (!attr[ctx->device & 15]) {
    B7_CUDA(cudaFuncSetAttribute(slice_step_kernel<B7_KERNEL_ARDSE>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    B7_CUDA(cudaFuncSetAttribute(slice_step_kernel<B7_KERNEL_MATERN52>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
    attr[ctx->device & 15] = true;
  }
  Args a;
  a.X = nullptr;
  a.N = gp->N; a.d = gp->d; a.noiseless = gp->noiseless; a.prior_order = prior_order; a.K = K;
  a.log_u = log_u; a.width = width; a.max_step = max_step; a.prior_std = prior_std;
  if (gp->kernel == B7_KERNEL_ARDSE)
    slice_step_kernel<B7_KERNEL_ARDSE><<<1, DIAG_THREADS, kSmem, ctx->stream>>>(gp->X, gp->y, io, a);
  else
    slice_step_kernel<B7_KERNEL_MATERN52><<<1, DIAG_THREADS, kSmem, ctx->stream>>>(gp->X, gp->y, io, a);
  b7_count(ctx);
  B7_CUDA(cudaGetLastError());
  return 0;
}

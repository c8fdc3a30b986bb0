// DNGO candidate pass on the FP64 tensor pipe: (optional) MLP basis (ReLU / tanh / no activation per layer) followed by the
// BLR head, tile by tile.
//
// Replaces, for the candidate grid, what models/dngo.lua:155-174 does in 32-row Lua minibatches: Z1 = basis(X_hid)
// (:165-171) and predictor:predict(Z0, Y0, Z1, ...) (:174).  One CTA works on tiles of 128 candidates that never
// leave shared memory between the layers:
//     act_0 = the tile's rows of the input grid (X, or precomputed features)
//     act_l+1 = act(W_l act_l + b_l)                      l = 0 .. n_layers-1   (nn.Linear + nn.ReLU / nn.Tanh / nothing)
//     v = L_A^-1 phi,  var = |v|^2 + 1/beta,  mean = m + w^T phi                 per (alpha_p, beta) draw
// Every product is a DMMA m8n8k4 fragment product: the weights (and, for the head, [L_A^-1 ; w^T] as one matrix whose
// last row yields the mean) sit in shared memory for the whole launch with a leading dimension = 4 mod 16 doubles
// (conflict-free fragment loads), a warp owns 16 candidates and all output rows, and the head skips the fragments
// above the diagonal of the triangular L_A^-1.  The one-DFMA-thread-per-candidate kernels of blr.cu ran at 27 %
// (BLR) and 22 % (MLP) of the FP64 pipe; they remain as the fallback for shapes whose weights do not fit.
// With the basis fused, the 8 D bytes per candidate of Z1 (1.7 GB at config 4) are never written or read.
// A tile's rows are contiguous in the grid, so the input tile arrives as ONE cp.async.bulk (TMA unit, mbarrier-tracked) in
// its raw layout [candidate][w_in]; the fragment loads read it with that leading dimension (2-way bank conflicts on the two
// B loads of a k-step at most) and mask the columns beyond w_in, so nothing is repacked: the first versions spent ~400 of
// their ~2 700 instructions per warp and tile on staging the tile through registers.
#include <algorithm>
#include <vector>

#include "b7_internal.h"
#include "gemm_tile.cuh"

using b7g::dmma884;

namespace {

constexpr int TC = 128;            // candidates per tile
constexpr int THREADS = 256;       // 8 warps x 16 candidates
constexpr int MAXL = 4;            // MLP layers
constexpr int MAXF = 8;            // output fragments of 8 rows (widths <= 64)

// leading dimension: >= width rounded up to 4, = 4 mod 16 (fragment rows land in distinct banks)
__host__ __device__ inline int ld_of(int width) {
  const int w4 = (width + 3) / 4 * 4;
  return w4 + ((4 - w4 % 16) + 16) % 16;
}

struct Plan {
  int n_layers;                 // MLP layers before the head
  int width[MAXL + 1];          // width[0] = input width, width[l + 1] = output of layer l
  int relu[MAXL];               // 1: ReLU after layer l
  int tanh[MAXL];               // 1: tanh after layer l (dngo_tile_kernel<true> only)
  int w_off[MAXL];              // offsets (doubles) of the staged weights / biases in shared memory
  int b_off[MAXL];
  int head_off;                 // [S][rows_pad][ld(D)] head matrices
  int head_rows;                // D + 1 rounded up to 8
  int raw_off;                  // input tile in its global layout [TC][width[0]] (one bulk copy)
  int act_off;                  // activation buffer [TC][act_ld] (only with layers); a layer >= 1 overwrites it in place
  int act_ld;
  int bar_off;                  // mbarrier of the bulk copy
  int S;                        // draws staged (0: no head, write the features)
};

struct Ptrs {
  const double* W[MAXL];
  const double* b[MAXL];
};

// acc[i][j] (+)= A[8i.., k] * B[cand.., k]^T over k < K4; A: rows x lda, Bt: [cand][ldb].
// MF (output fragments) and LDA (leading dimension of A) are compile-time constants: the fragment loop carries no branches
// and every A fragment is one LDS at a constant offset from one running pointer (with run-time shapes the compiler spent ~20
// integer instructions per fragment load on re-deriving addresses: 2 700 instructions per warp and tile, 4 % of them DMMAs).
// tri: A is [L^-1 ; w^T] -- fragment i is zero for k > 8 i + 7, except the last one (it holds the dense row w^T), so the
// fragments active at k0 are the suffix i >= k0 / 8.
template <int MF, int LDA>
__device__ __forceinline__ void tile_mma_t(const double* __restrict__ A, int K4, const double* __restrict__ Bt, int ldb, int kmax, int lane,
                                           double (&acc)[MAXF][2][2], bool tri) {
  const int r = lane >> 2, c = lane & 3;
  const double* B0 = Bt + r * ldb + c;
  const double* B1 = Bt + (8 + r) * ldb + c;
  const double* Ar = A + r * LDA + c;                  // LDA is a compile-time constant: fragment i is one LDS at [Ar + k0 + 8 i LDA]
  // A predicated-off DMMA still holds the FP64 tensor pipe for its 16 cycles (ncu dngo_r02: 47.7 M DMMAs issued, 28.8 M
  // predicated on, pipe busy for all of them): fragments above the diagonal are skipped at compile time, not by predicates.
  if (tri) {
    // [L^-1 ; w^T]: fragments i >= q (and the last one) are non-zero in columns 8 q .. 8 q + 7.  q is unrolled at compile
    // time, so every fragment load is one LDS at a constant offset and the skip costs nothing at run time.
#pragma unroll
    for (int q = 0; q < MF; ++q) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int k0 = 8 * q + 4 * h;
        if (k0 < K4) {                                   // warp-uniform
          const bool kin = k0 + c < kmax;
          const double b0 = kin ? B0[k0] : 0.0, b1 = kin ? B1[k0] : 0.0;
          double av[8];
#pragma unroll
          for (int i = 0; i < MF; ++i)
            if (i >= q || i == MF - 1) av[i] = Ar[8 * i * LDA + k0];
#pragma unroll
          for (int i = 0; i < MF; ++i)
            if (i >= q || i == MF - 1) {
              dmma884(acc[i][0][0], acc[i][0][1], av[i], b0);
              dmma884(acc[i][1][0], acc[i][1][1], av[i], b1);
            }
        }
      }
    }
    return;
  }
  // dense layers: one k-step (4 columns) at a time, the A fragments of the step, then its DMMAs (up to 14 independent
  // accumulators between two DMMAs on the same one; dmma884 is `asm volatile`, kept in program order)
  for (int k0 = 0; k0 < K4; k0 += 4, Ar += 4, B0 += 4, B1 += 4) {
    const bool kin = k0 + c < kmax;                    // the raw tile has no padding columns: mask instead
    const double b0 = kin ? *B0 : 0.0, b1 = kin ? *B1 : 0.0;
    double av[8];
#pragma unroll
    for (int i = 0; i < MF; ++i) av[i] = Ar[8 * i * LDA];
#pragma unroll
    for (int i = 0; i < MF; ++i) {
      dmma884(acc[i][0][0], acc[i][0][1], av[i], b0);
      dmma884(acc[i][1][0], acc[i][1][1], av[i], b1);
    }
  }
}

template <int LDA>
__device__ __forceinline__ void tile_mma_l(const double* __restrict__ A, int mf, int K4, const double* __restrict__ Bt, int ldb, int kmax,
                                           int lane, double (&acc)[MAXF][2][2], bool tri) {
  switch (mf) {
    case 1: tile_mma_t<1, LDA>(A, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 2: tile_mma_t<2, LDA>(A, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 3: tile_mma_t<3, LDA>(A, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 4: tile_mma_t<4, LDA>(A, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 5: tile_mma_t<5, LDA>(A, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 6: tile_mma_t<6, LDA>(A, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 7: tile_mma_t<7, LDA>(A, K4, Bt, ldb, kmax, lane, acc, tri); break;
    default: tile_mma_t<8, LDA>(A, K4, Bt, ldb, kmax, lane, acc, tri); break;
  }
}

// lda is ld_of(k width): one of 4, 20, 36, 52, 68
__device__ __forceinline__ void tile_mma(const double* __restrict__ A, int lda, int mf, int K4, const double* __restrict__ Bt, int ldb,
                                         int kmax, int lane, double (&acc)[MAXF][2][2], bool tri) {
  switch (lda) {
    case 4: tile_mma_l<4>(A, mf, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 20: tile_mma_l<20>(A, mf, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 36: tile_mma_l<36>(A, mf, K4, Bt, ldb, kmax, lane, acc, tri); break;
    case 52: tile_mma_l<52>(A, mf, K4, Bt, ldb, kmax, lane, acc, tri); break;
    default: tile_mma_l<68>(A, mf, K4, Bt, ldb, kmax, lane, acc, tri); break;
  }
}

// TANH: some layer has B7_ACT_TANH.  The tanh pass is compiled only into that instantiation, so that a stack without Tanh runs
// the instructions it ran before activation codes existed (the same SASS, register count and stack frame).
template <bool TANH>
__global__ void __launch_bounds__(THREADS, 2)
dngo_tile_kernel(const double* __restrict__ in, long long M, Plan pl, Ptrs pt, const double* __restrict__ Linv, const double* __restrict__ wv,
                 const double* __restrict__ par, int D, long long ld_out, double* __restrict__ mean, double* __restrict__ var,
                 double* __restrict__ feat_out) {
  extern __shared__ __align__(16) double sh[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, r = lane >> 2, c = lane & 3;
  // ---- stage the weights once per CTA (zero padded) ----
  for (int l = 0; l < pl.n_layers; ++l) {
    const int hi = pl.width[l], ho = pl.width[l + 1], ldw = ld_of(hi), rows = (ho + 7) / 8 * 8;
    for (int e = tid; e < rows * ldw; e += THREADS) {
      const int j = e / ldw, k = e % ldw;
      sh[pl.w_off[l] + e] = (j < ho && k < hi) ? pt.W[l][(long long)j * hi + k] : 0.0;
    }
    for (int e = tid; e < rows; e += THREADS) sh[pl.b_off[l] + e] = e < ho ? pt.b[l][e] : 0.0;
  }
  const int ldh = ld_of(D);
  for (int s = 0; s < pl.S; ++s)
    for (int e = tid; e < pl.head_rows * ldh; e += THREADS) {
      const int i = e / ldh, k = e % ldh;
      double v = 0.0;
      if (k < D) {
        if (i < D) v = k <= i ? Linv[((long long)s * D + i) * D + k] : 0.0;
        else if (i == D) v = wv[(long long)s * D + k];
      }
      sh[pl.head_off + s * pl.head_rows * ldh + e] = v;
    }
  __syncthreads();

  const long long n_tiles = (M + TC - 1) / TC;
  const int w_in = pl.width[0], lda = pl.act_ld;
  double* raw = sh + pl.raw_off;
  double* act = sh + pl.act_off;
  uint64_t* bar = reinterpret_cast<uint64_t*>(sh + pl.bar_off);
  // the tile is one contiguous run of nc * w_in doubles: a single bulk copy when rows are a multiple of 16 bytes
  const bool bulk = (w_in & 1) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0;
  auto issue = [&](long long tile) {                   // thread 0 only
    const long long c0 = tile * TC;
    const unsigned bytes = (unsigned)(min((long long)TC, M - c0) * w_in * 8);
    b7g::mbar_arrive_expect_tx(bar, bytes);
    b7g::bulk_g2s(raw, in + c0 * w_in, bytes, bar);
  };
  if (tid == 0) {
    b7g::mbar_init(bar, 1);
    b7g::mbar_fence_init();
    if (bulk && (long long)blockIdx.x < n_tiles) issue(blockIdx.x);
  }
  __syncthreads();
  unsigned phase = 0;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long c0 = tile * TC;
    const int nc = (int)min((long long)TC, M - c0);
    const bool more = tile + gridDim.x < n_tiles;
    if (bulk) {
      b7g::mbar_wait(bar, phase);
      phase ^= 1u;
    } else {
      // rows that are not a multiple of 16 bytes: flat coalesced copy into the same raw layout, 16 loads in flight per thread
      const double* src = in + c0 * w_in;
      const int total = nc * w_in;
      for (int f0 = tid; f0 < total; f0 += 16 * THREADS) {
        double buf[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) buf[i] = f0 + i * THREADS < total ? src[f0 + i * THREADS] : 0.0;
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (f0 + i * THREADS < total) raw[f0 + i * THREADS] = buf[i];
      }
      __syncthreads();
    }
    // rows >= nc of a partial last tile hold whatever the previous tile left: their results are never stored
    const double* X = raw + warp * 16 * w_in;          // this warp's 16 candidates
    int ldx = w_in;
    // ---- MLP layers ----
    for (int l = 0; l < pl.n_layers; ++l) {
      const int hi = pl.width[l], ho = pl.width[l + 1], mf = (ho + 7) / 8, K4 = (hi + 3) / 4 * 4;
      double acc[MAXF][2][2];
#pragma unroll
      for (int i = 0; i < MAXF; ++i) acc[i][0][0] = acc[i][0][1] = acc[i][1][0] = acc[i][1][1] = 0.0;
      tile_mma(sh + pl.w_off[l], ld_of(hi), mf, K4, X, ldx, hi, lane, acc, false);
      if (l == 0 && bulk) {                            // every warp is done with the raw tile: fetch the next one under the rest
        __syncthreads();
        if (tid == 0 && more) issue(tile + gridDim.x);
      }
      const double* bias = sh + pl.b_off[l];
      __syncwarp();                                    // every lane has read the warp's 16 input rows: overwrite them in place
      double* out = act + warp * 16 * lda;
#pragma unroll
      for (int i = 0; i < MAXF; ++i) {
        if (i >= mf) break;
        const int row = 8 * i + r;
        if (row >= ho) continue;
        const double bb = bias[row];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            double v = acc[i][j][e] + bb;
            if (pl.relu[l]) v = v > 0.0 ? v : 0.0;
            out[(8 * j + 2 * c + e) * lda + row] = v;
          }
      }
      __syncwarp();                                    // a warp only reads the 16 candidates it wrote
      if (TANH && pl.tanh[l]) {
        // a second pass over the warp's 16 x ho outputs in shared memory, one element per lane and step: tanh (libdevice,
        // DESIGN.md section 4.5) inlined once rather than in each of the 32 unrolled slots of the loop above, and no lane
        // idles while ho is not a multiple of 8
        int cc = lane / ho, j = lane - cc * ho;
        while (cc < 16) {
          double* p = out + cc * lda + j;
          *p = tanh(*p);
          for (j += 32; j >= ho && cc < 16; j -= ho) ++cc;
        }
        __syncwarp();
      }
      X = out;
      ldx = lda;
    }
    const int w_last = pl.width[pl.n_layers];
    if (pl.S == 0) {
      // ---- features out (b7_mlp_features): [cand][w_last] contiguous ----
      __syncthreads();
      for (int e = tid; e < nc * w_last; e += THREADS) feat_out[c0 * w_last + e] = act[(e / w_last) * lda + e % w_last];
    } else {
      // ---- BLR head per draw: rows 0 .. D-1 of the product are v = L_A^-1 phi, row D is w^T phi ----
      const int mf = pl.head_rows / 8, K4 = (D + 3) / 4 * 4;      // the dense row w^T sits in the last fragment (D / 8 = mf - 1)
      for (int s = 0; s < pl.S; ++s) {
        double acc[MAXF][2][2];
#pragma unroll
        for (int i = 0; i < MAXF; ++i) acc[i][0][0] = acc[i][0][1] = acc[i][1][0] = acc[i][1][1] = 0.0;
        tile_mma(sh + pl.head_off + s * pl.head_rows * ldh, ldh, mf, K4, X, ldx, D, lane, acc, true);
        if (pl.n_layers == 0 && bulk && s == pl.S - 1) {   // head only: the raw tile is free after the last draw's products
          __syncthreads();
          if (tid == 0 && more) issue(tile + gridDim.x);
        }
        double s2[2][2] = {{0.0, 0.0}, {0.0, 0.0}}, mu[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
        for (int i = 0; i < MAXF; ++i) {
          if (i >= mf) break;
          const int row = 8 * i + r;
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const double v = acc[i][j][e];
              if (row < D) s2[j][e] = fma(v, v, s2[j][e]);
              else if (row == D) mu[j][e] = v;
            }
        }
        // rows are spread over the 8 lanes that share lane & 3: fixed xor tree
#pragma unroll
        for (int o = 4; o < 32; o <<= 1)
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              s2[j][e] += __shfl_xor_sync(0xffffffffu, s2[j][e], o);
              mu[j][e] += __shfl_xor_sync(0xffffffffu, mu[j][e], o);
            }
        if (r == 0) {
          const double mconst = par[s * 4 + 2], inv_beta = par[s * 4 + 3];
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int cc = warp * 16 + 8 * j + 2 * c + e;
              if (cc < nc) {
                mean[(long long)s * ld_out + c0 + cc] = mconst + mu[j][e];
                var[(long long)s * ld_out + c0 + cc] = s2[j][e] + inv_beta;
              }
            }
        }
      }
    }
    __syncthreads();                                   // raw / act are rewritten by the next tile
  }
}

// Plans the shared memory of one launch; returns 1 if the shapes do not fit the tile kernel.
// act: n_layers B7_ACT_* codes (checked by the caller); nullptr plans the shared memory only.
int plan_tiles(int n_layers, const int* dims, const int* act, int D, int S, Plan* plan, size_t* smem_bytes) {
  if (n_layers > MAXL) return 1;
  Plan pl = {};
  pl.n_layers = n_layers;
  pl.S = S;
  int off = 0, wmax = dims[0];
  for (int l = 0; l <= n_layers; ++l) {
    if (dims[l] < 1 || dims[l] > 64) return 1;
    pl.width[l] = dims[l];
    wmax = std::max(wmax, dims[l]);
  }
  if (S > 0 && (D != dims[n_layers] || D + 1 > 64)) return 1;
  for (int l = 0; l < n_layers; ++l) {
    const int rows = (dims[l + 1] + 7) / 8 * 8;
    pl.relu[l] = act && act[l] == B7_ACT_RELU;
    pl.tanh[l] = act && act[l] == B7_ACT_TANH;
    pl.w_off[l] = off; off += rows * ld_of(dims[l]);
    pl.b_off[l] = off; off += rows;
  }
  pl.head_rows = S > 0 ? (D + 1 + 7) / 8 * 8 : 0;
  pl.head_off = off; off += S * pl.head_rows * (S > 0 ? ld_of(D) : 0);
  pl.act_ld = ld_of(wmax);
  off = (off + 1) / 2 * 2;                             // 16-byte aligned destination of the bulk copy
  pl.raw_off = off; off += TC * dims[0];
  off = (off + 1) / 2 * 2;
  pl.act_off = off; off += n_layers > 0 ? TC * pl.act_ld : 0;
  pl.bar_off = off; off += 2;
  const size_t smem = (size_t)off * sizeof(double);
  if (smem > 226 * 1024) return 1;
  *plan = pl;
  *smem_bytes = smem;
  return 0;
}

}  // namespace

// b7_dngo_score runs its head in chunks of at most four draws and halves the chunk down to one when a launch does not fit:
// the shapes are usable iff a one-draw launch fits.
bool b7_dngo_tiles_fit(int n_layers, const int* dims, int D) {
  Plan pl;
  size_t smem;
  return n_layers >= 1 && plan_tiles(n_layers, dims, nullptr, D, 1, &pl, &smem) == 0;
}

// Plans the shared memory, uploads nothing (all pointers are device pointers) and launches.  Returns 1 if the shapes
// do not fit the tile kernel (the caller then uses the per-candidate kernels of blr.cu).
int b7_launch_dngo_tiles(b7_ctx* ctx, const double* in, int64_t M, int n_layers, const int* dims, const double* const* W_dev,
                         const double* const* b_dev, const int* act, const double* Linv, const double* w, const double* par, int D, int S,
                         int64_t ld_out, double* mean, double* var, double* feat_out) {
  if (M <= 0) return 0;
  Plan pl;
  size_t smem;
  if (plan_tiles(n_layers, dims, act, D, S, &pl, &smem)) return 1;
  Ptrs pt = {};
  for (int l = 0; l < n_layers; ++l) {
    pt.W[l] = W_dev[l];
    pt.b[l] = b_dev[l];
  }
  static bool done[16] = {false};
  if (!done[ctx->device & 15]) {
    B7_CUDA(cudaFuncSetAttribute(dngo_tile_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    B7_CUDA(cudaFuncSetAttribute(dngo_tile_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    done[ctx->device & 15] = true;
  }
  bool tanh_any = false;
  for (int l = 0; l < n_layers; ++l) tanh_any = tanh_any || pl.tanh[l];
  const int64_t n_tiles = (M + TC - 1) / TC;
  const int per_sm = smem <= 110 * 1024 ? 2 : 1;
  const int grid = (int)std::min<int64_t>(n_tiles, (int64_t)ctx->sm_count * per_sm);
  if (tanh_any) dngo_tile_kernel<true><<<grid, THREADS, smem, ctx->stream>>>(in, M, pl, pt, Linv, w, par, D, ld_out, mean, var, feat_out);
  else dngo_tile_kernel<false><<<grid, THREADS, smem, ctx->stream>>>(in, M, pl, pt, Linv, w, par, D, ld_out, mean, var, feat_out);
  b7_count(ctx);
  B7_CUDA(cudaGetLastError());
  return 0;
}

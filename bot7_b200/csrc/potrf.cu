// Batched fp64 blocked Cholesky (kernel #2) with beta = L^-1 (y - m), log-determinant and LAPACK
// style info, plus the in-place triangular inversion used by the posterior pass.
//
// Replaces what Torch7 reaches through torch.potrf in utils.math.chol (reference
// utils/math.lua:159-218; LAPACK dpotrf, one matrix at a time) and the two triangular solves of
// gpTorch7's posterior.  One factor per slice-sampled hyper-parameter draw, all draws in one launch
// sequence (grid.z / grid.x = draw).
//
// Right-looking, block size 128 (= the DMMA tile edge of gemm_tile.cuh).  The matrices live in HBM in
// the tiled (fragment-order) layout of gemm_tile.cuh from the moment K is built until L^-1 is read by
// the posterior pass, so every operand k-step of every GEMM here is one 16 KB TMA bulk copy; lower
// storage, padded to a multiple of 128 with identity.  Per block column j:
//   diag  : one CTA per draw factors and inverts the 128x128 diagonal block inside shared memory,
//           blocked by 16 so that the work is DMMA fragment products; it also produces
//           x_j = L_jj^-1 r_j, the running log-determinant and info.
//   panel : L21 = A21 * inv(L11)^T as DMMA tiles; the epilogue folds r_i -= L21 x_j, so the forward
//           substitution for beta costs no extra pass over L.
//   trail : A22 -= L21 L21^T on the lower tiles (DMMA).  Two-level blocking: inside an outer panel of
//           4 blocks only the panel's own columns are updated per step (k = 128); the tiles to the
//           right of the panel are updated once per outer panel with k = 512, so most flops run in
//           long-k launches with a quarter of the read-modify-write traffic on C.
// Inversion (LAPACK dtrtri order, in place, column sweep from the right):
//   T = L[j+1:, j] * inv(L_jj)  (stored transposed), then  X[j+1:, j] = -Linv[j+1:, j+1:] * T.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "b7_internal.h"
#include "gemm_tile.cuh"

// tools/diag_probe.cu compiles this file with B7_DIAG_STAMPS to get a cycle stamp per phase of the diagonal-block kernel
#ifdef B7_DIAG_STAMPS
namespace {
__device__ long long b7_diag_stamps[128];
}  // namespace
#define DIAG_STAMP(i) do { if (threadIdx.x == 0 && blockIdx.x == 0) b7_diag_stamps[i] = clock64(); } while (0)
#endif
#include "potrf_diag.cuh"

using namespace b7g;

namespace {

// Programmatic dependent launch (single-factor schedule): a kernel launched with the programmatic-serialisation
// attribute may become resident once its stream predecessor has executed pdl_trigger() in every CTA; it must not touch
// global memory before pdl_wait(), which returns when the predecessor has completed and its writes are visible.
// Both are no-ops in a kernel that was launched without the attribute / has no dependent.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

__global__ void __launch_bounds__(DIAG_THREADS, 1)
diag_kernel(double* __restrict__ fac, long long fac_stride, int Np, int j, double* __restrict__ dinv, long long dinv_stride,
            double* __restrict__ beta, double* __restrict__ logdet, int* __restrict__ info, int s0) {
  extern __shared__ __align__(16) double sm[];
  double* M = sm;
  double* rj = M + NBK * DLD + 8 * SB * DSLD + 64 * TLD + 2 * NBK;
  double* lg = rj + NBK;
  __shared__ int s_info;
  const int s = s0 + blockIdx.x, tid = threadIdx.x;
  DIAG_STAMP(0);
  pdl_wait();
  double* blk = fac + (long long)s * fac_stride + tile_off(Np / TILE_K, j, j * (NBK / TILE_K));   // 8 tiles of block (j, j)
#pragma unroll 8
  for (int u = tid; u < NBK * NBK / 2; u += DIAG_THREADS) {
    // u enumerates pairs of doubles in the tiled order [kt][g4][row][kk]: 16 bytes per thread, consecutive threads
    // consecutive addresses; pairs above the diagonal are not read
    const int i = (u >> 1) & 127, k0 = (u >> 10) * TILE_K + ((u >> 8) & 3) * 4 + (u & 1) * 2;
    double2 v = make_double2(0.0, 0.0);
    if (k0 <= i) v = *reinterpret_cast<const double2*>(blk + 2 * u);
    *reinterpret_cast<double2*>(M + i * DLD + k0) = make_double2(v.x, k0 + 1 <= i ? v.y : 0.0);
  }
  if (tid < NBK) rj[tid] = beta[(long long)s * Np + j * NBK + tid];
  if (tid == 0) s_info = 0;
  __syncthreads();
  DIAG_STAMP(1);

  diag_factor_invert<true>(sm, &s_info, blk, j);
  // the panel kernel's CTAs may take their SMs now (not earlier: they would sit on 124 SMs that the side and far streams
  // use while this block is factored)
  pdl_trigger();
  // x_j = inv(L_jj) r_j : 4 threads per row, k interleaved, fixed shuffle tree
  {
    const double xv = diag_solve(M, rj, tid);
    if ((tid & 3) == 0) beta[(long long)s * Np + j * NBK + (tid >> 2)] = xv;
  }
  DIAG_STAMP(34);
  // the inverse in tiled order, ready to be a GEMM operand: only the pairs on or below the diagonal are written (the
  // buffer is zeroed once when the handle is created and nothing else writes to it; a single SM stores ~32 bytes per
  // cycle, so the 64 KB that are always zero would cost as much as the rest).  16 bytes per thread, consecutive
  // threads consecutive addresses.  The transposes (alpha_kernel, FP64 inversion sweep) are made by one launch for
  // all block columns after the factorisation (dinv_transpose_kernel).
  double* di = dinv + (long long)s * dinv_stride + (long long)j * NBK * NBK;
#pragma unroll 4
  for (int u = tid; u < NBK * NBK / 2; u += DIAG_THREADS) {
    const int i = (u >> 1) & 127, k0 = (u >> 10) * TILE_K + ((u >> 8) & 3) * 4 + (u & 1) * 2;
    if (k0 <= i) {
      const double2 v = *reinterpret_cast<const double2*>(M + i * DLD + k0);
      *reinterpret_cast<double2*>(di + 2 * u) = make_double2(v.x, k0 + 1 <= i ? v.y : 0.0);
    }
  }
  if (tid == 0) {
    logdet[s] = (j == 0 ? 0.0 : logdet[s]) + diag_logdet(lg);
    const int my_info = s_info;
    if (j == 0) info[s] = my_info;
    else if (info[s] == 0 && my_info != 0) info[s] = my_info;
  }
  DIAG_STAMP(35);
}

// dinvT(j) = dinv(j)^T for every block column and draw, tiled order on both sides
__global__ void dinv_transpose_kernel(const double* __restrict__ dinv, double* __restrict__ dinvT, long long dinv_stride, int s0) {
  const long long off = (long long)(s0 + blockIdx.y) * dinv_stride + (long long)blockIdx.x * NBK * NBK;
  const double* di = dinv + off;
  double* dt = dinvT + off;
  for (int e = threadIdx.x; e < NBK * NBK; e += blockDim.x) {
    const int kk = e & 3, i = (e >> 2) & 127, k = (e >> 11) * TILE_K + ((e >> 9) & 3) * 4 + kk;
    dt[e] = (k >= i) ? di[elem_off(k, i)] : 0.0;
  }
}

// ---- panel: L21 = A21 * inv(L11)^T, beta_i -= L21 x_j --------------------------------------------
__global__ void __launch_bounds__(THREADS, 1)
panel_kernel(double* __restrict__ fac, long long fac_stride, int Np, int j, const double* __restrict__ dinv,
             long long dinv_stride, double* __restrict__ beta, int s0) {
  extern __shared__ __align__(128) double smem[];
  const int s = s0 + blockIdx.z, it = j + 1 + blockIdx.x, KPB = NBK / TILE_K;
  double* tile = fac + (long long)s * fac_stride + tile_off(Np / TILE_K, it, j * KPB);
  const double* B = dinv + (long long)s * dinv_stride + (long long)j * NBK * NBK;
  Ring ring; ring.init(smem);
  Acc acc; acc.zero();
  mainloop_bulk(ring, tile, B, KPB, acc);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wm = warp >> 2, wn = warp & 3;
  const double* xj = beta + (long long)s * Np + j * NBK;
  double* red = smem;   // [128][4]
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int row = frag_row(wm, i, lane);
    double part = 0.0;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int col = frag_col(wn, jj, lane);
      *reinterpret_cast<double2*>(tile + elem_off(row, col)) = make_double2(acc.c[i][jj][0], acc.c[i][jj][1]);
      part += acc.c[i][jj][0] * xj[col] + acc.c[i][jj][1] * xj[col + 1];
    }
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    if ((lane & 3) == 0) red[row * 4 + wn] = part;
  }
  __syncthreads();
  if (tid < NBK) {
    double sum = ((red[tid * 4 + 0] + red[tid * 4 + 1]) + red[tid * 4 + 2]) + red[tid * 4 + 3];
    beta[(long long)s * Np + it * NBK + tid] -= sum;
  }
}

// ---- trailing update: C[it][nt] -= L[it][kb0:kb1] L[nt][kb0:kb1]^T on lower tiles ---------------
// it = it0 + blockIdx.x, nt = nt0 + blockIdx.y (tiles above the diagonal exit at once).  Used with
// one k block inside the current outer panel and with the whole outer panel (k = 128 * W) for the
// tiles to its right: the long-k launches carry most of the flops with one read-modify-write of C.
__global__ void __launch_bounds__(THREADS, 1)
trail_kernel(double* __restrict__ fac, long long fac_stride, int Np, int kb0, int kb1, int it0, int nt0, int s0) {
  extern __shared__ __align__(128) double smem[];
  const int it = it0 + blockIdx.x, nt = nt0 + blockIdx.y;
  if (nt > it) return;
  const int s = s0 + blockIdx.z, KPB = NBK / TILE_K, KTA = Np / TILE_K;
  double* base = fac + (long long)s * fac_stride;
  const double* A = base + tile_off(KTA, it, kb0 * KPB);
  const double* B = base + tile_off(KTA, nt, kb0 * KPB);
  double* C = base + tile_off(KTA, it, nt * KPB);
  Ring ring; ring.init(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wm = warp >> 2, wn = warp & 3;
  if (threadIdx.x == 0)   // start the operand stream before touching C
    for (int p = 0; p < 2 && p < (kb1 - kb0) * KPB; ++p) ring.produce(A + (long long)p * TILE_DOUBLES, B + (long long)p * TILE_DOUBLES);
  // acc starts at -C (loaded while the first bulk copies are in flight), accumulates +A B^T, and C_new = -acc:
  // the read of C is off the critical path and the epilogue is stores only
  Acc acc;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const double2 v = *reinterpret_cast<const double2*>(C + elem_off(frag_row(wm, i, lane), frag_col(wn, jj, lane)));
      acc.c[i][jj][0] = -v.x;
      acc.c[i][jj][1] = -v.y;
    }
  mainloop_bulk(ring, A, B, (kb1 - kb0) * KPB, acc, 2);
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
      *reinterpret_cast<double2*>(C + elem_off(frag_row(wm, i, lane), frag_col(wn, jj, lane))) =
          make_double2(-acc.c[i][jj][0], -acc.c[i][jj][1]);
}

// ---- row-sliced variants for one or two factors ----------------------------------------------------
// With a single factor a block column offers at most 31 tiles: one CTA per tile leaves most SMs idle for the ~17 us a
// 128 x 128 x 128 product takes on one SM's DMMA pipe, and the k = 512 updates hold an SM for ~70 us while the chain's
// next kernel waits for a free one.  Here a CTA owns SL_ROWS rows of a tile (first 32 rows = 4 CTAs per tile, now 16 = 8 CTAs per
// tile, see below): the B operand streams as whole 16 KB k-tiles, the A operand as the 4 row runs of its k-tile.  Every output element sees the
// same DMMA sequence (k ascending, one accumulator) and the beta reduction keeps the order of panel_kernel, so the
// results are bit-identical to the tile kernels.  Warp (wm, wn) owns rows 16 wm.., columns 32 wn.. : 2 x 4 fragments.
// Second step: SL_ROWS = 16 with 4 warps per CTA (8 CTAs per tile; N = 4096 refit 2.04 -> 1.99 ms, N = 2048 0.85 -> 0.82).  A warp keeps exactly the fragment shape and
// the instruction sequence it had with 32-row slices (16 rows x 32 columns), so every output element and every partial of the
// beta reduction is computed by the same operations in the same order -- only the DMMA time of a CTA halves (one warp per
// sub-core, 256 DMMAs = 4096 cycles per k = 128 product).  6 stages of 18 KB leave room for two CTAs per SM, so that the
// 8 x 31 CTAs of the first block columns at N = 4096 are one wave.
constexpr int SL_ROWS = 16, SL_STAGES = 6, SL_AHEAD = 5, SL_THREADS = (SL_ROWS / 16) * 128, SL_SPLIT = NBK / SL_ROWS;
constexpr int SL_A_DOUBLES = SL_ROWS * TILE_K;                     // 512
constexpr int SL_STAGE_DOUBLES = TILE_DOUBLES + SL_A_DOUBLES;      // B tile then A slice: 20 KB
constexpr int SL_SMEM = SL_STAGES * SL_STAGE_DOUBLES * 8 + 256;    // + 2 * SL_STAGES barriers

struct SliceAcc { double c[2][4][2]; };

struct SliceRing {
  double* smem;
  uint64_t *full, *empty;
  int issued, consumed;
  __device__ __forceinline__ void init(double* base) {
    smem = base;
    full = reinterpret_cast<uint64_t*>(base + SL_STAGES * SL_STAGE_DOUBLES);
    empty = full + SL_STAGES;
    issued = consumed = 0;
    if (threadIdx.x == 0) {
      for (int st = 0; st < SL_STAGES; ++st) { mbar_init(full + st, 1); mbar_init(empty + st, SL_THREADS / 32); }
      mbar_fence_init();
    }
    __syncthreads();
  }
  // thread 0: k-tile of B (128 rows) and rows r0 .. r0 + SL_ROWS - 1 of the matching k-tile of A
  __device__ __forceinline__ void produce(const double* a_tile, const double* b_tile, int r0) {
    const int slot = issued % SL_STAGES;
    if (issued >= SL_STAGES) mbar_wait(empty + slot, (unsigned)(((issued / SL_STAGES) - 1) & 1));
    double* st = smem + slot * SL_STAGE_DOUBLES;
    mbar_arrive_expect_tx(full + slot, SL_STAGE_DOUBLES * 8);
    bulk_g2s(st, b_tile, TILE_DOUBLES * 8, full + slot);
#pragma unroll
    for (int g4 = 0; g4 < KG; ++g4)
      bulk_g2s(st + TILE_DOUBLES + g4 * (SL_ROWS * 4), a_tile + g4 * (BM * 4) + r0 * 4, SL_ROWS * 4 * 8, full + slot);
    ++issued;
  }
};

// acc += A[r0 .. r0+31, :] * B^T over KT consecutive k-tiles
__device__ __forceinline__ void slice_mainloop(SliceRing& ring, const double* __restrict__ gA, const double* __restrict__ gB, int KT, int r0,
                                               SliceAcc& acc) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wm = warp >> 2, wn = warp & 3;
  int p = 0;
  if (tid == 0)
    for (; p < SL_AHEAD && p < KT; ++p) ring.produce(gA + (long long)p * TILE_DOUBLES, gB + (long long)p * TILE_DOUBLES, r0);
  for (int kt = 0; kt < KT; ++kt) {
    if (tid == 0 && p < KT) { ring.produce(gA + (long long)p * TILE_DOUBLES, gB + (long long)p * TILE_DOUBLES, r0); ++p; }
    const int slot = ring.consumed % SL_STAGES;
    mbar_wait(ring.full + slot, (unsigned)((ring.consumed / SL_STAGES) & 1));
    const double* sB = ring.smem + slot * SL_STAGE_DOUBLES;
    const double* sA = sB + TILE_DOUBLES;
#pragma unroll
    for (int g4 = 0; g4 < KG; ++g4) {
      double a[2], b[4];
      const double* pa = sA + g4 * (SL_ROWS * 4) + (16 * wm) * 4 + lane;
      const double* pb = sB + g4 * (BN * 4) + (32 * wn) * 4 + lane;
#pragma unroll
      for (int i = 0; i < 2; ++i) a[i] = pa[i * 32];
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) b[jj] = pb[jj * 32];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) dmma884(acc.c[i][jj][0], acc.c[i][jj][1], a[i], b[jj]);
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(ring.empty + slot);
    ++ring.consumed;
  }
  __syncthreads();   // every stage consumed: the ring memory may be reused by the caller's epilogue
}

// rows of accumulator fragment (i, jj) of this lane inside the 32-row slice / columns inside the tile
__device__ __forceinline__ int sl_row(int wm, int i, int lane) { return 16 * wm + 8 * i + (lane >> 2); }

// panel: L21 = A21 * inv(L11)^T and beta_i -= L21 x_j, rows r0 .. r0 + 31 of tile it = j + 1 + blockIdx.y
__global__ void __launch_bounds__(SL_THREADS, 2)
panel_slice_kernel(double* __restrict__ fac, long long fac_stride, int Np, int j, const double* __restrict__ dinv,
                   long long dinv_stride, double* __restrict__ beta, int s0) {
  extern __shared__ __align__(128) double smem[];
  const int s = s0 + blockIdx.z, it = j + 1 + blockIdx.y, r0 = blockIdx.x * SL_ROWS, KPB = NBK / TILE_K;
  double* tile = fac + (long long)s * fac_stride + tile_off(Np / TILE_K, it, j * KPB);
  const double* B = dinv + (long long)s * dinv_stride + (long long)j * NBK * NBK;
  SliceRing ring; ring.init(smem);
  SliceAcc acc;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) acc.c[i][jj][0] = acc.c[i][jj][1] = 0.0;
  pdl_trigger();
  pdl_wait();
  slice_mainloop(ring, tile, B, KPB, r0, acc);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, wm = warp >> 2, wn = warp & 3;
  const double* xj = beta + (long long)s * Np + j * NBK;
  double* red = smem;   // [SL_ROWS][4]
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int row = sl_row(wm, i, lane);
    double part = 0.0;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int col = frag_col(wn, jj, lane);
      *reinterpret_cast<double2*>(tile + elem_off(r0 + row, col)) = make_double2(acc.c[i][jj][0], acc.c[i][jj][1]);
      part += acc.c[i][jj][0] * xj[col] + acc.c[i][jj][1] * xj[col + 1];
    }
    part += __shfl_xor_sync(0xffffffffu, part, 1);
    part += __shfl_xor_sync(0xffffffffu, part, 2);
    if ((lane & 3) == 0) red[row * 4 + wn] = part;
  }
  __syncthreads();
  if (tid < SL_ROWS) {
    double sum = ((red[tid * 4 + 0] + red[tid * 4 + 1]) + red[tid * 4 + 2]) + red[tid * 4 + 3];
    beta[(long long)s * Np + it * NBK + r0 + tid] -= sum;
  }
}

// trailing update: C[it][nt] -= L[it][kb0:kb1] L[nt][kb0:kb1]^T, rows r0 .. r0 + 31 of the tile;
// it = it0 + blockIdx.x / 4, nt = nt0 + blockIdx.y (tiles above the diagonal exit at once)
__global__ void __launch_bounds__(SL_THREADS, 2)
trail_slice_kernel(double* __restrict__ fac, long long fac_stride, int Np, int kb0, int kb1, int it0, int nt0, int s0) {
  extern __shared__ __align__(128) double smem[];
  const int it = it0 + (int)(blockIdx.x / SL_SPLIT), nt = nt0 + blockIdx.y, r0 = (int)(blockIdx.x % SL_SPLIT) * SL_ROWS;
  pdl_trigger();
  if (nt > it) { pdl_wait(); return; }     // (a CTA that left without waiting would let the grid complete before its predecessor)
  const int s = s0 + blockIdx.z, KPB = NBK / TILE_K, KTA = Np / TILE_K;
  double* base = fac + (long long)s * fac_stride;
  const double* A = base + tile_off(KTA, it, kb0 * KPB);
  const double* B = base + tile_off(KTA, nt, kb0 * KPB);
  double* C = base + tile_off(KTA, it, nt * KPB);
  SliceRing ring; ring.init(smem);
  pdl_wait();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wm = warp >> 2, wn = warp & 3;
  // as trail_kernel: acc starts at -C, accumulates +A B^T, and C_new = -acc
  SliceAcc acc;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const double2 v = *reinterpret_cast<const double2*>(C + elem_off(r0 + sl_row(wm, i, lane), frag_col(wn, jj, lane)));
      acc.c[i][jj][0] = -v.x;
      acc.c[i][jj][1] = -v.y;
    }
  slice_mainloop(ring, A, B, (kb1 - kb0) * KPB, r0, acc);
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
      *reinterpret_cast<double2*>(C + elem_off(r0 + sl_row(wm, i, lane), frag_col(wn, jj, lane))) =
          make_double2(-acc.c[i][jj][0], -acc.c[i][jj][1]);
}

// ---- inversion sweep ------------------------------------------------------------------------------
__global__ void place_diag_kernel(double* __restrict__ fac, long long fac_stride, int Np, const double* __restrict__ dinv,
                                  long long dinv_stride, int s0) {
  const int s = s0 + blockIdx.y, j = blockIdx.x;
  double* blk = fac + (long long)s * fac_stride + tile_off(Np / TILE_K, j, j * (NBK / TILE_K));
  const double* di = dinv + (long long)s * dinv_stride + (long long)j * NBK * NBK;
  for (int e = threadIdx.x; e < NBK * NBK; e += blockDim.x) blk[e] = di[e];   // same tiled order on both sides
}

// T = L[it, j] * inv(L_jj), written transposed into the one-row-block tiled matrix tt (128 x Np):
// tt(c, it*128 + row) = T(row, c)
__global__ void __launch_bounds__(THREADS, 1)
inv_step1_kernel(const double* __restrict__ fac, long long fac_stride, int Np, int j, const double* __restrict__ dinvT,
                 long long dinv_stride, double* __restrict__ tt, long long tt_stride, int s0) {
  extern __shared__ __align__(128) double smem[];
  const int s = s0 + blockIdx.z, it = j + 1 + blockIdx.x, KPB = NBK / TILE_K;
  const double* A = fac + (long long)s * fac_stride + tile_off(Np / TILE_K, it, j * KPB);
  const double* B = dinvT + (long long)s * dinv_stride + (long long)j * NBK * NBK;
  Ring ring; ring.init(smem);
  Acc acc; acc.zero();
  mainloop_bulk(ring, A, B, KPB, acc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wm = warp >> 2, wn = warp & 3;
  double* T = tt + (long long)s * tt_stride;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      const int k = it * NBK + frag_row(wm, i, lane), col = frag_col(wn, jj, lane);
      T[elem_off(col, k)] = acc.c[i][jj][0];
      T[elem_off(col + 1, k)] = acc.c[i][jj][1];
    }
}

// X[it, j] = - sum_{k=(j+1)*128}^{(it+1)*128-1} Linv[it, k] * T[k, :]
__global__ void __launch_bounds__(THREADS, 1)
inv_step2_kernel(double* __restrict__ fac, long long fac_stride, int Np, int j, const double* __restrict__ tt,
                 long long tt_stride, int s0) {
  extern __shared__ __align__(128) double smem[];
  // longest rows first: better tail behaviour
  const int n_it = gridDim.x, it = j + n_it - (int)blockIdx.x, KPB = NBK / TILE_K, KTA = Np / TILE_K;
  const int s = s0 + blockIdx.z;
  double* base = fac + (long long)s * fac_stride;
  const double* A = base + tile_off(KTA, it, (j + 1) * KPB);
  const double* B = tt + (long long)s * tt_stride + (long long)(j + 1) * KPB * TILE_DOUBLES;
  double* C = base + tile_off(KTA, it, j * KPB);
  Ring ring; ring.init(smem);
  Acc acc; acc.zero();
  mainloop_bulk(ring, A, B, (it - j) * KPB, acc);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wm = warp >> 2, wn = warp & 3;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
      *reinterpret_cast<double2*>(C + elem_off(frag_row(wm, i, lane), frag_col(wn, jj, lane))) =
          make_double2(-acc.c[i][jj][0], -acc.c[i][jj][1]);
}

// tiled <-> row-major conversion of the N x N leading part (tests, b7_gp_read_factor)
__global__ void untile_kernel(const double* __restrict__ facT, double* __restrict__ out, int Np, int N) {
  const int row = blockIdx.x;
  const double* src = facT + tile_off(Np / TILE_K, row >> 7, 0);
  for (int k = threadIdx.x; k < N; k += blockDim.x) out[(long long)row * N + k] = src[elem_off(row & 127, k)];
}

bool g_attr_done[16] = {false};   // function attributes are per device
int set_attrs(int device) {
  if (g_attr_done[device & 15]) return 0;
  // every kernel of the chain asks for the same (largest) shared-memory carve-out: consecutive kernels with different
  // carve-outs make the SMs reconfigure between launches, which shows up as microseconds of gap in a chain of ~100
  // dependent launches
  auto set = [](const void* fn, int smem) -> cudaError_t {
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  };
  B7_CUDA(set((const void*)diag_kernel, DIAG_SMEM));
  B7_CUDA(set((const void*)panel_kernel, RING_SMEM));
  B7_CUDA(set((const void*)trail_kernel, RING_SMEM));
  B7_CUDA(set((const void*)panel_slice_kernel, SL_SMEM));
  B7_CUDA(set((const void*)trail_slice_kernel, SL_SMEM));
  B7_CUDA(set((const void*)inv_step1_kernel, RING_SMEM));
  B7_CUDA(set((const void*)inv_step2_kernel, RING_SMEM));
  g_attr_done[device & 15] = true;
  return 0;
}

// ---- alpha = L^-T beta ------------------------------------------------------------------------------
// The INT8 posterior path takes the mean from an fp64 dot product k*^T alpha (the arithmetic the oracle uses,
// `Ks @ alpha`) instead of v^T beta through the sliced operands, so alpha is needed once per fit.  Blocked back
// substitution on the factor before it is inverted in place: column sweep from the bottom, one CTA per draw,
//   alpha_ib = inv(L_ib,ib)^T r_ib ;   r[k] -= sum_row L[ib*128 + row][k] alpha_ib[row]   for k < 128 ib.
// Row block ib of L is one contiguous run of tiles; a warp owns a k-group (128 rows x 4 columns = 4 KB), lanes are
// rows, and the 4 column sums come out of a fixed shuffle tree (deterministic).
// FROM_INVERSE: fac already holds L^-1 (the path was switched after the fit, or the factor came from another
// rank): alpha = (L^-1)^T beta, the same row-block primitive without the solve.
constexpr int ALPHA_THREADS = 1024;

template <bool FROM_INVERSE>
__global__ void __launch_bounds__(ALPHA_THREADS, 1)
alpha_kernel(const double* __restrict__ fac, long long fac_stride, int Np, const double* __restrict__ dinvT, long long dinv_stride,
             const double* __restrict__ beta, double* __restrict__ alpha, int s0) {
  extern __shared__ __align__(16) double sm[];
  double* r = sm;            // Np
  double* xa = sm + Np;      // 128
  const int s = s0 + blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, NB = Np / NBK;
  const double* F = fac + (long long)s * fac_stride;
  for (int e = tid; e < Np; e += ALPHA_THREADS) r[e] = FROM_INVERSE ? 0.0 : beta[(long long)s * Np + e];
  __syncthreads();
  for (int step = 0; step < NB; ++step) {
    const int ib = FROM_INVERSE ? step : NB - 1 - step;
    if (tid < NBK) {
      if (FROM_INVERSE) {
        xa[tid] = beta[(long long)s * Np + ib * NBK + tid];
      } else {
        const double* dt = dinvT + (long long)s * dinv_stride + (long long)ib * NBK * NBK;
        double sum = 0.0;
#pragma unroll 4
        for (int q4 = 0; q4 < NBK / 4; ++q4) {
          const double4 m = *reinterpret_cast<const double4*>(dt + (q4 >> 2) * TILE_DOUBLES + (q4 & 3) * (BM * 4) + tid * 4);
          const double* rr = r + ib * NBK + 4 * q4;
          sum = fma(m.x, rr[0], sum); sum = fma(m.y, rr[1], sum); sum = fma(m.z, rr[2], sum); sum = fma(m.w, rr[3], sum);
        }
        xa[tid] = sum;
        alpha[(long long)s * Np + ib * NBK + tid] = sum;
      }
    }
    __syncthreads();
    const double* rowblk = F + tile_off(Np / TILE_K, ib, 0);
    const int n_kg = (FROM_INVERSE ? ib + 1 : ib) * (NBK / 4);       // k-groups of 4 columns left of (or including) the diagonal block
    for (int kg = warp; kg < n_kg; kg += ALPHA_THREADS / 32) {
      const double* p = rowblk + (long long)kg * (BM * 4);
      double4 v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = *reinterpret_cast<const double4*>(p + (lane + 32 * i) * 4);
      double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const double x = xa[lane + 32 * i];
        a0 = fma(v[i].x, x, a0); a1 = fma(v[i].y, x, a1); a2 = fma(v[i].z, x, a2); a3 = fma(v[i].w, x, a3);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a0 += __shfl_xor_sync(0xffffffffu, a0, o); a1 += __shfl_xor_sync(0xffffffffu, a1, o);
        a2 += __shfl_xor_sync(0xffffffffu, a2, o); a3 += __shfl_xor_sync(0xffffffffu, a3, o);
      }
      if (lane == 0) {
        double* out = r + kg * 4;
        if (FROM_INVERSE) { out[0] += a0; out[1] += a1; out[2] += a2; out[3] += a3; }
        else { out[0] -= a0; out[1] -= a1; out[2] -= a2; out[3] -= a3; }
      }
    }
    __syncthreads();
  }
  if (FROM_INVERSE)
    for (int e = tid; e < Np; e += ALPHA_THREADS) alpha[(long long)s * Np + e] = r[e];
}

// B7_POTRF_TRACE=1: an event after every launch of the main stream; b7_launch_potrf then synchronises and prints the time
// between consecutive events by kernel (stderr).  Debugging aid for the single-factor latency chain, off by default.
struct PotrfTrace {
  bool on = false;
  cudaStream_t st = nullptr;
  std::vector<cudaEvent_t> ev;
  std::vector<const char*> tag;
  void mark(const char* name) {
    if (!on) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, st);
    ev.push_back(e);
    tag.push_back(name);
  }
  void dump() {
    if (!on) return;
    cudaStreamSynchronize(st);
    const char* names[] = {"diag", "panel", "trail", "slice", "near", "wait_far", "transpose"};
    double sum[7] = {0, 0, 0, 0, 0, 0, 0};
    int cnt[7] = {0, 0, 0, 0, 0, 0, 0};
    for (size_t i = 1; i < ev.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
      for (int k = 0; k < 7; ++k)
        if (strcmp(tag[i], names[k]) == 0) { sum[k] += ms; ++cnt[k]; }
      if (getenv("B7_POTRF_TRACE") && atoi(getenv("B7_POTRF_TRACE")) > 1) fprintf(stderr, "  %-10s %8.1f us\n", tag[i], ms * 1e3);
    }
    float total = 0.f;
    if (ev.size() > 1) cudaEventElapsedTime(&total, ev.front(), ev.back());
    fprintf(stderr, "potrf trace: total %.1f us;", total * 1e3);
    for (int k = 0; k < 7; ++k)
      if (cnt[k]) fprintf(stderr, " %s %d x %.1f us;", names[k], cnt[k], sum[k] * 1e3 / cnt[k]);
    fprintf(stderr, "\n");
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
  }
};

// One or two factors: every kernel of the chain diag -> panel -> update of the next column is on the critical path of
// the whole fit (32 block columns at N = 4096), and the machine is otherwise empty.  Same operations on every tile in
// the same order as the batched schedule below (results are bit-identical), but
//   * panel and trailing updates run row-sliced (4 CTAs per tile: ~5 us instead of ~20 us per wave);
//   * on the main stream a column step only updates the NEXT column; the other columns of the outer panel get the same
//     update on a side stream while the next diagonal block is factored (they are needed one step later each);
//   * after an outer panel only the first column of the next one gets its k = 512 update on the main stream, the other
//     columns follow on the side stream, everything further right on the far stream as in the batched schedule.
int potrf_latency_enqueue(b7_gp* gp, int s0, int count, int W, bool allow_trace);

// The schedule above is ~100 dependent launches and as many event operations: enqueued one by one the host is not
// always ahead of the GPU and every dependent launch costs microseconds of gap.  A handle that is factorised again with
// the same (first draw, count) -- b7_gp_refit, i.e. every density evaluation of the slice sampler -- captures the
// schedule into a CUDA graph once (all kernel arguments are per-handle constants; the hyper-parameters live in device
// memory) and replays it from then on.  Measured (tools/fit_latency.py, refit ms with / without the graph): N = 2048
// 0.86 / 0.90, N = 4096 2.17 / 2.03, N = 8192 9.64 / 9.01 -- the replay wins while the chain is short and loses once the
// far updates are large (their nodes and the chain's are scheduled on equal terms whatever the node priorities say), so
// the graph is used up to 16 block columns.  B7_POTRF_GRAPH=0 disables it, =1 forces it at every size.
int potrf_latency(b7_gp* gp, int s0, int count, int W) {
  b7_ctx* ctx = gp->ctx;
  static const int graph_env = getenv("B7_POTRF_GRAPH") ? atoi(getenv("B7_POTRF_GRAPH")) : -1;
  const bool graph_ok = graph_env >= 0 ? graph_env != 0 : gp->NB <= 16;
  if (!graph_ok || getenv("B7_POTRF_TRACE")) return potrf_latency_enqueue(gp, s0, count, W, true);
  if (gp->potrf_graph && gp->potrf_graph_s0 == s0 && gp->potrf_graph_count == count) {
    B7_CUDA(cudaGraphLaunch(gp->potrf_graph, ctx->stream));
    b7_count(ctx, gp->potrf_graph_launches);
    return 0;
  }
  if (gp->potrf_calls_s0 == s0 && gp->potrf_calls_count == count) ++gp->potrf_calls;
  else { gp->potrf_calls_s0 = s0; gp->potrf_calls_count = count; gp->potrf_calls = 1; }
  if (gp->potrf_calls < 2) return potrf_latency_enqueue(gp, s0, count, W, false);
  // second call with this key: capture, instantiate, launch
  if (gp->potrf_graph) { cudaGraphExecDestroy(gp->potrf_graph); gp->potrf_graph = nullptr; }
  const int64_t before = ctx->launches;
  cudaGraph_t graph = nullptr;
  B7_CUDA(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
  const int rc = potrf_latency_enqueue(gp, s0, count, W, false);
  const cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
  if (rc != 0 || e != cudaSuccess || graph == nullptr) {
    if (getenv("B7_DEBUG")) fprintf(stderr, "potrf graph: capture failed (rc %d, %s)\n", rc, cudaGetErrorString(e));
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    ctx->launches = before;
    gp->potrf_calls = -(1 << 30);            // do not try again on this handle
    return potrf_latency_enqueue(gp, s0, count, W, false);
  }
  const cudaError_t ei = cudaGraphInstantiate(&gp->potrf_graph, graph, 0);
  cudaGraphDestroy(graph);
  if (ei != cudaSuccess) {
    if (getenv("B7_DEBUG")) fprintf(stderr, "potrf graph: instantiation failed (%s)\n", cudaGetErrorString(ei));
    gp->potrf_graph = nullptr;
    cudaGetLastError();
    ctx->launches = before;
    gp->potrf_calls = -(1 << 30);
    return potrf_latency_enqueue(gp, s0, count, W, false);
  }
  gp->potrf_graph_s0 = s0;
  gp->potrf_graph_count = count;
  gp->potrf_graph_launches = (int)(ctx->launches - before);
  if (getenv("B7_DEBUG")) fprintf(stderr, "potrf graph: %d kernel nodes captured\n", gp->potrf_graph_launches);
  B7_CUDA(cudaGraphLaunch(gp->potrf_graph, ctx->stream));
  return 0;
}

// launch with the programmatic-serialisation attribute (see pdl_wait)
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  // the stream's priority as a launch attribute as well: a captured graph keeps it per kernel node (without it the far
  // update's nodes compete with the chain's on equal terms: N = 8192 9.0 -> 10.0 ms)
  int prio = 0;
  cudaStreamGetPriority(st, &prio);
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributePriority;
  attr[0].val.priority = prio;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 2 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

int potrf_latency_enqueue(b7_gp* gp, int s0, int count, int W, bool allow_trace) {
  b7_ctx* ctx = gp->ctx;
  static const bool pdl = !(getenv("B7_POTRF_PDL") && atoi(getenv("B7_POTRF_PDL")) == 0);
  const int Np = gp->Np, NB = gp->NB, SPT = NBK / SL_ROWS;
  const long long fs = (long long)Np * Np, ds = (long long)NB * NBK * NBK;
  cudaStream_t sa = ctx->stream, sb = ctx->stream2, sc = ctx->stream3;
  bool far_pending = false, side_pending = false, near1_pending = false;
  PotrfTrace trace;
  trace.on = allow_trace && getenv("B7_POTRF_TRACE") != nullptr;
  trace.st = sa;
  trace.mark("start");
  // kernels of the main stream follow their predecessor programmatically; the side and far streams launch normally
  auto trail = [&](cudaStream_t st, int kb0, int kb1, int it0, int n_it, int nt0, int n_nt) {
    launch_pdl(trail_slice_kernel, dim3(n_it * SPT, n_nt, count), dim3(SL_THREADS), SL_SMEM, st, pdl && st == sa, gp->fac, fs, Np, kb0, kb1, it0, nt0, s0);
    b7_count(ctx);
  };
  for (int J = 0; J < NB; J += W) {
    const int Jend = J + W < NB ? J + W : NB;
    for (int j = J; j < Jend; ++j) {
      launch_pdl(diag_kernel, dim3(count), dim3(DIAG_THREADS), DIAG_SMEM, sa, pdl && j > 0, gp->fac, fs, Np, j, gp->dinv, ds, gp->beta, gp->logdet,
                 gp->info, s0);
      b7_count(ctx);
      trace.mark("diag");
      const int rem = NB - 1 - j;
      if (rem > 0) {
        launch_pdl(panel_slice_kernel, dim3(SPT, rem, count), dim3(SL_THREADS), SL_SMEM, sa, pdl, gp->fac, fs, Np, j, (const double*)gp->dinv, ds, gp->beta, s0);
        b7_count(ctx);
        trace.mark("panel");
      }
      if (j + 1 < Jend) {
        // column j + 1 <- column j, after whatever the side stream still had to do to that column
        if (near1_pending) { B7_CUDA(cudaStreamWaitEvent(sa, ctx->evS1, 0)); near1_pending = false; }
        // (at the first step of a panel the side stream may still be busy with the k = 128 W update of columns >= J + 2:
        //  not needed here, and ordered before this step's side launch by the stream itself)
        if (side_pending && j > J) { B7_CUDA(cudaStreamWaitEvent(sa, ctx->evS, 0)); side_pending = false; }
        trail(sa, j, j + 1, j + 1, rem, j + 1, 1);
        trace.mark("trail");
        if (j + 2 < Jend) {   // columns j + 2 .. Jend - 1 <- column j on the side stream (rows from j + 2: the lower tiles)
          B7_CUDA(cudaEventRecord(ctx->evA, sa));
          B7_CUDA(cudaStreamWaitEvent(sc, ctx->evA, 0));
          trail(sc, j, j + 1, j + 2, rem - 1, j + 2, Jend - 2 - j);
          B7_CUDA(cudaEventRecord(ctx->evS, sc));
          side_pending = true;
        }
      }
    }
    if (Jend >= NB) break;
    const int near_end = Jend + W < NB ? Jend + W : NB;
    if (side_pending) { B7_CUDA(cudaStreamWaitEvent(sa, ctx->evS, 0)); side_pending = false; }
    if (far_pending) B7_CUDA(cudaStreamWaitEvent(sa, ctx->evB, 0));     // it touched the next panel's tiles
    trace.mark("wait_far");
    trail(sa, J, Jend, Jend, NB - Jend, Jend, 1);                        // first column of the next panel, k = 128 W
    trace.mark("near");
    B7_CUDA(cudaEventRecord(ctx->evA, sa));
    if (near_end - Jend > 1) {
      B7_CUDA(cudaStreamWaitEvent(sc, ctx->evA, 0));
      trail(sc, J, Jend, Jend + 1, NB - Jend - 1, Jend + 1, 1);         // its second column: needed one step later
      B7_CUDA(cudaEventRecord(ctx->evS1, sc));
      near1_pending = true;
      if (near_end - Jend > 2) {
        trail(sc, J, Jend, Jend + 2, NB - Jend - 2, Jend + 2, near_end - Jend - 2);
        B7_CUDA(cudaEventRecord(ctx->evS, sc));
        side_pending = true;
      }
    }
    if (near_end < NB) {
      B7_CUDA(cudaStreamWaitEvent(sb, ctx->evA, 0));
      trail(sb, J, Jend, near_end, NB - near_end, near_end, NB - near_end);
      B7_CUDA(cudaEventRecord(ctx->evB, sb));
      far_pending = true;
    }
  }
  if (far_pending) B7_CUDA(cudaStreamWaitEvent(sa, ctx->evB, 0));
  if (side_pending) B7_CUDA(cudaStreamWaitEvent(sa, ctx->evS, 0));
  if (near1_pending) B7_CUDA(cudaStreamWaitEvent(sa, ctx->evS1, 0));
  trace.mark("wait_far");
  dinv_transpose_kernel<<<dim3(NB, count), 512, 0, sa>>>(gp->dinv, gp->dinvT, ds, s0);
  b7_count(ctx);
  trace.mark("transpose");
  trace.dump();
  B7_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace

int b7_launch_potrf(b7_gp* gp, int s0, int count) {
  b7_ctx* ctx = gp->ctx;
  B7_CHECK(set_attrs(ctx->device));
  const int Np = gp->Np, NB = gp->NB;
  const long long fs = (long long)Np * Np, ds = (long long)NB * NBK * NBK;
  static const int W_env = getenv("B7_POTRF_W") ? atoi(getenv("B7_POTRF_W")) : 0;
  const int W = W_env > 0 ? W_env : 4;   // outer panel = 4 blocks (512 columns)
  // one or two factors: the latency-oriented schedule with row-sliced kernels (bit-identical results)
  static const int slice_env = getenv("B7_POTRF_SLICE") ? atoi(getenv("B7_POTRF_SLICE")) : -1;
  // ... and small batches of small factors, where the machine is as empty (tools/refit_vs_s.py, refit ms batched -> latency
  // schedule: N = 512, 8 draws 0.385 -> 0.273; N = 2048, 4 draws 1.68 -> 1.15, 8 draws 2.09 -> 1.72, 16 draws 2.78 -> 2.94;
  // N = 4096, 4 draws 4.46 -> 4.83): up to S NB^2 = 2048 tile columns.  The test looks at the handle's total number of draws,
  // like the INT8 / FP64 choice below (which starts at 4096), so a sharded fit and the one-GPU fit take the same arithmetic.
  const bool small_batch = (long long)gp->S * NB * NB <= 2048;
  if (slice_env >= 0 ? slice_env != 0 : (count <= 2 || small_batch)) return potrf_latency(gp, s0, count, W);
  cudaStream_t sa = ctx->stream, sb = ctx->stream2;
  bool far_pending = false;
  PotrfTrace trace;
  trace.on = getenv("B7_POTRF_TRACE") != nullptr;
  trace.st = sa;
  trace.mark("start");
  // INT8 path (potrf_i8.cu): the panel rows are sliced once per outer panel into one of two scratch sets (the far
  // update of panel J still reads its set while panel J + W is sliced)
  // (batched fits only: a single factor is a latency chain that the extra slicing launch makes longer; measured
  // at N = 4096: S = 32 26.7 -> 17.7 ms, S = 1 4.1 -> 4.8 ms)
  // refit latency, ms, int8 / fp64 updates: N = 4096 S = 4 5.7 / 5.9, S = 8 7.4 / 8.8, S = 16 11.2 / 15.3;
  // N = 2048 S = 4 2.5 / 2.25, S = 16 3.5 / 3.5, S = 32 4.3 / 4.8 -> needs count * NB^2 >= 4096
  // The choice looks at the handle's total number of draws, not at how many of them this call factorises: a sharded fit
  // (each GPU factorises S / G draws) then uses the same arithmetic as the one-GPU fit and stays bit-identical to it.
  const int batch = gp->S;
  const bool i8 = ctx->use_i8 && ctx->potrf_i8 && batch >= 4 && (long long)batch * NB * NB >= 4096 && NB > W && Np <= B7_I8_MAX_NP;
  int8_t* pS[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  double* pSig[2] = {nullptr, nullptr};
  const size_t p_stride = i8 ? b7_i8_panel_bytes(Np, W) : 0;
  if (i8)
    for (int b = 0; b < 2; ++b) {
      B7_CHECK(b7_pool_alloc(ctx, (void**)&pS[b][0], p_stride * count));
      B7_CHECK(b7_pool_alloc(ctx, (void**)&pS[b][1], p_stride * count));
      B7_CHECK(b7_pool_alloc(ctx, (void**)&pSig[b], sizeof(double) * (size_t)Np * count));
    }
  int set = 0;
  for (int J = 0; J < NB; J += W) {
    const int Jend = J + W < NB ? J + W : NB;
    // --- the panel's own columns: latency-bound chain on the main stream ---
    for (int j = J; j < Jend; ++j) {
      diag_kernel<<<count, DIAG_THREADS, DIAG_SMEM, sa>>>(gp->fac, fs, Np, j, gp->dinv, ds, gp->beta, gp->logdet, gp->info, s0);
      b7_count(ctx);
      trace.mark("diag");
      const int rem = NB - 1 - j;
      if (rem > 0) {
        panel_kernel<<<dim3(rem, 1, count), THREADS, RING_SMEM, sa>>>(gp->fac, fs, Np, j, gp->dinv, ds, gp->beta, s0);
        b7_count(ctx);
        trace.mark("panel");
      }
      if (Jend - 1 - j > 0) {   // columns j+1 .. Jend-1 of the outer panel, all rows below
        trail_kernel<<<dim3(rem, Jend - 1 - j, count), THREADS, RING_SMEM, sa>>>(gp->fac, fs, Np, j, j + 1, j + 1, j + 1, s0);
        b7_count(ctx);
        trace.mark("trail");
      }
    }
    if (Jend >= NB) break;
    // --- update by this panel (k = 512).  "near": the next panel's columns, needed at once, main stream
    //     (after the previous far update, which touched the same tiles).  "far": everything to the right of
    //     the next panel, on the second stream, overlapping the next panel's chain of small kernels. ---
    const int near_end = Jend + W < NB ? Jend + W : NB;
    if (i8) B7_CHECK(b7_i8_panel_slice(ctx, sa, gp->fac, Np, J, Jend, Jend, pS[set][0], pS[set][1], p_stride, pSig[set], s0, count));
    if (far_pending) B7_CUDA(cudaStreamWaitEvent(sa, ctx->evB, 0));
    trace.mark("wait_far");
    if (i8) {
      B7_CHECK(b7_i8_trail(ctx, sa, gp->fac, Np, pS[set][0], pS[set][1], p_stride, pSig[set], J, Jend, Jend, Jend, NB - Jend, Jend,
                           near_end - Jend, s0, count));
    } else {
      trail_kernel<<<dim3(NB - Jend, near_end - Jend, count), THREADS, RING_SMEM, sa>>>(gp->fac, fs, Np, J, Jend, Jend, Jend, s0);
      b7_count(ctx);
    }
    trace.mark("near");
    if (near_end < NB) {
      B7_CUDA(cudaEventRecord(ctx->evA, sa));
      B7_CUDA(cudaStreamWaitEvent(sb, ctx->evA, 0));
      if (i8) {
        B7_CHECK(b7_i8_trail(ctx, sb, gp->fac, Np, pS[set][0], pS[set][1], p_stride, pSig[set], J, Jend, Jend, near_end, NB - near_end,
                             near_end, NB - near_end, s0, count));
      } else {
        trail_kernel<<<dim3(NB - near_end, NB - near_end, count), THREADS, RING_SMEM, sb>>>(gp->fac, fs, Np, J, Jend, near_end, near_end, s0);
        b7_count(ctx);
      }
      B7_CUDA(cudaEventRecord(ctx->evB, sb));
      far_pending = true;
    }
    set ^= 1;
  }
  if (far_pending) B7_CUDA(cudaStreamWaitEvent(sa, ctx->evB, 0));
  trace.mark("wait_far");
  dinv_transpose_kernel<<<dim3(NB, count), 512, 0, sa>>>(gp->dinv, gp->dinvT, ds, s0);
  b7_count(ctx);
  trace.mark("transpose");
  trace.dump();
  if (i8)
    for (int b = 0; b < 2; ++b) {
      b7_pool_free(ctx, pS[b][0]);
      b7_pool_free(ctx, pS[b][1]);
      b7_pool_free(ctx, pSig[b]);
    }
  B7_CUDA(cudaGetLastError());
  return 0;
}

// alpha = L^-T beta for draws [s0, s0 + count): from L (before the inversion) or from L^-1 (from_inverse)
int b7_launch_alpha(b7_gp* gp, int s0, int count, bool from_inverse) {
  b7_ctx* ctx = gp->ctx;
  const int Np = gp->Np;
  const size_t smem = (size_t)(Np + NBK) * sizeof(double);
  if (smem > 200 * 1024) { b7_set_error("alpha: %d observations exceed the shared-memory sweep", Np); return B7_ERR_ARG; }
  static bool attr[16][2] = {{false}};
  if (!attr[ctx->device & 15][from_inverse]) {
    if (from_inverse) B7_CUDA(cudaFuncSetAttribute(alpha_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    else B7_CUDA(cudaFuncSetAttribute(alpha_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr[ctx->device & 15][from_inverse] = true;
  }
  const long long fs = (long long)Np * Np, ds = (long long)gp->NB * NBK * NBK;
  if (from_inverse) alpha_kernel<true><<<count, ALPHA_THREADS, smem, ctx->stream>>>(gp->fac, fs, Np, gp->dinvT, ds, gp->beta, gp->alpha, s0);
  else alpha_kernel<false><<<count, ALPHA_THREADS, smem, ctx->stream>>>(gp->fac, fs, Np, gp->dinvT, ds, gp->beta, gp->alpha, s0);
  b7_count(ctx);
  B7_CUDA(cudaGetLastError());
  return 0;
}

int b7_launch_untile(b7_ctx* ctx, const double* facT, double* out, int Np, int N) {
  untile_kernel<<<N, 256, 0, ctx->stream>>>(facT, out, Np, N);
  b7_count(ctx);
  B7_CUDA(cudaGetLastError());
  return 0;
}

int b7_launch_trtri(b7_gp* gp, int s0, int count) {
  b7_ctx* ctx = gp->ctx;
  B7_CHECK(set_attrs(ctx->device));
  const int Np = gp->Np, NB = gp->NB;
  const long long fs = (long long)Np * Np, ds = (long long)NB * NBK * NBK, ts = (long long)NBK * Np;
  place_diag_kernel<<<dim3(NB, count), 256, 0, ctx->stream>>>(gp->fac, fs, Np, gp->dinv, ds, s0);
  b7_count(ctx);
  // INT8 path: block-recursive inversion with static operands per level (trtri_i8.cu)
  if (ctx->use_i8 && ctx->trtri_i8 && Np <= B7_I8_MAX_NP) return b7_launch_trtri_i8(gp, s0, count);
  for (int j = NB - 2; j >= 0; --j) {
    const int rem = NB - 1 - j;
    inv_step1_kernel<<<dim3(rem, 1, count), THREADS, RING_SMEM, ctx->stream>>>(gp->fac, fs, Np, j, gp->dinvT, ds, gp->tt, ts, s0);
    inv_step2_kernel<<<dim3(rem, 1, count), THREADS, RING_SMEM, ctx->stream>>>(gp->fac, fs, Np, j, gp->tt, ts, s0);
    b7_count(ctx, 2);
  }
  B7_CUDA(cudaGetLastError());
  return 0;
}

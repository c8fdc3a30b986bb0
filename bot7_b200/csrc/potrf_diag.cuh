// Diagonal-block factorisation of the blocked Cholesky (potrf.cu: diag_kernel): potf2 + inverse of one 128 x 128 block
// in shared memory, x = inv(L) r and the log-determinant.  Shared with the slice-step kernel (slice_step.cu), which
// factors fits of up to 128 observations (one block) with these operations in this order, so that its log likelihoods
// carry the bits of b7_gp_refit.
#pragma once
#include "b7_internal.h"
#include "gemm_tile.cuh"

#ifndef DIAG_STAMP
#define DIAG_STAMP(i) do { } while (0)
#endif

using namespace b7g;

namespace {

constexpr int NBK = B7_NB;          // 128
constexpr int DIAG_THREADS = 512;
constexpr int DIAG_WARPS = DIAG_THREADS / 32;
constexpr int DLD = 132;            // 132 = 4 mod 16: DMMA fragment loads (row- and column-wise) are conflict free
constexpr int SB = 16;              // sub-block width inside the 128 block
constexpr int DSLD = 20;            // leading dimension of the 16x16 sub-block inverses
constexpr int TLD = 68;             // scratch of the recursive inversion (64 x 68)
// shared: M[128][132] | DS[8][16][20] | T[64][68] | pivs,invs,rj,lg [4][128]
constexpr int DIAG_SMEM = (NBK * DLD + 8 * SB * DSLD + 64 * TLD + 4 * NBK) * 8;

// one 8x8 accumulator fragment: c += sign * A[m.., k0..k1) * op(B);  A row-major (k contiguous).
// NN = false: B is [n][k] row-major (C = A B^T);  NN = true: B is [k][n] row-major (C = A B).
template <bool NN>
__device__ __forceinline__ void frag_mac(double& c0, double& c1, const double* __restrict__ A, int lda,
                                         const double* __restrict__ B, int ldb, int k_begin, int k_end, double sign, int lane) {
  const int r = lane >> 2, c = lane & 3;
#pragma unroll 2
  for (int k = k_begin; k < k_end; k += 4) {     // every caller's k range is a multiple of 8
    const double a = sign * A[r * lda + k + c];
    const double b = NN ? B[(k + c) * ldb + r] : B[r * ldb + k + c];
    dmma884(c0, c1, a, b);
  }
}

// ---- diagonal block: potf2 + inverse + x_j + logdet + info -------------------------------------
// One CTA per draw; the block lives in shared memory (M, row-major, leading dimension 132).  The block column count
// times the duration of this kernel is the floor of a single-factor fit, so it is organised around its dependent chain:
//   * 16-wide sub-blocks.  Warp 0 ("chain") factors the 16x16 diagonal piece in registers: lane = row, the column is
//     broadcast by shuffles, every lane keeps its own copy of the running diagonal (no pivot broadcast), and the
//     reciprocal square root is a MUFU.RSQ64H seed + one cubic step with the scaling of the column folded in
//     (5 dependent FP64 operations per column; tools/lat_probe.cu: DFMA 8.3, SHFL 26, seed 19 cycles).
//   * lanes 16..31 of the chain warp carry the identity below the piece: the same eliminations turn [A; I] into
//     [L; L^-T], so the inverse of the piece costs no instruction of its own.
//   * look-ahead: the chain warp itself forms the 16 rows of the sub-panel and the 3 fragments of the trailing update
//     that the next piece needs and goes on factoring; warps 1..15 do the rest of the sub-panel
//     (L21 = A21 inv(L11)^T) and of the trailing update (A22 -= L21 L21^T) as DMMA fragment products behind it and
//     write the finished 16 columns of L to global memory.  Named barriers: S1 = "piece inverse and the chain's rows
//     are ready" (chain arrives, the others wait), U = between sub-panel and trailing update (warps 1..15),
//     S2 = "trailing update done" (the others arrive, the chain waits before it touches the next rows).
//   * the 128x128 inverse is assembled by recursive doubling ([[A,0],[B,C]]^-1 = [[A^-1,0],[-C^-1 B A^-1, C^-1]])
//     for h = 16, 32, 64 as fragment products, in place, fragments dealt so that every warp gets the same k length.
// History (tools/diag_probe.cu, cycles): 152 k with a lane-0 branch per column, float seed + 3 Newton steps, a separate
// inverse of the piece and no look-ahead (factor 79 k, inverse 18 k, updates 17 k, doubling 18 k, I/O 16 k).
constexpr int BAR_S1 = 1, BAR_U = 2, BAR_S2 = 3;
constexpr int UPD_THREADS = (DIAG_WARPS - DIAG_WARPS / 4) * 32;   // warps with (warp & 3) != 0
__device__ __forceinline__ void nbar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void nbar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ double rsq_seed(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  return y;
}

__device__ __forceinline__ void fence_cta() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }

// sub-panel of row group g (8 rows from i0 + 8 g): L21 = A21 * inv(L11)^T, all 16 columns, in place
__device__ __forceinline__ void diag_subpanel(double* M, const double* DSp, int i0, int j0, int g, int lane) {
  const int r = lane >> 2, c = lane & 3;
  double* Arow = M + (i0 + 8 * g) * DLD + j0;
  double a4[4];
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) a4[k4] = Arow[r * DLD + 4 * k4 + c];
  double c00 = 0, c01 = 0, c10 = 0, c11 = 0;
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) {
    dmma884(c00, c01, a4[k4], DSp[r * DSLD + 4 * k4 + c]);
    dmma884(c10, c11, a4[k4], DSp[(8 + r) * DSLD + 4 * k4 + c]);
  }
  __syncwarp();
  *reinterpret_cast<double2*>(Arow + r * DLD + 2 * c) = make_double2(c00, c01);
  *reinterpret_cast<double2*>(Arow + r * DLD + 8 + 2 * c) = make_double2(c10, c11);
}

// the chain warp's look-ahead: row groups 0 and 1 of the sub-panel with their four accumulator chains interleaved ...
__device__ __forceinline__ void diag_subpanel_pair(double* M, const double* DSp, int i0, int j0, int lane) {
  const int r = lane >> 2, c = lane & 3;
  double* Arow = M + i0 * DLD + j0;
  double a0[4], a1[4], b0[4], b1[4];
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) {
    a0[k4] = Arow[r * DLD + 4 * k4 + c];
    a1[k4] = Arow[(8 + r) * DLD + 4 * k4 + c];
    b0[k4] = DSp[r * DSLD + 4 * k4 + c];
    b1[k4] = DSp[(8 + r) * DSLD + 4 * k4 + c];
  }
  double c00 = 0, c01 = 0, c10 = 0, c11 = 0, e00 = 0, e01 = 0, e10 = 0, e11 = 0;
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) {
    dmma884(c00, c01, a0[k4], b0[k4]);
    dmma884(c10, c11, a0[k4], b1[k4]);
    dmma884(e00, e01, a1[k4], b0[k4]);
    dmma884(e10, e11, a1[k4], b1[k4]);
  }
  __syncwarp();
  *reinterpret_cast<double2*>(Arow + r * DLD + 2 * c) = make_double2(c00, c01);
  *reinterpret_cast<double2*>(Arow + r * DLD + 8 + 2 * c) = make_double2(c10, c11);
  *reinterpret_cast<double2*>(Arow + (8 + r) * DLD + 2 * c) = make_double2(e00, e01);
  *reinterpret_cast<double2*>(Arow + (8 + r) * DLD + 8 + 2 * c) = make_double2(e10, e11);
}

// ... and the three fragments (0,0), (1,0), (1,1) of the trailing update, i.e. the next 16x16 piece
__device__ __forceinline__ void diag_trail_next_piece(double* M, int i0, int j0, int lane) {
  const int r = lane >> 2, c = lane & 3;
  const double* L0 = M + i0 * DLD + j0;
  double a0[4], a1[4];
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) {
    a0[k4] = L0[r * DLD + 4 * k4 + c];
    a1[k4] = L0[(8 + r) * DLD + 4 * k4 + c];
  }
  double2* p00 = reinterpret_cast<double2*>(M + (i0 + r) * DLD + i0 + 2 * c);
  double2* p10 = reinterpret_cast<double2*>(M + (i0 + 8 + r) * DLD + i0 + 2 * c);
  double2* p11 = reinterpret_cast<double2*>(M + (i0 + 8 + r) * DLD + i0 + 8 + 2 * c);
  double2 v00 = *p00, v10 = *p10, v11 = *p11;
#pragma unroll
  for (int k4 = 0; k4 < 4; ++k4) {
    dmma884(v00.x, v00.y, -a0[k4], a0[k4]);
    dmma884(v10.x, v10.y, -a1[k4], a0[k4]);
    dmma884(v11.x, v11.y, -a1[k4], a1[k4]);
  }
  *p00 = v00; *p10 = v10; *p11 = v11;
}

// trailing fragment (gi, gk): C -= L21[gi] L21[gk]^T over the 16 columns from j0
__device__ __forceinline__ void diag_trail_frag(double* M, int i0, int j0, int gi, int gk, int lane) {
  const int r = lane >> 2, c = lane & 3;
  double2* cp = reinterpret_cast<double2*>(M + (i0 + 8 * gi + r) * DLD + i0 + 8 * gk + 2 * c);
  double2 cv = *cp;
  frag_mac<false>(cv.x, cv.y, M + (i0 + 8 * gi) * DLD + j0, DLD, M + (i0 + 8 * gk) * DLD + j0, DLD, 0, SB, -1.0, lane);
  *cp = cv;
}

// one k-tile (16 columns from 16 kt, all 128 rows) of the block back to global memory in tiled order, upper part zero;
// a thread moves 16 bytes, consecutive threads consecutive addresses
__device__ __forceinline__ void diag_store_tile(double* __restrict__ blk, const double* M, int kt, int t, int nthreads) {
  for (int u = t; u < NBK * 8; u += nthreads) {          // u = (g4 * 128 + row) * 2 + half
    const int i = (u >> 1) & 127, k0 = kt * TILE_K + (u >> 8) * 4 + (u & 1) * 2;
    const double2 v = *reinterpret_cast<const double2*>(M + i * DLD + k0);
    *reinterpret_cast<double2*>(blk + kt * TILE_DOUBLES + u * 2) = make_double2(k0 <= i ? v.x : 0.0, k0 + 1 <= i ? v.y : 0.0);
  }
}

// Factor the block held in M (lower triangle, zeros above) in place and replace it by the inverse of its factor; info
// (first bad pivot, 1-based from column 128 j) goes to *s_info and log L_ii to lg.  kStore: the columns of L are also
// written to the block's tiles `blk` in global memory as they are finished.  All DIAG_THREADS threads of the CTA.
template <bool kStore>
__device__ __forceinline__ void diag_factor_invert(double* sm, int* s_info, double* __restrict__ blk, int j) {
  double* M = sm;
  double* DS = M + NBK * DLD;
  double* T = DS + 8 * SB * DSLD;
  double* pivs = T + 64 * TLD;
  double* invs = pivs + NBK;
  double* lg = invs + 2 * NBK;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r = lane >> 2, c = lane & 3;
  if (warp == 0) {
    // ---- chain warp ----
    const bool is_row = lane < SB;
    const int li = lane & (SB - 1);
    int my_info = 0;
    for (int p = 0; p < NBK / SB; ++p) {
      const int j0 = p * SB, i0 = j0 + SB;
      double a[SB], d[SB];
#pragma unroll
      for (int k = 0; k < SB; ++k) {
        a[k] = is_row ? M[(j0 + li) * DLD + j0 + k] : (k == li ? 1.0 : 0.0);
        d[k] = M[(j0 + k) * DLD + j0 + k];
      }
      double mypiv = 1.0, myinv = 1.0;
#pragma unroll
      for (int q = 0; q < SB; ++q) {
        // inv = piv^-1/2: y (1 + e/2 + 3 e^2/8) with e = 1 - piv y^2 (|e| < 2^-19 from the seed: truncation below 2^-58);
        // my = a_q inv with the product by a_q folded into the correction
        const double piv = d[q];
        const double y = rsq_seed(piv);
        const double ay = a[q] * y, t = y * y;
        const double e = fma(-piv, t, 1.0);
        const double u = fma(e, 0.375, 0.5);
        const double my = fma(u, ay * e, ay);
        const double inv = fma(u, y * e, y);
        if (lane == q) { mypiv = piv; myinv = inv; }
#pragma unroll
        for (int k = 0; k < SB; ++k) {      // constant trip count: keeps a[], d[] in registers
          if (k > q) {
            // entries above the diagonal (lane < k <= 15) pick up values that are never read
            const double lk = __shfl_sync(0xffffffffu, my, k);
            a[k] = fma(-my, lk, a[k]);
            d[k] = fma(-lk, lk, d[k]);
          }
        }
        a[q] = my;
      }
      // LAPACK info: first pivot that is not positive -- or whose reciprocal root is not a finite positive number
      const unsigned bad = __ballot_sync(0xffffffffu, is_row && (!(mypiv > 0.0) || !(myinv > 0.0) || myinv > 1.79e308));
      if (bad != 0u && my_info == 0) my_info = j * NBK + j0 + __ffs((int)bad);
      if (is_row) {
#pragma unroll
        for (int k = 0; k < SB; k += 2)
          *reinterpret_cast<double2*>(M + (j0 + lane) * DLD + j0 + k) = make_double2(k <= lane ? a[k] : 0.0, k + 1 <= lane ? a[k + 1] : 0.0);
        pivs[j0 + lane] = mypiv;
        invs[j0 + lane] = myinv;
      } else {
        // lane 16 + col holds column col of the inverse: a[row] = X[row][col] (zero above the diagonal)
#pragma unroll
        for (int i = 0; i < SB; ++i) DS[(p * SB + i) * DSLD + li] = a[i];
      }
      __syncwarp();
      DIAG_STAMP(2 + 3 * p);
      if (p < NBK / SB - 1) {
        if (p >= 1) nbar_sync(BAR_S2, 32 + UPD_THREADS);      // trailing update p - 1 is complete
        DIAG_STAMP(3 + 3 * p);
        diag_subpanel_pair(M, DS + p * SB * DSLD, i0, j0, lane);
        if (p < NBK / SB - 2) {
          fence_cta();
          nbar_arrive(BAR_S1, 32 + UPD_THREADS);
        }
        __syncwarp();
        diag_trail_next_piece(M, i0, j0, lane);
        __syncwarp();
        DIAG_STAMP(4 + 3 * p);
      }
    }
    if (lane == 0) *s_info = my_info;
  } else if ((warp & 3) != 0) {
    // ---- update warps: sub-blocks 0..5 (the chain's look-ahead covers all of sub-block 6).  Warps 4, 8 and 12 sit out:
    //      they would share the chain warp's scheduler and FP64 pipe (a DFMA of the chain queued behind their DMMAs:
    //      5.5 k instead of 2.9 k cycles per piece) ----
    const int uw = warp - 1 - (warp >> 2), ut = uw * 32 + lane;
    constexpr int UW = UPD_THREADS / 32;
    for (int p = 0; p < NBK / SB - 2; ++p) {
      const int j0 = p * SB, i0 = j0 + SB, G = (NBK - i0) / 8;
      nbar_sync(BAR_S1, 32 + UPD_THREADS);
      if (ut < SB) lg[j0 + ut] = log(pivs[j0 + ut] * invs[j0 + ut]);
      for (int g = 2 + uw; g < G; g += UW) diag_subpanel(M, DS + p * SB * DSLD, i0, j0, g, lane);
      nbar_sync(BAR_U, UPD_THREADS);
      const int n_frag = G * (G + 1) / 2;
      int gi = 2, rem = uw;                 // fragment 3 + uw in the order (gi, gk <= gi); fragments 0..2 are the chain's
      for (int f = 3 + uw; f < n_frag; f += UW) {
        while (rem > gi) { rem -= gi + 1; ++gi; }
        diag_trail_frag(M, i0, j0, gi, rem, lane);
        rem += UW;
      }
      fence_cta();
      nbar_arrive(BAR_S2, 32 + UPD_THREADS);
      if (kStore) diag_store_tile(blk, M, p, ut, UPD_THREADS);          // columns j0 .. j0 + 15 are final
    }
  }
  __syncthreads();
  DIAG_STAMP(26);
  if (kStore) {
    diag_store_tile(blk, M, NBK / SB - 2, tid, DIAG_THREADS);
    diag_store_tile(blk, M, NBK / SB - 1, tid, DIAG_THREADS);
  }
  if (tid >= NBK - 2 * SB && tid < NBK) lg[tid] = log(pivs[tid] * invs[tid]);
  __syncthreads();
  // ---- inverse, in place: the 16x16 pieces first, then recursive doubling ----
  for (int e = tid; e < NBK * SB; e += DIAG_THREADS) {
    const int i = e >> 4, k = e & 15;
    M[i * DLD + (i & ~15) + k] = DS[i * DSLD + k];       // includes the zero upper part of the piece
  }
  __syncthreads();
  DIAG_STAMP(27);
  for (int h = SB; h < NBK; h <<= 1) {
    // fragment costs are (k length) h/8 - fn in the first phase and fi + 1 in the second: a warp takes that index from
    // both ends of the range so that every warp has the same total (h / 16 fragments per warp and phase)
    const int fpr = h / 8, wpp = DIAG_WARPS / (NBK / (2 * h));     // fragments per row; warps per pair: 4, 8, 16
    const int t = warp / wpp, wl = warp % wpp, base = 2 * h * t;
    const int half = fpr / 2, lo = wl % half, ypw = wpp / half;     // half = 1, 2, 4; ypw = 4
    // T = B * A^-1   (A^-1 lower triangular: k >= column fragment start)
    for (int fi = wl / half; fi < fpr; fi += ypw)
      for (int m = 0; m < 2; ++m) {
        const int fn = m == 0 ? lo : fpr - 1 - lo;
        double c0 = 0.0, c1 = 0.0;
        frag_mac<true>(c0, c1, M + (base + h + 8 * fi) * DLD + base, DLD, M + base * DLD + base + 8 * fn, DLD, 8 * fn, h, 1.0, lane);
        *reinterpret_cast<double2*>(T + (t * h + 8 * fi + r) * TLD + 8 * fn + 2 * c) = make_double2(c0, c1);
      }
    __syncthreads();
    DIAG_STAMP(h == 16 ? 28 : h == 32 ? 30 : 32);
    // X21 = -C^-1 * T  (C^-1 lower triangular: k < row fragment end)
    for (int fn = wl / half; fn < fpr; fn += ypw)
      for (int m = 0; m < 2; ++m) {
        const int fi = m == 0 ? lo : fpr - 1 - lo;
        double c0 = 0.0, c1 = 0.0;
        frag_mac<true>(c0, c1, M + (base + h + 8 * fi) * DLD + base + h, DLD, T + (t * h) * TLD + 8 * fn, TLD, 0, 8 * fi + 8, -1.0, lane);
        *reinterpret_cast<double2*>(M + (base + h + 8 * fi + r) * DLD + base + 8 * fn + 2 * c) = make_double2(c0, c1);
      }
    __syncthreads();
    DIAG_STAMP(h == 16 ? 29 : h == 32 ? 31 : 33);
  }
}

// x = inv(L) r from the inverse in M: 4 threads per row (row = tid / 4), k interleaved, fixed shuffle tree; the row's
// value is returned to the thread with tid % 4 == 0
__device__ __forceinline__ double diag_solve(const double* M, const double* rj, int tid) {
  const int row = tid >> 2, part = tid & 3;
  double xv = 0.0;
  for (int k = part; k <= row; k += 4) xv = fma(M[row * DLD + k], rj[k], xv);
  xv += __shfl_xor_sync(0xffffffffu, xv, 1);
  xv += __shfl_xor_sync(0xffffffffu, xv, 2);
  return xv;
}

// sum of the 128 log L_ii of the block, in row order
__device__ __forceinline__ double diag_logdet(const double* lg) {
  double ld_acc = 0.0;
  for (int q = 0; q < NBK; ++q) ld_acc += lg[q];
  return ld_acc;
}

}  // namespace

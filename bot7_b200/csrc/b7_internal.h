// Internal declarations shared by the translation units of libbot7_b200.so (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/bot7_b200.h"

#define B7_NB 128            // Cholesky / TRMM block size == GEMM tile edge
#define B7_MAX_DIMS 40       // grids/sobol.lua:31
#define B7_SOBOL_BITS 30     // grids/sobol.lua:32

void b7_set_error(const char* fmt, ...);

#define B7_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      b7_set_error("CUDA error %s at %s:%d (%s)", cudaGetErrorString(e_), __FILE__, __LINE__, #expr); \
      return B7_ERR_CUDA;                                                                          \
    }                                                                                              \
  } while (0)

#define B7_CHECK(expr)                 \
  do {                                 \
    int rc_ = (expr);                  \
    if (rc_ < 0) return rc_;           \
  } while (0)

enum { ST_SOBOL = 0, ST_KBUILD, ST_POTRF, ST_TRTRI, ST_KSTAR, ST_POSTERIOR, ST_SCORE, ST_BLR, ST_COUNT };

struct b7_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  cudaMemPool_t pool = nullptr;                   // private stream-ordered pool: the device's default pool is left alone
  cudaStream_t stream2 = nullptr;                 // far trailing updates of the Cholesky (overlaps the next panel)
  cudaStream_t stream3 = nullptr;                 // single-factor Cholesky: updates of the columns that are not needed next
  cudaEvent_t evA = nullptr, evB = nullptr, evS = nullptr, evS1 = nullptr;
  cudaEvent_t evK[2] = {nullptr, nullptr}, evP[2] = {nullptr, nullptr};   // K* pass of draw s + 1 under the posterior pass of draw s
  bool kstar_overlap = true;     // B7_KSTAR_OVERLAP=0: K* and posterior strictly one after the other
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, tm0 = nullptr, tm1 = nullptr;
  double stage_ms[ST_COUNT] = {0};
  int64_t stage_calls[ST_COUNT] = {0};
  bool profiling = false;
  bool use_i8 = false;           // posterior pass on the INT8 tensor pipe (posterior_i8.cu); default on, B7_POSTERIOR_I8=0 turns it off
  bool potrf_i8 = true;          // with use_i8: also the k = 512 trailing updates of the Cholesky (B7_POTRF_I8=0: FP64 DMMA)
  bool trtri_i8 = true;          // with use_i8: also the inversion of the factors (B7_TRTRI_I8=0: FP64 DMMA sweep)
  bool post_pair = true;         // INT8 posterior pass on CTA pairs (tcgen05 cta_group::2); B7_POST_PAIR=0: one CTA per tile
  int64_t launches = 0;
  // scratch for the posterior pass (grown on demand)
  double* ks = nullptr;        // K* panel, [panel_rows][Np]
  size_t ks_bytes = 0;
  double* moments = nullptr;   // [2][S][panel_rows] mean, var
  size_t moments_bytes = 0;
  double* xs_stage = nullptr;  // device staging of host candidate points
  size_t xs_bytes = 0;
  double* i8_partial = nullptr;   // [candidate tile][row block][64][2] partial sums of the INT8 posterior pass
  size_t i8_partial_bytes = 0;
  // size-keyed cache of freed device blocks (>= 1 MiB): a fit frees and re-requests the same multi-GB sizes, and even
  // the stream-ordered driver pool occasionally answers such a request with a fresh mapping (0.3-0.9 s; measured as
  // end-to-end steps of 0.25 / 0.85 s).  Everything is ordered on `stream`, so a cached block can be handed out at once.
  struct Block { void* p; size_t bytes; };
  std::vector<Block> cache;
  std::unordered_map<void*, size_t> live;
  size_t cache_bytes = 0, cache_cap = 0;
};

struct b7_grid {
  b7_ctx* ctx = nullptr;
  int64_t rows = 0;   // original rows
  int d = 0;
  double* X = nullptr;            // device, rows x d row-major
  std::vector<int64_t> removed;   // sorted original 0-based rows (tombstones)
  int64_t* removed_dev = nullptr; // device copy (capacity grows)
  int64_t removed_cap = 0;
  bool removed_dirty = false;
  // sharded grids (multi.cu): this handle holds rows [row_base, row_base + rows) of a grid of rows_total rows;
  // removed_global is the tombstone list of the whole grid (global original rows, sorted), replicated on every shard
  int64_t row_base = 0, rows_total = 0;
  std::vector<int64_t> removed_global;
};

struct b7_gp {
  b7_ctx* ctx = nullptr;
  int kernel = 0, N = 0, d = 0, S = 0, Np = 0, NB = 0, DT = 8, noiseless = 0;
  bool inverted = false, ready = false;
  double* X = nullptr;      // device N x d
  double* Xt = nullptr;     // device DT... x Np transposed, zero padded ([d][Np])
  double* y = nullptr;      // device N
  double* par = nullptr;    // device S x (B7_MAX_DIMS + 4): w[0..39], sf2, diag_add, m, sn2
  std::vector<double> par_host;
  std::vector<double> y_host;   // observations kept on the host for the residual upload of refits / retries
  double* fac = nullptr;    // device S x Np x Np : K -> L -> L^-1, lower, in the tiled (fragment-order) layout
  int8_t* facS = nullptr;   // device S x b7_i8_facs_stride(Np) : int8 slices of L^-1, pair-packed lower block triangle (only with ctx->use_i8)
  double* alpha = nullptr;  // device S x Np : L^-T beta = K_y^-1 (y - m) (the INT8 path's mean is m + k*^T alpha in fp64)
  double* sigma = nullptr;  // device S x Np : per-row power-of-two scales of the slices
  double* dinv = nullptr;   // device S x NB x (128 x 128 tiled) : inverse of the diagonal blocks of L
  double* dinvT = nullptr;  // device, transposes of dinv (tiled)
  double* beta = nullptr;   // device S x Np : r -> L^-1 (y - m)
  double* tt = nullptr;     // device S x (128 x Np tiled) : scratch of the inversion sweep
  double* logdet = nullptr; // device S : sum log L_ii
  int* info = nullptr;      // device S
  double* meta_dev = nullptr;   // device S x 3 : (info, log ml, jitter) per draw, exchanged by the sharded fit
  double* step_io = nullptr;    // device in / out of b7_gp_slice_step (grown on demand)
  size_t step_io_bytes = 0;
  // single-factor Cholesky replayed as a CUDA graph from the second call with the same (first draw, count) on
  // (the slice sampler's density evaluations: same handle, new hyper-parameters in device memory)
  cudaGraphExec_t potrf_graph = nullptr;
  int potrf_graph_s0 = -1, potrf_graph_count = 0, potrf_graph_launches = 0, potrf_calls_s0 = -1, potrf_calls_count = 0, potrf_calls = 0;
  bool fac_complete = true;     // fac holds L^-1 of every draw (false after a sharded fit that exchanged the int8 slices only)
  std::vector<char> sliced;   // per draw: facS/sigma hold the slices of the current L^-1
  std::vector<double> jitter;
  std::vector<int> info_host;
  std::vector<double> logml_host;
};

struct b7_blr {
  b7_ctx* ctx = nullptr;
  int N = 0, D = 0, S = 0;
  double* Linv = nullptr;  // device S x D x D : L_A^-1 (lower)
  double* w = nullptr;     // device S x D
  double* par = nullptr;   // device S x 4: alpha_p, beta, m, 1/beta
  std::vector<double> par_host;
  bool ready = true;       // Linv / w belong to par (false after a B7_FIT_LOGML_ONLY refit)
  // resident for b7_blr_refit (the log evidence the slice sampler evaluates, blr.cu)
  double* Z = nullptr;         // device N x D
  double* y = nullptr;         // device N
  double* partial = nullptr;   // device gram_blocks x (D*D + 2D): gram_kernel's per-block partials
  int gram_blocks = 0;
  double* gram = nullptr;      // device D*D + 2D: the partials summed in block order (first refit)
  double* hyp = nullptr;       // device S x 3: the rows of the last refit
  double* ev_w = nullptr;      // device S x D: w of the evidence pass
  double* ev_stat = nullptr;   // device S x 2: sum log (L_A)_ii, |w|^2
  double* ev_res = nullptr;    // device S x res_blocks: partial sums of |r - Z0 w|^2
  double* ev_out = nullptr;    // device S: log p(y | row)
  int* ev_info = nullptr;      // device 2S: evidence factor, predictor factor
};

// sharded fit (multi.cu): before / after the exchange of the per-draw state (api.cu)
int b7_gp_prepare_gather(b7_gp* gp, int s0, int count);
int b7_gp_finish_gather(b7_gp* gp, bool slices_exchanged);
// whether b7_dngo_score can run a basis of these widths (dims[0 .. n_layers]) in front of a head of width D (blr_dmma.cu)
bool b7_dngo_tiles_fit(int n_layers, const int* dims, int D);
// B7_ERR_ARG (message prefixed by `what`) unless act holds n_layers known B7_ACT_* codes (blr.cu)
int b7_check_act(const char* what, int n_layers, const int* act);
// the codes of the relu_last form of b7_mlp_features / b7_dngo_score(_multi): ReLU after every layer but the last, after the
// last one iff relu_last
inline std::vector<int> b7_relu_codes(int n_layers, int relu_last) {
  std::vector<int> act((size_t)(n_layers > 0 ? n_layers : 1), B7_ACT_RELU);
  if (n_layers > 0 && !relu_last) act[(size_t)n_layers - 1] = B7_ACT_NONE;
  return act;
}

// stream-ordered pool allocation on the context stream (api.cu)
int b7_pool_alloc(b7_ctx* ctx, void** p, size_t bytes);
void b7_pool_free(b7_ctx* ctx, void* p);

// ---- launch bookkeeping ----
static inline void b7_count(b7_ctx* ctx, int n = 1) { ctx->launches += n; }
// Brackets the launches of one stage with CUDA events on the context stream (only when profiling
// is on: it synchronises).  n = number of kernel launches of the stage inside the bracket.
struct StageTimer {
  b7_ctx* ctx; int stage;
  StageTimer(b7_ctx* c, int s) : ctx(c), stage(s) { if (ctx->profiling) cudaEventRecord(ctx->ev0, ctx->stream); }
  void stop(int n = 1) {
    if (!ctx->profiling) return;
    cudaEventRecord(ctx->ev1, ctx->stream);
    cudaEventSynchronize(ctx->ev1);
    float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    ctx->stage_ms[stage] += ms;
    ctx->stage_calls[stage] += n;
  }
};

// ---- kernels' host launchers (defined in the .cu files) ----
// sobol.cu
void b7_sobol_directions_host(int dims, uint32_t* out /* dims*30 */);
int b7_launch_sobol(b7_ctx* ctx, int dims, int64_t first_seed, int64_t count, const double* mins_dev,
                    const double* maxes_dev, double* out_dev);
// cov.cu
int b7_launch_cov_batched(b7_ctx* ctx, int kernel, const double* A /* rows x d */, int64_t rows, int64_t rows_pad, int d,
                          const double* Xt /* [d][Np] */, int N, int Np, const double* par, int64_t par_stride,
                          double* out /* rows_pad x Np */, int64_t out_stride, int batch, bool is_kxx, bool tiled = false);
// potrf.cu
int b7_launch_potrf(b7_gp* gp, int s0, int count);      // K -> L, beta, logdet, info for draws [s0,s0+count)
int b7_launch_trtri(b7_gp* gp, int s0, int count);      // L -> L^-1 in place
int b7_launch_alpha(b7_gp* gp, int s0, int count, bool from_inverse);   // alpha = L^-T beta (from L, or from L^-1)
// slice_step.cu: one directed slice step of a fit with Np == 128; io = [x0 | dir | u_right] (H each), u_shrink (K), then
// the outputs x1 (H), log p(x1), shrink uniforms used, evaluations, status (1: the K uniforms ran out)
int b7_launch_slice_step(b7_gp* gp, double* io, int K, double log_u, double width, double max_step, double prior_std,
                         int prior_order);
// posterior.cu
int b7_launch_untile(b7_ctx* ctx, const double* facT, double* out /* N x N row-major */, int Np, int N);
int b7_launch_posterior(b7_ctx* ctx, const double* LinvT /* tiled */, const double* beta, int Np, const double* ksT /* tiled */,
                        int64_t cols_pad, double sf2, double mconst, double* mean, double* var);
// potrf_i8.cu: k = 512 trailing updates of the Cholesky on the INT8 tensor pipe (scratch indexed by position in the batch)
size_t b7_i8_panel_bytes(int Np, int W);
int b7_i8_panel_slice(b7_ctx* ctx, cudaStream_t st, const double* fac, int Np, int kb0, int kb1, int row0_blk, int8_t* pA, int8_t* pB,
                      size_t p_stride, double* sig, int s0, int count);
int b7_i8_trail(b7_ctx* ctx, cudaStream_t st, double* fac, int Np, const int8_t* pA, const int8_t* pB, size_t p_stride, const double* sig,
                int kb0, int kb1, int row0_blk, int it0, int n_it, int nt0, int n_nt, int s0, int count);
// trtri_i8.cu: L -> L^-1 by block-recursive int8 products (the diagonal tiles must already hold their inverses)
int b7_launch_trtri_i8(b7_gp* gp, int s0, int count);
// posterior_i8.cu
#define B7_I8_SLICES 7        // radix-256 digit slices per operand
#define B7_I8_MAX_NP 16384    // 7 products x 2^14 x Np must stay below 2^31
size_t b7_i8_facs_stride(int Np);       // bytes of the pair-packed slice array of one draw
int b7_i8_slice_factor(b7_ctx* ctx, const double* fac, int Np, int8_t* facS, double* sigma, int s0, int count);
int b7_i8_cov_slices(b7_ctx* ctx, cudaStream_t st, int kernel, const double* A, int64_t rows, int64_t rows_pad, int d, const double* Xt,
                     int N, int Np, const double* par, double tau, const double* alpha, int8_t* ksS, double* meanP);
int b7_launch_posterior_i8(b7_ctx* ctx, const int8_t* facS, const double* sigma, int Np, const int8_t* ksS, const double* cand,
                           int64_t rows, int d, const double* Xt, const double* par, int kernel, int64_t cols_pad, double tau,
                           double sf2, double mconst, double* partial, double* mean, double* var);
size_t b7_i8_partial_bytes(int Np, int64_t cols_pad);   // scratch of the two launches above: sum v^2 and mean partials
double* b7_i8_mean_partials(double* partial, int Np, int64_t cols_pad);
// score.cu
int b7_launch_score(b7_ctx* ctx, int kind, const double* mean, const double* var, int S, int64_t M, int64_t ld,
                    double tradeoff, int bound, double sign, double fmin, const int64_t* removed, int64_t n_removed,
                    int64_t row_base, double* score_out /* nullable, M */, double* part_best, int64_t* part_idx,
                    int64_t* part_nan, int* n_parts);
int b7_argmax_finish(b7_ctx* ctx, const double* part_best, const int64_t* part_idx, const int64_t* part_nan,
                     int n_parts, double* best, int64_t* idx0, int64_t* nan_count);

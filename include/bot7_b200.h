/*
 * bot7_b200 -- C ABI of the B200-native surrogate-fit-and-acquisition path of bot7.
 *
 * The reference (montyhall/bot7, Lua/Torch7) has no FFI: its boundary is the Lua object protocol
 * of bot7.grids / bot7.models / bot7.scores / bots.bayesopt.  Every entry point below names the
 * reference interface whose body it replaces (file:line relative to the reference tree); the
 * LuaJIT-FFI glue that binds them is in lua/bot7_b200/ and INTEGRATION.md.
 *
 * Conventions
 *  - every function returns int: 0 ok; >0 LAPACK-style info; <0 error (text: b7_last_error()).
 *  - all matrices are row-major contiguous fp64 (torch.DoubleTensor:contiguous():data()).
 *  - host pointers are borrowed for the duration of the call; device state lives in opaque
 *    handles released by b7_*_free.  One host thread per context.  Calls are synchronous.
 *  - there is no CPU fallback: without a CUDA device b7_init fails.
 */
#ifndef BOT7_B200_H
#define BOT7_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b7_ctx b7_ctx;
typedef struct b7_grid b7_grid;
typedef struct b7_gp b7_gp;
typedef struct b7_blr b7_blr;
typedef struct b7_comm b7_comm;

enum { B7_KERNEL_ARDSE = 0, B7_KERNEL_MATERN52 = 1 };           /* bots/bayesopt.lua:41 model.kernel */
enum { B7_SCORE_EI = 0, B7_SCORE_CB = 1 };                       /* scores/init.lua */
enum { B7_BOUND_LOWER = 0, B7_BOUND_UPPER = 1 };                 /* scores/confidence_bound.lua:32 */
enum { B7_FIT_PREDICT = 0, B7_FIT_LOGML_ONLY = 1, B7_FIT_DEFER = 2 }; /* flags of b7_gp_fit */
enum { B7_ACT_NONE = 0, B7_ACT_RELU = 1, B7_ACT_TANH = 2 };         /* activation after a Linear of the DNGO basis */
enum { B7_ERR_ARG = -1, B7_ERR_CUDA = -2, B7_ERR_STATE = -3, B7_ERR_NOMEM = -4, B7_ERR_NCCL = -5 };

int         b7_version(void);
const char* b7_last_error(void);

/* context: one per (process, device) */
int  b7_init(int device, b7_ctx** out);
void b7_shutdown(b7_ctx* ctx);
int  b7_device_count(void);
int  b7_sync(b7_ctx* ctx);
/* stage timers (CUDA events on the context stream), accumulated since the last reset:
 * 0 sobol, 1 K build, 2 potrf, 3 trtri, 4 K* build, 5 posterior (TRMM), 6 scoring, 7 blr */
int  b7_set_profiling(b7_ctx* ctx, int on);   /* off by default: stage timing synchronises per launch */
int  b7_reset_stage_timers(b7_ctx* ctx);
int  b7_last_stage_ms(b7_ctx* ctx, int stage, double* ms_total, int64_t* launches);
/* Which tensor pipe carries the posterior pass (V = L^-1 K*^T, N^2 flop per candidate per draw):
 *   B7_PATH_FP64_DMMA  fp64 operands on DMMA tiles (posterior.cu);
 *   B7_PATH_INT8_OZAKI both operands split error-free into 7 radix-256 int8 slices, 28 exact int32 products on
 *                      tcgen05.mma.kind::i8 (CTA pairs), recombined in fp64 (posterior_i8.cu): variance to ~1e-12 sf2,
 *                      the mean an fp64 dot product k*^T alpha; 3x the throughput.  With this path the k = 512 trailing updates of batched factorisations
 *                      (potrf_i8.cu) and the inversion of the factors (trtri_i8.cu) use the same slicing
 *                      (B7_POTRF_I8=0 / B7_TRTRI_I8=0 keep those in FP64).  Default; B7_POSTERIOR_I8=0 in the
 *                      environment selects DMMA; fits with more than 16384 observations always use DMMA (int32
 *                      exactness bound). */
enum { B7_PATH_FP64_DMMA = 0, B7_PATH_INT8_OZAKI = 1 };
int  b7_set_posterior_path(b7_ctx* ctx, int path);
int  b7_get_posterior_path(b7_ctx* ctx);
/* device-side stopwatch: CUDA events recorded on the context stream (begin; ...calls...; end -> ms) */
int  b7_timer_begin(b7_ctx* ctx);
int  b7_timer_end(b7_ctx* ctx, double* ms);
/* number of kernels this library has launched on the context since b7_init */
int64_t b7_launch_count(b7_ctx* ctx);

/* ---- grids: replaces grid:generate / grid:i4_sobol (grids/sobol.lua:58-90,216-335) ---------- */
/* scaled direction integers V[i][j] (dims x 30, uint32): grids/sobol.lua:236-288 */
int b7_sobol_directions(int dims, uint32_t* out);
/* points seed = first_seed .. first_seed+count-1 (reference: seed = j + skip - 1, skip defaults 1,
 * grids/sobol.lua:70-75), rescaled by (maxes-mins), +mins as two rounded ops (:79-81) when both
 * are given.  out_host (count*dims) and out_grid are each optional. */
int b7_sobol_generate(b7_ctx* ctx, int dims, int64_t first_seed, int64_t count,
                      const double* mins, const double* maxes, double* out_host, b7_grid** out_grid);
/* grids/random.lua:23-35 or any user grid: upload an M x d host matrix */
int b7_grid_from_host(b7_ctx* ctx, const double* X, int64_t M, int d, b7_grid** out_grid);
int b7_grid_read(b7_grid* g, int64_t first_row, int64_t count, double* out_host);  /* original numbering */
int64_t b7_grid_size(b7_grid* g);        /* live rows (original rows minus removed) */
int64_t b7_grid_rows(b7_grid* g);        /* original rows */
int b7_grid_dims(b7_grid* g);
/* utils.tensor.steal / remove (utils/tensor.lua:158-193 via bots/abstract.lua:118): remove the row
 * with 1-based index `compacted_index` in the *current compacted* numbering.  The device grid keeps
 * its original layout; a sorted tombstone list reproduces the reference's numbering. */
int b7_grid_remove(b7_grid* g, int64_t compacted_index, double* removed_row /* nullable, d */);
int b7_grid_original_index(b7_grid* g, int64_t compacted_index, int64_t* original_index_1based);
void b7_grid_free(b7_grid* g);

/* ---- GP: replaces gp_regressor:predict / the density evaluated by sample_hypers -------------
 * (external gpTorch7; call sites bots/bayesopt.lua:68,74-75, scores/expected_improvement.lua:63).
 * hyp: S x H, H = d+3, row = [log l_1..log l_d, log sigma_f, log sigma_n, m]  (oracle/SPEC.md).
 * One Cholesky factor per draw with the jitter-retry policy of utils.math.chol
 * (utils/math.lua:159-218).  info[s]: 0 ok, >0 first failing pivot when even the retries failed
 * (chol(I) is then used, as the reference does); jitter[s]: eps finally added (0 if none).
 * flags: B7_FIT_PREDICT also inverts the factor for the posterior pass; B7_FIT_LOGML_ONLY stops
 * after K + potrf + beta + logdet (the slice sampler's density evaluation, samplers/slice.lua:100). */
int b7_gp_fit(b7_ctx* ctx, int kernel, const double* X, const double* y, int N, int d,
              const double* hyp, int S, int H, int noiseless, int flags,
              b7_gp** out, int* info /* S, nullable */, double* logml /* S, nullable */,
              double* jitter /* S, nullable */);
/* Same observations, new S x H hyper-parameter draws, every device buffer reused: the density
 * evaluation of the slice sampler (samplers/slice.lua:100-103) with X and y resident.
 * flags: B7_FIT_PREDICT or B7_FIT_LOGML_ONLY. */
int b7_gp_refit(b7_gp* gp, const double* hyp, int flags, int* info, double* logml, double* jitter);
/* One directed slice step (samplers/slice.lua:92-168) on the density log p(y | h) + log p(h) of this handle's
 * observations, in one launch, for N <= 128: every density is the value b7_gp_refit(B7_FIT_LOGML_ONLY) gives for that
 * row at this N (-inf unless info == 0 and finite) minus 1/2 sum (h_i / prior_std)^2, summed in prior_order (0 sequential
 * as Torch7, 1 numpy's pairwise sum).  The handle is only read (typically the one of B7_FIT_LOGML_ONLY); H = d + 3.
 * The caller draws the step's random numbers in the reference's order and passes them in: the direction (normalised:
 * dir), log U of the slice level, H uniforms of the bracket, then K shrink uniforms.  width: the scalar bracket width
 * (opt.width), max_step: the step-out limit per side.  Out: x1 = x0 + dir * dx (H), the shrink uniforms consumed, the
 * density evaluations made, log p(x1).  B7_ERR_ARG for N > 128 or a width that is not finite and positive;
 * B7_ERR_STATE when the K shrink uniforms ran out (call again with the same numbers and a larger K). */
int b7_gp_slice_step(b7_gp* gp, const double* x0 /* H */, const double* dir /* H, unit */, double log_u_level,
                     const double* u_right /* H */, const double* u_shrink /* K */, int K, double width,
                     double max_step, double prior_std, int prior_order, double* x1 /* H */, int* n_shrink_used,
                     int* n_evals, double* logp_x1);
int b7_gp_num_draws(b7_gp* gp);
int b7_gp_num_obs(b7_gp* gp);
/* model:predict(X_obs,Y_obs,X_hid,hyp,{mean,var}) for draw s (0-based): M x d host points ->
 * latent mean / variance (scores/expected_improvement.lua:63-66). */
int b7_gp_predict(b7_gp* gp, int s, const double* Xs, int64_t M, double* mean, double* var);
/* debugging / multi-GPU plumbing: device pointers of the per-draw state (row-major, ld = Npad):
 * what: 0 factor (L, or L^-1 after inversion), 1 beta = L^-1 (y-m), 2 diag-block inverses */
int b7_gp_device_ptr(b7_gp* gp, int what, void** ptr, int64_t* bytes);
int b7_gp_padded_n(b7_gp* gp);
/* copy factor rows of draw s back to the host (N x N, lower; what as above, 0 only) */
int b7_gp_read_factor(b7_gp* gp, int s, double* out_host);
/* draw-sharded fit (multi-GPU): with B7_FIT_DEFER in b7_gp_fit nothing is factorised; then
 * b7_gp_fit_range factorises draws [s0, s0+count) on this device.  The other slots are filled
 * by the host through b7_gp_device_ptr (NCCL all-gather) and b7_gp_mark_ready. */
int b7_gp_fit_range(b7_gp* gp, int s0, int count, int* info, double* logml, double* jitter);
int b7_gp_invert_range(b7_gp* gp, int s0, int count);
int b7_gp_mark_ready(b7_gp* gp);
void b7_gp_free(b7_gp* gp);

/* ---- acquisition: replaces bot:eval + bot:nominate (bots/bayesopt.lua:56-99) -----------------
 * For every live candidate of `grid`: posterior per draw, EI (scores/expected_improvement.lua:69-88)
 * or confidence bound (scores/confidence_bound.lua:70-106), sequential average over the S draws
 * (bots/bayesopt.lua:73-79) and first-maximum argmax (bots/bayesopt.lua:96).
 * score_host (nullable): averaged score of every ORIGINAL row (removed rows hold NaN).
 * argmax: 1-based index in the current compacted numbering (0 if no finite-or-inf score);
 * argmax_original: 1-based original row.  nan_count: NaN scores among live rows (they are skipped). */
int b7_acq_score(b7_gp* gp, b7_grid* grid, int kind, double tradeoff, int bound, double sign,
                 double fmin, double* score_host, int64_t* argmax, int64_t* argmax_original,
                 double* best, int64_t* nan_count);
/* Same, restricted to original rows [row0, row0+count): the per-GPU shard of the candidate grid.
 * argmax_original is global (1-based original row); combine across ranks with "max score, then
 * smallest original index". */
int b7_acq_score_range(b7_gp* gp, b7_grid* grid, int64_t row0, int64_t count, int kind,
                       double tradeoff, int bound, double sign, double fmin, double* score_host,
                       int64_t* argmax_original, double* best, int64_t* nan_count);
/* EI.compute / conf_bound.compute + MC average + argmax on given per-draw moments
 * (mean, var: S x M host arrays).  The fused scoring pass on its own. */
int b7_score_moments(b7_ctx* ctx, int kind, const double* mean, const double* var, int S, int64_t M,
                     double tradeoff, int bound, double sign, double fmin, double* score_host,
                     int64_t* argmax, double* best, int64_t* nan_count);

/* ---- DNGO head: replaces bayes_linear:predict called from models/dngo.lua:174 -----------------
 * hyp: S x 3 rows [log alpha_p, log beta, m] (oracle/SPEC.md). */
/* DNGO basis functions (models/dngo.lua:155-171: X -> output of the last hidden layer of the trained network):
 * Linear/ReLU MLP forward in fp64 on a device-resident grid.  dims[0..n_layers] are the widths (dims[0] = grid dims, each
 * <= 64), W[l] is dims[l+1] x dims[l] row-major (torch nn.Linear.weight), b[l] has dims[l+1] entries; every layer is
 * followed by ReLU (the last one only if relu_last).  The result is a new device grid of features that inherits the
 * removed rows of the input grid and feeds b7_blr_score. */
int b7_mlp_features(b7_ctx* ctx, b7_grid* in, int n_layers, const int* dims, const double* const* W,
                    const double* const* b, int relu_last, b7_grid** out);
/* Same, with one activation per layer instead of relu_last: act[l] (n_layers entries) follows layer l, B7_ACT_NONE (nothing,
 * nn.Linear alone), B7_ACT_RELU (nn.ReLU, max(0, x)) or B7_ACT_TANH (nn.Tanh, fp64 tanh within 2 ulp).  An unknown code is
 * B7_ERR_ARG before any device work.  b7_mlp_features is this call with B7_ACT_RELU for the inner layers and
 * relu_last ? B7_ACT_RELU : B7_ACT_NONE for the last one. */
int b7_mlp_features_act(b7_ctx* ctx, b7_grid* in, int n_layers, const int* dims, const double* const* W,
                        const double* const* b, const int* act, b7_grid** out);
int b7_blr_fit(b7_ctx* ctx, const double* Z0, const double* y, int N, int D, const double* hyp, int S,
               b7_blr** out, int* info);
/* Same features and responses, new S x 3 rows [log alpha_p, log beta, m], every device buffer reused: the density the
 * slice sampler evaluates for bayes_linear's hyper-parameters (declared arithmetic, DESIGN.md section 4.5):
 *   log p(y | h) = D/2 log alpha_p + N/2 log beta - E - sum_i log (L_A)_ii - N/2 log 2 pi,
 *   E = beta/2 |y - m - Z0 w|^2 + alpha_p/2 |w|^2.
 * flags: B7_FIT_PREDICT (also refresh L_A^-1, w for b7_blr_predict / b7_blr_score / b7_dngo_score, bit-identical to a
 * b7_blr_fit with the same rows) or B7_FIT_LOGML_ONLY (the handle cannot predict until the next B7_FIT_PREDICT).
 * logev[s]: log p(y | row s) (-inf when info[s] != 0 or the value is not finite); a row's result does not depend on the
 * other rows of the call. */
int b7_blr_refit(b7_blr* blr, const double* hyp, int flags, int* info /* S, nullable */, double* logev /* S, nullable */);
int b7_blr_num_draws(b7_blr* blr);
int b7_blr_predict(b7_blr* blr, int s, const double* Z1, int64_t M, double* mean, double* var);
int b7_blr_score(b7_blr* blr, b7_grid* features, int kind, double tradeoff, int bound, double sign,
                 double fmin, double* score_host, int64_t* argmax, int64_t* argmax_original,
                 double* best, int64_t* nan_count);
/* dngo:predict on the candidate grid in one pass (models/dngo.lua:155-174): the basis (same arguments as
 * b7_mlp_features, widths <= 63) is evaluated tile by tile in shared memory in front of the BLR head, so the M x D
 * feature matrix Z1 is never stored; then the same scoring / average / argmax as b7_blr_score. */
int b7_dngo_score(b7_blr* blr, b7_grid* grid, int n_layers, const int* dims, const double* const* W,
                  const double* const* b, int relu_last, int kind, double tradeoff, int bound, double sign, double fmin,
                  double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count);
/* b7_dngo_score with one activation code per layer (act as in b7_mlp_features_act) */
int b7_dngo_score_act(b7_blr* blr, b7_grid* grid, int n_layers, const int* dims, const double* const* W,
                      const double* const* b, const int* act, int kind, double tradeoff, int bound, double sign, double fmin,
                      double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count);
void b7_blr_free(b7_blr* blr);

/* ---- multi-GPU: candidate shards + draw-sharded fit (bots/bayesopt.lua:56-99 over config.bot.nGPU devices) ----
 * The path shards by candidates: rank g of G scores the contiguous original-row range
 * [g*floor(M/G) + min(g, M%G), ...) of the grid; the S factorisations are split the same way over the ranks and
 * exchanged once per fit with NCCL over NVLink (in the form the posterior pass reads: the packed int8 slices of
 * L^-1 + row scales + alpha on the INT8 path, L^-1 + beta on the FP64 path); the per-rank (best, index, nan)
 * triples are all-gathered and combined with "larger score, then smaller original index" -- the reference's
 * first-maximum scan for any G.  libnccl.so.2 is loaded at run time (dlopen) by the first b7_comm_* call.
 *
 * A communicator drives n_local devices of this process out of `world` ranks:
 *   b7_comm_init_all   one process, all listed devices (what the LuaJIT host calls): world = n_local = n_gpus;
 *   b7_comm_init_rank  one process per GPU (torchrun): rank 0 calls b7_comm_unique_id, the 128 bytes travel by any
 *                      means (torch.distributed, a file), every rank calls b7_comm_init_rank. */
int  b7_comm_init_all(int n_gpus, const int* device_ids /* nullable: 0 .. n_gpus-1 */, b7_comm** out);
int  b7_comm_unique_id(char* id128);
int  b7_comm_init_rank(int device, const char* id128, int world, int rank, b7_comm** out);
int  b7_comm_world(b7_comm* comm);
int  b7_comm_local_count(b7_comm* comm);
int  b7_comm_first_rank(b7_comm* comm);
b7_ctx* b7_comm_ctx(b7_comm* comm, int local_index);
void b7_comm_free(b7_comm* comm);
/* rows [row0, row0 + count) of M rows owned by `rank` of `world` (the same rule shards the S draws of a fit) */
int  b7_shard_range(int64_t M, int world, int rank, int64_t* row0, int64_t* count);
/* Sobol grid of `count` points from first_seed, each local device generating only its own shard;
 * out_grids: n_local handles (free each with b7_grid_free).  Indices reported for them are global. */
int  b7_sobol_generate_sharded(b7_comm* comm, int dims, int64_t first_seed, int64_t count, const double* mins,
                               const double* maxes, b7_grid** out_grids);
/* any host grid (grids/random.lua or cached candidates): X is the full M x d matrix on every process */
int  b7_grid_from_host_sharded(b7_comm* comm, const double* X, int64_t M, int d, b7_grid** out_grids);
/* utils.tensor.steal on the sharded grid: `compacted_index` is global (1-based, current compacted numbering);
 * every process makes the same call */
int  b7_grid_remove_sharded(b7_comm* comm, b7_grid** grids, int64_t compacted_index, double* removed_row /* nullable, d */);
/* b7_gp_fit over the communicator: every rank factorises and inverts its share of the S draws, one NCCL
 * all-gather fills the rest.  out_gps: n_local handles, each holding all S draws; info / logml / jitter: S entries.
 * gather_ms (nullable): device time of the exchange on the first local device. */
int  b7_gp_fit_sharded(b7_comm* comm, int kernel, const double* X, const double* y, int N, int d, const double* hyp, int S,
                       int H, int noiseless, b7_gp** out_gps, int* info, double* logml, double* jitter, double* gather_ms);
/* b7_acq_score over the communicator: each local device scores its shard with all S factors, then the triples are
 * combined.  score_host (nullable): the scores of the local shards, concatenated in local-device order (the whole
 * grid with b7_comm_init_all); argmax / argmax_original are global 1-based indices (compacted / original). */
int  b7_acq_score_multi(b7_comm* comm, b7_gp** gps, b7_grid** grids, int kind, double tradeoff, int bound, double sign,
                        double fmin, double* score_host, int64_t* argmax, int64_t* argmax_original, double* best,
                        int64_t* nan_count);
/* DNGO over the communicator (models/dngo.lua:155-174 under bots/bayesopt.lua:65-66 with config.bot.nGPU > 1).  With one
 * process per GPU every rank enters exactly one all-gather per call, also after its local step failed; then that rank
 * returns its own error and every other rank B7_ERR_STATE naming it.  With world == 1 both are the one-device calls. */
/* b7_blr_fit on every local device of the communicator: each handle holds all S rows and predicts / scores bit for bit like a
 * one-device b7_blr_fit with the same arguments.  out_blrs: n_local handles (free each with b7_blr_free); info: S entries. */
int  b7_blr_fit_multi(b7_comm* comm, const double* Z0, const double* y, int N, int D, const double* hyp, int S,
                      b7_blr** out_blrs, int* info /* S, nullable */);
/* b7_dngo_score over the communicator: each local device runs the fused basis + BLR head + score pass on its shard of the
 * candidate grid, then the per-rank triples are combined with the rule of b7_acq_score_multi.  Arguments and outputs as
 * b7_dngo_score and b7_acq_score_multi (score_host: the local shards concatenated in local-device order).  Every handle is
 * checked before any device work: B7_ERR_ARG for a handle of another device, dims that do not match the grid and the head,
 * or widths the tile kernel cannot take; B7_ERR_STATE for a head whose last refit was B7_FIT_LOGML_ONLY. */
int  b7_dngo_score_multi(b7_comm* comm, b7_blr** blrs, b7_grid** grids, int n_layers, const int* dims, const double* const* W,
                         const double* const* b, int relu_last, int kind, double tradeoff, int bound, double sign, double fmin,
                         double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count);
/* b7_dngo_score_multi with one activation code per layer (act as in b7_mlp_features_act); an unknown code is B7_ERR_ARG on
 * every rank, before any device work and without entering the all-gather, like the other argument checks. */
int  b7_dngo_score_multi_act(b7_comm* comm, b7_blr** blrs, b7_grid** grids, int n_layers, const int* dims, const double* const* W,
                             const double* const* b, const int* act, int kind, double tradeoff, int bound, double sign, double fmin,
                             double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count);

#ifdef __cplusplus
}
#endif
#endif /* BOT7_B200_H */

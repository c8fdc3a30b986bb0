// C ABI of libbot7_b200.so: handles, host<->device plumbing, jitter-retry policy, panel loop.
// See include/bot7_b200.h for the contract and the reference interface each entry replaces.
#include <math.h>
#include <stdarg.h>
#include <cmath>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include <algorithm>

#include "b7_internal.h"

static thread_local char g_err[512] = "";

void b7_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int b7_score_grid_size(b7_ctx* ctx, int64_t M);   // score.cu

namespace {

constexpr int kParStride = B7_MAX_DIMS + 4;
constexpr double kLog2Pi = 1.83787706640934548356;

// Stream-ordered allocation from the device's memory pool (release threshold = unlimited, set in
// b7_init): buffers freed by one fit are handed back to the next without a driver round trip
// (a fresh cudaMalloc of the 4.3 GB factor array costs tens of ms; the reference allocates and
// garbage-collects on every call, bots/bayesopt.lua:77).
constexpr size_t kCacheMin = (size_t)1 << 20;

void cache_flush(b7_ctx* ctx) {
  for (const b7_ctx::Block& b : ctx->cache) cudaFreeAsync(b.p, ctx->stream);
  ctx->cache.clear();
  ctx->cache_bytes = 0;
}

int dev_alloc_bytes(b7_ctx* ctx, void** p, size_t bytes) {
  *p = nullptr;
  bytes = (bytes + 255) / 256 * 256;
  if (bytes == 0) bytes = 256;
  if (bytes >= kCacheMin)
    for (size_t i = 0; i < ctx->cache.size(); ++i)
      if (ctx->cache[i].bytes == bytes) {                 // the same request as an earlier fit: same block
        *p = ctx->cache[i].p;
        ctx->cache_bytes -= bytes;
        ctx->cache[i] = ctx->cache.back();
        ctx->cache.pop_back();
        ctx->live[*p] = bytes;
        return 0;
      }
  cudaError_t e = cudaMallocFromPoolAsync(p, bytes, ctx->pool, ctx->stream);
  if (e != cudaSuccess && !ctx->cache.empty()) {          // give the cached blocks back and try again
    cudaGetLastError();
    cache_flush(ctx);
    cudaStreamSynchronize(ctx->stream);
    cudaMemPoolTrimTo(ctx->pool, 0);
    e = cudaMallocFromPoolAsync(p, bytes, ctx->pool, ctx->stream);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    b7_set_error("device allocation of %zu bytes failed: %s", bytes, cudaGetErrorString(e));
    return B7_ERR_NOMEM;
  }
  if (bytes >= kCacheMin) ctx->live[*p] = bytes;
  return 0;
}

template <typename T>
int dev_alloc(b7_ctx* ctx, T** p, size_t count) { return dev_alloc_bytes(ctx, (void**)p, (count ? count : 1) * sizeof(T)); }

inline void dev_free(b7_ctx* ctx, void* p) {
  if (!p) return;
  auto it = ctx->live.find(p);
  if (it != ctx->live.end()) {
    const size_t bytes = it->second;
    ctx->live.erase(it);
    if (ctx->cache_bytes + bytes <= ctx->cache_cap) {
      ctx->cache.push_back({p, bytes});
      ctx->cache_bytes += bytes;
      return;
    }
  }
  cudaFreeAsync(p, ctx->stream);
}

int grow(b7_ctx* ctx, double** p, size_t* have, size_t need_bytes) {
  if (*have >= need_bytes) return 0;
  dev_free(ctx, *p);
  *p = nullptr; *have = 0;
  B7_CHECK(dev_alloc(ctx, p, need_bytes / sizeof(double) + 1));
  *have = need_bytes;
  return 0;
}

inline int64_t pad128(int64_t n) { return (n + 127) / 128 * 128; }

// candidates per posterior launch: one 128-candidate tile per SM = one full wave
// Smaller fits get proportionally larger panels (up to 8x), so that a launch stays long against its fixed costs (barrier and
// TMEM set-up, pipeline fill and drain: a 148 x 128 panel at N = 512 was a 97 us launch at 0.35 of the INT8 peak) while
// the K* panel buffer keeps its size (rows x Np).
inline int64_t panel_rows(b7_ctx* ctx, int Np = 4096) {
  const int64_t base = (int64_t)ctx->sm_count * 128;
  const int64_t f = Np >= 4096 ? 1 : std::min<int64_t>(8, 4096 / std::max(Np, 128));
  return base * f;
}

int sync_removed(b7_grid* g) {
  if (!g->removed_dirty) return 0;
  int64_t n = (int64_t)g->removed.size();
  if (n > g->removed_cap) {
    dev_free(g->ctx, g->removed_dev);
    g->removed_cap = std::max<int64_t>(256, 2 * n);
    B7_CHECK(dev_alloc(g->ctx, &g->removed_dev, (size_t)g->removed_cap));
  }
  if (n > 0)
    B7_CUDA(cudaMemcpyAsync(g->removed_dev, g->removed.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, g->ctx->stream));
  g->removed_dirty = false;
  return 0;
}

// tiled-layout helpers (gemm_tile.cuh): element (row, k) of a matrix with Np columns
__device__ __forceinline__ long long tiled_index(int Np, int row, int k) {
  return ((long long)(row >> 7) * (Np >> 4) + (k >> 4)) * 2048 + ((k >> 2) & 3) * 512 + (row & 127) * 4 + (k & 3);
}

__global__ void frob_rows_kernel(const double* __restrict__ A, int Np, int N, double* __restrict__ out) {
  // sum of squares of row blockIdx.x of the symmetric matrix, read from its lower triangle only
  // (the upper blocks are never built): 2 * strictly-lower + diagonal; fixed-order tree
  __shared__ double sh[256];
  double s = 0.0;
  const int row = blockIdx.x;
  for (int k = threadIdx.x; k <= row; k += blockDim.x) {
    const double v = A[tiled_index(Np, row, k)];
    s += (k < row ? 2.0 : 1.0) * v * v;
  }
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sh[0];
}

__global__ void identity_kernel(double* __restrict__ A, int Np) {
  long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e < (long long)Np * Np) { const int row = (int)(e / Np), k = (int)(e % Np); A[tiled_index(Np, row, k)] = (row == k) ? 1.0 : 0.0; }
}

int upload_residual(b7_gp* gp, int s, const std::vector<double>& yh) {
  // r = y - m (padded with zeros) into beta[s]
  std::vector<double> r((size_t)gp->Np, 0.0);
  const double m = gp->par_host[(size_t)s * kParStride + B7_MAX_DIMS + 2];
  for (int i = 0; i < gp->N; ++i) r[i] = yh[i] - m;
  B7_CUDA(cudaMemcpyAsync(gp->beta + (size_t)s * gp->Np, r.data(), gp->Np * sizeof(double), cudaMemcpyHostToDevice, gp->ctx->stream));
  B7_CUDA(cudaStreamSynchronize(gp->ctx->stream));
  return 0;
}

int build_kxx(b7_gp* gp, int s0, int count) {
  b7_ctx* ctx = gp->ctx;
  StageTimer t(ctx, ST_KBUILD);
  B7_CHECK(b7_launch_cov_batched(ctx, gp->kernel, gp->X, gp->N, gp->Np, gp->d, gp->Xt, gp->N, gp->Np,
                                 gp->par + (size_t)s0 * kParStride, kParStride, gp->fac + (size_t)s0 * gp->Np * gp->Np,
                                 (int64_t)gp->Np * gp->Np, count, true, true));
  t.stop(1);
  return 0;
}

int factor(b7_gp* gp, int s0, int count) {
  b7_ctx* ctx = gp->ctx;
  StageTimer t(ctx, ST_POTRF);
  int64_t before = ctx->launches;
  B7_CHECK(b7_launch_potrf(gp, s0, count));
  t.stop((int)(ctx->launches - before));
  return 0;
}

}  // namespace

int b7_pool_alloc(b7_ctx* ctx, void** p, size_t bytes) {
  char* q = nullptr;
  int rc = dev_alloc(ctx, &q, bytes);
  *p = q;
  return rc;
}
void b7_pool_free(b7_ctx* ctx, void* p) { dev_free(ctx, p); }


extern "C" {

int b7_version(void) { return 100; }
const char* b7_last_error(void) { return g_err; }

int b7_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int b7_init(int device, b7_ctx** out) {
  if (!out) { b7_set_error("b7_init: out is null"); return B7_ERR_ARG; }
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    b7_set_error("b7_init: no CUDA device (%s); this library has no CPU path", e == cudaSuccess ? "count 0" : cudaGetErrorString(e));
    return B7_ERR_CUDA;
  }
  if (device < 0 || device >= n) { b7_set_error("b7_init: device %d out of range [0,%d)", device, n); return B7_ERR_ARG; }
  B7_CUDA(cudaSetDevice(device));
  b7_ctx* ctx = new b7_ctx();
  ctx->device = device;
  cudaDeviceProp p;
  B7_CUDA(cudaGetDeviceProperties(&p, device));
  ctx->sm_count = p.multiProcessorCount;
  if (p.major < 10) { b7_set_error("b7_init: device is sm_%d%d, this build is sm_100a only", p.major, p.minor); delete ctx; return B7_ERR_CUDA; }
  // main stream at the highest priority: when the far trailing update (stream2) fills the machine, the
  // small kernels of the next panel still get the first SMs that free up
  int prio_lo = 0, prio_hi = 0;
  B7_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
  B7_CUDA(cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi));
  B7_CUDA(cudaStreamCreateWithPriority(&ctx->stream2, cudaStreamNonBlocking, prio_lo));
  B7_CUDA(cudaEventCreateWithFlags(&ctx->evA, cudaEventDisableTiming));
  B7_CUDA(cudaEventCreateWithFlags(&ctx->evB, cudaEventDisableTiming));
  B7_CUDA(cudaStreamCreateWithPriority(&ctx->stream3, cudaStreamNonBlocking, (prio_hi + prio_lo) / 2));
  B7_CUDA(cudaEventCreateWithFlags(&ctx->evS, cudaEventDisableTiming));
  B7_CUDA(cudaEventCreateWithFlags(&ctx->evS1, cudaEventDisableTiming));
  for (int i = 0; i < 2; ++i) {
    B7_CUDA(cudaEventCreateWithFlags(&ctx->evK[i], cudaEventDisableTiming));
    B7_CUDA(cudaEventCreateWithFlags(&ctx->evP[i], cudaEventDisableTiming));
  }
  { const char* e = getenv("B7_KSTAR_OVERLAP"); ctx->kstar_overlap = !(e && e[0] == '0'); }
  // a pool of this context's own (the device's default pool, which torch or NCCL in the same process may use, keeps its
  // settings); never trimmed while the context lives: freed buffers stay in the pool for the next fit
  cudaMemPoolProps props = {};
  props.allocType = cudaMemAllocationTypePinned;
  props.handleTypes = cudaMemHandleTypeNone;
  props.location.type = cudaMemLocationTypeDevice;
  props.location.id = device;
  B7_CUDA(cudaMemPoolCreate(&ctx->pool, &props));
  unsigned long long keep = ~0ULL;
  B7_CUDA(cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep));
  // exact-size block cache in front of the pool: at most B7_CACHE_FRACTION (default 1/3) of the device memory
  {
    size_t free_b = 0, total_b = 0;
    B7_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const char* e = getenv("B7_CACHE_FRACTION");
    const double frac = e ? atof(e) : 1.0 / 3.0;
    ctx->cache_cap = (size_t)((frac < 0.0 ? 0.0 : (frac > 0.9 ? 0.9 : frac)) * (double)total_b);
  }
  { const char* e = getenv("B7_POSTERIOR_I8"); ctx->use_i8 = !(e && e[0] == '0'); }
  { const char* e = getenv("B7_POTRF_I8"); ctx->potrf_i8 = !(e && e[0] == '0'); }
  { const char* e = getenv("B7_TRTRI_I8"); ctx->trtri_i8 = !(e && e[0] == '0'); }
  { const char* e = getenv("B7_POST_PAIR"); ctx->post_pair = !(e && e[0] == '0') && ctx->sm_count >= 2; }
  B7_CUDA(cudaEventCreate(&ctx->ev0));
  B7_CUDA(cudaEventCreate(&ctx->ev1));
  B7_CUDA(cudaEventCreate(&ctx->tm0));
  B7_CUDA(cudaEventCreate(&ctx->tm1));
  *out = ctx;
  return 0;
}

void b7_shutdown(b7_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  dev_free(ctx, ctx->ks);
  dev_free(ctx, ctx->moments);
  dev_free(ctx, ctx->xs_stage);
  dev_free(ctx, ctx->i8_partial);
  cache_flush(ctx);
  cudaStreamSynchronize(ctx->stream);
  cudaStreamSynchronize(ctx->stream2);
  cudaStreamSynchronize(ctx->stream3);
  cudaEventDestroy(ctx->evS);
  cudaEventDestroy(ctx->evS1);
  cudaStreamDestroy(ctx->stream3);
  cudaEventDestroy(ctx->evA);
  cudaEventDestroy(ctx->evB);
  for (int i = 0; i < 2; ++i) { cudaEventDestroy(ctx->evK[i]); cudaEventDestroy(ctx->evP[i]); }
  cudaStreamDestroy(ctx->stream2);
  cudaEventDestroy(ctx->ev0);
  cudaEventDestroy(ctx->ev1);
  cudaEventDestroy(ctx->tm0);
  cudaEventDestroy(ctx->tm1);
  cudaStreamDestroy(ctx->stream);
  if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
  delete ctx;
}

int b7_sync(b7_ctx* ctx) {
  if (!ctx) return B7_ERR_ARG;
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int b7_set_posterior_path(b7_ctx* ctx, int path) {
  if (!ctx || (path != B7_PATH_FP64_DMMA && path != B7_PATH_INT8_OZAKI)) { b7_set_error("set_posterior_path: bad arguments"); return B7_ERR_ARG; }
  ctx->use_i8 = path == B7_PATH_INT8_OZAKI;
  return 0;
}
int b7_get_posterior_path(b7_ctx* ctx) { return ctx && ctx->use_i8 ? B7_PATH_INT8_OZAKI : B7_PATH_FP64_DMMA; }

int b7_timer_begin(b7_ctx* ctx) {
  if (!ctx) return B7_ERR_ARG;
  B7_CUDA(cudaSetDevice(ctx->device));
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  B7_CUDA(cudaEventRecord(ctx->tm0, ctx->stream));
  return 0;
}
int b7_timer_end(b7_ctx* ctx, double* ms) {
  if (!ctx || !ms) return B7_ERR_ARG;
  B7_CUDA(cudaEventRecord(ctx->tm1, ctx->stream));
  B7_CUDA(cudaEventSynchronize(ctx->tm1));
  float f = 0;
  B7_CUDA(cudaEventElapsedTime(&f, ctx->tm0, ctx->tm1));
  *ms = f;
  return 0;
}

int b7_set_profiling(b7_ctx* ctx, int on) { if (!ctx) return B7_ERR_ARG; ctx->profiling = on != 0; return 0; }
int b7_reset_stage_timers(b7_ctx* ctx) {
  if (!ctx) return B7_ERR_ARG;
  for (int i = 0; i < ST_COUNT; ++i) { ctx->stage_ms[i] = 0; ctx->stage_calls[i] = 0; }
  return 0;
}
int b7_last_stage_ms(b7_ctx* ctx, int stage, double* ms_total, int64_t* launches) {
  if (!ctx || stage < 0 || stage >= ST_COUNT) return B7_ERR_ARG;
  if (ms_total) *ms_total = ctx->stage_ms[stage];
  if (launches) *launches = ctx->stage_calls[stage];
  return 0;
}
int64_t b7_launch_count(b7_ctx* ctx) { return ctx ? ctx->launches : 0; }

/* ------------------------------------------------------------------ grids */

int b7_sobol_directions(int dims, uint32_t* out) {
  if (dims < 1 || dims >= B7_MAX_DIMS || !out) { b7_set_error("sobol: dims must satisfy 1 <= dims < 40"); return B7_ERR_ARG; }
  b7_sobol_directions_host(dims, out);
  return 0;
}

int b7_sobol_generate(b7_ctx* ctx, int dims, int64_t first_seed, int64_t count, const double* mins,
                      const double* maxes, double* out_host, b7_grid** out_grid) {
  if (!ctx) return B7_ERR_ARG;
  if (out_grid) *out_grid = nullptr;
  // grids/sobol.lua:36 assert(dims < max_dims); :318-324 "Too many calls" beyond 2^30 points
  if (dims < 1 || dims >= B7_MAX_DIMS) { b7_set_error("sobol: dims must satisfy 1 <= dims < 40"); return B7_ERR_ARG; }
  if (first_seed < 0) first_seed = 0;   // grids/sobol.lua:291 seed = max(0, floor(seed))
  if (count < 0 || first_seed + count > (1LL << B7_SOBOL_BITS)) { b7_set_error("sobol: too many calls (seed range exceeds 2^30)"); return B7_ERR_ARG; }
  if ((mins == nullptr) != (maxes == nullptr)) { b7_set_error("sobol: one-sided rescaling is done by the host wrapper; pass both mins and maxes or neither"); return B7_ERR_ARG; }
  B7_CUDA(cudaSetDevice(ctx->device));
  double* dev = nullptr;
  B7_CHECK(dev_alloc(ctx, &dev, (size_t)count * dims));
  double *dmin = nullptr, *dscale = nullptr;
  if (mins) {
    double h[2 * B7_MAX_DIMS];
    for (int i = 0; i < dims; ++i) { h[i] = mins[i]; h[B7_MAX_DIMS + i] = maxes[i] + (-mins[i]); }   // torch.add(maxes, -mins)
    B7_CHECK(dev_alloc(ctx, &dmin, 2 * B7_MAX_DIMS));
    dscale = dmin + B7_MAX_DIMS;
    B7_CUDA(cudaMemcpyAsync(dmin, h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
    B7_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  StageTimer t(ctx, ST_SOBOL);
  int rc = b7_launch_sobol(ctx, dims, first_seed, count, dmin, dscale, dev);
  t.stop(1);
  if (rc == 0 && out_host && count > 0) {
    cudaError_t e = cudaMemcpyAsync(out_host, dev, (size_t)count * dims * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e != cudaSuccess) { b7_set_error("sobol D2H: %s", cudaGetErrorString(e)); rc = B7_ERR_CUDA; }
  }
  cudaError_t e = cudaStreamSynchronize(ctx->stream);
  if (rc == 0 && e != cudaSuccess) { b7_set_error("sobol: %s", cudaGetErrorString(e)); rc = B7_ERR_CUDA; }
  dev_free(ctx, dmin);
  if (rc != 0 || !out_grid) { dev_free(ctx, dev); return rc; }
  b7_grid* g = new b7_grid();
  g->ctx = ctx; g->rows = count; g->d = dims; g->X = dev;
  *out_grid = g;
  return 0;
}

int b7_grid_from_host(b7_ctx* ctx, const double* X, int64_t M, int d, b7_grid** out_grid) {
  if (!ctx || !out_grid || M < 0 || d < 1 || (M > 0 && !X)) { b7_set_error("grid_from_host: bad arguments"); return B7_ERR_ARG; }
  *out_grid = nullptr;
  B7_CUDA(cudaSetDevice(ctx->device));
  double* dev = nullptr;
  B7_CHECK(dev_alloc(ctx, &dev, (size_t)M * d));
  if (M > 0) {
    B7_CUDA(cudaMemcpyAsync(dev, X, (size_t)M * d * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    B7_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  b7_grid* g = new b7_grid();
  g->ctx = ctx; g->rows = M; g->d = d; g->X = dev;
  *out_grid = g;
  return 0;
}

int b7_grid_read(b7_grid* g, int64_t first_row, int64_t count, double* out_host) {
  if (!g || first_row < 0 || count < 0 || first_row + count > g->rows || (count > 0 && !out_host)) { b7_set_error("grid_read: range"); return B7_ERR_ARG; }
  B7_CUDA(cudaSetDevice(g->ctx->device));
  if (count == 0) return 0;
  B7_CUDA(cudaMemcpyAsync(out_host, g->X + first_row * g->d, (size_t)count * g->d * sizeof(double), cudaMemcpyDeviceToHost, g->ctx->stream));
  B7_CUDA(cudaStreamSynchronize(g->ctx->stream));
  return 0;
}

int64_t b7_grid_size(b7_grid* g) { return g ? g->rows - (int64_t)g->removed.size() : 0; }
int64_t b7_grid_rows(b7_grid* g) { return g ? g->rows : 0; }
int b7_grid_dims(b7_grid* g) { return g ? g->d : 0; }

// compacted 1-based index -> original 0-based row: the smallest r with r - #removed(<= r) == c-1
static int64_t compacted_to_original(const b7_grid* g, int64_t c1) {
  int64_t r = c1 - 1;
  for (int64_t t : g->removed) {   // removed is sorted ascending
    if (t <= r) ++r; else break;
  }
  return r;
}

int b7_grid_original_index(b7_grid* g, int64_t compacted_index, int64_t* original_index_1based) {
  if (!g || compacted_index < 1 || compacted_index > b7_grid_size(g)) { b7_set_error("grid: compacted index out of range"); return B7_ERR_ARG; }
  if (original_index_1based) *original_index_1based = compacted_to_original(g, compacted_index) + 1;
  return 0;
}

int b7_grid_remove(b7_grid* g, int64_t compacted_index, double* removed_row) {
  if (!g || compacted_index < 1 || compacted_index > b7_grid_size(g)) { b7_set_error("grid_remove: index out of range"); return B7_ERR_ARG; }
  int64_t r = compacted_to_original(g, compacted_index);
  if (removed_row) B7_CHECK(b7_grid_read(g, r, 1, removed_row));
  g->removed.insert(std::upper_bound(g->removed.begin(), g->removed.end(), r), r);
  g->removed_dirty = true;
  return 0;
}

void b7_grid_free(b7_grid* g) {
  if (!g) return;
  cudaSetDevice(g->ctx->device);
  dev_free(g->ctx, g->X);
  dev_free(g->ctx, g->removed_dev);
  delete g;
}

/* ------------------------------------------------------------------ GP */

void b7_gp_free(b7_gp* gp) {
  if (!gp) return;
  cudaSetDevice(gp->ctx->device);
  cudaStreamSynchronize(gp->ctx->stream);
  void* ptrs[] = {gp->X, gp->Xt, gp->y, gp->par, gp->fac, gp->facS, gp->sigma, gp->dinv, gp->dinvT, gp->beta, gp->alpha, gp->tt, gp->logdet, gp->info, gp->meta_dev, gp->step_io};
  for (void* p : ptrs) dev_free(gp->ctx, p);
  if (gp->potrf_graph) cudaGraphExecDestroy(gp->potrf_graph);
  delete gp;
}

int b7_gp_num_draws(b7_gp* gp) { return gp ? gp->S : 0; }
int b7_gp_num_obs(b7_gp* gp) { return gp ? gp->N : 0; }
int b7_gp_padded_n(b7_gp* gp) { return gp ? gp->Np : 0; }

static int gp_retry_draw(b7_gp* gp, int s, int first_info);

// parameters per draw (oracle/SPEC.md): w = exp(-log l), sf2 = exp(2 log sf), sn2 = exp(2 log sn)
static void set_hypers_host(b7_gp* gp, const double* hyp) {
  const int d = gp->d, H = d + 3, S = gp->S;
  gp->par_host.assign((size_t)S * kParStride, 0.0);
  for (int s = 0; s < S; ++s) {
    const double* h = hyp + (size_t)s * H;
    double* p = gp->par_host.data() + (size_t)s * kParStride;
    for (int i = 0; i < d; ++i) p[i] = exp(-h[i]);
    const double sf2 = exp(2.0 * h[d]), sn2 = exp(2.0 * h[d + 1]);
    p[B7_MAX_DIMS] = sf2;
    p[B7_MAX_DIMS + 1] = sn2 + (gp->noiseless ? 1e-8 * sf2 : 0.0);
    p[B7_MAX_DIMS + 2] = h[d + 2];
    p[B7_MAX_DIMS + 3] = sn2;
  }
}

static void residuals_host(b7_gp* gp, const std::vector<double>& y, std::vector<double>& r) {
  r.assign((size_t)gp->S * gp->Np, 0.0);
  for (int s = 0; s < gp->S; ++s) {
    const double m = gp->par_host[(size_t)s * kParStride + B7_MAX_DIMS + 2];
    for (int i = 0; i < gp->N; ++i) r[(size_t)s * gp->Np + i] = y[i] - m;
  }
}

int b7_gp_fit_range(b7_gp* gp, int s0, int count, int* info, double* logml, double* jitter) {
  if (!gp || s0 < 0 || count < 0 || s0 + count > gp->S) { b7_set_error("gp_fit_range: draw range"); return B7_ERR_ARG; }
  b7_ctx* ctx = gp->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  if (count == 0) return 0;
  B7_CHECK(build_kxx(gp, s0, count));
  B7_CHECK(factor(gp, s0, count));
  std::vector<int> inf((size_t)count);
  B7_CUDA(cudaMemcpyAsync(inf.data(), gp->info + s0, count * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < count; ++i) {
    gp->jitter[s0 + i] = 0.0;
    gp->info_host[s0 + i] = 0;
    if (inf[i] != 0) B7_CHECK(gp_retry_draw(gp, s0 + i, inf[i]));   // utils/math.lua:168-216
  }
  // log marginal likelihood: -1/2 beta^T beta - sum log L_ii - N/2 log 2pi  (r^T K^-1 r = |L^-1 r|^2)
  std::vector<double> bh((size_t)count * gp->Np), ldh((size_t)count);
  B7_CUDA(cudaMemcpyAsync(bh.data(), gp->beta + (size_t)s0 * gp->Np, bh.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  B7_CUDA(cudaMemcpyAsync(ldh.data(), gp->logdet + s0, count * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < count; ++i) {
    double q = 0.0;
    for (int k = 0; k < gp->N; ++k) q += bh[(size_t)i * gp->Np + k] * bh[(size_t)i * gp->Np + k];
    gp->logml_host[s0 + i] = -0.5 * q - ldh[i] - 0.5 * gp->N * kLog2Pi;
  }
  for (int i = 0; i < count; ++i) {
    if (info) info[i] = gp->info_host[s0 + i];
    if (logml) logml[i] = gp->logml_host[s0 + i];
    if (jitter) jitter[i] = gp->jitter[s0 + i];
  }
  return 0;
}

// utils.math.chol retry policy (utils/math.lua:168-216) for one draw whose plain factorisation failed
static int gp_retry_draw(b7_gp* gp, int s, int first_info) {
  b7_ctx* ctx = gp->ctx;
  const size_t fs = (size_t)gp->Np * gp->Np;
  double* par_s = gp->par + (size_t)s * kParStride;
  const double diag0 = gp->par_host[(size_t)s * kParStride + B7_MAX_DIMS + 1];
  // max_eps = ||src||_F of the matrix that failed
  B7_CHECK(build_kxx(gp, s, 1));
  double* rows = nullptr;
  B7_CHECK(dev_alloc(ctx, &rows, (size_t)gp->N));
  frob_rows_kernel<<<gp->N, 256, 0, ctx->stream>>>(gp->fac + s * fs, gp->Np, gp->N, rows);
  b7_count(ctx);
  std::vector<double> rh((size_t)gp->N);
  B7_CUDA(cudaMemcpyAsync(rh.data(), rows, gp->N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  dev_free(ctx, rows);
  double ss = 0.0;
  for (double v : rh) ss += v;
  const double max_eps = sqrt(ss);
  double eps = 1e-8;
  const double growth = 1.1;
  while (true) {
    // a non-finite norm (NaN / inf entries, e.g. sigma_f^2 = exp(2 * 800)) can never be repaired by jitter and `eps > inf` never
    // becomes true: give up at once (the reference's loop would not terminate; declared deviation, oracle/SPEC.md)
    if (eps > max_eps || !std::isfinite(max_eps)) {
      // chol(I): L = I, beta = r, logdet = 0
      identity_kernel<<<(unsigned)((fs + 255) / 256), 256, 0, ctx->stream>>>(gp->fac + s * fs, gp->Np);
      b7_count(ctx);
      B7_CHECK(upload_residual(gp, s, gp->y_host));
      B7_CHECK(factor(gp, s, 1));
      gp->jitter[s] = INFINITY;
      gp->info_host[s] = first_info;
      return 0;
    }
    eps *= growth;
    double d = diag0 + eps;
    B7_CUDA(cudaMemcpyAsync(par_s + B7_MAX_DIMS + 1, &d, sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    B7_CUDA(cudaStreamSynchronize(ctx->stream));
    B7_CHECK(build_kxx(gp, s, 1));
    B7_CHECK(upload_residual(gp, s, gp->y_host));
    B7_CHECK(factor(gp, s, 1));
    int inf = 0;
    B7_CUDA(cudaMemcpyAsync(&inf, gp->info + s, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    B7_CUDA(cudaStreamSynchronize(ctx->stream));
    if (inf == 0) {
      gp->jitter[s] = eps;
      gp->info_host[s] = 0;
      // leave the nominal diagonal in par (posterior uses sf2 only)
      B7_CUDA(cudaMemcpyAsync(par_s + B7_MAX_DIMS + 1, &diag0, sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
      B7_CUDA(cudaStreamSynchronize(ctx->stream));
      return 0;
    }
  }
}

// the INT8 path keeps exact int32 sums only up to B7_I8_MAX_NP observations; larger fits stay on the FP64 DMMA kernel
static bool i8_path(const b7_gp* gp) { return gp->ctx->use_i8 && gp->Np <= B7_I8_MAX_NP; }

// INT8 path: slice L^-1 (allocated on first use)
static int gp_slice(b7_gp* gp, int s0, int count) {
  b7_ctx* ctx = gp->ctx;
  if (!gp->facS) {
    B7_CHECK(dev_alloc(ctx, &gp->facS, (size_t)gp->S * b7_i8_facs_stride(gp->Np)));
    B7_CHECK(dev_alloc(ctx, &gp->sigma, (size_t)gp->S * gp->Np));
  }
  B7_CHECK(b7_i8_slice_factor(ctx, gp->fac, gp->Np, gp->facS, gp->sigma, s0, count));
  for (int s = s0; s < s0 + count; ++s) gp->sliced[s] = 1;
  return 0;
}

static int gp_invert(b7_gp* gp, int s0, int count) {
  b7_ctx* ctx = gp->ctx;
  if (count <= 0) return 0;            // a rank of a sharded fit that owns no draw (S < number of GPUs)
  StageTimer t(ctx, ST_TRTRI);
  int64_t before = ctx->launches;
  // alpha = L^-T beta while L is still there (the INT8 path's mean is the fp64 dot product k*^T alpha)
  if (gp->Np <= B7_I8_MAX_NP) B7_CHECK(b7_launch_alpha(gp, s0, count, false));
  B7_CHECK(b7_launch_trtri(gp, s0, count));
  for (int s = s0; s < s0 + count; ++s) gp->sliced[s] = 0;
  if (i8_path(gp)) B7_CHECK(gp_slice(gp, s0, count));
  t.stop((int)(ctx->launches - before));
  return 0;
}

int b7_gp_mark_ready(b7_gp* gp) {
  if (!gp) return B7_ERR_ARG;
  // slots filled by the host (all-gather into fac, which already is the layout the posterior pass reads)
  std::fill(gp->sliced.begin(), gp->sliced.end(), 0);
  if (i8_path(gp)) {
    B7_CUDA(cudaSetDevice(gp->ctx->device));
    B7_CHECK(b7_launch_alpha(gp, 0, gp->S, true));      // the factors arrive inverted: alpha = (L^-1)^T beta
    B7_CHECK(gp_slice(gp, 0, gp->S));
    B7_CUDA(cudaStreamSynchronize(gp->ctx->stream));
  }
  gp->ready = true;
  gp->inverted = true;
  return 0;
}

}  // extern "C"

// sharded fit: own draws [s0, s0 + count) are factorised and inverted; make sure every buffer of the exchange exists
// and publish (info, log ml, jitter) of the own draws in device memory
int b7_gp_prepare_gather(b7_gp* gp, int s0, int count) {
  b7_ctx* ctx = gp->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  if (i8_path(gp) && !gp->facS) {
    B7_CHECK(dev_alloc(ctx, &gp->facS, (size_t)gp->S * b7_i8_facs_stride(gp->Np)));
    B7_CHECK(dev_alloc(ctx, &gp->sigma, (size_t)gp->S * gp->Np));
  }
  if (!gp->meta_dev) B7_CHECK(dev_alloc(ctx, &gp->meta_dev, (size_t)gp->S * 3));
  std::vector<double> m((size_t)std::max(count, 1) * 3);
  for (int i = 0; i < count; ++i) {
    m[3 * i] = (double)gp->info_host[s0 + i];
    m[3 * i + 1] = gp->logml_host[s0 + i];
    m[3 * i + 2] = gp->jitter[s0 + i];
  }
  if (count > 0) B7_CUDA(cudaMemcpyAsync(gp->meta_dev + 3 * (size_t)s0, m.data(), (size_t)count * 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  return 0;
}

int b7_gp_finish_gather(b7_gp* gp, bool slices_exchanged) {
  b7_ctx* ctx = gp->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  std::vector<double> m((size_t)gp->S * 3);
  B7_CUDA(cudaMemcpyAsync(m.data(), gp->meta_dev, m.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  for (int s = 0; s < gp->S; ++s) {
    gp->info_host[s] = (int)m[3 * s];
    gp->logml_host[s] = m[3 * s + 1];
    gp->jitter[s] = m[3 * s + 2];
  }
  std::fill(gp->sliced.begin(), gp->sliced.end(), slices_exchanged ? 1 : 0);
  gp->fac_complete = !slices_exchanged;
  gp->ready = true;
  gp->inverted = true;
  return 0;
}

extern "C" {

int b7_gp_fit(b7_ctx* ctx, int kernel, const double* X, const double* y, int N, int d, const double* hyp, int S,
              int H, int noiseless, int flags, b7_gp** out, int* info, double* logml, double* jitter) {
  if (!ctx || !out) { b7_set_error("gp_fit: null ctx/out"); return B7_ERR_ARG; }
  *out = nullptr;
  if (!X || !y || !hyp || N < 1 || d < 1 || d >= B7_MAX_DIMS || S < 1 || H != d + 3 ||
      (kernel != B7_KERNEL_ARDSE && kernel != B7_KERNEL_MATERN52)) {
    b7_set_error("gp_fit: bad arguments (N=%d d=%d S=%d H=%d kernel=%d; H must be d+3, d < 40)", N, d, S, H, kernel);
    return B7_ERR_ARG;
  }
  B7_CUDA(cudaSetDevice(ctx->device));
  b7_gp* gp = new b7_gp();
  gp->ctx = ctx; gp->kernel = kernel; gp->N = N; gp->d = d; gp->S = S; gp->noiseless = noiseless;
  gp->Np = (int)pad128(N); gp->NB = gp->Np / B7_NB;
  gp->jitter.assign(S, 0.0); gp->info_host.assign(S, 0); gp->logml_host.assign(S, 0.0); gp->sliced.assign(S, 0);
  const size_t Np = gp->Np, fs = Np * Np, ds = (size_t)gp->NB * B7_NB * B7_NB;
  int rc = 0;
  auto fail = [&](int code) { b7_gp_free(gp); return code; };
  if ((rc = dev_alloc(ctx, &gp->X, (size_t)N * d)) || (rc = dev_alloc(ctx, &gp->Xt, (size_t)d * Np)) || (rc = dev_alloc(ctx, &gp->y, (size_t)N)) ||
      (rc = dev_alloc(ctx, &gp->par, (size_t)S * kParStride)) || (rc = dev_alloc(ctx, &gp->fac, (size_t)S * fs)) ||
      (rc = dev_alloc(ctx, &gp->dinv, (size_t)S * ds)) || (rc = dev_alloc(ctx, &gp->dinvT, (size_t)S * ds)) ||
      (rc = dev_alloc(ctx, &gp->beta, (size_t)S * Np)) || (rc = dev_alloc(ctx, &gp->alpha, (size_t)S * Np)) ||
      (rc = dev_alloc(ctx, &gp->tt, (size_t)S * B7_NB * Np)) ||
      (rc = dev_alloc(ctx, &gp->logdet, (size_t)S)) || (rc = dev_alloc(ctx, &gp->info, (size_t)S)))
    return fail(rc);
  // diag_kernel only writes the lower triangles of the inverted diagonal blocks: the zeros above them are set here, once
  if (cudaMemsetAsync(gp->dinv, 0, (size_t)S * ds * sizeof(double), ctx->stream) != cudaSuccess) return fail(B7_ERR_CUDA);
  gp->y_host.assign(y, y + N);
  set_hypers_host(gp, hyp);
  std::vector<double> xt((size_t)d * Np, 0.0), r;
  for (int i = 0; i < N; ++i)
    for (int k = 0; k < d; ++k) xt[(size_t)k * Np + i] = X[(size_t)i * d + k];
  residuals_host(gp, gp->y_host, r);
  cudaStream_t st = ctx->stream;
  cudaError_t e;
  if ((e = cudaMemcpyAsync(gp->X, X, (size_t)N * d * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
      (e = cudaMemcpyAsync(gp->Xt, xt.data(), xt.size() * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
      (e = cudaMemcpyAsync(gp->y, y, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
      (e = cudaMemcpyAsync(gp->par, gp->par_host.data(), gp->par_host.size() * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
      (e = cudaMemcpyAsync(gp->beta, r.data(), r.size() * sizeof(double), cudaMemcpyHostToDevice, st)) != cudaSuccess ||
      (e = cudaStreamSynchronize(st)) != cudaSuccess) {
    b7_set_error("gp_fit upload: %s", cudaGetErrorString(e));
    return fail(B7_ERR_CUDA);
  }
  if (flags == B7_FIT_DEFER) { *out = gp; return 0; }
  if ((rc = b7_gp_fit_range(gp, 0, S, info, logml, jitter)) < 0) return fail(rc);
  if (flags == B7_FIT_PREDICT) {
    if ((rc = gp_invert(gp, 0, S)) < 0) return fail(rc);
    gp->inverted = true;
  }
  if ((e = cudaStreamSynchronize(st)) != cudaSuccess) { b7_set_error("gp_fit: %s", cudaGetErrorString(e)); return fail(B7_ERR_CUDA); }
  gp->ready = true;
  *out = gp;
  return 0;
}

// Same observations, new hyper-parameter draws: the slice sampler's density evaluation
// (samplers/slice.lua:100-103) with X, y and every buffer resident -- only S x H doubles go in and
// S log-likelihoods come out.
int b7_gp_refit(b7_gp* gp, const double* hyp, int flags, int* info, double* logml, double* jitter) {
  if (!gp || !hyp || (flags != B7_FIT_PREDICT && flags != B7_FIT_LOGML_ONLY)) { b7_set_error("gp_refit: bad arguments"); return B7_ERR_ARG; }
  b7_ctx* ctx = gp->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  set_hypers_host(gp, hyp);
  std::vector<double> r;
  residuals_host(gp, gp->y_host, r);
  gp->ready = false; gp->inverted = false;
  B7_CUDA(cudaMemcpyAsync(gp->par, gp->par_host.data(), gp->par_host.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  B7_CUDA(cudaMemcpyAsync(gp->beta, r.data(), r.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  B7_CHECK(b7_gp_fit_range(gp, 0, gp->S, info, logml, jitter));
  if (flags == B7_FIT_PREDICT) {
    B7_CHECK(gp_invert(gp, 0, gp->S));
    gp->inverted = true;
  }
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  gp->ready = true;
  return 0;
}

// One directed slice step in one launch (slice_step.cu): the random numbers go in, the new point comes out.
int b7_gp_slice_step(b7_gp* gp, const double* x0, const double* dir, double log_u_level, const double* u_right,
                     const double* u_shrink, int K, double width, double max_step, double prior_std, int prior_order,
                     double* x1, int* n_shrink_used, int* n_evals, double* logp_x1) {
  if (!gp || !x0 || !dir || !u_right || K < 0 || (K > 0 && !u_shrink) || !x1 || (prior_order != 0 && prior_order != 1)) {
    b7_set_error("gp_slice_step: bad arguments");
    return B7_ERR_ARG;
  }
  if (gp->N > B7_NB) {
    b7_set_error("gp_slice_step: %d observations; the one-launch step takes at most %d", gp->N, B7_NB);
    return B7_ERR_ARG;
  }
  if (!(width > 0.0) || !std::isfinite(width)) {
    b7_set_error("gp_slice_step: width %g is not a finite positive number", width);
    return B7_ERR_ARG;
  }
  b7_ctx* ctx = gp->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  const int H = gp->d + 3;
  std::vector<double> in((size_t)3 * H + K), out((size_t)H + 4);
  std::copy(x0, x0 + H, in.begin());
  std::copy(dir, dir + H, in.begin() + H);
  std::copy(u_right, u_right + H, in.begin() + 2 * H);
  if (K > 0) std::copy(u_shrink, u_shrink + K, in.begin() + 3 * H);
  B7_CHECK(grow(ctx, &gp->step_io, &gp->step_io_bytes, (in.size() + out.size()) * sizeof(double)));
  B7_CUDA(cudaMemcpyAsync(gp->step_io, in.data(), in.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  B7_CHECK(b7_launch_slice_step(gp, gp->step_io, K, log_u_level, width, max_step, prior_std, prior_order));
  B7_CUDA(cudaMemcpyAsync(out.data(), gp->step_io + in.size(), out.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  if (out[H + 3] != 0.0) {
    b7_set_error("gp_slice_step: the %d shrink uniforms ran out; call again with more", K);
    return B7_ERR_STATE;
  }
  std::copy(out.begin(), out.begin() + H, x1);
  if (logp_x1) *logp_x1 = out[H];
  if (n_shrink_used) *n_shrink_used = (int)out[H + 1];
  if (n_evals) *n_evals = (int)out[H + 2];
  return 0;
}

int b7_gp_invert_range(b7_gp* gp, int s0, int count) {   // used with B7_FIT_DEFER
  if (!gp || s0 < 0 || count < 0 || s0 + count > gp->S) return B7_ERR_ARG;
  B7_CUDA(cudaSetDevice(gp->ctx->device));
  B7_CHECK(gp_invert(gp, s0, count));
  B7_CUDA(cudaStreamSynchronize(gp->ctx->stream));
  return 0;
}

int b7_gp_device_ptr(b7_gp* gp, int what, void** ptr, int64_t* bytes) {
  if (!gp || !ptr) return B7_ERR_ARG;
  const int64_t Np = gp->Np;
  switch (what) {
    case 0: *ptr = gp->fac; if (bytes) *bytes = (int64_t)gp->S * Np * Np * 8; return 0;
    case 1: *ptr = gp->beta; if (bytes) *bytes = (int64_t)gp->S * Np * 8; return 0;
    case 2: *ptr = gp->dinv; if (bytes) *bytes = (int64_t)gp->S * gp->NB * B7_NB * B7_NB * 8; return 0;
    default: b7_set_error("gp_device_ptr: what=%d", what); return B7_ERR_ARG;
  }
}

int b7_gp_read_factor(b7_gp* gp, int s, double* out_host) {
  if (!gp || !out_host || s < 0 || s >= gp->S) return B7_ERR_ARG;
  B7_CUDA(cudaSetDevice(gp->ctx->device));
  double* tmp = nullptr;
  B7_CHECK(dev_alloc(gp->ctx, &tmp, (size_t)gp->N * gp->N));
  int rc = b7_launch_untile(gp->ctx, gp->fac + (size_t)s * gp->Np * gp->Np, tmp, gp->Np, gp->N);
  cudaError_t e = cudaMemcpyAsync(out_host, tmp, (size_t)gp->N * gp->N * 8, cudaMemcpyDeviceToHost, gp->ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(gp->ctx->stream);
  dev_free(gp->ctx, tmp);
  if (rc < 0) return rc;
  if (e != cudaSuccess) { b7_set_error("gp_read_factor: %s", cudaGetErrorString(e)); return B7_ERR_CUDA; }
  return 0;
}

// posterior of draw s over `rows` device points (A: rows x d) -> mean/var device arrays (rows_pad long)
static int posterior_panel(b7_gp* gp, int s, const double* A, int64_t rows, double* mean, double* var) {
  b7_ctx* ctx = gp->ctx;
  const int64_t rp = pad128(rows);
  B7_CHECK(grow(ctx, &ctx->ks, &ctx->ks_bytes, (size_t)rp * gp->Np * 8));
  const double* p = gp->par_host.data() + (size_t)s * kParStride;
  if (!gp->fac_complete && (!i8_path(gp) || !gp->sliced[s])) {
    b7_set_error("gp: this handle came from a sharded fit that exchanged the int8 slices only; refit to use the FP64 path");
    return B7_ERR_STATE;
  }
  if (i8_path(gp)) {
    if (!gp->sliced[s]) B7_CHECK(gp_slice(gp, s, 1));     // the path was switched after the fit
    // error-free sliced operands on the INT8 tensor pipe (posterior_i8.cu); K* needs no max: 0 < k* <= sf2 <= tau
    int e = 0;
    frexp(p[B7_MAX_DIMS], &e);
    const double tau = ldexp(1.0, e);
    const int64_t rp64 = (rows + 63) / 64 * 64;
    int8_t* ksS = reinterpret_cast<int8_t*>(ctx->ks);
    B7_CHECK(grow(ctx, &ctx->i8_partial, &ctx->i8_partial_bytes, b7_i8_partial_bytes(gp->Np, rp64)));
    {
      StageTimer t(ctx, ST_KSTAR);
      B7_CHECK(b7_i8_cov_slices(ctx, ctx->stream, gp->kernel, A, rows, rp64, gp->d, gp->Xt, gp->N, gp->Np, gp->par + (size_t)s * kParStride, tau,
                                gp->alpha + (size_t)s * gp->Np, ksS, b7_i8_mean_partials(ctx->i8_partial, gp->Np, rp64)));
      t.stop(1);
    }
    StageTimer t(ctx, ST_POSTERIOR);
    B7_CHECK(b7_launch_posterior_i8(ctx, gp->facS + (size_t)s * b7_i8_facs_stride(gp->Np), gp->sigma + (size_t)s * gp->Np, gp->Np, ksS, A, rows,
                                    gp->d, gp->Xt, gp->par + (size_t)s * kParStride, gp->kernel, rp64, tau, p[B7_MAX_DIMS], p[B7_MAX_DIMS + 2],
                                    ctx->i8_partial, mean, var));
    t.stop(1);   // one posterior pass (the few-microsecond finish kernel rides along)
    return 0;
  }
  {
    StageTimer t(ctx, ST_KSTAR);
    B7_CHECK(b7_launch_cov_batched(ctx, gp->kernel, A, rows, rp, gp->d, gp->Xt, gp->N, gp->Np,
                                   gp->par + (size_t)s * kParStride, 0, ctx->ks, 0, 1, false, true));
    t.stop(1);
  }
  {
    StageTimer t(ctx, ST_POSTERIOR);
    B7_CHECK(b7_launch_posterior(ctx, gp->fac + (size_t)s * gp->Np * gp->Np, gp->beta + (size_t)s * gp->Np, gp->Np, ctx->ks,
                                 rp, p[B7_MAX_DIMS], p[B7_MAX_DIMS + 2], mean, var));
    t.stop(1);
  }
  return 0;
}

// All S draws of one candidate panel on the INT8 path with the K* pass of draw s + 1 (FP64 / integer pipes, second
// stream) running under the posterior pass of draw s (tensor pipe, main stream): two sets of K* slices and partials.
// Used when stage profiling is off (the stage timers need the two passes one after the other).
static int posterior_panel_draws_i8(b7_gp* gp, const double* A, int64_t rows, double* dm, double* dv, int64_t ld) {
  b7_ctx* ctx = gp->ctx;
  const int S = gp->S;
  const int64_t rp64 = (rows + 63) / 64 * 64;
  const size_t ks_bytes = ((size_t)rp64 * gp->Np * B7_I8_SLICES + 255) / 256 * 256;
  const size_t part_bytes = (b7_i8_partial_bytes(gp->Np, rp64) + 255) / 256 * 256;
  B7_CHECK(grow(ctx, &ctx->ks, &ctx->ks_bytes, 2 * ks_bytes));
  B7_CHECK(grow(ctx, &ctx->i8_partial, &ctx->i8_partial_bytes, 2 * part_bytes));
  for (int s = 0; s < S; ++s)
    if (!gp->sliced[s]) B7_CHECK(gp_slice(gp, s, 1));
  auto tau_of = [&](int s) {
    int e = 0;
    frexp(gp->par_host[(size_t)s * kParStride + B7_MAX_DIMS], &e);
    return ldexp(1.0, e);
  };
  auto ks_of = [&](int s) { return reinterpret_cast<int8_t*>(ctx->ks) + (size_t)(s & 1) * ks_bytes; };
  auto part_of = [&](int s) { return reinterpret_cast<double*>(reinterpret_cast<char*>(ctx->i8_partial) + (size_t)(s & 1) * part_bytes); };
  auto kstar = [&](int s) {
    return b7_i8_cov_slices(ctx, ctx->stream2, gp->kernel, A, rows, rp64, gp->d, gp->Xt, gp->N, gp->Np, gp->par + (size_t)s * kParStride, tau_of(s),
                            gp->alpha + (size_t)s * gp->Np, ks_of(s), b7_i8_mean_partials(part_of(s), gp->Np, rp64));
  };
  // the second stream starts after everything already queued on the main one (the grid, the factors)
  B7_CUDA(cudaEventRecord(ctx->evA, ctx->stream));
  B7_CUDA(cudaStreamWaitEvent(ctx->stream2, ctx->evA, 0));
  B7_CHECK(kstar(0));
  B7_CUDA(cudaEventRecord(ctx->evK[0], ctx->stream2));
  for (int s = 0; s < S; ++s) {
    if (s + 1 < S) {
      if (s >= 1) B7_CUDA(cudaStreamWaitEvent(ctx->stream2, ctx->evP[(s + 1) & 1], 0));   // posterior s - 1 has released that set
      B7_CHECK(kstar(s + 1));
      B7_CUDA(cudaEventRecord(ctx->evK[(s + 1) & 1], ctx->stream2));
    }
    B7_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->evK[s & 1], 0));
    const double* p = gp->par_host.data() + (size_t)s * kParStride;
    B7_CHECK(b7_launch_posterior_i8(ctx, gp->facS + (size_t)s * b7_i8_facs_stride(gp->Np), gp->sigma + (size_t)s * gp->Np, gp->Np, ks_of(s), A, rows,
                                    gp->d, gp->Xt, gp->par + (size_t)s * kParStride, gp->kernel, rp64, tau_of(s), p[B7_MAX_DIMS], p[B7_MAX_DIMS + 2],
                                    part_of(s), dm + (size_t)s * ld, dv + (size_t)s * ld));
    B7_CUDA(cudaEventRecord(ctx->evP[s & 1], ctx->stream));
  }
  return 0;
}

static bool all_sliced_or_sliceable(const b7_gp* gp) {
  if (gp->fac_complete) return true;
  for (char c : gp->sliced) if (!c) return false;
  return true;
}

static int require_predict_state(b7_gp* gp) {
  if (!gp->ready || !gp->inverted) {
    b7_set_error("gp: factor not inverted (fit with B7_FIT_PREDICT, or b7_gp_invert_range + b7_gp_mark_ready)");
    return B7_ERR_STATE;
  }
  return 0;
}

int b7_gp_predict(b7_gp* gp, int s, const double* Xs, int64_t M, double* mean, double* var) {
  if (!gp || s < 0 || s >= gp->S || M < 0 || (M > 0 && (!Xs || !mean || !var))) { b7_set_error("gp_predict: bad arguments"); return B7_ERR_ARG; }
  B7_CHECK(require_predict_state(gp));
  b7_ctx* ctx = gp->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  const int64_t P = panel_rows(ctx, gp->Np);
  B7_CHECK(grow(ctx, &ctx->xs_stage, &ctx->xs_bytes, (size_t)std::min(P, pad128(M)) * gp->d * 8));
  B7_CHECK(grow(ctx, &ctx->moments, &ctx->moments_bytes, (size_t)2 * std::min(P, pad128(M)) * 8));
  for (int64_t c0 = 0; c0 < M; c0 += P) {
    const int64_t n = std::min(P, M - c0), np = pad128(n);
    B7_CUDA(cudaMemcpyAsync(ctx->xs_stage, Xs + c0 * gp->d, (size_t)n * gp->d * 8, cudaMemcpyHostToDevice, ctx->stream));
    double* dm = ctx->moments; double* dv = ctx->moments + np;
    B7_CHECK(posterior_panel(gp, s, ctx->xs_stage, n, dm, dv));
    B7_CUDA(cudaMemcpyAsync(mean + c0, dm, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    B7_CUDA(cudaMemcpyAsync(var + c0, dv, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    B7_CUDA(cudaStreamSynchronize(ctx->stream));
  }
  return 0;
}

/* ------------------------------------------------------------------ acquisition */

struct PartBuf {
  b7_ctx* ctx = nullptr;
  double* best = nullptr; int64_t* idx = nullptr; int64_t* nan = nullptr; int cap = 0;
  explicit PartBuf(b7_ctx* c) : ctx(c) {}
  ~PartBuf() { dev_free(ctx, best); dev_free(ctx, idx); dev_free(ctx, nan); }
};

static int finish_argmax(b7_ctx* ctx, PartBuf& pb, int n_parts, double* best, int64_t* row0based, int64_t* nan_count) {
  std::vector<double> hb((size_t)n_parts); std::vector<int64_t> hi((size_t)n_parts), hn((size_t)n_parts);
  if (n_parts > 0) {
    B7_CUDA(cudaMemcpyAsync(hb.data(), pb.best, n_parts * 8, cudaMemcpyDeviceToHost, ctx->stream));
    B7_CUDA(cudaMemcpyAsync(hi.data(), pb.idx, n_parts * 8, cudaMemcpyDeviceToHost, ctx->stream));
    B7_CUDA(cudaMemcpyAsync(hn.data(), pb.nan, n_parts * 8, cudaMemcpyDeviceToHost, ctx->stream));
  }
  B7_CUDA(cudaStreamSynchronize(ctx->stream));
  double bv = -INFINITY; int64_t bi = INT64_MAX, nn = 0;
  for (int p = 0; p < n_parts; ++p) {
    nn += hn[p];
    if (hi[p] == INT64_MAX) continue;
    if (hb[p] > bv || (hb[p] == bv && hi[p] < bi)) { bv = hb[p]; bi = hi[p]; }
  }
  if (bi == INT64_MAX) { *best = NAN; *row0based = -1; } else { *best = bv; *row0based = bi; }
  *nan_count = nn;
  return 0;
}

int b7_acq_score_range(b7_gp* gp, b7_grid* grid, int64_t row0, int64_t count, int kind, double tradeoff, int bound,
                       double sign, double fmin, double* score_host, int64_t* argmax_original, double* best,
                       int64_t* nan_count) {
  if (!gp || !grid || row0 < 0 || count < 0 || row0 + count > grid->rows || grid->d != gp->d ||
      (kind != B7_SCORE_EI && kind != B7_SCORE_CB)) {
    b7_set_error("acq_score: bad arguments (grid dims %d vs model dims %d)", grid ? grid->d : -1, gp ? gp->d : -1);
    return B7_ERR_ARG;
  }
  if (grid->ctx != gp->ctx) { b7_set_error("acq_score: the grid and the model live on different contexts / devices"); return B7_ERR_ARG; }
  B7_CHECK(require_predict_state(gp));
  b7_ctx* ctx = gp->ctx;
  B7_CUDA(cudaSetDevice(ctx->device));
  B7_CHECK(sync_removed(grid));
  const int64_t P = panel_rows(ctx, gp->Np), Pp = std::min(P, pad128(std::max<int64_t>(count, 1)));
  const int S = gp->S;
  B7_CHECK(grow(ctx, &ctx->moments, &ctx->moments_bytes, (size_t)2 * S * Pp * 8));
  const int64_t n_panels = (count + P - 1) / P;
  PartBuf pb(ctx);
  pb.cap = (int)(n_panels * b7_score_grid_size(ctx, P)) + 1;
  B7_CHECK(dev_alloc(ctx, &pb.best, (size_t)pb.cap)); B7_CHECK(dev_alloc(ctx, &pb.idx, (size_t)pb.cap)); B7_CHECK(dev_alloc(ctx, &pb.nan, (size_t)pb.cap));
  struct ScoreBuf { b7_ctx* c; double* p; ~ScoreBuf() { dev_free(c, p); } } sb{ctx, nullptr};
  if (score_host) B7_CHECK(dev_alloc(ctx, &sb.p, (size_t)std::max<int64_t>(count, 1)));
  double* const score_dev = sb.p;
  int n_parts = 0, rc = 0;
  for (int64_t c0 = 0; c0 < count && rc == 0; c0 += P) {
    const int64_t n = std::min(P, count - c0), np = pad128(n);
    double* dm = ctx->moments; double* dv = ctx->moments + (size_t)S * np;
    if (i8_path(gp) && ctx->kstar_overlap && !ctx->profiling && S > 1 && all_sliced_or_sliceable(gp))
      rc = posterior_panel_draws_i8(gp, grid->X + (row0 + c0) * grid->d, n, dm, dv, np);
    else
      for (int s = 0; s < S && rc == 0; ++s)
        rc = posterior_panel(gp, s, grid->X + (row0 + c0) * grid->d, n, dm + (size_t)s * np, dv + (size_t)s * np);
    if (rc < 0) break;
    StageTimer t(ctx, ST_SCORE);
    int parts = 0;
    rc = b7_launch_score(ctx, kind, dm, dv, S, n, np, tradeoff, bound, sign, fmin, grid->removed_dev,
                         (int64_t)grid->removed.size(), row0 + c0, score_dev ? score_dev + c0 : nullptr, pb.best + n_parts,
                         pb.idx + n_parts, pb.nan + n_parts, &parts);
    t.stop(1);
    n_parts += parts;
  }
  double bv = NAN; int64_t r0 = -1, nn = 0;
  if (rc == 0) rc = finish_argmax(ctx, pb, n_parts, &bv, &r0, &nn);
  if (rc == 0 && score_host && count > 0) {
    cudaError_t e = cudaMemcpyAsync(score_host, score_dev, (size_t)count * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { b7_set_error("acq_score D2H: %s", cudaGetErrorString(e)); rc = B7_ERR_CUDA; }
  }
  if (rc < 0) return rc;
  if (argmax_original) *argmax_original = r0 + 1;
  if (best) *best = bv;
  if (nan_count) *nan_count = nn;
  return 0;
}

int b7_acq_score(b7_gp* gp, b7_grid* grid, int kind, double tradeoff, int bound, double sign, double fmin,
                 double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count) {
  if (!grid) { b7_set_error("acq_score: null grid"); return B7_ERR_ARG; }
  int64_t orig = 0;
  B7_CHECK(b7_acq_score_range(gp, grid, 0, grid->rows, kind, tradeoff, bound, sign, fmin, score_host, &orig, best, nan_count));
  if (argmax_original) *argmax_original = orig;
  if (argmax) {
    if (orig <= 0) *argmax = 0;
    else {
      int64_t r = orig - 1;
      int64_t below = std::lower_bound(grid->removed.begin(), grid->removed.end(), r) - grid->removed.begin();
      *argmax = r - below + 1;
    }
  }
  return 0;
}

int b7_score_moments(b7_ctx* ctx, int kind, const double* mean, const double* var, int S, int64_t M, double tradeoff,
                     int bound, double sign, double fmin, double* score_host, int64_t* argmax, double* best,
                     int64_t* nan_count) {
  if (!ctx || S < 1 || M < 0 || (M > 0 && (!mean || !var)) || (kind != B7_SCORE_EI && kind != B7_SCORE_CB)) { b7_set_error("score_moments: bad arguments"); return B7_ERR_ARG; }
  B7_CUDA(cudaSetDevice(ctx->device));
  const size_t n = (size_t)S * std::max<int64_t>(M, 1);
  double *dm = nullptr, *dv = nullptr, *ds = nullptr;
  B7_CHECK(dev_alloc(ctx, &dm, n)); B7_CHECK(dev_alloc(ctx, &dv, n)); B7_CHECK(dev_alloc(ctx, &ds, (size_t)std::max<int64_t>(M, 1)));
  PartBuf pb(ctx); pb.cap = b7_score_grid_size(ctx, M) + 1;
  B7_CHECK(dev_alloc(ctx, &pb.best, (size_t)pb.cap)); B7_CHECK(dev_alloc(ctx, &pb.idx, (size_t)pb.cap)); B7_CHECK(dev_alloc(ctx, &pb.nan, (size_t)pb.cap));
  int rc = 0, parts = 0;
  if (M > 0) {
    B7_CUDA(cudaMemcpyAsync(dm, mean, (size_t)S * M * 8, cudaMemcpyHostToDevice, ctx->stream));
    B7_CUDA(cudaMemcpyAsync(dv, var, (size_t)S * M * 8, cudaMemcpyHostToDevice, ctx->stream));
    StageTimer t(ctx, ST_SCORE);
    rc = b7_launch_score(ctx, kind, dm, dv, S, M, M, tradeoff, bound, sign, fmin, nullptr, 0, 0, ds, pb.best, pb.idx, pb.nan, &parts);
    t.stop(1);
  }
  double bv = NAN; int64_t r0 = -1, nn = 0;
  if (rc == 0) rc = finish_argmax(ctx, pb, parts, &bv, &r0, &nn);
  if (rc == 0 && score_host && M > 0) {
    cudaError_t e = cudaMemcpyAsync(score_host, ds, (size_t)M * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { b7_set_error("score_moments D2H: %s", cudaGetErrorString(e)); rc = B7_ERR_CUDA; }
  }
  dev_free(ctx, dm); dev_free(ctx, dv); dev_free(ctx, ds);
  if (rc < 0) return rc;
  if (argmax) *argmax = r0 + 1;
  if (best) *best = bv;
  if (nan_count) *nan_count = nn;
  return 0;
}

}  // extern "C"

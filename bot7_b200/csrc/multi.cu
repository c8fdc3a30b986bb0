// Multi-GPU entry points of the C ABI (include/bot7_b200.h, "multi-GPU" block): candidate shards, draw-sharded fit
// with one NCCL all-gather per fit, and the (best, index, nan) combine -- bots/bayesopt.lua:56-99 spread over
// config.bot.nGPU devices.  NCCL is bound at run time (dlopen of libnccl.so.2): the library keeps no link-time
// dependency besides libcudart, and a single-GPU host never loads NCCL at all.
//
// One b7_comm drives `n_local` devices of this process out of `world` ranks.  Work on the local devices is issued
// from one host thread per device (the per-device entry points are synchronous), the exchanges are grouped NCCL calls
// on the devices' own streams.
#include <dlfcn.h>
#include <math.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include "b7_internal.h"

namespace {

// ---- the few NCCL declarations this file needs (ABI-stable since NCCL 2.0; nccl.h is not required to build) ----
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
enum { ncclInt8 = 0, ncclInt64 = 4, ncclFloat64 = 8 };

struct Nccl {
  void* h = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
Nccl g_nccl;

int load_nccl() {
  if (g_nccl.h) return 0;
  const char* env = getenv("B7_NCCL_LIB");
  const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  // a copy the process already holds (torch's bundled one under torchrun) wins: one NCCL per process
  for (const char* n : names)
    if (n && !h) h = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
  for (const char* n : names)
    if (n && !h) h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
  if (!h) { b7_set_error("multi-GPU: cannot load libnccl.so.2 (set B7_NCCL_LIB): %s", dlerror()); return B7_ERR_NCCL; }
#define B7_SYM(field, name)                                                                      \
  *(void**)(&g_nccl.field) = dlsym(h, name);                                                     \
  if (!g_nccl.field) { b7_set_error("multi-GPU: %s missing from the NCCL library", name); return B7_ERR_NCCL; }
  B7_SYM(GetVersion, "ncclGetVersion");
  B7_SYM(GetUniqueId, "ncclGetUniqueId");
  B7_SYM(CommInitRank, "ncclCommInitRank");
  B7_SYM(CommInitAll, "ncclCommInitAll");
  B7_SYM(CommDestroy, "ncclCommDestroy");
  B7_SYM(AllGather, "ncclAllGather");
  B7_SYM(Broadcast, "ncclBroadcast");
  B7_SYM(GroupStart, "ncclGroupStart");
  B7_SYM(GroupEnd, "ncclGroupEnd");
  B7_SYM(GetErrorString, "ncclGetErrorString");
#undef B7_SYM
  g_nccl.h = h;
  return 0;
}

#define B7_NCCL(expr)                                                                              \
  do {                                                                                             \
    ncclResult_t r_ = (expr);                                                                      \
    if (r_ != 0) {                                                                                 \
      b7_set_error("NCCL error %s at %s:%d (%s)", g_nccl.GetErrorString(r_), __FILE__, __LINE__, #expr); \
      return B7_ERR_NCCL;                                                                          \
    }                                                                                              \
  } while (0)

void shard(int64_t M, int world, int rank, int64_t* row0, int64_t* count) {
  const int64_t base = M / world, extra = M % world;
  *row0 = rank * base + std::min<int64_t>(rank, extra);
  *count = base + (rank < extra ? 1 : 0);
}

}  // namespace

struct b7_comm {
  int world = 1, rank0 = 0;
  bool owns_ctx = true;
  std::vector<b7_ctx*> ctx;          // one per local device
  std::vector<ncclComm_t> nccl;      // one per local device (empty when world == 1)
  std::vector<double*> triple;       // per local device: world x 4 words for the exchanges of the combine (see exchange_status)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;   // exchange timing on the first local device (the context's own timer events
                                              // belong to the caller's b7_timer_begin / b7_timer_end)
  int n_local() const { return (int)ctx.size(); }
};

namespace {

// runs fn(i) for every local device on its own host thread (the per-device entry points block their caller);
// the first negative return code wins and its message is re-published on the calling thread
template <typename F>
int for_each_local(b7_comm* c, F fn) {
  const int n = c->n_local();
  std::vector<int> rc((size_t)n, 0);
  std::vector<std::string> msg((size_t)n);
  auto body = [&](int i) {
    cudaSetDevice(c->ctx[i]->device);
    rc[i] = fn(i);
    if (rc[i] < 0) msg[i] = b7_last_error();
  };
  if (n == 1) {
    body(0);
  } else {
    std::vector<std::thread> th;
    for (int i = 0; i < n; ++i) th.emplace_back(body, i);
    for (auto& t : th) t.join();
  }
  for (int i = 0; i < n; ++i)
    if (rc[i] < 0) { b7_set_error("device %d: %s", c->ctx[i]->device, msg[i].c_str()); return rc[i]; }
  return 0;
}

// In-place all-gather of a per-draw device array (`per` bytes per draw, draws split over the ranks by the shard
// rule): ncclAllGather when every rank owns the same number of draws, otherwise one grouped broadcast per owner.
int gather_draws(b7_comm* c, const std::vector<void*>& bufs, size_t per, int S) {
  const bool even = S % c->world == 0;
  B7_NCCL(g_nccl.GroupStart());
  for (int i = 0; i < c->n_local(); ++i) {
    char* base = (char*)bufs[i];
    if (even) {
      const size_t bytes = per * (size_t)(S / c->world);
      B7_NCCL(g_nccl.AllGather(base + (size_t)(c->rank0 + i) * bytes, base, bytes, ncclInt8, c->nccl[i], c->ctx[i]->stream));
    } else {
      for (int r = 0; r < c->world; ++r) {
        int64_t s0, cnt;
        shard(S, c->world, r, &s0, &cnt);
        if (cnt > 0) B7_NCCL(g_nccl.Broadcast(base + (size_t)s0 * per, base + (size_t)s0 * per, per * (size_t)cnt, ncclInt8, r, c->nccl[i], c->ctx[i]->stream));
      }
    }
  }
  B7_NCCL(g_nccl.GroupEnd());
  return 0;
}

int comm_finish_init(b7_comm* c) {
  for (int i = 0; i < c->n_local(); ++i) {
    B7_CUDA(cudaSetDevice(c->ctx[i]->device));
    double* t = nullptr;
    B7_CHECK(b7_pool_alloc(c->ctx[i], (void**)&t, sizeof(double) * 4 * (size_t)c->world));
    c->triple.push_back(t);
  }
  B7_CUDA(cudaSetDevice(c->ctx[0]->device));
  B7_CUDA(cudaEventCreate(&c->ev0));
  B7_CUDA(cudaEventCreate(&c->ev1));
  return 0;
}

}  // namespace

extern "C" {

int b7_shard_range(int64_t M, int world, int rank, int64_t* row0, int64_t* count) {
  if (M < 0 || world < 1 || rank < 0 || rank >= world || !row0 || !count) { b7_set_error("shard_range: bad arguments"); return B7_ERR_ARG; }
  shard(M, world, rank, row0, count);
  return 0;
}

int b7_comm_init_all(int n_gpus, const int* device_ids, b7_comm** out) {
  if (!out || n_gpus < 1) { b7_set_error("comm_init_all: bad arguments"); return B7_ERR_ARG; }
  *out = nullptr;
  if (n_gpus > b7_device_count()) { b7_set_error("comm_init_all: %d devices asked for, %d present", n_gpus, b7_device_count()); return B7_ERR_ARG; }
  b7_comm* c = new b7_comm();
  c->world = n_gpus; c->rank0 = 0;
  std::vector<int> devs((size_t)n_gpus);
  for (int i = 0; i < n_gpus; ++i) devs[i] = device_ids ? device_ids[i] : i;
  int rc = 0;
  for (int i = 0; i < n_gpus && rc == 0; ++i) {
    b7_ctx* x = nullptr;
    rc = b7_init(devs[i], &x);
    if (rc == 0) c->ctx.push_back(x);
  }
  if (rc == 0 && n_gpus > 1) {
    rc = load_nccl();
    if (rc == 0) {
      c->nccl.assign((size_t)n_gpus, nullptr);
      ncclResult_t r = g_nccl.CommInitAll(c->nccl.data(), n_gpus, devs.data());
      if (r != 0) { b7_set_error("ncclCommInitAll: %s", g_nccl.GetErrorString(r)); c->nccl.clear(); rc = B7_ERR_NCCL; }
    }
  }
  if (rc == 0) rc = comm_finish_init(c);
  if (rc < 0) { b7_comm_free(c); return rc; }
  *out = c;
  return 0;
}

int b7_comm_unique_id(char* id128) {
  if (!id128) return B7_ERR_ARG;
  B7_CHECK(load_nccl());
  ncclUniqueId id;
  B7_NCCL(g_nccl.GetUniqueId(&id));
  memcpy(id128, id.internal, 128);
  return 0;
}

int b7_comm_init_rank(int device, const char* id128, int world, int rank, b7_comm** out) {
  if (!out || world < 1 || rank < 0 || rank >= world || (world > 1 && !id128)) { b7_set_error("comm_init_rank: bad arguments"); return B7_ERR_ARG; }
  *out = nullptr;
  b7_comm* c = new b7_comm();
  c->world = world; c->rank0 = rank;
  b7_ctx* x = nullptr;
  int rc = b7_init(device, &x);
  if (rc == 0) c->ctx.push_back(x);
  if (rc == 0 && world > 1) {
    rc = load_nccl();
    if (rc == 0) {
      ncclUniqueId id;
      memcpy(id.internal, id128, 128);
      c->nccl.assign(1, nullptr);
      cudaSetDevice(device);
      ncclResult_t r = g_nccl.CommInitRank(c->nccl.data(), world, id, rank);
      if (r != 0) { b7_set_error("ncclCommInitRank: %s", g_nccl.GetErrorString(r)); c->nccl.clear(); rc = B7_ERR_NCCL; }
    }
  }
  if (rc == 0) rc = comm_finish_init(c);
  if (rc < 0) { b7_comm_free(c); return rc; }
  *out = c;
  return 0;
}

int b7_comm_world(b7_comm* c) { return c ? c->world : 0; }
int b7_comm_local_count(b7_comm* c) { return c ? c->n_local() : 0; }
int b7_comm_first_rank(b7_comm* c) { return c ? c->rank0 : 0; }
b7_ctx* b7_comm_ctx(b7_comm* c, int i) { return (c && i >= 0 && i < c->n_local()) ? c->ctx[i] : nullptr; }

void b7_comm_free(b7_comm* c) {
  if (!c) return;
  for (size_t i = 0; i < c->ctx.size(); ++i) {
    cudaSetDevice(c->ctx[i]->device);
    cudaStreamSynchronize(c->ctx[i]->stream);
    if (i < c->triple.size()) b7_pool_free(c->ctx[i], c->triple[i]);
  }
  if (!c->ctx.empty()) cudaSetDevice(c->ctx[0]->device);
  if (c->ev0) cudaEventDestroy(c->ev0);
  if (c->ev1) cudaEventDestroy(c->ev1);
  for (ncclComm_t n : c->nccl)
    if (n) g_nccl.CommDestroy(n);
  if (c->owns_ctx)
    for (b7_ctx* x : c->ctx) b7_shutdown(x);
  delete c;
}

/* ------------------------------------------------------------------ sharded grids */

static void free_grids(b7_grid** g, int n) {
  for (int i = 0; i < n; ++i) { b7_grid_free(g[i]); g[i] = nullptr; }
}

int b7_sobol_generate_sharded(b7_comm* c, int dims, int64_t first_seed, int64_t count, const double* mins, const double* maxes,
                              b7_grid** out) {
  if (!c || !out || count < 0) { b7_set_error("sobol_generate_sharded: bad arguments"); return B7_ERR_ARG; }
  for (int i = 0; i < c->n_local(); ++i) out[i] = nullptr;
  if (first_seed < 0) first_seed = 0;
  int rc = for_each_local(c, [&](int i) {
    int64_t r0, n;
    shard(count, c->world, c->rank0 + i, &r0, &n);
    int rc_ = b7_sobol_generate(c->ctx[i], dims, first_seed + r0, n, mins, maxes, nullptr, &out[i]);
    if (rc_ == 0) { out[i]->row_base = r0; out[i]->rows_total = count; }
    return rc_;
  });
  if (rc < 0) free_grids(out, c->n_local());
  return rc;
}

int b7_grid_from_host_sharded(b7_comm* c, const double* X, int64_t M, int d, b7_grid** out) {
  if (!c || !out || M < 0 || d < 1 || (M > 0 && !X)) { b7_set_error("grid_from_host_sharded: bad arguments"); return B7_ERR_ARG; }
  for (int i = 0; i < c->n_local(); ++i) out[i] = nullptr;
  int rc = for_each_local(c, [&](int i) {
    int64_t r0, n;
    shard(M, c->world, c->rank0 + i, &r0, &n);
    int rc_ = b7_grid_from_host(c->ctx[i], X + r0 * d, n, d, &out[i]);
    if (rc_ == 0) { out[i]->row_base = r0; out[i]->rows_total = M; }
    return rc_;
  });
  if (rc < 0) free_grids(out, c->n_local());
  return rc;
}

// global compacted 1-based index -> global original 0-based row, with the replicated tombstone list
static int64_t global_original(const std::vector<int64_t>& removed, int64_t c1) {
  int64_t r = c1 - 1;
  for (int64_t t : removed) {
    if (t <= r) ++r; else break;
  }
  return r;
}

int b7_grid_remove_sharded(b7_comm* c, b7_grid** grids, int64_t compacted_index, double* removed_row) {
  if (!c || !grids || !grids[0]) { b7_set_error("grid_remove_sharded: bad arguments"); return B7_ERR_ARG; }
  const int64_t total = grids[0]->rows_total, live = total - (int64_t)grids[0]->removed_global.size();
  if (compacted_index < 1 || compacted_index > live) { b7_set_error("grid_remove_sharded: index out of range"); return B7_ERR_ARG; }
  const int64_t r = global_original(grids[0]->removed_global, compacted_index);
  bool have_row = false;
  for (int i = 0; i < c->n_local(); ++i) {
    b7_grid* g = grids[i];
    if (r >= g->row_base && r < g->row_base + g->rows) {        // the owner: tombstone in its local numbering
      const int64_t lr = r - g->row_base;
      if (removed_row) { B7_CHECK(b7_grid_read(g, lr, 1, removed_row)); have_row = true; }
      g->removed.insert(std::upper_bound(g->removed.begin(), g->removed.end(), lr), lr);
      g->removed_dirty = true;
    }
    g->removed_global.insert(std::upper_bound(g->removed_global.begin(), g->removed_global.end(), r), r);
  }
  if (removed_row && c->world > c->n_local()) {
    // one process per GPU: the owner's row travels to everybody (d doubles through the triple scratch's stream)
    const int d = grids[0]->d;
    int owner = 0;
    for (int q = 0; q < c->world; ++q) { int64_t r0, n; shard(total, c->world, q, &r0, &n); if (r >= r0 && r < r0 + n) owner = q; }
    b7_ctx* x = c->ctx[0];
    double* dev = nullptr;
    B7_CHECK(b7_pool_alloc(x, (void**)&dev, sizeof(double) * d));
    if (have_row) B7_CUDA(cudaMemcpyAsync(dev, removed_row, sizeof(double) * d, cudaMemcpyHostToDevice, x->stream));
    B7_NCCL(g_nccl.Broadcast(dev, dev, sizeof(double) * d, ncclInt8, owner, c->nccl[0], x->stream));
    B7_CUDA(cudaMemcpyAsync(removed_row, dev, sizeof(double) * d, cudaMemcpyDeviceToHost, x->stream));
    B7_CUDA(cudaStreamSynchronize(x->stream));
    b7_pool_free(x, dev);
  }
  return 0;
}

/* ------------------------------------------------------------------ sharded fit */

int b7_gp_fit_sharded(b7_comm* c, int kernel, const double* X, const double* y, int N, int d, const double* hyp, int S, int H,
                      int noiseless, b7_gp** out, int* info, double* logml, double* jitter, double* gather_ms) {
  if (!c || !out) { b7_set_error("gp_fit_sharded: null comm/out"); return B7_ERR_ARG; }
  const int n = c->n_local();
  for (int i = 0; i < n; ++i) out[i] = nullptr;
  if (gather_ms) *gather_ms = 0.0;
  if (c->world == 1) return b7_gp_fit(c->ctx[0], kernel, X, y, N, d, hyp, S, H, noiseless, B7_FIT_PREDICT, &out[0], info, logml, jitter);
  // 1. every rank: upload, then factorise + invert (+ alpha, slices) its own draws
  int rc = for_each_local(c, [&](int i) {
    int rc_ = b7_gp_fit(c->ctx[i], kernel, X, y, N, d, hyp, S, H, noiseless, B7_FIT_DEFER, &out[i], nullptr, nullptr, nullptr);
    if (rc_ < 0) return rc_;
    int64_t s0, cnt;
    shard(S, c->world, c->rank0 + i, &s0, &cnt);
    if ((rc_ = b7_gp_fit_range(out[i], (int)s0, (int)cnt, nullptr, nullptr, nullptr)) < 0) return rc_;
    if ((rc_ = b7_gp_invert_range(out[i], (int)s0, (int)cnt)) < 0) return rc_;
    return b7_gp_prepare_gather(out[i], (int)s0, (int)cnt);
  });
  auto fail = [&](int code) { for (int i = 0; i < n; ++i) { b7_gp_free(out[i]); out[i] = nullptr; } return code; };
  // one process per GPU: agree on the outcome of phase 1 before anybody enters the big exchange (a rank that failed,
  // e.g. out of memory, must not leave the others waiting inside ncclAllGather)
  if (c->world > n) {
    b7_ctx* x = c->ctx[0];
    cudaSetDevice(x->device);
    double mine = rc < 0 ? 1.0 : 0.0;
    std::string my_msg = rc < 0 ? b7_last_error() : "";
    std::vector<double> all((size_t)c->world, 0.0);
    cudaError_t e = cudaMemcpyAsync(c->triple[0] + c->rank0, &mine, sizeof(double), cudaMemcpyHostToDevice, x->stream);
    ncclResult_t r = e == cudaSuccess ? g_nccl.AllGather(c->triple[0] + c->rank0, c->triple[0], 1, ncclFloat64, c->nccl[0], x->stream) : 1;
    if (r == 0) e = cudaMemcpyAsync(all.data(), c->triple[0], all.size() * sizeof(double), cudaMemcpyDeviceToHost, x->stream);
    if (r == 0 && e == cudaSuccess) e = cudaStreamSynchronize(x->stream);
    if (r != 0 || e != cudaSuccess) { b7_set_error("gp_fit_sharded: status exchange failed"); return fail(B7_ERR_NCCL); }
    for (int q = 0; q < c->world; ++q)
      if (all[q] != 0.0 && rc == 0) { b7_set_error("gp_fit_sharded: rank %d failed in its share of the fit", q); rc = B7_ERR_STATE; }
    if (rc < 0 && !my_msg.empty()) b7_set_error("%s", my_msg.c_str());
  }
  if (rc < 0) return fail(rc);
  // 2. one exchange, in the form the posterior pass reads
  const bool i8 = out[0]->ctx->use_i8 && out[0]->Np <= B7_I8_MAX_NP;
  const size_t Np = out[0]->Np;
  std::vector<void*> b0((size_t)n), b1((size_t)n), b2((size_t)n), bm((size_t)n);
  for (int i = 0; i < n; ++i) {
    b0[i] = i8 ? (void*)out[i]->facS : (void*)out[i]->fac;
    b1[i] = i8 ? (void*)out[i]->sigma : (void*)out[i]->beta;
    b2[i] = (void*)out[i]->alpha;
    bm[i] = (void*)out[i]->meta_dev;
  }
  b7_ctx* x0 = c->ctx[0];
  cudaSetDevice(x0->device);
  if (gather_ms) cudaEventRecord(c->ev0, x0->stream);
  if ((rc = gather_draws(c, b0, i8 ? b7_i8_facs_stride((int)Np) : Np * Np * sizeof(double), S)) < 0) return fail(rc);
  if ((rc = gather_draws(c, b1, Np * sizeof(double), S)) < 0) return fail(rc);
  if ((rc = gather_draws(c, b2, Np * sizeof(double), S)) < 0) return fail(rc);
  if ((rc = gather_draws(c, bm, 3 * sizeof(double), S)) < 0) return fail(rc);
  cudaSetDevice(x0->device);
  if (gather_ms) cudaEventRecord(c->ev1, x0->stream);
  // 3. bookkeeping on every handle
  rc = for_each_local(c, [&](int i) { return b7_gp_finish_gather(out[i], i8); });
  if (rc < 0) return fail(rc);
  if (gather_ms) {
    float ms = 0;
    cudaSetDevice(x0->device);
    if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess) *gather_ms = ms;
  }
  for (int s = 0; s < S; ++s) {
    if (info) info[s] = out[0]->info_host[s];
    if (logml) logml[s] = out[0]->logml_host[s];
    if (jitter) jitter[s] = out[0]->jitter[s];
  }
  return 0;
}

/* ------------------------------------------------------------------ sharded acquisition */

// The per-rank triples (best score, global original row 1-based or 0, nan count) -> the result every rank reports: larger
// score, then smaller global original row (the reference's first-maximum scan, bots/bayesopt.lua:96); the compacted index
// comes from the tombstone list of the whole grid, which every shard holds.
static void combine_triples(const std::vector<double>& ab, const std::vector<int64_t>& ai, const std::vector<int64_t>& an,
                            const b7_grid* g, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count) {
  double bv = NAN;
  int64_t bi = 0, nn = 0;
  for (size_t r = 0; r < ab.size(); ++r) {
    nn += an[r];
    if (ai[r] <= 0 || ab[r] != ab[r]) continue;
    if (bi == 0 || ab[r] > bv || (ab[r] == bv && ai[r] < bi)) { bv = ab[r]; bi = ai[r]; }
  }
  if (best) *best = bv;
  if (nan_count) *nan_count = nn;
  if (argmax_original) *argmax_original = bi;
  if (argmax) {
    if (bi <= 0) *argmax = 0;
    else {
      const std::vector<int64_t>& rem = g->removed_global;
      *argmax = bi - (int64_t)(std::lower_bound(rem.begin(), rem.end(), bi - 1) - rem.begin());
    }
  }
}

// One process per GPU: every rank, whether its local step failed or not, enters this one all-gather of its status and the
// words `mine[0 .. k)` (k <= 3; doubles travel as their exact bit patterns), so that a rank-local failure cannot leave the
// other ranks waiting inside a collective (a rank whose CUDA context is lost cannot reach it: that case stays fatal, as in
// b7_gp_fit_sharded's phase-1 exchange).  On success `all` holds world x (1 + k) words.  If a rank failed, that rank
// returns its own code and message, every other rank B7_ERR_STATE naming the first failed rank.
static int exchange_status(b7_comm* c, int rc, const int64_t* mine, int k, std::vector<int64_t>& all, const char* what) {
  b7_ctx* x = c->ctx[0];
  const int w = 1 + k;
  const std::string my_msg = rc < 0 ? b7_last_error() : "";
  int64_t h[4] = {rc < 0 ? rc : 0, 0, 0, 0};
  for (int j = 0; j < k; ++j) h[1 + j] = mine[j];
  all.assign((size_t)w * c->world, 0);
  int64_t* buf = (int64_t*)c->triple[0];
  cudaError_t e = cudaSetDevice(x->device);
  if (e == cudaSuccess) e = cudaMemcpyAsync(buf + (size_t)w * c->rank0, h, w * sizeof(int64_t), cudaMemcpyHostToDevice, x->stream);
  ncclResult_t r = e == cudaSuccess ? g_nccl.AllGather(buf + (size_t)w * c->rank0, buf, w, ncclInt64, c->nccl[0], x->stream) : 1;
  if (r == 0) e = cudaMemcpyAsync(all.data(), buf, all.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, x->stream);
  if (r == 0 && e == cudaSuccess) e = cudaStreamSynchronize(x->stream);
  if (r != 0 || e != cudaSuccess) { b7_set_error("%s: status exchange failed", what); return B7_ERR_NCCL; }
  if (rc < 0) { b7_set_error("%s", my_msg.c_str()); return rc; }
  for (int q = 0; q < c->world; ++q)
    if (all[(size_t)w * q] != 0) { b7_set_error("%s: rank %d failed in its local step", what, q); return B7_ERR_STATE; }
  return 0;
}

int b7_acq_score_multi(b7_comm* c, b7_gp** gps, b7_grid** grids, int kind, double tradeoff, int bound, double sign, double fmin,
                       double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count) {
  if (!c || !gps || !grids) { b7_set_error("acq_score_multi: null arguments"); return B7_ERR_ARG; }
  const int n = c->n_local();
  for (int i = 0; i < n; ++i)
    if (!gps[i] || !grids[i] || gps[i]->ctx != c->ctx[i] || grids[i]->ctx != c->ctx[i]) {
      b7_set_error("acq_score_multi: handle %d does not belong to local device %d of the communicator", i, i);
      return B7_ERR_ARG;
    }
  std::vector<double> tb((size_t)n, NAN);
  std::vector<int64_t> ti((size_t)n, 0), tn((size_t)n, 0), off((size_t)n, 0);
  for (int i = 1; i < n; ++i) off[i] = off[i - 1] + grids[i - 1]->rows;
  int rc = for_each_local(c, [&](int i) {
    int64_t o = 0;
    int rc_ = b7_acq_score_range(gps[i], grids[i], 0, grids[i]->rows, kind, tradeoff, bound, sign, fmin,
                                 score_host ? score_host + off[i] : nullptr, &o, &tb[i], &tn[i]);
    ti[i] = o > 0 ? o + grids[i]->row_base : 0;      // global original row, 1-based
    return rc_;
  });
  if (rc < 0) return rc;
  std::vector<double> ab((size_t)c->world, NAN);
  std::vector<int64_t> ai((size_t)c->world, 0), an((size_t)c->world, 0);
  if (c->world == n) {
    for (int i = 0; i < n; ++i) { ab[i] = tb[i]; ai[i] = ti[i]; an[i] = tn[i]; }
  } else {
    // one process per GPU: all-gather of the triples (index and count travel as exact int64 bit patterns)
    b7_ctx* x = c->ctx[0];
    double h[3];
    h[0] = tb[0];
    memcpy(&h[1], &ti[0], 8);
    memcpy(&h[2], &tn[0], 8);
    B7_CUDA(cudaSetDevice(x->device));
    B7_CUDA(cudaMemcpyAsync(c->triple[0] + 3 * c->rank0, h, sizeof(h), cudaMemcpyHostToDevice, x->stream));
    B7_NCCL(g_nccl.AllGather(c->triple[0] + 3 * c->rank0, c->triple[0], 3, ncclInt64, c->nccl[0], x->stream));
    std::vector<double> all((size_t)3 * c->world);
    B7_CUDA(cudaMemcpyAsync(all.data(), c->triple[0], all.size() * sizeof(double), cudaMemcpyDeviceToHost, x->stream));
    B7_CUDA(cudaStreamSynchronize(x->stream));
    for (int r = 0; r < c->world; ++r) {
      ab[r] = all[3 * r];
      memcpy(&ai[r], &all[3 * r + 1], 8);
      memcpy(&an[r], &all[3 * r + 2], 8);
    }
  }
  combine_triples(ab, ai, an, grids[0], argmax, argmax_original, best, nan_count);
  return 0;
}

/* ------------------------------------------------------------------ DNGO over the communicator */

int b7_blr_fit_multi(b7_comm* c, const double* Z0, const double* y, int N, int D, const double* hyp, int S, b7_blr** out, int* info) {
  if (!c || !out || S < 1) { b7_set_error("blr_fit_multi: bad arguments (null comm/out or S=%d)", S); return B7_ERR_ARG; }
  const int n = c->n_local();
  for (int i = 0; i < n; ++i) out[i] = nullptr;
  if (c->world == 1) return b7_blr_fit(c->ctx[0], Z0, y, N, D, hyp, S, &out[0], info);
  // the head is fitted on every device rather than broadcast: the fit has no atomics, so every device holds the same bits
  std::vector<std::vector<int>> inf((size_t)n, std::vector<int>((size_t)S, 0));
  std::vector<int> worst((size_t)n, 0);
  int rc = for_each_local(c, [&](int i) {
    worst[i] = b7_blr_fit(c->ctx[i], Z0, y, N, D, hyp, S, &out[i], inf[i].data());
    return worst[i];
  });
  if (c->world > n) {
    std::vector<int64_t> all;
    rc = exchange_status(c, rc, nullptr, 0, all, "blr_fit_multi");
  }
  if (rc < 0) {
    for (int i = 0; i < n; ++i) { b7_blr_free(out[i]); out[i] = nullptr; }
    return rc;
  }
  if (info)
    for (int s = 0; s < S; ++s) info[s] = inf[0][s];
  return worst[0];
}

int b7_dngo_score_multi(b7_comm* c, b7_blr** blrs, b7_grid** grids, int n_layers, const int* dims, const double* const* W,
                        const double* const* b, int relu_last, int kind, double tradeoff, int bound, double sign, double fmin,
                        double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count) {
  return b7_dngo_score_multi_act(c, blrs, grids, n_layers, dims, W, b, b7_relu_codes(n_layers, relu_last).data(), kind, tradeoff, bound,
                                 sign, fmin, score_host, argmax, argmax_original, best, nan_count);
}

int b7_dngo_score_multi_act(b7_comm* c, b7_blr** blrs, b7_grid** grids, int n_layers, const int* dims, const double* const* W,
                            const double* const* b, const int* act, int kind, double tradeoff, int bound, double sign, double fmin,
                            double* score_host, int64_t* argmax, int64_t* argmax_original, double* best, int64_t* nan_count) {
  if (!c || !blrs || !grids || n_layers < 1 || !dims || !W || !b || (kind != B7_SCORE_EI && kind != B7_SCORE_CB)) {
    b7_set_error("dngo_score_multi: bad arguments");
    return B7_ERR_ARG;
  }
  const int n = c->n_local();
  for (int i = 0; i < n; ++i) {
    if (!blrs[i] || !grids[i] || blrs[i]->ctx != c->ctx[i] || grids[i]->ctx != c->ctx[i]) {
      b7_set_error("dngo_score_multi: handle %d does not belong to local device %d of the communicator", i, i);
      return B7_ERR_ARG;
    }
    if (dims[0] != grids[i]->d || dims[n_layers] != blrs[i]->D) {
      b7_set_error("dngo_score_multi: dims[0] = %d must equal the grid's dims (%d), dims[%d] = %d the head's D (%d)", dims[0], grids[i]->d,
                   n_layers, dims[n_layers], blrs[i]->D);
      return B7_ERR_ARG;
    }
    if (!blrs[i]->ready) {
      b7_set_error("dngo_score_multi: the last refit of handle %d was B7_FIT_LOGML_ONLY; refit with B7_FIT_PREDICT first", i);
      return B7_ERR_STATE;
    }
  }
  // an empty shard launches nothing and would not notice: check the shapes and the activation codes here, for every rank alike
  if (!b7_dngo_tiles_fit(n_layers, dims, dims[n_layers])) {
    b7_set_error("dngo_score: layer shapes do not fit the tile kernel (widths <= 63, at most 4 layers)");
    return B7_ERR_ARG;
  }
  B7_CHECK(b7_check_act("dngo_score_multi", n_layers, act));
  if (c->world == 1)
    return b7_dngo_score_act(blrs[0], grids[0], n_layers, dims, W, b, act, kind, tradeoff, bound, sign, fmin, score_host, argmax,
                         argmax_original, best, nan_count);
  std::vector<double> tb((size_t)n, NAN);
  std::vector<int64_t> ti((size_t)n, 0), tn((size_t)n, 0), off((size_t)n, 0);
  for (int i = 1; i < n; ++i) off[i] = off[i - 1] + grids[i - 1]->rows;
  int rc = for_each_local(c, [&](int i) {
    int64_t o = 0;
    int rc_ = b7_dngo_score_act(blrs[i], grids[i], n_layers, dims, W, b, act, kind, tradeoff, bound, sign, fmin,
                            score_host ? score_host + off[i] : nullptr, nullptr, &o, &tb[i], &tn[i]);
    ti[i] = o > 0 ? o + grids[i]->row_base : 0;      // local original row + the shard's first row: global, 1-based
    return rc_;
  });
  std::vector<double> ab((size_t)c->world, NAN);
  std::vector<int64_t> ai((size_t)c->world, 0), an((size_t)c->world, 0);
  if (c->world == n) {
    if (rc < 0) return rc;
    for (int i = 0; i < n; ++i) { ab[i] = tb[i]; ai[i] = ti[i]; an[i] = tn[i]; }
  } else {
    int64_t mine[3];
    memcpy(&mine[0], &tb[0], 8);
    mine[1] = ti[0];
    mine[2] = tn[0];
    std::vector<int64_t> all;
    if ((rc = exchange_status(c, rc, mine, 3, all, "dngo_score_multi")) < 0) return rc;
    for (int r = 0; r < c->world; ++r) {
      memcpy(&ab[r], &all[4 * (size_t)r + 1], 8);
      ai[r] = all[4 * (size_t)r + 2];
      an[r] = all[4 * (size_t)r + 3];
    }
  }
  combine_triples(ab, ai, an, grids[0], argmax, argmax_original, best, nan_count);
  return 0;
}

}  // extern "C"

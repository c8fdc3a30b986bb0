"""Multi-GPU plumbing: one process per GPU, torch.distributed (NCCL on GPUs, gloo in CPU tests).

The path shards by candidates (SURVEY section 8e): rank g owns the contiguous original-row range
shard_range(M, G, g) of the Sobol sequence and generates it locally.  The only exchanges are
  * fit:     draws are factorised S/G per rank, then L^-1 and beta are all-gathered (NCCL over
             NVLink; in place on the library's own device buffers), or every rank factorises all
             draws when S < G;
  * combine: an all-gather of one (best score, global original index, nan count) triple per rank,
             then every rank applies the same rule -- larger score wins, ties go to the smaller
             global index -- which reproduces the reference's first-maximum scan
             (bots/bayesopt.lua:96) for any G.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np


def shard_range(M: int, world: int, rank: int):
    """Contiguous shard [row0, row0+count) of M rows; the first M % world ranks get one extra row."""
    base, extra = divmod(int(M), int(world))
    row0 = rank * base + min(rank, extra)
    return row0, base + (1 if rank < extra else 0)


def draw_range(S: int, world: int, rank: int):
    return shard_range(S, world, rank)


def combine_argmax(triples):
    """triples: iterable of (best, global_index_1based or 0, nan_count).  Deterministic reduction:
    NaN/empty shards (index 0) are skipped; max score, ties -> smallest index."""
    best, idx, nans = float("nan"), 0, 0
    for b, i, n in triples:
        nans += int(n)
        if int(i) <= 0 or (isinstance(b, float) and math.isnan(b)):
            continue
        if idx == 0 or b > best or (b == best and int(i) < idx):
            best, idx = float(b), int(i)
    return best, idx, nans


def allgather_argmax(best, idx, nans, group=None):
    """All ranks get the same (best, idx, nans).  CPU (gloo) and CUDA (NCCL) tensors both work."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return combine_argmax([(best, idx, nans)])
    dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    world = dist.get_world_size(group)
    # index and count travel as exact int64; the score as float64
    f = torch.tensor([float(best)], dtype=torch.float64, device=dev)
    i = torch.tensor([int(idx), int(nans)], dtype=torch.int64, device=dev)
    fs = [torch.empty_like(f) for _ in range(world)]
    is_ = [torch.empty_like(i) for _ in range(world)]
    dist.all_gather(fs, f, group=group)
    dist.all_gather(is_, i, group=group)
    return combine_argmax([(float(a[0]), int(b[0]), int(b[1])) for a, b in zip(fs, is_)])


class _DevBuf:
    """__cuda_array_interface__ view of a raw device pointer so torch can wrap library memory."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes // 8,), "typestr": "<f8", "data": (int(ptr), False),
                                         "version": 3, "strides": None}


def allgather_draws(full, per_draw, S, world, rank, group=None):
    """In-place all-gather of a flat per-draw buffer: rank r owns draws draw_range(S, world, r) of `full`
    (S * per_draw elements) and receives everybody else's.  Works on CPU (gloo) and CUDA (NCCL) tensors."""
    import torch.distributed as dist
    chunks = []
    for r in range(world):
        s0, cnt = draw_range(S, world, r)
        chunks.append(full[s0 * per_draw:(s0 + cnt) * per_draw])
    if all(c.numel() == chunks[0].numel() for c in chunks):
        dist.all_gather(chunks, chunks[rank].clone(), group=group)
    else:                                   # S not divisible by the world size: one broadcast per owner
        for r in range(world):
            if chunks[r].numel():
                dist.broadcast(chunks[r], src=r, group=group)
    return full


def allgather_factors(factors, S, world, rank, group=None):
    """After each rank factorised + inverted its draw range: all-gather L^-1 (S x Np x Np, tiled layout) and
    beta (S x Np) in place on the library's own device buffers (NCCL over NVLink)."""
    import torch
    Np = factors.padded_n()
    for what, per_draw in ((0, Np * Np), (1, Np)):
        ptr, nbytes = factors.device_ptr(what)
        full = torch.as_tensor(_DevBuf(ptr, nbytes), device="cuda")
        torch.cuda.synchronize()
        allgather_draws(full, per_draw, S, world, rank, group)
        torch.cuda.synchronize()


class Comm:
    """The multi-GPU block of the C ABI (include/bot7_b200.h): b7_comm_* / b7_gp_fit_sharded / b7_acq_score_multi, and for DNGO
    b7_blr_fit_multi / b7_dngo_score_multi.

    Comm.all(n)            one process driving n devices (ncclCommInitAll) -- what the LuaJIT glue does with config.bot.nGPU;
    Comm.from_env()        one process per GPU under torchrun: rank 0 makes the NCCL unique id, torch.distributed carries its
                           128 bytes to the other ranks, every rank joins with b7_comm_init_rank.
    Everything after that (draw-sharded fit, all-gather of the factors, shard scoring, argmax combine) runs inside the library."""

    def __init__(self, handle):
        from . import _lib as L
        self._L = L
        self.handle = handle
        lib = L.lib()
        self.world = lib.b7_comm_world(handle)
        self.n_local = lib.b7_comm_local_count(handle)
        self.first_rank = lib.b7_comm_first_rank(handle)
        self.ctxs = []
        for i in range(self.n_local):
            c = L.Context.__new__(L.Context)          # borrowed: the communicator owns its contexts
            c.handle = C.c_void_p(lib.b7_comm_ctx(handle, i))
            c.device = None
            self.ctxs.append(c)

    @classmethod
    def all(cls, n_gpus, device_ids=None):
        from . import _lib as L
        h = C.c_void_p()
        ids = (C.c_int * n_gpus)(*device_ids) if device_ids is not None else None
        L.check(L.lib().b7_comm_init_all(n_gpus, ids, C.byref(h)), "b7_comm_init_all")
        return cls(h)

    @classmethod
    def from_env(cls, device, world, rank, group=None):
        from . import _lib as L
        buf = C.create_string_buffer(128)
        if world > 1:
            import torch.distributed as dist
            if rank == 0:
                L.check(L.lib().b7_comm_unique_id(buf), "b7_comm_unique_id")
            box = [buf.raw]
            dist.broadcast_object_list(box, src=0, group=group)
            buf = C.create_string_buffer(box[0], 128)
        h = C.c_void_p()
        L.check(L.lib().b7_comm_init_rank(device, buf, world, rank, C.byref(h)), "b7_comm_init_rank")
        return cls(h)

    def _handles(self, objs):
        return (C.c_void_p * self.n_local)(*[o.handle if hasattr(o, "handle") else o for o in objs])

    def sobol_grid(self, dims, first_seed, count, mins=None, maxes=None):
        """Sharded Sobol grid: points first_seed .. first_seed + count - 1, each device generating its own shard."""
        from .grids import DeviceGrid
        L = self._L
        out = (C.c_void_p * self.n_local)()
        mn = None if mins is None else L.as_f64(mins)
        mx = None if maxes is None else L.as_f64(maxes)
        L.check(L.lib().b7_sobol_generate_sharded(self.handle, dims, first_seed, count, L.dptr(mn), L.dptr(mx), out), "b7_sobol_generate_sharded")
        return [DeviceGrid(C.c_void_p(out[i]), self.ctxs[i]) for i in range(self.n_local)]

    def grid_from_host(self, X):
        from .grids import DeviceGrid
        L = self._L
        X = L.as_f64(X)
        out = (C.c_void_p * self.n_local)()
        L.check(L.lib().b7_grid_from_host_sharded(self.handle, L.dptr(X), X.shape[0], X.shape[1], out), "b7_grid_from_host_sharded")
        return [DeviceGrid(C.c_void_p(out[i]), self.ctxs[i]) for i in range(self.n_local)]

    def grid_remove(self, grids, compacted_index):
        L = self._L
        d = grids[0].dims()
        row = np.empty(d)
        L.check(L.lib().b7_grid_remove_sharded(self.handle, self._handles(grids), int(compacted_index), L.dptr(row)), "b7_grid_remove_sharded")
        return row

    def fit(self, X, y, hyp, kernel=0, noiseless=False):
        """b7_gp_fit_sharded -> (list of per-device factor handles, info, logml, jitter, gather_ms)."""
        L = self._L
        X, y = L.as_f64(X), L.as_f64(y).reshape(-1)
        hyp = np.atleast_2d(L.as_f64(hyp))
        S, H = hyp.shape
        out = (C.c_void_p * self.n_local)()
        info = (C.c_int * S)()
        logml, jitter, gms = np.zeros(S), np.zeros(S), C.c_double()
        L.check(L.lib().b7_gp_fit_sharded(self.handle, int(kernel), L.dptr(X), L.dptr(y), X.shape[0], X.shape[1], L.dptr(hyp), S, H,
                                          int(bool(noiseless)), out, info, L.dptr(logml), L.dptr(jitter), C.byref(gms)), "b7_gp_fit_sharded")
        return [C.c_void_p(out[i]) for i in range(self.n_local)], np.array(list(info)), logml, jitter, gms.value

    def free_fit(self, gps):
        for g in gps:
            self._L.lib().b7_gp_free(g)

    def acq_score(self, gps, grids, kind=0, tradeoff=0.0, bound=0, sign=-1.0, fmin=0.0, want_scores=False):
        """b7_acq_score_multi -> (best, argmax (global, compacted), argmax_original, nan_count, scores of the local shards or None)."""
        L = self._L
        n = sum(int(L.lib().b7_grid_rows(g.handle)) for g in grids)
        sc = np.empty(n) if want_scores else None
        am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
        L.check(L.lib().b7_acq_score_multi(self.handle, (C.c_void_p * self.n_local)(*gps), self._handles(grids), kind, tradeoff, bound, sign,
                                           fmin, L.dptr(sc), C.byref(am), C.byref(amo), C.byref(best), C.byref(nn)), "b7_acq_score_multi")
        return best.value, am.value, amo.value, nn.value, sc

    def blr_fit(self, Z0, y, hyp):
        """b7_blr_fit_multi -> (list of per-device BLR head handles, each holding all S rows, info)."""
        L = self._L
        Z0, y = np.atleast_2d(L.as_f64(Z0)), L.as_f64(y).reshape(-1)
        hyp = np.atleast_2d(L.as_f64(hyp))
        S = hyp.shape[0]
        out = (C.c_void_p * self.n_local)()
        info = (C.c_int * S)()
        L.check(L.lib().b7_blr_fit_multi(self.handle, L.dptr(Z0), L.dptr(y), Z0.shape[0], Z0.shape[1], L.dptr(hyp), S, out, info),
                "b7_blr_fit_multi")
        return [C.c_void_p(out[i]) for i in range(self.n_local)], np.array(list(info))

    def free_blr(self, blrs):
        for h in blrs:
            self._L.lib().b7_blr_free(h)

    def dngo_score(self, blrs, grids, weights, biases, relu_last=True, kind=0, tradeoff=0.0, bound=0, sign=-1.0, fmin=0.0,
                   want_scores=False, act=None):
        """b7_dngo_score_multi -> (best, argmax (global, compacted), argmax_original, nan_count, scores of the local shards or None).
        weights[l]: (h_out x h_in) like torch nn.Linear.weight; biases[l]: (h_out,).
        act: one code per layer (b7_dngo_score_multi_act); None is the relu_last form."""
        L = self._L
        Ws = [L.as_f64(w) for w in weights]
        bs = [L.as_f64(b).reshape(-1) for b in biases]
        n = len(Ws)
        dims = (C.c_int * (n + 1))(*([Ws[0].shape[1]] + [w.shape[0] for w in Ws]))
        Wp = (C.POINTER(C.c_double) * n)(*[L.dptr(w) for w in Ws])
        bp = (C.POINTER(C.c_double) * n)(*[L.dptr(b) for b in bs])
        rows = sum(int(L.lib().b7_grid_rows(g.handle)) for g in grids)
        sc = np.empty(rows) if want_scores else None
        am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
        if act is None:
            L.check(L.lib().b7_dngo_score_multi(self.handle, (C.c_void_p * self.n_local)(*blrs), self._handles(grids), n, dims, Wp, bp,
                                                int(bool(relu_last)), kind, tradeoff, bound, sign, fmin, L.dptr(sc), C.byref(am),
                                                C.byref(amo), C.byref(best), C.byref(nn)), "b7_dngo_score_multi")
        else:
            from .models import act_codes
            L.check(L.lib().b7_dngo_score_multi_act(self.handle, (C.c_void_p * self.n_local)(*blrs), self._handles(grids), n, dims, Wp,
                                                    bp, act_codes(act, n), kind, tradeoff, bound, sign, fmin, L.dptr(sc), C.byref(am),
                                                    C.byref(amo), C.byref(best), C.byref(nn)), "b7_dngo_score_multi_act")
        return best.value, am.value, amo.value, nn.value, sc

    def close(self):
        if self.handle:
            self._L.lib().b7_comm_free(self.handle)
            self.handle = None

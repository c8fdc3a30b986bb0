#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on the B200-native path.

metric : EI candidates scored per second at N_obs = 4096, S = 32 hyper-parameter draws (Hartmann6, d = 6, ARD-SE GP),
         GP fit ms (K build + batched Cholesky) beside it.                      [--config headline, the default]
step   : headline / c2 / c4 (weak scaling, factors and grid resident): one pass of the hot path over this rank's
         candidate shard -- per draw the K* tile, the posterior (V = L^-1 K*^T: exact int8 slice products on tcgen05 CTA
         pairs; FP64 DMMA tiles timed beside it at 1 GPU), the fused EI / bound + S-average + argmax pass -- and the
         combine of the per-rank (best, index, nan) triples.
         c3 / c5 (--scaling strong, fixed total work): the draw-sharded fit, its NCCL exchange, the scoring of the whole
         sharded grid and the combine, all inside the timed region.
value  : whole-job candidates/s, inputs resident in HBM when the timed region starts (device time between two CUDA
         events on the library's stream, max over ranks).
e2e    : the same through the C ABI with HOST buffers: b7_gp_fit_sharded (X, y, hyp from the host), the candidate batch
         uploaded with b7_grid_from_host_sharded, b7_acq_score_multi with the score vector read back.  Headline: one
         acquisition over 2^20 candidates per GPU (the survey's headline shape, SURVEY 8d); the same with a batch the size
         of the timed step is reported beside it as e2e_step_batch.
multi  : one process per GPU (torchrun); everything that crosses GPUs runs inside libbot7_b200.so (b7_comm_init_rank,
         b7_gp_fit_sharded, b7_acq_score_multi: NCCL over NVLink); torch.distributed (gloo) only carries the 128-byte
         NCCL id, the barriers and the max over ranks of the timings.
Launch : python bench.py --gpus N --steps K --warmup W [--config headline|c1|c2|c3|c4|c5] [--scaling weak|strong] [--dump-outputs DIR]
         python bench.py --impl reference ...     (CPU arm: the oracle port on the host cores, same config)
Prints ONE JSON line on rank 0; exits 3 if the two posterior paths select different candidates.
--dump-outputs DIR: also writes what the last timed step returned as DIR/<name>.npy, so that two builds run with the same
         arguments can be compared output for output: the combined best score, argmax and NaN count (rank 0) and the score vector
         of every rank's shard (scores.npy on one GPU, scores_rank<r>.npy on several).  The scores come from one more step after
         the timed window, on the same inputs, which must return the timed step's result bit for bit.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True            # the benchmark leaves the tree it runs from as it found it (it may be read-only)

N_OBS, DIMS, S_DRAWS = 4096, 6, 32
SMS = 148
PANELS_PER_STEP = 2                       # 2 x (148 SMs x 128 candidates) = 37 888 candidates per GPU per step
M_STEP = PANELS_PER_STEP * SMS * 128
METRIC = "EI candidates scored/s at N=4096, S=32 hypers"
UNIT = "candidates/s"
EI, CB = 0, 1

# BASELINE.json configs (SURVEY 8d shapes).  weak: candidates per GPU fixed; strong: total fixed, fit inside the step.
CONFIGS = {
    "headline": dict(N=4096, d=6, S=32, kind=EI, obj="hartmann6", M=M_STEP, scaling="weak",
                     workload="Hartmann6 integrated EI, N_obs=4096, d=6, S=32 draws (headline of BASELINE.json metric; fits one GPU)"),
    "c1": dict(N=50, d=2, S=10, kind=EI, obj="braninhoo", M=20000, scaling="weak",
               workload="config 1: examples/run_benchmark.lua shape -- Branin-Hoo 2D, bayesopt EI, GP ARD-SE, N=50 obs, S=10 draws, 20k Sobol candidates"),
    "c2": dict(N=512, d=6, S=1, kind=CB, obj="hartmann6", M=1 << 20, scaling="weak",
               workload="config 2: Hartmann6 6D, UCB (-LCB, kappa=1), single MAP GP, N=512 obs, 2^20 Sobol candidates per GPU"),
    "c3": dict(N=2048, d=6, S=32, kind=EI, obj="hartmann6", M=1 << 22, scaling="strong",
               workload="config 3: Hartmann6 integrated EI, S=32 draws (batched Cholesky), N=2048, 2^22 Sobol candidates in total; "
                        "step = draw-sharded fit + exchange + scoring"),
    "c4": dict(N=20000, d=6, D=50, S=1, kind=EI, obj="hartmann6", M=1 << 22, scaling="weak",
               workload="config 4: DNGO BLR head on 50-d last-layer features, N=20k obs, 2^22 Sobol candidates per GPU"),
    "c5": dict(N=8192, d=20, S=1, kind=EI, obj="ackley", M=1 << 26, scaling="strong",
               workload="config 5: Ackley d=20, N=8192 obs, 2^26 Sobol candidates in total sharded over the GPUs; step = fit + scoring"),
}


# ------------------------------------------------------------------ synthetic workload (SURVEY 8d)

def splitmix64(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    z = x
    z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    return z ^ (z >> np.uint64(31))


def u01(seed, idx):
    """Counter-based uniform: (splitmix64(seed * 2^32 + i) >> 11) * 2^-53."""
    with np.errstate(over="ignore"):
        i = np.asarray(idx, dtype=np.uint64)
        return (splitmix64(np.uint64(seed) * np.uint64(1 << 32) + i) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def hartmann6(X):
    """benchmarks/hartmann6.lua:36-63 (restated; only synthesises Y_obs)."""
    A = -np.array([[10.0, 3.00, 17.0, 3.50, 1.70, 8.00], [0.05, 10.0, 17.0, 0.10, 8.00, 14.0],
                   [3.00, 3.50, 1.70, 10.0, 17.0, 8.00], [17.0, 8.00, 0.05, 10.0, 0.10, 14.0]])
    P = -np.array([[.1312, .1696, .5569, .0124, .8283, .5886], [.2329, .4135, .8307, .3736, .1004, .9991],
                   [.2348, .1451, .3522, .2883, .3047, .6650], [.4047, .8828, .8732, .5743, .1091, .0381]])
    a = -np.array([1.0, 1.2, 3.0, 3.2])
    return np.exp((A[None] * (X[:, None, :] + P[None]) ** 2).sum(2)) @ a


def ackley(X):
    """benchmarks/ackley.lua:28-48 on [-32.768, 32.768]^d mapped from the unit cube (restated; only synthesises Y_obs)."""
    Z = (X - 0.5) * 65.536
    d = Z.shape[1]
    return -20.0 * np.exp(-0.2 * np.sqrt((Z ** 2).sum(1) / d)) - np.exp(np.cos(2 * np.pi * Z).sum(1) / d) + 20.0 + np.e


def hyper_draws(S, d):
    s = np.arange(S)
    hyp = np.zeros((S, d + 3))
    for dd in range(d):
        hyp[:, dd] = np.log(0.1) + u01(2, s * d + dd) * (np.log(2.0) - np.log(0.1))
    hyp[:, d] = 0.5 * (u01(3, s) - 0.5)
    hyp[:, d + 1] = 0.5 * np.log(1e-2)            # noisy case sigma_n^2 = 1e-2
    hyp[:, d + 2] = 0.1 * (u01(4, s) - 0.5)
    return hyp


def dngo_basis(d, D):
    """SURVEY 8d: Z = ReLU(X W + b), W (d x D), b from u(5, .) mapped to N(0, 1) by Box-Muller."""
    n = d * D + D
    u1, u2 = u01(5, np.arange(n)), u01(5, n + np.arange(n))
    z = np.sqrt(-2.0 * np.log(np.maximum(u1, 2.0 ** -53))) * np.cos(2 * np.pi * u2)
    return z[:d * D].reshape(d, D), z[d * D:]


def braninhoo(X):
    """benchmarks/braninhoo.lua:21-44 on [-5, 10] x [0, 15] mapped from the unit square (restated; only synthesises Y_obs)."""
    x1, x2 = 15.0 * X[:, 0] - 5.0, 15.0 * X[:, 1]
    return (x2 - 5.1 / (4 * np.pi ** 2) * x1 ** 2 + 5.0 / np.pi * x1 - 6.0) ** 2 + 10.0 * (1 - 1.0 / (8 * np.pi)) * np.cos(x1) + 10.0


def objective(cfg, X):
    y = {"hartmann6": hartmann6, "braninhoo": braninhoo}.get(cfg["obj"], ackley)(X)
    return (y - y.mean()) / y.std()


# ------------------------------------------------------------------ clocks

class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.samples, self.stop, self.t = index, [], False, None

    def _run(self):
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.t.join(6)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s and s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------ CPU arm (oracle port)

CPU_SAMPLE_CANDIDATES = 65536            # SURVEY 8d: scoring timed on a 65 536-candidate slice, scaled linearly in M


def cpu_sample(cfg, n_draws=None, m_cand=None):
    """Oracle (numpy / LAPACK / BLAS on all host threads; the K* element loops threaded like TH's OpenMP loops) on a bounded
    sample of the config: min(S, n_draws) draws x m_cand candidates, factors pre-fit for the weak configs, fit inside
    for the strong ones.  Returns dict(candidates/s scaled to the config, fit ms per factor, GFLOP/s of the scoring, cores, text)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import b7_oracle as o
    try:    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to every host core
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass
    N, d, S = cfg["N"], cfg["d"], cfg["S"]
    m = m_cand or CPU_SAMPLE_CANDIDATES
    if cfg["scaling"] == "strong":
        m = min(m, cfg["M"])
    X = o.sobol_points(d, N + m)
    Xo, Xc = X[:N], X[N:]
    y = objective(cfg, Xo)
    fmin = float(y.min())
    if "D" in cfg:                        # DNGO head: basis on the host, BLR fit, BLR scoring
        W, b = dngo_basis(d, cfg["D"])
        t0 = time.perf_counter()
        Z0 = np.maximum(Xo @ W + b, 0.0)
        fit = o.blr_fit(Z0, y, np.array([0.0, np.log(1e2), 0.0]))
        t_fit = time.perf_counter() - t0
        t0 = time.perf_counter()
        Z1 = np.maximum(Xc @ W + b, 0.0)
        mu, var = o.blr_predict(fit, Z1)
        o.argmax_first(o.ei_compute(mu, var, fmin, 0.0))
        t = time.perf_counter() - t0
        return {"value": m / t, "fit_ms_per_factor": t_fit * 1e3, "cores": os.cpu_count(), "gflops": m * (cfg["D"] ** 2) / t * 1e-9,
                "sample": f"{m} of {cfg['M']} candidates (basis + BLR predict + EI + argmax), scaled linearly in M; numpy/OpenBLAS on all host threads"}
    nd = min(S, n_draws or 2)
    hyp = hyper_draws(S, d)[:nd]
    t0 = time.perf_counter()
    fits = [o.gp_fit(Xo, y, h, 0, False) for h in hyp]
    t_fit = (time.perf_counter() - t0) / nd
    t0 = time.perf_counter()
    acc = np.zeros(m)
    for f in fits:
        mu, var = o.gp_predict(f, Xc)
        acc = acc + (o.ei_compute(mu, var, fmin, 0.0) if cfg["kind"] == EI else o.cb_compute(mu, var, 1.0, "lower", -1.0))
    o.argmax_first(acc / nd)
    t_draw = (time.perf_counter() - t0) / nd            # seconds per draw for m candidates
    per_cand = t_draw * S / m                           # scoring seconds per candidate at S draws
    if cfg["scaling"] == "strong":
        per_cand += t_fit * S / cfg["M"]                # the fit is part of the strong-scaling step
    return {"value": 1.0 / per_cand, "fit_ms_per_factor": t_fit * 1e3, "cores": os.cpu_count(),
            "gflops": m * (float(N) ** 2 + 4.0 * N) / t_draw * 1e-9,
            "sample": f"{nd} of {S} draws x {m} candidates (K* + TRSM + col-sum-sq + score per draw), "
                      f"{'fit timed and added per step' if cfg['scaling'] == 'strong' else 'factors pre-fit'}; scaled linearly in S and M; "
                      "numpy/scipy (OpenBLAS) on all host threads"}


def run_reference(args, cfg, rank):
    if rank != 0:
        return
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        last = cpu_sample(cfg, n_draws=1, m_cand=32768)     # ~5 s of CPU work per step: K + W steps end within a few minutes
        if i >= args.warmup:
            vals.append(last["value"])
    value = statistics.mean(vals)
    line = {"impl": "reference", "metric": METRIC if args.config == "headline" else f"candidates scored/s ({args.config})", "value": value, "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": cfg["M"] / value * 1e3, "higher_is_better": True,
            "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            # the same workload description as the GPU arm's line (its `arithmetic` and `l2` entries describe that arm and are left out);
            # what a step of this arm actually computes is in `cpu_sample` / `cpu_baseline.sample`
            "config": {"workload": cfg["workload"], "kernel": "ARD-SE" if "D" not in cfg else "BLR head",
                       "candidates_per_gpu_per_step": cfg["M"] if cfg["scaling"] == "weak" else cfg["M"] // max(args.gpus, 1),
                       "candidates_total": cfg["M"] * (args.gpus if cfg["scaling"] == "weak" else 1),
                       "grid": "Sobol", "cpu_sample": last["sample"]},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": last["cores"], "kind": "port", "sample": last["sample"],
                             "fit_ms_per_factor": last["fit_ms_per_factor"], "scoring_gflops": last["gflops"],
                             "note": "CPU restatement (Torch7/gpTorch7 unavailable: no Lua runtime, gp rock not vendored)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------ peaks

def measured_peaks():
    pk = {"hbm_gbs": 6451.8, "hbm_source": "fallback constant", "fp64_dmma_tflops": 37.1, "fp64_source": "fallback constant",
          "int8_tops": 4216.1, "int8_source": "fallback constant"}
    try:
        pk["hbm_gbs"] = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        pk["hbm_source"] = "MEASURED_PEAKS.json (driver-written copy bandwidth)"
    except Exception:
        pass
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "fp64_peak_r01.json")))
        pk["fp64_dmma_tflops"] = max(v for k, v in d.items() if k.startswith("dmma_"))
        pk["fp64_source"] = "profiles/fp64_peak_r01.json: DMMA.8x8x4 issue-rate probe on this pool's B200 (tools/fp64_peak.cu); MEASURED_PEAKS.json has no FP64 figure"
    except Exception:
        pass
    try:
        pk["int8_tops_sustained"] = json.load(open(os.path.join(ROOT, "profiles", "i8_sustained_r01.json")))[
            "p_major_A_collector_7_class_accumulators"]["tops_sustained"]
    except Exception:
        pk["int8_tops_sustained"] = 4075.5
    try:
        pk["int8_tops"] = json.load(open(os.path.join(ROOT, "profiles", "i8_mma_peak_r01.json")))["i8_mma_m128n128_tops"]
        pk["int8_source"] = "profiles/i8_mma_peak_r01.json: tcgen05.mma.kind::i8 M128 N128 issue-rate probe on this pool's B200 (tools/i8_mma_probe.cu); MEASURED_PEAKS.json has no INT8 figure"
    except Exception:
        pass
    return pk


def slices_bytes_per_draw(Np):
    P = (Np // 128 + 1) // 2
    return 4 * P * (P + 1) * 57344


# ------------------------------------------------------------------ outputs

DUMP_MAX_VALUES = 1 << 21                 # per array: 16 MB of float64, so a dump stays well under 64 MB


def dump_outputs(out_dir, arrays, max_values=DUMP_MAX_VALUES):
    """arrays: name -> values, written as out_dir/<name>.npy in float64.  An array with more than max_values elements is
    stored as a fixed, seeded sample of them, the sampled positions beside it as <name>_rows.npy: the same elements every run."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).reshape(-1)
        if a.size > max_values:
            rows = np.sort(np.random.default_rng(0).choice(a.size, max_values, replace=False))
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dump_last_step(args, world, rank, res, step, names):
    """--dump-outputs: `res` is what the last timed step returned, `step(True)` repeats it outside the timed window and also returns
    this rank's score vector (last element).  names: the output names of res.  Every rank takes part (the step may hold collectives)."""
    again = step(True)
    if not np.array_equal(np.array(again[:len(names)], float), np.array(res[:len(names)], float), equal_nan=True):
        raise RuntimeError(f"--dump-outputs: the repeated step returned {again[:len(names)]}, the timed step {res[:len(names)]}")
    arrays = {n: [v] for n, v in zip(names, res)} if rank == 0 else {}
    arrays["scores" if world == 1 else f"scores_rank{rank}"] = again[-1]
    dump_outputs(args.dump_outputs, arrays, DUMP_MAX_VALUES // world)     # at most 32 MB over all ranks


# ------------------------------------------------------------------ GPU arm

_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line, on the process's real stdout (main() points file descriptor 1 at stderr for everything else)."""
    sys.stdout.flush()
    if _REAL_STDOUT is not None:
        os.dup2(_REAL_STDOUT, 1)
    print(json.dumps(line), flush=True)
    if _REAL_STDOUT is not None:
        os.dup2(2, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default=None, choices=["weak", "strong"])
    ap.add_argument("--candidates", type=int, default=None, help="override the config's candidate count (per GPU if weak, total if strong)")
    ap.add_argument("--e2e-candidates", type=int, default=None, help="candidates per GPU of the end-to-end leg (default: 2^20 at the headline, else the step's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-path", action="store_true", help="skip the FP64 DMMA path that the 1-GPU headline run times beside the default one")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write what the last timed step returned as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = dict(CONFIGS[args.config])
    if args.scaling:
        cfg["scaling"] = args.scaling
    if args.candidates:
        cfg["M"] = args.candidates
    if args.impl == "reference":
        return run_reference(args, cfg, rank)
    if args.warmup < 3:
        args.warmup = 3

    # NCCL's own log lines (the version banner at NCCL_DEBUG=WARN / VERSION, INFO lines) go to stderr: stdout carries ONE JSON line.
    # NCCL honours NCCL_DEBUG_FILE only above the VERSION level, so VERSION becomes WARN (which prints the banner too); and because
    # a library may still write to file descriptor 1 directly, the descriptor itself points at stderr until the line is printed.
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    sys.stdout.flush()
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    from bot7_b200 import _lib as L
    from bot7_b200 import models, parallel
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("gloo")
    comm = parallel.Comm.from_env(local, world, rank)
    ctx = comm.ctxs[0]
    lib = L.lib()
    pk = measured_peaks()
    N, d, S, kind = cfg["N"], cfg["d"], cfg["S"], cfg["kind"]
    strong = cfg["scaling"] == "strong"
    M_total = cfg["M"] if strong else cfg["M"] * world
    row0, cnt = parallel.shard_range(M_total, world, rank)
    tradeoff = 0.0 if kind == EI else 1.0

    def allmax(*vals):
        if not dist:
            return list(vals)
        import torch
        t = torch.tensor(list(vals), dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def allsum(v):
        if not dist:
            return v
        import torch
        t = torch.tensor([float(v)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    def barrier():
        if dist:
            dist.barrier()

    # observations: the first N Sobol points; candidates: the rest, sharded by b7_shard_range
    Xo = np.empty((N, d))
    L.check(lib.b7_sobol_generate(ctx.handle, d, 1, N, None, None, L.dptr(Xo), None), "b7_sobol_generate")
    y = objective(cfg, Xo)
    fmin = float(y.min())
    ctx.set_profiling(True)
    ctx.reset_timers()
    grids_ = comm.sobol_grid(d, 1 + N, M_total)
    sobol_ms = ctx.stage_times()["sobol"][0]
    ctx.set_profiling(False)
    env = dict(args=args, cfg=cfg, comm=comm, ctx=ctx, L=L, lib=lib, models=models, parallel=parallel, dist=dist, pk=pk, Xo=Xo, y=y, fmin=fmin,
               grids_=grids_, cnt=cnt, row0=row0, sobol_ms=sobol_ms, world=world, rank=rank, local=local, allmax=allmax, allsum=allsum,
               barrier=barrier)
    if "D" in cfg:
        return bench_dngo(**env)

    hyp = hyper_draws(S, d)

    # ---- fit (timed separately: "GP fit ms") -----------------------------------------------------
    fit_ms = {}
    gps = None
    for rep in range(2):
        if gps:
            comm.free_fit(gps)
        ctx.set_profiling(True)
        ctx.reset_timers()
        barrier()
        t0 = time.perf_counter()
        gps, info, logml, jit, gather_ms = comm.fit(Xo, y, hyp)
        fit_wall = (time.perf_counter() - t0) * 1e3
        st = ctx.stage_times()
        ctx.set_profiling(False)
        own = parallel.draw_range(S, world, rank)[1]
        fit_ms.update(kbuild_ms=st["kbuild"][0], potrf_ms=st["potrf"][0], trtri_ms=st["trtri"][0], exchange_ms=gather_ms,
                      fit_wall_ms=fit_wall, draws_on_this_rank=own)
    assert (info == 0).all()
    if world == 1 and args.config == "headline":
        # single-factor density evaluation (the slice sampler's f): X, y resident, new hyper-parameters each call
        f1 = models.GPFactors(Xo, y, hyp[:1], "ardse", False, L.FIT_LOGML_ONLY, ctx)
        for i in range(2):
            f1.refit(hyp[1:2], L.FIT_LOGML_ONLY)
        t0 = time.perf_counter()
        for i in range(5):
            f1.refit(hyp[i:i + 1], L.FIT_LOGML_ONLY)
        fit_ms["single_factor_refit_ms"] = (time.perf_counter() - t0) / 5 * 1e3
        f1.free()

    state = {"gps": gps}

    def step(want_scores=False):
        """-> (best, argmax, argmax_original, nan_count, scores of this rank's shard or None), as comm.acq_score returns them."""
        if strong:                         # fit + exchange inside the step
            comm.free_fit(state["gps"])
            state["gps"] = comm.fit(Xo, y, hyp)[0]
        return comm.acq_score(state["gps"], grids_, kind, tradeoff, 0, -1.0, fmin, want_scores=want_scores)

    def timed(path, warmup, steps, profiled):
        """`steps` timed steps; returns (device ms per step (max over ranks), wall ms, launches (sum over ranks), stage times, clocks,
        result of the last step).  profiled = False: the number that counts (no per-stage synchronisation, K* of draw s + 1 runs under
        the posterior pass of draw s); profiled = True: per-launch CUDA-event times for the roofline (every stage synchronises)."""
        if ctx.posterior_path() != path:
            ctx.set_posterior_path(path)
            if not strong:                 # the resident factors were exchanged in the other path's form
                comm.free_fit(state["gps"])
                state["gps"] = comm.fit(Xo, y, hyp)[0]
        ctx.set_profiling(profiled)
        r = None
        for _ in range(warmup):
            r = step()
        barrier()
        ctx.sync()
        ctx.reset_timers()
        l0 = ctx.launch_count()
        with ClockSampler(local) as clk_:
            ctx.timer_begin()
            t0 = time.perf_counter()
            for _ in range(steps):
                r = step()
            dev = ctx.timer_end()
            wall = (time.perf_counter() - t0) * 1e3
        barrier()
        n_l = allsum(ctx.launch_count() - l0)
        st_ = ctx.stage_times()
        ctx.set_profiling(False)
        dev, wall = allmax(dev, wall)
        return dev / steps, wall / steps, n_l, st_, clk_.summary(), r

    default_path = ctx.posterior_path()
    other_path = L.PATH_FP64_DMMA if default_path == L.PATH_INT8_OZAKI else L.PATH_INT8_OZAKI
    path_name = {L.PATH_FP64_DMMA: "fp64_dmma", L.PATH_INT8_OZAKI: "int8_ozaki"}
    other = None
    if world == 1 and args.config == "headline" and not args.no_other_path:
        # secondary path first (so that the default path is the one left selected), then the default path = `value`
        o_ms, _, o_launches, _, o_clk, o_res = timed(other_path, 2, args.steps, False)
        _, _, _, o_st, _, _ = timed(other_path, 0, 1, True)
        other = (o_ms, o_launches, o_clk, o_res, o_st)
    ms_per_step, wall_ms, launches, _, clocks, res = timed(default_path, args.warmup, args.steps, False)
    if args.dump_outputs:
        dump_last_step(args, world, rank, res, step, ["best", "argmax", "argmax_original", "nan_count"])
    prof_steps = 1 if strong else 2
    prof_ms, _, _, st, _, _ = timed(default_path, 0, prof_steps, True)
    value = M_total / (ms_per_step * 1e-3)

    # ---- end to end through the C ABI with host buffers (fit + upload + score + read back) ------
    # headline: the survey's shape, 2^20 candidates per GPU and acquisition (SURVEY 8d); the step-sized batch beside it
    def e2e_leg(m):
        if m <= cnt:
            Xc_host = grids_[0].read(0, m)
        else:                              # more rows than the resident shard holds: this rank's next m Sobol points, made on the host side
            Xc_host = np.empty((m, d))
            L.check(lib.b7_sobol_generate(ctx.handle, d, 1 + N + row0, m, None, None, L.dptr(Xc_host), None), "b7_sobol_generate")
        Xc_all = np.concatenate([Xc_host] * world) if world > 1 else Xc_host   # every rank uploads its own m rows
        untimed = 1 if m >= (1 << 19) else 2
        times = []
        for i in range(untimed + 3):
            barrier()
            t0 = time.perf_counter()
            g2 = comm.grid_from_host(Xc_all)
            gp2 = comm.fit(Xo, y, hyp)[0]
            b_, a_, ao_, n_, sc = comm.acq_score(gp2, g2, kind, tradeoff, 0, -1.0, fmin, want_scores=True)
            times.append(time.perf_counter() - t0)
            comm.free_fit(gp2)
            for g in g2:
                g.free()
        sec = allmax(float(np.median(times[untimed:])))[0]
        return {"value": world * m / sec, "unit": UNIT, "h2d_bytes_per_step": int(Xc_host.nbytes + Xo.nbytes + y.nbytes + hyp.nbytes),
                "d2h_bytes_per_step": int(m * 8 + 32), "candidates_per_gpu": int(m),
                "includes": "b7_gp_fit_sharded from host X/y/hyp (K build, batched potrf, inversion, exchange) + b7_grid_from_host_sharded + "
                            f"b7_acq_score_multi with the score vector copied back; median of 3 steps after {untimed} untimed",
                "seconds_per_step": sec, "all_steps_s": [round(x, 4) for x in times]}

    if args.e2e_candidates:
        m_e2e = args.e2e_candidates
    elif args.config == "headline" and not args.candidates:
        m_e2e = 1 << 20
    else:
        m_e2e = cnt if not strong else min(cnt, 1 << 20)
    if strong:
        m_e2e = min(m_e2e, cnt)
    e2e = e2e_leg(m_e2e)
    e2e_step_batch = e2e_leg(cnt) if (m_e2e != cnt and not strong) else None

    if rank != 0:
        comm.free_fit(state["gps"])
        if dist:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: the posterior pass (V = L^-1 K*^T) -----------------------
    Np = (N + 127) // 128 * 128

    def posterior_roofline(path, st_, ms_step, n_steps):
        post_ms, post_n = st_["posterior"]
        if not post_n:
            return None
        flops_total = float(cnt) * S * n_steps * (float(N) ** 2 + 4.0 * N)      # algorithmic: N^2 + 4N flop per candidate per draw
        common = {"launches_timed": post_n, "avg_launch_ms": post_ms / post_n, "share_of_step": post_ms / n_steps / ms_step,
                  "algorithmic_flop_per_candidate_per_draw": float(N) ** 2 + 4.0 * N,
                  "timing": "per-launch CUDA events in a separate profiled pass (every stage synchronised); share_of_step = posterior ms per "
                            "profiled step / ms_per_step of the unprofiled timed loop"}
        ach = flops_total / (post_ms * 1e-3) * 1e-12
        if path == L.PATH_FP64_DMMA:
            return {"bound": "tensor", "kernel": "posterior_kernel (FP64 DMMA.8x8x4)", "achieved": ach, "peak": pk["fp64_dmma_tflops"], "unit": "TFLOP/s",
                    "frac": ach / pk["fp64_dmma_tflops"], "traffic": traffic.get("fp64"), "peak_source": pk["fp64_source"], **common}
        return {"bound": "tensor", "kernel": "posterior_i8_pair_kernel (tcgen05.mma.cta_group::2.kind::i8, 7x7 error-free radix-256 slices, 28 products)",
                "achieved": 28.0 * ach, "peak": pk["int8_tops"], "unit": "TOP/s", "frac": 28.0 * ach / pk["int8_tops"], "traffic": traffic.get("int8"),
                "fp64_equivalent_tflops": ach, "fp64_dmma_peak_tflops": pk["fp64_dmma_tflops"], "peak_source": pk["int8_source"],
                "peak_sustained": pk["int8_tops_sustained"], "frac_of_sustained_peak": 28.0 * ach / pk["int8_tops_sustained"],
                "note": "N = 64 MMAs (7 int32 accumulators x 64 columns = 448 of the 512 TMEM columns) with the A operand held in the collector; "
                        "peak is the N = 128 issue-rate figure (burst: each launch is timed alone, but inside a long power-capped step, for which "
                        "the sustained figure of the same 28-product pattern, profiles/i8_sustained_r01.json, is given beside it)", **common}

    traffic = {}
    if args.config == "headline":
        try:
            traffic["fp64"] = json.load(open(os.path.join(ROOT, "profiles", "posterior_ncu_r01.json"))).get("dram_bytes_per_launch")
            traffic["int8"] = json.load(open(os.path.join(ROOT, "profiles", "posterior_i8_pair_ncu_r02.json"))).get("dram_bytes_per_launch")
        except Exception:
            pass
    roofline = posterior_roofline(default_path, st, ms_per_step, prof_steps)
    own = fit_ms["draws_on_this_rank"]

    def rate(num, ms):
        return num / (ms * 1e-3) if ms else None

    recv_bytes = (S - own) * (slices_bytes_per_draw(Np) + 2 * Np * 8 + 24) if world > 1 else 0
    stages = {
        "profiled_ms_per_step": prof_ms,
        "sobol": {"ms": sobol_ms, "bound": "hbm", "achieved_gbs": rate(cnt * d * 8 * 1e-9, sobol_ms), "peak_gbs": pk["hbm_gbs"],
                  "points_per_s": rate(cnt, sobol_ms)},
        "kstar": {"ms_per_step": st["kstar"][0] / prof_steps, "bound": "fp64 issue (hbm by bytes)",
                  "achieved_gbs": rate(cnt * S * Np * 7 * 1e-9, st["kstar"][0] / prof_steps), "peak_gbs": pk["hbm_gbs"],
                  "note": "serialised in the profiled pass; in the timed loop it runs on a second stream under the posterior pass"},
        "score": {"ms_per_step": st["score"][0] / prof_steps, "bound": "hbm",
                  "achieved_gbs": rate(cnt * (16 * S + 8) * 1e-9, st["score"][0] / prof_steps), "peak_gbs": pk["hbm_gbs"]},
        "fit_kbuild": {"ms": fit_ms["kbuild_ms"], "bound": "hbm", "achieved_gbs": rate(own * Np * Np * 8 * 1e-9, fit_ms["kbuild_ms"]),
                       "peak_gbs": pk["hbm_gbs"]},
        # fp64-equivalent rates: on the int8_ozaki path the k = 512 trailing updates (potrf_i8.cu) and the inversion
        # (trtri_i8.cu) run as exact int8 slice products, so the figure can exceed the FP64 DMMA peak it is shown next to
        "fit_potrf": {"ms": fit_ms["potrf_ms"], "bound": "tensor", "achieved_tflops": rate(own * Np ** 3 / 3 * 1e-12, fit_ms["potrf_ms"]),
                      "peak_tflops": pk["fp64_dmma_tflops"], "arithmetic": "fp64 DMMA + int8 slices (k=512 updates)"},
        "fit_trtri": {"ms": fit_ms["trtri_ms"], "bound": "tensor", "achieved_tflops": rate(own * Np ** 3 / 3 * 1e-12, fit_ms["trtri_ms"]),
                      "peak_tflops": pk["fp64_dmma_tflops"], "arithmetic": "int8 slices, block-recursive (+ alpha back-substitution, slicing)"},
        "fit_exchange": {"ms": fit_ms["exchange_ms"], "bound": "nvlink", "bytes_received_per_rank": recv_bytes,
                         "achieved_gbs": rate(recv_bytes * 1e-9, fit_ms["exchange_ms"]), "peak_gbs": 770.0,
                         "form": "packed int8 slices of L^-1 (lower block triangle) + row scales + alpha, ncclAllGather in place"},
    }
    line = {
        "metric": METRIC if args.config == "headline" else f"candidates scored/s ({args.config})", "value": value, "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": cfg["scaling"],
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["workload"],
                   "arithmetic": "fp64 results; on the int8_ozaki path the N^2 products are 28 exact int8 slice products recombined in fp64, the "
                                 "posterior mean is the fp64 dot product k*^T alpha",
                   "kernel": "ARD-SE", "candidates_per_gpu_per_step": cnt, "candidates_total": M_total,
                   "e2e_candidates_per_gpu": int(m_e2e),
                   "grid": "Sobol (generated on device, per-rank shard)",
                   "l2": f"inputs larger than L2: {S} inverse factors = {S * slices_bytes_per_draw(Np) / 1e9:.2f} GB of int8 slices "
                         f"+ {min(cnt, SMS * 128) * Np * 7 / 1e6:.0f} MB K* panel per launch vs 126 MB L2",
                   "parallelism": f"candidate-sharded x{world}" + (", draw-sharded fit + in-library ncclAllGather of the sliced factors" if world > 1 else "")},
        "gp_fit_ms": {"k_build_plus_cholesky": fit_ms["kbuild_ms"] + fit_ms["potrf_ms"], "draws_on_this_rank": own,
                      "per_factor": (fit_ms["kbuild_ms"] + fit_ms["potrf_ms"]) / max(own, 1),
                      "inversion_for_predict": fit_ms["trtri_ms"], **{k: v for k, v in fit_ms.items() if k.endswith("_ms")}},
        "e2e": e2e,
        "gpu_launches": int(launches), "wall_ms_per_step": wall_ms,
        "clocks": clocks, "roofline": roofline, "stages": stages, "peaks": pk,
        "posterior_path": path_name[default_path],
        "result": {"best": res[0], "global_index": res[2], "nan_count": res[3]},
    }
    if e2e_step_batch:
        line["e2e_step_batch"] = e2e_step_batch
    if other:
        o_ms, o_launches, o_clk, o_res, o_st = other
        line["other_path"] = {"posterior_path": path_name[other_path], "value": M_total / (o_ms * 1e-3), "unit": UNIT, "ms_per_step": o_ms,
                              "gpu_launches": int(o_launches), "roofline": posterior_roofline(other_path, o_st, o_ms, 1), "clocks": o_clk,
                              "same_argmax": bool(o_res[2] == res[2]), "best_rel_diff": abs(o_res[0] - res[0]) / abs(res[0]) if res[0] else None}
    if not args.no_cpu_baseline and world == 1:
        c = cpu_sample(cfg)
        line["cpu_baseline"] = {"value": c["value"], "unit": UNIT, "cores": c["cores"], "kind": "port", "sample": c["sample"],
                                "fit_ms_per_factor": c["fit_ms_per_factor"], "scoring_gflops": c["gflops"],
                                "note": "CPU restatement (Torch7/gpTorch7 unavailable)"}
    emit(line)
    comm.free_fit(state["gps"])
    if dist:
        dist.destroy_process_group()
    if other and not line["other_path"]["same_argmax"]:
        print("bench: the two posterior paths selected different candidates", file=sys.stderr)
        sys.exit(3)


def bench_dngo(args, cfg, comm, ctx, L, lib, models, parallel, dist, pk, Xo, y, fmin, grids_, cnt, row0, sobol_ms, world, rank, local,
               allmax, allsum, barrier):
    """config 4: DNGO BLR head (models/dngo.lua:155-174).  step = the BLR scoring pass over this rank's resident feature grid
    (posterior moments + EI + argmax) and the combine of the triples; the basis (ReLU MLP over the Sobol grid) and the fit
    are timed beside it; e2e = basis + fit + scoring from host observations with the scores read back."""
    d, D = cfg["d"], cfg["D"]
    W, b = dngo_basis(d, D)
    Ws, bs = [np.ascontiguousarray(W.T)], [b]
    hyp = np.array([[0.0, np.log(1e2), 0.0]])
    grid = grids_[0]
    ctx.set_profiling(True)
    ctx.reset_timers()
    feats = models.mlp_features(grid, Ws, bs, True, ctx)
    basis_ms = ctx.stage_times()["blr"][0]
    Z0 = np.maximum(Xo @ W + b, 0.0)
    ctx.reset_timers()
    blr = models.BLRFactors(Z0, y, hyp, ctx)
    fit_ms = ctx.stage_times()["blr"][0]
    ctx.set_profiling(False)

    def step(want_scores=False):
        """-> (best, global argmax_original, nan_count, scores of this rank's shard or None)."""
        am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
        sc = np.empty(cnt) if want_scores else None
        L.check(lib.b7_blr_score(blr.handle, feats.handle, EI, 0.0, 0, -1.0, fmin, L.dptr(sc), C.byref(am), C.byref(amo), C.byref(best),
                                 C.byref(nn)), "b7_blr_score")
        gi = amo.value + row0 if amo.value > 0 else 0
        return (*(parallel.allgather_argmax(best.value, gi, nn.value) if dist else (best.value, gi, nn.value)), sc)

    def timed(warmup, steps, profiled):
        ctx.set_profiling(profiled)
        r = None
        for _ in range(warmup):
            r = step()
        barrier()
        ctx.sync()
        ctx.reset_timers()
        l0 = ctx.launch_count()
        with ClockSampler(local) as clk_:
            ctx.timer_begin()
            t0 = time.perf_counter()
            for _ in range(steps):
                r = step()
            dev = ctx.timer_end()
            wall = (time.perf_counter() - t0) * 1e3
        barrier()
        n_l = allsum(ctx.launch_count() - l0)
        st_ = ctx.stage_times()
        ctx.set_profiling(False)
        dev, wall = allmax(dev, wall)
        return dev / steps, wall / steps, n_l, st_, clk_.summary(), r

    ms_per_step, wall_ms, launches, _, clocks, res = timed(args.warmup, args.steps, False)
    if args.dump_outputs:
        dump_last_step(args, world, rank, res, step, ["best", "argmax_original", "nan_count"])
    _, _, _, st, _, _ = timed(0, 3, True)
    blr_ms = st["blr"][0] / 3
    e2e_times = []
    for i in range(5):
        barrier()
        t0 = time.perf_counter()
        Z0_ = np.maximum(Xo @ W + b, 0.0)
        b2 = models.BLRFactors(Z0_, y, hyp, ctx)
        # dngo:predict + score + argmax in one pass over the device grid: the basis is evaluated in front of the head,
        # the 1.7 GB feature matrix Z1 is never stored (b7_dngo_score)
        sc, am_, amo_, best_, nn_ = models.dngo_score(b2, grid, Ws, bs, True, EI, 0.0, 0, -1.0, fmin, want_scores=True)
        if dist:
            parallel.allgather_argmax(best_, amo_ + row0, nn_)
        e2e_times.append(time.perf_counter() - t0)
        b2.free()
    ctx.set_profiling(True)
    ctx.reset_timers()
    models.dngo_score(blr, grid, Ws, bs, True, EI, 0.0, 0, -1.0, fmin)
    fused_ms = ctx.stage_times()["blr"][0]
    ctx.set_profiling(False)
    e2e_s = allmax(float(np.median(e2e_times[2:])))[0]
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return
    bytes_alg = cnt * (8 * D + 16)
    line = {
        "metric": "candidates scored/s (c4)", "value": world * cnt / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": cfg["workload"], "candidates_per_gpu_per_step": cnt, "features": D,
                   "l2": f"inputs larger than L2: {cnt * D * 8 / 1e9:.2f} GB feature grid vs 126 MB L2",
                   "parallelism": f"candidate-sharded x{world} (no data-path collective; triples combined over gloo)"},
        "e2e": {"value": world * cnt / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(Xo.nbytes + y.nbytes + Z0.nbytes + hyp.nbytes),
                "d2h_bytes_per_step": int(cnt * 8 + 32),
                "includes": "host basis of the observations + b7_blr_fit + b7_dngo_score (basis + BLR head + EI + argmax in one pass over the "
                            "device Sobol grid, Z1 never stored) with the score vector copied back; median of 3 steps after 2 untimed ones",
                "seconds_per_step": e2e_s},
        "gpu_launches": int(launches), "wall_ms_per_step": wall_ms, "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "BLR moments kernel (blr.cu): mean / variance of the BLR head per candidate",
                     "achieved": bytes_alg / (blr_ms * 1e-3) * 1e-9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": bytes_alg / (blr_ms * 1e-3) * 1e-9 / pk["hbm_gbs"], "traffic": None,
                     "algorithmic_bytes_per_candidate": 8 * D + 16, "avg_launch_ms": blr_ms,
                     "fp64_tflops": cnt * (D * D + 2 * D) * 2 / (blr_ms * 1e-3) * 1e-12, "fp64_peak_tflops": pk["fp64_dmma_tflops"],
                     "peak_source": pk["hbm_source"]},
        "stages": {"sobol": {"ms": sobol_ms}, "basis_mlp": {"ms": basis_ms, "tflops": cnt * (d * D) * 2 / (basis_ms * 1e-3) * 1e-12 if basis_ms else None},
                   "blr_fit": {"ms": fit_ms}, "blr_moments": {"ms_per_step": blr_ms}, "score": {"ms_per_step": st["score"][0] / 3},
                   "fused_basis_plus_head": {"ms": fused_ms, "note": "b7_dngo_score's tile kernel: basis + head per tile, reads 8 d bytes per candidate"}},
        "peaks": pk, "result": {"best": res[0], "global_index": res[1], "nan_count": res[2]},
    }
    if not args.no_cpu_baseline and world == 1:
        c = cpu_sample(cfg)
        line["cpu_baseline"] = {"value": c["value"], "unit": UNIT, "cores": c["cores"], "kind": "port", "sample": c["sample"],
                                "fit_ms_per_factor": c["fit_ms_per_factor"], "note": "CPU restatement (Torch7/gpTorch7 unavailable)"}
    emit(line)
    if dist:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

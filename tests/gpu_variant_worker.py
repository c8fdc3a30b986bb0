"""One seeded workload in a process of its own: `python gpu_variant_worker.py WORKLOAD OUT.npz [--profile]`.

Most of the library's B7_* switches are read once per process (`static const ... getenv`) or at b7_init, so
tests/test_gpu_coverage.py runs every execution variant as a child process with its own environment.  The child
builds the workload from fixed seeds, writes the raw float64 outputs and exits; the parent compares them with the
reference run and with the oracle.  The problem builders are imported by the parent as well, so both sides see the
same inputs.  This is a helper of the GPU tests, not a test module.
"""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (HERE, os.path.join(ROOT, "oracle"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import b7_oracle as oracle                      # noqa: E402
from test_gpu_parity import make_problem        # noqa: E402

# batched: 18 row blocks x 13 draws = 4212 >= 4096 -> INT8 trailing updates of the Cholesky and trtri_i8
BATCHED = dict(N=2304, d=6, S=13, M=64 * 37 + 5)
BATCHED_DRAWS = (0, 12)
JITTER_DRAW = 7
# latency: two draws -> the row-sliced schedule; fit + two refits, the third factorisation replays the CUDA graph
LATENCY = dict(N=1100, d=6, S=2, M=64 * 37 + 5)
# blr: every `dp` bucket of launch_moments_dp (8 ... 64) through D, every launch_mlp_layer bucket through the input width
# (BLR_INPUT_DIMS) and the hidden widths; D = 64 and a 64-wide hidden layer are what the DMMA tile kernels decline
BLR_D = (1, 9, 17, 25, 33, 41, 50, 63, 64)
BLR_HIDDEN = (5, 12, 20, 28, 36, 44, 52, 60, 64)
BLR_INPUT_DIMS = 6
BLR_N, BLR_M = 300, 128 * 37 + 5

WORKLOADS = ("batched_ardse", "batched_matern52", "jitter", "latency", "blr")


def batched_problem(jitter=False):
    """N = 2304, d = 6, S = 13, sigma_n^2 = 1e-2.  With `jitter`: observations 2104..2303 repeat observations 0..199 and draw 7
    has sigma_n^2 = 1e-18, so its K_y is singular and only that draw of the INT8 batch takes the jitter retry."""
    Xo, y, hyp, Xc = make_problem(oracle, BATCHED["N"], BATCHED["d"], BATCHED["S"], BATCHED["M"], 1e-2, seed=11)
    if jitter:
        d = BATCHED["d"]
        Xo[-200:] = Xo[:200]
        y[-200:] = y[:200]
        hyp[JITTER_DRAW, :d] = np.log(0.15)
        hyp[JITTER_DRAW, d + 1] = 0.5 * np.log(1e-18)
    return Xo, y, hyp, Xc


def latency_problem():
    Xo, y, hyp, Xc = make_problem(oracle, LATENCY["N"], LATENCY["d"], LATENCY["S"], LATENCY["M"], 1e-2, seed=12)
    return Xo, y, hyp, Xc, [hyp, hyp + 0.1, hyp]          # fit, refit, refit (graph replay)


def blr_problem(D, H):
    r = np.random.default_rng(1000 + D)
    dims = [BLR_INPUT_DIMS, H, D]
    Ws = [r.normal(size=(dims[i + 1], dims[i])) / np.sqrt(dims[i]) for i in range(2)]
    bs = [0.1 * r.normal(size=dims[i + 1]) for i in range(2)]
    Xo, Xc = r.random((BLR_N, BLR_INPUT_DIMS)), r.random((BLR_M, BLR_INPUT_DIMS))
    y = r.normal(size=BLR_N)
    hyp = np.array([[0.0, np.log(30.0), 0.05], [np.log(2.0), np.log(60.0), -0.1]])
    return Ws, bs, Xo, y, hyp, Xc


def _acq(f, grid, fmin):
    from bot7_b200 import _lib as L
    sc = np.empty(grid.rows())
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
    L.check(L.lib().b7_acq_score(f.handle, grid.handle, L.SCORE_EI, 0.0, 0, -1.0, fmin, L.dptr(sc), C.byref(am), C.byref(amo),
                                 C.byref(best), C.byref(nn)), "b7_acq_score")
    return sc, np.array([am.value, amo.value, nn.value], dtype=np.float64), np.array([best.value])


def run_batched(kernel, jitter):
    from bot7_b200 import grids, models
    Xo, y, hyp, Xc = batched_problem(jitter)
    f = models.GPFactors(Xo, y, hyp, kernel)
    out = {"info": f.info.astype(np.float64), "jitter": f.jitter.copy(), "logml": f.logml.copy()}
    draws = (0, JITTER_DRAW, 12) if jitter else BATCHED_DRAWS
    for s in draws:
        if not jitter:
            out[f"factor{s}"] = f.read_factor(s)
        out[f"mean{s}"], out[f"var{s}"] = f.predict(s, Xc)
    grid = grids.DeviceGrid.from_host(Xc)
    out["score"], out["argmax"], out["best"] = _acq(f, grid, float(y.min()))
    grid.free()
    f.free()
    return out


def run_latency():
    from bot7_b200 import _lib as L
    from bot7_b200 import grids, models
    Xo, y, hyp, Xc, steps = latency_problem()
    f = models.GPFactors(Xo, y, steps[0], "ardse")
    out = {"logml0": f.logml.copy(), "info0": f.info.astype(np.float64)}
    for k in (1, 2):
        f.refit(steps[k], L.FIT_PREDICT)
        out[f"logml{k}"], out[f"info{k}"] = f.logml.copy(), f.info.astype(np.float64)
    for s in range(LATENCY["S"]):
        out[f"mean{s}"], out[f"var{s}"] = f.predict(s, Xc)
    grid = grids.DeviceGrid.from_host(Xc)
    out["score"], out["argmax"], out["best"] = _acq(f, grid, float(y.min()))
    grid.free()
    f.free()
    return out


def run_blr():
    from bot7_b200 import _lib as L
    from bot7_b200 import grids, models
    out = {}
    for D, H in zip(BLR_D, BLR_HIDDEN):
        Ws, bs, Xo, y, hyp, Xc = blr_problem(D, H)
        Z0, Z1 = oracle.mlp_features(Xo, Ws, bs), oracle.mlp_features(Xc, Ws, bs)
        f = models.BLRFactors(Z0, y, hyp)
        out[f"D{D}_info"] = f.info.astype(np.float64)
        for s in range(hyp.shape[0]):
            out[f"D{D}_mean{s}"], out[f"D{D}_var{s}"] = f.predict(s, Z1)
        grid = grids.DeviceGrid.from_host(Xc)
        feats = models.mlp_features(grid, Ws, bs)
        out[f"D{D}_features"] = feats.read()
        sc = np.empty(BLR_M)
        am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
        L.check(L.lib().b7_blr_score(f.handle, feats.handle, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), L.dptr(sc), C.byref(am),
                                     C.byref(amo), C.byref(best), C.byref(nn)), "b7_blr_score")
        out[f"D{D}_blr_score"], out[f"D{D}_blr_argmax"] = sc, np.array([am.value, nn.value], dtype=np.float64)
        try:
            sc2, am2, _, _, nn2 = models.dngo_score(f, grid, Ws, bs, True, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), want_scores=True)
            out[f"D{D}_dngo_score"], out[f"D{D}_dngo_argmax"] = sc2, np.array([am2, nn2], dtype=np.float64)
        except L.B7Error as e:
            out[f"D{D}_dngo_error"] = np.array([1.0 if "tile kernel" in str(e) else -1.0])
        feats.free()
        grid.free()
        f.free()
    return out


def run(workload):
    if workload == "batched_ardse":
        return run_batched("ardse", False)
    if workload == "batched_matern52":
        return run_batched("matern52", False)
    if workload == "jitter":
        return run_batched("ardse", True)
    if workload == "latency":
        return run_latency()
    if workload == "blr":
        return run_blr()
    raise SystemExit(f"unknown workload {workload!r}; one of {WORKLOADS}")


def main(argv):
    workload, path = argv[1], argv[2]
    from bot7_b200 import _lib as L
    ctx = L.Context.default(0)
    if "--profile" in argv[3:]:
        ctx.set_profiling(True)
    out = run(workload)
    ctx.sync()
    np.savez(path, **out)


if __name__ == "__main__":
    main(sys.argv)

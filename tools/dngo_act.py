"""Cost of the basis activations at config 4's shape (2^22 Sobol candidates, basis 6 -> 50 -> 50 -> 50, S = 1 and 5):
for ReLU and for Tanh, the basis alone (b7_mlp_features(_act)), the fused b7_dngo_score(_act) and the per-layer fallback
(B7_BLR_DMMA=0), each the mean of many calls after warm-up on the device stopwatch (CUDA events, b7_timer_begin / end).
With --parent-lib, a build of the parent commit is timed on ReLU in the same job, alternating with this build (ABBA), one
child process per library and round.  tools/tanh_bench.cu compares libdevice tanh(), which the library uses, with a table-driven
candidate.  Writes one JSON file.

    python tools/dngo_act.py [--parent-lib path/to/libbot7_b200.so] [--rounds 3] [--out profiles/dngo_act_r01.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M, DIMS, WIDTHS = 1 << 22, 6, [6, 50, 50, 50]
ACTS = {"relu": [1, 1, 1], "tanh": [2, 2, 2]}


def child(lib_path, acts, warmup, calls):
    """Times one library (raw ctypes: the parent build has no _act symbols and the package binding would refuse it)."""
    lib = C.CDLL(lib_path)
    p, dp = C.c_void_p, C.POINTER(C.c_double)
    lib.b7_last_error.restype = C.c_char_p

    def ok(rc, what):
        if rc < 0:
            raise RuntimeError(f"{what}: {lib.b7_last_error().decode()}")

    ctx = p()
    ok(lib.b7_init(0, C.byref(ctx)), "b7_init")
    grid = p()
    ok(lib.b7_sobol_generate(ctx, DIMS, C.c_int64(1), C.c_int64(M), None, None, None, C.byref(grid)), "b7_sobol_generate")
    r = np.random.default_rng(4)
    Ws = [np.ascontiguousarray(r.standard_normal((WIDTHS[l + 1], WIDTHS[l])) / np.sqrt(WIDTHS[l])) for l in range(3)]
    bs = [0.1 * r.standard_normal(WIDTHS[l + 1]) for l in range(3)]
    n = len(Ws)
    dims = (C.c_int * (n + 1))(*WIDTHS)
    Wp = (dp * n)(*[w.ctypes.data_as(dp) for w in Ws])
    bp = (dp * n)(*[b.ctypes.data_as(dp) for b in bs])
    Z0 = np.ascontiguousarray(r.standard_normal((400, 50)))
    y = r.standard_normal(400)
    heads = {}
    for S in (1, 5):
        hyp = np.ascontiguousarray(np.column_stack([np.log(0.5) + r.random(S), np.log(20.0) + r.random(S), np.zeros(S)]))
        h = p()
        ok(lib.b7_blr_fit(ctx, Z0.ctypes.data_as(dp), y.ctypes.data_as(dp), 400, 50, hyp.ctypes.data_as(dp), S, C.byref(h), None),
           "b7_blr_fit")
        heads[S] = h
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()

    def timed(fn):
        for _ in range(warmup):
            fn()
        ms = C.c_double()
        ok(lib.b7_timer_begin(ctx), "b7_timer_begin")
        for _ in range(calls):
            fn()
        ok(lib.b7_timer_end(ctx, C.byref(ms)), "b7_timer_end")
        return ms.value / calls

    out = {}
    for name in acts:
        codes = (C.c_int * n)(*ACTS[name])
        relu = name == "relu"                          # ReLU through the relu_last entries: what the parent build has

        def features():
            f = p()
            if relu:
                ok(lib.b7_mlp_features(ctx, grid, n, dims, Wp, bp, 1, C.byref(f)), "b7_mlp_features")
            else:
                ok(lib.b7_mlp_features_act(ctx, grid, n, dims, Wp, bp, codes, C.byref(f)), "b7_mlp_features_act")
            lib.b7_grid_free(f)

        def score(S):
            def fn():
                if relu:
                    ok(lib.b7_dngo_score(heads[S], grid, n, dims, Wp, bp, 1, 0, C.c_double(0.0), 0, C.c_double(-1.0), C.c_double(0.0),
                                         None, C.byref(am), C.byref(amo), C.byref(best), C.byref(nn)), "b7_dngo_score")
                else:
                    ok(lib.b7_dngo_score_act(heads[S], grid, n, dims, Wp, bp, codes, 0, C.c_double(0.0), 0, C.c_double(-1.0),
                                             C.c_double(0.0), None, C.byref(am), C.byref(amo), C.byref(best), C.byref(nn)),
                       "b7_dngo_score_act")
            return fn

        out[name] = {"basis_ms": timed(features), "dngo_score_S1_ms": timed(score(1)), "dngo_score_S5_ms": timed(score(5)),
                     "argmax_S5": am.value}
    for h in heads.values():
        lib.b7_blr_free(h)
    lib.b7_grid_free(grid)
    lib.b7_shutdown(ctx)
    return out


def run_child(lib_path, acts, warmup, calls, env=None):
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", lib_path, "--acts", ",".join(acts), "--warmup", str(warmup),
                        "--calls", str(calls)], capture_output=True, text=True, env=dict(os.environ, **(env or {})), timeout=1800)
    if r.returncode != 0:
        raise RuntimeError(r.stdout[-2000:] + r.stderr[-2000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def tanh_bench():
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "tanh_bench")
        subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                        os.path.join(ROOT, "tools", "tanh_bench.cu"), "-o", exe], check=True)
        r = subprocess.run([exe], capture_output=True, text=True, check=True, timeout=600)
        return json.loads(r.stdout.strip().splitlines()[-1])


def spread(v):
    return {"mean": float(np.mean(v)), "min": float(np.min(v)), "max": float(np.max(v)), "runs": [float(x) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--child")
    ap.add_argument("--acts", default="relu,tanh")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--calls", type=int, default=40)
    ap.add_argument("--parent-lib")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "dngo_act_r01.json"))
    a = ap.parse_args()
    if a.child:
        print(json.dumps(child(a.child, a.acts.split(","), a.warmup, a.calls)))
        return
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                          check=True).stdout.strip().splitlines()[0]
    lib = os.path.join(ROOT, "bot7_b200", "libbot7_b200.so")
    res = {"card": card, "shape": {"M": M, "widths": WIDTHS, "S": [1, 5]},
           "method": f"mean of {a.calls} calls after {a.warmup} warm-up calls, CUDA events on the context stream; each call is "
                     "synchronous (weights uploaded, scores reduced on the host), as a user calls it",
           "this": run_child(lib, ["relu", "tanh"], a.warmup, a.calls),
           "fallback_B7_BLR_DMMA_0": run_child(lib, ["relu", "tanh"], 2, 8, {"B7_BLR_DMMA": "0"}),
           "tanh_bench": tanh_bench()}
    if a.parent_lib:
        keys = ("basis_ms", "dngo_score_S1_ms", "dngo_score_S5_ms")
        runs = {"this": {k: [] for k in keys}, "parent": {k: [] for k in keys}}
        pair = (("this", lib), ("parent", a.parent_lib))
        for rnd in range(a.rounds):
            for who, path in (pair if rnd % 2 == 0 else pair[::-1]):         # ABBA: neither build always runs first
                r = run_child(path, ["relu"], a.warmup, a.calls)["relu"]
                for k in keys:
                    runs[who][k].append(r[k])
        res["relu_vs_parent"] = {who: {k: spread(v) for k, v in d.items()} for who, d in runs.items()}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

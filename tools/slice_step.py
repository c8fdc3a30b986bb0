"""Cost of gp_regressor.sample_hypers with 11 slice steps (the priming draw + nSamples = 10 of the reference experiment) by
the three samplers that walk the same chain:

  * sequential: bot7_b200.samplers.slice, one b7_gp_refit per density evaluation;
  * speculative: slice_speculative, batches of spec_width = 8 evaluations per b7_gp_refit;
  * device step: slice_device, one b7_gp_slice_step per step (config device_step = True, N <= 128).

Shapes: config c1 (Branin, d = 2, N = 100), and d = 6 at N = 100 and N = 128.  Each variant runs `reps` times from a fresh model
and the same seed (the chains are checked to be identical); the time of a run is CUDA events on the library's stream around the
whole call (b7_timer_begin / b7_timer_end: the call ends in a synchronisation, so this is its wall time), the median is
reported with the host clock's median beside it, and the device calls and kernel launches per step.  Prints one JSON object
(and writes it to --out when given).  Needs a CUDA device; there is no CPU path.
Run: python tools/slice_step.py [--out profiles/slice_step_r01.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]

VARIANTS = {"sequential": {"speculative": False}, "speculative": {"speculative": True}, "device_step": {"device_step": True}}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--steps", type=int, default=11)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import b7_oracle as o
    from bot7_b200 import _lib as L
    from bot7_b200 import models
    ctx = L.Context.default(0)
    calls = {"n": 0}
    for name in ("refit", "slice_step"):
        orig = getattr(models.GPFactors, name)

        def counted(self, *args, _orig=orig, **kw):
            calls["n"] += 1
            return _orig(self, *args, **kw)
        setattr(models.GPFactors, name, counted)
    orig_init = models.GPFactors.__init__

    def counted_init(self, *args, **kw):
        calls["n"] += 1
        orig_init(self, *args, **kw)
    models.GPFactors.__init__ = counted_init

    res = {"tool": "tools/slice_step.py", "date": time.strftime("%Y-%m-%d"), "gpu": gpu_info(), "reps": a.reps, "steps": a.steps,
           "timing": "median over reps of CUDA events around one sample_hypers call (ends in a synchronisation); fresh model, same seed",
           "shapes": []}
    for label, N, d in (("c1", 100, 2), ("d6_N100", 100, 6), ("d6_N128", 128, 6)):
        X = o.sobol_points(d, N + 7)[7:]
        y = {2: o.braninhoo, 6: o.hartmann6}[d](X)
        y = (y - y.mean()) / y.std()
        shape = {"label": label, "N": N, "d": d}
        chains = {}
        for vname, cfg in VARIANTS.items():
            def run():
                m = models.gp_regressor(dict(cfg, nSamples=a.steps), rng=np.random.default_rng(7))
                return m.sample_hypers(X, y)
            run()                                             # warm-up: module loads, graph capture, pool
            ev, wall = [], []
            c0, l0 = calls["n"], ctx.launch_count()
            for _ in range(a.reps):
                ms = C.c_double()
                L.check(L.lib().b7_timer_begin(ctx.handle))
                t0 = time.perf_counter()
                out = run()
                wall.append((time.perf_counter() - t0) * 1e3)
                L.check(L.lib().b7_timer_end(ctx.handle, C.byref(ms)))
                ev.append(ms.value)
            per = a.reps * a.steps
            chains[vname] = out
            shape[vname] = {"ms_median": float(np.median(ev)), "ms_min": float(np.min(ev)), "ms_max": float(np.max(ev)),
                            "host_ms_median": float(np.median(wall)),
                            "device_calls_per_step": (calls["n"] - c0) / per, "launches_per_step": (ctx.launch_count() - l0) / per}
        shape["chains_identical"] = all(np.array_equal(chains["sequential"], c) for c in chains.values())
        shape["device_step_speedup_vs_speculative"] = shape["speculative"]["ms_median"] / shape["device_step"]["ms_median"]
        res["shapes"].append(shape)
        print(json.dumps(shape), flush=True)
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
            fh.write("\n")


if __name__ == "__main__":
    main()

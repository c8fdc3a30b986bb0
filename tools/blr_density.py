"""Cost of the DNGO head's hyper-parameter density (b7_blr_refit with B7_FIT_LOGML_ONLY) at config 4's shape, N = 20 000
observations, D = 50 features:

  * device ms per batched evaluation at W = 1 and W = 8 rows per call (CUDA events around `reps` calls), and the host
    wall time per call (launches + copies + synchronisation included);
  * wall ms of bayes_linear.sample_hypers with nSamples = 10, speculative (8 evaluations per call) and sequential;
  * the reference evaluation's host time for the same evaluations (tests/blr_evidence_oracle.py: numpy / LAPACK, fp64).

Prints one JSON object (and writes it to --out when given).  Needs a CUDA device; there is no CPU path.
Run: python tools/blr_density.py [--out profiles/blr_density_r01.json]"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]


def features(N, D, seed=0):
    r = np.random.default_rng(seed)
    X = r.uniform(-1, 1, (N, 6))
    H = np.maximum(X @ (r.standard_normal((6, 32)) / math.sqrt(6)) + 0.2 * r.standard_normal(32), 0.0)
    Z = np.maximum(H @ (r.standard_normal((32, D)) / math.sqrt(8)) + 0.2 * r.standard_normal(D), 0.0)
    y = np.sin(2 * X[:, 0]) + X[:, 1] * X[:, 2] + 0.05 * r.standard_normal(N)
    return Z, y


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=20000)
    ap.add_argument("--D", type=int, default=50)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from blr_evidence_oracle import blr_log_evidence
    from bot7_b200 import _lib as L
    from bot7_b200 import models
    ctx = L.Context.default(0)
    Z, y = features(a.N, a.D)
    r = np.random.default_rng(1)
    rows = np.column_stack([r.uniform(-3, 2, 8), r.uniform(1, 7, 8), y.mean() + r.uniform(-0.3, 0.3, 8)])
    res = {"tool": "tools/blr_density.py", "date": time.strftime("%Y-%m-%d"), "gpu": gpu_info(), "N": a.N, "D": a.D, "reps": a.reps}
    for W in (1, 8):
        f = models.BLRFactors(Z, y, rows[:W])
        for _ in range(20):
            f.refit(rows[:W], L.FIT_LOGML_ONLY)
        ctx.timer_begin()
        t0 = time.perf_counter()
        for k in range(a.reps):
            f.refit(rows[:W], L.FIT_LOGML_ONLY)
        wall = (time.perf_counter() - t0) * 1e3 / a.reps
        dev = ctx.timer_end() / a.reps
        res[f"W{W}"] = {"device_ms_per_call": dev, "wall_ms_per_call": wall, "wall_ms_per_evaluation": wall / W}
        f.free()
    t0 = time.perf_counter()
    for h in rows:
        blr_log_evidence(Z, y, h)
    res["oracle_ms_per_evaluation"] = (time.perf_counter() - t0) * 1e3 / len(rows)
    for spec in (True, False):
        bl = models.bayes_linear({"sampler": "slice", "nSamples": 10, "speculative": spec}, rng=np.random.default_rng(2))
        bl.sample_hypers(Z, y, single=True)                            # resident handle built, chain under way
        n0 = ctx.launch_count()
        t0 = time.perf_counter()
        bl.sample_hypers(Z, y)
        ms = (time.perf_counter() - t0) * 1e3
        res["sample_hypers_speculative" if spec else "sample_hypers_sequential"] = {
            "wall_ms_nSamples_10": ms, "kernel_launches": ctx.launch_count() - n0}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()

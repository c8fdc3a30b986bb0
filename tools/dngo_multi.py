"""DNGO acquisition over G GPUs of one process (b7_comm_init_all) at config 4's shape: N = 20 000 observations, d = 6, a ReLU
basis 6 -> 50 (D = 50), one head row, EI.  For every G in {1, 2, 4, 8} the box has:

  * weak scaling: 2^22 Sobol candidates per GPU, median wall ms of b7_dngo_score_multi (argmax only, no scores read back);
  * strong scaling: 2^24 candidates in total, the same; the nominee must equal G = 1's;
  * median wall ms of b7_blr_fit_multi;
  * end to end: host basis of the observations + b7_blr_fit_multi + b7_dngo_score_multi over the weak-scaling grid.

Each call is synchronous (it returns after every device finished), so host wall time around it is the step time, thread fan-out
and combine included.  Prints one JSON object (and writes it to --out when given).  Needs CUDA devices; there is no CPU path.
Run: python tools/dngo_multi.py [--out profiles/dngo_multi_r01.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle")]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()
        return out
    except Exception:
        return ["unknown"]


def median_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import b7_oracle as o
    from bot7_b200 import _lib as L
    from bot7_b200 import parallel
    d, D, N = 6, 50, a.N
    r = np.random.default_rng(0)
    W, b = r.standard_normal((D, d)) * np.sqrt(2.0 / d), 0.1 * r.standard_normal(D)      # He-scaled: EI is not 0 everywhere
    Xo = o.sobol_points(d, N)
    y = o.hartmann6(Xo)
    y = (y - y.mean()) / y.std()
    fmin = float(y.min())
    hyp = np.array([[0.0, np.log(1e2), float(y.mean())]])
    n_dev = L.lib().b7_device_count()
    res = {"tool": "tools/dngo_multi.py", "date": time.strftime("%Y-%m-%d"), "gpus": gpu_info(), "N": N, "d": d, "D": D, "S": 1,
           "score": "EI", "reps": a.reps, "weak_per_gpu": 1 << 22, "strong_total": 1 << 24, "runs": []}
    ref = None
    for G in (1, 2, 4, 8):
        if G > n_dev:
            continue
        comm = parallel.Comm.all(G)
        Z0 = np.maximum(Xo @ W.T + b, 0.0)
        blrs, _ = comm.blr_fit(Z0, y, hyp)
        row = {"G": G}
        for label, M in (("weak", G << 22), ("strong", 1 << 24)):
            gs = comm.sobol_grid(d, 1 + N, M)
            out = {}

            def score():
                out["r"] = comm.dngo_score(blrs, gs, [W], [b], True, L.SCORE_EI, 0.0, 0, -1.0, fmin)
            med, lo, hi = median_ms(score, a.reps)
            row[label] = {"M": M, "ms_median": med, "ms_min": lo, "ms_max": hi, "candidates_per_s": M / (med * 1e-3),
                          "argmax": out["r"][1], "best": out["r"][0]}
            if label == "weak":
                def e2e():
                    Z = np.maximum(Xo @ W.T + b, 0.0)
                    hs, _ = comm.blr_fit(Z, y, hyp)
                    comm.dngo_score(hs, gs, [W], [b], True, L.SCORE_EI, 0.0, 0, -1.0, fmin)
                    comm.free_blr(hs)
                med, lo, hi = median_ms(e2e, max(5, a.reps // 3))
                row["e2e_weak"] = {"ms_median": med, "ms_min": lo, "ms_max": hi,
                                   "includes": "host basis of the observations + b7_blr_fit_multi + b7_dngo_score_multi"}
            for g in gs:
                g.free()
        if ref is None:
            ref = row["strong"]["argmax"], row["strong"]["best"]
        assert (row["strong"]["argmax"], row["strong"]["best"]) == ref, ("strong-scaling nominee differs from G = 1", row, ref)

        def fit():
            hs, _ = comm.blr_fit(Z0, y, hyp)
            comm.free_blr(hs)
        med, lo, hi = median_ms(fit, a.reps)
        row["blr_fit_multi"] = {"ms_median": med, "ms_min": lo, "ms_max": hi}
        comm.free_blr(blrs)
        comm.close()
        res["runs"].append(row)
        print(json.dumps(row), flush=True)
    g1 = res["runs"][0]
    for row in res["runs"]:
        row["weak_efficiency"] = g1["weak"]["ms_median"] / row["weak"]["ms_median"]
        row["strong_speedup"] = g1["strong"]["ms_median"] / row["strong"]["ms_median"]
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()

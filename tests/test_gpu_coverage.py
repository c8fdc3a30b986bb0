"""Breadth of the GPU path: the kernel instantiations, candidate panels and execution variants that the library selects at
run time, each against the oracle and, where the code claims it, against another variant bit for bit.

A. every DT bucket of the two covariance ladders (cov.cu, posterior_i8.cu), both kernels, both posterior paths;
B. scoring passes of several candidate panels with a partial last one and removed rows at the panel boundaries;
C. the B7_* execution variants, one child process each (tests/gpu_variant_worker.py).

Bars are the suite's own (test_gpu_parity.py): mean 1e-9 of max(|m|, 1); variance 1e-9 sf2 and 1e-9 relative where
var >= 1e-3 sf2; log marginal likelihood 1e-11 relative; EI 1e-7 relative with a floor of 1e-6 of the largest score;
argmax identical, or a near-tie with a score gap <= 1e-12 relative.  Importing this module needs no GPU:
tests/test_coverage_inventory.py reads the lists below.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import gpu_variant_worker as W
from bot7_b200 import _lib as L
from bot7_b200 import grids, models, parallel
from test_gpu_parity import make_problem, posterior_errors, record_parity, rel

pytestmark = pytest.mark.gpu

# A: lower and upper edge of every DT bucket of cov.cu (2, 4, 6, 8, 16, 24, 40) and posterior_i8.cu (2, 4, ..., 32, 40)
SWEEP_D = (1, 4, 5, 7, 8, 9, 12, 13, 16, 17, 20, 21, 24, 25, 32, 33, 39)
SWEEP_N, SWEEP_S, SWEEP_M = 300, 2, 64 * 31 + 5
BLR_D, BLR_HIDDEN, BLR_INPUT_DIMS = W.BLR_D, W.BLR_HIDDEN, W.BLR_INPUT_DIMS

# C: (id, environment, workloads, expectation).  "same": bit-identical to the default run of the workload;
# "same_as:<id>": bit-identical to that variant's run; "oracle": the oracle bars, INT8 <-> FP64 agreement with the default
# run where that pairing exists, and at least one output differs in bits from the default run (the knob changed the arithmetic).
BATCHED = ("batched_ardse", "batched_matern52")
VARIANTS = [
    ("post_pair_0", {"B7_POST_PAIR": "0"}, BATCHED + ("latency",), "same"),
    ("post_pair_0_chunk_1", {"B7_POST_PAIR": "0", "B7_POST_CHUNK": "1"}, BATCHED, "same"),
    ("post_pair_0_chunk_3", {"B7_POST_PAIR": "0", "B7_POST_CHUNK": "3"}, BATCHED, "same"),
    ("post_group_1", {"B7_POST_GROUP": "1"}, BATCHED, "same"),
    ("post_group_5", {"B7_POST_GROUP": "5"}, BATCHED, "same"),
    ("post_pair_0_group_1", {"B7_POST_PAIR": "0", "B7_POST_GROUP": "1"}, BATCHED, "same"),
    ("post_pair_0_group_5", {"B7_POST_PAIR": "0", "B7_POST_GROUP": "5"}, BATCHED, "same"),
    ("kstar_overlap_0", {"B7_KSTAR_OVERLAP": "0"}, BATCHED + ("latency",), "same"),
    ("profiling", {}, BATCHED + ("latency",), "same"),
    ("trail_chunk_1", {"B7_TRAIL_CHUNK": "1"}, BATCHED, "same"),
    ("trail_chunk_3", {"B7_TRAIL_CHUNK": "3"}, BATCHED, "same"),
    ("trtri_chunk_1", {"B7_TRTRI_CHUNK": "1"}, BATCHED, "same"),
    ("trtri_chunk_7", {"B7_TRTRI_CHUNK": "7"}, BATCHED, "same"),
    ("potrf_pdl_0", {"B7_POTRF_PDL": "0"}, ("latency",), "same"),
    ("potrf_graph_0", {"B7_POTRF_GRAPH": "0"}, ("latency",), "same"),
    ("potrf_graph_1", {"B7_POTRF_GRAPH": "1"}, ("latency",), "same"),
    ("cache_fraction_0", {"B7_CACHE_FRACTION": "0"}, BATCHED + ("latency",), "same"),
    ("potrf_slice_0", {"B7_POTRF_SLICE": "0"}, ("latency",), "same"),
    ("potrf_i8_0", {"B7_POTRF_I8": "0"}, BATCHED, "oracle"),
    # the row-sliced schedule runs the FP64 DMMA sequence of the batched tile kernels, not the INT8 trailing updates
    ("potrf_slice_1", {"B7_POTRF_SLICE": "1"}, BATCHED, "same_as:potrf_i8_0"),
    ("trtri_i8_0", {"B7_TRTRI_I8": "0"}, BATCHED, "oracle"),
    ("posterior_i8_0", {"B7_POSTERIOR_I8": "0"}, BATCHED + ("latency",), "oracle"),
    ("potrf_w_2", {"B7_POTRF_W": "2"}, BATCHED, "oracle"),
    ("potrf_w_8", {"B7_POTRF_W": "8"}, BATCHED, "oracle"),
    ("blr_dmma_0", {"B7_BLR_DMMA": "0"}, ("blr",), "oracle"),
]
PROFILED = {"profiling"}
# knobs that no variant runs, and why
EXCLUDED_KNOBS = {
    "B7_POST_DBG": "measurement switch of the pair kernel: its results are wrong by design",
    "B7_POTRF_TRACE": "prints per-kernel timings of the factorisation to stderr; forces the un-captured schedule",
    "B7_NCCL_LIB": "path of the NCCL library of the multi-GPU path, covered by the multi-GPU tests",
    "B7_DEBUG": "stderr messages about the CUDA graph capture of the factorisation",
}
VARIANT_TIMEOUT_S = 600


_worst = {}


def note(part, bar, value):
    """Largest measured error per part and bar: printed at the end of the module, and written to
    $BOT7_PARITY_DIR/parity_r02.json (key gpu_coverage) when that variable is set."""
    d = _worst.setdefault(part, {})
    d[bar] = max(d.get(bar, 0.0), float(value))
    return value


@pytest.fixture(scope="module", autouse=True)
def report_worst_errors():
    yield
    if _worst:
        print("\nworst measured errors:", _worst)
        record_parity("gpu_coverage", _worst)


def _acq_score(f, grid, fmin, kind=L.SCORE_EI):
    sc = np.empty(grid.rows())
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
    L.check(L.lib().b7_acq_score(f.handle, grid.handle, kind, 0.0, 0, -1.0, fmin, L.dptr(sc), C.byref(am), C.byref(amo), C.byref(best),
                                 C.byref(nn)))
    return sc, am.value, amo.value, best.value, nn.value


def check_argmax(idx, ref_score, ref_idx, what=""):
    """Selected candidate (1-based, indexing ref_score): identical to the oracle's, or a near-tie that is reported."""
    if idx == ref_idx:
        return 0.0
    assert idx >= 1, f"{what}: no candidate selected (oracle {ref_idx})"
    best = ref_score[ref_idx - 1]
    gap = abs(ref_score[idx - 1] - best) / abs(best)
    print(f"{what}: argmax {idx} vs oracle {ref_idx}, near-tie gap {gap:.2e}")
    assert gap <= 1e-12, f"{what}: argmax differs beyond a near-tie: {idx} vs {ref_idx} (gap {gap})"
    return gap


def assert_posterior_bars(mu, var, mu_ref, var_ref, sf2, what, part):
    e = posterior_errors(mu, var, mu_ref, var_ref, sf2)
    for bar in ("mean", "var_over_sf2", "var_rel_where_ge_1e-3_sf2"):
        note(part, bar, e[bar])
    assert e["mean"] <= 1e-9, (what, e)                          # mean 1e-9 of max(|m|, 1)
    assert e["var_over_sf2"] <= 1e-9, (what, e)                  # variance 1e-9 sf2
    assert e["var_rel_where_ge_1e-3_sf2"] <= 1e-9, (what, e)     # and 1e-9 relative down to 1e-3 sf2
    return e


def oracle_draws(oracle, Xo, y, hyp, Xc, kernel):
    """fit + predict of every draw: (fits, means[S, M], vars[S, M])."""
    fits = [oracle.gp_fit(Xo, y, h, kernel) for h in hyp]
    mv = [oracle.gp_predict(fit, Xc) for fit in fits]
    return fits, np.array([m for m, _ in mv]), np.array([v for _, v in mv])


def ei_average(oracle, means, variances, fmin):
    return oracle.mc_average([oracle.ei_compute(m, v, fmin, 0.0) for m, v in zip(means, variances)])


@pytest.fixture
def restore_path(ctx):
    keep = ctx.posterior_path()
    yield
    ctx.set_posterior_path(keep)


# ---------------------------------------------------------------------------------- A. dimension and kernel sweep

def sweep_problem(oracle, d):
    """N = 300 (3 row blocks: the pair kernel has a phantom block), S = 2, M = 64 * 31 + 5.  Length-scales are set from the
    median distance of a candidate to its nearest observation (half of it, times exp(U(-0.4, 0.4)) per dimension): scaling
    with sqrt(d) alone leaves K* ~ 0 or ~ sf2 for every candidate at large d, where any kernel passes.  Every third
    candidate is moved next to an observation (scaled distance 0.05 ... 1 under draw 0), which gives the low-variance tail."""
    Xo, y, hyp, Xc = make_problem(oracle, SWEEP_N, d, SWEEP_S, SWEEP_M, 1e-2, seed=d)
    r = np.random.default_rng(100 + d)
    nn2 = ((Xc[:, None, :] - Xo[None, :, :]) ** 2).sum(-1).min(1)
    hyp[:, :d] = np.log(0.5 * np.sqrt(np.median(nn2))) + r.uniform(-0.4, 0.4, (SWEEP_S, d))
    near = np.arange(0, SWEEP_M, 3)
    u = r.normal(size=(near.size, d))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    Xc[near] = Xo[r.integers(0, SWEEP_N, near.size)] + r.uniform(0.05, 1.0, (near.size, 1)) * u * np.exp(hyp[0, :d])
    return Xo, y, hyp, Xc


@pytest.mark.parametrize("kern", ["ardse", "matern52"])
@pytest.mark.parametrize("d", SWEEP_D)
def test_every_dimension_bucket_both_kernels_both_paths(ctx, oracle, restore_path, d, kern):
    Xo, y, hyp, Xc = sweep_problem(oracle, d)
    kid = models.KERNELS[kern]
    fits, m_ref, v_ref = oracle_draws(oracle, Xo, y, hyp, Xc, kid)
    sf2 = np.array([fit["sf2"] for fit in fits])
    # not a trivial problem: both a well-determined and a prior-like population of candidates
    for s in range(SWEEP_S):
        assert np.mean(v_ref[s] <= 0.5 * sf2[s]) >= 0.1 and np.mean(v_ref[s] >= 0.9 * sf2[s]) >= 0.1
    fmin = float(y.min())
    ref = ei_average(oracle, m_ref, v_ref, fmin)
    _, ref_idx, _ = oracle.argmax_first(ref)
    # non-finite coordinate d - 1 (the last term of every distance and of the finish kernel's NaN test)
    i_nan, i_inf = 7, SWEEP_M - 2
    bad = Xc.copy()
    bad[i_nan, d - 1] = np.nan
    bad[i_inf, d - 1] = np.inf
    nan_rows, prior_rows = ([i_nan], [i_inf]) if kern == "ardse" else ([i_nan, i_inf], [])
    ok = np.ones(SWEEP_M, bool)
    ok[[i_nan, i_inf]] = False
    grid, grid_bad = grids.DeviceGrid.from_host(Xc), grids.DeviceGrid.from_host(bad)
    out = {}
    for path in (L.PATH_FP64_DMMA, L.PATH_INT8_OZAKI):
        ctx.set_posterior_path(path)
        f = models.GPFactors(Xo, y, hyp, kern)
        assert (f.info == 0).all() and (f.jitter == 0).all()
        assert note("A", "logml_rel", rel(f.logml, np.array([fit["logml"] for fit in fits]), 1e-300)) <= 1e-11
        mv = [f.predict(s, Xc) for s in range(SWEEP_S)]
        for s in range(SWEEP_S):
            assert_posterior_bars(mv[s][0], mv[s][1], m_ref[s], v_ref[s], sf2[s], (d, kern, path, s), "A")
        sc, am, amo, best, nn = _acq_score(f, grid, fmin)
        assert note("A", "ei_rel", rel(sc, ref, 1e-6 * max(ref.max(), 1e-300))) <= 1e-7
        assert nn == 0 and am == amo
        check_argmax(am, ref, ref_idx, f"d={d} {kern} path {path}")
        for s in range(SWEEP_S):
            m1, v1 = f.predict(s, bad)
            assert np.isnan(m1[nan_rows]).all() and np.isnan(v1[nan_rows]).all()
            for r_ in prior_rows:                                    # ARD-SE, infinite coordinate: k* = 0, the prior
                assert m1[r_] == hyp[s, d + 2] and abs(v1[r_] / sf2[s] - 1) <= 1e-15
            assert np.array_equal(m1[ok], mv[s][0][ok]) and np.array_equal(v1[ok], mv[s][1][ok])
        _, am_b, _, _, nn_b = _acq_score(f, grid_bad, fmin)
        assert nn_b == len(nan_rows) and am_b - 1 not in nan_rows
        out[path] = mv
        f.free()
    for s in range(SWEEP_S):                                         # the path-agreement bars of test_gpu_parity.py
        a, b = out[L.PATH_FP64_DMMA][s], out[L.PATH_INT8_OZAKI][s]
        assert note("A", "paths_var_over_sf2", np.max(np.abs(a[1] - b[1])) / sf2[s]) <= 1e-12
        assert note("A", "paths_mean", np.max(np.abs(a[0] - b[0]))) <= 1e-10
    grid.free()
    grid_bad.free()


# ---------------------------------------------------------------------------------- B. several candidate panels

PANEL_N, PANEL_D, PANEL_S = 2100, 6, 5
_panel_cache = {}


@pytest.fixture(scope="module")
def panel_problem(ctx, oracle):
    """N = 2100 (Np = 2176: one panel = 128 x SMs candidates), M = 2P + 777 (three panels, the last partial), 5 draws.  The
    oracle's moments of all 5 draws are computed once and shared by every case."""
    if "p" not in _panel_cache:
        import torch
        P = 128 * torch.cuda.get_device_properties(0).multi_processor_count
        M = 2 * P + 777
        Xo, y, hyp, Xc = make_problem(oracle, PANEL_N, PANEL_D, PANEL_S, M, 1e-2, seed=21)
        _, m_ref, v_ref = oracle_draws(oracle, Xo, y, hyp, Xc, 0)
        removed = sorted({P - 1, P, 2 * P - 1, 2 * P, M - 1})          # both sides of each panel boundary, and the last row
        _panel_cache["p"] = dict(P=P, M=M, Xo=Xo, y=y, hyp=hyp, Xc=Xc, m_ref=m_ref, v_ref=v_ref, removed=removed)
    return _panel_cache["p"]


@pytest.mark.parametrize("S,path", [(1, L.PATH_INT8_OZAKI), (2, L.PATH_FP64_DMMA), (5, L.PATH_INT8_OZAKI), (5, L.PATH_FP64_DMMA)])
def test_multi_panel_acquisition(ctx, oracle, restore_path, panel_problem, S, path):
    # (1, INT8): one draw, per-draw posterior passes; (5, INT8): the two-stream double-buffered pass, an odd S wraps the
    # buffer parity; FP64: per-draw passes on the DMMA kernels
    p = panel_problem
    P, M, Xo, y, hyp, Xc = p["P"], p["M"], p["Xo"], p["y"], p["hyp"][:S], p["Xc"]
    ctx.set_posterior_path(path)
    f = models.GPFactors(Xo, y, hyp)
    assert (f.info == 0).all() and f.padded_n() == 2176
    grid = grids.DeviceGrid.from_host(Xc)
    for r_ in reversed(p["removed"]):                                # descending: compacted index = original index + 1
        grid.remove(r_ + 1)
    live = np.ones(M, bool)
    live[p["removed"]] = False
    fmin = float(y.min())
    sc, am, amo, best, nn = _acq_score(f, grid, fmin)
    # 1. against the oracle; removed rows read NaN and are not counted as NaN scores
    ref = ei_average(oracle, p["m_ref"][:S], p["v_ref"][:S], fmin)
    assert np.isnan(sc[~live]).all() and nn == 0
    assert note("B", "ei_rel", rel(sc[live], ref[live], 1e-6 * ref[live].max())) <= 1e-7
    _, ref_idx, _ = oracle.argmax_first(np.where(live, ref, np.nan))
    check_argmax(amo, ref, ref_idx, f"S={S} path {path}")
    assert am == amo - int(np.sum(~live[:amo - 1]))
    # 2. the same kernels grouped differently: per-draw moments of b7_gp_predict scored by b7_score_moments, bit for bit
    mv = [f.predict(s, Xc) for s in range(S)]
    mean = np.ascontiguousarray(np.array([m for m, _ in mv])[:, live])
    var = np.ascontiguousarray(np.array([v for _, v in mv])[:, live])
    sc2 = np.empty(int(live.sum()))
    am2, best2, nn2 = C.c_int64(), C.c_double(), C.c_int64()
    L.check(L.lib().b7_score_moments(ctx.handle, L.SCORE_EI, L.dptr(mean), L.dptr(var), S, sc2.size, 0.0, 0, -1.0, fmin, L.dptr(sc2),
                                     C.byref(am2), C.byref(best2), C.byref(nn2)))
    assert np.array_equal(sc2, sc[live])
    assert (am2.value, best2.value, nn2.value) == (am, best, nn)
    # 3. three shards with boundaries off the 64-candidate tiles and off the panels: same scores, same combined triple
    bounds = [0, P // 2 + 3, P + P // 2 + 5, M]
    assert all(b % 64 and b % P for b in bounds[1:-1])
    parts, trips = [], []
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        part = np.empty(r1 - r0)
        o_, b_, n_ = C.c_int64(), C.c_double(), C.c_int64()
        L.check(L.lib().b7_acq_score_range(f.handle, grid.handle, r0, r1 - r0, L.SCORE_EI, 0.0, 0, -1.0, fmin, L.dptr(part), C.byref(o_),
                                           C.byref(b_), C.byref(n_)))
        parts.append(part)
        trips.append((b_.value, o_.value, n_.value))
    assert np.array_equal(np.concatenate(parts), sc, equal_nan=True)
    assert parallel.combine_argmax(trips) == (best, amo, nn)
    grid.free()
    f.free()


# ---------------------------------------------------------------------------------- C. execution variants

_runs = {}
_oracle_cache = {}


def run_variant(tmp_dir, workload, env_extra, profile=False):
    """One child process: the parent's environment without any inherited B7_* variable, plus the variant's, plus
    B7_CACHE_FRACTION=0.05 (unless the variant sets it).  Returns the worker's outputs."""
    key = (workload, tuple(sorted(env_extra.items())), profile)
    if key in _runs:
        return _runs[key]
    env = {k: v for k, v in os.environ.items() if not k.startswith("B7_")}
    env["B7_CACHE_FRACTION"] = "0.05"
    env.update(env_extra)
    out_path = os.path.join(tmp_dir, "run%d.npz" % len(_runs))
    cmd = [sys.executable, os.path.join(os.path.dirname(os.path.abspath(__file__)), "gpu_variant_worker.py"), workload, out_path]
    if profile:
        cmd.append("--profile")
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=VARIANT_TIMEOUT_S)
    assert p.returncode == 0, f"{workload} {env_extra}: exit {p.returncode}\n{p.stdout[-2000:]}\n{p.stderr[-3000:]}"
    with np.load(out_path) as z:
        out = {k: z[k] for k in z.files}
    os.remove(out_path)
    _runs[key] = out
    return out


def bit_differences(a, b):
    assert sorted(a) == sorted(b)
    return [k for k in sorted(a) if not np.array_equal(a[k], b[k], equal_nan=True)]


def oracle_batched(oracle, workload):
    if workload not in _oracle_cache:
        kernel = {"batched_ardse": 0, "batched_matern52": 1, "jitter": 0}[workload]
        Xo, y, hyp, Xc = W.batched_problem(workload == "jitter")
        fits, m_ref, v_ref = oracle_draws(oracle, Xo, y, hyp, Xc, kernel)
        _oracle_cache[workload] = dict(y=y, hyp=hyp, fits=fits, m_ref=m_ref, v_ref=v_ref,
                                       score=ei_average(oracle, m_ref, v_ref, float(y.min())))
    return _oracle_cache[workload]


def check_batched_against_oracle(oracle, workload, out):
    o = oracle_batched(oracle, workload)
    fits = o["fits"]
    assert (out["info"] == 0).all() and (out["jitter"] == 0).all()
    assert note("C", "logml_rel", rel(out["logml"], np.array([fit["logml"] for fit in fits]), 1e-300)) <= 1e-11
    for s in W.BATCHED_DRAWS:
        assert_posterior_bars(out[f"mean{s}"], out[f"var{s}"], o["m_ref"][s], o["v_ref"][s], fits[s]["sf2"], (workload, s), "C")
        inv = np.linalg.inv(np.tril(fits[s]["L"]))                   # the handle holds L^-1 (the bar of the inversion tests)
        scale = np.max(np.abs(out[f"factor{s}"]))
        assert note("C", "inverse_factor_over_max", np.max(np.abs(out[f"factor{s}"] - np.tril(inv))) / scale) <= 1e-9
    assert note("C", "ei_rel", rel(out["score"], o["score"], 1e-6 * o["score"].max())) <= 1e-7
    _, ref_idx, _ = oracle.argmax_first(o["score"])
    check_argmax(int(out["argmax"][0]), o["score"], ref_idx, workload)
    assert out["argmax"][2] == 0


def check_latency_against_oracle(oracle, out):
    Xo, y, hyp, Xc, steps = W.latency_problem()
    for k, h in enumerate(steps):
        assert (out[f"info{k}"] == 0).all()
        assert note("C", "logml_rel", rel(out[f"logml{k}"], np.array([oracle.gp_fit(Xo, y, row, 0)["logml"] for row in h]), 1e-300)) <= 1e-11
    fits, m_ref, v_ref = oracle_draws(oracle, Xo, y, steps[-1], Xc, 0)
    for s in range(len(fits)):
        assert_posterior_bars(out[f"mean{s}"], out[f"var{s}"], m_ref[s], v_ref[s], fits[s]["sf2"], ("latency", s), "C")
    ref = ei_average(oracle, m_ref, v_ref, float(y.min()))
    assert note("C", "ei_rel", rel(out["score"], ref, 1e-6 * ref.max())) <= 1e-7
    check_argmax(int(out["argmax"][0]), ref, oracle.argmax_first(ref)[1], "latency")


def check_blr_against_oracle(oracle, out):
    for D, H in zip(W.BLR_D, W.BLR_HIDDEN):
        Ws, bs, Xo, y, hyp, Xc = W.blr_problem(D, H)
        Z0, Z1 = oracle.mlp_features(Xo, Ws, bs), oracle.mlp_features(Xc, Ws, bs)
        assert (out[f"D{D}_info"] == 0).all()
        assert note("C", "blr_features", np.max(np.abs(out[f"D{D}_features"] - Z1)) / max(1.0, np.max(np.abs(Z1)))) <= 1e-12
        per = []
        for s in range(hyp.shape[0]):
            mr, vr = oracle.blr_predict(oracle.blr_fit(Z0, y, hyp[s]), Z1)
            assert note("C", "blr_mean", rel(out[f"D{D}_mean{s}"], mr, 1.0)) <= 1e-10, (D, s)
            assert note("C", "blr_var_rel", rel(out[f"D{D}_var{s}"], vr, 1e-300)) <= 1e-9, (D, s)
            per.append(oracle.ei_compute(mr, vr, float(y.min()), 0.0))
        ref = oracle.mc_average(per)
        _, i, _ = oracle.argmax_first(ref)
        assert note("C", "ei_rel", rel(out[f"D{D}_blr_score"], ref, 1e-6 * max(ref.max(), 1e-300))) <= 1e-7
        check_argmax(int(out[f"D{D}_blr_argmax"][0]), ref, i, f"blr D={D}")
        if D <= 63:
            assert note("C", "ei_rel", rel(out[f"D{D}_dngo_score"], ref, 1e-6 * max(ref.max(), 1e-300))) <= 1e-7
            check_argmax(int(out[f"D{D}_dngo_argmax"][0]), ref, i, f"dngo D={D}")
        else:                                                        # as test_dngo_tile_kernel_shapes_vs_oracle expects
            assert out[f"D{D}_dngo_error"][0] == 1.0


def check_paths_agree(workload, out, ref):
    """INT8 <-> FP64 agreement with the default run, at the bars of the path tests of test_gpu_parity.py: log ml 1e-12
    relative and the factor 1e-11 of its largest entry (INT8 trailing update / inversion against FP64), mean 1e-10 and
    variance 1e-12 sf2 (INT8 against FP64 posterior)."""
    if workload == "blr":
        return
    key = "logml" if "logml" in out else "logml2"
    assert note("C", "paths_logml_rel", rel(out[key], ref[key], 1e-300)) <= 1e-12
    hyp = W.batched_problem()[2] if workload in BATCHED else W.latency_problem()[4][-1]
    d = hyp.shape[1] - 3
    for key in sorted(out):
        if key.startswith("factor"):
            assert note("C", "paths_factor_over_max", np.max(np.abs(out[key] - ref[key])) / np.max(np.abs(ref[key]))) <= 1e-11, key
        elif key.startswith("mean"):
            assert note("C", "paths_mean", np.max(np.abs(out[key] - ref[key]))) <= 1e-10, key
        elif key.startswith("var"):
            sf2 = np.exp(2 * hyp[int(key[3:]), d])
            assert note("C", "paths_var_over_sf2", np.max(np.abs(out[key] - ref[key])) / sf2) <= 1e-12, key


CASES = [(vid, env, wl, expect) for vid, env, wls, expect in VARIANTS for wl in wls]


@pytest.mark.parametrize("vid,env,workload,expect", CASES, ids=[f"{c[0]}-{c[2]}" for c in CASES])
def test_execution_variant(ctx, oracle, tmp_path_factory, vid, env, workload, expect):
    tmp = str(tmp_path_factory.getbasetemp())
    out = run_variant(tmp, workload, env, vid in PROFILED)
    ref = run_variant(tmp, workload, {})
    if expect == "same":
        assert bit_differences(out, ref) == []
        return
    if expect.startswith("same_as:"):
        other = dict(VARIANTS_BY_ID[expect.split(":", 1)[1]][1])
        assert bit_differences(out, run_variant(tmp, workload, other)) == []
        return
    if workload in BATCHED:
        check_batched_against_oracle(oracle, workload, out)
    elif workload == "latency":
        check_latency_against_oracle(oracle, out)
    else:
        check_blr_against_oracle(oracle, out)
    check_paths_agree(workload, out, ref)
    assert bit_differences(out, ref), f"{vid} on {workload}: bit-identical to the default run, the knob changed nothing"


VARIANTS_BY_ID = {v[0]: v for v in VARIANTS}


@pytest.mark.parametrize("workload", ["batched_ardse", "batched_matern52", "latency", "blr"])
def test_default_run_of_every_workload_meets_the_oracle(ctx, oracle, tmp_path_factory, workload):
    out = run_variant(str(tmp_path_factory.getbasetemp()), workload, {})
    if workload in BATCHED:
        check_batched_against_oracle(oracle, workload, out)
    elif workload == "latency":
        check_latency_against_oracle(oracle, out)
    else:
        check_blr_against_oracle(oracle, out)


def test_jitter_retry_of_one_draw_inside_an_int8_batch(ctx, oracle, tmp_path_factory):
    # 13 draws, 18 row blocks: the batched factorisation runs the INT8 trailing updates; draw 7 (sigma_n^2 = 1e-18 on
    # repeated observations) fails and takes the utils.math.chol retry alone, with the exact eps sequence of the oracle
    out = run_variant(str(tmp_path_factory.getbasetemp()), "jitter", {})
    o = oracle_batched(oracle, "jitter")
    fits = o["fits"]
    j = W.JITTER_DRAW
    assert fits[j]["iters"] >= 1 and out["jitter"][j] == fits[j]["jitter"]
    assert (out["info"] == 0).all()
    healthy = [s for s in range(len(fits)) if s != j]
    assert (out["jitter"][healthy] == 0).all()
    assert note("C_jitter", "logml_rel", rel(out["logml"][healthy], np.array([fits[s]["logml"] for s in healthy]), 1e-300)) <= 1e-11
    for s in (0, 12):
        assert_posterior_bars(out[f"mean{s}"], out[f"var{s}"], o["m_ref"][s], o["v_ref"][s], fits[s]["sf2"], ("jitter", s), "C_jitter")
    # the jittered draw: the ill-conditioned bars of the noiseless tests (variance 1e-9 sf2, mean 1e-6 absolute)
    assert note("C_jitter", "jittered_var_over_sf2", np.max(np.abs(out[f"var{j}"] - o["v_ref"][j])) / fits[j]["sf2"]) <= 1e-9
    assert note("C_jitter", "jittered_mean_abs", np.max(np.abs(out[f"mean{j}"] - o["m_ref"][j]))) <= 1e-6

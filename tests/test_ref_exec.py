"""Oracle and CUDA path against vectors produced by EXECUTING the reference's own Lua (tests/golden/ref_exec.npz).

The vectors come from tests/golden/make_ref_exec.py: the reference modules grids/sobol.lua + utils/bits.lua, utils/math.lua,
scores/*.lua, utils/tensor.lua and benchmarks/*.lua run unmodified under tools/minilua (a Lua 5.1 interpreter with a
numpy-backed Torch7 stand-in written for this repository, because the image has no Lua runtime).  This pins the functions that
`oracle/b7_oracle.py` marks PINNED to outputs of the reference source itself instead of to hand-traced known answers only.
Caveat, stated once: the runtime under the reference code is numpy, not TH -- same IEEE operations in the same order, but `exp`
is numpy's.

CPU: the oracle equals the vectors (bit for bit wherever the arithmetic is +, -, *, /, sqrt, exp in a fixed order); where the
reference tree is present a subset is re-executed live and compared with the committed file.
GPU: the CUDA path equals the vectors at the north-star bars (Sobol and compaction bit-exact, EI 1e-7, bound bit-exact).
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "ref_exec.npz")
REF = os.environ.get("BOT7_REFERENCE", "")         # a checkout of the reference bot7 Lua source, if any


@pytest.fixture(scope="module")
def G():
    return np.load(GOLD)


SOBOL_CASES = {                      # name -> (dims, size, skip, mins?, maxes?)
    "sobol_d2_n200": (2, 200, 1, False, False), "sobol_d6_n256": (6, 256, 1, False, False), "sobol_d20_n48": (20, 48, 1, False, False),
    "sobol_d39_n24": (39, 24, 1, False, False), "sobol_d6_n40_skip37": (6, 40, 37, False, False),
    "sobol_d6_n64_scaled": (6, 64, 1, True, True), "sobol_d6_n64_mins": (6, 64, 1, True, False), "sobol_d6_n64_maxes": (6, 64, 1, False, True),
}


# ---------------------------------------------------------------------------------- oracle vs executed reference (CPU)

@pytest.mark.parametrize("name", sorted(SOBOL_CASES))
def test_oracle_sobol_equals_the_executed_reference(oracle, G, name):
    dims, size, skip, lo, hi = SOBOL_CASES[name]
    mins = G["sobol_mins6"] if lo else None
    maxes = G["sobol_maxes6"] if hi else None
    assert np.array_equal(oracle.sobol_points(dims, size, skip, mins, maxes), G[name])


def test_oracle_sobol_state_and_direction_numbers(oracle, G):
    # a second generate() on the same object and the __call__ form restart from the same seed: the same 16 points twice
    two = G["sobol_d3_two_calls"]
    assert np.array_equal(two[:16], oracle.sobol_points(3, 16)) and np.array_equal(two[16:], two[:16])
    # create_bank's initial values, then the recurrence-filled, column-scaled integers after the first point
    b0, b1 = G["sobol_bank_initial"][:39], G["sobol_bank_scaled"][:39]
    unscaled = oracle.sobol_bank_unscaled(39)
    assert np.array_equal(b0[b0 != 0], unscaled[b0 != 0])
    assert np.array_equal(b1, oracle.sobol_direction_integers(39))
    assert G["sobol_recipd"][0] == 2.0 ** -30
    # the doubles-based XOR of utils/bits.lua is the integer XOR
    assert np.array_equal(G["xor_out"], [float(int(a) ^ int(b)) for a, b in G["xor_pairs"]])
    for a, b in G["xor_pairs"]:
        assert oracle.bitwise_xor_literal(float(a), float(b)) == float(int(a) ^ int(b))


def test_oracle_erf_cdf_pdf_equal_the_executed_reference(oracle, G):
    x = G["math_x"]
    assert np.array_equal(oracle.erf_ref(x), G["math_erf"])
    assert np.array_equal(oracle.norm_pdf_ref(x), G["math_pdf"])
    assert np.array_equal(oracle.norm_cdf_ref(x), G["math_cdf"])


def test_oracle_scores_equal_the_executed_reference(oracle, G):
    m, v, fmin = G["score_mean"], G["score_var"], float(G["score_fmin"][0])
    for key, t in (("score_ei_t0", 0.0), ("score_ei_t01", 0.1)):
        assert np.array_equal(oracle.ei_compute(m, v, fmin, t), G[key], equal_nan=True)
    assert np.isnan(G["score_ei_t0"]).sum() == 1 and np.isnan(G["score_ei_t0"][2])       # 0 / 0 at sigma = 0, improvement = 0: NaN survives the clamp
    assert np.array_equal(oracle.cb_compute(m, v, 1.0, "lower", -1.0), G["score_lcb"])
    assert np.array_equal(oracle.cb_compute(m, v, 2.0, "upper", 1.0), G["score_ucb"])
    assert np.array_equal(oracle.cb_compute(m, v, 0.5, "lower", 1.0), G["score_lcb_pos"])
    # scores/expected_improvement.lua:70 reads the GLOBAL `config`: without it EI.compute raises (the oracle takes the tradeoff as an argument)
    assert G["score_ei_without_global"][0] == 1.0


def test_oracle_jitter_policy_equals_the_executed_reference(oracle, G):
    for name in ("spd", "semi", "neg"):
        L, jit, iters = oracle.chol_jitter(G["chol_%s_in" % name])
        assert np.allclose(np.tril(L), G["chol_%s_L" % name], rtol=1e-13, atol=0.0)
        assert iters == int(G["chol_%s_iterations" % name][0])
        printed = float(G["chol_%s_jitter_printed" % name][0])                       # the reference prints it with %.2e
        assert (jit == 0.0 and printed == 0.0) or abs(jit - printed) <= 0.006 * printed
    assert int(G["chol_semi_iterations"][0]) == 1 and int(G["chol_neg_iterations"][0]) == 194


def test_compaction_and_objectives_equal_the_executed_reference(oracle, G):
    src = G["steal_src"]
    rest = np.delete(src, 3, axis=0)                     # steal row 4
    res = [np.zeros(3), src[3]]
    res.append(rest[3])                                  # steal row 4 of the COMPACTED tensor
    rest = np.delete(rest, 3, axis=0)
    res += [rest[0], rest[7]]                            # steal rows {1, 8} in one call
    rest = np.delete(rest, [0, 7], axis=0)
    assert np.array_equal(G["steal_res"], np.array(res)) and np.array_equal(G["steal_rest"], rest)
    assert np.array_equal(G["remove_out"], np.delete(src, [9, 0, 4], axis=0))
    for name in ("braninhoo", "hartmann6", "ackley"):
        x, y = G["bench_%s_x" % name], G["bench_%s_y" % name]
        ref = getattr(oracle, name)(x)
        assert np.max(np.abs(ref - y) / np.maximum(np.abs(y), 1.0)) <= 4e-16


def _draw_scores(oracle, G, kind):
    m, v, fmin = G["bo_means"], G["bo_vars"], float(G["bo_yobs"].min())
    order = G["bo_%s_order" % kind].astype(int)
    S = m.shape[0]
    # eval: one priming draw (result unused, bots/bayesopt.lua:68), then S draws; nominate calls eval again
    assert order.shape == (2 * (S + 1),) and np.array_equal(order[:S + 1], order[S + 1:])
    used = order[1:S + 1] - 1
    if kind == "ei":
        return np.array([oracle.ei_compute(m[s], v[s], fmin, 0.0) for s in used]), used
    return np.array([oracle.cb_compute(m[s], v[s], 2.0, "upper", 1.0) for s in used]), used


@pytest.mark.parametrize("kind", ["ei", "ucb"])
def test_oracle_draw_average_and_argmax_equal_the_executed_bayesopt(oracle, G, kind):
    """bots/bayesopt.lua:56-99 executed with the reference's own score objects: sequential sum from zero in draw order, one
    divide, first maximum (candidates 5 and 18 tie by construction in the EI case)."""
    per_draw, _ = _draw_scores(oracle, G, kind)
    score = oracle.mc_average(per_draw)
    assert np.array_equal(score, G["bo_%s_score" % kind])
    best, idx, nans = oracle.argmax_first(score)
    assert idx == int(G["bo_%s_idx" % kind][0]) and nans == 0
    if kind == "ei":
        assert idx == 5 and score[4] == score[17]


@pytest.mark.skipif(not os.path.isdir(REF), reason="bot7 reference source not found (set BOT7_REFERENCE to a checkout)")
def test_committed_vectors_are_what_the_reference_produces_here():
    """Re-executes a subset of the generator live (one Sobol case; all of math / scores / chol / steal / objectives) and compares it
    with the committed file: the fixture cannot drift from the reference source or from the interpreter."""
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_ref_exec
    os.environ["REF_EXEC_FAST"] = "1"
    try:
        live, _ = make_ref_exec.generate()
    finally:
        del os.environ["REF_EXEC_FAST"]
    committed = np.load(GOLD)
    assert len(live) >= 38
    for k, v in live.items():
        assert np.array_equal(v, committed[k], equal_nan=True), k


# ---------------------------------------------------------------------------------- CUDA path vs executed reference (GPU)

@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SOBOL_CASES))
def test_cuda_sobol_equals_the_executed_reference(ctx, G, name):
    from bot7_b200 import grids
    dims, size, skip, lo, hi = SOBOL_CASES[name]
    cfg = {"size": size, "dims": dims, "skip": skip}
    if lo:
        cfg["mins"] = G["sobol_mins6"]
    if hi:
        cfg["maxes"] = G["sobol_maxes6"]
    assert np.array_equal(grids.sobol(cfg)(), G[name])


@pytest.mark.gpu
def test_cuda_scores_equal_the_executed_reference(ctx, G):
    from bot7_b200 import scores
    m, v, fmin = G["score_mean"], G["score_var"], G["score_fmin"]
    for key, t in (("score_ei_t0", 0.0), ("score_ei_t01", 0.1)):
        ei, ref = scores.expected_improvement.compute(m, v, fmin, t), G[key]
        ok = ~np.isnan(ref)
        assert np.array_equal(np.isnan(ei), np.isnan(ref))
        assert float(np.max(np.abs(ei[ok] - ref[ok]) / np.maximum(np.abs(ref[ok]), 1e-300))) <= 1e-7        # north_star: EI 1e-7 relative
        assert np.array_equal(ei[:4][ok[:4]], ref[:4][ok[:4]])                                                # sigma = 0 rows exactly
    assert np.array_equal(scores.confidence_bound.compute(m, v, {"tradeoff": 1.0, "bound": "lower", "sign": -1.0}), G["score_lcb"])
    assert np.array_equal(scores.confidence_bound.compute(m, v, {"tradeoff": 2.0, "bound": "upper", "sign": 1.0}), G["score_ucb"])
    assert np.array_equal(scores.confidence_bound.compute(m, v, {"tradeoff": 0.5, "bound": "lower", "sign": 1.0}), G["score_lcb_pos"])


@pytest.mark.gpu
def test_cuda_grid_compaction_equals_the_executed_reference(ctx, G):
    from bot7_b200 import grids
    g = grids.DeviceGrid.from_host(G["steal_src"])
    stolen = [g.remove(4)[0], g.remove(4)[0], g.remove(1)[0], g.remove(7)[0]]      # {1, 8} of one call = 1, then 8 - 1 = 7 of what is left
    assert np.array_equal(np.array(stolen), G["steal_res"][1:])
    rest = np.array([g.read(g.original_index(c) - 1, 1)[0] for c in range(1, g.size() + 1)])
    assert np.array_equal(rest, G["steal_rest"])
    g.free()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["ei", "ucb"])
def test_cuda_draw_average_and_argmax_equal_the_executed_bayesopt(ctx, oracle, G, kind):
    """The fused scoring pass (per-draw EI / bound, sequential average, first-max argmax) on the moments the executed
    bots/bayesopt.lua saw, in the draw order it used."""
    import ctypes as C
    from bot7_b200 import _lib as L
    _, used = _draw_scores(oracle, G, kind)
    mean = np.ascontiguousarray(G["bo_means"][used])
    var = np.ascontiguousarray(G["bo_vars"][used])
    S, M = mean.shape
    out = np.empty(M)
    am, best, nn = C.c_int64(), C.c_double(), C.c_int64()
    k, trade, bound, sign = (L.SCORE_EI, 0.0, 0, -1.0) if kind == "ei" else (L.SCORE_CB, 2.0, 1, 1.0)
    L.check(L.lib().b7_score_moments(ctx.handle, k, L.dptr(mean), L.dptr(var), S, M, trade, bound, sign, float(G["bo_yobs"].min()),
                                     L.dptr(out), C.byref(am), C.byref(best), C.byref(nn)), "b7_score_moments")
    ref = G["bo_%s_score" % kind]
    assert am.value == int(G["bo_%s_idx" % kind][0]) and nn.value == 0              # selected index: bit-exact requirement
    if kind == "ucb":
        assert np.array_equal(out, ref)                                              # sqrt / mul / add only
    else:
        assert float(np.max(np.abs(out - ref) / np.maximum(np.abs(ref), 1e-300))) <= 1e-7

"""GPU parity: the CUDA path, called through the C ABI / the host mirror of the reference API,
against the CPU oracle on the same seeded inputs and against the committed golden fixtures.

Bars (BASELINE.json north_star): Sobol points and the selected candidate index bit-exact;
posterior mean / variance 1e-9; EI / UCB 1e-7 relative.  Tolerances are written at each assert.
mean/var "relative" is taken against max(|value|, scale) with scale = 1 for the mean (Y is
standardised) and sigma_f^2 for the variance: both quantities are differences of O(scale) terms,
so their absolute error is what two correct fp64 algorithms can agree on (DESIGN.md, numerics).
"""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

from bot7_b200 import _lib as L
from bot7_b200 import bots, grids, models, parallel, scores

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def rel(a, b, floor):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


# ---------------------------------------------------------------------------------- Sobol

@pytest.mark.parametrize("dims,size,skip", [(2, 20000, 1), (6, 65536, 1), (20, 30000, 1), (39, 5000, 1), (6, 5000, 4090),
                                            (1, 100, 1), (3, 1, 1), (6, 7, 0)])
def test_sobol_bit_exact(ctx, oracle, dims, size, skip):
    out = grids.sobol({"size": size, "dims": dims, "skip": skip})()
    assert out.shape == (size, dims)
    assert np.array_equal(out, oracle.sobol_points(dims, size, skip))


def test_sobol_golden_sha256(ctx):
    out = grids.sobol({"size": 65536, "dims": 6})()
    num = (out * 2.0 ** 30).astype("<u4")
    assert hashlib.sha256(num.tobytes()).hexdigest() == "6ed6741e43f7e1a738ef44a3ed0db34e02aee5adfa796f2ff8f7f8140f4d81a1"
    g = np.load(os.path.join(GOLD, "pinned.npz"))
    assert np.array_equal(num[:4096], g["sobol6"])


def test_sobol_rescale_and_one_sided(ctx, oracle):
    mins, maxes = np.linspace(-1, 0.5, 6), np.linspace(1, 3.3, 6)
    for kw in ({"mins": mins, "maxes": maxes}, {"mins": mins}, {"maxes": maxes}):
        out = grids.sobol(dict(size=3000, dims=6, **kw))()
        assert np.array_equal(out, oracle.sobol_points(6, 3000, 1, kw.get("mins"), kw.get("maxes")))


def test_sobol_large_index_range_property(ctx, oracle):
    # index-range independence: any sub-range equals the same rows of the full sequence (what the
    # multi-GPU sharding relies on); checked deep into the sequence where the oracle is still cheap
    first = (1 << 29) + 12345
    dev = grids.sobol({"size": 1 << 30, "dims": 8}).generate_device(first=first - 1, count=10000)
    got = dev.read()
    assert np.array_equal(got, oracle.sobol_numerators(8, first, 10000) * 2.0 ** -30)
    dev.free()


def test_sobol_limits(ctx):
    with pytest.raises(AssertionError):
        grids.sobol({"size": 10, "dims": 40})                       # grids/sobol.lua:36
    with pytest.raises(L.B7Error, match="too many calls"):
        grids.sobol({"size": 10, "dims": 2, "skip": 1 << 30})()     # grids/sobol.lua:318-324
    assert grids.sobol({"size": 0, "dims": 2})().shape == (0, 2)


# ---------------------------------------------------------------------------------- scoring pass

def test_scoring_golden_and_edge_cases(ctx, oracle):
    g = np.load(os.path.join(GOLD, "pinned.npz"))
    mean, var, fmin = g["mean"], g["var"], float(g["fmin"])
    ei = scores.expected_improvement.compute(mean, var, np.array([fmin]), 0.0)
    ok = ~np.isnan(g["ei"])
    assert np.array_equal(np.isnan(ei), np.isnan(g["ei"]))           # NaN policy: same entries
    assert rel(ei[ok], g["ei"][ok], 1e-300) <= 1e-7                  # north_star: EI 1e-7 relative
    assert np.mean(ei[ok] == g["ei"][ok]) > 0.9                      # in fact mostly bit-equal (exp differs by <= 1 ulp)
    ei_t = scores.expected_improvement.compute(mean, var, np.array([fmin]), 0.1)
    assert rel(ei_t[ok], g["ei_t"][ok], 1e-300) <= 1e-7
    lcb = scores.confidence_bound.compute(mean, var, {"tradeoff": 1.0, "bound": "lower", "sign": -1.0})
    ucb = scores.confidence_bound.compute(mean, var, {"tradeoff": 2.0, "bound": "upper", "sign": 1.0})
    assert np.array_equal(lcb, g["lcb"], equal_nan=True)             # sqrt/mul/add only: bit-exact
    assert np.array_equal(ucb, g["ucb"], equal_nan=True)
    # sigma = 0 rows: ei = max(imprv, 0) exactly
    assert np.array_equal(ei[:5], np.maximum(fmin - mean[:5], 0.0))


def test_scoring_average_order_and_argmax_rule(ctx, oracle):
    r = np.random.default_rng(5)
    S, M = 7, 50001
    mean, var = r.normal(size=(S, M)), r.random((S, M)) ** 2
    lib = L.lib()
    for kind in (L.SCORE_EI, L.SCORE_CB):
        sc = np.empty(M)
        am, best, nn = C.c_int64(), C.c_double(), C.c_int64()
        trade = 0.0 if kind == L.SCORE_EI else 1.0
        L.check(lib.b7_score_moments(ctx.handle, kind, L.dptr(mean), L.dptr(var), S, M, trade, 0, -1.0, -0.2, L.dptr(sc),
                                     C.byref(am), C.byref(best), C.byref(nn)))
        per = [oracle.ei_compute(mean[s], var[s], -0.2, trade) if kind == L.SCORE_EI else oracle.cb_compute(mean[s], var[s], trade)
               for s in range(S)]
        ref = oracle.mc_average(per)
        assert rel(sc, ref, 1e-300) <= 1e-7
        b, i, n = oracle.argmax_first(sc)                            # argmax of the GPU's own scores: exact rule
        assert (am.value, best.value, nn.value) == (i, b, n)
    # ties: EI clamps to exactly 0 for hopeless candidates -> first index must win
    mean = np.full((1, 1000), 50.0)
    var = np.full((1, 1000), 1e-4)
    mean[0, 400] = mean[0, 700] = -1.0
    am = C.c_int64()
    L.check(lib.b7_score_moments(ctx.handle, L.SCORE_EI, L.dptr(mean), L.dptr(var), 1, 1000, 0.0, 0, -1.0, 0.0, None,
                                 C.byref(am), None, None))
    assert am.value == 401
    mean[:] = 50.0
    L.check(lib.b7_score_moments(ctx.handle, L.SCORE_EI, L.dptr(mean), L.dptr(var), 1, 1000, 0.0, 0, -1.0, 0.0, None,
                                 C.byref(am), None, None))
    assert am.value == 1                                             # all zero -> first
    # empty and all-NaN inputs
    nn, best = C.c_int64(), C.c_double()
    L.check(lib.b7_score_moments(ctx.handle, L.SCORE_EI, None, None, 1, 0, 0.0, 0, -1.0, 0.0, None, C.byref(am), C.byref(best), C.byref(nn)))
    assert am.value == 0 and nn.value == 0
    mean[:] = np.nan
    L.check(lib.b7_score_moments(ctx.handle, L.SCORE_EI, L.dptr(mean), L.dptr(var), 1, 1000, 0.0, 0, -1.0, 0.0, None,
                                 C.byref(am), C.byref(best), C.byref(nn)))
    assert am.value == 0 and nn.value == 1000 and np.isnan(best.value)


# ---------------------------------------------------------------------------------- GP fit / predict / acquisition

@pytest.mark.parametrize("name", ["gp_c1", "gp_h6", "gp_m52"])
def test_gp_against_golden_and_oracle(ctx, oracle, name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    X, y, hyp, Xc, kern = g["X"], g["y"], g["hyp"], g["Xc"], int(g["kernel"])
    f = models.GPFactors(X, y, hyp, kern)
    assert (f.info == 0).all() and (f.jitter == 0).all()
    assert rel(f.logml, g["logml"], 1e-300) <= 1e-11
    for s in range(hyp.shape[0]):
        mu, var = f.predict(s, Xc)
        sf2 = np.exp(2 * hyp[s, X.shape[1]])
        assert rel(mu, g["mean"][s], 1.0) <= 1e-9                    # north_star: mean 1e-9
        assert rel(var, g["var"][s], sf2) <= 1e-9                    # north_star: variance 1e-9
        assert rel(var, g["var"][s], 1e-3 * sf2) <= 1e-9             # and strictly relative down to 1e-3 sf2
    grid = grids.DeviceGrid.from_host(Xc)
    for kind, key in ((L.SCORE_EI, "ei"), (L.SCORE_CB, "cb")):
        sc = np.empty(Xc.shape[0])
        am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
        L.check(L.lib().b7_acq_score(f.handle, grid.handle, kind, 0.0 if kind == L.SCORE_EI else 1.0, 0, -1.0, float(y.min()),
                                     L.dptr(sc), C.byref(am), C.byref(amo), C.byref(best), C.byref(nn)))
        assert rel(sc, g[key], 1e-6 * np.max(np.abs(g[key]))) <= 1e-7   # north_star: EI/UCB 1e-7
        assert am.value == int(g[key + "_idx"]) == amo.value         # selected candidate: bit-exact index
        assert nn.value == 0
    f.free()


def make_problem(oracle, N, d, S, M, noise, seed=3):
    r = np.random.default_rng(seed)
    X = oracle.sobol_points(d, N + M)
    perm = r.permutation(N + M)
    Xo, Xc = X[np.sort(perm[:N])], X[np.sort(perm[N:])]
    y = {2: oracle.braninhoo, 6: oracle.hartmann6}.get(d, oracle.ackley)(Xo)
    y = (y - y.mean()) / y.std()
    hyp = np.zeros((S, d + 3))
    hyp[:, :d] = np.log(0.1) + r.random((S, d)) * (np.log(2) - np.log(0.1))
    hyp[:, d] = 0.5 * (r.random(S) - 0.5)
    hyp[:, d + 1] = 0.5 * np.log(noise)
    hyp[:, d + 2] = 0.1 * (r.random(S) - 0.5)
    return Xo, y, hyp, Xc


@pytest.mark.parametrize("N,d,S,M,noise", [(127, 6, 2, 1000, 1e-2), (128, 6, 1, 129, 1e-2), (129, 3, 2, 300, 1e-2),
                                           (640, 6, 3, 20000, 1e-2), (1100, 20, 2, 4000, 1e-2), (1, 2, 1, 10, 1e-2)])
def test_gp_ragged_sizes_vs_oracle(ctx, oracle, N, d, S, M, noise):
    # block-boundary sizes (127/128/129), several blocks, several candidate panels, N = 1
    Xo, y, hyp, Xc = make_problem(oracle, N, d, S, M, noise)
    if N == 1:
        y = np.array([0.3])
    f = models.GPFactors(Xo, y, hyp, "ardse")
    ref = oracle.acquisition(Xo, y, hyp, Xc, 0, False, oracle.SCORE_EI)
    for s in range(S):
        mu, var = f.predict(s, Xc)
        sf2 = np.exp(2 * hyp[s, d])
        assert rel(mu, ref["mean"][s], 1.0) <= 1e-9
        assert rel(var, ref["var"][s], sf2) <= 1e-9
    grid = grids.DeviceGrid.from_host(Xc)
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
    sc = np.empty(M)
    L.check(L.lib().b7_acq_score(f.handle, grid.handle, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), L.dptr(sc), C.byref(am),
                                 C.byref(amo), C.byref(best), C.byref(nn)))
    assert rel(sc, ref["score"], 1e-6 * max(np.max(ref["score"]), 1e-300)) <= 1e-7
    # index: equal, or a genuine near-tie (|score gap| within 1e-7 relative) -- reported separately
    if am.value != ref["idx"]:
        gap = abs(ref["score"][am.value - 1] - ref["best"]) / abs(ref["best"])
        assert gap <= 1e-12, f"argmax differs beyond a near-tie: {am.value} vs {ref['idx']} (gap {gap})"
    f.free()


@pytest.mark.parametrize("kern,bound,sign,tradeoff", [(1, "upper", 1.0, 2.0), (0, "upper", -1.0, 0.5), (1, "lower", 1.0, 1.0)])
def test_confidence_bound_variants_and_matern_at_size(ctx, oracle, kern, bound, sign, tradeoff):
    # config 2 of BASELINE.json in miniature (UCB, single MAP draw), both kernels, every bound/sign branch
    Xo, y, hyp, Xc = make_problem(oracle, 640, 6, 1, 9000, 1e-2, seed=kern + 5)
    f = models.GPFactors(Xo, y, hyp, kern)
    grid = grids.DeviceGrid.from_host(Xc)
    sc = np.empty(Xc.shape[0])
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
    L.check(L.lib().b7_acq_score(f.handle, grid.handle, L.SCORE_CB, tradeoff, L.BOUND_UPPER if bound == "upper" else L.BOUND_LOWER,
                                 sign, float(y.min()), L.dptr(sc), C.byref(am), C.byref(amo), C.byref(best), C.byref(nn)))
    ref = oracle.acquisition(Xo, y, hyp, Xc, kern, False, oracle.SCORE_CB, tradeoff, bound, sign)
    assert rel(sc, ref["score"], 1e-6 * np.max(np.abs(ref["score"]))) <= 1e-7
    assert am.value == ref["idx"] and best.value == sc[am.value - 1]
    f.free()


def test_empty_and_tiny_grids(ctx, oracle):
    Xo, y, hyp, Xc = make_problem(oracle, 64, 3, 2, 5, 1e-2)
    f = models.GPFactors(Xo, y, hyp)
    am, amo, best, nn = C.c_int64(7), C.c_int64(7), C.c_double(), C.c_int64(7)
    g0 = grids.DeviceGrid.from_host(np.zeros((0, 3)))
    L.check(L.lib().b7_acq_score(f.handle, g0.handle, L.SCORE_EI, 0.0, 0, -1.0, 0.0, None, C.byref(am), C.byref(amo), C.byref(best), C.byref(nn)))
    assert (am.value, amo.value, nn.value) == (0, 0, 0) and np.isnan(best.value)
    g1 = grids.DeviceGrid.from_host(Xc)
    for i in range(4):
        g1.remove(1)                                                # only the last original row stays live
    L.check(L.lib().b7_acq_score(f.handle, g1.handle, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), None, C.byref(am), C.byref(amo),
                                 C.byref(best), C.byref(nn)))
    assert (am.value, amo.value) == (1, 5)
    g2 = grids.DeviceGrid.from_host(np.zeros((3, 4)))
    with pytest.raises(L.B7Error, match="grid dims"):
        L.check(L.lib().b7_acq_score(f.handle, g2.handle, L.SCORE_EI, 0.0, 0, -1.0, 0.0, None, C.byref(am), C.byref(amo),
                                     C.byref(best), C.byref(nn)))
    f.free()


def test_gp_noiseless_illconditioned_reports_scaled_error(ctx, oracle):
    # sigma_n^2 = 1e-6: cond(K) ~ 1e8; two correct fp64 algorithms differ by cond*eps.  Bar: absolute
    # error scaled by the prior variance (what the subtraction sf2 - sum v^2 can resolve).
    Xo, y, hyp, Xc = make_problem(oracle, 700, 6, 2, 3000, 1e-6)
    f = models.GPFactors(Xo, y, hyp, "ardse", noiseless=True)
    for s in range(2):
        fit = oracle.gp_fit(Xo, y, hyp[s], 0, True)
        mr, vr = oracle.gp_predict(fit, Xc)
        mu, var = f.predict(s, Xc)
        assert np.max(np.abs(var - vr)) / fit["sf2"] <= 1e-9
        assert np.max(np.abs(mu - mr)) <= 1e-6
    f.free()


def test_jitter_retry_policy_matches_reference_policy(ctx, oracle, capsys):
    # duplicated observations + negligible noise: the plain factorisation fails; the retry adds
    # eps = 1e-8 * 1.1^k exactly like utils.math.chol (utils/math.lua:168-216)
    r = np.random.default_rng(0)
    X = r.random((200, 3))
    X[100:] = X[:100]
    y = r.normal(size=200)
    hyp = np.array([[np.log(0.5)] * 3 + [0.0, 0.5 * np.log(1e-18), 0.0]])
    f = models.GPFactors(X, y, hyp, "ardse", flags=L.FIT_LOGML_ONLY)
    fr = oracle.gp_fit(X, y, hyp[0], 0)
    assert f.info[0] == 0 and fr["iters"] >= 1
    assert f.jitter[0] == fr["jitter"]                               # same eps sequence
    assert "jitter of" in capsys.readouterr().out                    # warning printed, as in the reference
    f.free()


def test_both_posterior_paths_agree_with_the_oracle(ctx, oracle):
    # FP64 DMMA tiles vs error-free int8 slices on tcgen05 (28 exact products recombined in fp64): same handle,
    # path switched on the fly; both against the oracle and against each other
    Xo, y, hyp, Xc = make_problem(oracle, 900, 6, 3, 12000, 1e-2)
    f = models.GPFactors(Xo, y, hyp)
    grid = grids.DeviceGrid.from_host(Xc)
    ref = oracle.acquisition(Xo, y, hyp, Xc, 0, False, oracle.SCORE_EI)
    keep = ctx.posterior_path()
    out = {}
    try:
        for path in (L.PATH_FP64_DMMA, L.PATH_INT8_OZAKI, L.PATH_FP64_DMMA):
            ctx.set_posterior_path(path)
            assert ctx.posterior_path() == path
            mv = [f.predict(s, Xc) for s in range(3)]
            sc = np.empty(Xc.shape[0])
            am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
            L.check(L.lib().b7_acq_score(f.handle, grid.handle, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), L.dptr(sc), C.byref(am),
                                         C.byref(amo), C.byref(best), C.byref(nn)))
            for s in range(3):
                sf2 = np.exp(2 * hyp[s, 6])
                assert rel(mv[s][0], ref["mean"][s], 1.0) <= 1e-9 and rel(mv[s][1], ref["var"][s], sf2) <= 1e-9
            assert am.value == ref["idx"] and rel(sc, ref["score"], 1e-6 * ref["score"].max()) <= 1e-7
            out[path] = (mv, sc)
    finally:
        ctx.set_posterior_path(keep)
    a, b = out[L.PATH_FP64_DMMA], out[L.PATH_INT8_OZAKI]
    for s in range(3):
        assert np.max(np.abs(a[0][s][1] - b[0][s][1])) <= 1e-12 * np.exp(2 * hyp[s, 6])      # variance: 1e-12 sf2
        assert np.max(np.abs(a[0][s][0] - b[0][s][0])) <= 1e-10
    f.free()


def test_nonfinite_candidate_poisons_only_its_own_row(ctx, oracle):
    # integers cannot carry a NaN through the int8 slices: the kernel re-derives which K* rows the fp64 path would
    # see as NaN (NaN coordinate; infinite coordinate under Matern, inf * 0).  ARD-SE with an infinite coordinate
    # is a clean k* = 0: prior mean and prior variance.
    Xo, y, hyp, Xc = make_problem(oracle, 300, 6, 2, 1000, 1e-2)
    bad = Xc.copy()
    bad[5, 2] = np.nan
    bad[70, 0] = np.inf
    bad[999, 5] = -np.inf
    keep = ctx.posterior_path()
    try:
        for kern, nan_rows, prior_rows in (("ardse", [5], [70, 999]), ("matern52", [5, 70, 999], [])):
            f = models.GPFactors(Xo, y, hyp, kern)
            for path in (L.PATH_FP64_DMMA, L.PATH_INT8_OZAKI):
                ctx.set_posterior_path(path)
                m0, v0 = f.predict(1, Xc)
                m1, v1 = f.predict(1, bad)
                assert np.isnan(m1[nan_rows]).all() and np.isnan(v1[nan_rows]).all()
                for r_ in prior_rows:
                    assert m1[r_] == hyp[1, 8] and abs(v1[r_] / np.exp(2 * hyp[1, 6]) - 1) <= 1e-15
                ok = np.ones(1000, bool)
                ok[[5, 70, 999]] = False
                assert np.array_equal(m0[ok], m1[ok]) and np.array_equal(v0[ok], v1[ok])
                grid = grids.DeviceGrid.from_host(bad)
                am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
                L.check(L.lib().b7_acq_score(f.handle, grid.handle, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), None, C.byref(am),
                                             C.byref(amo), C.byref(best), C.byref(nn)))
                assert nn.value == len(nan_rows) and am.value - 1 not in nan_rows
            f.free()
    finally:
        ctx.set_posterior_path(keep)


def test_int8_trailing_update_of_the_cholesky_matches_the_fp64_one(ctx, oracle):
    # potrf_i8.cu: with the INT8 path selected, batched fits (S >= 4 draws and S * NB^2 >= 4096) run the k = 512
    # trailing updates as exact int8 slice products; the factor must agree with the all-FP64 factorisation to
    # rounding level, and both with the oracle.  18 row blocks x 13 draws = 4212.
    Xo, y, hyp, _ = make_problem(oracle, 2304, 6, 13, 10, 1e-3)
    keep = ctx.posterior_path()
    out = {}
    try:
        for path in (L.PATH_FP64_DMMA, L.PATH_INT8_OZAKI):
            ctx.set_posterior_path(path)
            f = models.GPFactors(Xo, y, hyp, flags=L.FIT_LOGML_ONLY)
            assert (np.asarray(f.info) == 0).all()
            out[path] = (np.array(f.logml), [f.read_factor(s) for s in (0, 12)])
            f.free()
    finally:
        ctx.set_posterior_path(keep)
    a, b = out[L.PATH_FP64_DMMA], out[L.PATH_INT8_OZAKI]
    assert rel(a[0], b[0], 1e-300) <= 1e-12
    for La, Lb, s in zip(a[1], b[1], (0, 12)):
        assert np.max(np.abs(La - Lb)) <= 1e-12 * np.max(np.abs(La))
        assert not np.array_equal(La, Lb)                                # the two arithmetic paths really differ
        ref = oracle.gp_fit(Xo, y, hyp[s], 0)
        assert np.max(np.abs(Lb - np.tril(ref["L"]))) <= 1e-10 * np.max(np.abs(ref["L"]))
        assert rel(b[0][s:s + 1], np.array([ref["logml"]]), 1e-300) <= 1e-11


@pytest.mark.parametrize("N,S", [(300, 2), (600, 2), (1700, 1), (2304, 4)])
def test_block_recursive_int8_inverse_matches_the_fp64_sweep(ctx, oracle, N, S):
    # trtri_i8.cu: X21 = -X22 (L21 X11) per level with exact int8 slice products; 3, 5, 14 and 18 row blocks leave the
    # last pair of a level short or empty at different levels.  Against the FP64 column sweep and against numpy.
    Xo, y, hyp, _ = make_problem(oracle, N, 6, S, 10, 1e-3)
    keep = ctx.posterior_path()
    out = {}
    try:
        for path in (L.PATH_FP64_DMMA, L.PATH_INT8_OZAKI):
            ctx.set_posterior_path(path)
            f = models.GPFactors(Xo, y, hyp)
            assert (np.asarray(f.info) == 0).all()
            out[path] = [f.read_factor(s) for s in range(S)]
            f.free()
    finally:
        ctx.set_posterior_path(keep)
    for s in range(S):
        a, b = out[L.PATH_FP64_DMMA][s], out[L.PATH_INT8_OZAKI][s]
        scale = np.max(np.abs(a))
        assert np.max(np.abs(a - b)) <= 1e-11 * scale
        assert N <= 128 or not np.array_equal(a, b)
        ref = np.linalg.inv(np.tril(oracle.gp_fit(Xo, y, hyp[s], 0)["L"]))
        assert np.max(np.abs(b - np.tril(ref))) <= 1e-9 * scale


def test_more_than_16384_observations_stay_on_the_fp64_kernels(ctx, oracle):
    # the int8 slice sums are exact in int32 up to Np = 16384 (7 products x 2^14 x Np < 2^31); beyond that the fit,
    # the inversion and the posterior must run on the FP64 DMMA kernels even with the INT8 path selected.
    # Size-independent checks: interpolation of the observations to noise level, 0 <= var <= prior, finite logml.
    N, d = 16500, 2
    r = np.random.default_rng(2)
    X = oracle.sobol_points(d, N)
    y = oracle.braninhoo(X)
    y = (y - y.mean()) / y.std()
    hyp = np.array([[np.log(0.3), np.log(0.3), 0.0, 0.5 * np.log(1e-2), 0.0]])
    assert ctx.posterior_path() == L.PATH_INT8_OZAKI
    f = models.GPFactors(X, y, hyp)
    assert f.info[0] == 0 and np.isfinite(f.logml[0]) and f.padded_n() == 16512
    idx = r.choice(N, 300, replace=False)
    mean, var = f.predict(0, X[idx])
    assert np.all(np.isfinite(mean)) and np.all(var >= 0.0) and np.all(var <= 1.0 + 1e-12)
    assert np.max(np.abs(mean - y[idx])) <= 0.5 and np.max(var) <= 1e-2          # dense data: posterior hugs the observations
    far = np.full((1, d), 50.0)
    m_far, v_far = f.predict(0, far)
    assert abs(m_far[0] - hyp[0, 4]) <= 1e-12 and abs(v_far[0] - 1.0) <= 1e-12      # no correlation left: the prior
    f.free()


def refined_alpha(oracle, fit, y):
    """alpha = K_y^-1 (y - m) with two steps of iterative refinement whose residual is formed in extended precision
    (numpy longdouble, 64-bit mantissa) from the fp64 entries of K_y: an estimate of the exact solution of the
    system the fp64 algorithms solve, good to ~cond * 2^-64.  Test infrastructure (used to measure the oracle's own
    error where cond(K) * eps exceeds the 1e-9 bar)."""
    import scipy.linalg as sla
    X, L_ = fit["X"], fit["L"]
    K = oracle.cov(fit["kernel"], X, X, fit["w"], fit["sf2"])
    K[np.diag_indices(K.shape[0])] += fit["sn2"] + fit["jitter"]
    r = (y - fit["m"]).astype(np.longdouble)
    alpha = fit["alpha"].astype(np.longdouble)
    for _ in range(2):
        res = r.copy()
        for c0 in range(0, K.shape[0], 2048):                      # K in longdouble, 2048 rows at a time
            res[c0:c0 + 2048] -= K[c0:c0 + 2048].astype(np.longdouble) @ alpha
        dz = sla.solve_triangular(L_.T, sla.solve_triangular(L_, res.astype(np.float64), lower=True), lower=False)
        alpha = alpha + dz.astype(np.longdouble)
    return alpha


def test_int8_path_at_its_largest_size_matches_the_fp64_path(ctx, oracle):
    # N = 16384: the longest int32 accumulations the INT8 kernels are allowed to run (posterior k = 16384, inversion
    # k = 8192); inverse and posterior of both paths against the oracle on 2048 candidates.
    # Bars: variance 1e-9 sf2 (north_star).  Mean: cond(K) ~ N sf2 / sn2 = 2e6 and |alpha| ~ 1e2, so two correct fp64
    # algorithms differ by ~cond * eps * |alpha| ~ 1e-8 -- the 1e-9 bar is below what fp64 can resolve for this system.
    # The test therefore measures the oracle's own error against an extended-precision refinement of alpha and holds
    # the GPU paths to the same reference: GPU error <= max(1e-9, 3 x the LAPACK oracle's error).
    N, d, M = 16384, 3, 2048
    r = np.random.default_rng(3)
    X = oracle.sobol_points(d, N)
    y = oracle.ackley(X)
    y = (y - y.mean()) / y.std()
    hyp = np.array([[np.log(0.2), np.log(0.3), np.log(0.25), 0.1, 0.5 * np.log(1e-2), 0.05]])
    Xc = r.random((M, d))
    keep = ctx.posterior_path()
    out = {}
    try:
        for path in (L.PATH_FP64_DMMA, L.PATH_INT8_OZAKI):
            ctx.set_posterior_path(path)
            f = models.GPFactors(X, y, hyp)
            assert f.info[0] == 0
            out[path] = (f.logml[0],) + f.predict(0, Xc)
            f.free()
    finally:
        ctx.set_posterior_path(keep)
    a, b = out[L.PATH_FP64_DMMA], out[L.PATH_INT8_OZAKI]
    sf2 = np.exp(2 * hyp[0, 3])
    assert a[0] == b[0]                                               # single factor: the same FP64 factorisation
    dm, dv = np.max(np.abs(a[1] - b[1])), np.max(np.abs(a[2] - b[2])) / sf2
    assert dm <= 5e-8 and dv <= 1e-9
    assert np.all(b[2] >= 0) and np.all(b[2] <= sf2 * (1 + 1e-12))
    ref = oracle.gp_fit(X, y, hyp[0], 0)
    m_ref, v_ref = oracle.gp_predict(ref, Xc)
    alpha_x = refined_alpha(oracle, ref, y)
    Ks = oracle.cov(0, Xc, X, ref["w"], ref["sf2"])
    m_x = (ref["m"] + Ks.astype(np.longdouble) @ alpha_x).astype(np.float64)
    oracle_err = float(np.max(np.abs(m_ref - m_x)))
    report = {"N": N, "candidates": M, "cond_estimate": N * sf2 / 1e-2, "oracle_mean_vs_extended_precision": oracle_err,
              "paths_mean_diff": float(dm), "paths_var_diff_over_sf2": float(dv)}
    for name, mv in (("fp64_dmma", a), ("int8_ozaki", b)):
        e = posterior_errors(mv[1], mv[2], m_ref, v_ref, sf2)
        e["mean_vs_extended_precision"] = float(np.max(np.abs(mv[1] - m_x)))
        report[name] = e
    record_parity("largest_int8_N16384", report)
    print("N = 16384:", report)
    for name in ("fp64_dmma", "int8_ozaki"):
        e = report[name]
        assert e["var_over_sf2"] <= 1e-9, report                                          # north_star bar
        assert e["mean_vs_extended_precision"] <= max(1e-9, 3 * oracle_err), report       # see the comment above
        assert e["mean"] <= max(1e-9, 4 * oracle_err), report


@pytest.mark.parametrize("N", [300, 1100, 2304])
def test_one_factor_latency_path_gives_the_bits_of_the_batched_fit(ctx, oracle, N):
    # potrf.cu: one or two factors per call run the row-sliced panel / trailing kernels (4 CTAs per tile); three use the
    # tile kernels.  Same DMMA sequence per element, same reduction order for beta: factor, log marginal likelihood and
    # beta-dependent results must be bit-identical.  FP64 path on both sides (three draws never take the INT8 updates).
    Xo, y, hyp, _ = make_problem(oracle, N, 6, 3, 10, 1e-3)
    keep = ctx.posterior_path()
    try:
        ctx.set_posterior_path(L.PATH_FP64_DMMA)
        three = models.GPFactors(Xo, y, hyp, flags=L.FIT_LOGML_ONLY)
        one = models.GPFactors(Xo, y, hyp[1:2], flags=L.FIT_LOGML_ONLY)
        assert (np.asarray(three.info) == 0).all() and (np.asarray(one.info) == 0).all()
        assert np.array_equal(one.logml, three.logml[1:2])
        assert np.array_equal(one.read_factor(0), three.read_factor(1))
        ref = oracle.gp_fit(Xo, y, hyp[1], 0)
        assert np.max(np.abs(one.read_factor(0) - np.tril(ref["L"]))) <= 1e-10 * np.max(np.abs(ref["L"]))
        assert rel(np.asarray(one.logml), np.array([ref["logml"]]), 1e-300) <= 1e-11
        one.free()
        three.free()
    finally:
        ctx.set_posterior_path(keep)


def test_fit_is_deterministic_and_predict_needs_inverse(ctx, oracle):
    Xo, y, hyp, Xc = make_problem(oracle, 300, 6, 3, 2000, 1e-2)
    a = models.GPFactors(Xo, y, hyp)
    b = models.GPFactors(Xo, y, hyp)
    assert np.array_equal(a.logml, b.logml)
    assert all(np.array_equal(x, z) for x, z in zip(a.predict(1, Xc), b.predict(1, Xc)))   # run-to-run bit-exact
    c = models.GPFactors(Xo, y, hyp, flags=L.FIT_LOGML_ONLY)
    assert np.array_equal(c.logml, a.logml)
    with pytest.raises(L.B7Error, match="not inverted"):
        c.predict(0, Xc)
    for f in (a, b, c):
        f.free()


def test_refit_reuses_handle(ctx, oracle):
    # slice-sampler density path: same observations, new draws, no reallocation
    Xo, y, hyp, Xc = make_problem(oracle, 300, 6, 2, 1500, 1e-2)
    f = models.GPFactors(Xo, y, hyp, flags=L.FIT_LOGML_ONLY)
    hyp2 = hyp + 0.1
    f.refit(hyp2, L.FIT_LOGML_ONLY)
    ref = [oracle.gp_fit(Xo, y, h, 0)["logml"] for h in hyp2]
    assert rel(f.logml, np.array(ref), 1e-300) <= 1e-11
    f.refit(hyp, L.FIT_PREDICT)
    g = models.GPFactors(Xo, y, hyp)
    assert np.array_equal(f.logml, g.logml)
    assert all(np.array_equal(a, b) for a, b in zip(f.predict(1, Xc), g.predict(1, Xc)))
    f.free()
    g.free()


def test_second_device_in_the_same_process(ctx, oracle):
    # the Lua host is one process that may drive several GPUs: contexts are per device
    if L.lib().b7_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx1 = L.Context(1)
    Xo, y, hyp, Xc = make_problem(oracle, 300, 6, 2, 3000, 1e-2)
    f0 = models.GPFactors(Xo, y, hyp, ctx=ctx)
    f1 = models.GPFactors(Xo, y, hyp, ctx=ctx1)
    assert np.array_equal(f0.logml, f1.logml)
    assert all(np.array_equal(a, b) for a, b in zip(f0.predict(1, Xc), f1.predict(1, Xc)))
    out = np.empty((1000, 5))
    L.check(L.lib().b7_sobol_generate(ctx1.handle, 5, 1, 1000, None, None, L.dptr(out), None))
    assert np.array_equal(out, oracle.sobol_points(5, 1000))
    f0.free()
    f1.free()
    ctx1.close()


def test_argument_errors(ctx):
    X, y = np.zeros((4, 2)), np.zeros(4)
    with pytest.raises(L.B7Error, match="H must be d\\+3"):
        models.GPFactors(X, y, np.zeros((1, 4)))
    with pytest.raises(ValueError):
        models.GPFactors(X, np.zeros(3), np.zeros((1, 5)))


# ---------------------------------------------------------------------------------- properties at scale

def test_posterior_properties_large(ctx, oracle):
    # size-independent properties on a shape the oracle would not finish quickly:
    # N = 2048, S = 4, 40k candidates (three posterior panels)
    N, d, S, M = 2048, 6, 4, 40000
    X = oracle.sobol_points(d, N + M)
    Xo, Xc = X[:N], X[N:]
    y = oracle.hartmann6(Xo)
    y = (y - y.mean()) / y.std()
    r = np.random.default_rng(9)
    hyp = np.zeros((S, d + 3))
    hyp[:, :d] = np.log(0.2) + r.random((S, d)) * np.log(5)
    hyp[:, d + 1] = 0.5 * np.log(1e-2)
    f = models.GPFactors(Xo, y, hyp)
    assert (f.info == 0).all()
    for s in range(S):
        sf2 = np.exp(2 * hyp[s, d])
        mu, var = f.predict(s, Xc)
        assert (var >= 0).all() and (var <= sf2 * (1 + 1e-12)).all()     # 0 <= latent variance <= prior
        mo, vo = f.predict(s, Xo[:512])
        # at observed points the latent variance is below the noise level sigma_n^2
        assert (vo <= 1e-2 * 1.0001).all()
    # linearity of the mean in y: mean(y1 + y2) - m = (mean(y1)-m) + (mean(y2)-m)
    h0 = hyp[:1].copy()
    h0[0, d + 2] = 0.0
    y2 = np.cos(5 * Xo.sum(1))
    m1 = models.GPFactors(Xo, y, h0).predict(0, Xc[:5000])[0]
    m2 = models.GPFactors(Xo, y2, h0).predict(0, Xc[:5000])[0]
    m12 = models.GPFactors(Xo, y + y2, h0).predict(0, Xc[:5000])[0]
    assert np.max(np.abs(m12 - (m1 + m2))) <= 1e-9
    # spot-check a slice against the oracle at this size
    fit = oracle.gp_fit(Xo, y, hyp[0], 0)
    mr, vr = oracle.gp_predict(fit, Xc[:2000])
    mu, var = f.predict(0, Xc[:2000])
    assert rel(mu, mr, 1.0) <= 1e-9 and rel(var, vr, fit["sf2"]) <= 1e-9
    f.free()


def record_parity(key, values):
    """Measured maxima of the headline-size parity tests -> $BOT7_PARITY_DIR/parity_r02.json (the source of
    profiles/parity_r02.json).  Without BOT7_PARITY_DIR nothing is written: the suite leaves the checkout as it found it."""
    import json
    out = os.environ.get("BOT7_PARITY_DIR")
    if not out:
        return
    os.makedirs(out, exist_ok=True)
    path = os.path.join(out, "parity_r02.json")
    try:
        data = json.load(open(path))
    except Exception:
        data = {}
    data[key] = values
    json.dump(data, open(path, "w"), indent=1, sort_keys=True)


def posterior_errors(mu, var, mu_ref, var_ref, sf2):
    """The four figures every size-parity test reports: mean (against max(|mean|, 1)), variance against the prior
    variance, variance strictly relative where var >= 1e-3 sf2, and the smallest variance seen."""
    big = var_ref >= 1e-3 * sf2
    return {"mean": rel(mu, mu_ref, 1.0), "var_over_sf2": float(np.max(np.abs(var - var_ref)) / sf2),
            "var_rel_where_ge_1e-3_sf2": float(np.max(np.abs(var - var_ref)[big] / var_ref[big])) if big.any() else 0.0,
            "frac_var_ge_1e-3_sf2": float(np.mean(big)), "min_var_over_sf2": float(var_ref.min() / sf2)}


def test_headline_config_both_paths_against_the_oracle(ctx, oracle):
    """The shape BASELINE.json's metric is quoted on and bench.py times -- N = 4096, d = 6, sigma_n^2 = 1e-2, bench.py's own
    hyper_draws() and Sobol grid -- against oracle.acquisition, on both posterior paths.  4 of the 32 draws (the rows with
    the shortest and the longest length-scales and two more), 2 posterior panels = 37 888 candidates.
    Call sites matched: scores/expected_improvement.lua:63-66 (predict + fmin), bots/bayesopt.lua:73-79,96 (average, argmax).
    Bars (north_star): mean 1e-9, variance 1e-9 sf2 and 1e-9 relative where var >= 1e-3 sf2, EI 1e-7, argmax identical."""
    import bench
    N, d, M = bench.N_OBS, bench.DIMS, bench.M_STEP
    pts = grids.sobol({"size": N + M, "dims": d})()
    assert np.array_equal(pts, oracle.sobol_points(d, N + M))
    Xo, Xc = pts[:N], pts[N:]
    y = bench.hartmann6(Xo)
    assert np.allclose(y, oracle.hartmann6(Xo), rtol=1e-14, atol=0)
    y = (y - y.mean()) / y.std()
    hyp32 = bench.hyper_draws(bench.S_DRAWS, d)
    ls = hyp32[:, :d].sum(1)
    rows = [int(np.argmin(ls)), int(np.argmax(ls))]
    rows = sorted(rows + [s for s in range(bench.S_DRAWS) if s not in rows][:2])
    assert len(set(rows)) == 4
    hyp = hyp32[rows]
    ref = oracle.acquisition(Xo, y, hyp, Xc, 0, False, oracle.SCORE_EI)
    keep = ctx.posterior_path()
    report = {"N": N, "d": d, "candidates": M, "draw_rows": rows, "sigma_n2": 1e-2}
    try:
        for path, name in ((L.PATH_INT8_OZAKI, "int8_ozaki"), (L.PATH_FP64_DMMA, "fp64_dmma")):
            ctx.set_posterior_path(path)
            f = models.GPFactors(Xo, y, hyp)
            assert (f.info == 0).all() and (f.jitter == 0).all()
            worst = {}
            for s in range(len(rows)):
                sf2 = np.exp(2 * hyp[s, d])
                mu, var = f.predict(s, Xc)
                e = posterior_errors(mu, var, ref["mean"][s], ref["var"][s], sf2)
                worst = {k: (max(worst.get(k, 0.0), v) if k != "min_var_over_sf2" else min(worst.get(k, 1.0), v)) for k, v in e.items()}
            grid = grids.DeviceGrid.from_host(Xc)
            sc = np.empty(M)
            am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
            L.check(L.lib().b7_acq_score(f.handle, grid.handle, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), L.dptr(sc), C.byref(am),
                                         C.byref(amo), C.byref(best), C.byref(nn)))
            worst["ei_rel"] = rel(sc, ref["score"], 1e-6 * ref["score"].max())
            worst["logml_rel"] = rel(f.logml, np.array([oracle.gp_fit(Xo, y, h, 0)["logml"] for h in hyp]), 1e-300)
            worst["argmax"] = int(am.value)
            worst["argmax_oracle"] = int(ref["idx"])
            report[name] = worst
            record_parity("headline_N4096", report)
            assert worst["mean"] <= 1e-9, worst                           # north_star: mean 1e-9
            assert worst["var_over_sf2"] <= 1e-9, worst                   # variance 1e-9 of the prior variance
            assert worst["var_rel_where_ge_1e-3_sf2"] <= 1e-9, worst      # and 1e-9 strictly relative down to 1e-3 sf2
            assert worst["ei_rel"] <= 1e-7, worst                         # EI 1e-7
            assert am.value == ref["idx"] == amo.value and nn.value == 0  # selected candidate: identical
            assert worst["logml_rel"] <= 1e-11
            grid.free()
            f.free()
    finally:
        ctx.set_posterior_path(keep)


def test_headline_noiseless_variant_reports_scaled_error(ctx, oracle):
    """Noiseless variant (diag = 1e-6 + 1e-8 sf2, cond(K) ~ 1e9) at N = 2048 with bench.py's draws: two correct fp64
    algorithms differ by cond * eps here (LAPACK against an extended-precision solve differs by ~3e-9 relative, DESIGN.md
    section 2), so the bar is the scaled one: variance 1e-9 of the prior variance, mean 1e-6 absolute; argmax identical
    or a tie within 1e-9 relative."""
    import bench
    N, d, M = 2048, 6, 18944
    pts = grids.sobol({"size": N + M, "dims": d})()
    Xo, Xc = pts[:N], pts[N:]
    y = bench.hartmann6(Xo)
    y = (y - y.mean()) / y.std()
    hyp = bench.hyper_draws(bench.S_DRAWS, d)[[3, 11]]
    hyp[:, d + 1] = 0.5 * np.log(1e-6)
    ref = oracle.acquisition(Xo, y, hyp, Xc, 0, True, oracle.SCORE_EI)
    keep = ctx.posterior_path()
    report = {"N": N, "candidates": M, "sigma_n2": 1e-6, "noiseless": True}
    try:
        for path, name in ((L.PATH_INT8_OZAKI, "int8_ozaki"), (L.PATH_FP64_DMMA, "fp64_dmma")):
            ctx.set_posterior_path(path)
            f = models.GPFactors(Xo, y, hyp, "ardse", noiseless=True)
            assert (f.info == 0).all()
            worst = {}
            for s in range(2):
                mu, var = f.predict(s, Xc)
                e = posterior_errors(mu, var, ref["mean"][s], ref["var"][s], np.exp(2 * hyp[s, d]))
                worst = {k: (max(worst.get(k, 0.0), v) if k != "min_var_over_sf2" else min(worst.get(k, 1.0), v)) for k, v in e.items()}
            grid = grids.DeviceGrid.from_host(Xc)
            sc = np.empty(M)
            am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
            L.check(L.lib().b7_acq_score(f.handle, grid.handle, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), L.dptr(sc), C.byref(am),
                                         C.byref(amo), C.byref(best), C.byref(nn)))
            worst["ei_abs_over_max"] = float(np.max(np.abs(sc - ref["score"])) / ref["score"].max())
            worst["argmax"], worst["argmax_oracle"] = int(am.value), int(ref["idx"])
            report[name] = worst
            record_parity("noiseless_N2048", report)
            assert worst["var_over_sf2"] <= 1e-9 and worst["mean"] <= 1e-6, worst
            if am.value != ref["idx"]:
                gap = abs(ref["score"][am.value - 1] - ref["best"]) / abs(ref["best"])
                assert gap <= 1e-9, f"argmax differs beyond a near-tie: {am.value} vs {ref['idx']} (gap {gap})"
            grid.free()
            f.free()
    finally:
        ctx.set_posterior_path(keep)


def test_sharded_acquisition_equals_single(ctx, oracle):
    # (e) multi-GPU: G candidate shards scored independently + the deterministic combine give the
    # same index/score as one pass, for G = 1, 2, 4, 8 (the ranks are emulated on one GPU here;
    # tests/test_host_logic.py covers the 2-rank gloo exchange)
    Xo, y, hyp, Xc = make_problem(oracle, 256, 6, 4, 30011, 1e-2)
    f = models.GPFactors(Xo, y, hyp)
    grid = grids.DeviceGrid.from_host(Xc)
    grid.remove(17)
    grid.remove(20000)
    lib = L.lib()
    full = np.empty(Xc.shape[0])
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
    L.check(lib.b7_acq_score(f.handle, grid.handle, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), L.dptr(full), C.byref(am),
                             C.byref(amo), C.byref(best), C.byref(nn)))
    assert np.isnan(full[16]) and np.isnan(full[20000])              # removed rows (20000 compacted -> original 20001)
    for G in (2, 4, 8):
        trips, parts = [], []
        for g in range(G):
            r0, cnt = parallel.shard_range(Xc.shape[0], G, g)
            sc = np.empty(cnt)
            o_, b_, n_ = C.c_int64(), C.c_double(), C.c_int64()
            L.check(lib.b7_acq_score_range(f.handle, grid.handle, r0, cnt, L.SCORE_EI, 0.0, 0, -1.0, float(y.min()), L.dptr(sc),
                                           C.byref(o_), C.byref(b_), C.byref(n_)))
            trips.append((b_.value, o_.value, n_.value))
            parts.append(sc)
        b, i, n = parallel.combine_argmax(trips)
        assert (b, i, n) == (best.value, amo.value, nn.value)
        assert np.array_equal(np.concatenate(parts), full, equal_nan=True)   # scores bit-identical for any sharding
    f.free()


def _two_gpus():
    return L.lib().b7_device_count() >= 2


@pytest.mark.parametrize("S,path", [(8, L.PATH_INT8_OZAKI), (5, L.PATH_INT8_OZAKI), (4, L.PATH_FP64_DMMA)])
def test_multi_gpu_c_abi_equals_single_gpu(ctx, oracle, S, path):
    """(e) on real GPUs, through the C ABI only: b7_comm_init_all over every device of the box, Sobol shards generated
    per device, draw-sharded fit + NCCL exchange inside the library (all-gather when S divides, broadcasts otherwise),
    shard scoring and the (best, index, nan) combine -- must reproduce the one-GPU result bit for bit: log marginal
    likelihoods, every score, the selected candidate and the grid row it removes (bots/bayesopt.lua:56-99, bots/abstract.lua:118)."""
    if not _two_gpus():
        pytest.skip("needs at least 2 GPUs")
    G = min(L.lib().b7_device_count(), 8)
    N, d, M = 700, 6, 30011
    pts = oracle.sobol_points(d, N + M)
    Xo = pts[:N]
    y = oracle.hartmann6(Xo)
    y = (y - y.mean()) / y.std()
    r = np.random.default_rng(S)
    hyp = np.zeros((S, d + 3))
    hyp[:, :d] = np.log(0.15) + r.random((S, d)) * np.log(8)
    hyp[:, d + 1] = 0.5 * np.log(1e-2)
    fmin = float(y.min())
    keep = ctx.posterior_path()
    comm = parallel.Comm.all(G)
    try:
        ctx.set_posterior_path(path)
        for c in comm.ctxs:
            c.set_posterior_path(path)
        f = models.GPFactors(Xo, y, hyp)
        g1 = grids.sobol({"size": N + M, "dims": d}).generate_device(first=N, count=M)
        one = np.empty(M)
        am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
        L.check(L.lib().b7_acq_score(f.handle, g1.handle, L.SCORE_EI, 0.0, 0, -1.0, fmin, L.dptr(one), C.byref(am), C.byref(amo),
                                     C.byref(best), C.byref(nn)))
        gs = comm.sobol_grid(d, 1 + N, M)
        assert sum(g.rows() for g in gs) == M
        gps, info, logml, jit, gather_ms = comm.fit(Xo, y, hyp)
        assert (info == 0).all() and np.array_equal(logml, f.logml)
        b, a, ao, n_, sc = comm.acq_score(gps, gs, L.SCORE_EI, 0.0, 0, -1.0, fmin, want_scores=True)
        assert np.array_equal(sc, one)                                   # every score, bit for bit
        assert (b, a, ao, n_) == (best.value, am.value, amo.value, nn.value)
        # steal the nominated row on both, score again: compacted numbering stays global
        row_m = comm.grid_remove(gs, a)
        row_1 = g1.remove(am.value)
        assert np.array_equal(row_m, row_1.reshape(-1))
        L.check(L.lib().b7_acq_score(f.handle, g1.handle, L.SCORE_EI, 0.0, 0, -1.0, fmin, None, C.byref(am), C.byref(amo), C.byref(best),
                                     C.byref(nn)))
        b, a, ao, n_, _ = comm.acq_score(gps, gs, L.SCORE_EI, 0.0, 0, -1.0, fmin)
        assert (b, a, ao, n_) == (best.value, am.value, amo.value, nn.value)
        comm.free_fit(gps)
        for g in gs:
            g.free()
        g1.free()
        f.free()
    finally:
        ctx.set_posterior_path(keep)
        comm.close()


def test_multi_gpu_one_process_per_gpu(ctx):
    """The same exchange with one process per GPU (torchrun): b7_comm_unique_id / b7_comm_init_rank, the unique id
    carried by torch.distributed (gloo); rank 0 compares against its own one-GPU result (tools/multi_check.py)."""
    if not _two_gpus():
        pytest.skip("needs at least 2 GPUs")
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    G = min(L.lib().b7_device_count(), 8)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={G}", "--master-addr", "127.0.0.1",
                          "--master-port", "29517", os.path.join(root, "tools", "multi_check.py")], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "multi_check ok" in out.stdout


# ---------------------------------------------------------------------------------- grid bookkeeping

def test_grid_compaction_semantics(ctx):
    # utils.tensor.steal/remove (utils/tensor.lua:158-193): indices refer to the compacted tensor
    X = np.arange(40, dtype=np.float64).reshape(20, 2)
    ref = X.copy()
    g = grids.DeviceGrid.from_host(X)
    r = np.random.default_rng(2)
    for _ in range(12):
        idx = int(r.integers(1, ref.shape[0] + 1))
        row = g.remove(idx)
        assert np.array_equal(row[0], ref[idx - 1])
        ref = np.delete(ref, idx - 1, axis=0)
        assert g.size() == ref.shape[0]
        for c in (1, ref.shape[0]):
            assert np.array_equal(g.read(g.original_index(c) - 1, 1)[0], ref[c - 1])
    with pytest.raises(L.B7Error):
        g.remove(ref.shape[0] + 1)
    g.free()


# ---------------------------------------------------------------------------------- BLR head

def test_blr_against_golden(ctx, oracle):
    g = np.load(os.path.join(GOLD, "blr.npz"))
    f = models.BLRFactors(g["Z0"], g["y"], g["hyp"])
    assert (f.info == 0).all()
    for s in range(2):
        mu, var = f.predict(s, g["Z1"])
        assert rel(mu, g["mean"][s], 1.0) <= 1e-9
        assert rel(var, g["var"][s], 1e-300) <= 1e-9
    feats = grids.DeviceGrid.from_host(g["Z1"])
    sc = np.empty(g["Z1"].shape[0])
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
    fmin = float(g["y"].min())
    L.check(L.lib().b7_blr_score(f.handle, feats.handle, L.SCORE_EI, 0.0, 0, -1.0, fmin, L.dptr(sc), C.byref(am), C.byref(amo),
                                 C.byref(best), C.byref(nn)))
    ref = oracle.mc_average([oracle.ei_compute(g["mean"][s], g["var"][s], fmin, 0.0) for s in range(2)])
    assert rel(sc, ref, 1e-6 * ref.max()) <= 1e-7
    assert am.value == oracle.argmax_first(ref)[1]
    f.free()


@pytest.mark.parametrize("N,D", [(33, 1), (1000, 7), (5000, 50), (300, 64)])
def test_blr_shapes_vs_oracle(ctx, oracle, N, D):
    r = np.random.default_rng(N + D)
    Z0, y, Z1 = np.maximum(r.normal(size=(N, D)), 0), r.normal(size=N), np.maximum(r.normal(size=(1111, D)), 0)
    hyp = np.array([[0.0, np.log(50.0), 0.05]])
    f = models.BLRFactors(Z0, y, hyp)
    mr, vr = oracle.blr_predict(oracle.blr_fit(Z0, y, hyp[0]), Z1)
    mu, var = f.predict(0, Z1)
    assert rel(mu, mr, 1.0) <= 1e-9 and rel(var, vr, 1e-300) <= 1e-9
    f.free()
    with pytest.raises(L.B7Error):
        models.BLRFactors(np.zeros((10, 65)), np.zeros(10), hyp)


def test_dngo_device_pipeline(ctx, oracle):
    # config 4 of BASELINE.json in miniature, entirely on the device: Sobol grid -> MLP basis -> BLR moments
    # -> EI -> argmax, with a removed candidate carried from the input grid to the feature grid
    r = np.random.default_rng(21)
    d, h, N, M = 6, 50, 400, 30000
    Ws = [r.normal(size=(h, d)) / np.sqrt(d), r.normal(size=(h, h)) / np.sqrt(h), r.normal(size=(h, h)) / np.sqrt(h)]
    bs = [0.1 * r.normal(size=h) for _ in range(3)]
    sob = grids.sobol({"size": N + M, "dims": d})
    Xo = sob.generate({"size": N, "dims": d})
    y = oracle.hartmann6(Xo)
    y = (y - y.mean()) / y.std()
    grid = sob.generate_device(first=N, count=M)
    grid.remove(123)
    feats = models.mlp_features(grid, Ws, bs)
    Xc = grid.read()
    Zref = oracle.mlp_features(Xc, Ws, bs)
    Z = feats.read()
    assert Z.shape == (M, h) and np.max(np.abs(Z - Zref)) <= 1e-12 * max(1.0, np.max(np.abs(Zref)))
    Z0 = oracle.mlp_features(Xo, Ws, bs)
    hyp = np.array([[0.0, np.log(1e2), 0.0], [np.log(2.0), np.log(30.0), 0.1]])
    f = models.BLRFactors(Z0, y, hyp)
    sc = np.empty(M)
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
    fmin = float(y.min())
    L.check(L.lib().b7_blr_score(f.handle, feats.handle, L.SCORE_EI, 0.0, 0, -1.0, fmin, L.dptr(sc), C.byref(am), C.byref(amo),
                                 C.byref(best), C.byref(nn)))
    per = []
    for s in range(2):
        mr, vr = oracle.blr_predict(oracle.blr_fit(Z0, y, hyp[s]), Zref)
        per.append(oracle.ei_compute(mr, vr, fmin, 0.0))
    ref = oracle.mc_average(per)
    assert np.isnan(sc[122])                                        # removed row travels with the grid
    live = np.ones(M, dtype=bool)
    live[122] = False
    assert rel(sc[live], ref[live], 1e-6 * ref[live].max()) <= 1e-7
    b, i, n = oracle.argmax_first(np.where(live, ref, np.nan))
    assert amo.value == i and am.value == i - (1 if i > 123 else 0)
    # dngo:predict in one pass (b7_dngo_score): the basis is evaluated tile by tile in front of the head and Z1 is never
    # stored; same scores as the two-step path to rounding, same selected candidate
    sc2, am2, amo2, best2, nn2 = models.dngo_score(f, grid, Ws, bs, True, L.SCORE_EI, 0.0, 0, -1.0, fmin, want_scores=True)
    assert np.isnan(sc2[122]) and rel(sc2[live], ref[live], 1e-6 * ref[live].max()) <= 1e-7
    assert rel(sc2[live], sc[live], 1e-6 * ref[live].max()) <= 1e-12
    assert (am2, amo2) == (am.value, amo.value) and abs(best2 - best.value) <= 1e-12 * abs(best.value)
    with pytest.raises(L.B7Error, match="widths"):
        models.mlp_features(grid, [r.normal(size=(65, d))], [np.zeros(65)])
    f.free()


@pytest.mark.parametrize("D,S,layers", [(1, 1, (3,)), (7, 3, (4, 9)), (50, 5, (6,)), (63, 3, (20, 33, 40)), (64, 1, (6,))])
def test_dngo_tile_kernel_shapes_vs_oracle(ctx, oracle, D, S, layers):
    # DMMA tile kernels (blr_dmma.cu) at ragged widths: 1, below / above a fragment, the 63-wide limit of the head, more than
    # 4 draws (chunked), and D = 64 (falls back to the per-candidate kernels); ragged candidate counts (last tile partial)
    r = np.random.default_rng(D * 7 + S)
    dims = list(layers) + [D]
    Ws = [r.normal(size=(dims[i + 1], dims[i])) / np.sqrt(dims[i]) for i in range(len(dims) - 1)]
    bs = [0.1 * r.normal(size=dims[i + 1]) for i in range(len(dims) - 1)]
    N, M = 300, 128 * 37 + 5
    Xo, Xc = r.random((N, dims[0])), r.random((M, dims[0]))
    y = r.normal(size=N)
    Z0, Zref = oracle.mlp_features(Xo, Ws, bs), oracle.mlp_features(Xc, Ws, bs)
    hyp = np.stack([np.array([np.log(0.5 + s), np.log(20.0 + 10 * s), 0.05 * s]) for s in range(S)])
    f = models.BLRFactors(Z0, y, hyp)
    grid = grids.DeviceGrid.from_host(Xc)
    feats = models.mlp_features(grid, Ws, bs)
    assert np.max(np.abs(feats.read() - Zref)) <= 1e-12 * max(1.0, np.max(np.abs(Zref)))
    for s in range(S):
        mu, var = f.predict(s, Zref)
        mr, vr = oracle.blr_predict(oracle.blr_fit(Z0, y, hyp[s]), Zref)
        assert rel(mu, mr, 1.0) <= 1e-10 and rel(var, vr, 1e-300) <= 1e-9
    fmin = float(y.min())
    per = [oracle.ei_compute(*oracle.blr_predict(oracle.blr_fit(Z0, y, hyp[s]), Zref), fmin, 0.0) for s in range(S)]
    ref = oracle.mc_average(per)
    b, i, n = oracle.argmax_first(ref)
    if D <= 63:
        sc, am, amo, best, nn = models.dngo_score(f, grid, Ws, bs, True, L.SCORE_EI, 0.0, 0, -1.0, fmin, want_scores=True)
        assert rel(sc, ref, 1e-6 * max(ref.max(), 1e-300)) <= 1e-7 and am == i
    else:
        with pytest.raises(L.B7Error, match="tile kernel"):
            models.dngo_score(f, grid, Ws, bs, True, L.SCORE_EI, 0.0, 0, -1.0, fmin)
    f.free()


# ---------------------------------------------------------------------------------- the reference-facing API end to end

def test_reference_api_predict_and_scores(ctx, oracle):
    Xo, y, hyp, Xc = make_problem(oracle, 100, 2, 1, 4000, 1e-2)
    model = models.gp_regressor({"kernel": "ardse"})
    model.hyp = hyp[0]
    pred = model.predict(Xo, y, Xc, None, {"mean": True, "var": True})
    assert pred["mean"].shape == (4000, 1) and pred["var"].shape == (4000, 1)
    fit = oracle.gp_fit(Xo, y, hyp[0], 0)
    mr, vr = oracle.gp_predict(fit, Xc)
    assert rel(pred["mean"][:, 0], mr, 1.0) <= 1e-9 and rel(pred["var"][:, 0], vr, fit["sf2"]) <= 1e-9
    ei = scores.expected_improvement()(model, None, Xo, y, Xc)
    ref = oracle.ei_compute(mr, vr, float(y.min()), 0.0)
    assert ei.shape == (4000,) and rel(ei, ref, 1e-6 * ref.max()) <= 1e-7
    cb = scores.confidence_bound()(model, hyp[0], Xo, y, Xc)
    assert rel(cb, oracle.cb_compute(mr, vr), 1e-6) <= 1e-7


def test_speculative_hyper_sampling_gives_the_same_experiment(ctx, oracle):
    # batched density evaluations (one fit of 4 factors per device call) vs one factor per call: the factors
    # are computed independently per draw with a fixed order, so the chains and the nominations coincide
    import time
    hypers = [{"name": "x%d" % i, "size": 1, "min": 0.0, "max": 1.0} for i in range(2)]
    runs, walls = [], []
    for spec in (True, False):
        cfg = {"bot": {"budget": 9, "nInitial": 3, "nSamples": 3, "verbose": 0}, "grid": {"size": 3000},
               "model": {"speculative": spec}}
        bot = bots.bayesopt(lambda x: oracle.braninhoo(x)[0], hypers, cfg, rng=np.random.default_rng(11))
        t0 = time.perf_counter()
        bot.run_experiment()
        walls.append(time.perf_counter() - t0)
        runs.append((bot.observed.copy(), bot.responses.copy(), bot.model.hyp.copy()))
    assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1])
    assert np.array_equal(runs[0][2], runs[1][2])
    print("bayesopt 9 trials: speculative %.2f s, sequential %.2f s" % tuple(walls))


def test_bayesopt_loop_branin(ctx, oracle):
    # config 1 of BASELINE.json in miniature: Branin-Hoo 2D, EI, Sobol grid, fixed hyper draws
    hypers = [{"name": "x1", "size": 1, "min": 0.0, "max": 1.0}, {"name": "x2", "size": 1, "min": 0.0, "max": 1.0}]
    cfg = {"bot": {"budget": 12, "nInitial": 3, "nSamples": 4, "verbose": 0}, "grid": {"size": 5000}}
    bot = bots.bayesopt(lambda x: oracle.braninhoo(x)[0], hypers, cfg, rng=np.random.default_rng(4))
    assert bot.grid.rows() == 5000 and bot.config["grid"]["type"] == "sobol" and bot.config["bot"]["msg_freq"] == 1
    best = bot.run_experiment()
    assert bot.observed.shape == (12, 2) and bot.responses.shape == (12, 1) and bot.grid.size() == 5000 - 12
    assert best["y"].item() == bot.responses.min()
    # the nominated points are distinct grid rows and the last acquisition picked a live candidate
    assert len({tuple(r) for r in bot.observed}) == 12
    assert 1 <= bot.last["argmax"] <= 5000 - 11 and bot.last["nan_count"] == 0
    # an acquisition with given draws equals the oracle's choice on the compacted candidates
    hyps = np.tile(np.array([[np.log(0.3), np.log(0.3), 0.0, 0.5 * np.log(1e-2), 0.0]]), (2, 1))
    hyps[1, :2] = np.log(0.6)
    score, idx, bestv, _ = bot.acquire(hyps, want_score=True)
    ref = oracle.acquisition(bot.observed, bot.responses[:, 0], hyps, bot.candidates, 0, False, oracle.SCORE_EI)
    assert score.shape == (5000 - 12,) and idx == ref["idx"]
    assert rel(score, ref["score"], 1e-6 * ref["score"].max()) <= 1e-7


def test_bot_save_and_resume_through_the_t7_result_file(ctx, oracle, tmp_path):
    # bots/abstract.lua:234-240 (save) + :19-44 (cache protocol): a run persisted in Torch7 format resumes with its
    # observations, on the candidates that were still live, and then behaves like the uninterrupted run's state
    from bot7_b200 import t7
    hypers = [{"name": "x1", "size": 1, "min": 0.0, "max": 1.0}, {"name": "x2", "size": 1, "min": 0.0, "max": 1.0}]
    cfg = {"bot": {"budget": 6, "nInitial": 3, "nSamples": 2, "verbose": 0}, "grid": {"size": 2000}}
    bot = bots.bayesopt(lambda x: oracle.braninhoo(x)[0], hypers, cfg, rng=np.random.default_rng(5))
    bot.run_experiment()
    path = bot.save(str(tmp_path / "demo_bayesopt.t7"))
    res = t7.load(path)
    assert list(res) == ["best", "x", "y"] and np.array_equal(res["x"], bot.observed) and np.array_equal(res["y"], bot.responses)
    assert res["best"]["t"] == bot.best["t"] and np.array_equal(res["best"]["y"], bot.best["y"])
    cache = bots.cache_from_results(path, candidates=bot.candidates)
    again = bots.bayesopt(lambda x: oracle.braninhoo(x)[0], hypers, cfg, cache=cache, rng=np.random.default_rng(6))
    assert again.nTrials == 6 and again.grid.size() == 2000 - 6
    assert again.best["y"].item() == bot.responses.min() and again.best["t"] == int(bot.responses[:, 0].argmin()) + 1
    x, y = again.run_trial()
    assert again.nTrials == 7 and again.observed.shape == (7, 2) and np.array_equal(again.observed[:6], bot.observed)
    assert not any(np.array_equal(x[0], o) for o in bot.observed)              # a fresh grid row, not a repeat


def test_nonfinite_hyper_parameters_return_instead_of_hanging(ctx, oracle):
    """sigma_f^2 = exp(1600) = inf makes every entry of K infinite: the jitter policy's give-up test `eps > ||K||_F` can never
    fire (utils/math.lua:184), so the retry loop must treat a non-finite norm as give-up (oracle/SPEC.md).  The call returns at
    once with jitter = inf / a non-finite likelihood, and the handle stays usable."""
    import time
    Xo, y, hyp, _ = make_problem(oracle, 150, 2, 2, 10, 1e-2)
    bad = hyp.copy()
    bad[1, 2] = 800.0
    t0 = time.perf_counter()
    f = models.GPFactors(Xo, y, bad, flags=L.FIT_LOGML_ONLY)
    assert time.perf_counter() - t0 < 5.0
    ref = oracle.gp_fit(Xo, y, hyp[0], 0)["logml"]
    assert abs(f.logml[0] - ref) <= 1e-9 * abs(ref)                     # the healthy draw next to it is unaffected
    assert f.info[1] != 0 or not np.isfinite(f.logml[1]) or np.isinf(f.jitter[1])
    g = f.refit(hyp, L.FIT_LOGML_ONLY)                                  # and the handle still works
    assert abs(g.logml[1] - oracle.gp_fit(Xo, y, hyp[1], 0)["logml"]) <= 1e-9 * abs(ref)
    f.free()
    # the same draw through the full fit (factor + inversion + slicing) and a prediction: returns, and the healthy draw is exact
    t0 = time.perf_counter()
    p = models.GPFactors(Xo, y, bad)
    Xs = oracle.sobol_points(2, 64)
    m0, v0 = p.predict(0, Xs)
    m1, v1 = p.predict(1, Xs)
    assert time.perf_counter() - t0 < 5.0
    mr, vr = oracle.gp_predict(oracle.gp_fit(Xo, y, hyp[0], 0), Xs)
    assert rel(m0, mr, 1.0) <= 1e-9 and m1.shape == (64,) and v1.shape == (64,)
    p.free()

"""The DNGO head's hyper-parameter chain on the GPU: b7_blr_refit's log evidence against the oracle, refit = fit bit for bit,
slot independence, failing rows, the chains of the Python twin and of the Lua glue, and DNGO end to end with sampling on.

Bars: log evidence 1e-11 * max(|log p|, N); mean 1e-9; variance 1e-9 relative; EI 1e-7 relative with the same argmax.
Each check prints its worst error against its bar (run with -s to see them)."""
import math
import os
import sys

import numpy as np
import pytest

from blr_evidence_oracle import blr_log_evidence

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DS = [1, 7, 8, 9, 16, 33, 50, 63, 64]
NS = [1, 37, 20000]


def features(N, D, seed, dead=0, fit=False):
    """ReLU features of a two-layer net on 6 inputs (the last `dead` units never fire: all-zero columns), and responses:
    a smooth function of the inputs, or (fit=True) a linear function of the features plus 1e-3 noise."""
    r = np.random.default_rng(seed)
    X = r.uniform(-1, 1, (N, 6))
    W1, b1 = r.standard_normal((6, 32)) / math.sqrt(6), 0.2 * r.standard_normal(32)
    H = np.maximum(X @ W1 + b1, 0.0)
    W2, b2 = r.standard_normal((32, D)) / math.sqrt(8), 0.2 * r.standard_normal(D)
    b2[D - dead:] = -1e3
    Z = np.maximum(H @ W2 + b2, 0.0)
    if fit:
        y = Z @ r.standard_normal(D) / math.sqrt(D) + 1e-3 * r.standard_normal(N)
    else:
        y = np.sin(2 * X[:, 0]) + X[:, 1] * X[:, 2] - 0.5 * X[:, 3] ** 2 + 0.05 * r.standard_normal(N)
    return Z, y


def rows_for(N, D, y):
    """(alpha_p, beta) rows spanning alpha_p 1e-3 .. 1e2 and beta 1e-1 .. 1e4, m off the data mean.  With N <= D the Gram has a
    null space, where the rounding of any two fp64 Gram sums (about eps beta |G|) is divided by alpha_p: there the rows keep
    beta / alpha_p <= 100 and still cover both ends of both ranges."""
    m0 = float(np.mean(y)) if N else 0.0
    if N > D:
        pairs = [(a, b) for a in (1e-3, 1.0, 1e2) for b in (1e-1, 1e2, 1e4)]
    else:
        pairs = [(1e-3, 1e-1), (1e-1, 1e-1), (1.0, 1e2), (1e2, 1e4), (1e2, 1e-1), (1e-2, 1.0)]
    return np.array([[math.log(a), math.log(b), m0 + 0.3 * (k % 3 - 1)] for k, (a, b) in enumerate(pairs)])


def rel(a, b, floor):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


@pytest.fixture(scope="module")
def M(ctx):
    from bot7_b200 import _lib, grids, models
    return models, _lib, grids


@pytest.mark.gpu
@pytest.mark.parametrize("N", NS)
def test_log_evidence_matches_the_oracle(M, oracle, N):
    models, L, _ = M
    worst = (0.0, None)
    for D in DS:
        cases = [features(N, D, 100 + D, dead=min(3, D - 1) if D > 3 else 0)]
        if N > D:
            cases.append(features(N, D, 200 + D, fit=True))       # features explain y: the residual is small at beta = 1e4
        for Z, y in cases:
            H = rows_for(N, D, y)
            f = models.BLRFactors(Z, y, H)
            lev, info = f.refit(H, L.FIT_LOGML_ONLY)
            assert f.S == len(H) and L.lib().b7_blr_num_draws(f.handle) == len(H)
            for s, h in enumerate(H):
                ref = blr_log_evidence(Z, y, h)
                assert math.isfinite(ref) and info[s] == 0, (N, D, h)
                err = abs(lev[s] - ref) / max(abs(ref), N)
                if err > worst[0]:
                    worst = (err, (N, D, tuple(np.exp(h[:2]))))
                assert err <= 1e-11, (N, D, h, lev[s], ref)
            f.free()
    print(f"\nlog evidence N={N}: worst {worst[0]:.2e} of max(|log p|, N) at (N, D, (alpha_p, beta)) = {worst[1]} [bar 1e-11]")


def _dngo_problem(N, M_, seed=3):
    r = np.random.default_rng(seed)
    X = r.uniform(0, 1, (N + M_, 4))
    Xo, Xc = X[:N], X[N:]
    Ws = [r.standard_normal((24, 4)) / 2.0, r.standard_normal((40, 24)) / 5.0]
    bs = [0.1 * r.standard_normal(24), 0.1 * r.standard_normal(40)]
    y = np.sin(4 * Xo[:, 0]) * np.cos(3 * Xo[:, 1]) + Xo[:, 2] - Xo[:, 3] ** 2
    return Xo, (y - y.mean()) / y.std(), Xc, Ws, bs


def _oracle_scores(oracle, Z0, y, Z1, H):
    per, means, vars_ = [], [], []
    for h in H:
        mu, var = oracle.blr_predict(oracle.blr_fit(Z0, y, h), Z1)
        means.append(mu)
        vars_.append(var)
        per.append(oracle.ei_compute(mu, var, float(y.min()), 0.0))
    return np.array(means), np.array(vars_), oracle.mc_average(per)


@pytest.mark.gpu
def test_refit_equals_fit_and_new_rows_match_the_oracle(M, oracle):
    models, L, grids = M
    Xo, y, Xc, Ws, bs = _dngo_problem(700, 6000)
    Z0, Z1 = oracle.mlp_features(Xo, Ws, bs), oracle.mlp_features(Xc, Ws, bs)
    R0 = np.array([[0.0, math.log(1e2), y.mean()], [math.log(0.3), math.log(20.0), 0.1], [math.log(5.0), math.log(400.0), -0.2]])
    R1 = np.array([[math.log(2.0), math.log(50.0), 0.05], [math.log(1e-2), math.log(1e3), -0.1], [math.log(10.0), math.log(5.0), 0.3]])
    grid = grids.DeviceGrid.from_host(Xc)

    def outputs(f):
        mv = [f.predict(s, Z1) for s in range(f.S)]
        sc = models.dngo_score(f, grid, Ws, bs, want_scores=True, fmin=float(y.min()))
        return mv, sc
    fresh = models.BLRFactors(Z0, y, R0)
    a_mv, a_sc = outputs(fresh)
    f = models.BLRFactors(Z0, y, R1)
    f.refit(R1, L.FIT_LOGML_ONLY)
    with pytest.raises(L.B7Error, match="LOGML_ONLY"):
        f.predict(0, Z1)                                            # a log-evidence refit leaves no predictor behind
    lev, info = f.refit(R0, L.FIT_PREDICT)
    b_mv, b_sc = outputs(f)
    for (ma, va), (mb, vb) in zip(a_mv, b_mv):
        assert np.array_equal(ma, mb) and np.array_equal(va, vb)
    assert np.array_equal(a_sc[0], b_sc[0]) and a_sc[1:] == b_sc[1:]
    assert np.array_equal(info, [0, 0, 0]) and np.isfinite(lev).all()
    # new rows on the refitted handle against the oracle
    fresh.refit(R1, L.FIT_PREDICT)
    means, vars_, ei = _oracle_scores(oracle, Z0, y, Z1, R1)
    em = ev = 0.0
    for s in range(3):
        mu, var = fresh.predict(s, Z1)
        em, ev = max(em, rel(mu, means[s], 1.0)), max(ev, rel(var, vars_[s], 1e-300))
    sc, am, amo, best, nn = models.dngo_score(fresh, grid, Ws, bs, want_scores=True, fmin=float(y.min()))
    eei = rel(sc, ei, 1e-300 + 1e-6 * ei.max())
    b, i, _ = oracle.argmax_first(ei)
    print(f"\nrefit to new rows: mean {em:.2e} [1e-9], var rel {ev:.2e} [1e-9], EI rel {eei:.2e} [1e-7], argmax {am} vs {i}")
    assert em <= 1e-9 and ev <= 1e-9 and eei <= 1e-7 and am == i and nn == 0


@pytest.mark.gpu
def test_slots_are_independent(M, oracle):
    models, L, _ = M
    Z, y = features(5000, 50, 7)
    r = np.random.default_rng(1)
    H = np.column_stack([r.uniform(-5, 4, 8), r.uniform(-2, 9, 8), y.mean() + r.uniform(-0.5, 0.5, 8)])
    f8 = models.BLRFactors(Z, y, H)
    lev8, _ = f8.refit(H, L.FIT_LOGML_ONLY)
    f1 = models.BLRFactors(Z, y, H[:1])
    for s in range(8):
        lev1, _ = f1.refit(H[s:s + 1], L.FIT_LOGML_ONLY)
        assert lev1[0] == lev8[s], s
    # the same rows in another order: every slot keeps its bits
    perm = r.permutation(8)
    levp, _ = f8.refit(H[perm], L.FIT_LOGML_ONLY)
    assert np.array_equal(levp, lev8[perm])
    # a short batch through the twin (padded by repeating its last row) = one evaluation at a time
    bl = models.bayes_linear({"sampler": "slice", "spec_width": 8})
    batch = bl.log_density_batch(H[:5], Z, y)
    assert np.array_equal(batch, [bl.log_density(h, Z, y) for h in H[:5]])
    assert np.array_equal(batch, [lev8[s] - 0.5 * np.sum((H[s] / 2.0) ** 2) for s in range(5)])


@pytest.mark.gpu
def test_failing_rows_are_minus_inf_and_leave_their_neighbours_alone(M, oracle):
    models, L, _ = M
    Z, y = features(3000, 33, 9, dead=2)
    H = np.array([[0.0, math.log(1e2), y.mean()]] * 8) + np.linspace(-0.5, 0.5, 8)[:, None] * [1.0, 1.0, 0.1]
    f = models.BLRFactors(Z, y, H)
    good, _ = f.refit(H, L.FIT_LOGML_ONLY)
    bad = H.copy()
    bad[2, 0] = 800.0                                               # alpha_p = exp(800) overflows: the factor fails
    bad[5, :2] = [800.0, -800.0]
    bad[6, 1] = -800.0                                              # beta underflows to 0: a finite (tiny) evidence
    lev, info = f.refit(bad, L.FIT_LOGML_ONLY)
    assert lev[2] == -np.inf and lev[5] == -np.inf and info[2] != 0 and info[5] != 0
    ref6 = blr_log_evidence(Z, y, bad[6])
    assert abs(lev[6] - ref6) <= 1e-11 * max(abs(ref6), len(y))
    for s in (0, 1, 3, 4, 7):
        assert lev[s] == good[s] and info[s] == 0
    bl = models.bayes_linear()
    assert bl.log_density_batch(bad, Z, y)[2] == -np.inf


class _Recorder:
    """numpy Generator stand-in that records the uniform draws, to recover the slice level Y = f(x0) + log u."""

    def __init__(self, rng):
        self.rng, self.u = rng, []

    def random(self, *a):
        v = self.rng.random(*a)
        self.u.append(v)
        return v

    def standard_normal(self, *a):
        return self.rng.standard_normal(*a)


@pytest.mark.gpu
def test_chains_speculative_sequential_and_oracle(M, oracle):
    models, L, _ = M
    from bot7_b200 import samplers
    Z, y = features(20000, 50, 11)
    cfg = {"sampler": "slice", "nSamples": 6}
    spec = models.bayes_linear(dict(cfg, speculative=True), rng=np.random.default_rng(21))
    seq = models.bayes_linear(dict(cfg, speculative=False), rng=np.random.default_rng(21))
    a = np.concatenate([spec.sample_hypers(Z, y), spec.sample_hypers(Z, y)])       # the chain state is kept across calls
    b = np.concatenate([seq.sample_hypers(Z, y), seq.sample_hypers(Z, y)])
    assert np.array_equal(a, b) and a.shape == (12, 3)
    assert spec.rng.random() == seq.rng.random()
    assert len({tuple(r) for r in a}) == 12                                        # the chain moves
    # the same chain driven by the oracle's density
    rec = _Recorder(np.random.default_rng(21))
    x = spec.default_hyp(y)
    out, margin = [], math.inf
    for _ in range(12):
        vals = []

        def dens(v):
            h = np.asarray(v).reshape(-1)
            vals.append(blr_log_evidence(Z, y, h) - 0.5 * float(np.sum((h / 2.0) ** 2)))
            return vals[-1]
        rec.u.clear()
        x = samplers.slice()(lambda v, _a: dens(v), x, {"nSamples": 1}, None, rng=rec)
        Y = vals[0] + math.log(rec.u[0])
        margin = min([margin] + [abs(v - Y) for v in vals[1:]])
        out.append(x[0].copy())
    err = float(np.max(np.abs(np.array(out) - a)))
    print(f"\nGPU chain vs oracle chain: max |diff| {err:.2e} [atol 1e-9]; smallest slice margin |f(x) - Y| met: {margin:.3e}")
    assert err <= 1e-9


@pytest.mark.gpu
def test_lua_chain_matches_the_python_twin(ctx, oracle):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from minilua.harness import GlueRuntime
    from bot7_b200 import models
    Z, y = features(4000, 40, 13)
    h0 = np.array([[0.0, math.log(1e2), float(y.mean())]])
    rt = GlueRuntime(seed=9)
    rt.run("require('bot7_b200').install()")
    for name, v in [("Z0", Z), ("Y0", y.reshape(-1, 1)), ("H0", h0)]:
        rt.set_global(name, rt.tensor(v))
    r = rt.run(r"""
local net = nn.Sequential():add(nn.Linear(6, 24)):add(nn.ReLU()):add(nn.Linear(24, 40)):add(nn.ReLU()):add(nn.Linear(40, 1))
local model = bot7.models.dngo({network = net, basis = net:get(4), zDim = 40, update = {schedule = {batchsize = 32}},
                                predictor = {sampler = 'slice', nSamples = 5, spec_width = 8}})
model.blr_state = H0:clone()
torch.manualSeed(9)                          -- the network's initialisation drew from the generator: restart it for the chain
local draws = model:sample_blr_hypers(Z0, Y0)
return draws, model.blr_state, torch.rand(1)[1]
""")
    draws, state, nxt, calls = r[0].a.copy(), r[1].a.copy(), r[2], list(rt.ffi.calls)
    rt.close()
    tw = models.bayes_linear({"sampler": "slice", "nSamples": 5, "spec_width": 8}, rng=np.random.default_rng(9))
    tw.hyp = h0[0].copy()
    ref = tw.sample_hypers(Z, y)
    # eight density evaluations per device call: one b7_blr_fit for the resident handle, then one b7_blr_refit per batch
    n_fit, n_refit = calls.count("b7_blr_fit"), calls.count("b7_blr_refit")
    print(f"\nLua chain vs twin: max |diff| {float(np.max(np.abs(draws - ref))):.2e} [atol 1e-9]; device calls: "
          f"{n_fit} b7_blr_fit + {n_refit} b7_blr_refit for 5 draws")
    assert n_fit == 1 and 5 <= n_refit <= 40
    assert draws.shape == (5, 3) and np.allclose(draws, ref, rtol=0.0, atol=1e-9)
    assert np.allclose(state[0], tw.hyp, rtol=0.0, atol=1e-9)
    assert nxt == tw.rng.random()


@pytest.mark.gpu
def test_dngo_end_to_end_with_sampling(ctx, oracle):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from minilua.harness import GlueRuntime
    from bot7_b200 import grids, models
    Xo, y, Xc, _, _ = _dngo_problem(400, 5000, seed=5)
    rt = GlueRuntime(seed=5)
    rt.run("require('bot7_b200').install()")
    for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("XC", Xc)]:
        rt.set_global(name, rt.tensor(v))
    r = rt.run(r"""
local B, ffi = require('bot7_b200.ffi'), require('ffi')
local net = nn.Sequential():add(nn.Linear(4, 24)):add(nn.ReLU()):add(nn.Linear(24, 50)):add(nn.ReLU()):add(nn.Linear(50, 1))
local model = bot7.models.dngo({network = net, basis = net:get(4), zDim = 50, update = {schedule = {batchsize = 32}},
                                predictor = {sampler = 'slice', nSamples = 4}})
local p = model:predict(X0, Y0, XC, nil, {mean = true, var = true})
local rows_p = model.blr_rows:clone()
local box = ffi.new('b7_grid*[1]')
B.check(B.C.b7_grid_from_host(B.context(), XC:data(), XC:size(1), XC:size(2), box), 'b7_grid_from_host')
local grid = ffi.gc(box[0], B.C.b7_grid_free)
local argmax, best, nans = model:acquire(X0, Y0, grid, B.C.B7_SCORE_EI, 0.0, B.C.B7_BOUND_LOWER, -1.0)
return p.mean, p.var, rows_p, argmax, best, nans, model.blr_rows, net:get(1).weight, net:get(1).bias, net:get(3).weight, net:get(3).bias
""")
    rt.close()
    W1, b1, W2, b2 = r[7].a, r[8].a, r[9].a, r[10].a
    rows_p, rows_a = r[2].a, r[6].a
    assert rows_p.shape == (4, 3) and rows_a.shape == (4, 3) and not np.array_equal(rows_p, rows_a)   # the chain went on
    Z0, Z1 = oracle.mlp_features(Xo, [W1, W2], [b1, b2]), oracle.mlp_features(Xc, [W1, W2], [b1, b2])
    means, vars_, _ = _oracle_scores(oracle, Z0, y, Z1, rows_p)
    em, ev = rel(r[0].a[:, 0], means.mean(0), 1.0), rel(r[1].a[:, 0], vars_.mean(0), 1e-300)
    _, _, ei = _oracle_scores(oracle, Z0, y, Z1, rows_a)
    best, idx, _ = oracle.argmax_first(ei)
    eb = abs(r[4] - best) / abs(best)
    # the Python twin: dngo.predict and dngo_score on the rows of its own chain
    Ws, bs = [W1, W2], [b1, b2]
    basis = lambda X: oracle.mlp_features(X, Ws, bs)                  # noqa: E731
    cfg = {"predictor": {"sampler": "slice", "nSamples": 4}}
    tw = models.dngo(cfg, basis, rng=np.random.default_rng(3))
    pr = tw.predict(Xo, y, Xc)
    rows_t = models.dngo(cfg, basis, rng=np.random.default_rng(3)).predictor.sample_hypers(Z0, y)
    tm, tv, _ = _oracle_scores(oracle, Z0, y, Z1, rows_t)
    etm, etv = rel(pr["mean"][:, 0], tm.mean(0), 1.0), rel(pr["var"][:, 0], tv.mean(0), 1e-300)
    f = tw.predictor.factors(Z0, y, "marginalize")                   # the next four states of the twin's chain
    _, _, ei_t = _oracle_scores(oracle, Z0, y, Z1, f.hyp)
    sc, am, _, bt, nn = models.dngo_score(f, grids.DeviceGrid.from_host(Xc), Ws, bs, want_scores=True, fmin=float(y.min()))
    et = rel(sc, ei_t, 1e-300 + 1e-6 * ei_t.max())
    print(f"\nDNGO with sampling: Lua mean {em:.2e} var {ev:.2e} EI(best) {eb:.2e} argmax {r[3]} vs {idx}; "
          f"twin mean {etm:.2e} var {etv:.2e} EI {et:.2e} argmax {am} vs {oracle.argmax_first(ei_t)[1]}")
    assert em <= 1e-9 and ev <= 1e-9 and r[3] == idx and eb <= 1e-7 and r[5] == 0
    assert etm <= 1e-9 and etv <= 1e-9 and et <= 1e-7 and am == oracle.argmax_first(ei_t)[1] and nn == 0


@pytest.mark.gpu
def test_default_dngo_uses_the_one_fixed_row(ctx, oracle):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from minilua.harness import GlueRuntime
    from bot7_b200 import models
    Xo, y, Xc, Ws, bs = _dngo_problem(300, 2000, seed=8)
    Z0 = oracle.mlp_features(Xo, Ws, bs)
    bl = models.bayes_linear()
    f = bl.factors(Z0, y, "marginalize")
    assert f.S == 1 and np.array_equal(f.hyp, [[0.0, math.log(1e2), float(np.mean(y))]]) and bl.hyp is None
    rt = GlueRuntime(seed=5)
    rt.run("require('bot7_b200').install()")
    for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("XC", Xc)]:
        rt.set_global(name, rt.tensor(v))
    r = rt.run(r"""
local net = nn.Sequential():add(nn.Linear(4, 24)):add(nn.ReLU()):add(nn.Linear(24, 50)):add(nn.ReLU()):add(nn.Linear(50, 1))
local model = bot7.models.dngo({network = net, basis = net:get(4), zDim = 50, update = {schedule = {batchsize = 32}}, predictor = {}})
model:predict(X0, Y0, XC, nil, {mean = true, var = true})
return model.blr_rows, model.blr_state == nil
""")
    calls = list(rt.ffi.calls)
    rt.close()
    assert calls.count("b7_blr_fit") == 1 and calls.count("b7_blr_refit") == 0 and r[1] is True
    assert np.array_equal(r[0].a, [[0.0, math.log(1e2), y.mean()]]) or np.allclose(r[0].a, [[0.0, math.log(1e2), y.mean()]], atol=1e-15)

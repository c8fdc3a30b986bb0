"""Per-layer activations of the DNGO basis (B7_ACT_NONE / RELU / TANH): the device tanh against mpmath, the features and the
fused score against the oracle on the tile kernel and on the per-layer fallback (B7_BLR_DMMA=0, in a child process), the ReLU
codes against the relu_last entries bit for bit, the multi-GPU entry, and the Lua glue's basis_stack.  The last tests run on
the CPU: the glue against the oracle-backed stand-in library of tests/fake_b7_act.py.  The reference features with activation
codes are tests/act_oracle.py's."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import act_oracle  # noqa: E402

NONE, RELU, TANH = 0, 1, 2
DIMS = 6


def rel(a, b, floor):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


def tanh_sweep():
    """Arguments of the tanh check: +-0, subnormals, 1e-300 .. 1e-8, both sides of the polynomial / quotient switch at 0.625,
    around the saturation point (1 - tanh x < 2^-54 from x ~ 19.06), 19 .. 40, +-inf, NaN; each with both signs."""
    r = np.random.default_rng(3)
    sw = np.array([0.625])
    near = lambda x, k: x * (1.0 + np.arange(-k, k + 1) * 2.0 ** -52)          # noqa: E731
    pos = np.concatenate([
        [0.0, 5e-324, 1e-320, 1e-310, 2.2250738585072009e-308, 2.2250738585072014e-308],
        np.logspace(-300, -8, 600), np.logspace(-8, 0, 2000), near(sw, 40), np.linspace(0.55, 0.7, 3000),
        np.linspace(0.7, 19.0, 3000), near(np.array([19.06154746539849]), 40), np.linspace(18.9, 19.3, 1000),
        np.linspace(19.0, 40.0, 500), [354.0, 709.0, 1e300, np.inf], r.random(4000) * 3.0])
    return np.concatenate([pos, -pos, [np.nan]])


def ulp_error(x, y):
    """|y - tanh(x)| in ulps of the correctly rounded tanh(x) (mpmath at 40 digits); inf where a special value is not exact."""
    import mpmath as mp
    mp.mp.dps = 40
    out = np.empty(len(x))
    for i, (a, b) in enumerate(zip(x, y)):
        if np.isnan(a):
            out[i] = 0.0 if np.isnan(b) else np.inf
        elif np.isinf(a):
            out[i] = 0.0 if b == math.copysign(1.0, a) else np.inf
        else:
            t = mp.tanh(mp.mpf(float(a)))
            out[i] = float(abs(mp.mpf(float(b)) - t) / np.spacing(abs(float(t))))
    return out


def net(widths, seed, scale=1.5):
    """A Linear stack of the given widths; pre-activations of order 1 so that tanh sees both sides of its switch point."""
    r = np.random.default_rng(seed)
    Ws = [r.standard_normal((widths[l + 1], widths[l])) * scale / math.sqrt(widths[l]) for l in range(len(widths) - 1)]
    bs = [0.3 * r.standard_normal(widths[l + 1]) for l in range(len(widths) - 1)]
    return Ws, bs


FEATURE_CASES = [  # widths, codes
    ([1, 7], [TANH]),
    ([DIMS, 50, 50, 50], [TANH, TANH, TANH]),
    ([7, 63, 1], [NONE, TANH]),
    ([DIMS, 64, 7, 50, 63], [TANH, RELU, NONE, TANH]),
    ([63, 50], [NONE]),
    ([64, 64, 64], [RELU, TANH]),
    ([1, 64, 63, 7], [TANH, NONE, RELU]),
]
M_FEAT = 128 * 23 + 45                                   # the last tile is partial


def feature_inputs(widths, k):
    return np.random.default_rng(100 + k).standard_normal((M_FEAT, widths[0]))


def device_outputs():
    """Everything the kernel comparison needs, computed with the library of this process: the tanh sweep through a 1 x 1
    identity layer, the mixed-code features and
    the ReLU codes next to relu_last."""
    from bot7_b200 import grids, models
    out = {}
    x = tanh_sweep()
    g = grids.DeviceGrid.from_host(x.reshape(-1, 1))
    out["tanh"] = models.mlp_features(g, [np.ones((1, 1))], [np.zeros(1)], act=[TANH]).read()[:, 0]
    for k, (widths, codes) in enumerate(FEATURE_CASES):
        Ws, bs = net(widths, k)
        g = grids.DeviceGrid.from_host(feature_inputs(widths, k))
        out[f"feat{k}"] = models.mlp_features(g, Ws, bs, act=codes).read()
    Ws, bs = net([DIMS, 24, 50], 9)
    g = grids.DeviceGrid.from_host(feature_inputs([DIMS], 9))
    for last in (0, 1):
        out[f"relu_old{last}"] = models.mlp_features(g, Ws, bs, bool(last)).read()
        out[f"relu_act{last}"] = models.mlp_features(g, Ws, bs, act=[RELU, RELU if last else NONE]).read()
    return out


@pytest.fixture(scope="module")
def fallback(ctx, tmp_path_factory):
    """device_outputs() of a child process with B7_BLR_DMMA=0: every layer on the per-layer kernels of blr.cu."""
    path = str(tmp_path_factory.mktemp("act") / "fallback.npz")
    env = dict(os.environ, B7_BLR_DMMA="0")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), path], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return dict(np.load(path))


@pytest.fixture(scope="module")
def tiles(ctx):
    return device_outputs()


def check_tanh(x, y):
    err = ulp_error(x, y)
    worst = int(np.argmax(err))
    print(f"\ntanh: {len(x)} points, max {err[worst]:.3f} ulp at x = {x[worst]!r}")
    assert err[worst] <= 2.0, (x[worst], y[worst])
    # a Linear output is never -0 on either kernel (the tile kernel's accumulator starts at +0, the per-layer kernel adds the
    # +0 products of its padding), so tanh(-0) = -0 cannot be observed through a layer: both zeros give +0
    z = x == 0
    assert np.all(y[z] == 0.0) and not np.signbit(y[z]).any()


@pytest.mark.gpu
def test_device_tanh_on_the_tile_kernel(tiles):
    x, y = tanh_sweep(), tiles["tanh"]
    check_tanh(x, y)


@pytest.mark.gpu
def test_device_tanh_on_the_fallback(fallback):
    check_tanh(tanh_sweep(), fallback["tanh"])


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["tiles", "fallback"])
def test_mixed_codes_features_vs_oracle(request, oracle, kernel):
    out = request.getfixturevalue(kernel)
    for k, (widths, codes) in enumerate(FEATURE_CASES):
        Ws, bs = net(widths, k)
        ref = act_oracle.mlp_features(feature_inputs(widths, k), Ws, bs, codes)
        Z = out[f"feat{k}"]
        assert Z.shape == ref.shape
        assert np.max(np.abs(Z - ref)) <= 1e-12 * max(1.0, np.max(np.abs(ref))), (widths, codes)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["tiles", "fallback"])
def test_relu_codes_are_the_relu_last_entry_bit_for_bit(request, kernel):
    out = request.getfixturevalue(kernel)
    for last in (0, 1):
        assert np.array_equal(out[f"relu_old{last}"].view(np.int64), out[f"relu_act{last}"].view(np.int64))


def head(oracle, widths, codes, S, seed):
    Ws, bs = net(widths, seed)
    r = np.random.default_rng(seed + 1)
    Xo = r.random((400, widths[0]))
    y = oracle.hartmann6(Xo) if widths[0] == 6 else np.sin(3 * Xo).sum(1)
    y = (y - y.mean()) / y.std()
    Z0 = act_oracle.mlp_features(Xo, Ws, bs, codes)
    hyp = np.column_stack([np.log(0.5) + r.random(S), np.log(20.0) + r.random(S), y.mean() + 0.1 * (r.random(S) - 0.5)])
    return Ws, bs, Z0, y, hyp


SCORE_CASES = [  # widths, codes, S, kind, bound
    ([DIMS, 50, 50, 50], [TANH, TANH, TANH], 1, 0, 0),
    ([DIMS, 50, 50, 50], [TANH, TANH, TANH], 5, 1, 0),
    ([DIMS, 24, 40], [TANH, NONE], 5, 0, 0),
    ([DIMS, 33, 17], [RELU, TANH], 1, 1, 1),
    ([DIMS, 20, 7, 40, 50], [TANH, NONE, RELU, TANH], 5, 1, 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("widths,codes,S,kind,bound", SCORE_CASES)
def test_dngo_score_act_vs_oracle(ctx, oracle, widths, codes, S, kind, bound):
    """Head moments (through b7_mlp_features_act + b7_blr_predict), the fused score, the argmax; then a NaN candidate and a
    removed nominee: the NaN row is counted and skipped, the removed row scores NaN and the next nominee is the oracle's."""
    from bot7_b200 import _lib as L
    from bot7_b200 import grids, models
    Ws, bs, Z0, y, hyp = head(oracle, widths, codes, S, seed=len(widths) + 10 * S + kind + 3 * bound)
    M = 128 * 151 + 77
    Xc = np.random.default_rng(5).random((M, widths[0]))
    has_nan = RELU not in codes         # ReLU maps a NaN pre-activation to 0 on the device (v > 0 ? v : 0), as it always has
    if has_nan:
        Xc[1000, 2] = np.nan
    Zref = act_oracle.mlp_features(Xc, Ws, bs, codes)
    f = models.BLRFactors(Z0, y, hyp)
    grid = grids.DeviceGrid.from_host(Xc)
    try:
        feats = models.mlp_features(grid, Ws, bs, act=codes)
        Z = feats.read()
        fin = np.isfinite(Zref).all(1)
        assert np.array_equal(fin, np.isfinite(Z).all(1))
        per = []
        fmin, tradeoff, sign = float(y.min()), (0.0 if kind == 0 else 2.0), -1.0
        for s in range(S):
            mu, var = f.predict(s, Z[fin])
            mr, vr = oracle.blr_predict(oracle.blr_fit(Z0, y, hyp[s]), Zref[fin])
            assert rel(mu, mr, 1.0) <= 1e-10 and rel(var, vr, 1e-300) <= 1e-9
            mr, vr = np.full(M, np.nan), np.full(M, np.nan)
            mr[fin], vr[fin] = oracle.blr_predict(oracle.blr_fit(Z0, y, hyp[s]), Zref[fin])
            per.append(oracle.ei_compute(mr, vr, fmin, tradeoff) if kind == 0 else
                       oracle.cb_compute(mr, vr, tradeoff, "upper" if bound == 1 else "lower", sign))
        ref = oracle.mc_average(np.array(per))
        b, i, n = oracle.argmax_first(ref)
        sc, am, amo, best, nn = models.dngo_score(f, grid, Ws, bs, kind=kind, tradeoff=tradeoff, bound=bound, sign=sign, fmin=fmin,
                                                  want_scores=True, act=codes)
        live = np.isfinite(ref)
        floor = 1e-6 * max(np.abs(ref[live]).max(), 1e-300)
        assert np.isnan(sc[1000]) == has_nan and nn == n == int(has_nan)
        assert rel(sc[live], ref[live], floor) <= 1e-7 and am == amo == i and abs(best - b) <= 1e-7 * max(abs(b), floor)
        grid.remove(i)
        sc2, am2, amo2, best2, nn2 = models.dngo_score(f, grid, Ws, bs, kind=kind, tradeoff=tradeoff, bound=bound, sign=sign, fmin=fmin,
                                                       want_scores=True, act=codes)
        ref2 = ref.copy()
        ref2[i - 1] = np.nan
        b2, i2, _ = oracle.argmax_first(ref2)
        assert np.isnan(sc2[i - 1]) and amo2 == i2 and am2 == i2 - (1 if i2 > i else 0) and nn2 == nn
    finally:
        f.free()


@pytest.mark.gpu
def test_relu_codes_score_bit_for_bit(ctx, oracle):
    from bot7_b200 import grids, models
    for last in (0, 1):
        widths = [DIMS, 32, 50]
        codes = [RELU, RELU if last else NONE]
        Ws, bs, Z0, y, hyp = head(oracle, widths, codes, 5, seed=40 + last)
        grid = grids.DeviceGrid.from_host(np.random.default_rng(6).random((128 * 40 + 3, DIMS)))
        f = models.BLRFactors(Z0, y, hyp)
        old = models.dngo_score(f, grid, Ws, bs, bool(last), fmin=float(y.min()), want_scores=True)
        new = models.dngo_score(f, grid, Ws, bs, fmin=float(y.min()), want_scores=True, act=codes)
        assert np.array_equal(old[0].view(np.int64), new[0].view(np.int64)) and old[1:] == new[1:]
        f.free()


@pytest.mark.gpu
def test_unknown_codes_are_refused_before_device_work(ctx, oracle):
    from bot7_b200 import _lib as L
    from bot7_b200 import grids, models
    Ws, bs, Z0, y, hyp = head(oracle, [DIMS, 32, 50], [TANH, TANH], 2, seed=51)
    grid = grids.DeviceGrid.from_host(np.random.default_rng(7).random((5000, DIMS)))
    f = models.BLRFactors(Z0, y, hyp)
    before = ctx.launch_count()
    for bad in ([TANH, 3], [-1, RELU]):
        with pytest.raises(L.B7Error, match="unknown activation code"):
            models.mlp_features(grid, Ws, bs, act=bad)
        with pytest.raises(L.B7Error, match="unknown activation code"):
            models.dngo_score(f, grid, Ws, bs, fmin=0.0, act=bad)
    assert ctx.launch_count() == before and grid.size() == 5000
    f.free()


def _n_gpus():
    from bot7_b200 import _lib as L
    return min(L.lib().b7_device_count(), 8)


@pytest.fixture(scope="module")
def comm(ctx):
    from bot7_b200 import parallel
    c = parallel.Comm.all(_n_gpus())
    yield c
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("S,kind,bound", [(1, 0, 0), (5, 1, 1)])
def test_dngo_score_multi_act_equals_one_device(ctx, comm, oracle, S, kind, bound):
    if comm.world < 2:
        pytest.skip("needs at least 2 GPUs")
    from bot7_b200 import grids, models
    widths, codes = [DIMS, 50, 50, 50], [TANH, TANH, TANH]
    Ws, bs, Z0, y, hyp = head(oracle, widths, codes, S, seed=70 + S)
    M = 128 * 97 + 13
    Xc = np.random.default_rng(8).random((M, DIMS))
    Xc[17, 0] = np.nan
    fmin, tradeoff = float(y.min()), 1.5
    one, gs = models.BLRFactors(Z0, y, hyp), comm.grid_from_host(Xc)
    blrs, _ = comm.blr_fit(Z0, y, hyp)
    g1 = grids.DeviceGrid.from_host(Xc)
    try:
        sc, am, amo, best, nn = models.dngo_score(one, g1, Ws, bs, kind=kind, tradeoff=tradeoff, bound=bound, fmin=fmin, want_scores=True,
                                                  act=codes)
        bm, amm, aomm, nm, scm = comm.dngo_score(blrs, gs, Ws, bs, kind=kind, tradeoff=tradeoff, bound=bound, fmin=fmin, want_scores=True,
                                                 act=codes)
        assert (amm, aomm, nm) == (am, amo, nn) and np.array_equal(np.array([bm]), np.array([best]), equal_nan=True)
        assert np.array_equal(scm.view(np.int64), sc.view(np.int64))
    finally:
        comm.free_blr(blrs)
        one.free()
        for g in gs:
            g.free()


@pytest.mark.gpu
def test_dngo_score_multi_act_refuses_unknown_codes_on_every_rank(ctx, comm, oracle):
    from bot7_b200 import _lib as L
    Ws, bs, Z0, y, hyp = head(oracle, [DIMS, 32, 50], [TANH, TANH], 2, seed=81)
    M = 10007
    gs = comm.sobol_grid(DIMS, 1, M)
    blrs, _ = comm.blr_fit(Z0, y, hyp)
    try:
        before = [c.launch_count() for c in comm.ctxs]
        sizes = [g.size() for g in gs]
        dims = (C.c_int * 3)(DIMS, 32, 50)
        Wa, ba = [L.as_f64(w) for w in Ws], [L.as_f64(b) for b in bs]
        Wp = (C.POINTER(C.c_double) * 2)(*[L.dptr(w) for w in Wa])
        bp = (C.POINTER(C.c_double) * 2)(*[L.dptr(b) for b in ba])
        sc = np.full(M, 7.0)
        am, amo, best, nn = C.c_int64(-5), C.c_int64(-5), C.c_double(-5.0), C.c_int64(-5)
        rc = L.lib().b7_dngo_score_multi_act(comm.handle, (C.c_void_p * comm.n_local)(*blrs), comm._handles(gs), 2, dims, Wp, bp,
                                             (C.c_int * 2)(TANH, 7), 0, 0.0, 0, -1.0, 0.0, L.dptr(sc), C.byref(am), C.byref(amo),
                                             C.byref(best), C.byref(nn))
        assert rc == -1 and "unknown activation code" in L.lib().b7_last_error().decode()
        assert (sc == 7.0).all() and (am.value, amo.value, best.value, nn.value) == (-5, -5, -5.0, -5)
        assert [c.launch_count() for c in comm.ctxs] == before and [g.size() for g in gs] == sizes
        m = comm.dngo_score(blrs, gs, Ws, bs, fmin=float(y.min()), act=[TANH, TANH])
        assert m[1] >= 1
    finally:
        comm.free_blr(blrs)
        for g in gs:
            g.free()


# ---------------------------------------------------------------------------------- the Lua glue (tools/minilua)

LUA_STANDINS = r"""
if not nn.Identity then
  local I, pI = torch.class('nn.Identity', 'nn.Module')
  function I:__init() pI.__init(self) end
  function I:updateOutput(input) self.output = input; return input end
  -- Torch7 nn.Dropout(p, v1): v2 (the default) scales by 1 / (1 - p) in training and is the identity in evaluation mode
  local D, pD = torch.class('nn.Dropout', 'nn.Module')
  function D:__init(p, v1) pD.__init(self); self.p = p or 0.5; self.v2 = not v1 end
  function D:updateOutput(input)
    if self.train or self.v2 then self.output = input else self.output = input:clone():mul(1 - self.p) end
    return self.output
  end
  local S, pS = torch.class('nn.Sigmoid', 'nn.Module')
  function S:__init() pS.__init(self) end
end
function MODEL(net, basis, zDim)
  return bot7.models.dngo({network = net, basis = basis, zDim = zDim, update = {schedule = {batchsize = 32}}, predictor = {}})
end
function CODES(net, basis)
  local st = MODEL(net, basis, 1):basis_stack()
  return table.concat(st.codes, ','), st.relu_form, st.relu_last, st.n
end
"""

LUA_ACQUIRE = r"""
local B, ffi = require('bot7_b200.ffi'), require('ffi')
local net = NET()
local model = MODEL(net, net:get(BASIS), ZDIM)
local p = model:predict(X0, Y0, XC, nil, {mean = true, var = true})
local box = ffi.new('b7_grid*[1]')
B.check(B.C.b7_grid_from_host(B.context(), XC:data(), XC:size(1), XC:size(2), box), 'b7_grid_from_host')
local grid = ffi.gc(box[0], B.C.b7_grid_free)
local argmax, best, nans = model:acquire(X0, Y0, grid, B.C.B7_SCORE_EI, 0.0, B.C.B7_BOUND_LOWER, -1.0)
local Ws, bs = {}, {}
for i = 1, net:size() do local m = net:get(i); if m.weight then Ws[#Ws + 1] = m.weight; bs[#bs + 1] = m.bias end end
return p.mean, argmax, best, Ws[1], bs[1], Ws[2], bs[2]
"""

NETS = {
    "tanh": ("nn.Sequential():add(nn.Linear(6, 24)):add(nn.Tanh()):add(nn.Linear(24, 50)):add(nn.Tanh()):add(nn.Linear(50, 1))",
             4, 50, [TANH, TANH]),
    "relu_dropout": ("nn.Sequential():add(nn.Linear(6, 24)):add(nn.ReLU()):add(nn.Dropout(0.5)):add(nn.Linear(24, 50)):add(nn.ReLU())"
                     ":add(nn.Identity()):add(nn.Linear(50, 1))", 6, 50, [RELU, RELU]),
}


def lua_acquire(rt, oracle, name):
    """The DNGO model of NETS[name]: predict and acquire through the glue, then the oracle's head mean and EI argmax."""
    src, basis, zdim, codes = NETS[name]
    r = np.random.default_rng(2)
    Xo, Xc = r.random((300, DIMS)), r.random((3000, DIMS))
    y = np.sin(3 * Xo).sum(1)
    y = (y - y.mean()) / y.std()
    rt.run("require('bot7_b200').install()")
    rt.run(LUA_STANDINS)
    for n, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("XC", Xc)]:
        rt.set_global(n, rt.tensor(v))
    rt.set_global("BASIS", basis)
    rt.set_global("ZDIM", zdim)
    rt.run("function NET() torch.manualSeed(4); return %s end" % src)
    res = rt.run(LUA_ACQUIRE)
    Ws, bs = [res[3].a, res[5].a], [res[4].a, res[6].a]
    Z0, Z1 = act_oracle.mlp_features(Xo, Ws, bs, codes), act_oracle.mlp_features(Xc, Ws, bs, codes)
    mr, vr = oracle.blr_predict(oracle.blr_fit(Z0, y, [0.0, np.log(1e2), float(y.mean())]), Z1)
    _, idx, _ = oracle.argmax_first(oracle.ei_compute(mr, vr, float(y.min()), 0.0))
    return res, mr, idx


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tanh", "relu_dropout"])
def test_lua_dngo_act_on_the_gpu(ctx, oracle, name):
    """models.dngo under tools/minilua with the real library: a Linear/Tanh network through the _act entries, a
    Linear/ReLU/Dropout/Identity network through the relu_last entries, both against the oracle."""
    from minilua.harness import GlueRuntime
    rt = GlueRuntime(seed=5)
    try:
        res, mr, idx = lua_acquire(rt, oracle, name)
        calls = list(rt.ffi.calls)
    finally:
        rt.close()
    assert rel(res[0].a[:, 0], mr, 1.0) <= 1e-9 and res[1] == idx
    act = name == "tanh"
    assert ("b7_dngo_score_act" in calls) == act and ("b7_dngo_score" in calls) != act
    assert ("b7_mlp_features_act" in calls) == act and ("b7_mlp_features" in calls) != act


def _fake_rt(oracle):
    from fake_b7_act import FakeB7Act
    from minilua.harness import GlueRuntime
    fake = FakeB7Act(oracle)
    return GlueRuntime(seed=5, lib_resolver=lambda name: fake), fake


def test_lua_basis_stack_codes_and_refusals(oracle):
    """CPU: the codes basis_stack reads out of the network, which stacks keep the relu_last form, and the modules it refuses."""
    rt, _ = _fake_rt(oracle)
    try:
        rt.run("require('bot7_b200').install()")
        rt.run(LUA_STANDINS)
        L, T, R = "nn.Linear(6, 8)", "nn.Tanh()", "nn.ReLU()"

        def codes(mods, basis):
            return tuple(rt.run("local net = nn.Sequential()%s; return CODES(net, net:get(%d))"
                                % ("".join(":add(%s)" % m for m in mods), basis)))

        assert codes([L, T, "nn.Linear(8, 5)", T, "nn.Linear(5, 1)"], 4) == ("2,2", False, 0, 2)
        assert codes([L, T, "nn.Linear(8, 5)", "nn.Linear(5, 1)"], 3) == ("2,0", False, 0, 2)
        assert codes([L, "nn.Linear(8, 5)", R], 3) == ("0,1", False, 1, 2)
        assert codes([L, R, "nn.Dropout(0.5)", "nn.Linear(8, 5)", R, "nn.Identity()"], 6) == ("1,1", True, 1, 2)
        assert codes([L, R, "nn.Linear(8, 5)", "nn.Dropout(0.0, true)"], 4) == ("1,0", True, 0, 2)
        for mods, basis, msg in [([L, "nn.Sigmoid()", "nn.Linear(8, 5)"], 3, r"module 2 of the network \(nn.Sigmoid\) is not supported"),
                                 ([L, R, T, "nn.Linear(8, 5)"], 4, r"module 3 of the network \(nn.Tanh\) is a second activation"),
                                 ([L, "nn.Dropout(0.5, true)", "nn.Linear(8, 5)"], 3, r"module 2 of the network \(nn.Dropout\) is a v1"),
                                 ([T, L], 2, r"module 1 of the network \(nn.Tanh\) comes before the first nn.Linear")]:
            with pytest.raises(Exception, match=msg):
                codes(mods, basis)
    finally:
        rt.close()


def test_lua_tanh_acquire_with_the_stand_in_library(oracle):
    """CPU: a Linear/Tanh model's predict and acquire go through b7_mlp_features_act and b7_dngo_score_act with the codes
    [TANH, TANH] and nominate the oracle's argmax; a Linear/ReLU/Dropout model keeps the relu_last entries."""
    for name in ("tanh", "relu_dropout"):
        rt, fake = _fake_rt(oracle)
        try:
            res, mr, idx = lua_acquire(rt, oracle, name)
        finally:
            rt.close()
        assert rel(res[0].a[:, 0], mr, 1.0) <= 1e-9 and res[1] == idx
        if name == "tanh":
            assert fake.calls.count("b7_mlp_features_act") == 1 and fake.calls.count("b7_dngo_score_act") == 1
            assert "b7_dngo_score" not in fake.calls and fake.codes == [[TANH, TANH]] * 2
        else:
            assert fake.calls.count("b7_mlp_features") == 1 and fake.calls.count("b7_dngo_score") == 1 and not fake.codes


if __name__ == "__main__":
    # child process of the `fallback` fixture (B7_BLR_DMMA=0 in its environment)
    np.savez(sys.argv[1], **device_outputs())

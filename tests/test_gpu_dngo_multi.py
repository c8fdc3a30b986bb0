"""DNGO over several GPUs: b7_blr_fit_multi and b7_dngo_score_multi against the one-device b7_blr_fit / b7_dngo_score, and the
Lua glue's bots.bayesopt with a DNGO model and config.bot.nGPU > 1.

Each candidate's basis, head and score, including the sequential average over the S rows, do not depend on the tile or the
shard that holds it, and the head's fit has no atomics: every comparison with the one-device result below is bit for bit.
The communicator spans every device of the box up to 8; tests that need two or more devices skip on one.  The last test runs
on the CPU: the glue's multi-GPU DNGO branch against the stand-in library of tests/fake_b7_dngo_multi.py."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

N_OBS, DIMS = 600, 6


def _n_gpus():
    from bot7_b200 import _lib as L
    return min(L.lib().b7_device_count(), 8)


@pytest.fixture(scope="module")
def comm(ctx):
    from bot7_b200 import parallel
    c = parallel.Comm.all(_n_gpus())
    yield c
    c.close()


def _need_two(comm):
    if comm.world < 2:
        pytest.skip("needs at least 2 GPUs")


def net(widths, seed):
    """A Linear / ReLU stack of the given widths (widths[0] = DIMS): weights h_out x h_in like torch nn.Linear.weight."""
    r = np.random.default_rng(seed)
    Ws = [r.standard_normal((widths[l + 1], widths[l])) * math.sqrt(2.0 / widths[l]) for l in range(len(widths) - 1)]
    bs = [0.1 * r.standard_normal(widths[l + 1]) for l in range(len(widths) - 1)]
    return Ws, bs


def head_problem(oracle, widths, S, seed):
    """Observations through the basis (relu_last) and S rows [log alpha_p, log beta, m] of the head."""
    Ws, bs = net(widths, seed)
    r = np.random.default_rng(seed + 1)
    Xo = r.random((N_OBS, DIMS))
    y = oracle.hartmann6(Xo)
    y = (y - y.mean()) / y.std()
    Z0 = oracle.mlp_features(Xo, Ws, bs, True)
    hyp = np.column_stack([np.log(0.1) + r.random(S) * np.log(100), np.log(10) + r.random(S) * np.log(100),
                           y.mean() + 0.2 * (r.random(S) - 0.5)])
    if S == 1:
        hyp[0, :2] = [0.0, math.log(1e2)]
    return Ws, bs, Z0, y, hyp


def one_device(L, blr, grid, Ws, bs, kind, tradeoff, bound, sign, fmin):
    """b7_dngo_score on one device over the whole grid -> (best, argmax, argmax_original, nan_count, scores)."""
    from bot7_b200 import models
    sc, am, amo, best, nn = models.dngo_score(blr, grid, Ws, bs, True, kind, tradeoff, bound, sign, fmin, want_scores=True)
    return best, am, amo, nn, sc


def same(multi, one):
    """Every output bit for bit: best (NaN == NaN), argmax, argmax_original, nan_count, every score."""
    bm, am, aom, nm, scm = multi
    b1, a1, ao1, n1, sc1 = one
    assert (am, aom, nm) == (a1, ao1, n1), ((am, aom, nm), (a1, ao1, n1))
    assert np.array_equal(np.array([bm]), np.array([b1]), equal_nan=True), (bm, b1)
    if scm is not None:
        assert np.array_equal(scm.view(np.int64), sc1.view(np.int64)), "scores differ in their bits"


def sobol_one_device(L, ctx, first, M):
    from bot7_b200 import grids
    h = C.c_void_p()
    L.check(L.lib().b7_sobol_generate(ctx.handle, DIMS, first, M, None, None, None, C.byref(h)), "b7_sobol_generate")
    return grids.DeviceGrid(h, ctx)


def compacted(removed, row):
    """1-based compacted index of the 0-based original row `row` given the removed original rows."""
    return row + 1 - sum(1 for t in removed if t < row)


CASES = [  # S, kind, bound, widths
    (1, 0, 0, [DIMS, 32, 50]),
    (5, 0, 0, [DIMS, 24, 40, 50]),
    (5, 1, 0, [DIMS, 32, 50]),
    (5, 1, 1, [DIMS, 24, 40, 50]),
    (1, 1, 1, [DIMS, 20, 33, 17]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("S,kind,bound,widths", CASES)
def test_dngo_score_multi_equals_one_device(ctx, comm, oracle, S, kind, bound, widths):
    """Sobol shards and host shards (with non-finite candidates) against b7_dngo_score over the whole grid; then the nominee
    and the first and last rows of a shard are removed and everything is compared again."""
    from bot7_b200 import _lib as L
    from bot7_b200 import grids, models
    Ws, bs, Z0, y, hyp = head_problem(oracle, widths, S, seed=S + 10 * kind + bound + len(widths))
    tradeoff, sign, fmin = (0.0, -1.0, float(y.min())) if kind == 0 else (1.5, -1.0 if bound == 0 else 1.0, 0.0)
    one = models.BLRFactors(Z0, y, hyp, ctx=ctx)
    blrs, info = comm.blr_fit(Z0, y, hyp)
    assert np.array_equal(info, one.info)
    M = 40009
    X = oracle.sobol_points(DIMS, M, 7)
    bad = np.arange(5, M, 4001)                      # non-finite and extreme candidates spread over every shard
    X[bad[0::4]] = np.nan
    X[bad[1::4], 2] = 1e308
    X[bad[2::4]] = 1e300
    X[bad[3::4], 0] = -np.inf
    try:
        for label in ("sobol", "host"):
            if label == "sobol":
                gs, g1 = comm.sobol_grid(DIMS, 1 + N_OBS, M), sobol_one_device(L, ctx, 1 + N_OBS, M)
            else:
                gs, g1 = comm.grid_from_host(X), grids.DeviceGrid.from_host(X, ctx)
            args = (kind, tradeoff, bound, sign, fmin)
            m = comm.dngo_score(blrs, gs, Ws, bs, True, *args, want_scores=True)
            o = one_device(L, one, g1, Ws, bs, *args)
            same(m, o)
            print(f"\n{label} S={S} kind={kind} bound={bound} layers={len(widths) - 1} G={comm.world}: argmax {m[1]} best {m[0]:.6g} "
                  f"nan {m[3]}")
            # fmin = NaN: every EI is NaN, no shard has a nominee
            if kind == 0:
                m_nan = comm.dngo_score(blrs, gs, Ws, bs, True, kind, tradeoff, bound, sign, float("nan"), want_scores=True)
                same(m_nan, one_device(L, one, g1, Ws, bs, kind, tradeoff, bound, sign, float("nan")))
                assert m_nan[1] == 0 and m_nan[3] == M and math.isnan(m_nan[0])
            # steal the nominee, then the first and the last row of the second shard (the first shard on one device)
            from bot7_b200 import parallel
            r0, cnt = parallel.shard_range(M, comm.world, min(1, comm.world - 1))
            removed = []
            for row in (m[2] - 1, r0, r0 + cnt - 1):
                if row in removed:
                    continue
                k = compacted(sorted(removed), row)
                row_m = comm.grid_remove(gs, k)
                row_1 = g1.remove(k)
                assert np.array_equal(row_m.view(np.int64), row_1.reshape(-1).view(np.int64))
                removed.append(row)
                m = comm.dngo_score(blrs, gs, Ws, bs, True, *args, want_scores=True)
                same(m, one_device(L, one, g1, Ws, bs, *args))
                assert m[2] - 1 not in removed and np.isnan(m[4][removed]).all()
            for g in gs:
                g.free()
            g1.free()
    finally:
        comm.free_blr(blrs)
        one.free()


@pytest.mark.gpu
def test_fewer_candidates_than_devices(ctx, comm, oracle):
    """M < G: some shards are empty; then every row of one shard is removed."""
    _need_two(comm)
    from bot7_b200 import _lib as L
    from bot7_b200 import grids, models, parallel
    Ws, bs, Z0, y, hyp = head_problem(oracle, [DIMS, 32, 50], 5, seed=41)
    one = models.BLRFactors(Z0, y, hyp, ctx=ctx)
    blrs, _ = comm.blr_fit(Z0, y, hyp)
    args = (0, 0.0, 0, -1.0, float(y.min()))
    try:
        for M in (1, comm.world - 1):
            X = oracle.sobol_points(DIMS, M, 3)
            gs, g1 = comm.grid_from_host(X), grids.DeviceGrid.from_host(X, ctx)
            assert sum(g.rows() for g in gs) == M and any(g.rows() == 0 for g in gs)
            m = comm.dngo_score(blrs, gs, Ws, bs, True, *args, want_scores=True)
            same(m, one_device(L, one, g1, Ws, bs, *args))
            assert m[1] >= 1
            for g in gs:
                g.free()
            g1.free()
        # a shard whose rows are all removed
        M = 3 * comm.world + 1
        X = oracle.sobol_points(DIMS, M, 5)
        gs, g1 = comm.grid_from_host(X), grids.DeviceGrid.from_host(X, ctx)
        r0, cnt = parallel.shard_range(M, comm.world, 1)
        removed = []
        for row in range(r0, r0 + cnt):
            k = compacted(removed, row)
            comm.grid_remove(gs, k)
            g1.remove(k)
            removed.append(row)
        m = comm.dngo_score(blrs, gs, Ws, bs, True, *args, want_scores=True)
        same(m, one_device(L, one, g1, Ws, bs, *args))
        assert not (r0 < m[2] <= r0 + cnt) and np.isnan(m[4][r0:r0 + cnt]).all()
        for g in gs:
            g.free()
        g1.free()
    finally:
        comm.free_blr(blrs)
        one.free()


@pytest.mark.gpu
def test_tie_across_a_shard_boundary_goes_to_the_smaller_index(ctx, comm, oracle):
    """The same candidate as the last row of one shard and the first row of the next, where it is the best of the grid: the
    nominee is the smaller original row, and after it is removed its twin on the other side."""
    _need_two(comm)
    from bot7_b200 import _lib as L
    from bot7_b200 import grids, models, parallel
    Ws, bs, Z0, y, hyp = head_problem(oracle, [DIMS, 32, 50], 5, seed=43)
    one = models.BLRFactors(Z0, y, hyp, ctx=ctx)
    blrs, _ = comm.blr_fit(Z0, y, hyp)
    args = (0, 0.0, 0, -1.0, float(y.min()))
    M = 20011
    X = oracle.sobol_points(DIMS, M, 9)
    try:
        g0 = grids.DeviceGrid.from_host(X, ctx)
        _, _, amo, _, _ = one_device(L, one, g0, Ws, bs, *args)
        g0.free()
        r0, _ = parallel.shard_range(M, comm.world, 1)
        X[r0 - 1] = X[r0] = X[amo - 1]                  # the best candidate on both sides of the boundary
        gs, g1 = comm.grid_from_host(X), grids.DeviceGrid.from_host(X, ctx)
        m = comm.dngo_score(blrs, gs, Ws, bs, True, *args, want_scores=True)
        same(m, one_device(L, one, g1, Ws, bs, *args))
        assert m[2] == min(r0, amo) and m[4][r0 - 1] == m[4][r0]
        comm.grid_remove(gs, m[1])
        g1.remove(m[1])
        m2 = comm.dngo_score(blrs, gs, Ws, bs, True, *args, want_scores=True)
        same(m2, one_device(L, one, g1, Ws, bs, *args))
        assert m2[0] == m[0] and m2[2] == sorted({r0, r0 + 1, amo} - {m[2]})[0]
        for g in gs:
            g.free()
        g1.free()
    finally:
        comm.free_blr(blrs)
        one.free()


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 5])
def test_blr_fit_multi_equals_one_device(ctx, comm, oracle, S):
    """Every handle predicts bit for bit like a one-device b7_blr_fit, and info is the same."""
    from bot7_b200 import _lib as L
    from bot7_b200 import models
    _, _, Z0, y, hyp = head_problem(oracle, [DIMS, 32, 50], S, seed=50 + S)
    hyp[-1, 0] = -40.0                                  # alpha_p = 4e-18: a row whose factorisation may fail, with its info
    one = models.BLRFactors(Z0, y, hyp, ctx=ctx)
    blrs, info = comm.blr_fit(Z0, y, hyp)
    try:
        assert np.array_equal(info, one.info)
        Z1 = np.random.default_rng(S).random((5000, Z0.shape[1])) * Z0.max(0)
        for s in range(S):
            m1, v1 = one.predict(s, Z1)
            for h in blrs:
                mm, vm = np.empty(len(Z1)), np.empty(len(Z1))
                L.check(L.lib().b7_blr_predict(h, s, L.dptr(Z1), len(Z1), L.dptr(mm), L.dptr(vm)), "b7_blr_predict")
                assert np.array_equal(mm.view(np.int64), m1.view(np.int64)) and np.array_equal(vm.view(np.int64), v1.view(np.int64))
        print(f"\nS={S} G={comm.world}: info {list(info)}")
    finally:
        comm.free_blr(blrs)
        one.free()


@pytest.mark.gpu
def test_bad_arguments_touch_nothing(ctx, comm, oracle):
    """A head of the wrong device, mismatched dims, a width of 64 and a B7_FIT_LOGML_ONLY head are refused before any device
    work: no launch, no score written, the grids unchanged."""
    from bot7_b200 import _lib as L
    Ws, bs, Z0, y, hyp = head_problem(oracle, [DIMS, 32, 50], 3, seed=61)
    M = 10007
    gs = comm.sobol_grid(DIMS, 1, M)
    blrs, _ = comm.blr_fit(Z0, y, hyp)
    W64, b64 = net([DIMS, 32, 64], 62)
    Z64 = oracle.mlp_features(np.random.default_rng(1).random((N_OBS, DIMS)), W64, b64, True)
    blrs64, _ = comm.blr_fit(Z64, y, hyp)

    def refused(handles, Ws_, bs_, code):
        before = [c.launch_count() for c in comm.ctxs]
        sizes = [g.size() for g in gs]
        n = len(Ws_)
        dims = (C.c_int * (n + 1))(*([Ws_[0].shape[1]] + [w.shape[0] for w in Ws_]))
        Wa, ba = [L.as_f64(w) for w in Ws_], [L.as_f64(b) for b in bs_]
        Wp = (C.POINTER(C.c_double) * n)(*[L.dptr(w) for w in Wa])
        bp = (C.POINTER(C.c_double) * n)(*[L.dptr(b) for b in ba])
        sc = np.full(M, 7.0)
        am, amo, best, nn = C.c_int64(-5), C.c_int64(-5), C.c_double(-5.0), C.c_int64(-5)
        rc = L.lib().b7_dngo_score_multi(comm.handle, (C.c_void_p * comm.n_local)(*handles), comm._handles(gs), n, dims, Wp, bp, 1, 0, 0.0,
                                         0, -1.0, 0.0, L.dptr(sc), C.byref(am), C.byref(amo), C.byref(best), C.byref(nn))
        msg = L.lib().b7_last_error().decode()
        assert rc == code, (rc, msg)
        assert (sc == 7.0).all() and (am.value, amo.value, best.value, nn.value) == (-5, -5, -5.0, -5)
        assert [c.launch_count() for c in comm.ctxs] == before and [g.size() for g in gs] == sizes
        return msg

    try:
        if comm.world >= 2:
            msg = refused(blrs[::-1], Ws, bs, -1)
            assert "does not belong" in msg
        refused(blrs, [Ws[0][:, :5]] + Ws[1:], bs, -1)                        # dims[0] = 5, the grid has 6
        refused(blrs, Ws[:1], bs[:1], -1)                                    # dims[n_layers] = 32, the head has 50
        msg = refused(blrs64, W64, b64, -1)                                  # D = 64: wider than the tile kernel takes
        assert "tile kernel" in msg
        L.check(L.lib().b7_blr_refit(blrs[-1], L.dptr(L.as_f64(hyp)), L.FIT_LOGML_ONLY, None, None), "b7_blr_refit")
        refused(blrs, Ws, bs, -3)
        L.check(L.lib().b7_blr_refit(blrs[-1], L.dptr(L.as_f64(hyp)), L.FIT_PREDICT, None, None), "b7_blr_refit")
        m = comm.dngo_score(blrs, gs, Ws, bs, True, 0, 0.0, 0, -1.0, float(y.min()))
        assert m[1] >= 1                                                      # the handles still score after the refusals
    finally:
        comm.free_blr(blrs)
        comm.free_blr(blrs64)
        for g in gs:
            g.free()


@pytest.mark.gpu
def test_dngo_multi_one_process_per_gpu(ctx):
    """b7_comm_init_rank under torchrun, one process per GPU (tools/dngo_multi_check.py): rank 0 compares the result of the
    sharded fit and score with its own one-device result."""
    if _n_gpus() < 2:
        pytest.skip("needs at least 2 GPUs")
    G = _n_gpus()
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={G}", "--master-addr", "127.0.0.1",
                          "--master-port", "29519", os.path.join(ROOT, "tools", "dngo_multi_check.py")], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "dngo_multi_check ok" in out.stdout


LUA_BOT = r"""
local out = {}
for _, n in ipairs{1, 2} do
  torch.manualSeed(SEED)
  local net = nn.Sequential():add(nn.Linear(6, 24)):add(nn.ReLU()):add(nn.Linear(24, 50)):add(nn.ReLU()):add(nn.Linear(50, 1))
  local model = bot7.models.dngo({network = net, basis = net:get(4), zDim = 50, update = {schedule = {batchsize = 32}}, predictor = PRED})
  local bot = bot7.bots.bayesopt(nil, nil, {bot = {nInitial = 0, nGPU = n}, candidates = XC, model = model,
                                            score = bot7.scores.expected_improvement(), observed = X0, responses = Y0, nTrials = 3})
  local first = bot:nominate()[1]
  local rows1 = model.blr_rows:clone()
  local second = bot:nominate()[1]
  out[n] = {first, second, rows1, model.blr_rows:clone(), net:get(1).weight, net:get(1).bias, net:get(3).weight, net:get(3).bias}
end
return out[1][1], out[1][2], out[2][1], out[2][2], out[1][3], out[1][4], out[2][3], out[2][4],
       out[1][5], out[1][6], out[1][7], out[1][8]
"""


@pytest.mark.gpu
@pytest.mark.parametrize("sampler", [None, "slice"])
def test_lua_dngo_bayesopt_on_two_gpus_equals_one(ctx, oracle, sampler):
    """bots.bayesopt with a DNGO model, nGPU = 1 and 2: the same two nominations, the first one the oracle's argmax, and with
    predictor.sampler = 'slice' the same sampled rows."""
    if _n_gpus() < 2:
        pytest.skip("needs at least 2 GPUs")
    from minilua.harness import GlueRuntime
    r = np.random.default_rng(7)
    Xo, Xc = r.random((300, DIMS)), oracle.sobol_points(DIMS, 20000, 11)
    y = oracle.hartmann6(Xo)
    y = (y - y.mean()) / y.std()
    rt = GlueRuntime(seed=5)
    rt.run("require('bot7_b200').install()")
    for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("XC", Xc)]:
        rt.set_global(name, rt.tensor(v))
    rt.set_global("SEED", 3)
    rt.run("PRED = {}" if sampler is None else "PRED = {sampler = 'slice', nSamples = 4}")
    res = rt.run(LUA_BOT)
    calls = list(rt.ffi.calls)
    rt.close()
    first1, second1, first2, second2 = res[0], res[1], res[2], res[3]
    rows = [res[k].a.copy() for k in range(4, 8)]
    W1, b1, W2, b2 = res[8].a, res[9].a, res[10].a, res[11].a
    assert (first1, second1) == (first2, second2) and first1 != second1
    assert np.array_equal(rows[0], rows[2]) and np.array_equal(rows[1], rows[3])
    assert calls.count("b7_blr_fit_multi") == 2 and calls.count("b7_dngo_score_multi") == 2
    Z0 = oracle.mlp_features(Xo, [W1, W2], [b1, b2], True)
    Z1 = oracle.mlp_features(Xc, [W1, W2], [b1, b2], True)
    per = []
    for h in rows[0]:
        m, v = oracle.blr_predict(oracle.blr_fit(Z0, y, h), Z1)
        per.append(oracle.ei_compute(m, v, float(y.min()), 0.0))
    _, idx, _ = oracle.argmax_first(oracle.mc_average(np.array(per)))
    print(f"\nsampler={sampler}: nominations {first1}, {second1} on 1 and 2 GPUs; oracle {idx}; rows {rows[0].shape[0]}")
    assert first1 == idx
    if sampler == "slice":
        assert rows[0].shape == (4, 3) and not np.array_equal(rows[0], rows[1])


def test_lua_dngo_nGPU_branch_with_the_stand_in_library(oracle):
    """CPU: bots.bayesopt with a DNGO model and nGPU = 2 drives b7_comm_init_all, b7_blr_fit_multi and b7_dngo_score_multi of
    the oracle-backed stand-in library, frees the per-device heads of every acquisition and nominates what nGPU = 1 does."""
    from fake_b7_dngo_multi import FakeB7DngoMulti
    from minilua.harness import GlueRuntime
    fake = FakeB7DngoMulti(oracle)
    rt = GlueRuntime(seed=5, lib_resolver=lambda name: fake)
    rt.run("require('bot7_b200').install()")
    r = np.random.default_rng(1)
    Xo, Xc = r.random((40, DIMS)), r.random((300, DIMS))
    y = np.sin(3 * Xo).sum(1)
    for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("XC", Xc)]:
        rt.set_global(name, rt.tensor(v))
    rt.set_global("SEED", 3)
    rt.run("PRED = {}")
    res = rt.run(LUA_BOT)
    rt.close()
    assert (res[0], res[1]) == (res[2], res[3]) and res[0] != res[1]
    calls = fake.calls
    assert calls.count("b7_comm_init_all") == 1 and calls.count("b7_grid_from_host_sharded") == 1
    assert calls.count("b7_blr_fit_multi") == 2 and calls.count("b7_dngo_score_multi") == 2 and calls.count("b7_grid_remove_sharded") == 2
    assert calls.count("b7_dngo_score") == 2
    assert [f[0] for f in fake.freed].count("blr") >= 2 * 2

"""b7_gp_slice_step -- one directed slice step of the GP hyper-parameter chain in one launch (N <= 128) -- against the paths the
samplers use today: its densities against b7_gp_refit(B7_FIT_LOGML_ONLY) + the host's prior bit for bit, the chains of
`device_step = True` against the speculative and the sequential samplers, the Lua twin against the Python twin, and the
refusals.  Every comparison is exact: the device step is meant to walk the same chain, not a close one."""
import copy
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

NS = [1, 2, 50, 100, 127, 128]
DS = [2, 6, 20]


def data(oracle, N, d, seed=3):
    r = np.random.default_rng(seed)
    X = oracle.sobol_points(d, N + 7)[7:]
    y = {2: oracle.braninhoo, 6: oracle.hartmann6}.get(d, oracle.ackley)(X)
    y = (y - y.mean()) / (y.std() if N > 1 else 1.0)
    return X, y, r


def rows(d, r):
    """Two ordinary rows, a row whose sigma_f^2 overflows (exp(800)), and one whose K is the all-ones matrix to the last bit
    (length scales e^30, noise e^-80): with two or more observations and noise its plain factorisation fails and the jitter
    retry takes over."""
    out = []
    for _ in range(2):
        h = np.empty(d + 3)
        h[:d] = np.log(0.1) + r.random(d) * (np.log(2) - np.log(0.1))
        h[d], h[d + 1], h[d + 2] = 0.5 * (r.random() - 0.5), 0.5 * np.log(1e-2), 0.1 * (r.random() - 0.5)
        out.append(h)
    h = out[0].copy()
    h[d] = 400.0
    out.append(h)
    h = out[1].copy()
    h[:d], h[d + 1] = 30.0, -40.0
    out.append(h)
    return out


def device_density(f, h, prior_std, prior_order):
    """The kernel's density at h: a step with no step-out (max_step 0), the bracket [-1, 0] (u_right = 0) and the shrink uniform
    1, so that its one shrink proposal is dx = 0, i.e. x1 = h, and the level log U = -inf, so that it is the last one."""
    H = h.size
    d_vec = np.zeros(H)
    d_vec[0] = 1.0
    res = f.slice_step(h, d_vec, -np.inf, np.zeros(H), np.ones(1), 1.0, 0.0, prior_std, prior_order)
    assert res is not None
    x1, used, evals, logp = res
    assert np.array_equal(x1[0], h) and used == 1 and evals == 4
    return logp


@pytest.fixture(scope="module")
def M(ctx):
    from bot7_b200 import _lib, models
    return models, _lib


@pytest.mark.gpu
@pytest.mark.parametrize("N", NS)
def test_density_is_the_refit_density_bit_for_bit(M, oracle, N):
    models, L = M
    seen = {"jitter": 0, "inf": 0}
    for d in DS:
        X, y, r = data(oracle, N, d, seed=N + d)
        for kernel in ("ardse", "matern52"):
            for noiseless in (False, True):
                hs = rows(d, r)
                f = models.GPFactors(X, y, hs[0], kernel, noiseless, L.FIT_LOGML_ONLY)
                ref = models.gp_regressor({"kernel": kernel, "noiseless": noiseless})
                for h in hs:
                    want = ref.log_density(h, X, y)                     # b7_gp_refit + guard + numpy's prior sum
                    got = device_density(f, h, 2.0, 1)
                    assert got == want, (N, d, kernel, noiseless, h, got, want)
                    assert math.copysign(1.0, got) == math.copysign(1.0, want)
                    # Torch7's order for the prior: the sequential sum
                    f2 = ref._density
                    lp = float(f2.logml[0]) if f2.info[0] == 0 and np.isfinite(f2.logml[0]) else -np.inf
                    s = 0.0
                    for v in (h / 2.0) ** 2:
                        s += float(v)
                    assert device_density(f, h, 2.0, 0) == lp - 0.5 * s
                    seen["jitter"] += int(f2.jitter[0] > 0 and np.isfinite(f2.jitter[0]))
                    seen["inf"] += int(want == -np.inf)
                f.free()
                ref._density.free()
    print(f"N={N}: {seen}")
    assert seen["inf"] >= 12                     # the overflow row in every case
    if N >= 2:
        assert seen["jitter"] >= 1               # the all-ones K needed the retry somewhere


def chain(models, X, y, cfg, steps, seed):
    m = models.gp_regressor(dict(cfg, nSamples=steps), rng=np.random.default_rng(seed))
    out = m.sample_hypers(X, y)
    return out, m.rng.bit_generator.state


@pytest.mark.gpu
@pytest.mark.parametrize("N,d", [(100, 2), (128, 6)])
def test_device_chain_is_the_speculative_and_the_sequential_chain(M, oracle, N, d):
    models, L = M
    X, y, _ = data(oracle, N, d)
    dev, s_dev = chain(models, X, y, {"device_step": True}, 20, 5)
    spec, s_spec = chain(models, X, y, {"speculative": True}, 20, 5)
    seq, s_seq = chain(models, X, y, {"speculative": False}, 20, 5)
    assert dev.shape == (20, d + 3) and len({tuple(r) for r in dev}) > 10      # the chain moves
    assert np.array_equal(dev, spec) and np.array_equal(dev, seq)
    assert s_dev == s_spec == s_seq


@pytest.mark.gpu
def test_device_chain_with_too_few_shrink_uniforms_leaves_the_generator_untouched(M, oracle):
    """Start every step with one shrink uniform: steps that need more are refused (None) and made again from the same draws;
    the generator does not move on a refused attempt and the chain is the sequential one."""
    from bot7_b200.samplers import slice_device
    models, L = M
    X, y, _ = data(oracle, 100, 2)
    m = models.gp_regressor({"device_step": True}, rng=np.random.default_rng(5))
    m.init(X, y)
    log = []

    def step(*a):
        before = copy.deepcopy(m.rng.bit_generator.state)
        res = m.device_step(X, y, *a)
        log.append((before, res is None, len(a[4])))
        return res
    sampler = slice_device()
    x = m.hyp.reshape(1, -1)
    out = []
    for _ in range(20):
        x = sampler(step, x, {"nSamples": 1}, None, rng=m.rng, k=1)
        out.append(x[0])
    refused = [i for i, (_, none, _) in enumerate(log) if none]
    assert refused, "no step needed a second shrink uniform"
    for i in refused:
        assert log[i + 1][0] == log[i][0] and log[i + 1][2] == 2 * log[i][2]
    seq, s_seq = chain(models, X, y, {"speculative": False}, 20, 5)
    assert np.array_equal(np.array(out), seq) and m.rng.bit_generator.state == s_seq


@pytest.mark.gpu
def test_refusals_come_before_device_work(M, oracle):
    import ctypes as C
    models, L = M
    ctx = L.Context.default()

    def call(f, K=4, width=1.0, order=1):
        H = f.d + 3
        x0, d_vec, ur, us, x1 = np.zeros(H), np.eye(H)[0], np.full(H, 0.5), np.full(max(K, 1), 0.5), np.empty(H)
        used, ev, lp = C.c_int(), C.c_int(), C.c_double()
        before = ctx.launch_count()
        rc = L.lib().b7_gp_slice_step(f.handle, L.dptr(x0), L.dptr(d_vec), -0.1, L.dptr(ur), L.dptr(us), K, width, 1e3, 2.0, order,
                                      L.dptr(x1), C.byref(used), C.byref(ev), C.byref(lp))
        return rc, ctx.launch_count() - before
    X, y, r = data(oracle, 129, 2)
    big = models.GPFactors(X, y, rows(2, r)[0], "ardse", False, L.FIT_LOGML_ONLY)
    assert call(big) == (L.ERR_ARG, 0)
    assert "129 observations" in L.lib().b7_last_error().decode()
    X, y, r = data(oracle, 128, 2)
    f = models.GPFactors(X, y, rows(2, r)[0], "ardse", False, L.FIT_LOGML_ONLY)
    for kw in ({"width": 0.0}, {"width": float("inf")}, {"width": float("nan")}, {"order": 2}, {"K": -1}):
        assert call(f, **kw) == (L.ERR_ARG, 0), kw
    with pytest.raises(ValueError, match="H = 5"):
        f.slice_step(np.zeros(6), np.eye(6)[0], -0.1, np.zeros(6), np.ones(4), 1.0, 1e3, 2.0, 1)
    # K = 0: the first shrink proposal has no uniform -> B7_ERR_STATE after the launch
    rc, launches = call(f, K=0)
    assert rc == L.ERR_STATE and launches == 1 and "ran out" in L.lib().b7_last_error().decode()
    # the N > 128 route of the model is the speculative sampler
    Xb, yb, _ = data(oracle, 129, 2)
    a, s_a = chain(models, Xb, yb, {"device_step": True}, 3, 2)
    b, s_b = chain(models, Xb, yb, {"speculative": True}, 3, 2)
    assert np.array_equal(a, b) and s_a == s_b
    big.free()
    f.free()


@pytest.mark.gpu
def test_lua_device_sampler_walks_the_python_twin_chain(M, oracle):
    """lua/bot7_b200/sampler_device.lua under tools/minilua with the real library: the chain of the Lua speculative sampler bit
    for bit, and the chain and the generator's final state of the Python twin (d = 2: H = 5 < 8 terms, where Torch7's sequential
    prior sum and numpy's pairwise one are the same sum).  The twins normalise the direction with norms of different rounding
    (the stand-in's Torch7 norm against numpy's), so their chains agree to that rounding, as the speculative twins do."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from minilua.harness import GlueRuntime
    models, L = M
    X, y, _ = data(oracle, 100, 2)

    def lua_chain(device):
        rt = GlueRuntime(seed=9)
        rt.run("require('bot7_b200').install()")
        rt.set_global("X0", rt.tensor(X))
        rt.set_global("Y0", rt.tensor(y.reshape(-1, 1)))
        rt.set_global("DEV", device)
        r = rt.run(r"""
local model = bot7.models.gp_regressor{kernel = 'ardse', nSamples = 8, device_step = DEV}
local draws = model:sample_hypers(X0, Y0)
return draws, model.hyp, torch.rand(1)[1]
""")
        out = (r[0].a.copy(), r[1].a.copy(), r[2], list(rt.ffi.calls))
        rt.close()
        return out
    dev, dev_state, dev_next, calls = lua_chain(True)
    assert calls.count("b7_gp_slice_step") >= 8 and calls.count("b7_gp_refit") == 0 and calls.count("b7_gp_fit") == 1
    spec, _, spec_next, _ = lua_chain(False)
    tw = models.gp_regressor({"kernel": "ardse", "nSamples": 8, "device_step": True}, rng=np.random.default_rng(9))
    ref = tw.sample_hypers(X, y)
    assert np.array_equal(dev, spec)
    assert dev.shape == (8, 5) and np.allclose(dev, ref, rtol=0.0, atol=1e-9) and np.allclose(dev_state[0], tw.hyp, rtol=0.0, atol=1e-9)
    assert dev_next == tw.rng.random() and dev_next == spec_next

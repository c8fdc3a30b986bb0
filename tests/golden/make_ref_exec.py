"""Golden vectors produced by EXECUTING the reference's own Lua (a read-only checkout named by BOT7_REFERENCE) under tools/minilua.

The image has no Lua runtime and the reference holds no test vectors, so until now the oracle was pinned by hand-traced known
answers only.  tools/minilua (a Lua 5.1 interpreter with a numpy-backed Torch7 tensor stand-in, written for this repository)
runs the reference modules UNMODIFIED -- grids/sobol.lua with utils/bits.lua (the doubles-based XOR), utils/math.lua (erf,
norm_pdf, norm_cdf, chol with its jitter policy), scores/expected_improvement.lua, scores/confidence_bound.lua,
utils/tensor.lua (steal / remove), benchmarks/{braninhoo,hartmann6,ackley}.lua -- and their outputs are stored here as
tests/golden/ref_exec.npz.  tests/test_ref_exec.py compares the oracle (CPU) and the CUDA path (GPU) with them.

What this is and is not: the control flow and every arithmetic operation are the reference's own source lines; the runtime
underneath is not LuaJIT + TH but Python floats + numpy (IEEE doubles, element-wise operations in storage order; `exp` is
numpy's, which may differ from glibc's in the last ulp).  torch.potrf is LAPACK dpotrf through scipy, as TH's is.

Run (with a checkout of the reference):  BOT7_REFERENCE=<bot7 checkout> python tests/golden/make_ref_exec.py
"""
import io
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from minilua import Interpreter, LuaError  # noqa: E402
from minilua import torch7  # noqa: E402
from minilua.interp import LuaTable  # noqa: E402

REF = os.environ.get("BOT7_REFERENCE", "")         # a checkout of the reference bot7 Lua source, if any
OUT = os.path.join(ROOT, "tests", "golden", "ref_exec.npz")


def reference_runtime(seed=0):
    """An interpreter with the reference's utils / grids / scores / benchmarks modules loaded from the reference tree."""
    if not os.path.isdir(REF):
        raise RuntimeError("set BOT7_REFERENCE to a checkout of the reference bot7 source")
    out = io.StringIO()
    I = Interpreter(stdout=out)
    T = torch7.install(I, seed)

    # torch.potrf(res, src, uplo): LAPACK dpotrf; raises like TH when a leading minor is not positive definite
    def t_potrf(*a):
        import scipy.linalg as sla
        if isinstance(a[0], torch7.Tensor) and len(a) >= 2 and isinstance(a[1], torch7.Tensor):
            res, src, uplo = a[0], a[1], (a[2] if len(a) > 2 else "U")
        else:
            res, src, uplo = None, a[0], (a[1] if len(a) > 1 else "U")
        c, info = sla.lapack.dpotrf(np.array(src.a, dtype=np.float64), lower=1 if uplo == "L" else 0, clean=1)
        if info > 0:
            raise LuaError("potrf: the leading minor of order %d is not positive definite" % info)
        if info < 0:
            raise LuaError("potrf: illegal value in argument %d" % -info)
        if res is None:
            return torch7.Tensor(np.ascontiguousarray(c), src.ttype)
        res.a = np.ascontiguousarray(c)
        return res
    T.set("potrf", t_potrf)

    I.run("bot7 = {grids = {}, scores = {}, utils = {}, benchmarks = {}}")
    loaded = I.G.get("package").get("loaded")
    bot7 = I.G.get("bot7")
    utils = bot7.get("utils")
    ut = I.run_file(os.path.join(REF, "utils", "tensor.lua"))[0]
    loaded.set("bot7.utils.tensor", ut)
    utils.set("tensor", ut)
    um = I.run_file(os.path.join(REF, "utils", "math.lua"))[0]
    utils.set("math", um)
    loaded.set("bot7.utils.math", um)
    loaded.set("bot7.utils", utils)
    ub = I.run_file(os.path.join(REF, "utils", "bits.lua"))[0]
    loaded.set("bot7.utils.bits", ub)
    utils.set("bits", ub)
    I.run_file(os.path.join(REF, "grids", "abstract.lua"))
    I.run_file(os.path.join(REF, "grids", "sobol.lua"))
    I.run_file(os.path.join(REF, "scores", "abstract.lua"))
    I.run_file(os.path.join(REF, "scores", "expected_improvement.lua"))
    I.run_file(os.path.join(REF, "scores", "confidence_bound.lua"))
    return I, out


def tensor(a):
    return torch7.Tensor(np.ascontiguousarray(np.array(a, dtype=np.float64)), "torch.DoubleTensor")


def generate():
    I, out = reference_runtime()
    G = {}
    rng = np.random.default_rng(20261019)

    # ---- grids/sobol.lua (+ utils/bits.lua): plain, skipped, rescaled, one-sided ----------------------------------------
    mins6, maxes6 = np.array([-1.0, 0.0, 2.0, -5.0, 0.5, 0.0]), np.array([1.0, 3.0, 4.0, 5.0, 0.75, 10.0])
    I.G.set("MINS", tensor(mins6.reshape(1, -1)))          # 1 x d, the shape bots/abstract.lua hands to the grid
    I.G.set("MAXES", tensor(maxes6.reshape(1, -1)))
    cases = {
        "sobol_d2_n200": "return bot7.grids.sobol{size = 200, dims = 2}:generate()",
        "sobol_d6_n256": "return bot7.grids.sobol{size = 256, dims = 6}:generate()",
        "sobol_d20_n48": "return bot7.grids.sobol{size = 48, dims = 20}:generate()",
        "sobol_d39_n24": "return bot7.grids.sobol{size = 24, dims = 39}:generate()",
        "sobol_d6_n40_skip37": "return bot7.grids.sobol{size = 40, dims = 6, skip = 37}:generate()",
        "sobol_d6_n64_scaled": "return bot7.grids.sobol{size = 64, dims = 6, mins = MINS, maxes = MAXES}:generate()",
        "sobol_d6_n64_mins": "return bot7.grids.sobol{size = 64, dims = 6, mins = MINS}:generate()",
        "sobol_d6_n64_maxes": "return bot7.grids.sobol{size = 64, dims = 6, maxes = MAXES}:generate()",
        # the generator object keeps state (seed, lastq): a second call on the same object, and __call__
        "sobol_d3_two_calls": "local g = bot7.grids.sobol{size = 16, dims = 3}; local a = g:generate(); local b = g(); return torch.cat(a, b, 1)",
    }
    if os.environ.get("REF_EXEC_FAST"):                  # debugging aid: one small Sobol case only
        cases = {"sobol_d3_two_calls": cases["sobol_d3_two_calls"]}
    for name, src in cases.items():
        G[name] = I.run(src, "=" + name)[0].a.copy()
    G["sobol_mins6"], G["sobol_maxes6"] = mins6, maxes6
    # create_bank's initial direction numbers, and the bank after the first point was generated (recurrence filled in and every
    # column scaled by 2^(maxcol - j): the integers the CUDA path keeps in its host table)
    if not os.environ.get("REF_EXEC_FAST"):              # (the 39-dimensional recurrence is ~1000 emulated XORs: a minute)
        r = I.run("local g = bot7.grids.sobol{size = 2, dims = 39}; local b0 = g.bank:clone(); g:generate(); return b0, g.bank, g.recipd")
        G["sobol_bank_initial"], G["sobol_bank_scaled"], G["sobol_recipd"] = r[0].a.copy(), r[1].a.copy(), np.array([r[2]])
    G["xor_pairs"] = np.array([[5, 3], [1023, 512], [2 ** 31 - 1, 2 ** 30 + 12345], [0, 77], [123456789, 987654321]], dtype=np.float64)
    I.G.set("XP", tensor(G["xor_pairs"]))
    G["xor_out"] = I.run("local u = require('bot7.utils.bits'); local o = torch.Tensor(XP:size(1)); "
                         "for i = 1, XP:size(1) do o[i] = u.bitwise_xor(XP[i][1], XP[i][2]) end; return o")[0].a.copy()

    # ---- utils/math.lua: erf (A&S 7.1.26), norm_pdf, norm_cdf -----------------------------------------------------------
    x = np.concatenate([np.linspace(-6.0, 6.0, 97), [0.0, -0.0, 0.5, -0.5, 1e-9, -1e-9, 37.0, -37.0], rng.standard_normal(64) * 2])
    I.G.set("X", tensor(x))
    G["math_x"] = x
    G["math_erf"] = I.run("return bot7.utils.math.erf(X)")[0].a.copy()
    G["math_pdf"] = I.run("return bot7.utils.math.norm_pdf(X)")[0].a.copy()
    G["math_cdf"] = I.run("return bot7.utils.math.norm_cdf(X)")[0].a.copy()

    # ---- scores: EI.compute / conf_bound.compute on M x 1 moments -------------------------------------------------------
    M = 512
    mean, var = rng.standard_normal(M), np.abs(rng.standard_normal(M)) * 0.4
    var[:4] = 0.0                                       # sigma = 0 rows
    mean[2] = -0.25                                     # ... one of them with zero improvement at fmin = -0.25 (0 / 0)
    G["score_mean"], G["score_var"], G["score_fmin"] = mean, var, np.array([-0.25])
    I.G.set("MEAN", tensor(mean.reshape(-1, 1)))
    I.G.set("VAR", tensor(var.reshape(-1, 1)))
    I.G.set("FMIN", tensor([[-0.25]]))
    # EI.compute reads an undefined GLOBAL `config` (scores/expected_improvement.lua:70; its 4th parameter is shadowed): the global
    # is defined here with the tradeoff under test, which is the value the function then uses
    for name, trade in [("ei_t0", 0.0), ("ei_t01", 0.1)]:
        I.G.set("config", LuaTable({"tradeoff": trade}))
        G["score_" + name] = I.run("return bot7.scores.expected_improvement.compute(MEAN, VAR, FMIN, nil)")[0].a.copy().reshape(-1)
    I.G.set("config", None)
    G["score_ei_without_global"] = np.array([0.0 if I.run("return (pcall(bot7.scores.expected_improvement.compute, MEAN, VAR, FMIN, 0.0))")[0] else 1.0])
    for name, cfg in [("lcb", "{tradeoff = 1.0, bound = 'lower', sign = -1.0}"), ("ucb", "{tradeoff = 2.0, bound = 'Upper', sign = 1.0}"),
                      ("lcb_pos", "{tradeoff = 0.5, bound = 'lower', sign = 1.0}")]:
        G["score_" + name] = I.run("return bot7.scores.confidence_bound.compute(MEAN, VAR, %s)" % cfg)[0].a.copy().reshape(-1)

    # ---- bots/bayesopt.lua eval + nominate (:56-99): priming draw, S draws, sequential sum, one divide, score:max(1) -------
    # The real bot class and the real EI / bound objects run; the model is a stand-in whose predict returns prescribed moments
    # per draw (the GP itself lives in the absent gp rock), and the parent class bots/abstract.lua is replaced by a stub that
    # only carries the fields eval / nominate read.
    S, Mb = 5, 300
    means, vars_ = rng.standard_normal((S, Mb)) * 0.5, np.abs(rng.standard_normal((S, Mb))) * 0.2 + 1e-3
    means[:, 17] = means[:, 4]                          # two candidates with identical moments in every draw: a tie for the argmax
    vars_[:, 17] = vars_[:, 4]
    means[:, 4] -= 3.0                                  # ... made the best ones
    means[:, 17] -= 3.0
    yobs = rng.standard_normal((40, 1))
    G["bo_means"], G["bo_vars"], G["bo_yobs"] = means, vars_, yobs
    I.G.set("MEANS", tensor(means))
    I.G.set("VARS", tensor(vars_))
    I.G.set("YOBS", tensor(yobs))
    loaded = I.G.get("package").get("loaded")
    loaded.set("bot7.models", LuaTable())
    loaded.set("bot7.scores", I.G.get("bot7").get("scores"))
    I.run("bot7.bots = {}; local a = torch.class('bot7.bots.abstract'); function a:__init() end; function a:configure(c) return c or {} end")
    I.run_file(os.path.join(REF, "bots", "bayesopt.lua"))
    BO = r"""
local S = MEANS:size(1)
local order = {}
local fake = {k = 0}
function fake:class() return 'gp.models.gp_regressor' end
function fake:sample_hypers(X, Y, a, b, single) self.k = self.k + 1; local s = (self.k - 1) % S + 1; order[#order + 1] = s; return torch.Tensor{{s}} end
function fake:parse_hypers(h) return h end
function fake:predict(X0, Y0, X1, hyp, req) local s = hyp[1][1]; return {mean = MEANS[s]:clone():view(-1, 1), var = VARS[s]:clone():view(-1, 1)} end
local bot = bot7.bots.bayesopt(nil, nil, {bot = {nSamples = S, nInitial = 0}}, {model = fake, score = SCORE})
bot.observed, bot.responses, bot.candidates, bot.nTrials = torch.zeros(YOBS:size(1), 2), YOBS, torch.zeros(MEANS:size(2), 2), 3
local score = bot:eval()
fake.k = 0
local idx = bot:nominate()
return score, idx, torch.Tensor(order)
"""
    for name, ctor, trade in [("ei", "bot7.scores.expected_improvement{tradeoff = 0.0}", 0.0),
                              ("ucb", "bot7.scores.confidence_bound{tradeoff = 2.0, bound = 'upper', sign = 1.0}", None)]:
        I.G.set("config", LuaTable({"tradeoff": trade}) if trade is not None else None)     # EI.compute's global (see above)
        I.G.set("SCORE", I.run("return " + ctor)[0])
        r = I.run(BO, "=bayesopt " + name)
        G["bo_%s_score" % name], G["bo_%s_idx" % name], G["bo_%s_order" % name] = r[0].a.copy(), r[1].a.copy(), r[2].a.copy()
    I.G.set("config", None)

    # ---- utils.math.chol: plain success, jitter success, give-up ---------------------------------------------------------
    A = rng.standard_normal((6, 6))
    spd = A @ A.T + 6 * np.eye(6)
    v = rng.standard_normal((6, 1))
    semi = v @ v.T                                       # rank one: needs jitter
    neg = -np.eye(4)                                     # never succeeds: eps passes ||src||_F = 2 and chol(I) is returned
    for name, mat in [("spd", spd), ("semi", semi), ("neg", neg)]:
        I.G.set("K", tensor(mat))
        r = I.run("local msgs = {}; local p = print; print = function(s) msgs[#msgs + 1] = s end; "
                  "local L = bot7.utils.math.chol(K, 'L', {verbose = 1}); print = p; return L, #msgs, msgs[#msgs]")
        G["chol_" + name + "_in"] = mat
        G["chol_" + name + "_L"] = np.tril(r[0].a)
        msg = r[2] or ""
        jit = 0.0
        if "jitter of" in msg:
            jit = float(msg.split("jitter of")[1])
        elif "returning chol(I)" in msg:
            jit = np.inf
        G["chol_" + name + "_jitter_printed"] = np.array([jit])
        G["chol_" + name + "_iterations"] = np.array([max(int(r[1]) - 1, 0)])    # one 'Iteration %d' line per pass + the final warning

    # ---- utils.tensor.steal / remove: the grid compaction of bots/abstract.lua:118 ---------------------------------------
    src = np.arange(1, 31, dtype=np.float64).reshape(10, 3)
    I.G.set("SRC", tensor(src))
    r = I.run("local U = bot7.utils.tensor; local res, rest = U.steal(torch.Tensor{{0, 0, 0}}, SRC, torch.LongTensor{4}); "
              "local res2, rest2 = U.steal(res, rest, torch.LongTensor{4}); "
              "local res3, rest3 = U.steal(res2, rest2, torch.LongTensor{1, 8}); return res3, rest3, U.remove(SRC, torch.LongTensor{10, 1, 5})")
    G["steal_src"], G["steal_res"], G["steal_rest"], G["remove_out"] = src, r[0].a.copy(), r[1].a.copy(), r[2].a.copy()

    # ---- benchmarks: the three objectives used to synthesise observations -------------------------------------------------
    loaded = I.G.get("package").get("loaded")
    I.run_file(os.path.join(REF, "benchmarks", "abstract.lua")) if os.path.exists(os.path.join(REF, "benchmarks", "abstract.lua")) else None
    pts = {"braninhoo": rng.random((32, 2)), "hartmann6": rng.random((32, 6)), "ackley": rng.random((32, 5))}
    for name, X in pts.items():
        path = os.path.join(REF, "benchmarks", name + ".lua")
        try:
            f = I.run_file(path)
            f = f[0] if f else I.G.get("bot7").get("benchmarks").get(name)
            I.G.set("F", f)
            I.G.set("XB", tensor(X))
            vals = I.run("local o = torch.Tensor(XB:size(1)); for i = 1, XB:size(1) do local v = F(XB[{{i}, {}}]); "
                         "o[i] = torch.isTensor(v) and v:view(-1)[1] or v end; return o")[0].a.copy()
            G["bench_" + name + "_x"], G["bench_" + name + "_y"] = X, vals
        except LuaError as e:                               # recorded, not fatal: the objectives only synthesise test data
            print("benchmark %s not executed: %s" % (name, e))
    del loaded
    return G, out.getvalue()


if __name__ == "__main__":
    if not os.path.isdir(REF):
        sys.exit("set BOT7_REFERENCE to a checkout of the reference bot7 source: nothing to execute")
    G, printed = generate()
    if os.environ.get("REF_EXEC_FAST"):
        OUT = "/tmp/ref_exec_fast.npz"                   # the debugging subset never replaces the committed file
    np.savez_compressed(OUT, **G)
    print("wrote %s: %d arrays, %d bytes" % (OUT, len(G), os.path.getsize(OUT)))
    for k in sorted(G):
        print("  %-28s %s" % (k, G[k].shape))

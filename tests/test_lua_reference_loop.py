"""The reference's OWN control plane driving the LuaJIT glue: init.lua, hyperparam.lua, bots/abstract.lua, bots/bayesopt.lua,
samplers/slice.lua, grids/abstract.lua, scores/abstract.lua, utils/*.lua, benchmarks/*.lua and examples/run_benchmark.lua are
loaded UNMODIFIED from the read-only reference tree under tools/minilua, `require('bot7_b200').install()` swaps in the glue
classes, and whole Bayesian-optimisation experiments run -- BASELINE.json's config 1 (examples/run_benchmark.lua: Branin-Hoo,
bayesopt EI, GP ARD-SE, Sobol candidates) through the reference's own example script.

This needs a checkout of the reference (named by BOT7_REFERENCE) and runs without a GPU; the library has no CPU path.  So the
glue's `ffi.load` is answered by tests/fake_b7_lib.py, an oracle-backed object with the C ABI's signatures.  What is under test
is therefore the PROTOCOL between the reference's classes, the glue and the C ABI -- constructor chains, which object owns which
field, compacted vs original numbering across `utils.tensor.steal` and `b7_grid_remove`, handle lifetimes -- in the one setting
where the real reference classes are the callers.  (The glue against the REAL library is tests/test_lua_exec.py on the GPU.)
Absent dependencies are stubbed and named: penlight's tablex (deepcopy / find), the `gp` rock (an empty `gp.models` table, which is
exactly what install() fills), nnTools (DNGO's trainer: not on this path), torch.CmdLine.
"""
import io
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("BOT7_REFERENCE", "")         # a checkout of the reference bot7 Lua source, if any
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from minilua import Interpreter, LuaError  # noqa: E402,F401
from minilua import ffi as ffi_mod  # noqa: E402
from minilua import torch7  # noqa: E402
from minilua.harness import LUA_DIR  # noqa: E402
from minilua.interp import LuaTable  # noqa: E402

pytestmark = pytest.mark.skipif(not os.path.isdir(REF), reason="bot7 reference source not found (set BOT7_REFERENCE to a checkout)")

CMDLINE = r"""
local Cmd = torch.class('torch.CmdLine')
function Cmd:__init() self.opts = {} end
function Cmd:text() end
function Cmd:option(name, default, help) self.opts[#self.opts + 1] = {name = name:gsub('^%-+', ''), default = default} end
function Cmd:parse(arg)
  local o = {}
  for _, op in ipairs(self.opts) do o[op.name] = op.default end
  local i = 1
  while i <= #arg do
    local key = arg[i]:gsub('^%-+', '')
    local def = o[key]
    assert(def ~= nil, 'unknown option ' .. arg[i])
    local v = arg[i + 1]
    if type(def) == 'number' then v = tonumber(v) elseif type(def) == 'boolean' then v = (v == 'true') end
    o[key] = v
    i = i + 2
  end
  return o
end
"""


# nnTools (the network builder / trainer of the reference's DNGO) is out of scope and needs nn's backward pass, optim and
# torch.Timer: stand-ins with the call signatures models/dngo.lua uses.  The "trained" network is a fixed random Linear / ReLU
# stack; training is a forward pass (so that every module has an output, which dngo:init reads to find the basis layer).
NNTOOLS = r"""
local function builder(config, data)
  local d = data.xr:size(2)
  return nn.Sequential():add(nn.Linear(d, 12)):add(nn.ReLU()):add(nn.Linear(12, 20)):add(nn.ReLU()):add(nn.Linear(20, 1))
end
local trained = 0
local function trainer(network, data, config, cache)
  network:forward(data.xr)
  cache.state.dfdx = cache.state.dfdx or torch.zeros(1)
  trained = trained + 1
  return {loss = 0, err = 0}
end
package.loaded['bot7.nnTools.builder']   = builder
package.loaded['bot7.nnTools.trainer']   = trainer
package.loaded['bot7.nnTools.evaluator'] = function() return 0, 0 end
package.loaded['bot7.nnTools.buffers']   = function(config, data) return {} end
function nnTools_trained() return trained end
nn.MSECriterion = function() return {} end
optim = package.loaded['optim']        -- models/dngo.lua:34 reads the global
optim.sgd = function() end
-- gp.models.bayes_linear: constructed by dngo:init (models/dngo.lua:74) and never used by the override
do
  gp = gp or {models = {}}
  local B = torch.class('gp.models.bayes_linear')
  function B:__init(...) end
  function B:init(X, Y) end
  package.loaded['gp.models'].bayes_linear = B
end
"""


class Runtime:
    def __init__(self, oracle, seed=7):
        from fake_b7_lib import FakeB7
        self.out = io.StringIO()
        self.I = I = Interpreter(search_path=[("bot7", REF), ("bot7_b200", LUA_DIR)], stdout=self.out)
        torch7.install(I, seed)
        loaded = I.G.get("package").get("loaded")

        def deepcopy(t):                                   # penlight tablex.deepcopy: tables recursively, metatables kept
            if isinstance(t, LuaTable):
                n = LuaTable()
                n.meta = t.meta
                for k, v in t.hash.items():
                    n.hash[k] = deepcopy(v)
                return n
            return t

        def find(t, v, start=1):
            for k in range(int(start), t.length() + 1):
                if I.eq(t.get(k), v):
                    return k
            return [None]
        tablex = LuaTable()
        tablex.set("deepcopy", deepcopy)
        tablex.set("find", find)
        loaded.set("pl.tablex", tablex)
        loaded.set("gp.models", LuaTable())                 # the absent rock: an empty module table
        for n in ("optim", "xlua"):
            loaded.set(n, LuaTable())
        loaded.set("nn", I.G.get("nn"))
        I.run(CMDLINE, "=torch.CmdLine")
        I.run(NNTOOLS, "=nnTools stand-ins")
        self.fake = FakeB7(oracle)
        self.ffi = ffi_mod.Runtime(I, lambda name: self.fake)
        self.ffi.install()
        I.run("require 'bot7'; require('bot7_b200').install()", "=setup")

    def close(self):
        self.ffi.close()


@pytest.fixture()
def rt(oracle):
    r = Runtime(oracle)
    yield r
    r.close()


def test_reference_example_script_runs_config_1_through_the_glue(rt, oracle):
    """examples/run_benchmark.lua, unmodified, with its own command line: Branin-Hoo, bayesopt + EI, noiseless GP, Sobol grid."""
    I, fake = rt.I, rt.fake
    args = LuaTable({k + 1: v for k, v in enumerate(["-budget", "9", "-grid_size", "300", "-nInitial", "3", "-verbose", "1", "-benchmark", "braninhoo"])})
    I.G.set("arg", args)
    I.run_file(os.path.join(REF, "examples", "run_benchmark.lua"))
    text = rt.out.getvalue()
    assert "Trial: 9 of 9" in text and "Best response" in text and "Error" not in text
    calls = fake.calls
    # one Sobol grid by the glue's generator (host tensor, as the reference's Grids[...](config)() returns it) + its device copy
    assert calls.count("b7_sobol_generate") == 1 and calls.count("b7_grid_from_host") == 1
    assert calls.count("b7_grid_remove") == 9                           # every nomination leaves the device grid too
    assert calls.count("b7_acq_score") == 6                             # trials 4 .. 9 (nTrials <= nInitial picks at random)
    assert calls.count("b7_gp_refit") > 50                              # the reference's slice sampler evaluating the glue's density
    # everything that was created has been released once the bot is gone, the context last
    import gc
    del I
    rt.I.G.set("bot", None)
    gc.collect()
    rt.close()
    kinds = [f[0] for f in fake.freed]
    assert kinds[-1] == "ctx" and fake.freed[-1][2] == 0, fake.freed[-3:]
    assert kinds.count("grid") == 1 and kinds.count("gp") >= 6


def test_reference_bot_and_glue_stay_consistent_trial_by_trial(rt, oracle):
    """The same experiment driven trial by trial: after every run_trial the host candidates (compacted by the reference's
    utils.tensor.steal) and the device grid (compacted by b7_grid_remove) hold the same rows in the same order, the nominee is
    the row the acquisition selected, and the model's chain state follows bots/abstract.lua:148 / bots/bayesopt.lua:68-75."""
    I, fake = rt.I, rt.fake
    seen = []

    def check(bot):
        cand = I.index(bot, "candidates").a
        grids = [o for o in fake.handles.values() if o["kind"] == "grid"]
        assert len(grids) == 1
        dev = grids[0]["X"][grids[0]["live"]]
        assert np.array_equal(cand, dev)
        obs, resp = I.index(bot, "observed"), I.index(bot, "responses")
        seen.append((None if obs is None else obs.a.copy(), None if resp is None else resp.a.copy(), int(I.index(bot, "nTrials"))))
        return True
    I.G.set("CHECK", check)
    r = I.run(r"""
local benchmarks = require('bot7.benchmarks')
local hypers = {bot7.hyperparam('x1', 0, 1), bot7.hyperparam('x2', 0, 1)}
local expt = {xDim = 2, yDim = 1,
              bot = {type = 'bo', nInitial = 2, budget = 7, nSamples = 3, verbose = 0},
              model = {noiseless = true, nSamples = 2, speculative = false},   -- the reference's own slice sampler over the glue's density
              grid = {type = 'sobol', size = 200},
              score = {type = 'confidence_bound', tradeoff = 1.5}}
local bot = bot7.bots.bayesopt(benchmarks.braninhoo, hypers, expt)
assert(torch.type(bot) == 'bot7_b200.bots.bayesopt' and torch.type(bot.model) == 'bot7_b200.models.gp_regressor')
assert(torch.type(bot.score) == 'bot7_b200.scores.confidence_bound' and bot.score.config.tradeoff == 1.5)
CHECK(bot)
for t = 1, 7 do
  bot:run_trial()
  CHECK(bot)
end
-- the reference's own bot:eval (bots/bayesopt.lua:56-82, not overridden by the glue) with the glue's model and score objects:
-- per draw model:predict + score.compute through the library, summed and averaged by the reference code
local sc = bot:eval()
assert(sc:dim() == 1 and sc:size(1) == bot.candidates:size(1) and sc:eq(sc):all())
return bot.observed, bot.responses, bot.model.hyp, bot.candidates:size(1)
""", "=trial loop")
    obs, resp, hyp, n_left = r[0].a, r[1].a, r[2].a, r[3]
    assert obs.shape == (7, 2) and resp.shape == (7, 1) and n_left == 193
    assert np.allclose(resp[:, 0], oracle.braninhoo(obs), rtol=1e-14, atol=0.0)
    assert hyp.shape == (1, 5) and np.isfinite(hyp).all()
    # all observed points are distinct rows of the original Sobol grid, i.e. nothing was nominated twice
    grid = oracle.sobol_points(2, 200)
    rows = [int(np.flatnonzero((grid == x).all(1))[0]) for x in obs]
    assert len(set(rows)) == 7
    assert [s[2] for s in seen] == list(range(0, 8))
    assert fake.calls.count("b7_acq_score") == 5 and fake.calls.count("b7_grid_remove") == 7
    assert fake.calls.count("b7_gp_predict") == 3 and fake.calls.count("b7_score_moments") == 3      # bot:eval, nSamples = 3
    assert fake.calls.count("b7_gp_refit") > 100                      # one device call per density evaluation of samplers/slice.lua


def test_reference_dngo_class_and_bot_drive_the_glue_override(rt, oracle):
    """models/dngo.lua (reference, unmodified) is the parent of the glue's DNGO class: its __init / init build the network, find
    the basis layer and set config.zDim; the override's predict / acquire hand the basis stack and the BLR head to the library;
    bots/bayesopt.lua reaches it through model:class() == 'bot7.models.dngo' (:65).  nnTools is a stand-in (see NNTOOLS)."""
    I, fake = rt.I, rt.fake
    g = np.random.default_rng(1)
    X0, X1 = g.random((30, 2)), g.random((400, 2))
    y0 = oracle.braninhoo(X0)
    y0 = (y0 - y0.mean()) / y0.std()
    for name, v in (("X0", X0), ("Y0", y0.reshape(-1, 1)), ("X1", X1)):
        I.G.set(name, torch7.Tensor(np.ascontiguousarray(v), "torch.DoubleTensor"))
    r = I.run(r"""
local cfg = {model = {}, update = {schedule = {batchsize = 8}}, predictor = {}}
local model = bot7.models.dngo(cfg, nil, X0, Y0)
assert(torch.type(model) == 'bot7_b200.models.dngo' and model:class() == 'bot7.models.dngo')
assert(model.config.zDim == 20 and torch.type(model.basis) == 'nn.ReLU' and model.basis == model.network:get(4))
local before = nnTools_trained()
local p = model:predict(X0, Y0, X1, nil, {mean = true, var = true})
local net = model.network
return p.mean, p.var, nnTools_trained() - before, net:get(1).weight, net:get(1).bias, net:get(3).weight, net:get(3).bias
""", "=dngo predict")
    W1, b1, W2, b2 = (t.a for t in r[3:7])
    Z0 = oracle.mlp_features(X0, [W1, W2], [b1, b2], True)
    Z1 = oracle.mlp_features(X1, [W1, W2], [b1, b2], True)
    fit = oracle.blr_fit(Z0, y0, [0.0, np.log(1e2), float(y0.mean())])
    mr, vr = oracle.blr_predict(fit, Z1)
    assert r[2] == 1                                                   # the parent's network update ran once (models/dngo.lua:126-153)
    assert np.allclose(r[0].a[:, 0], mr, rtol=1e-10, atol=1e-12) and np.allclose(r[1].a[:, 0], vr, rtol=1e-10, atol=1e-12)
    # the host basis went through the reference's own minibatch loop (batchsize 8 over 30 rows) and the network's forward
    assert fake.calls.count("b7_blr_fit") == 1 and fake.calls.count("b7_mlp_features") == 1 and fake.calls.count("b7_blr_predict") == 1

    # a whole experiment with the DNGO model under the reference's bot
    r = I.run(r"""
local benchmarks = require('bot7.benchmarks')
local hypers = {bot7.hyperparam('x1', 0, 1), bot7.hyperparam('x2', 0, 1)}
local expt = {xDim = 2, yDim = 1, bot = {type = 'bo', nInitial = 3, budget = 7, verbose = 0},
              model = {type = 'dngo', model = {}, update = {schedule = {batchsize = 4}}, predictor = {}},
              grid = {type = 'sobol', size = 150}, score = {type = 'expected_improvement'}}
local bot = bot7.bots.bayesopt(benchmarks.braninhoo, hypers, expt)
assert(torch.type(bot.model) == 'bot7_b200.models.dngo')
for t = 1, 7 do bot:run_trial() end
return bot.observed, bot.responses, bot.candidates, bot
""", "=dngo experiment")
    obs, resp, cand = r[0].a, r[1].a, r[2].a
    assert obs.shape == (7, 2) and cand.shape == (143, 2) and np.allclose(resp[:, 0], oracle.braninhoo(obs), rtol=1e-14, atol=0.0)
    assert fake.calls.count("b7_dngo_score") == 4                       # trials 4 .. 7: one fused pass over the device grid each
    grids = [o for o in fake.handles.values() if o["kind"] == "grid" and o["X"].shape == (150, 2)]
    assert len(grids) == 1 and np.array_equal(cand, grids[0]["X"][grids[0]["live"]])


@pytest.mark.parametrize("extra, acq_calls", [(["-score", "ucb"], 4), (["-bot", "rs"], 0), (["-benchmark", "hartmann6", "-noisy", "true"], 4)])
def test_reference_example_script_variants(rt, extra, acq_calls):
    """The same script with its other switches: the confidence bound, the random-search bot (which the glue leaves alone apart
    from the Sobol grid it draws from), a 6-dimensional noisy objective."""
    I, fake = rt.I, rt.fake
    argv = ["-budget", "6", "-grid_size", "120", "-nInitial", "2", "-verbose", "0"] + extra
    I.G.set("arg", LuaTable({k + 1: v for k, v in enumerate(argv)}))
    I.run_file(os.path.join(REF, "examples", "run_benchmark.lua"))
    assert "Error" not in rt.out.getvalue()
    assert fake.calls.count("b7_sobol_generate") == 1 and fake.calls.count("b7_acq_score") == acq_calls
    assert fake.calls.count("b7_grid_remove") == (6 if acq_calls else 0)


def test_reference_bot_with_nGPU_2_uses_the_multi_gpu_block(rt, oracle):
    """config.bot.nGPU = 2 under the reference's bot: the glue creates one communicator, shards the host candidates over it, fits
    through b7_gp_fit_sharded, scores through b7_acq_score_multi and removes through b7_grid_remove_sharded; the per-device factor
    handles of every acquisition are freed, and the nominations equal those of the one-GPU bot on the same generator."""
    I, fake = rt.I, rt.fake
    LOOP = r"""
local benchmarks = require('bot7.benchmarks')
local hypers = {bot7.hyperparam('x1', 0, 1), bot7.hyperparam('x2', 0, 1)}
local out = {}
for _, n in ipairs{1, 2} do
  torch.manualSeed(5)
  local expt = {xDim = 2, yDim = 1, bot = {type = 'bo', nInitial = 2, budget = 6, nSamples = 2, verbose = 0, nGPU = n},
                model = {noiseless = true}, grid = {type = 'sobol', size = 160}, score = {type = 'expected_improvement'}}
  local bot = bot7.bots.bayesopt(benchmarks.braninhoo, hypers, expt)
  for t = 1, 6 do bot:run_trial() end
  out[n] = bot.observed:clone()
  bot = nil
  collectgarbage()
end
return out[1], out[2]
"""
    r = I.run(LOOP, "=nGPU loop")
    assert np.array_equal(r[0].a, r[1].a) and r[0].a.shape == (6, 2)
    calls = fake.calls
    assert calls.count("b7_comm_init_all") == 1 and calls.count("b7_grid_from_host_sharded") == 1
    assert calls.count("b7_gp_fit_sharded") == 4 and calls.count("b7_acq_score_multi") == 4 and calls.count("b7_grid_remove_sharded") == 6
    import gc
    gc.collect()
    kinds = [f[0] for f in fake.freed]
    assert kinds.count("gp") >= 8 + 4                                  # 2 per sharded acquisition, 1 per one-GPU acquisition (+ density handles)


def test_glue_grid_class_reproduces_the_executed_reference_grids(rt):
    """bot7.grids.sobol after install() (the glue class under the reference's grids/abstract.lua, unit-cube points from the
    stand-in library) against the vectors of the reference's own generator (tests/golden/ref_exec.npz), including the one-sided
    rescale variants that the glue computes with its own tensor arithmetic."""
    I = rt.I
    G = np.load(os.path.join(ROOT, "tests", "golden", "ref_exec.npz"))
    I.G.set("MINS", torch7.Tensor(np.ascontiguousarray(G["sobol_mins6"].reshape(1, -1)), "torch.DoubleTensor"))
    I.G.set("MAXES", torch7.Tensor(np.ascontiguousarray(G["sobol_maxes6"].reshape(1, -1)), "torch.DoubleTensor"))
    r = I.run(r"""
local S = bot7.grids.sobol
assert(torch.type(S{size = 1, dims = 2}) == 'bot7_b200.grids.sobol')
return S{size = 256, dims = 6}:generate(), S{size = 40, dims = 6, skip = 37}:generate(), S{size = 24, dims = 39}(),
       S{size = 64, dims = 6, mins = MINS, maxes = MAXES}:generate(), S{size = 64, dims = 6, mins = MINS}:generate(),
       S{size = 64, dims = 6, maxes = MAXES}:generate()
""")
    for got, key in zip(r, ["sobol_d6_n256", "sobol_d6_n40_skip37", "sobol_d39_n24", "sobol_d6_n64_scaled", "sobol_d6_n64_mins", "sobol_d6_n64_maxes"]):
        assert np.array_equal(got.a, G[key]), key

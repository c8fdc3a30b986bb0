"""The LuaJIT glue (lua/bot7_b200/*.lua) EXECUTED: tools/minilua is a Lua 5.1 interpreter with Torch7-tensor and LuaJIT-FFI
stand-ins, written for this repository because the image has no Lua runtime.  The FFI stand-in parses the glue's own
`ffi.cdef` block and calls the real libbot7_b200.so through ctypes, so on a GPU box every glue method runs the CUDA path
exactly as a `th` process would drive it -- and is compared with the CPU oracle like the Python twin is.

CPU part (no GPU): the interpreter's Lua semantics, the tensor and FFI stand-ins, and everything of the glue that does not need
a device (module loading, install(), class wiring, argument conversion errors, the loud failure without a CUDA device).
GPU part: Sobol grid, EI / confidence bound, GP predict / log density / hyper sampling, bayesopt nomination, DNGO head.
"""
import io
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from minilua import Interpreter, LuaError  # noqa: E402
from minilua import torch7  # noqa: E402
from minilua.harness import GlueRuntime  # noqa: E402


def lua(src, *args):
    out = io.StringIO()
    I = Interpreter(stdout=out)
    r = I.run(src, "=t", *args)
    return r, out.getvalue()


# ---------------------------------------------------------------------------------- interpreter semantics (CPU)

SEMANTICS = r"""
local function fib(n) if n < 2 then return n end return fib(n - 1) + fib(n - 2) end
print(fib(15))
local t = {10, 20, 30, x = 'a', [5] = 50}
print(#t, t.x, t[5])
local function va(...) local a, b = ...; return select('#', ...), a, b end
print(va(1, nil, 3))
local cnt = 0
local function counter() return function() cnt = cnt + 1; return cnt end end
local c1, c2 = counter(), counter()
c1(); c1(); c2()
print(cnt)
local A = {}; A.__index = A
function A.new(v) return setmetatable({v = v}, A) end
function A:get() return self.v end
A.__add = function(a, b) return A.new(a.v + b.v) end
A.__call = function(self, x) return self.v * x end
A.__tostring = function(self) return 'A(' .. self.v .. ')' end
A.__eq = function(a, b) return a.v == b.v end
local a = A.new(3) + A.new(4)
print(a:get(), a(2), tostring(a), a == A.new(7), a ~= A.new(8))
print(string.format('%5.2f|%d|%s|%-4s|%e|%5d|%%', 3.14159, 42.0, 'hi', 'ab', 12345.678, 7))
print(('Hello'):lower(), ('confidence_bound'):find('bound'))
print(pcall(function() error({code = 7}) end))
print(pcall(function() local x = nil; return x.y end))
print(pcall(error, 'plain'))
for i = 10, 1, -3 do io.write(i, ' ') end print()
for k, v in ipairs({'a', 'b', 'c'}) do io.write(k, v, ' ') end print()
local keys = {} for k in pairs({x = 1, y = 2}) do keys[#keys + 1] = k end table.sort(keys) print(table.concat(keys, ','))
local i = 0 repeat local j = i; i = i + 1 until j >= 2 print(i)
print(1e3, 2^10, 10 / 4, 7 % 3, -7 % 3, 1/0, -1/0, math.huge == 1/0, 0/0 ~= 0/0)
print(type(nil), type(1), type('s'), type({}), type(print), type(fib))
print(tostring(1e15), tostring(0.1), 1e100, 2^53)
local p, q, r = (function() return 1, 2, 3 end)()
print(p, q, r, (va(1, 2)))
print(({(function() return 1, 2 end)(), (function() return 3, 4 end)()})[3])
print(not nil, nil == false, 1 == 1.0, '1' == 1, 'a' < 'b', '10' + 5, '3' * '4')
print(select(-1, 1, 2, 3), #'abc', ('x'):rep(3), ('abcdef'):sub(2, -2))
print(tonumber('0x10'), tonumber('  12  '), tonumber('1e2'), tonumber('abc'), tonumber('10', 2))
print(string.gsub('hello world', 'o', '0'), ('key=val'):match('(%w+)=(%w+)'))
print(next({}), rawget(t, 'x'), unpack({1, 2, 3}))
local x, y = 1, 2; x, y = y, x; print(x, y)
local tt = {}; local k = 1; k, tt[k] = 2, 'v'; print(k, tt[1], tt[2])
do local s = 0; for _, v in ipairs{1, 2, 3} do if v == 2 then break end s = s + v end print(s) end
local function outer() local n = 0; return function() n = n + 1; return n end, function() return n end end
local inc, get = outer(); inc(); inc(); print(get())
print(math.floor(-3.5), math.ceil(3.2), math.max(1, 5, 3), math.min(2, -1), math.abs(-2), math.sqrt(16), math.log(1), math.pi > 3.14)
goto_like = 5; print(goto_like, _G.goto_like, _G['goto_like'])
print(#{1, 2, nil, 4} >= 2, #'', ('%d items'):format(3))
local mt = setmetatable({}, {__index = function(_, key) return key .. '!' end, __newindex = function(tb, key, v) rawset(tb, key, v * 2) end})
mt.z = 4; print(mt.foo, mt.z, getmetatable(mt) ~= nil, getmetatable('s').__index == string)
print(pcall(function() return 1 + {} end))
print(pcall(function() return #5 end))
print(pcall(function() local f; f() end))
print(tostring(nil), tostring(true), tostring(12), 1 .. 2, 'a' .. 1.5)
print(-2^2, 2^3^2, not 1 == 2, 1 .. 2 .. 3, 2 * 3 % 4, -3 % 5, 1 + 2 < 4 and 'y' or 'n', #'ab' + 1, -2 ^ -2, -0.0, 100 * 1.1, 1e16)
for i = 1, 2, 0.5 do io.write(i, ';') end print()
return 'done', 42
"""

EXPECTED = """610
3\ta\t50
3\t1\tnil
3
7\t14\tA(7)\ttrue\ttrue
 3.14|42|hi|ab  |1.234568e+04|    7|%
hello\t12\t16
false\ttable
false\tattempt to index 'x' (a nil value) with key 'y'
false\tplain
10 7 4 1
1a 2b 3c
x,y
3
1000\t1024\t2.5\t1\t2\tinf\t-inf\ttrue\ttrue
nil\tnumber\tstring\ttable\tfunction\tfunction
1e+15\t0.1\t1e+100\t9.007199254741e+15
1\t2\t3\t2
4
true\tfalse\ttrue\tfalse\ttrue\t15\t12
3\t3\txxx\tbcde
16\t12\t100\tnil\t2
hell0 w0rld\tkey\tval
nil\ta\t1\t2\t3
2\t1
2\tv\tnil
1
2
-4\t4\t5\t-1\t2\t4\t0\ttrue
5\t5\t5
true\t0\t3 items
foo!\t8\ttrue\ttrue
false\tattempt to perform arithmetic on a table value
false\tattempt to get length of a number value
false\tattempt to call 'f' (a nil value)
nil\ttrue\t12\t12\ta1.5
-4\t512\tfalse\t123\t2\t2\ty\t3\t-0.25\t-0\t110\t1e+16
1;1.5;2;
"""


def test_interpreter_semantics():
    r, out = lua(SEMANTICS)
    got = [(ln if "table: 0x" not in ln else ln.split("table: 0x")[0] + "table").rstrip() for ln in out.splitlines()]
    for k, (g, e) in enumerate(zip(got, EXPECTED.splitlines())):
        assert g == e, f"output line {k + 1}"
    assert len(got) == len(EXPECTED.splitlines())
    assert r == ["done", 42]


def test_interpreter_varargs_methods_and_errors():
    r, _ = lua("""
local C = {}; C.__index = C
function C.new(...) local o = setmetatable({}, C); o.args = {...}; o.n = select('#', ...); return o end
function C:sum() local s = 0; for i = 1, self.n do s = s + (self.args[i] or 0) end; return s end
local o = C.new(1, 2, nil, 4)
local ok, err = pcall(function() return o:missing() end)
local ok2, err2 = pcall(function() error('boom', 2) end)
local function tail(n) if n == 0 then return 'end' end return tail(n - 1) end
return o:sum(), o.n, ok, err, err2, tail(100), ...
""", "extra")
    assert r[0] == 7 and r[1] == 4 and r[2] is False and "missing" in r[3] and r[4] == "boom" and r[5] == "end" and r[6] == "extra"


def test_require_search_path_and_preload(tmp_path):
    d = tmp_path / "pkg"
    d.mkdir()
    (d / "init.lua").write_text("local M = {name = ...}; M.sub = require('pkg.sub'); return M")
    (d / "sub.lua").write_text("return {value = 7, loaded_as = ...}")
    out = io.StringIO()
    I = Interpreter(search_path=[("pkg", str(d))], stdout=out)
    r = I.run("package.preload['virt'] = function(n) return {n = n} end\n"
              "local a, b = require('pkg'), require('pkg')\n"
              "return a == b, a.name, a.sub.value, a.sub.loaded_as, require('virt').n, pcall(require, 'nope')")
    assert r[:5] == [True, "pkg", 7, "pkg.sub", "virt"] and r[5] is False and "not found" in r[6]


# ---------------------------------------------------------------------------------- Torch7 stand-in (CPU)

def test_tensor_standin_follows_torch7_semantics():
    out = io.StringIO()
    I = Interpreter(stdout=out)
    torch7.install(I, seed=1)
    r = I.run(r"""
local t = torch.DoubleTensor{{1, 2, 3}, {4, 5, 6}}
local v = t:narrow(2, 2, 2)                       -- view: columns 2..3
v:fill(9)
local mn, imn = t:min(2)                          -- keeps the dimension, indices are 1-based
local row = t[2]; row[1] = -1                     -- t[i] is a view of row i
local h = torch.zeros(1, 4); h:narrow(2, 1, 2):fill(0.5); h[1][4] = 7
local e = torch.DoubleTensor{1, 2}:view(2, 1):expand(2, 3)
local c = torch.cat({torch.ones(1, 2), torch.zeros(1, 2)}, 1)
local s = torch.DoubleTensor{1, 4, 9}:sqrt():add(1):mul(2)        -- in place, chained
local l = torch.rand(1):mul(10):long():add(1)
local cls, par = torch.class('t.A'), nil
return t, mn, imn, h, e:isContiguous(), e:size(2), c, s, t:view(-1):size(1), t:sum(), t:mean(), torch.type(t), torch.type(l),
       #torch.DoubleTensor(3, 2):size(), t:t():isContiguous(), torch.type(cls), (#t)[2], pcall(function() return t:narrow(2, 3, 2) end)
""".replace("local cls, par = torch.class('t.A'), nil", "t_ = {}; local cls = torch.class('t_.A')"))
    t, mn, imn, h, e_contig, e_size2, c, s = r[:8]
    assert np.array_equal(t.a, [[1, 9, 9], [-1, 9, 9]])
    assert np.array_equal(mn.a, [[1], [4]]) and np.array_equal(imn.a, [[1], [1]]) and imn.ttype == "torch.LongTensor"
    assert np.array_equal(h.a, [[0.5, 0.5, 0, 7]])
    assert e_contig is False and e_size2 == 3
    assert np.array_equal(c.a, [[1, 1], [0, 0]]) and np.array_equal(s.a, [4, 6, 8])
    assert r[8] == 6 and r[9] == 36.0 and r[10] == 6.0 and r[11] == "torch.DoubleTensor" and r[12] == "torch.LongTensor"
    assert r[13] == 2 and r[14] is False and r[15] == "table" and r[16] == 3    # a transposed view is not contiguous: :data() on it is an error here
    assert r[17] is False and "out of range" in r[18]
    # uninitialised tensors are poisoned, so a glue that reads before writing is caught
    assert np.isnan(I.run("return torch.DoubleTensor(2, 2)")[0].a).all()
    # torch.class needs the package table of a dotted name (luaT_getinnerparent)
    with pytest.raises(LuaError, match="invalid module name"):
        I.run("torch.class('nowhere.Thing')")


def test_torch_class_inheritance_and_call_protocol():
    out = io.StringIO()
    I = Interpreter(stdout=out)
    torch7.install(I)
    r = I.run(r"""
pk = {}
local P = torch.class('pk.Parent')
function P:__init(a) self.a = a end
function P:who() return 'parent' end
function P:__call__(x) return self.a + x end
local C, parent = torch.class('pk.Child', 'pk.Parent')
function C:__init(a, b) parent.__init(self, a); self.b = b end
function C:who() return 'child of ' .. parent.who(self) end
local o = pk.Child(1, 2)
return o.a, o.b, o:who(), o(10), torch.type(o), parent == P, torch.type(P(5)), torch.typename(3) == nil, torch.type(3)
""")
    assert r == [1, 2, "child of parent", 11, "pk.Child", True, "pk.Parent", True, "number"]


# ---------------------------------------------------------------------------------- FFI stand-in + glue without a device (CPU)

def test_ffi_standin_conversions_and_checks():
    with GlueRuntime(fixture=False) as rt:
        r = rt.run(r"""
local ffi = require('ffi')
ffi.cdef[[ typedef struct b7_ctx b7_ctx; typedef struct b7_gp b7_gp; enum { K_A = 0, K_B = 5, K_C };
           int b7_version(void); const char* b7_last_error(void); int b7_init(int device, b7_ctx** out);
           int b7_device_count(void); void b7_gp_free(b7_gp* gp); ]]
local lib = ffi.load('bot7_b200')
local box = ffi.new('b7_ctx*[1]')
local arr = ffi.new('int[?]', 3, {7, 8})
local one = ffi.new('double[1]'); one[0] = 2.5
local wrong = ffi.new('b7_gp*[1]')
local function E(f, ...) local ok, e = pcall(f, ...); return tostring(ok) .. '|' .. tostring(e) end
return lib.b7_version(), lib.K_B, lib.K_C, box[0] == nil, arr[0], arr[1], arr[2], one[0], ffi.sizeof('int'), ffi.sizeof(arr),
       E(lib.b7_version, 1),                          -- wrong number of arguments
       E(lib.b7_init, 0, 5),                          -- a number where a pointer is expected
       E(lib.b7_init, 0, wrong),                      -- pointer to another struct type
       E(lib.b7_init, 'x', box),                      -- a string where an int is expected
       E(function() return arr[3] end),               -- out of bounds
       E(function() return lib.b7_nope end),          -- undeclared symbol
       E(ffi.new, 'b7_ctx')                           -- opaque type
""")
        assert r[0] == 100 and r[1] == 5 and r[2] == 6 and r[3] is True and r[4:8] == [7, 8, 0, 2.5] and r[8] == 4 and r[9] == 12
        errs = r[10:]
        assert all(e.startswith("false|") for e in errs)
        assert "wrong number of arguments" in errs[0]
        assert "cannot convert 'number'" in errs[1]
        assert "cannot convert 'b7_gp **' to 'b7_ctx **'" in errs[2]
        assert "cannot convert 'string' to 'int'" in errs[3]
        assert "out of bounds" in errs[4]
        assert "missing declaration" in errs[5]
        assert "opaque" in errs[6]


def test_glue_cdef_declares_the_whole_header():
    """The ffi.cdef block of lua/bot7_b200/ffi.lua parses with the stand-in's C declaration parser and declares every function of
    include/bot7_b200.h with the same number of parameters."""
    import re
    with GlueRuntime() as rt:
        rt.require("bot7_b200.ffi")
        header = open(os.path.join(ROOT, "include", "bot7_b200.h")).read()
        header = re.sub(r"//[^\n]*", "", re.sub(r"/\*.*?\*/", "", header, flags=re.S))
        n = 0
        for m in re.finditer(r"\b(b7_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S):
            args = m.group(2).strip()
            want = 0 if args in ("", "void") else len(args.split(","))
            assert m.group(1) in rt.ffi.decls.funcs, m.group(1)
            assert len(rt.ffi.decls.funcs[m.group(1)][1]) == want, m.group(1)
            n += 1
        assert n >= 50 and {"B7_KERNEL_ARDSE", "B7_SCORE_CB", "B7_FIT_LOGML_ONLY", "B7_BOUND_UPPER"} <= set(rt.ffi.decls.enums)


def test_glue_loads_installs_and_fails_loudly_without_a_device():
    with GlueRuntime() as rt:
        r = rt.run(r"""
local M = require('bot7_b200')
local before = bot7.models.dngo
M.install()
local gp = bot7.models.gp_regressor{kernel = 'matern52', nSamples = 3}
local ei, cb = bot7.scores.expected_improvement(), bot7.scores.confidence_bound{bound = 'Upper'}
local grid = bot7.grids.sobol{size = 10, dims = 3}
local X = torch.rand(5, 2)
gp:init(X, torch.rand(5, 1))
return torch.type(gp), gp:class(), gp.config.kernel, gp.config.prior_std, gp.hyp, torch.type(ei), ei.config.tradeoff, cb.config.bound,
       torch.type(grid), grid.config.max_dims, bot7.models.dngo ~= before, before.update_network ~= nil,
       gp:parse_hypers(torch.zeros(5)):dim(), gp:cache().hyp == gp.hyp,
       M.ffi.C.b7_device_count(), pcall(function() return grid:generate() end)
""")
        assert r[0] == "bot7_b200.models.gp_regressor" and r[1] == "gp.models.gp_regressor" and r[2] == "matern52" and r[3] == 2.0
        hyp = r[4].a
        assert hyp.shape == (1, 5) and np.allclose(hyp[0, :2], np.log(0.5)) and hyp[0, 2] == 0.0 and np.isclose(hyp[0, 3], 0.5 * np.log(1e-2))
        assert r[5] == "bot7_b200.scores.expected_improvement" and r[6] == 0.0 and r[7] == "Upper"
        assert r[8] == "bot7_b200.grids.sobol" and r[9] == 40 and r[10] is True and r[11] is True and r[12] == 2 and r[13] is True
        if r[14] == 0:                                     # no device: the first call that needs one fails loudly, no CPU path
            assert r[15] is False and "no CUDA device" in r[16] and "no CPU path" in r[16]


# ---------------------------------------------------------------------------------- the glue on the GPU

def _has_gpu():
    try:
        from bot7_b200 import _lib
        return _lib.lib().b7_device_count() > 0
    except Exception:
        return False


@pytest.fixture()
def rt():
    if not _has_gpu():
        pytest.skip("no CUDA device")
    runtime = GlueRuntime(seed=5)
    runtime.run("require('bot7_b200').install()")
    yield runtime
    runtime.close()


def rel(a, b, floor):
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor)))


def problem(oracle, N, d, S, M, noise=1e-2, seed=3):
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


@pytest.mark.gpu
def test_lua_sobol_grid_is_bit_exact(rt, oracle):
    rt.set_global("MINS", rt.tensor([-1.0, 0.0, 2.0, -5.0, 0.5, 0.0]))
    rt.set_global("MAXES", rt.tensor([1.0, 3.0, 4.0, 5.0, 0.75, 10.0]))
    r = rt.run(r"""
local B, ffi = require('bot7_b200.ffi'), require('ffi')
local g = bot7.grids.sobol{size = 5000, dims = 6}
local a = g:generate()
local b = g:generate{size = 300, dims = 6, skip = 4090, mins = MINS, maxes = MAXES}
local c = bot7.grids.sobol{size = 64, dims = 39}:generate()
local dev = g:generate_device(nil, 100, 50)             -- rows 100 .. 149 as a device-resident grid
local back = torch.DoubleTensor(50, 6)
B.check(B.C.b7_grid_read(dev, 0, 50, back:data()), 'b7_grid_read')
return a, b, c, back
""")
    assert np.array_equal(r[0].a, oracle.sobol_points(6, 5000))
    assert np.array_equal(r[1].a, oracle.sobol_points(6, 300, 4090, rt.I.G.get("MINS").a, rt.I.G.get("MAXES").a))
    assert np.array_equal(r[2].a, oracle.sobol_points(39, 64))
    assert np.array_equal(r[3].a, oracle.sobol_points(6, 5000)[100:150])


@pytest.mark.gpu
def test_lua_sobol_grid_equals_the_executed_reference(rt):
    """The glue's grid class against the vectors the reference's own grids/sobol.lua produced under the interpreter
    (tests/golden/ref_exec.npz): plain, skipped, two-sided rescale (done by the library) and the one-sided variants (done by the
    glue's own tensor arithmetic, grids/sobol.lua:82-86) -- bit for bit."""
    G = np.load(os.path.join(ROOT, "tests", "golden", "ref_exec.npz"))
    rt.set_global("MINS", rt.tensor(G["sobol_mins6"].reshape(1, -1)))            # 1 x d, as bots/abstract.lua builds them
    rt.set_global("MAXES", rt.tensor(G["sobol_maxes6"].reshape(1, -1)))
    r = rt.run(r"""
local S = bot7.grids.sobol
return S{size = 256, dims = 6}:generate(), S{size = 40, dims = 6, skip = 37}:generate(), S{size = 24, dims = 39}(),
       S{size = 64, dims = 6, mins = MINS, maxes = MAXES}:generate(), S{size = 64, dims = 6, mins = MINS}:generate(),
       S{size = 64, dims = 6, maxes = MAXES}:generate()
""")
    for got, key in zip(r, ["sobol_d6_n256", "sobol_d6_n40_skip37", "sobol_d39_n24", "sobol_d6_n64_scaled", "sobol_d6_n64_mins", "sobol_d6_n64_maxes"]):
        assert np.array_equal(got.a, G[key]), key


@pytest.mark.gpu
def test_lua_scores_match_the_oracle(rt, oracle):
    g = np.random.default_rng(0)
    mean, var = g.standard_normal(4000), np.abs(g.standard_normal(4000)) * 0.3
    var[:5] = 0.0
    rt.set_global("MEAN", rt.tensor(mean.reshape(-1, 1)))
    rt.set_global("VAR", rt.tensor(var.reshape(-1, 1)))
    r = rt.run(r"""
local EI, CB = bot7.scores.expected_improvement, bot7.scores.confidence_bound
return EI.compute(MEAN, VAR, torch.DoubleTensor{-0.3}, 0.1), CB.compute(MEAN, VAR, CB{tradeoff = 2.0, bound = 'upper', sign = 1.0}.config),
       CB.compute(MEAN, VAR, CB().config)
""")
    ei = oracle.ei_compute(mean, var, -0.3, 0.1)
    assert rel(r[0].a, ei, 1e-300) <= 1e-7 and np.mean(r[0].a == ei) > 0.9   # north_star: EI 1e-7 relative (exp differs by <= 1 ulp)
    assert np.array_equal(r[0].a[:5], np.maximum((-0.3 + (-mean[:5])) + (-0.1), 0.0))  # sigma = 0 rows: max(improvement, 0) exactly
    assert np.array_equal(r[1].a, oracle.cb_compute(mean, var, 2.0, "upper", 1.0))
    assert np.array_equal(r[2].a, oracle.cb_compute(mean, var))


@pytest.mark.gpu
def test_lua_gp_model_predict_density_and_sampling(rt, oracle):
    Xo, y, hyp, Xc = problem(oracle, 150, 2, 3, 2000)
    for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("X1", Xc), ("HYP", hyp[:1]), ("HYPS", hyp)]:
        rt.set_global(name, rt.tensor(v))
    r = rt.run(r"""
local model = bot7.models.gp_regressor{kernel = 'ardse', nSamples = 4}
local p   = model:predict(X0, Y0, X1, HYP, {mean = true, var = true})
local one = model:predict(X0, Y0, X1[7], HYP, {mean = true})            -- a single point (1-D) and only the mean
local ld  = model:log_density(HYP[1], X0, Y0)
local ldb = model:log_density_batch(HYPS, X0, Y0)                       -- 3 rows through the 8-slot resident handle
local ld2 = model:log_density(HYPS[3], X0, Y0)                          -- resident single-slot handle re-used (b7_gp_refit)
local bad = HYP:clone(); bad[1][3] = 800                                 -- sigma_f^2 = exp(1600) overflows: the density must be -inf, not an error
local ldbad = model:log_density(bad, X0, Y0)
local ei  = bot7.scores.expected_improvement()(model, HYP, X0, Y0, X1)
model:init(X0, Y0)
local start = model.hyp:clone()
local draws = model:sample_hypers(X0, Y0)
local single = model:sample_hypers(X0, Y0, nil, nil, true)
local fant = model:fantasize(5, X0, Y0, X1:narrow(1, 1, 3), HYP)
return p.mean, p.var, one.mean, one.var, ld, ldb, ld2, ldbad, ei, start, draws, single, model.hyp, fant
""")
    fit = oracle.gp_fit(Xo, y, hyp[0], 0)
    mr, vr = oracle.gp_predict(fit, Xc)
    assert r[0].a.shape == (2000, 1) and rel(r[0].a[:, 0], mr, 1.0) <= 1e-9 and rel(r[1].a[:, 0], vr, fit["sf2"]) <= 1e-9
    assert r[2].a.shape == (1, 1) and abs(r[2].a[0, 0] - mr[6]) <= 1e-9 and r[3] is None
    dens = [oracle.gp_fit(Xo, y, h, 0)["logml"] - 0.5 * np.sum((h / 2.0) ** 2) for h in hyp]
    assert abs(r[4] - dens[0]) <= 1e-9 * abs(dens[0])
    assert np.allclose(r[5].a, dens, rtol=1e-9, atol=0) and abs(r[6] - dens[2]) <= 1e-9 * abs(dens[2])
    assert r[7] == -np.inf
    ei = oracle.ei_compute(mr, vr, float(y.min()), 0.0)
    assert rel(r[8].a, ei, 1e-6 * ei.max()) <= 1e-7
    start, draws, single, state, fant = r[9].a, r[10].a, r[11].a, r[12].a, r[13].a
    assert draws.shape == (4, 5) and np.isfinite(draws).all() and single.shape == (1, 5)
    assert not np.array_equal(draws[0], start[0]) and np.array_equal(state[0], single[0])      # the chain moved and its state is the last draw
    assert fant.shape == (3, 5) and np.isfinite(fant).all()


@pytest.mark.gpu
def test_lua_speculative_hyper_sampling_matches_the_python_twin(oracle):
    """model:sample_hypers through lua/bot7_b200/sampler_spec.lua (batches of 8 density evaluations per b7_gp_refit) against the
    Python twin's slice_speculative on the same device library: both draw from numpy generators with the same seed in the same
    order, so the chains coincide (to the rounding of the direction's norm), and the sequential setting gives the same chain."""
    if not _has_gpu():
        pytest.skip("no CUDA device")
    sys.path.insert(0, ROOT)
    from bot7_b200 import models
    Xo, y, hyp, _ = problem(oracle, 200, 2, 1, 10)

    def lua_chain(speculative):
        r_ = GlueRuntime(seed=9)
        r_.run("require('bot7_b200').install()")
        for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("H0", hyp[:1])]:
            r_.set_global(name, r_.tensor(v))
        r_.set_global("SPEC", speculative)
        r = r_.run(r"""
local model = bot7.models.gp_regressor{kernel = 'ardse', nSamples = 5, speculative = SPEC, spec_width = 8}
model.hyp = H0:clone()
local draws = model:sample_hypers(X0, Y0)
return draws, model.hyp, torch.rand(1)[1]
""")
        out = (r[0].a.copy(), r[1].a.copy(), r[2], list(r_.ffi.calls))
        r_.close()
        return out
    spec, spec_state, spec_next, calls = lua_chain(True)
    # eight density evaluations per device call: one b7_gp_fit for the resident handle, then b7_gp_refit per batch
    n_batches = calls.count("b7_gp_fit") + calls.count("b7_gp_refit")
    assert calls.count("b7_gp_fit") == 1 and 5 <= n_batches <= 40
    tw = models.gp_regressor({"kernel": "ardse", "nSamples": 5, "speculative": True, "spec_width": 8}, rng=np.random.default_rng(9))
    tw.hyp = hyp[0].copy()
    ref = tw.sample_hypers(Xo, y)
    assert spec.shape == (5, 5) and np.allclose(spec, ref, rtol=0.0, atol=1e-9)
    assert np.allclose(spec_state[0], tw.hyp, rtol=0.0, atol=1e-9)
    assert abs(spec_next - tw.rng.random()) == 0.0                       # both generators were left in the same state
    # the fixture's sequential stand-in sampler draws in another order, so the sequential setting is compared through the twin
    tw2 = models.gp_regressor({"kernel": "ardse", "nSamples": 5, "speculative": False}, rng=np.random.default_rng(9))
    tw2.hyp = hyp[0].copy()
    assert np.array_equal(tw2.sample_hypers(Xo, y), ref)


@pytest.mark.gpu
def test_lua_bayesopt_nominates_the_oracle_argmax(rt, oracle):
    Xo, y, hyp, Xc = problem(oracle, 120, 2, 1, 3000)
    for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("XC", Xc)]:
        rt.set_global(name, rt.tensor(v))
    r = rt.run(r"""
local model = bot7.models.gp_regressor{kernel = 'ardse'}
local score = bot7.scores.expected_improvement()
local cfg = {bot = {nInitial = 2, nSamples = 3}, candidates = XC, model = model, score = score, observed = X0, responses = Y0, nTrials = 5}
local bot = bot7.bots.bayesopt(nil, nil, cfg)
local rec, orig = {}, model.sample_hypers
model.sample_hypers = function(self, ...) local h = orig(self, ...); rec[#rec + 1] = h:clone(); return h end
local first = bot:nominate()
-- the nominated row left the device grid (utils.tensor.steal): with the same draws the next nomination is another point,
-- numbered in the compacted grid
local n_draws, replay = #rec, 0
model.sample_hypers = function(self, X, Y, a, b, single)
  if not single then return rec[1] end
  replay = replay % 3 + 1
  return rec[1 + replay]
end
local second = bot:nominate()
local fresh = bot7.bots.bayesopt(nil, nil, {bot = {nInitial = 2, nSamples = 3}, candidates = XC, model = model, score = score,
                                            observed = X0, responses = Y0, nTrials = 1})
local rnd = fresh:nominate()                             -- still in the initial design: a random row
model.sample_hypers = function(self, X, Y, a, b, single) return rec[4] end
local ucb = bot7.bots.bayesopt(nil, nil, {bot = {nInitial = 0, nSamples = 1}, candidates = XC, model = model,
                                          score = bot7.scores.confidence_bound{tradeoff = 2.0}, observed = X0, responses = Y0, nTrials = 3})
local third = ucb:nominate()
return first, second, rnd, third, torch.cat(rec, 1), n_draws, torch.type(first)
""")
    first, second, rnd, third, rec, n_draws = r[0].a, r[1].a, r[2].a, r[3].a, r[4].a, r[5]
    assert n_draws == 4 and rec.shape[1] == 5 and r[6] == "torch.LongTensor"
    hyps = rec[1:4]                                                          # the priming draw is discarded (bots/bayesopt.lua:68)
    ref = oracle.acquisition(Xo, y, hyps, Xc, 0, False, oracle.SCORE_EI)
    assert first.shape == (1,) and int(first[0]) == ref["idx"]
    keep = np.ones(len(Xc), bool)
    keep[ref["idx"] - 1] = False
    ref2 = oracle.acquisition(Xo, y, hyps, Xc[keep], 0, False, oracle.SCORE_EI)
    assert int(second[0]) == ref2["idx"]
    assert 1 <= int(rnd[0]) <= len(Xc)
    keep3 = np.ones(len(Xc), bool)                                          # `ucb` has its own device grid: nothing removed yet
    ref3 = oracle.acquisition(Xo, y, hyps[2:3], Xc[keep3], 0, False, oracle.SCORE_CB, 2.0)
    assert int(third[0]) == ref3["idx"]


@pytest.mark.gpu
def test_lua_dngo_head_matches_the_oracle(rt, oracle):
    Xo, y, _, Xc = problem(oracle, 400, 6, 1, 5000)
    for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("XC", Xc)]:
        rt.set_global(name, rt.tensor(v))
    r = rt.run(r"""
local B, ffi = require('bot7_b200.ffi'), require('ffi')
local net = nn.Sequential():add(nn.Linear(6, 24)):add(nn.ReLU()):add(nn.Linear(24, 50)):add(nn.ReLU()):add(nn.Linear(50, 1))
local model = bot7.models.dngo({network = net, basis = net:get(4), zDim = 50, update = {schedule = {batchsize = 32}}, predictor = {}})
local p = model:predict(X0, Y0, XC, nil, {mean = true, var = true})
local box = ffi.new('b7_grid*[1]')
B.check(B.C.b7_grid_from_host(B.context(), XC:data(), XC:size(1), XC:size(2), box), 'b7_grid_from_host')
local grid = ffi.gc(box[0], B.C.b7_grid_free)
local argmax, best, nans = model:acquire(X0, Y0, grid, B.C.B7_SCORE_EI, 0.0, B.C.B7_BOUND_LOWER, -1.0)
return p.mean, p.var, argmax, best, nans, model.updates, net:get(1).weight, net:get(1).bias, net:get(3).weight, net:get(3).bias, model:class()
""")
    W1, b1, W2, b2 = r[6].a, r[7].a, r[8].a, r[9].a
    Z0 = oracle.mlp_features(Xo, [W1, W2], [b1, b2], True)
    Z1 = oracle.mlp_features(Xc, [W1, W2], [b1, b2], True)
    fit = oracle.blr_fit(Z0, y, [0.0, np.log(1e2), float(y.mean())])
    mr, vr = oracle.blr_predict(fit, Z1)
    assert r[0].a.shape == (5000, 1) and rel(r[0].a[:, 0], mr, 1.0) <= 1e-9 and rel(r[1].a[:, 0], vr, 1e-2) <= 1e-9
    ei = oracle.ei_compute(mr, vr, float(y.min()), 0.0)
    best, idx, nan_count = oracle.argmax_first(ei)
    assert r[2] == idx and abs(r[3] - best) <= 1e-7 * abs(best) and r[4] == 0
    assert r[5] == 2 and r[10] == "bot7.models.dngo"                       # predict and acquire both ran the parent's network update


@pytest.mark.gpu
def test_lua_bayesopt_on_two_gpus_equals_one(rt, oracle):
    from bot7_b200 import _lib
    if _lib.lib().b7_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    Xo, y, hyp, Xc = problem(oracle, 200, 2, 4, 6000)
    for name, v in [("X0", Xo), ("Y0", y.reshape(-1, 1)), ("XC", Xc), ("HYPS", hyp)]:
        rt.set_global(name, rt.tensor(v))
    r = rt.run(r"""
local model = bot7.models.gp_regressor{kernel = 'ardse'}
local k = 0
model.sample_hypers = function(self, X, Y, a, b, single) if not single then return HYPS end; k = k % 4 + 1; return HYPS[k]:view(1, -1) end
local out = {}
for _, n in ipairs{1, 2} do
  k = 0
  local bot = bot7.bots.bayesopt(nil, nil, {bot = {nInitial = 0, nSamples = 4, nGPU = n}, candidates = XC, model = model,
                                            score = bot7.scores.expected_improvement(), observed = X0, responses = Y0, nTrials = 3})
  out[#out + 1] = bot:nominate()[1]
  out[#out + 1] = bot:nominate()[1]
end
return out[1], out[2], out[3], out[4]
""")
    ref = oracle.acquisition(Xo, y, hyp, Xc, 0, False, oracle.SCORE_EI)
    assert r[0] == ref["idx"] and r[2] == r[0] and r[3] == r[1] and r[1] != r[0]


# ---------------------------------------------------------------------------------- the interpreter on the reference's own Lua (CPU)

REF = os.environ.get("BOT7_REFERENCE", "")         # a checkout of the reference bot7 Lua source, if any


def _lua_spec_chain(rt, speculative, width):
    """120 draws of a correlated 2-D Gaussian from seed 11 in `rt`, by lua/bot7_b200/sampler_spec.lua (batch width `width`) or,
    not speculative, by bot7.samplers.slice (the reference's, loaded into `rt` by the caller): alternately narrow brackets that
    step out and wide ones that shrink.  -> (chain 120 x 2, density evaluations, batched calls, the generator's next draw)."""
    rt.set_global("SPEC", speculative)
    rt.set_global("WIDTH", width)
    r = rt.run(r"""
local evals, calls = 0, 0
local function logp1(x, a) return -0.5 * (x[1] ^ 2 / a.v1 + x[2] ^ 2 / a.v2 + 0.3 * x[1] * x[2]) end
local function f(x, a) evals = evals + 1; return logp1(x[1], a) end
local function fb(P, a) calls = calls + 1; local o = torch.Tensor(P:size(1)); for i = 1, P:size(1) do evals = evals + 1; o[i] = logp1(P[i], a) end; return o end
local sampler = SPEC and require('bot7_b200.sampler_spec')() or bot7.samplers.slice()
local out, x = torch.Tensor(120, 2), torch.Tensor{{0.3, -0.2}}
for i = 1, 120 do
  local opt = {nSamples = 1, width = (i % 2 == 0) and 0.05 or 6.0}        -- narrow brackets step out, wide ones shrink
  if SPEC then x = sampler(fb, x, opt, {v1 = 1.0, v2 = 4.0}, WIDTH) else x = sampler(f, x, opt, {v1 = 1.0, v2 = 4.0}) end
  out[i]:copy(x[1])
end
return out, evals, calls, torch.rand(1)[1]
""")
    rt.close()
    return r[0].a, r[1], r[2], r[3]


@pytest.mark.skipif(not os.path.isdir(REF), reason="bot7 reference source not found (set BOT7_REFERENCE to a checkout)")
def test_interpreter_runs_the_reference_slice_sampler_unchanged():
    """Validation of the interpreter and the tensor stand-in on code that was written for the real runtime: the reference's
    samplers/abstract.lua, samplers/slice.lua and utils/tensor.lua are loaded from the read-only reference tree, unmodified, and
    sample a correlated-scale Gaussian; the same call protocol (sampler(f, X0, opt, f_args) -> nSamples x dim tensor) is what
    lua/bot7_b200/models_gp.lua:sample_hypers relies on and what the test fixture's stand-in sampler implements."""
    out = io.StringIO()
    I = Interpreter(stdout=out)
    torch7.install(I, seed=3)
    I.run("bot7 = {samplers = {}, utils = {}}")
    utils_tensor = I.run_file(os.path.join(REF, "utils", "tensor.lua"))[0]
    I.G.get("bot7").get("utils").set("tensor", utils_tensor)
    I.G.get("package").get("loaded").set("bot7.utils", I.G.get("bot7").get("utils"))
    I.run_file(os.path.join(REF, "samplers", "abstract.lua"))
    I.run_file(os.path.join(REF, "samplers", "slice.lua"))
    r = I.run(r"""
local sampler = bot7.samplers.slice()
local evals = 0
local function logp(x, args) evals = evals + 1; return -0.5 * (x[1][1] ^ 2 / args.v1 + x[1][2] ^ 2 / args.v2) end
local x = torch.zeros(1, 2)
local out = torch.Tensor(400, 2)
for i = 1, 400 do
  x = sampler(logp, x, {nSamples = 1}, {v1 = 1.0, v2 = 4.0})
  out[i]:copy(x[1])
end
local gibbs = sampler(logp, torch.zeros(1, 2), {nSamples = 3, gibbs = true}, {v1 = 1.0, v2 = 4.0})
return out, evals, gibbs, torch.type(sampler)
""")
    xs, evals, gibbs = r[0].a, r[1], r[2].a
    assert xs.shape == (400, 2) and np.isfinite(xs).all() and evals > 1200 and r[3] == "bot7.samplers.slice"
    # The Python twin (bot7_b200/samplers.py) restates this control flow and draws its random numbers in the same order: fed
    # by the same generator it must walk the SAME chain -- which pins the twin (and with it the speculative
    # sampler that the GPU tests compare with it) to the executed reference.
    sys.path.insert(0, ROOT)
    from bot7_b200 import samplers
    rng = np.random.default_rng(3)
    count = [0]

    def logp(x, args):
        count[0] += 1
        return -0.5 * (x[0, 0] ** 2 / args["v1"] + x[0, 1] ** 2 / args["v2"])
    tw = samplers.slice()
    x = np.zeros((1, 2))
    chain = np.empty((400, 2))
    for i in range(400):
        x = tw(logp, x, {"nSamples": 1}, {"v1": 1.0, "v2": 4.0}, rng)
        chain[i] = x[0]
    g2 = tw(logp, np.zeros((1, 2)), {"nSamples": 3, "gibbs": True}, {"v1": 1.0, "v2": 4.0}, rng)
    # same number of density evaluations = every accept / reject / step-out decision coincided; the values differ by rounding only
    # (the direction's norm: BLAS dot in numpy vs a sum of squares), the Gibbs draws (no norm) not at all
    assert count[0] == evals and np.allclose(chain, xs, rtol=0.0, atol=1e-12) and np.array_equal(g2, gibbs)
    assert abs(xs[:, 0].mean()) < 0.35 and abs(xs[:, 1].mean()) < 0.7
    assert 0.6 < xs[:, 0].var() < 1.6 and 2.4 < xs[:, 1].var() < 6.4          # N(0, diag(1, 4)); 400 correlated draws
    assert gibbs.shape == (3, 2) and np.isfinite(gibbs).all()
    assert "Error" not in out.getvalue()


@pytest.mark.skipif(not os.path.isdir(REF), reason="bot7 reference source not found (set BOT7_REFERENCE to a checkout)")
@pytest.mark.parametrize("width", [1, 3, 4, 8])
def test_lua_speculative_sampler_walks_the_executed_reference_chain(width):
    """lua/bot7_b200/sampler_spec.lua (batched density evaluations, generator rewound after discarded speculation) against
    the reference's samplers/slice.lua executed next to it: from the same generator state the two chains are bit-identical,
    for every batch width, with step-out, with a narrow initial bracket (stepping out needed) and a wide one (shrinking)."""
    def chain(speculative):
        rt = GlueRuntime(seed=11, fixture=False)
        I = rt.I
        I.run("bot7 = {samplers = {}, utils = {}}")
        ut = I.run_file(os.path.join(REF, "utils", "tensor.lua"))[0]
        I.G.get("bot7").get("utils").set("tensor", ut)
        I.G.get("package").get("loaded").set("bot7.utils", I.G.get("bot7").get("utils"))
        I.run_file(os.path.join(REF, "samplers", "abstract.lua"))
        I.run_file(os.path.join(REF, "samplers", "slice.lua"))
        return _lua_spec_chain(rt, speculative, width)
    ref, ref_evals, _, ref_next = chain(False)
    got, evals, calls, nxt = chain(True)
    assert np.array_equal(got, ref)                       # the same chain, bit for bit
    assert nxt == ref_next                                # and the generator is left where the sequential sampler leaves it
    assert calls < ref_evals                              # in fewer sequential (device) calls
    if width >= 4:
        assert calls < 0.5 * ref_evals


@pytest.mark.parametrize("width", [1, 3, 4, 8])
def test_lua_speculative_sampler_walks_the_python_twin_chain(width):
    """lua/bot7_b200/sampler_spec.lua against bot7_b200/samplers.py:slice, the Python restatement of samplers/slice.lua, on the
    chain of the test above and without the reference tree: from the same seed the two walk the same chain (to the rounding of
    the direction's norm: BLAS dot in numpy vs a sum of squares), draw the same random numbers (the generator is left in the same
    state) and the speculative one needs fewer sequential density calls."""
    sys.path.insert(0, ROOT)
    from bot7_b200 import samplers
    got, _, calls, nxt = _lua_spec_chain(GlueRuntime(seed=11, fixture=False), True, width)
    rng, evals = np.random.default_rng(11), [0]

    def logp(x, a):
        evals[0] += 1
        return -0.5 * (x[0, 0] ** 2 / a["v1"] + x[0, 1] ** 2 / a["v2"] + 0.3 * x[0, 0] * x[0, 1])
    tw, x, chain = samplers.slice(), np.array([[0.3, -0.2]]), np.empty((120, 2))
    for i in range(1, 121):
        x = tw(logp, x, {"nSamples": 1, "width": 0.05 if i % 2 == 0 else 6.0}, {"v1": 1.0, "v2": 4.0}, rng)
        chain[i - 1] = x[0]
    assert np.allclose(got, chain, rtol=0.0, atol=1e-12)
    assert nxt == rng.random()
    assert calls < evals[0]
    if width >= 4:
        assert calls < 0.5 * evals[0]

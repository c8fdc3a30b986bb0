"""Static checks of the LuaJIT drop-in (lua/bot7_b200/*.lua); its execution under tools/minilua is tests/test_lua_exec.py and
tests/test_lua_reference_loop.py.  Checked here, without running anything: the glue is complete with respect to the reference's own
call sites and well-formed:

* every method the reference calls on the model / score / grid / sampler objects of the accelerated path
  (extracted from the reference named by BOT7_REFERENCE when it is present, otherwise from the committed list below, which was extracted
  from it) is defined by the replacement class, or inherited from the reference parent it subclasses;
* every C symbol the glue calls through `B.C.` is declared in include/bot7_b200.h (and therefore in the generated cdef);
* block keywords balance (the first, parser-free check) and, with tools/lua_check.py, the full grammar, every name, every
  `self:method()`, the arity of every FFI call and the existence of every method name (second half of this file).
"""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LUA = os.path.join(ROOT, "lua", "bot7_b200")
REF = os.environ.get("BOT7_REFERENCE", "")         # a checkout of the reference bot7 Lua source, if any

# method names the reference calls on `self.model` / `model` in the files of the path (SURVEY section 8b):
#   bots/abstract.lua:148 init; bots/bayesopt.lua:65,68,74,75 class, sample_hypers, parse_hypers;
#   scores/expected_improvement.lua:57,63 and scores/confidence_bound.lua:57,63 fantasize, predict; models/abstract.lua cache
MODEL_METHODS = {"init", "sample_hypers", "parse_hypers", "class", "predict", "fantasize", "cache"}
DNGO_METHODS = {"init", "predict", "class"}            # bots/bayesopt.lua:65 + models/dngo.lua protocol used by the scores
CALL_SITES = ["bots/abstract.lua", "bots/bayesopt.lua", "scores/expected_improvement.lua", "scores/confidence_bound.lua"]


def lua(name):
    return open(os.path.join(LUA, name)).read()


def strip_comments(text):
    text = re.sub(r"--\[\[.*?\]\]", "", text, flags=re.S)
    return re.sub(r"--[^\n]*", "", text)


def defined_methods(text, cls):
    return set(re.findall(r"function\s+%s[:.]([A-Za-z_]\w*)\s*\(" % re.escape(cls), text))


def test_reference_call_sites_match_the_committed_list():
    if not os.path.isdir(REF):
        pytest.skip("bot7 reference source not found (set BOT7_REFERENCE to a checkout)")
    called = set()
    for f in CALL_SITES:
        src = strip_comments(open(os.path.join(REF, f)).read())
        called |= set(re.findall(r"\bmodel:([A-Za-z_]\w*)\s*\(", src))
    assert called <= MODEL_METHODS, f"the reference calls model methods missing from the list: {called - MODEL_METHODS}"
    assert {"init", "sample_hypers", "parse_hypers", "class", "predict", "fantasize"} <= called


def test_gp_regressor_defines_every_method_the_reference_calls():
    got = defined_methods(lua("models_gp.lua"), "model")
    assert MODEL_METHODS <= got, f"missing: {MODEL_METHODS - got}"
    # the density the sampler sees carries the prior and the failure guard, like the Python twin (ADVICE r01)
    text = lua("models_gp.lua")
    assert "prior_std" in text and "-math.huge" in text and "info[" in text


def test_dngo_override_defines_the_hand_off():
    text = lua("models_dngo.lua")
    got = defined_methods(text, "dngo")
    assert {"predict", "class", "acquire", "basis_stack"} <= got
    assert "'bot7.models.dngo'" in text                      # subclasses the reference class: init / report / network stay the parent's
    for sym in ("b7_mlp_features", "b7_blr_fit", "b7_blr_predict", "b7_dngo_score"):
        assert "B.C.%s" % sym in text


def test_bayesopt_calls_only_defined_model_methods_and_uses_nGPU():
    text = strip_comments(lua("bayesopt.lua"))
    called = set(re.findall(r"self\.model:([A-Za-z_]\w*)\s*\(", text))
    gp = defined_methods(lua("models_gp.lua"), "model")
    dn = defined_methods(lua("models_dngo.lua"), "dngo")
    for m in called:
        assert m in gp or m in dn, f"bayesopt.lua calls model:{m}, which no replacement model defines"
    assert "config.bot.nGPU" in text
    for sym in ("b7_comm_init_all", "b7_gp_fit_sharded", "b7_acq_score_multi", "b7_grid_remove_sharded"):
        assert "B.C.%s" % sym in text


def test_glue_calls_only_declared_symbols():
    header = open(os.path.join(ROOT, "include", "bot7_b200.h")).read()
    declared = set(re.findall(r"\b(b7_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", header, flags=re.S)))
    enums = set(re.findall(r"\b(B7_[A-Z0-9_]+)\b", header))
    for f in os.listdir(LUA):
        if not f.endswith(".lua") or f == "ffi.lua":
            continue
        text = strip_comments(lua(f))
        for sym in set(re.findall(r"B\.C\.(b7_[a-z0-9_]+)", text)):
            assert sym in declared, f"{f} calls {sym}, not declared in include/bot7_b200.h"
        for e in set(re.findall(r"B\.C\.(B7_[A-Z0-9_]+)", text)):
            assert e in enums, f"{f} uses {e}, not an enum of include/bot7_b200.h"


def test_install_replaces_every_accelerated_class():
    text = lua("init.lua")
    for target in ("bot7.grids.sobol", "bot7.scores.expected_improvement", "bot7.scores.confidence_bound", "bot7.models.gp_regressor",
                   "bot7.models.dngo", "bot7.bots.bayesopt"):
        assert re.search(re.escape(target) + r"\s*=", text), f"install() does not replace {target}"


@pytest.mark.parametrize("name", sorted(f for f in os.listdir(LUA) if f.endswith(".lua")))
def test_block_keywords_balance(name):
    text = strip_comments(lua(name))
    text = re.sub(r"\[\[.*?\]\]", "", text, flags=re.S)           # long strings (the cdef)
    text = re.sub(r"'(?:[^'\\\n]|\\.)*'|\"(?:[^\"\\\n]|\\.)*\"", "''", text)
    opens = len(re.findall(r"\bfunction\b", text)) + len(re.findall(r"\bif\b", text)) + len(re.findall(r"\bdo\b", text))
    # `for ... do` and `while ... do` are counted once through their `do`; `repeat ... until` has no `end`
    ends = len(re.findall(r"\bend\b", text))
    assert opens == ends, f"{name}: {opens} block openers vs {ends} `end`"
    assert text.count("(") == text.count(")") and text.count("{") == text.count("}")


# ---- full-grammar checks (tools/lua_check.py: Lua 5.1 / LuaJIT lexer + parser + scope resolution) ------------------
import sys  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tools"))
import lua_check  # noqa: E402

GLUE_FILES = sorted(f for f in os.listdir(LUA) if f.endswith(".lua"))


@pytest.mark.parametrize("name", GLUE_FILES)
def test_glue_parses_and_every_name_resolves(name):
    """The whole file is valid Lua 5.1 and every name it reads is a local in scope or a global that a `th` process provides:
    a misspelt local or a forgotten `local` would surface here as an unknown global."""
    rep = lua_check.check_file(os.path.join(LUA, name))
    assert not lua_check.unknown_globals(rep), f"{name}: unknown globals {lua_check.unknown_globals(rep)}"
    # the one global the glue owns: the package table torch.class stores its classes in (luaT_getinnerparent needs it to exist)
    allowed = {"bot7_b200"} if name == "ffi.lua" else set()
    assert set(rep.global_writes) <= allowed, f"{name}: assigns globals {rep.global_writes} (the glue must not leak names into _G)"


@pytest.mark.parametrize("name", GLUE_FILES)
def test_self_method_calls_resolve(name):
    """`self:m(...)` inside a glue class: m is defined by the class itself, or by the reference parent it subclasses."""
    text = lua(name)
    rep = lua_check.check_text(text, name)
    own = {path.split(":")[1] for path, _ in rep.functions if ":" in path} | \
          {path.split(".")[-1] for path, _ in rep.functions if "." in path}
    # methods of the reference parents that the glue relies on (bots/abstract.lua, grids/abstract.lua, models/abstract.lua,
    # models/dngo.lua, scores/abstract.lua); extracted from the reference when it is present, else this committed list
    parents = {"bayesopt.lua": ["bots/bayesopt.lua", "bots/abstract.lua"], "grids_sobol.lua": ["grids/sobol.lua", "grids/abstract.lua"],
               "models_dngo.lua": ["models/dngo.lua", "models/abstract.lua"], "models_gp.lua": ["models/abstract.lua"],
               "scores.lua": ["scores/abstract.lua"]}
    committed = {"__init", "cache", "class", "init", "predict", "report", "update", "eval", "nominate", "run_experiment", "generate",
                 "create_bank", "i4_sobol", "fantasize", "parse_hypers", "sample_hypers", "network", "train", "extract_features"}
    inherited = set(committed)
    if os.path.isdir(REF):
        inherited = set()
        for f in parents.get(name, []):
            p = os.path.join(REF, f)
            if os.path.exists(p):
                r = lua_check.check_file(p)
                inherited |= {path.split(":")[1] for path, _ in r.functions if ":" in path}
                inherited |= {path.split(".")[-1] for path, _ in r.functions if "." in path}
    for obj, m, line in rep.method_calls:
        if obj == "self":
            assert m in own or m in inherited, f"{name}:{line}: self:{m}() is defined neither here nor in {parents.get(name)}"


def test_checker_parses_the_whole_reference_tree():
    """Validation of the checker itself: all of the reference's Lua (5 k lines written for the real interpreter) parses."""
    if not os.path.isdir(REF):
        pytest.skip("bot7 reference source not found (set BOT7_REFERENCE to a checkout)")
    n = 0
    for dirpath, _, files in os.walk(REF):
        for f in files:
            if f.endswith(".lua"):
                lua_check.check_file(os.path.join(dirpath, f))
                n += 1
    assert n >= 40


@pytest.mark.parametrize("src, msg", [
    ("local function f(a)\n  if a then return 1\nend\n", "'end'"),                       # unclosed function
    ("local t = {1, 2\nlocal u = 3\n", "'}'"),                                           # unclosed table
    ("local function f() return ... end\n", "vararg"),                                    # ... outside a vararg function
    ("break\n", "break"),                                                                 # break outside a loop
    ("local x = = 3\n", "unexpected"),                                                    # garbage expression
    ("f() = 3\n", "assign"),                                                              # call as assignment target
    ("return 1\nlocal x = 2\n", "last statement"),                                       # code after return
    ("x = 3 +\n", "unexpected"),                                                          # dangling operator
    ("local s = 'abc\n", "unexpected character"),                                         # unfinished string
])
def test_checker_rejects_broken_lua(src, msg):
    with pytest.raises(lua_check.LuaSyntaxError) as e:
        lua_check.check_text(src, "t.lua")
    assert msg in str(e.value)


def test_checker_scope_rules():
    rep = lua_check.check_text("""
local a = 1
local function f(x, ...) local n = select('#', ...); return x + a + n + undefined_name end
for i = 1, 3 do local b = i end
repeat local c = 1 until c == 1
function M.g(self) return self end
function obj:h() return self, misspelt end
leak = b
""", "t.lua")
    assert set(rep.global_reads) == {"select", "undefined_name", "M", "obj", "misspelt", "b"}   # b is out of scope after the loop
    assert set(lua_check.unknown_globals(rep)) == {"undefined_name", "M", "obj", "misspelt", "b"}
    assert set(rep.global_writes) == {"leak"}
    assert ("obj:h", 7) in rep.functions and ("M.g", 6) in rep.functions


def test_ffi_call_arity_matches_the_header():
    """Every C call of the glue passes exactly as many arguments as include/bot7_b200.h declares (LuaJIT raises
    'wrong number of arguments for function call' otherwise -- at run time, which nothing here can reach)."""
    header = open(os.path.join(ROOT, "include", "bot7_b200.h")).read()
    header = re.sub(r"//[^\n]*", "", re.sub(r"/\*.*?\*/", "", header, flags=re.S))
    protos = {}
    for m in re.finditer(r"\b(b7_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S):
        args = m.group(2).strip()
        protos[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    assert len(protos) >= 50
    checked = 0
    for f in GLUE_FILES:
        rep = lua_check.check_file(os.path.join(LUA, f))
        for path, line, n_args in rep.field_calls:
            m = re.search(r"(?:^|\.)(b7_[a-z0-9_]+)$", path)
            if not m:
                continue
            assert m.group(1) in protos, f"{f}:{line}: {m.group(1)} is not declared in the header"
            assert n_args == protos[m.group(1)], f"{f}:{line}: {m.group(1)} called with {n_args} arguments, the header declares {protos[m.group(1)]}"
            checked += 1
    assert checked >= 20


# Torch7 tensor / storage methods (torch7/doc/tensor.md, maths.md), nn.Module methods and Lua string methods the glue may call
TORCH7_METHODS = {
    "add", "addmm", "addmv", "abs", "apply", "byte", "cdiv", "clone", "cmul", "contiguous", "copy", "csub", "cumsum", "data", "dim",
    "div", "dot", "double", "eq", "exp", "expand", "expandAs", "fill", "float", "ge", "gt", "index", "indexCopy", "int", "isContiguous",
    "isSameSizeAs", "le", "log", "long", "lt", "max", "mean", "min", "mm", "mul", "mv", "nDimension", "nElement", "narrow", "ne", "neg",
    "norm", "numel", "pow", "prod", "repeatTensor", "reshape", "resize", "resizeAs", "select", "set", "size", "sort", "sqrt", "squeeze",
    "std", "storage", "stride", "sub", "sum", "t", "transpose", "type", "typeAs", "unfold", "var", "view", "viewAs", "zero",
    "any", "all", "maskedCopy", "maskedFill", "maskedSelect", "nonzero", "indexFill", "cat", "clamp", "cdiv", "cpow",
    "forward", "evaluate", "training", "get", "parameters", "getParameters", "updateOutput",
    "find", "format", "gmatch", "gsub", "len", "lower", "match", "rep", "sub", "upper",
}


def test_every_method_called_by_the_glue_exists_somewhere():
    """obj:method(...) with a misspelt method name is a run-time 'attempt to call method (a nil value)': every method name the
    glue calls is a Torch7 tensor / nn / string method, a method one of the glue classes defines, or one the reference defines."""
    defined = set()
    for f in GLUE_FILES:
        rep = lua_check.check_file(os.path.join(LUA, f))
        defined |= {re.split(r"[:.]", path)[-1] for path, _ in rep.functions}
    ref_defined = {"init", "class", "cache", "predict", "fantasize", "sample_hypers", "parse_hypers", "eval", "nominate", "update",
                   "report", "generate", "network", "train"}
    if os.path.isdir(REF):
        ref_defined = set()
        for dirpath, _, files in os.walk(REF):
            for fn in files:
                if fn.endswith(".lua"):
                    r = lua_check.check_file(os.path.join(dirpath, fn))
                    ref_defined |= {re.split(r"[:.]", path)[-1] for path, _ in r.functions}
    for f in GLUE_FILES:
        rep = lua_check.check_file(os.path.join(LUA, f))
        for obj, m, line in rep.method_calls:
            assert m in TORCH7_METHODS or m in defined or m in ref_defined, f"{f}:{line}: {obj}:{m}() -- no such method anywhere"

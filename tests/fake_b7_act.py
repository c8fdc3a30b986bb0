"""TEST INFRASTRUCTURE: fake_b7_dngo_multi.FakeB7DngoMulti extended with oracle-backed stand-ins of b7_mlp_features_act,
b7_dngo_score_act and b7_dngo_score_multi_act, so that the glue's per-layer activation codes (lua/bot7_b200/models_dngo.lua:
basis_stack) can run under tools/minilua without a GPU.  Like FakeB7, it checks the protocol between the glue and the C ABI
(which entry is called with which codes), not the numerics; the features come from tests/act_oracle.py.  Never importable
from the product: it lives under tests/ and needs oracle/."""
import ctypes as C

import numpy as np

import act_oracle
from fake_b7_dngo_multi import FakeB7DngoMulti
from fake_b7_lib import FakeError, _arr


class FakeB7Act(FakeB7DngoMulti):
    def __init__(self, oracle):
        super().__init__(oracle)
        self.codes = []                                                        # the act arrays the _act entries received

    def _codes(self, n_layers, act):
        codes = [int(a) for a in _arr(act, (n_layers,), C.c_int)]
        if any(a not in (0, 1, 2) for a in codes):
            raise FakeError("unknown activation code in %r" % codes)
        self.codes.append(codes)
        return codes

    def b7_mlp_features_act(self, ctx, g, n_layers, dims, W, b, act, out):
        self._get(ctx, "ctx")
        grid = self._get(g, "grid")
        Ws, bs = self._stack(n_layers, dims, W, b)
        Z = act_oracle.mlp_features(grid["X"], Ws, bs, self._codes(n_layers, act))
        C.c_void_p.from_address(out).value = self._new({"kind": "grid", "X": Z, "live": list(grid["live"])})
        return 0

    def b7_dngo_score_act(self, blr, g, n_layers, dims, W, b, act, kind, tradeoff, bound, sign, fmin, score_host, argmax,
                          argmax_original, best, nan_count):
        f, grid = self._get(blr, "blr"), self._get(g, "grid")
        Ws, bs = self._stack(n_layers, dims, W, b)
        Z1 = act_oracle.mlp_features(grid["X"][grid["live"]], Ws, bs, self._codes(n_layers, act))
        per = []
        for fit in f["fits"]:
            mu, v = self.o.blr_predict(fit, Z1)
            per.append(self.o.ei_compute(mu, v, fmin, tradeoff) if kind == 0 else
                       self.o.cb_compute(mu, v, tradeoff, "upper" if bound == 1 else "lower", sign))
        score = self.o.mc_average(np.array(per))
        bst, idx, nans = self.o.argmax_first(score)
        if score_host:
            _arr(score_host, (len(score),))[...] = score
        C.c_int64.from_address(argmax).value = idx
        if argmax_original:
            C.c_int64.from_address(argmax_original).value = grid["live"][idx - 1] + 1 if idx else 0
        C.c_double.from_address(best).value = bst
        C.c_int64.from_address(nan_count).value = nans
        return 0

    def b7_dngo_score_multi_act(self, comm, blrs, grids, n_layers, dims, W, b, act, kind, tradeoff, bound, sign, fmin, score_host,
                                argmax, argmax_original, best, nan_count):
        c = self._get(comm, "comm")
        bh = [C.c_void_p.from_address(blrs + g * C.sizeof(C.c_void_p)).value for g in range(c["n"])]
        rh = [C.c_void_p.from_address(grids + g * C.sizeof(C.c_void_p)).value for g in range(c["n"])]
        for h in bh:
            self._get(h, "blr")
        for h in rh:
            self._get(h, "grid")
        return FakeB7Act.b7_dngo_score_act(self, bh[0], rh[0], n_layers, dims, W, b, act, kind, tradeoff, bound, sign, fmin, score_host,
                                           argmax, argmax_original, best, nan_count)

"""TEST INFRASTRUCTURE: fake_b7_lib.FakeB7 extended with oracle-backed stand-ins of b7_blr_fit_multi and b7_dngo_score_multi, so
that the glue's DNGO branch for config.bot.nGPU > 1 (lua/bot7_b200/models_dngo.lua:acquire_multi) can run under tools/minilua
without a GPU.  Like FakeB7, it checks the protocol between the glue and the C ABI (handles per device, which are freed, global
numbering across the shards), not the numerics.  Never importable from the product: it lives under tests/ and needs oracle/."""
import ctypes as C

from fake_b7_lib import FakeB7, _arr


class FakeB7DngoMulti(FakeB7):
    def b7_blr_fit_multi(self, comm, Z0, y, N, D, hyp, S, out_blrs, info):
        c = self._get(comm, "comm")
        Z, yy, H = _arr(Z0, (N, D)).copy(), _arr(y, (N,)).copy(), _arr(hyp, (S, 3)).copy()
        fits = [self.o.blr_fit(Z, yy, H[s]) for s in range(S)]
        if info:
            _arr(info, (S,), C.c_int)[...] = 0
        for g in range(c["n"]):                                                # every device fits the whole head
            C.c_void_p.from_address(out_blrs + g * C.sizeof(C.c_void_p)).value = self._new({"kind": "blr", "fits": fits, "D": D})
        return 0

    def b7_dngo_score_multi(self, comm, blrs, grids, n_layers, dims, W, b, relu_last, kind, tradeoff, bound, sign, fmin, score_host, argmax,
                            argmax_original, best, nan_count):
        c = self._get(comm, "comm")
        bh = [C.c_void_p.from_address(blrs + g * C.sizeof(C.c_void_p)).value for g in range(c["n"])]
        rh = [C.c_void_p.from_address(grids + g * C.sizeof(C.c_void_p)).value for g in range(c["n"])]
        for h in bh:
            self._get(h, "blr")
        for h in rh:
            self._get(h, "grid")
        # the shard handles share one logical grid (see FakeB7.b7_grid_from_host_sharded): score it whole
        return FakeB7.b7_dngo_score(self, bh[0], rh[0], n_layers, dims, W, b, relu_last, kind, tradeoff, bound, sign, fmin, score_host, argmax,
                                    argmax_original, best, nan_count)

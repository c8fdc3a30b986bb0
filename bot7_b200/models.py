"""bot7.models -- surrogates (host-side mirror of the Lua object protocol over the C ABI).

In the reference `bot7.models` *is* gpTorch7's `gp.models` (models/init.lua:15) plus
models/dngo.lua.  The protocol kept here is the one bot7 itself uses (call sites:
bots/abstract.lua:148, bots/bayesopt.lua:65-75, scores/expected_improvement.lua:57,63):
`init`, `predict -> {mean, var}`, `sample_hypers`, `parse_hypers`, `fantasize`, `class`, `cache`,
field `hyp`.  The arithmetic follows oracle/SPEC.md (gpTorch7 is not available: declared spec).
All numerics run in libbot7_b200.so; nothing here computes a covariance or a factorisation.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib as L
from .samplers import slice as slice_sampler
from .samplers import slice_device, slice_speculative

DEVICE_STEP_MAX_N = 128    # b7_gp_slice_step: one 128 x 128 block
KERNELS = {"ardse": L.KERNEL_ARDSE, "matern52": L.KERNEL_MATERN52, "matern_52": L.KERNEL_MATERN52}


class GPFactors:
    """Handle on one batched fit: S hyper-parameter draws -> S Cholesky factors on the device."""

    def __init__(self, X, y, hyp, kernel="ardse", noiseless=False, flags=L.FIT_PREDICT, ctx=None):
        self.ctx = ctx or L.Context.default()
        X = L.as_f64(X)
        if X.ndim == 1:
            X = X.reshape(1, -1)
        y = L.as_f64(y).reshape(-1)
        hyp = np.atleast_2d(L.as_f64(hyp))
        self.N, self.d = X.shape
        self.S, H = hyp.shape
        if y.shape[0] != self.N:
            raise ValueError("X_obs and Y_obs disagree on the number of observations")
        self.hyp = hyp
        self.handle = C.c_void_p()
        info = (C.c_int * self.S)()
        self.logml = np.zeros(self.S)
        self.jitter = np.zeros(self.S)
        kid = KERNELS[kernel] if isinstance(kernel, str) else int(kernel)
        L.check(L.lib().b7_gp_fit(self.ctx.handle, kid, L.dptr(X), L.dptr(y), self.N, self.d, L.dptr(hyp), self.S, H,
                                  int(bool(noiseless)), flags, C.byref(self.handle), info, L.dptr(self.logml),
                                  L.dptr(self.jitter)), "b7_gp_fit")
        self.info = np.array(list(info), dtype=np.int32)
        for s in np.nonzero(self.jitter > 0)[0]:
            # utils/math.lua:204-215 prints a warning; same policy
            if math.isinf(self.jitter[s]):
                print("Warning: utils.math.chol failed to find a PSD version\nof the input matrix; returning chol(I).")
            else:
                print("Warning: utils.math.chol succeeded in factorizing the\ninput matrix after applying "
                      "a jitter of %.2e" % self.jitter[s])

    def refit(self, hyp, flags=L.FIT_PREDICT):
        """New hyper-parameter draws on the same observations; all device buffers are reused."""
        hyp = np.atleast_2d(L.as_f64(hyp))
        if hyp.shape != self.hyp.shape:
            raise ValueError("refit needs the same S x H shape as the original fit")
        info = (C.c_int * self.S)()
        L.check(L.lib().b7_gp_refit(self.handle, L.dptr(hyp), flags, info, L.dptr(self.logml), L.dptr(self.jitter)), "b7_gp_refit")
        self.hyp = hyp
        self.info = np.array(list(info), dtype=np.int32)
        return self

    def slice_step(self, x0, d_vec, log_u, u_right, u_shrink, width, max_step, prior_std, prior_order):
        """One directed slice step on this handle's observations in one device call (b7_gp_slice_step, N <= 128) ->
        (x1 (1 x H), shrink uniforms used, density evaluations, log p(x1)), or None when `u_shrink` ran out."""
        H = self.d + 3
        x0, d_vec, u_right = (L.as_f64(v).reshape(-1) for v in (x0, d_vec, u_right))
        u_shrink = L.as_f64(u_shrink).reshape(-1)
        if x0.size != H or d_vec.size != H or u_right.size != H:
            raise ValueError(f"slice_step: the handle's hyper-parameter rows have H = {H} entries")
        x1, used, evals, logp = np.empty((1, H)), C.c_int(), C.c_int(), C.c_double()
        rc = L.lib().b7_gp_slice_step(self.handle, L.dptr(x0), L.dptr(d_vec), float(log_u), L.dptr(u_right), L.dptr(u_shrink),
                                      u_shrink.size, float(width), float(max_step), float(prior_std), int(prior_order),
                                      L.dptr(x1), C.byref(used), C.byref(evals), C.byref(logp))
        if rc == L.ERR_STATE:
            return None
        L.check(rc, "b7_gp_slice_step")
        return x1, used.value, evals.value, logp.value

    def predict(self, s, Xs):
        Xs = L.as_f64(Xs)
        if Xs.ndim == 1:
            Xs = Xs.reshape(1, -1)
        M = Xs.shape[0]
        mean, var = np.empty(M), np.empty(M)
        L.check(L.lib().b7_gp_predict(self.handle, int(s), L.dptr(Xs), M, L.dptr(mean), L.dptr(var)), "b7_gp_predict")
        return mean, var

    def read_factor(self, s):
        """Lower triangle of draw s's factor as an N x N array: L after a fit without inversion (FIT_LOGML_ONLY /
        FIT_DEFER), L^-1 once the handle can predict."""
        out = np.empty((self.N, self.N))
        L.check(L.lib().b7_gp_read_factor(self.handle, int(s), L.dptr(out)), "b7_gp_read_factor")
        return np.tril(out)

    def padded_n(self):
        return int(L.lib().b7_gp_padded_n(self.handle))

    def device_ptr(self, what):
        p, n = C.c_void_p(), C.c_int64()
        L.check(L.lib().b7_gp_device_ptr(self.handle, what, C.byref(p), C.byref(n)))
        return p.value, n.value

    def fit_range(self, s0, count):
        info = (C.c_int * max(count, 1))()
        logml, jit = np.zeros(max(count, 1)), np.zeros(max(count, 1))
        L.check(L.lib().b7_gp_fit_range(self.handle, s0, count, info, L.dptr(logml), L.dptr(jit)), "b7_gp_fit_range")
        L.check(L.lib().b7_gp_invert_range(self.handle, s0, count), "b7_gp_invert_range")
        self.logml[s0:s0 + count] = logml[:count]
        self.jitter[s0:s0 + count] = jit[:count]
        return np.array(list(info)[:count])

    def mark_ready(self):
        L.check(L.lib().b7_gp_mark_ready(self.handle))

    def free(self):
        if getattr(self, "handle", None):
            L.lib().b7_gp_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class gp_regressor:
    """GP regression surrogate with the gp.models.gp_regressor protocol.

    config keys (bots/bayesopt.lua:38-45, examples/run_benchmark.lua:61): kernel ('ardse'), nzModel
    ('GaussianNoise_iso'), mean ('constant'), sampler ('slice'), noiseless.
    hyp vector layout (oracle/SPEC.md): [log l_1..log l_d, log sigma_f, log sigma_n, m].
    """

    def __init__(self, config=None, ctx=None, rng=None):
        c = dict(config or {})
        c.setdefault("kernel", "ardse")
        c.setdefault("nzModel", "GaussianNoise_iso")
        c.setdefault("mean", "constant")
        c.setdefault("sampler", "slice")
        c.setdefault("noiseless", False)
        c.setdefault("nSamples", 1)
        c.setdefault("burnin", 0)
        c.setdefault("prior_std", 2.0)     # declared: independent N(0, prior_std^2) on every hyp entry
        # declared initial state of the chain (bots/abstract.lua:148 model:init; gpTorch7's own values are unknown)
        c.setdefault("init_lengthscale", 0.5)
        c.setdefault("init_sigma_f", 1.0)
        c.setdefault("init_noise", None)   # sigma_n^2; None: 1e-2, or 1e-6 with `noiseless`
        c.setdefault("speculative", True)  # batched density evaluations; the chain is identical either way
        c.setdefault("spec_width", 8)     # profiles/refit_vs_width_r01.json: 8 evaluations cost 1.0-2.1x one
        # one device call per slice step (b7_gp_slice_step) for fits of up to 128 observations; the chain is identical, larger
        # fits keep the route above
        c.setdefault("device_step", False)
        self.config = c
        self.ctx = ctx
        self.rng = rng or np.random.default_rng(0)
        self.hyp = None
        self._cache_key = None
        self._factors = None
        self._density_key = None
        self._density = None

    def class_(self):
        return "gp.models.gp_regressor"

    def cache(self):
        return {"config": self.config, "hyp": self.hyp}

    # -- protocol ---------------------------------------------------------------------------
    def init(self, X, Y):
        """bots/abstract.lua:148 -- set the initial hyper-parameter state from the data."""
        X = np.atleast_2d(L.as_f64(X))
        d = X.shape[1]
        h = np.zeros(d + 3)
        noise = self.config["init_noise"]
        if noise is None:
            noise = 1e-6 if self.config["noiseless"] else 1e-2
        h[:d] = math.log(self.config["init_lengthscale"])
        h[d] = math.log(self.config["init_sigma_f"])
        h[d + 1] = 0.5 * math.log(noise)
        h[d + 2] = float(np.mean(Y))
        self.hyp = h
        return self

    def parse_hypers(self, h):
        return np.atleast_2d(L.as_f64(h))

    def log_density(self, h, X, Y):
        """log p(y | h) + log p(h): one density evaluation of the slice sampler = one GP fit
        (K build + potrf + beta + logdet) with nothing but a scalar coming back."""
        h = L.as_f64(h).reshape(1, -1)
        key = (np.asarray(X).tobytes(), np.asarray(Y).tobytes(), 1)
        if self._density_key != key:                 # X, y stay resident across the sampler's evaluations
            if self._density is not None:
                self._density.free()
            self._density = GPFactors(X, Y, h, self.config["kernel"], self.config["noiseless"], L.FIT_LOGML_ONLY, self.ctx)
            self._density_key = key
        else:
            self._density.refit(h, L.FIT_LOGML_ONLY)
        f = self._density
        lp = float(f.logml[0]) if f.info[0] == 0 and np.isfinite(f.logml[0]) else -np.inf
        sd = self.config["prior_std"]
        return lp - 0.5 * float(np.sum((h / sd) ** 2))

    def log_density_batch(self, H, X, Y):
        """k density evaluations in one device call (one batched fit of k factors): what the speculative
        sampler asks for.  The handle keeps `spec_width` slots; short batches repeat their last row."""
        H = np.atleast_2d(L.as_f64(H))
        k, W = H.shape[0], max(int(self.config["spec_width"]), 3)
        out = []
        for c0 in range(0, k, W):
            chunk = H[c0:c0 + W]
            n = chunk.shape[0]
            padded = np.concatenate([chunk, np.repeat(chunk[-1:], W - n, 0)], 0) if n < W else chunk
            key = (np.asarray(X).tobytes(), np.asarray(Y).tobytes(), W)
            if self._density_key != key:
                if self._density is not None:
                    self._density.free()
                self._density = GPFactors(X, Y, padded, self.config["kernel"], self.config["noiseless"], L.FIT_LOGML_ONLY, self.ctx)
                self._density_key = key
            else:
                self._density.refit(padded, L.FIT_LOGML_ONLY)
            f = self._density
            sd = self.config["prior_std"]
            for i in range(n):
                lp = float(f.logml[i]) if f.info[i] == 0 and np.isfinite(f.logml[i]) else -np.inf
                out.append(lp - 0.5 * float(np.sum((chunk[i] / sd) ** 2)))
        return out

    def device_step(self, X, Y, x0, d_vec, log_u, u_right, u_shrink, width, max_step):
        """One slice step in one device call on the single-slot handle of log_density (X, y resident); numpy's pairwise
        order for the prior's sum, as log_density's np.sum."""
        key = (np.asarray(X).tobytes(), np.asarray(Y).tobytes(), 1)
        if self._density_key != key:
            self.log_density(x0, X, Y)
        return self._density.slice_step(x0, d_vec, log_u, u_right, u_shrink, width, max_step, self.config["prior_std"], 1)

    def sample_hypers(self, X, Y, _a=None, _b=None, single=False):
        """bots/bayesopt.lua:68,74: slice-sample the hyper-parameter posterior, keep the chain state."""
        if self.hyp is None:
            self.init(X, Y)
        n = 1 if single else int(self.config["nSamples"])
        out = np.empty((n, self.hyp.size))
        x = self.hyp.reshape(1, -1).copy()
        device = self.config["device_step"] and np.atleast_2d(X).shape[0] <= DEVICE_STEP_MAX_N
        for i in range(n):
            if device:
                x = slice_device()(lambda *a: self.device_step(X, Y, *a), x, {"nSamples": 1}, None, rng=self.rng)
            elif self.config["speculative"]:
                x = slice_speculative()(lambda V, a: self.log_density_batch(V, X, Y), x, {"nSamples": 1}, None,
                                        rng=self.rng, width=int(self.config["spec_width"]))
            else:
                x = slice_sampler()(lambda v, a: self.log_density(v, X, Y), x, {"nSamples": 1}, None, rng=self.rng)
            out[i] = x[0]
        self.hyp = out[-1].copy()
        return out[0] if single else out

    def _fit(self, X0, Y0, hyp):
        hyp = self.parse_hypers(self.hyp if hyp is None else hyp)
        key = (np.asarray(X0).tobytes(), np.asarray(Y0).tobytes(), hyp.tobytes())
        if key != self._cache_key:
            if self._factors is not None:
                self._factors.free()
            self._factors = GPFactors(X0, Y0, hyp, self.config["kernel"], self.config["noiseless"], L.FIT_PREDICT, self.ctx)
            self._cache_key = key
        return self._factors

    def factors(self, X0, Y0, hyp=None) -> GPFactors:
        return self._fit(L.as_f64(X0), L.as_f64(Y0), hyp)

    def predict(self, X0, Y0, X1, hyp=None, req=None):
        """model:predict(X_obs, Y_obs, X_hid, hyp, {mean=true, var=true}) -> {mean=, var=} (M x 1 each)."""
        f = self._fit(L.as_f64(X0), L.as_f64(Y0), hyp)
        mean, var = f.predict(0, X1)
        out = {}
        if req is None or req.get("mean", True):
            out["mean"] = mean.reshape(-1, 1)
        if req is None or req.get("var", True):
            out["var"] = var.reshape(-1, 1)
        return out

    def fantasize(self, n, X0, Y0, Xp, hyp=None):
        """Y_pend ~ N(mean, var) at the pending points (independent marginals; host RNG)."""
        p = self.predict(X0, Y0, Xp, hyp)
        z = self.rng.standard_normal((p["mean"].shape[0], int(n)))
        return p["mean"] + np.sqrt(p["var"]) * z


class BLRFactors:
    def __init__(self, Z0, y, hyp, ctx=None):
        self.ctx = ctx or L.Context.default()
        Z0 = np.atleast_2d(L.as_f64(Z0))
        y = L.as_f64(y).reshape(-1)
        hyp = np.atleast_2d(L.as_f64(hyp))
        if hyp.shape[1] != 3:
            raise ValueError("BLR hyp rows are [log alpha_p, log beta, m]")
        self.N, self.D = Z0.shape
        self.S = hyp.shape[0]
        self.hyp = hyp
        self.handle = C.c_void_p()
        info = (C.c_int * self.S)()
        L.check(L.lib().b7_blr_fit(self.ctx.handle, L.dptr(Z0), L.dptr(y), self.N, self.D, L.dptr(hyp), self.S,
                                   C.byref(self.handle), info), "b7_blr_fit")
        self.info = np.array(list(info))
        self.logev = None

    def refit(self, hyp, flags=L.FIT_PREDICT):
        """New S x 3 rows on the same features and responses (all device buffers reused) -> (logev, info):
        log p(y | row) per row (-inf where info != 0).  FIT_LOGML_ONLY leaves the handle unable to predict until the
        next FIT_PREDICT refit."""
        hyp = np.atleast_2d(L.as_f64(hyp))
        if hyp.shape != self.hyp.shape:
            raise ValueError("refit needs the same S x 3 shape as the original fit")
        info = (C.c_int * self.S)()
        self.logev = np.empty(self.S)
        L.check(L.lib().b7_blr_refit(self.handle, L.dptr(hyp), flags, info, L.dptr(self.logev)), "b7_blr_refit")
        self.hyp = hyp
        self.info = np.array(list(info))
        return self.logev, self.info

    def predict(self, s, Z1):
        Z1 = np.atleast_2d(L.as_f64(Z1))
        M = Z1.shape[0]
        mean, var = np.empty(M), np.empty(M)
        L.check(L.lib().b7_blr_predict(self.handle, int(s), L.dptr(Z1), M, L.dptr(mean), L.dptr(var)), "b7_blr_predict")
        return mean, var

    def free(self):
        if getattr(self, "handle", None):
            L.lib().b7_blr_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def act_codes(act, n):
    """n activation codes (L.ACT_NONE / ACT_RELU / ACT_TANH, one per layer) as a C int array; an unknown code is the library's
    to refuse."""
    if len(act) != n:
        raise ValueError(f"act: {len(act)} codes for {n} layers")
    return (C.c_int * n)(*[int(a) for a in act])


def mlp_features(grid, weights, biases, relu_last=True, ctx=None, act=None):
    """DNGO basis on the device (models/dngo.lua:164-171 without the 32-row minibatch loop and without
    the host round trip of Z1): MLP forward of a DeviceGrid, returns a DeviceGrid of features.
    weights[l]: (h_out x h_in) like torch nn.Linear.weight; biases[l]: (h_out,).
    act: one code per layer (b7_mlp_features_act); None is the relu_last form (b7_mlp_features)."""
    from .grids import DeviceGrid
    ctx = ctx or grid.ctx
    Ws = [L.as_f64(w) for w in weights]
    bs = [L.as_f64(b).reshape(-1) for b in biases]
    n = len(Ws)
    dims = (C.c_int * (n + 1))(*([Ws[0].shape[1]] + [w.shape[0] for w in Ws]))
    Wp = (C.POINTER(C.c_double) * n)(*[L.dptr(w) for w in Ws])
    bp = (C.POINTER(C.c_double) * n)(*[L.dptr(b) for b in bs])
    out = C.c_void_p()
    if act is None:
        L.check(L.lib().b7_mlp_features(ctx.handle, grid.handle, n, dims, Wp, bp, int(bool(relu_last)), C.byref(out)), "b7_mlp_features")
    else:
        L.check(L.lib().b7_mlp_features_act(ctx.handle, grid.handle, n, dims, Wp, bp, act_codes(act, n), C.byref(out)),
                "b7_mlp_features_act")
    return DeviceGrid(out, ctx)


def dngo_score(blr, grid, weights, biases, relu_last=True, kind=L.SCORE_EI, tradeoff=0.0, bound=0, sign=-1.0, fmin=0.0,
               want_scores=False, act=None):
    """dngo:predict + score + argmax over a device grid in one pass (b7_dngo_score; models/dngo.lua:155-174): the basis is
    evaluated in front of the BLR head tile by tile, the feature matrix Z1 is never stored.
    act: one code per layer (b7_dngo_score_act); None is the relu_last form.
    Returns (scores or None, argmax (compacted), argmax_original, best, nan_count)."""
    Ws = [L.as_f64(w) for w in weights]
    bs = [L.as_f64(b).reshape(-1) for b in biases]
    n = len(Ws)
    dims = (C.c_int * (n + 1))(*([Ws[0].shape[1]] + [w.shape[0] for w in Ws]))
    Wp = (C.POINTER(C.c_double) * n)(*[L.dptr(w) for w in Ws])
    bp = (C.POINTER(C.c_double) * n)(*[L.dptr(b) for b in bs])
    sc = np.empty(grid.rows()) if want_scores else None
    am, amo, best, nn = C.c_int64(), C.c_int64(), C.c_double(), C.c_int64()
    if act is None:
        L.check(L.lib().b7_dngo_score(blr.handle, grid.handle, n, dims, Wp, bp, int(bool(relu_last)), kind, tradeoff, bound, sign, fmin,
                                      L.dptr(sc), C.byref(am), C.byref(amo), C.byref(best), C.byref(nn)), "b7_dngo_score")
    else:
        L.check(L.lib().b7_dngo_score_act(blr.handle, grid.handle, n, dims, Wp, bp, act_codes(act, n), kind, tradeoff, bound, sign, fmin,
                                          L.dptr(sc), C.byref(am), C.byref(amo), C.byref(best), C.byref(nn)), "b7_dngo_score_act")
    return sc, am.value, amo.value, best.value, nn.value


class bayes_linear:
    """gp.models.bayes_linear as used by models/dngo.lua:77-79,174:
    predict(Z0, Y0, Z1, nil, hyp, req) with hyp == 'marginalize' or a S x 3 array.

    config keys: alpha_p (1), beta (1e2) -- the fixed row [log alpha_p, log beta, mean(Y0)] that 'marginalize' uses by
    default; sampler (None; 'slice': 'marginalize' averages over `nSamples` successive states of a slice-sampling chain on
    log p(y | h) + log p(h), started at the fixed row and kept across calls like gp_regressor.sample_hypers keeps its
    chain), nSamples (10), prior_std (2), speculative (True), spec_width (8), burnin (0: chain steps discarded when the
    chain starts).
    """

    def __init__(self, config=None, ctx=None, rng=None):
        c = dict(config or {})
        c.setdefault("alpha_p", 1.0)
        c.setdefault("beta", 1e2)
        c.setdefault("sampler", None)
        c.setdefault("nSamples", 10)
        c.setdefault("prior_std", 2.0)     # declared: independent N(0, prior_std^2) on every hyp entry, as for the GP
        c.setdefault("speculative", True)  # batched density evaluations; the chain is identical either way
        c.setdefault("spec_width", 8)
        c.setdefault("burnin", 0)
        self.config = c
        self.ctx = ctx
        self.rng = rng or np.random.default_rng(0)
        self.hyp = None
        self._density_key = None
        self._density = None

    def class_(self):
        return "gp.models.bayes_linear"

    def default_hyp(self, Y0):
        return np.array([[math.log(self.config["alpha_p"]), math.log(self.config["beta"]), float(np.mean(Y0))]])

    def _density_handle(self, Z0, Y0, rows, W):
        """The resident handle of W slots for (Z0, Y0), refitted to `rows` (W x 3) for the log evidence only."""
        key = (np.asarray(Z0).tobytes(), np.asarray(Y0).tobytes(), W)
        if self._density_key != key:                 # Z0, y and the Gram partials stay resident across the evaluations
            if self._density is not None:
                self._density.free()
            self._density = BLRFactors(Z0, Y0, rows, self.ctx)
            self._density_key = key
        self._density.refit(rows, L.FIT_LOGML_ONLY)
        return self._density

    def log_density(self, h, Z0, Y0):
        """log p(y | h) + log p(h): one density evaluation of the slice sampler on a single-slot handle."""
        h = L.as_f64(h).reshape(1, -1)
        f = self._density_handle(Z0, Y0, h, 1)
        lp = float(f.logev[0]) if f.info[0] == 0 and np.isfinite(f.logev[0]) else -np.inf
        sd = self.config["prior_std"]
        return lp - 0.5 * float(np.sum((h / sd) ** 2))

    def log_density_batch(self, H, Z0, Y0):
        """k density evaluations in one device call per `spec_width` rows: what the speculative sampler asks for.
        The handle keeps `spec_width` slots; short batches repeat their last row."""
        H = np.atleast_2d(L.as_f64(H))
        k, W = H.shape[0], max(int(self.config["spec_width"]), 3)
        out = []
        for c0 in range(0, k, W):
            chunk = H[c0:c0 + W]
            n = chunk.shape[0]
            padded = np.concatenate([chunk, np.repeat(chunk[-1:], W - n, 0)], 0) if n < W else chunk
            f = self._density_handle(Z0, Y0, padded, W)
            sd = self.config["prior_std"]
            for i in range(n):
                lp = float(f.logev[i]) if f.info[i] == 0 and np.isfinite(f.logev[i]) else -np.inf
                out.append(lp - 0.5 * float(np.sum((chunk[i] / sd) ** 2)))
        return out

    def _step(self, x, Z0, Y0):
        if self.config["speculative"]:
            return slice_speculative()(lambda V, a: self.log_density_batch(V, Z0, Y0), x, {"nSamples": 1}, None,
                                       rng=self.rng, width=int(self.config["spec_width"]))
        return slice_sampler()(lambda v, a: self.log_density(v, Z0, Y0), x, {"nSamples": 1}, None, rng=self.rng)

    def sample_hypers(self, Z0, Y0, single=False):
        """Slice-sample the (alpha_p, beta, m) posterior; the chain starts at the fixed row and its state is kept."""
        Z0 = np.atleast_2d(L.as_f64(Z0))
        Y0 = L.as_f64(Y0).reshape(-1)
        if self.hyp is None:
            x = self.default_hyp(Y0)
            for _ in range(int(self.config["burnin"])):
                x = self._step(x, Z0, Y0)
            self.hyp = x[0].copy()
        n = 1 if single else int(self.config["nSamples"])
        out = np.empty((n, self.hyp.size))
        x = self.hyp.reshape(1, -1).copy()
        for i in range(n):
            x = self._step(x, Z0, Y0)
            out[i] = x[0]
        self.hyp = out[-1].copy()
        return out[0] if single else out

    def factors(self, Z0, Y0, hyp=None) -> BLRFactors:
        if hyp is None or (isinstance(hyp, str) and hyp == "marginalize"):
            if self.config["sampler"] == "slice":
                hyp = self.sample_hypers(Z0, Y0)
            else:
                hyp = self.hyp if self.hyp is not None else self.default_hyp(Y0)
        return BLRFactors(Z0, Y0, hyp, self.ctx)

    def predict(self, Z0, Y0, Z1, _unused=None, hyp=None, req=None):
        f = self.factors(Z0, Y0, hyp)
        means, vars_ = zip(*[f.predict(s, Z1) for s in range(f.S)])
        f.free()
        return {"mean": np.mean(means, axis=0).reshape(-1, 1), "var": np.mean(vars_, axis=0).reshape(-1, 1)}


class dngo:
    """models/dngo.lua BLR head only (SURVEY a-16): `basis` maps X -> features (the trained network of
    the reference, models/dngo.lua:83-105,155-171, is out of scope and is passed in as a callable)."""

    def __init__(self, config=None, basis=None, ctx=None, rng=None):
        self.config = dict(config or {})
        self.basis = basis
        self.predictor = bayes_linear(self.config.get("predictor"), ctx, rng)

    def class_(self):
        return "bot7.models.dngo"

    def init(self, X, Y):
        return self

    def predict(self, X0, Y0, X1, hyp=None, req=None):
        hyp = "marginalize" if hyp is None else hyp          # models/dngo.lua:110
        Z0 = self.basis(np.atleast_2d(L.as_f64(X0)))         # :155-162
        Z1 = self.basis(np.atleast_2d(L.as_f64(X1)))         # :165-171
        return self.predictor.predict(Z0, Y0, Z1, None, hyp, req)   # :174

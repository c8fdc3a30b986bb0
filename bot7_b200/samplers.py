"""bot7.samplers.slice -- host control flow of reference samplers/slice.lua (SURVEY a-15).

Strictly sequential; every call of `f` is one device evaluation (for GP hyper-parameters: one
b7_gp_fit with B7_FIT_LOGML_ONLY).  The RNG is host state (torch MT19937 in the reference, numpy
here) and is not reproduced; the control flow is.
"""
from __future__ import annotations

import copy

import numpy as np


class slice:  # noqa: A001  (name kept from the reference)
    def __call__(self, f, X0, opt=None, f_args=None, rng=None):
        opt = self.configure(opt)                                   # samplers/slice.lua:26
        return self.sample(f, X0, opt, f_args, rng or np.random.default_rng())

    @staticmethod
    def configure(opt=None):
        """samplers/slice.lua:32-48."""
        opt = dict(opt or {})
        opt["max_step"] = opt.get("max_step") or 1e3
        opt["nSamples"] = opt.get("nSamples") or 1
        if opt.get("step_out") is not False:
            opt["step_out"] = True
        if opt.get("logspace") is not False:
            opt["logspace"] = True
        return opt

    @staticmethod
    def sample(f, X0, opt, f_args, rng):
        """samplers/slice.lua:51-89."""
        X0 = np.atleast_2d(np.asarray(X0, dtype=np.float64))
        X0 = np.tile(X0.copy(), (int(opt["nSamples"]), 1))
        N, xDim = X0.shape
        samples = np.empty((N, xDim))
        if opt.get("gibbs"):
            for n in range(N):
                x0 = X0[n:n + 1]
                x1 = np.zeros((1, xDim))
                d_vec = np.zeros((1, xDim))
                order = rng.permutation(xDim)
                for itr in range(xDim):
                    d = order[itr]
                    d_vec[0, d] = 1.0
                    x1[0, d] = slice.directed_slice(opt, f, f_args, d_vec, x0, rng)[0, d]
                    d_vec[0, d] = 0.0
                samples[n] = x1
        else:
            for n in range(N):
                x0 = X0[n:n + 1]
                d_vec = rng.standard_normal((1, xDim))
                d_vec = d_vec / np.linalg.norm(d_vec)
                samples[n] = slice.directed_slice(opt, f, f_args, d_vec, x0, rng)
        return samples

    @staticmethod
    def directed_slice(opt, f, f_args, d_vec, x0, rng):
        """samplers/slice.lua:92-168."""
        xDim = x0.shape[1]
        stepsize = opt.get("widths")
        if stepsize is None:
            stepsize = np.full((1, xDim), opt.get("width") or 1.0)   # :95

        def f_dx(dx=None):                                            # :100-103
            dx = np.zeros((1, xDim)) if dx is None else dx
            return f(x0 + d_vec * dx, f_args)

        Y = f_dx()                                                    # :106
        if opt["logspace"]:
            Y = Y + np.log(rng.random())                              # :108
        else:
            Y = Y * rng.random()
        right = rng.random((1, xDim)) * stepsize                      # :114
        left = right - stepsize                                       # :115
        if opt["step_out"]:                                           # :118-130
            itr = 0
            while f_dx(right) > Y and itr < opt["max_step"]:
                itr += 1
                right = right + stepsize
            itr = 0
            while f_dx(left) > Y and itr < opt["max_step"]:
                itr += 1
                left = left - stepsize
        dx = np.zeros((1, xDim))
        while True:                                                   # :134-164
            dx = left + (right - left) * rng.random()
            y = f_dx(dx)
            if y != y:                                                # :139-142
                print("Error: samplers.slice encountered a NaN")
                break
            if y > Y:                                                 # :144
                break
            if (dx == 0.0).any():                                     # :148-151
                print("Error: samplers.slice shrank to zero")
                break
            pos = dx > 0                                              # :153-161
            right = np.where(pos, dx, right)
            neg = dx < 0
            left = np.where(neg, dx, left)
        return x0 + d_vec * dx


class slice_speculative(slice):
    """Same chain as `slice`, fewer sequential density evaluations (SURVEY section 8f rank 1).

    The reference sampler (samplers/slice.lua:92-168) calls `f` strictly one point at a time, and for
    GP hyper-parameters every call is a device fit whose cost at small and medium N is launch latency,
    not arithmetic.  Here `f_batch(points[k x h]) -> k values` evaluates several points in one device
    call (one batched fit), and the control flow asks for points *before* it knows it needs them:

      * the current point, the first right and the first left bracket end (their positions depend on the
        RNG only) go out as one batch;
      * stepping out evaluates the next `width` ends of the side being extended at once;
      * stepping in pre-computes the next `width` proposals under the assumption that each one is
        rejected (the bracket update after a rejection depends only on the sign of the proposal).

    Speculative results that the sequential algorithm would not have requested are discarded, and the
    RNG is rewound to exactly the state the sequential algorithm would have left it in, so for a given
    generator the samples are bit-identical to `slice` (tests/test_host_logic.py).
    """

    def __call__(self, f_batch, X0, opt=None, f_args=None, rng=None, width=4):
        opt = self.configure(opt)
        rng = rng or np.random.default_rng()
        X0 = np.atleast_2d(np.asarray(X0, dtype=np.float64))
        X0 = np.tile(X0.copy(), (int(opt["nSamples"]), 1))
        N, xDim = X0.shape
        samples = np.empty((N, xDim))
        self.calls = 0          # device calls (batches)
        self.evals = 0          # points evaluated, speculative ones included
        if opt.get("gibbs"):
            raise NotImplementedError("gibbs sweeps use the sequential sampler")
        for n in range(N):
            x0 = X0[n:n + 1]
            d_vec = rng.standard_normal((1, xDim))
            d_vec = d_vec / np.linalg.norm(d_vec)
            samples[n] = self._directed(opt, f_batch, f_args, d_vec, x0, rng, int(width))
        return samples

    def _eval(self, f_batch, f_args, x0, d_vec, dxs):
        pts = np.concatenate([x0 + d_vec * dx for dx in dxs], 0)
        self.calls += 1
        self.evals += len(dxs)
        return [float(v) for v in f_batch(pts, f_args)]

    def _propose(self, rng, left, right, width):
        """`width` shrink proposals under the assumption that each earlier one is rejected; records the RNG state
        after every draw so that the caller can rewind to exactly where the sequential algorithm would be."""
        l, r, props, states = left, right, [], []
        for _ in range(width):
            u = rng.random()
            states.append(rng.bit_generator.state)
            p = l + (r - l) * u
            props.append((p, l, r))
            if (p == 0.0).any():
                break
            r = np.where(p > 0, p, r)
            l = np.where(p < 0, p, l)
        return props, states

    def _directed(self, opt, f_batch, f_args, d_vec, x0, rng, width):
        xDim = x0.shape[1]
        stepsize = opt.get("widths")
        if stepsize is None:
            stepsize = np.full((1, xDim), opt.get("width") or 1.0)
        zero = np.zeros((1, xDim))
        # RNG order of the reference: log U (:108), then the bracket (:114)
        logu = np.log(rng.random()) if opt["logspace"] else rng.random()
        right = rng.random((1, xDim)) * stepsize
        left = right - stepsize
        # first device call: the point itself, both bracket ends, and -- betting that no stepping out will be
        # needed -- the first shrink proposals for this bracket (stepping out draws no random numbers, so the
        # proposals are the ones the sequential algorithm would make if the bet holds)
        state0 = rng.bit_generator.state
        props, states = self._propose(rng, left, right, max(width - 3, 1))
        vals = self._eval(f_batch, f_args, x0, d_vec, [zero, right, left] + [p for p, _, _ in props])
        f0, fr, fl, ys = vals[0], vals[1], vals[2], vals[3:]
        Y = f0 + logu if opt["logspace"] else f0 * logu
        pending = (props, states, ys)
        if opt["step_out"] and (fr > Y or fl > Y):
            pending = None                           # bet lost: discard the proposals, rewind the RNG
            rng.bit_generator.state = state0
            for side in (+1, -1):
                end, fe, itr = (right, fr, 0) if side > 0 else (left, fl, 0)
                cache = []
                while fe > Y and itr < opt["max_step"]:
                    itr += 1
                    end = end + side * stepsize
                    if not cache:
                        ends, e = [], end
                        for _ in range(width):        # repeated addition, exactly like the sequential loop
                            ends.append(e)
                            e = e + side * stepsize
                        cache = list(zip(ends, self._eval(f_batch, f_args, x0, d_vec, ends)))
                    end, fe = cache.pop(0)
                if side > 0:
                    right = end
                else:
                    left = end
        dx = zero
        while True:
            if pending is not None:
                props, states, ys = pending
                pending = None
            else:
                props, states = self._propose(rng, left, right, width)
                ys = self._eval(f_batch, f_args, x0, d_vec, [p for p, _, _ in props])
            done = False
            for (p, l_before, r_before), y, st in zip(props, ys, states):
                dx, left, right = p, l_before, r_before
                rng.bit_generator.state = st          # RNG exactly as after this proposal's draw
                if y != y:
                    print("Error: samplers.slice encountered a NaN")
                    done = True
                    break
                if y > Y:
                    done = True
                    break
                if (dx == 0.0).any():
                    print("Error: samplers.slice shrank to zero")
                    done = True
                    break
                right = np.where(dx > 0, dx, right)
                left = np.where(dx < 0, dx, left)
            if done:
                break
        return x0 + d_vec * dx


class slice_device(slice):
    """Same chain as `slice`, one device call per step: `step` runs the whole directed slice step (b7_gp_slice_step).

    The generator stays on the host.  Each step pre-draws, from a copy of it, what the sequential sampler would consume in its
    order -- H normals for the direction, one uniform for the level, H for the bracket, then `k` shrink uniforms -- and passes
    the normalised direction, log U and the uniforms to `step(x0, d_vec, log_u, u_right, u_shrink, width, max_step)`, which
    returns (x1, shrink uniforms used, density evaluations, log p(x1)), or None when the `k` shrink uniforms ran out (the step
    is then made again from the same draws with twice as many).  The real generator then advances by exactly what the
    sequential sampler would have drawn, so for a given generator the samples are bit-identical to `slice`.  The NaN exit
    prints the reference's message; the shrink-to-zero exit ends the step the same way but is not reported.  Gibbs sweeps and
    per-dimension `widths` stay on the other samplers.
    """

    def __call__(self, step, X0, opt=None, f_args=None, rng=None, k=16):
        opt = self.configure(opt)
        rng = rng or np.random.default_rng()
        if opt.get("gibbs") or opt.get("widths") is not None or not opt["logspace"] or not opt["step_out"]:
            raise NotImplementedError("the device step runs the log-space directed step with step-out and a scalar width")
        X0 = np.atleast_2d(np.asarray(X0, dtype=np.float64))
        X0 = np.tile(X0.copy(), (int(opt["nSamples"]), 1))
        N, xDim = X0.shape
        samples = np.empty((N, xDim))
        self.calls = 0          # device calls (one per step, more when the shrink uniforms ran out)
        self.evals = 0          # density evaluations
        width = float(opt.get("width") or 1.0)
        for n in range(N):
            x0 = X0[n:n + 1]
            while True:
                r = copy.deepcopy(rng)
                d_vec = r.standard_normal((1, xDim))
                d_vec = d_vec / np.linalg.norm(d_vec)
                log_u = float(np.log(r.random()))
                u_right = r.random((1, xDim))
                res = step(x0, d_vec, log_u, u_right, r.random(int(k)), width, float(opt["max_step"]))
                self.calls += 1
                if res is not None:
                    break
                k = 2 * int(k)
            x1, used, evals, logp = res
            self.evals += evals
            if logp != logp:
                print("Error: samplers.slice encountered a NaN")
            rng.standard_normal((1, xDim))
            rng.random()
            rng.random((1, xDim))
            rng.random(used)
            samples[n] = x1
        return samples

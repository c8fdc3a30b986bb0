"""The reference BLR log evidence (tests/blr_evidence_oracle.py:blr_log_evidence, the density the DNGO head's hyper-parameter
chain samples) against independent evaluations, and the host side of that chain.  CPU only.

* 50-digit mpmath evaluation of log N(y; m 1, beta^-1 I + alpha_p^-1 Z0 Z0^T), the Gaussian marginal the declared formula
  restates (N x N covariance, no Cholesky of A, no w);
* the closed form at D = 1;
* the speculative slice sampler driven by the oracle density walks the sequential sampler's chain;
* the opt-in defaults of bayes_linear and the Lua glue (static).
"""
import math
import os

import numpy as np
import pytest

from blr_evidence_oracle import blr_log_evidence

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALPHAS = [1e-3, 1e-1, 1.0, 1e2]
BETAS = [1e-1, 1.0, 1e2, 1e4]


def _features(N, D, seed):
    r = np.random.default_rng(seed)
    X = r.uniform(-1, 1, (N, 3))
    Z = np.maximum(X @ r.standard_normal((3, D)) + 0.3 * r.standard_normal(D), 0.0)
    y = np.sin(3 * X[:, 0]) + X[:, 1] * X[:, 2] + 0.05 * r.standard_normal(N)
    return Z, y


def _mp_log_evidence(Z, y, alpha_p, beta, m):
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 50
    N, D = Z.shape
    Zm = mp.matrix(Z.tolist())
    a, b = mp.mpf(alpha_p), mp.mpf(beta)
    C = Zm * Zm.T / a
    for i in range(N):
        C[i, i] += 1 / b
    r = mp.matrix([mp.mpf(v) - mp.mpf(m) for v in y])
    q = (r.T * mp.lu_solve(C, r))[0]
    return -q / 2 - mp.log(mp.det(C)) / 2 - N * mp.log(2 * mp.pi) / 2


@pytest.mark.parametrize("D", [1, 6])
def test_log_evidence_against_50_digits(oracle, D):
    N = 40
    Z, y = _features(N, D, 10 + D)
    m = float(y.mean()) + 0.37                      # off the data mean: r^T r is not the centred sum of squares
    worst = 0.0
    for alpha_p in ALPHAS:
        for beta in BETAS:
            got = blr_log_evidence(Z, y, [math.log(alpha_p), math.log(beta), m])
            # the row carries log alpha_p, log beta: the reference value is taken at the same rounded exponentials
            ref = _mp_log_evidence(Z, y, math.exp(math.log(alpha_p)), math.exp(math.log(beta)), m)
            err = abs(got - float(ref)) / max(abs(float(ref)), N)
            worst = max(worst, err)
            assert err <= 1e-12, (alpha_p, beta, got, float(ref))
    print(f"D={D}: worst error {worst:.2e} of max(|log p|, N)")


def test_log_evidence_closed_form_d1(oracle):
    mp = pytest.importorskip("mpmath")
    mp.mp.dps = 40
    N = 40
    Z, y = _features(N, 1, 3)
    z = [mp.mpf(v) for v in Z[:, 0]]
    for alpha_p in ALPHAS:
        for beta in BETAS:
            m = float(y.mean()) - 0.21
            a, b = mp.mpf(math.exp(math.log(alpha_p))), mp.mpf(math.exp(math.log(beta)))
            r = [mp.mpf(v) - mp.mpf(m) for v in y]
            s = mp.fsum(v * v for v in z)
            zr = mp.fsum(p * q for p, q in zip(z, r))
            rr = mp.fsum(v * v for v in r)
            # y ~ N(m, beta^-1 I + alpha_p^-1 z z^T): det = beta^-N (1 + beta s / alpha_p), inverse by Sherman-Morrison
            ref = (N * mp.log(b) / 2 - mp.log(1 + b * s / a) / 2 - b * rr / 2 + b * b * zr * zr / (2 * (a + b * s))
                   - N * mp.log(2 * mp.pi) / 2)
            got = blr_log_evidence(Z, y, [math.log(alpha_p), math.log(beta), m])
            assert abs(got - float(ref)) <= 1e-12 * max(abs(float(ref)), N), (alpha_p, beta)


def test_log_evidence_failures_are_minus_inf(oracle):
    Z, y = _features(30, 4, 5)
    assert blr_log_evidence(Z, y, [800.0, 0.0, 0.0]) == -math.inf          # alpha_p = exp(800) overflows
    assert blr_log_evidence(Z, y, [800.0, -800.0, 0.0]) == -math.inf
    lp = blr_log_evidence(Z, y, [0.0, -800.0, 0.0])                       # beta underflows to 0: finite, tiny
    assert math.isfinite(lp) and lp < -1e3 * 30 / 2 * 0.7


@pytest.mark.parametrize("width", [1, 3, 8])
def test_speculative_chain_on_the_oracle_density_is_the_sequential_one(oracle, width):
    from bot7_b200 import samplers
    Z, y = _features(60, 5, 7)

    def dens(h):
        h = np.asarray(h, dtype=np.float64).reshape(-1)
        return blr_log_evidence(Z, y, h) - 0.5 * float(np.sum((h / 2.0) ** 2))
    x0 = np.array([[0.0, math.log(1e2), float(y.mean())]])
    seq, spec = [], []
    rng_a, rng_b = np.random.default_rng(4), np.random.default_rng(4)
    xa, xb = x0.copy(), x0.copy()
    for _ in range(12):
        xa = samplers.slice()(lambda v, a: dens(v), xa, {"nSamples": 1}, None, rng=rng_a)
        xb = samplers.slice_speculative()(lambda V, a: [dens(v) for v in V], xb, {"nSamples": 1}, None, rng=rng_b, width=width)
        seq.append(xa[0].copy())
        spec.append(xb[0].copy())
    assert np.array_equal(np.array(seq), np.array(spec))
    assert rng_a.random() == rng_b.random()
    assert not np.array_equal(seq[-1], x0[0])


def test_bayes_linear_sampling_is_opt_in():
    from bot7_b200 import models
    c = models.bayes_linear().config
    assert c["sampler"] is None and c["alpha_p"] == 1.0 and c["beta"] == 1e2
    assert (c["nSamples"], c["prior_std"], c["speculative"], c["spec_width"], c["burnin"]) == (10, 2.0, True, 8, 0)
    assert models.bayes_linear({"sampler": "slice", "nSamples": 4}).config["nSamples"] == 4


def test_lua_glue_samples_only_when_asked():
    text = open(os.path.join(ROOT, "lua", "bot7_b200", "models_dngo.lua")).read()
    assert "function dngo:sample_blr_hypers(" in text and "function dngo:blr_log_density_batch(" in text
    assert "B.C.b7_blr_refit(" in text and "B.C.B7_FIT_LOGML_ONLY" in text
    assert "chain_config(self).sampler == 'slice'" in text and "require('bot7_b200.sampler_spec')" in text

"""Reference evaluation of the DNGO head's log evidence -- TEST INFRASTRUCTURE, like oracle/ (nothing in bot7_b200/ imports it).

The density the hyper-parameter chain of the BLR head samples (declared arithmetic, DESIGN.md section 4.5; the BLR head's other
forms are oracle/SPEC.md's, gpTorch7 being absent -- PARITY UNPINNED), in the direct form, on top of the oracle's jitter
Cholesky.  Needs oracle/ on sys.path (tests/conftest.py puts it there)."""
import math

import numpy as np
import scipy.linalg as sla

import b7_oracle


def blr_log_evidence(Z0, y, hyp):
    """DECLARED. log p(y | h) of the BLR head, h = [log alpha_p, log beta, m]:
    D/2 log alpha_p + N/2 log beta - E - sum_i log (L_A)_ii - N/2 log 2 pi with E = beta/2 |r - Z0 w|^2 + alpha_p/2 |w|^2,
    r = y - m, the residual formed explicitly and L_A from the oracle's chol_jitter.  A factorisation that needs jitter (the
    device does not retry) or a non-finite value gives -inf."""
    Z0 = np.asarray(Z0, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64).reshape(-1)
    hyp = np.asarray(hyp, dtype=np.float64).reshape(-1)
    N, D = Z0.shape
    with np.errstate(all="ignore"):
        alpha_p, beta, m = float(np.exp(hyp[0])), float(np.exp(hyp[1])), float(hyp[2])   # overflow -> inf, as exp() on the device
        A = beta * (Z0.T @ Z0) + alpha_p * np.eye(D)
        if not np.isfinite(A).all():
            return -math.inf
        L, jit, _ = b7_oracle.chol_jitter(A)
        if jit != 0.0:
            return -math.inf
        r = y - m
        w = sla.solve_triangular(L.T, sla.solve_triangular(L, beta * (Z0.T @ r), lower=True), lower=False)
        res = r - Z0 @ w
        E = 0.5 * beta * float(res @ res) + 0.5 * alpha_p * float(w @ w)
        lp = 0.5 * D * hyp[0] + 0.5 * N * hyp[1] - E - float(np.log(np.diag(L)).sum()) - 0.5 * N * b7_oracle.LOG2PI
    return lp if math.isfinite(lp) else -math.inf

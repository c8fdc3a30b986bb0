"""Reference for the per-layer activations of the DNGO basis (B7_ACT_NONE / RELU / TANH), used by tests/test_gpu_dngo_act.py and
tests/fake_b7_act.py.  DECLARED semantics (the reference's nnTools/builder.lua is not in the tree): each nn.Linear (x W^T + b)
is followed by its code's activation -- ACT_NONE nothing, ACT_RELU Torch7 nn.ReLU max(0, x), ACT_TANH Torch7 nn.Tanh tanh(x)
element-wise.  The ReLU-only stacks are oracle/b7_oracle.py's mlp_features; this module adds the other codes without
changing it.  Never importable from the product: it lives under tests/."""
import numpy as np

ACT_NONE, ACT_RELU, ACT_TANH = 0, 1, 2


def mlp_features(X, weights, biases, act):
    """Output of the last Linear of the stack after its activation; act holds one code per layer."""
    if len(act) != len(weights) or any(a not in (ACT_NONE, ACT_RELU, ACT_TANH) for a in act):
        raise ValueError(f"mlp_features: act must hold one of ACT_NONE / ACT_RELU / ACT_TANH per layer (got {list(act)})")
    Z = np.asarray(X, dtype=np.float64)
    for l, (W, b) in enumerate(zip(weights, biases)):
        Z = Z @ np.asarray(W, dtype=np.float64).T + np.asarray(b, dtype=np.float64).reshape(1, -1)
        if act[l] == ACT_RELU:
            Z = np.maximum(Z, 0.0)
        elif act[l] == ACT_TANH:
            Z = np.tanh(Z)
    return Z

"""Host bookkeeping of samplers.slice_device (CPU): with a step that replays samplers/slice.lua's directed step from the numbers it
is given, the device sampler walks the sequential sampler's chain and leaves the generator where the sequential sampler does,
also when steps run out of shrink uniforms and are made again."""
import numpy as np
import pytest

from bot7_b200.samplers import slice as slice_sampler
from bot7_b200.samplers import slice_device


def logp(x):
    """A correlated 2-D Gaussian with a hole: points with x_0 > 1.5 have density -inf."""
    x = np.asarray(x).reshape(-1)
    if x[0] > 1.5:
        return -np.inf
    return float(-0.5 * (x[0] ** 2 + 4.0 * (x[1] - 0.5 * x[0]) ** 2))


def replay_step(x0, d_vec, log_u, u_right, u_shrink, width, max_step):
    """samplers/slice.lua:92-168 on the given random numbers -> (x1, shrink uniforms used, evaluations, log p(x1)), or None."""
    f = lambda dx: logp(x0 + d_vec * dx)  # noqa: E731
    Y = f(np.zeros_like(x0)) + log_u
    evals = 1
    right = u_right * width
    left = right - width
    for side in (1, -1):
        itr = 0
        while True:
            end = right if side > 0 else left
            evals += 1
            if not (f(end) > Y and itr < max_step):
                break
            itr += 1
            if side > 0:
                right = right + width
            else:
                left = left - width
    used = 0
    while True:
        if used == len(u_shrink):
            return None
        dx = left + (right - left) * u_shrink[used]
        used += 1
        y = f(dx)
        evals += 1
        if y != y or y > Y or (dx == 0.0).any():
            return x0 + d_vec * dx, used, evals, y
        right = np.where(dx > 0, dx, right)
        left = np.where(dx < 0, dx, left)


@pytest.mark.parametrize("k", [1, 2, 16])
def test_device_sampler_walks_the_sequential_chain(k):
    r_seq, r_dev = np.random.default_rng(4), np.random.default_rng(4)
    x_seq = x_dev = np.array([[0.3, -0.2]])
    dev = slice_device()
    calls = 0
    for _ in range(60):
        x_seq = slice_sampler()(lambda v, a: logp(v), x_seq, {"nSamples": 1}, None, rng=r_seq)
        x_dev = dev(replay_step, x_dev, {"nSamples": 1}, None, rng=r_dev, k=k)
        calls += dev.calls
        assert np.array_equal(x_seq, x_dev)
    assert r_seq.bit_generator.state == r_dev.bit_generator.state
    assert k > 1 or calls > 60                # one shrink uniform is too few for some steps


def test_device_sampler_refuses_what_it_does_not_run():
    with pytest.raises(NotImplementedError):
        slice_device()(replay_step, np.zeros((1, 2)), {"gibbs": True}, None, rng=np.random.default_rng(0))
    with pytest.raises(NotImplementedError):
        slice_device()(replay_step, np.zeros((1, 2)), {"widths": np.ones((1, 2))}, None, rng=np.random.default_rng(0))

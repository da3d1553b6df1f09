"""CPU: the per-segment bins -> weight-gradient contraction of the CGNNI backward (oracle/pwl_grad.py) against fp64 autograd of
Linear(1, 10) - ReLU - Linear(10, 1), including a unit with zero input weight and units with negative slopes."""
import numpy as np
import pytest
import torch

from oracle import pwl_grad


def _weights(seed):
    rng = np.random.RandomState(seed)
    w1 = rng.randn(10).astype(np.float32)
    b1 = rng.randn(10).astype(np.float32)
    w2 = rng.randn(10).astype(np.float32)
    w1[0] = 0.0                                           # a unit without input: active everywhere iff b1 > 0
    b1[0] = abs(b1[0]) + 0.1
    w1[1] = 0.0                                           # ... and one that is never active
    b1[1] = -abs(b1[1]) - 0.1
    w1[2:5] = -np.abs(w1[2:5]) - 0.05                     # negative slopes: active left of their breakpoint
    return w1, b1, w2, np.float32(rng.randn())


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_bins_contraction_matches_autograd(seed):
    w1, b1, w2, b2 = _weights(seed)
    rng = np.random.RandomState(100 + seed)
    x = (rng.randn(5000) * 3).astype(np.float32)
    g = rng.randn(5000)
    mlp = torch.nn.Sequential(torch.nn.Linear(1, 10), torch.nn.ReLU(), torch.nn.Linear(10, 1)).double()
    with torch.no_grad():
        mlp[0].weight.copy_(torch.from_numpy(w1).double().reshape(10, 1))
        mlp[0].bias.copy_(torch.from_numpy(b1).double())
        mlp[2].weight.copy_(torch.from_numpy(w2).double().reshape(1, 10))
        mlp[2].bias.fill_(float(b2))
    out = mlp(torch.from_numpy(x).double().reshape(-1, 1)).reshape(-1)
    (out * torch.from_numpy(g)).sum().backward()
    Sg, Sgx = pwl_grad.bins(w1, b1, x, g)
    assert np.count_nonzero(Sg) >= 5                       # the inputs do spread over several segments
    dW1, db1, dW2, db2 = pwl_grad.contract(w1, b1, w2, Sg, Sgx)
    ref = [mlp[0].weight.grad.reshape(-1), mlp[0].bias.grad, mlp[2].weight.grad.reshape(-1), mlp[2].bias.grad.reshape(-1)]
    for got, want in zip([dW1, db1, dW2, np.array([db2])], ref):
        want = want.numpy()
        assert np.abs(got - want).max() <= 1e-10 * max(np.abs(want).max(), 1.0)
    assert dW1[1] == 0.0 and db1[1] == 0.0 and dW2[1] == 0.0    # the dead unit gets nothing
    assert dW1[0] != 0.0                                        # the always-on unit gets dW1 = c * sum g x


def test_segments_follow_the_breakpoints():
    w1 = np.array([1.0, -2.0, 0.0, 4.0], np.float32)
    b1 = np.array([-1.0, 2.0, 1.0, 0.0], np.float32)      # breakpoints 1, 1, inf, 0 -> sorted 0, 1, 1
    t, rank = pwl_grad.breakpoints(w1, b1)
    assert list(rank) == [1, 2, 3, 0]
    assert list(pwl_grad.segments(w1, b1, [-1.0, 0.5, 2.0])) == [0, 1, 3]

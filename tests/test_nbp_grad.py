"""CPU: the hand-derived neural BP backward (oracle/nbp_grad.py, the recurrence gd_backward_nbp.cu implements) against torch
autograd through oracle/restate.py::_forward_neural_bp, in fp64, on the toric L = 4 fixture and a random irregular graph with
isolated and degree-1 variables and checks of degree up to 12."""
import numpy as np
import pytest
import torch

from conftest import Golden
from oracle import nbp_grad, restate


def _autograd(edge_index, V, C, x, w, T, dlogit):
    wg = {k: v.detach().double().clone().requires_grad_(True) for k, v in w.items()}
    logit = restate._forward_neural_bp(edge_index, V, C, x, wg, T, torch.float64)["logit"]
    (logit * dlogit).sum().backward()
    return logit.detach(), {k: v.grad for k, v in wg.items()}


def _seeded(E, T, seed):
    g = torch.Generator().manual_seed(seed)
    w = {}
    for l in range(T):
        w["layers.%d.W" % (2 * l)] = torch.rand((E, 1), generator=g, dtype=torch.float64) * 0.6 + 0.6
        w["layers.%d.W_p" % (2 * l)] = torch.rand((E, 1), generator=g, dtype=torch.float64) * 0.6 + 0.6
    w["W"] = torch.rand((E, 1), generator=g, dtype=torch.float64) * 0.6 + 0.6
    w["W_p"] = torch.rand((E, 1), generator=g, dtype=torch.float64) * 0.6 + 0.6
    w["alpha"] = torch.tensor([[0.25]], dtype=torch.float64)
    return w


def _irregular(seed):
    """Random checks of degree 2 .. 12 over V variables; variable V - 1 is isolated, some variables have one edge.  (A check of
    degree 1 always sends the clamped message +-34.5: past it, fp64 autograd through 1 - o loses digits the recurrence keeps.)"""
    rng = np.random.RandomState(seed)
    V, C = 40, 14
    rows = []
    for c in range(C):
        d = 12 if c == 1 else rng.randint(2, 9)
        rows.append(np.sort(rng.choice(V - 1, d, replace=False)))
    pcm = np.zeros((C, V), np.uint8)
    for c, r in enumerate(rows):
        pcm[c, r] = 1
    ci, vi = np.nonzero(pcm)                         # (check, variable) pairs
    order = np.lexsort((ci, vi))                     # canonical: sorted by variable, then check
    ei = torch.from_numpy(np.stack([vi[order], ci[order]])).long()
    return ei, V, C


def _inputs(V, C, B, seed):
    g = torch.Generator().manual_seed(seed)
    prior = torch.rand((B, 1), generator=g, dtype=torch.float64) * 2 + 0.5
    sign = torch.where(torch.rand((B, C), generator=g) < 0.3, -1.0, 1.0).double()
    x = torch.cat([prior.expand(B, V), sign], 1)
    dlogit = torch.randn((B, V), generator=g, dtype=torch.float64)
    return x, dlogit


def _check(edge_index, V, C, x, w, T, dlogit):
    logit_ref, ref = _autograd(edge_index, V, C, x, w, T, dlogit)
    logit, got = nbp_grad.grads(edge_index, V, C, x, w, T, dlogit)
    # (the recurrence keeps digits of saturated messages that restate's op sequence rounds away: not bit-equal)
    assert torch.allclose(logit, logit_ref, rtol=1e-6, atol=1e-6)
    for k, want in ref.items():
        if k not in got:                                 # the target_to_source layers' W / W_p: unused by the forward
            assert want is None or not want.any(), k
            continue
        err = (got[k] - want).abs().max().item()
        scale = want.abs().max().item()
        assert scale > 0.0 or k == "layers.0.W", k        # m^0 = 0: the first layer's W gets nothing
        assert err <= 1e-9 * scale, "%s: max err %.3g of max |g| %.3g" % (k, err, scale)


def test_toric_fixture_weights_match_autograd():
    g = Golden("ext_neural_bp_toricL4")
    dlogit = torch.randn((g.B, g.V), generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    _check(g.edge_index, g.V, g.C, g.x.double(), g.weights, g.T, dlogit)


@pytest.mark.parametrize("seed", [0, 1])
def test_random_irregular_graph_matches_autograd(seed):
    ei, V, C = _irregular(seed)
    T, B = 5, 6
    x, dlogit = _inputs(V, C, B, seed)
    _check(ei, V, C, x, _seeded(ei.size(1), T, seed), T, dlogit)

"""GPU suite: training the CGNNI decoder (classical/CGNNI.py) through the node-owner forward with stash and its backward kernel
(csrc/gd_backward_light.cu), against fp64 autograd through the oracle's restatement of the forward (oracle/restate.py).

Bar, per parameter tensor the forward uses (ggc2.mlp2, mlp): max |g - g_ref| <= 1e-4 max |g_ref|; loss within 1e-5 relative.
The other state_dict tensors are never used by the forward: their .grad stays None, as under autograd in the reference."""
import ctypes as ct

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import Golden
from oracle import restate

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GRAD_RTOL = 1e-4
USED = ("ggc2.mlp2.0.weight", "ggc2.mlp2.0.bias", "ggc2.mlp2.2.weight", "ggc2.mlp2.2.bias",
        "mlp.0.weight", "mlp.0.bias", "mlp.2.weight", "mlp.2.bias")
CLAMP_LOGIT = float(np.log(1.0 / 1e-7 - 1.0))          # |logit| where sigmoid(-logit) reaches the clamp bounds, ~16.12


class _Data(object):
    pass


def _decoder(weights, T=25):
    from gnn_decode_b200.classical import CGNNI
    dec = CGNNI.GNNI(T)
    dec.load_state_dict(weights, strict=True)
    return dec.to(DEV).train()


def _step(dec, edge_index, V, C, x, loss_fn):
    """The drop-in train step: loss = loss_fn(decoder(datas)); loss.backward()."""
    B, N, E = x.size(0), V + C, edge_index.size(1)
    d = _Data()
    d.x = x.reshape(-1, 1).to(DEV)
    d.edge_index = (edge_index.repeat(1, B) + (torch.arange(B) * N).repeat_interleave(E)).to(DEV)
    dec.zero_grad(set_to_none=True)
    pred = dec(d)
    assert pred.requires_grad
    loss = loss_fn(pred.reshape(B, V))
    loss.backward()
    grads = {k: (p.grad.detach().clone() if p.grad is not None else None) for k, p in dec.named_parameters()}
    return loss.item(), grads, pred.detach().reshape(B, V)


def _oracle(weights, edge_index, V, C, x, loss_fn, T=25):
    loss, grads, prob = restate.decode_grad("cgnni", edge_index, V, C, x.cpu().double(), weights, loss_fn, T=T, dtype=torch.float64)
    return loss.item(), grads, prob


def _check(loss, grads, loss_ref, grads_ref, what=""):
    assert abs(loss - loss_ref) <= 1e-5 * abs(loss_ref), (what, loss, loss_ref)
    for k in USED:
        g, gr = grads[k].double().cpu(), grads_ref[k]
        err, scale = (g - gr).abs().max().item(), gr.abs().max().item()
        assert err <= GRAD_RTOL * scale, "%s %s: max err %.3g vs max |g_ref| %.3g" % (what, k, err, scale)
    for k, g in grads.items():
        if k not in USED:
            assert g is None, k


def _bce_away_from_clamp(x, edge_index, V, C, weights, y, T=25):
    """Weighted BCE against y whose weights vanish where the fp64 logit lies within 0.6 of the clamp thresholds."""
    lg = restate.decode("cgnni", edge_index, V, C, x.cpu().double(), weights, T=T, dtype=torch.float64)["logit"]
    wt = ((lg.abs() - CLAMP_LOGIT).abs() > 0.6).double()
    yd = y.double()

    def loss(prob):
        return F.binary_cross_entropy(prob, yd.to(prob.device, prob.dtype), weight=wt.to(prob.device, prob.dtype))
    return loss


def _weighted_sum(B, V, seed):
    r = torch.from_numpy(np.random.RandomState(seed).randn(B, V))

    def loss(prob):
        return (r.to(prob.device, prob.dtype) * prob).sum()
    return loss


@pytest.mark.parametrize("loss_kind", ["bce", "rsum"])
@pytest.mark.parametrize("name", ["cgnni_bch_epoch18", "cgnni_ldpc_epoch18", "cgnni_bch_seeded"])
def test_fixture_gradients_match_fp64_autograd(name, loss_kind, gd_opt):
    g = Golden(name)
    loss_fn = (_bce_away_from_clamp(g.x, g.edge_index, g.V, g.C, g.weights, g.y, g.T) if loss_kind == "bce"
               else _weighted_sum(g.B, g.V, 7))
    dec = _decoder(g.weights, g.T)
    loss, grads, prob = _step(dec, g.edge_index, g.V, g.C, g.x.float(), loss_fn)
    loss_ref, grads_ref, _ = _oracle(g.weights, g.edge_index, g.V, g.C, g.x, loss_fn, g.T)
    _check(loss, grads, loss_ref, grads_ref, name)
    # the train-mode forward is the node-owner inference kernel plus the stash: bit-identical outputs
    from gnn_decode_b200.graph import TannerGraph
    gd_opt.set("GD_FORCE_LIGHT")
    dec.eval()
    with torch.no_grad():
        p_inf = dec.decode(g.x.float().to(DEV), graph=TannerGraph(g.edge_index, g.V, g.C, DEV))
    assert torch.equal(p_inf, prob)


def _sampled(B, seed=11, snr=(1.0, 2.0, 3.0, 4.0, 5.0, 6.0)):
    from gnn_decode_b200 import codes
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.sampler import sample_syndromes
    pcm = codes.bch_63_45_pcm()
    g = TannerGraph.from_pcm(pcm, DEV)
    x, err = sample_syndromes(g, B, list(snr), noise=2, seed=seed)
    return torch.from_numpy(codes.edge_index_of(pcm)), g.V, g.C, x, err


def test_batch_the_gpu_fills():
    """4096 sampled BCH(63,45) syndromes (~44 M syndrome-edge-iteration items through the bins).  At this size some items sit
    within fp32 rounding of a ReLU breakpoint or of tanh saturation, so fp32 arithmetic itself -- the reference's own CGNNI dtype
    (restate.decode_grad in fp32) -- is up to ~2e-3 max|g| away from fp64 on ggc2.mlp2 at 1-6 dB.  Bar per tensor: 1e-4 max|g|,
    or, where the fp32 reference is further than that from fp64, no more than twice its distance."""
    w = Golden("cgnni_bch_epoch18").weights
    ei, V, C, x, err = _sampled(4096)
    loss_fn = _bce_away_from_clamp(x, ei, V, C, w, err)
    loss, grads, _ = _step(_decoder(w), ei, V, C, x, loss_fn)
    loss_ref, grads_ref, _ = _oracle(w, ei, V, C, x, loss_fn)
    _, grads32, _ = restate.decode_grad("cgnni", ei, V, C, x.cpu(), w, loss_fn, dtype=torch.float32)
    assert abs(loss - loss_ref) <= 1e-5 * abs(loss_ref)
    for k in USED:
        gr = grads_ref[k]
        scale = gr.abs().max().item()
        err32 = (grads32[k].double() - gr).abs().max().item()
        err = (grads[k].double().cpu() - gr).abs().max().item()
        assert err <= max(GRAD_RTOL * scale, 2.0 * err32), "%s: max err %.3g, fp32 reference %.3g, max |g_ref| %.3g" % (
            k, err, err32, scale)


def test_clamp_saturation():
    """Large priors: most outputs saturate.  The trained BCH weights bound |logit| near 1 whatever the priors, so this uses the
    seeded fixture's weights, whose read-out does reach the clamp.  Gradients match the oracle, and a loss on clamped outputs
    only has gradient 0."""
    g = Golden("cgnni_bch_seeded")
    x = g.x.clone()
    x[:, :g.V] *= 300.0
    lg = restate.decode("cgnni", g.edge_index, g.V, g.C, x.double(), g.weights, dtype=torch.float64)["logit"]
    clamped = lg.abs() > CLAMP_LOGIT + 0.6
    assert clamped.double().mean().item() > 0.5
    far = ((lg.abs() - CLAMP_LOGIT).abs() > 0.6).double()
    r = torch.from_numpy(np.random.RandomState(3).randn(g.B, g.V)) * far

    def loss_fn(prob):
        return (r.to(prob.device, prob.dtype) * prob).sum()
    dec = _decoder(g.weights)
    loss, grads, _ = _step(dec, g.edge_index, g.V, g.C, x.float(), loss_fn)
    loss_ref, grads_ref, _ = _oracle(g.weights, g.edge_index, g.V, g.C, x, loss_fn)
    _check(loss, grads, loss_ref, grads_ref)
    mask = clamped.double()

    def clamped_only(prob):
        return (mask.to(prob.device, prob.dtype) * prob).sum()
    _, grads, _ = _step(dec, g.edge_index, g.V, g.C, x.float(), clamped_only)
    for k in USED:
        assert torch.count_nonzero(grads[k]).item() == 0, k


def test_determinism_accumulate_and_linearity():
    from gnn_decode_b200 import _cabi
    from gnn_decode_b200.graph import TannerGraph
    g = Golden("cgnni_bch_epoch18")
    dec = _decoder(g.weights)
    loss_fn = _weighted_sum(g.B, g.V, 5)
    l1, g1, _ = _step(dec, g.edge_index, g.V, g.C, g.x.float(), loss_fn)
    l2, g2, _ = _step(dec, g.edge_index, g.V, g.C, g.x.float(), loss_fn)
    assert l1 == l2 and all(torch.equal(g1[k], g2[k]) for k in USED)
    loss3 = _weighted_sum(g.B, g.V, 5)
    r3 = lambda prob: loss3(prob[:g.B]) + loss3(prob[g.B:2 * g.B]) + loss3(prob[2 * g.B:])   # noqa: E731
    _, g3, _ = _step(dec, g.edge_index, g.V, g.C, g.x.float().repeat(3, 1), r3)
    for k in USED:
        assert (g3[k] - 3 * g1[k]).abs().max().item() <= 2e-4 * (3 * g1[k]).abs().max().item(), k
    # gd_decode_bwd with accumulate != 0 adds exactly the same gradient
    lib = _cabi.lib()
    graph = TannerGraph(g.edge_index, g.V, g.C, DEV)
    model = dec.gd_model()
    w = dec.packed_weights(DEV)
    x = g.x.float().contiguous().to(DEV)
    B = g.B
    stash = torch.empty(lib.gd_stash_floats(graph.handle, ct.byref(model), B), device=DEV)
    assert stash.numel() == g.T * g.E * B
    prob = torch.empty((B, g.V), device=DEV)
    logit = torch.empty((B, g.V), device=DEV)
    st = ct.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ct.c_void_p(t.data_ptr())   # noqa: E731
    _cabi.check(lib.gd_decode_fwd_train(graph.handle, ct.byref(model), p(w), p(x), p(prob), p(logit), p(stash), B, st))
    gl = torch.from_numpy(np.random.RandomState(1).randn(B, g.V)).float().to(DEV)
    ws = torch.empty(lib.gd_bwd_workspace_floats(graph.handle, ct.byref(model), B), device=DEV)
    gw = torch.empty(w.numel(), device=DEV)
    _cabi.check(lib.gd_decode_bwd(graph.handle, ct.byref(model), p(w), p(x), p(stash), p(gl), p(gw), p(ws), 0, B, st))
    first = gw.clone()
    _cabi.check(lib.gd_decode_bwd(graph.handle, ct.byref(model), p(w), p(x), p(stash), p(gl), p(gw), p(ws), 1, B, st))
    assert torch.count_nonzero(first).item() > 0 and torch.equal(gw, 2 * first)


@pytest.mark.parametrize("B", [1, 7, 129])
def test_batch_sizes(B):
    """One syndrome, a batch that is no multiple of 4, and one more than the largest tile (two tiles, the second partial)."""
    w = Golden("cgnni_bch_epoch18").weights
    ei, V, C, x, err = _sampled(B, seed=20 + B)
    loss_fn = _weighted_sum(B, V, B)
    loss, grads, _ = _step(_decoder(w), ei, V, C, x, loss_fn)
    loss_ref, grads_ref, _ = _oracle(w, ei, V, C, x, loss_fn)
    _check(loss, grads, loss_ref, grads_ref, "B=%d" % B)


def _random_pcm(seed):
    """Isolated variables, degree-1 nodes, one check of degree 30 and variables of degree above 4."""
    rng = np.random.RandomState(seed)
    C, V = int(rng.randint(8, 14)), int(rng.randint(36, 48))
    pcm = np.zeros((C, V), dtype=np.uint8)
    for v in range(2, V):
        deg = int(rng.choice([1, 1, 2, 3, 5, 6])) if v % 7 else min(C, 7)
        pcm[rng.permutation(C)[:deg], v] = 1
    pcm[0, :] = 0
    pcm[0, 2:32] = 1                                        # a check of degree 30
    pcm[1, :] = 0
    pcm[1, 5] = 1                                           # a degree-1 check
    pcm[:, :2] = 0                                          # two isolated variables
    return pcm


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_graphs(seed):
    from gnn_decode_b200 import codes
    from gnn_decode_b200.classical import CGNNI
    from gnn_decode_b200.graph import TannerGraph
    pcm = _random_pcm(seed)
    assert pcm.sum(1).max() == 30 and pcm.sum(0).max() > 4 and (pcm.sum(0) == 0).any() and (pcm.sum(0) == 1).any()
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    C, V = pcm.shape
    g = TannerGraph(ei, V, C, DEV)
    torch.manual_seed(seed)
    T = 6
    dec = CGNNI.GNNI(T)
    weights = {k: v.detach().clone() for k, v in dec.state_dict().items()}
    dec = dec.to(DEV).train()
    rng = np.random.RandomState(seed)
    B = 300
    x = torch.cat([torch.from_numpy(rng.randn(B, V) * 2 + 2), torch.zeros(B, C, dtype=torch.float64)], 1).float()
    loss_fn = _weighted_sum(B, V, seed)
    dec.zero_grad(set_to_none=True)
    prob = dec.decode(x.to(DEV), graph=g)
    loss = loss_fn(prob)
    loss.backward()
    grads = {k: p.grad for k, p in dec.named_parameters()}
    loss_ref, grads_ref, _ = _oracle(weights, ei, V, C, x, loss_fn, T)
    _check(loss.item(), grads, loss_ref, grads_ref, "seed=%d" % seed)


def test_sgd_trajectory():
    """Five torch.optim.SGD steps on the GPU against the same five steps on the fp64 oracle's weights."""
    g = Golden("cgnni_ldpc_epoch18")
    dec = _decoder(g.weights)
    opt = torch.optim.SGD(dec.parameters(), lr=0.05)
    w_ref = {k: v.double().clone() for k, v in g.weights.items()}
    y = g.y.double()

    def bce(prob):
        return F.binary_cross_entropy(prob, y.to(prob.device, prob.dtype))
    for _ in range(5):
        _step(dec, g.edge_index, g.V, g.C, g.x.float(), bce)
        opt.step()
        _, gr, _ = _oracle(w_ref, g.edge_index, g.V, g.C, g.x, bce)
        w_ref = {k: v - 0.05 * gr[k] for k, v in w_ref.items()}
    moved = 0.0
    for k in USED:
        got, want = dec.state_dict()[k].double().cpu(), w_ref[k]
        assert (got - want).abs().max().item() <= 1e-4 * want.abs().max().item(), k
        moved = max(moved, (want - g.weights[k].double()).abs().max().item())
    assert moved > 1e-3                                      # the steps did move the weights


def test_refusals():
    """Graphs the node-owner kernel cannot take, and programs without a backward, raise GdError (no kernel runs)."""
    from gnn_decode_b200 import _cabi, codes
    from gnn_decode_b200.graph import TannerGraph
    g = Golden("cgnni_ldpc_epoch18")
    dec = _decoder(g.weights)
    perm = torch.from_numpy(np.random.RandomState(0).permutation(g.E))
    x = g.x.float().to(DEV)
    with pytest.raises(_cabi.GdError, match="canonical"):
        dec.decode(x, graph=TannerGraph(g.edge_index[:, perm], g.V, g.C, DEV))
    pcm = codes.hgp_pcm()
    big = TannerGraph.from_pcm(pcm, DEV)
    xb = torch.zeros((4, big.N), device=DEV)
    xb[:, :big.V] = 3.0
    with pytest.raises(_cabi.GdError, match="shared memory"):
        dec.decode(xb, graph=big)
    model = _cabi.GdModel(_cabi.PROG_QGNNI, 10, 25, 0)
    assert _cabi.lib().gd_bwd_workspace_floats(TannerGraph(g.edge_index, g.V, g.C, DEV).handle, ct.byref(model), 24) == -1
    torch.cuda.synchronize()

"""Training neural BP (quantum/neural_BP.py) and decoder_v1_1 on the GPU: the streamed forward with stash and the per-edge-weight
backward (gd_backward_nbp.cu), against fp64 autograd through oracle/restate.py (bar: max |g - g_ref| <= 1e-4 max |g_ref| per
parameter tensor, loss within 1e-5 relative), on the golden fixtures through the drop-in `criterion(decoder(datas)).backward()`,
seeded weights on toric L = 5 and HGP [[1600,64]], random irregular graphs and batch shapes; reproducibility, accumulate, Adam
steps, a saturating case, the refusals and the kernels one step launches.

The loss neural_BP.py's own train() calls is not in this tree; SURVEY.md (L4) records its LossFunc (neural_BP.py:317-350) as the
sin-relaxed syndrome + logical parity of decoder_v2_4 in training, so train.LossFunc is the first of the two losses used here.

Which kernels a call launches is read with torch.profiler in a child process (this file run as a script): profiler sessions
early in a pytest process make later sessions of other test files miss kernels."""
import ctypes as ct
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

if __name__ == "__main__":
    _ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [_ROOT, os.path.join(_ROOT, "tests")]
from conftest import Golden  # noqa: E402
from gnn_decode_b200 import _cabi, codes, options  # noqa: E402
from gnn_decode_b200.graph import TannerGraph  # noqa: E402
from gnn_decode_b200.sampler import sample_syndromes  # noqa: E402
from oracle import nbp_grad, restate  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
GRAD_BAR, LOSS_BAR = 1e-4, 1e-5
GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ---- decoders and references ---------------------------------------------------------------------------------------------
def _seeded_neural_bp(T, E, seed=0, lo=0.6, hi=1.2, alpha=0.25):
    from gnn_decode_b200.quantum import neural_BP
    g = torch.Generator().manual_seed(seed)
    dec = neural_BP.GNNI(T, n_edges=E)
    with torch.no_grad():
        for n_, p_ in dec.named_parameters():
            p_.copy_(torch.full_like(p_, alpha) if n_ == "alpha" else torch.rand(p_.shape, generator=g, dtype=p_.dtype) * (hi - lo) + lo)
    return dec


def _golden_decoder(name):
    g = Golden(name)
    if name == "ext_neural_bp_toricL4":
        from gnn_decode_b200.quantum import neural_BP
        dec = neural_BP.GNNI(g.T, n_edges=g.E)
        types = None
    else:
        from gnn_decode_b200.quantum import decoder_v1_1
        z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        types = torch.from_numpy(z["edge_types"]).long()
        dec = decoder_v1_1.GNNI(g.T, edge_types=types, nb_digits=int(z["nb_digits"]))
    dec.load_state_dict(g.weights, strict=True)
    return g, dec, types


def _trained_names(dec):
    """The parameters the kernel's weights come from (the target_to_source layers of neural_BP.py own unused W / W_p)."""
    T = dec.Nc
    return [n for l in range(T) for n in ("layers.%d.W" % (2 * l), "layers.%d.W_p" % (2 * l))] + ["W", "W_p", "alpha"]


def _ref(tg, x, state, T, loss_fn, types=None, key="prob"):
    """fp64 autograd through restate._forward_neural_bp: (loss, {name: grad}) w.r.t. the decoder's own parameters (decoder_v1_1:
    its type tables, the per-edge weights gathered from them with autograd)."""
    names = [n for l in range(T) for n in ("layers.%d.W" % (2 * l), "layers.%d.W_p" % (2 * l))] + ["W", "W_p", "alpha"]
    w = {n: state[n].detach().double().cpu().clone().requires_grad_(True) for n in names}
    we = dict(w) if types is None else {n: (w[n] if n == "alpha" else w[n][types]) for n in names}
    out = restate._forward_neural_bp(tg.edge_index.cpu(), tg.V, tg.C, x.double().cpu(), we, T, torch.float64)
    loss = loss_fn(out[key])
    loss.backward()
    return loss.item(), {n: w[n].grad for n in names}


def _gpu(dec, tg, x, loss_fn):
    """One drop-in step on the device: prob = decoder.decode(x) in train mode, loss, backward."""
    dec.zero_grad(set_to_none=True)
    dec.train()
    prob = dec.decode(x, graph=tg)
    loss = loss_fn(prob.double())
    loss.backward()
    return loss.item(), {n: p.grad.detach().double().cpu() for n, p in dec.named_parameters() if n in _trained_names(dec)}


def _distances(got, ref):
    out = {}
    for n, want in ref.items():
        scale = want.abs().max().item()
        out[n] = ((got[n] - want).abs().max().item(), scale)
    return out


def _assert_bar(got, ref, what):
    """Every case is held to GRAD_BAR."""
    for n, (err, scale) in _distances(got, ref).items():
        assert torch.isfinite(got[n]).all(), "%s %s: non-finite gradient" % (what, n)
        assert err <= GRAD_BAR * scale or (scale == 0.0 and err == 0.0), \
            "%s %s: max |g - g_ref| %.3g > %.0e x max |g_ref| %.3g" % (what, n, err, GRAD_BAR, scale)


def _wsum(B, V, seed):
    c = torch.randn((B, V), generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    fn = lambda prob: (prob * (c if not prob.is_cuda else c.to(prob.device))).sum()      # noqa: E731
    fn.c = c
    return fn


def _recurrence(tg, x, state, T, c):
    """The fp64 recurrence (oracle/nbp_grad.py, pinned to autograd on the CPU) for the loss sum c * prob."""
    w = {n: v.detach().double().cpu() for n, v in state.items()}
    ei, xc = tg.edge_index.cpu(), x.double().cpu()
    logit, _ = nbp_grad.grads(ei, tg.V, tg.C, xc, w, T, torch.zeros_like(c))
    prob = torch.sigmoid(-logit)
    return nbp_grad.grads(ei, tg.V, tg.C, xc, w, T, -c * prob * (1 - prob))[1]


def _check(dec, tg, x, loss_seed=3, what="", autograd=True):
    """GPU gradients against the fp64 recurrence (oracle/nbp_grad.py) and, where asked, against fp64 autograd through restate.
    Autograd's op sequence (tanh(u/2) and 1 - o from exp(S), sums over a node's other edges as the total minus the own term)
    rounds away the digits of saturated messages in fp64 too; the recurrence keeps them, and is pinned to autograd where
    nothing saturates (tests/test_nbp_grad.py).  On random irregular graphs and larger batches some messages saturate, so
    there the recurrence is the only reference; autograd's distance is printed."""
    T = dec.Nc
    loss_fn = _wsum(x.size(0), tg.V, loss_seed)
    dec = dec.to(DEV)
    loss, got = _gpu(dec, tg, x, loss_fn)
    loss_ref, ref = _ref(tg, x, dec.state_dict(), T, loss_fn)
    rec = _recurrence(tg, x, dec.state_dict(), T, loss_fn.c)
    print(what, "vs recurrence", {n: e / s if s else e for n, (e, s) in _distances(got, rec).items()},
          "vs autograd", {n: e / s if s else e for n, (e, s) in _distances(got, ref).items()})
    assert abs(loss - loss_ref) <= LOSS_BAR * abs(loss_ref), "%s: loss %.9g vs %.9g" % (what, loss, loss_ref)
    _assert_bar(got, rec, what + " vs the fp64 recurrence")
    if autograd:
        _assert_bar(got, ref, what + " vs fp64 autograd")
    return got, ref


# ---- 1. golden fixtures through the drop-in decoder(datas) + criterion + backward ----------------------------------------
class _Data(object):
    def __init__(self, g, dev):
        self.x = g.x.reshape(-1, 1).to(dev)
        self.edge_index = g.batched_edge_index().to(dev)
        self.y = g.y.reshape(-1, 1).to(dev)


@pytest.mark.parametrize("loss_kind", ["LossFunc", "weighted_prob"])
@pytest.mark.parametrize("name", ["ext_neural_bp_toricL4", "ext_v1_1_onehot_toricL4"])
def test_golden_fixture_drop_in_training(name, loss_kind):
    from gnn_decode_b200 import train
    g, dec, types = _golden_decoder(name)
    dec = dec.to(DEV).train()
    tg = TannerGraph(g.edge_index, g.V, g.C, DEV)
    datas = _Data(g, DEV)
    if loss_kind == "LossFunc":
        criterion = train.LossFunc(graph=tg)
        no_logical = torch.zeros((0, g.V), dtype=torch.float64)
        ref_loss = lambda prob: restate.loss_v2_4(prob, g.y, g.H, no_logical)      # noqa: E731
    else:
        wsum = _wsum(g.B, g.V, 11)
        criterion = lambda pred, d: wsum(pred.reshape(g.B, g.V))                    # noqa: E731
        ref_loss = wsum
    pred = dec(datas)
    assert pred.requires_grad and pred.dtype == torch.float64
    loss = criterion(pred, datas)
    loss.backward()
    got = {n: p.grad.detach().double().cpu() for n, p in dec.named_parameters() if n in _trained_names(dec)}
    loss_ref, ref = _ref(tg, g.x, dec.state_dict(), g.T, ref_loss, types)
    assert abs(loss.item() - loss_ref) <= LOSS_BAR * abs(loss_ref)
    _assert_bar(got, ref, name)
    if types is not None:     # the index backward sums the per-edge gradients per type, bit-reproducibly
        first = {n: p.grad.clone() for n, p in dec.named_parameters() if p.grad is not None}
        dec.zero_grad(set_to_none=True)
        criterion(dec(datas), datas).backward()
        for n, p in dec.named_parameters():
            if n in first:
                assert torch.equal(p.grad, first[n]), n


# ---- 2. seeded weights on toric L = 5 and HGP [[1600,64]] ---------------------------------------------------------------
def test_seeded_toric5_T8():
    tg = TannerGraph.from_pcm(codes.toric_pcm(5), DEV)
    x, _ = sample_syndromes(tg, 200, [0.03, 0.08], noise=1, seed=5)
    _check(_seeded_neural_bp(8, tg.E, seed=1), tg, x, what="toric5")


def test_seeded_hgp_T6_B8():
    tg = TannerGraph.from_pcm(codes.hgp_pcm(), DEV)
    x, _ = sample_syndromes(tg, 8, [0.02, 0.05], noise=1, seed=9)
    _check(_seeded_neural_bp(6, tg.E, seed=2), tg, x, what="hgp")


# ---- 3. random irregular graphs (check degree up to 12, isolated and degree-1 variables) ---------------------------------
def _irregular_pcm(seed):
    rng = np.random.RandomState(seed)
    V, C = 60, 20
    pcm = np.zeros((C, V), dtype=np.uint8)
    for c in range(C):
        d = 12 if c < 2 else rng.randint(2, 10)
        pcm[c, rng.choice(V - 2, size=d, replace=False)] = 1
    pcm[0, V - 2] = 1                         # variable V - 2 has one edge; V - 1 none
    return pcm


@pytest.mark.parametrize("seed", [0, 1])
def test_random_irregular_graph(seed):
    tg = TannerGraph.from_pcm(_irregular_pcm(seed), DEV)
    x, _ = sample_syndromes(tg, 96, [0.05, 0.1], noise=1, seed=seed)
    # Seed 0's inputs hold an item with |u| = 1.5e-6: before log|tanh(u/2)| formed 1 - e^-|u| by series at small |u|
    # (gd_math.cuh, bp_one_minus_exp), layers 0-2 and alpha were up to 4.5e-4 of max |g| from the recurrence here.
    _check(_seeded_neural_bp(5, tg.E, seed=seed), tg, x, what="irregular %d" % seed, autograd=False)


# ---- 4. batch shapes: scalar stash stores, partial tiles, several tiles per CTA ------------------------------------------
@pytest.mark.parametrize("B", [1, 7, 129, 40000])
def test_batch_shapes(B):
    tg = TannerGraph.from_pcm(codes.toric_pcm(5), DEV)
    x, _ = sample_syndromes(tg, B, [0.03, 0.08], noise=1, seed=B)
    T = 3 if B > 1000 else 5
    # B = 129 holds an item with |u| = 1.3e-4 (layers 0 and 2 were 1.03e-4 of max |g| away while 1 - e^-|u| was a subtraction)
    _check(_seeded_neural_bp(T, tg.E, seed=4), tg, x, what="B=%d" % B, autograd=False)


# ---- 4b. small messages: |u| well below 1e-2 on most items -----------------------------------------------------------------
@pytest.mark.parametrize("graph", ["toric5", "irregular0"])
def test_small_message_arguments(graph):
    """Priors near 0 (p close to 0.5) and per-layer W_p spread through 0 keep every |u| below 0.1 and put ~10% of the
    (syndrome, edge, layer) items below 1e-3, where log|tanh(u/2)| = log(1 - q) - log(1 + q), q = e^-|u|, is hardest to form
    in fp32 (1 - q by subtraction carries q's ~2.4e-7 absolute error: ~2.4e-7 / |u| in the value) and the backward's exact
    1 / sinh(u) is large.  The check outputs are tiny too (down to ~1e-10): formed as log(1 + p) - log(1 - p) from rounded
    1 +- p they come out 0, and the W gradients, sums of dq m, lose their digits.  Nothing saturates and no clamp binds, so
    every tensor is held to GRAD_BAR."""
    pcm = codes.toric_pcm(5) if graph == "toric5" else _irregular_pcm(0)
    tg = TannerGraph.from_pcm(pcm, DEV)
    B, T = 128, 5
    gen = torch.Generator().manual_seed(31)
    x = torch.ones((B, tg.N), dtype=torch.float64)
    x[:, :tg.V] = (torch.rand((B, tg.V), generator=gen, dtype=torch.float64) * 2 - 1) * 0.05
    x[:, tg.V:] = torch.where(torch.rand((B, tg.C), generator=gen) < 0.3, -1.0, 1.0)
    x = x.float()
    dec = _seeded_neural_bp(T, tg.E, seed=31)
    with torch.no_grad():
        for n_, p_ in dec.named_parameters():
            if n_.startswith("layers.") and n_.endswith("W_p"):
                p_.copy_(torch.rand(p_.shape, generator=gen) * 2 - 1)
    info = {}
    w = {n: v.detach().double() for n, v in dec.state_dict().items()}
    nbp_grad.grads(tg.edge_index.cpu(), tg.V, tg.C, x, w, T, torch.zeros((B, tg.V), dtype=torch.float64), info)
    print(graph, info)
    # 13695 of 122880 items on toric L = 5, 7742 of 80000 on the irregular graph
    assert info["small_u"] >= 5000 and info["max_abs_u"] < 0.1 and info["o_clamped"] == 0, info
    _check(dec, tg, x.to(DEV), what="small |u| %s" % graph, autograd=False)


# ---- 5. the paths: forward = streamed inference, bit-reproducible backward, accumulate ------------------------------------
def _abi_step(dec, tg, x, dlogit, gw, accumulate):
    lib = _cabi.lib()
    model = dec.gd_model()
    w = torch.cat([p.detach().reshape(-1).float() for p in dec._gd_params()]).to(DEV)
    B = x.size(0)
    p = lambda t: ct.c_void_p(t.data_ptr())                                             # noqa: E731
    st = ct.c_void_p(torch.cuda.current_stream().cuda_stream)
    stash = torch.empty(lib.gd_stash_floats(tg.handle, ct.byref(model), B), device=DEV)
    assert stash.numel() == dec.Nc * tg.E * B
    prob = torch.empty((B, tg.V), device=DEV)
    logit = torch.empty((B, tg.V), device=DEV)
    _cabi.check(lib.gd_decode_fwd_train(tg.handle, ct.byref(model), p(w), p(x), p(prob), p(logit), p(stash), B, st))
    ws = torch.empty(lib.gd_bwd_workspace_floats(tg.handle, ct.byref(model), B), device=DEV)
    _cabi.check(lib.gd_decode_bwd(tg.handle, ct.byref(model), p(w), p(x), p(stash), p(dlogit), p(gw), p(ws), accumulate, B, st))
    torch.cuda.synchronize()
    return prob, logit


def test_forward_equals_streamed_inference_and_backward_is_reproducible(gd_opt):
    tg = TannerGraph.from_pcm(codes.toric_pcm(5), DEV)
    x, _ = sample_syndromes(tg, 3000, [0.03, 0.08], noise=1, seed=21)
    dec = _seeded_neural_bp(6, tg.E, seed=6).to(DEV)
    dlogit = torch.randn((x.size(0), tg.V), generator=torch.Generator().manual_seed(2)).to(DEV)
    n_w = (2 * dec.Nc + 2) * tg.E + 1
    g1, g2 = torch.empty(n_w, device=DEV), torch.empty(n_w, device=DEV)
    prob, logit = _abi_step(dec, tg, x, dlogit, g1, 0)
    _abi_step(dec, tg, x, dlogit, g2, 0)
    assert torch.equal(g1, g2)
    g3 = g1.clone()
    _abi_step(dec, tg, x, dlogit, g3, 1)
    assert torch.equal(g3, g1 + g1)
    gd_opt.set("GD_FORCE_STREAMED")
    dec.eval()
    with torch.no_grad():
        p_inf, l_inf = dec.decode(x, graph=tg, return_logits=True)
    assert torch.equal(prob, p_inf) and torch.equal(logit, l_inf)


# ---- 6. Adam steps with WeightClipper against the same steps on fp64 oracle gradients -------------------------------------
def test_adam_steps_follow_the_oracle():
    """Five Adam steps on the device's gradients against five on fp64 autograd's.  Adam divides each element's gradient by its own
    running RMS, so an element whose gradient is 1e-2 of its tensor's largest carries up to 1e-2 relative error from the 1e-4
    gradient bar into its step: the weights are held to 1e-3 of how far the steps moved them."""
    from gnn_decode_b200.quantum.neural_BP import WeightClipper
    tg = TannerGraph.from_pcm(codes.toric_pcm(5), DEV)
    x, _ = sample_syndromes(tg, 256, [0.03, 0.08], noise=1, seed=8)
    T = 5
    dec = _seeded_neural_bp(T, tg.E, seed=8).to(DEV)
    ref = _seeded_neural_bp(T, tg.E, seed=8)
    names = _trained_names(dec)
    loss_fn = _wsum(x.size(0), tg.V, 13)
    opt = torch.optim.Adam(dec.parameters(), lr=1e-2)
    opt_ref = torch.optim.Adam(ref.parameters(), lr=1e-2)
    clip = WeightClipper()
    start = {n: p.detach().double().cpu().clone() for n, p in ref.named_parameters()}
    for _ in range(5):
        _gpu(dec, tg, x, loss_fn)
        opt.step()
        dec.apply(clip)
        _, g_ref = _ref(tg, x, ref.state_dict(), T, loss_fn)
        opt_ref.zero_grad(set_to_none=True)
        for n, p in ref.named_parameters():
            if n in g_ref:
                p.grad = g_ref[n].to(p.dtype)
        opt_ref.step()
        ref.apply(clip)
    mine = dict(dec.named_parameters())
    apart = {}
    for n, p in ref.named_parameters():
        if n in names:
            apart[n] = ((mine[n].detach().double().cpu() - p.detach()).abs().max().item(), (p.detach() - start[n]).abs().max().item())
    print("adam: (max |w - w_ref|, max |w_ref - w_0|)", apart)
    for n, (err, moved) in apart.items():
        if n == "layers.0.W":
            assert moved == 0.0 and err == 0.0         # m^0 = 0: no gradient, no step
            continue
        assert moved > 0.0, n
        assert err <= 1e-3 * moved, "%s: weights %.3g apart after 5 steps that moved them %.3g" % (n, err, moved)


# ---- 7. saturating inputs: |u| past 87, the o-clamp binds ------------------------------------------------------------------
def test_saturating_inputs_give_finite_gradients_near_fp64():
    """Priors +-25 and weights near 1.5 saturate the logits (prob(1 - prob) underflows), so the loss here is a weighted sum of
    the logits, through the C entry points.  The reference is the fp64 recurrence (oracle/nbp_grad.py): fp64 autograd through
    1 - o and 1 - tanh^2 loses the digits of the saturated terms; both distances are printed for the record."""
    tg = TannerGraph.from_pcm(codes.toric_pcm(5), DEV)
    B = 64
    gen = torch.Generator().manual_seed(17)
    x = torch.ones((B, tg.N))
    x[:, :tg.V] = 25.0 * torch.where(torch.rand((B, tg.V), generator=gen) < 0.1, -1.0, 1.0)
    x[:, tg.V:] = torch.where(torch.rand((B, tg.C), generator=gen) < 0.3, -1.0, 1.0)
    x = x.to(DEV)
    dec = _seeded_neural_bp(5, tg.E, seed=17, lo=1.4, hi=1.6).to(DEV)
    c = torch.randn((B, tg.V), generator=torch.Generator().manual_seed(19), dtype=torch.float64)
    gw = torch.empty((2 * dec.Nc + 2) * tg.E + 1, device=DEV)
    _, logit = _abi_step(dec, tg, x, c.float().to(DEV), gw, 0)
    assert torch.isfinite(gw).all()
    got, off = {}, 0
    for n in _trained_names(dec):
        k = tg.E if n != "alpha" else 1
        got[n] = gw[off:off + k].double().cpu().reshape(dict(dec.named_parameters())[n].shape)
        off += k
    w = {n: v.detach().double().cpu() for n, v in dec.state_dict().items()}
    info = {}
    _, rec = nbp_grad.grads(tg.edge_index.cpu(), tg.V, tg.C, x.cpu(), w, dec.Nc, c, info)
    assert info["max_abs_u"] > 87.0 and info["o_clamped"] > 0, info
    _, ref = _ref(tg, x, dec.state_dict(), dec.Nc, lambda logit: (logit * c).sum(), key="logit")
    d_rec, d_ref = _distances(got, rec), _distances(got, ref)
    print("saturating", info, "max|g - g_fp64 recurrence| / max|g|", {n: e / s if s else e for n, (e, s) in d_rec.items()},
          "max|g - g_fp64 autograd| / max|g|", {n: e / s if s else e for n, (e, s) in d_ref.items()})
    assert torch.isfinite(logit).all()
    logit_rec, _ = nbp_grad.grads(tg.edge_index.cpu(), tg.V, tg.C, x.cpu(), w, dec.Nc, torch.zeros_like(c))
    loss, loss_rec = (logit.double().cpu() * c).sum().item(), (logit_rec * c).sum().item()
    print("saturating loss", loss, loss_rec)
    assert abs(loss - loss_rec) <= LOSS_BAR * abs(loss_rec)
    _assert_bar(got, rec, "saturating vs the fp64 recurrence")


# ---- 8. refusals and routing (profiler in a child process) ----------------------------------------------------------------
def _kernels(fn):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    out = []
    for ev in events:
        if ev.get("cat") == "kernel" and "gd::" in ev.get("name", ""):
            m = re.search(r"(\w+)\s*(?:<|\()", ev["name"].split("gd::", 1)[1])
            out.append(m.group(1) if m else ev["name"])
    return out


def _probe_main():
    tg = TannerGraph.from_pcm(codes.toric_pcm(5), DEV)
    x, _ = sample_syndromes(tg, 300, [0.03, 0.08], noise=1, seed=3)
    dec = _seeded_neural_bp(4, tg.E).to(DEV).train()
    perm = torch.from_numpy(np.random.RandomState(0).permutation(tg.E))
    tp = TannerGraph(tg.edge_index[:, perm], tg.V, tg.C, DEV)
    out = {}
    for name, graph in (("step", tg), ("permuted", tp)):
        err = []

        def run():
            try:
                dec.zero_grad(set_to_none=True)
                dec.decode(x, graph=graph).sum().backward()
            except _cabi.GdError as e:
                err.append(str(e))
        out[name] = {"kernels": _kernels(run), "error": err[0] if err else None}
    print(json.dumps(out))


@pytest.fixture(scope="module")
def launched():
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_one_step_launches_the_streamed_forward_the_backward_and_its_reduction(launched):
    assert launched["step"]["error"] is None
    assert launched["step"]["kernels"] == ["decode_streamed_tma_kernel", "nbp_bwd_kernel", "nbp_reduce_kernel"]


def test_permuted_edge_order_is_refused_without_a_launch(launched):
    assert launched["permuted"]["error"] is not None and "canonical" in launched["permuted"]["error"]
    assert launched["permuted"]["kernels"] == []


def test_hidden_not_E_is_invalid():
    lib = _cabi.lib()
    tg = TannerGraph.from_pcm(codes.toric_pcm(4), DEV)
    model = _cabi.GdModel(_cabi.PROG_NEURAL_BP, tg.E + 1, 3, 0)
    B = 8
    x = torch.zeros((B, tg.N), device=DEV)
    buf = torch.zeros(1 << 16, device=DEV)
    p = lambda t: ct.c_void_p(t.data_ptr())                                             # noqa: E731
    rc = lib.gd_decode_fwd_train(tg.handle, ct.byref(model), p(buf), p(x), p(buf), None, p(buf), B, None)
    assert rc == _cabi.GD_ERR_INVALID
    rc = lib.gd_decode_bwd(tg.handle, ct.byref(model), p(buf), p(x), p(buf), p(buf), p(buf), p(buf), 0, B, None)
    assert rc == _cabi.GD_ERR_INVALID
    assert lib.gd_bwd_workspace_floats(tg.handle, ct.byref(model), B) == -1
    torch.cuda.synchronize()


if __name__ == "__main__":
    _probe_main()

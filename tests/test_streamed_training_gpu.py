"""GPU suite: training decoder_v2_4 on codes whose training state does not fit shared memory -- the TMA-staged streamed
forward with stash (csrc/gd_streamed_tma.cu, STASH) and the backward with its work arrays in global memory
(csrc/gd_backward.cu, decode_bwd_kernel<true>) -- against the reference's own gradients and fp64 autograd through the
oracle's restatement (oracle/restate.py).  GD_FORCE_STREAMED puts small codes on both streamed kernels.

Bars as in tests/test_training_gpu.py: per parameter tensor max |g - g_ref| <= 1e-4 max |g_ref|, loss within 1e-5 relative."""
import ctypes as ct
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import restate
from oracle.adam import AdamOracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GRAD_RTOL = 1e-4
FIXTURES = ["grad_v2_4_toricL4_epoch1", "grad_v2_4_toricL5_epoch3_T6"]


class _Case(object):
    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN, name + ".npz"))
        self.V, self.C, self.E, self.B, self.T = (int(z[k]) for k in ("V", "C", "E", "B", "T"))
        self.edge_index = torch.from_numpy(z["edge_index"])
        self.x, self.y = torch.from_numpy(z["x"]), torch.from_numpy(z["y"])
        self.H, self.logical = torch.from_numpy(z["H"]).double(), torch.from_numpy(z["logical"]).double()
        self.weights = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
        self.grads = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("g:")}
        self.loss = float(z["loss"])


class _Data(object):
    pass


def _decoder(weights, T):
    from gnn_decode_b200.quantum import decoder_v2_4
    dec = decoder_v2_4.GNNI(T)
    dec.load_state_dict(weights)
    return dec.to(DEV).train()


def _kernels(fn):
    """Names of the CUDA kernels fn() launches."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def _ran(names, what):
    return any(what in n for n in names)


def _check(loss, grads, loss_ref, grads_ref, what=""):
    assert abs(loss - loss_ref) <= 1e-5 * abs(loss_ref), (what, loss, loss_ref)
    for k, gr in grads_ref.items():
        g = grads[k].double().cpu()
        err, scale = (g - gr).abs().max().item(), gr.abs().max().item()
        assert err <= GRAD_RTOL * scale + 1e-12, "%s %s: max err %.3g vs max |g_ref| %.3g" % (what, k, err, scale)


def _code(pcm):
    """(graph, edge_index, H [V, C] fp64, pcm) of a CSS code given as blockdiag(Hz, Hx)."""
    from gnn_decode_b200 import codes
    from gnn_decode_b200.graph import TannerGraph
    return TannerGraph.from_pcm(pcm, DEV), torch.from_numpy(codes.edge_index_of(pcm)), torch.from_numpy(pcm.T.astype(np.float64))


def _hgp(n_checks, n_vars):
    from gnn_decode_b200 import codes
    Hz, Hx = codes.hgp_checks(codes.regular_ldpc(n_checks, n_vars, 3, 4, 1234))
    pcm = codes.css_pcm(Hz, Hx)
    return pcm, codes.css_logicals(Hz, Hx)


def _against_oracle(dec, weights, g, ei, H, logical, x, y, T, what):
    """train_step_grads (forward with stash -> fused loss -> backward) against fp64 autograd through the oracle."""
    from gnn_decode_b200.train import train_step_grads
    loss, _ = train_step_grads(dec, g, x, y, logical)
    grads = {k: p.grad.clone() for k, p in dec.named_parameters()}
    L = torch.from_numpy(np.asarray(logical, dtype=np.float64))
    yd = y.cpu().double()
    loss_ref, grads_ref, _ = restate.decode_grad("v2_4", ei, g.V, g.C, x.cpu().double(), weights,
                                                 lambda prob: restate.loss_v2_4(prob, yd, H, L), T=T, dtype=torch.float64)
    _check(loss.item(), grads, loss_ref.item(), grads_ref, what)
    return grads


@pytest.mark.parametrize("name", FIXTURES)
def test_reference_gradients_on_the_streamed_kernels(name, gd_opt):
    """GD_FORCE_STREAMED: both training calls on the streamed kernels reproduce the reference's own loss.backward()
    gradients, through train_step_grads and through the drop-in decoder + LossFunc autograd."""
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.train import LossFunc, train_step_grads
    gd_opt.set("GD_FORCE_STREAMED")
    case = _Case(name)
    dec = _decoder(case.weights, case.T)
    g = TannerGraph(case.edge_index, case.V, case.C, DEV)
    out = {}

    def fused():
        out["loss"], _ = train_step_grads(dec, g, case.x.to(DEV), case.y.to(DEV), case.logical)
    names = _kernels(fused)
    assert _ran(names, "decode_streamed_tma_kernel") and _ran(names, "decode_bwd_kernel<true>"), names
    assert not _ran(names, "lean_") and not _ran(names, "decode_bwd_kernel<false>"), names
    _check(out["loss"].item(), {k: p.grad for k, p in dec.named_parameters()}, case.loss, case.grads, "fused")
    fused_grads = {k: p.grad.clone() for k, p in dec.named_parameters()}
    crit = LossFunc(None, None, graph=g, logical=case.logical)
    N = case.V + case.C
    d = _Data()
    d.x = case.x.reshape(-1, 1).to(DEV)
    d.edge_index = (case.edge_index.repeat(1, case.B) + (torch.arange(case.B) * N).repeat_interleave(case.E)).to(DEV)
    d.y = case.y.reshape(-1, 1).to(DEV)
    dec.zero_grad()
    loss = crit(dec(d), d)
    loss.backward()
    grads = {k: p.grad.clone() for k, p in dec.named_parameters()}
    _check(loss.item(), grads, case.loss, case.grads, "drop-in")
    for k in grads:
        assert (grads[k] - fused_grads[k]).abs().max().item() <= 1e-5 * fused_grads[k].abs().max().item() + 1e-12, k


def _raw(dec, g, x, train):
    from gnn_decode_b200 import _cabi
    lib = _cabi.lib()
    model = dec.gd_model()
    w = dec.packed_weights(DEV)
    B = x.size(0)
    prob = torch.empty((B, g.V), device=DEV)
    st = ct.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ct.c_void_p(t.data_ptr())   # noqa: E731
    if train:
        stash = torch.empty(lib.gd_stash_floats(g.handle, ct.byref(model), B), device=DEV)
        _cabi.check(lib.gd_decode_fwd_train(g.handle, ct.byref(model), p(w), p(x), p(prob), None, p(stash), B, st))
        return prob, stash
    _cabi.check(lib.gd_decode_fwd(g.handle, ct.byref(model), p(w), p(x), p(prob), None, None, B, st))
    return prob, None


def test_training_forward_equals_streamed_inference(gd_opt):
    """Rotated d = 5, B = 20000 (a batch the streamed inference kernel takes): the training forward is that kernel plus the
    stash, so its output is bit-identical."""
    from gnn_decode_b200 import codes
    from gnn_decode_b200.sampler import sample_syndromes
    gd_opt.set("GD_FORCE_STREAMED")
    g, _, _ = _code(codes.css_pcm(*codes.rotated_surface_checks(5)))
    case = _Case(FIXTURES[1])
    dec = _decoder(case.weights, case.T)
    x, _ = sample_syndromes(g, 20000, [0.03, 0.08, 0.12], noise=1, seed=3)
    holder = {}
    names = _kernels(lambda: holder.update(train=_raw(dec, g, x, True)))
    assert _ran(names, "decode_streamed_tma_kernel"), names
    names = _kernels(lambda: holder.update(infer=_raw(dec, g, x, False)))
    assert _ran(names, "decode_streamed_tma_kernel"), names
    assert torch.equal(holder["train"][0], holder["infer"][0])


def test_resident_and_global_memory_backward_agree(gd_opt):
    """One stash (the resident edge-owner forward, rotated d = 7, B = 4096), both backward forms.  The weight-gradient partials
    are grouped differently (other tiles, 64-bit check-table bins), so the results are close but need not be bit-equal;
    measured on a B200: the largest per-tensor gap is 4.1e-7 of max |g| (ggc1.mlp.0.bias)."""
    from gnn_decode_b200 import _cabi, codes
    from gnn_decode_b200.sampler import sample_syndromes
    from gnn_decode_b200.train import sin_loss
    Hz, Hx = codes.rotated_surface_checks(7)
    g, _, _ = _code(codes.css_pcm(Hz, Hx))
    case = _Case(FIXTURES[1])
    dec = _decoder(case.weights, case.T)
    x, err = sample_syndromes(g, 4096, [0.03, 0.08, 0.12], noise=1, seed=9)
    gd_opt.set("GD_NO_LEAN")                                      # the edge-owner stash layout, no table-kernel header
    prob, stash = _raw(dec, g, x, True)
    _, _, gl = sin_loss(g, prob, err, codes.css_logicals(Hz, Hx))
    lib = _cabi.lib()
    model = dec.gd_model()
    w = dec.packed_weights(DEV)
    st = ct.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ct.c_void_p(t.data_ptr())   # noqa: E731

    def bwd():
        ws = torch.empty(lib.gd_bwd_workspace_floats(g.handle, ct.byref(model), 4096), device=DEV)
        gw = torch.empty(w.numel(), device=DEV)
        _cabi.check(lib.gd_decode_bwd(g.handle, ct.byref(model), p(w), p(x), p(stash), p(gl), p(gw), p(ws), 0, 4096, st))
        return gw
    out = {}
    names = _kernels(lambda: out.update(a=bwd()))
    assert _ran(names, "decode_bwd_kernel<false>"), names
    gd_opt.set("GD_FORCE_STREAMED")
    names = _kernels(lambda: out.update(b=bwd()))
    assert _ran(names, "decode_bwd_kernel<true>"), names
    off = 0
    for k, prm in dec.named_parameters():
        n = prm.numel()
        a, b = out["a"][off:off + n], out["b"][off:off + n]
        gap = (a - b).abs().max().item() / a.abs().max().item()
        print("%s: gap %.3g of max |g|" % (k, gap))
        assert gap <= 1e-5, (k, gap)
        off += n


def test_mid_size_code_default_route():
    """hgp_pcm(9, 12) (E = 1512): the forward is resident, the backward's work arrays do not fit shared memory (it was
    refused before the global-memory form existed) -- against fp64 autograd at B = 16, T = 6."""
    from gnn_decode_b200.sampler import sample_syndromes
    pcm, logical = _hgp(9, 12)
    g, ei, H = _code(pcm)
    assert g.E == 1512
    case = _Case(FIXTURES[1])
    dec = _decoder(case.weights, 6)
    x, err = sample_syndromes(g, 16, [0.03, 0.06, 0.1], noise=1, seed=4)
    names = _kernels(lambda: _against_oracle(dec, case.weights, g, ei, H, logical, x, err, 6, "hgp(9,12)"))
    assert _ran(names, "decode_bwd_kernel<true>") and not _ran(names, "decode_bwd_kernel<false>"), names
    assert _ran(names, "decode_kernel") or _ran(names, "decode_streamed_tma_kernel"), names


def test_hgp_1600():
    """HGP [[1600,64]] (BASELINE config 5, E = 10752): B = 2, T = 3 against fp64 autograd.  The check-table adjoint bins see
    E * tile items per phase here (64-bit bins keep every item's resolution)."""
    from gnn_decode_b200 import codes
    from gnn_decode_b200.sampler import sample_syndromes
    pcm, logical = _hgp(24, 32)
    assert np.array_equal(pcm, codes.hgp_pcm())
    g, ei, H = _code(pcm)
    case = _Case(FIXTURES[1])
    dec = _decoder(case.weights, 3)
    x, err = sample_syndromes(g, 2, [0.05, 0.1], noise=1, seed=6)
    names = _kernels(lambda: _against_oracle(dec, case.weights, g, ei, H, logical, x, err, 3, "hgp1600"))
    assert _ran(names, "decode_streamed_tma_kernel") and _ran(names, "decode_bwd_kernel<true>"), names


@pytest.mark.parametrize("B", [1, 7, 129])
def test_batch_sizes(B, gd_opt):
    """GD_FORCE_STREAMED on toric L = 5: one syndrome, a batch that is no multiple of 4 (scalar stash stores), and 129 (the
    backward's tiles of 4 end with one partial tile of 1 syndrome; the forward's last tile is partial too)."""
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.sampler import sample_syndromes
    gd_opt.set("GD_FORCE_STREAMED")
    case = _Case(FIXTURES[1])
    g = TannerGraph(case.edge_index, case.V, case.C, DEV)
    dec = _decoder(case.weights, case.T)
    x, err = sample_syndromes(g, B, [0.03, 0.08, 0.12], noise=1, seed=30 + B)
    _against_oracle(dec, case.weights, g, case.edge_index, case.H, case.logical.numpy().astype(np.uint8), x, err, case.T,
                    "B=%d" % B)


def test_bit_reproducible_and_accumulate():
    """Mid-size code, default route: two identical steps give bit-identical gradients, and accumulate = 1 adds exactly the
    same gradient."""
    from gnn_decode_b200 import _cabi
    from gnn_decode_b200.sampler import sample_syndromes
    from gnn_decode_b200.train import sin_loss
    pcm, logical = _hgp(9, 12)
    g, _, _ = _code(pcm)
    dec = _decoder(_Case(FIXTURES[1]).weights, 6)
    B = 300
    x, err = sample_syndromes(g, B, [0.03, 0.06, 0.1], noise=1, seed=8)
    lib = _cabi.lib()
    model = dec.gd_model()
    w = dec.packed_weights(DEV)
    st = ct.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ct.c_void_p(t.data_ptr())   # noqa: E731
    ws = torch.empty(lib.gd_bwd_workspace_floats(g.handle, ct.byref(model), B), device=DEV)

    def step():
        prob, stash = _raw(dec, g, x, True)
        _, _, gl = sin_loss(g, prob, err, logical)
        gw = torch.empty(w.numel(), device=DEV)
        _cabi.check(lib.gd_decode_bwd(g.handle, ct.byref(model), p(w), p(x), p(stash), p(gl), p(gw), p(ws), 0, B, st))
        return gw, stash, gl
    g1, stash, gl = step()
    g2, _, _ = step()
    assert torch.count_nonzero(g1).item() > 0 and torch.equal(g1, g2)
    _cabi.check(lib.gd_decode_bwd(g.handle, ct.byref(model), p(w), p(x), p(stash), p(gl), p(g2), p(ws), 1, B, st))
    assert torch.equal(g2, 2 * g1)


def test_fused_trainer_adam_steps():
    """Three FusedTrainer steps (forward -> gd_loss_v2_4 -> backward -> Adam) on the mid-size code against the same three Adam
    steps of oracle/adam.py on fp64 oracle gradients.  Each step's gradient is also the fused train step's, bit for bit (its
    accuracy against fp64 autograd on this code and route is test_mid_size_code_default_route's).  Adam moves every weight by
    about lr per step whatever the size of its gradient, so where a gradient is near 0 the step's direction rests on rounding:
    the trajectory is compared where every step's oracle gradient is at least 5e-2 of its tensor's largest (within 0.1 lr),
    and everywhere within the 2 lr per step Adam can move."""
    from gnn_decode_b200.sampler import sample_syndromes
    from gnn_decode_b200.train import FusedTrainer, train_step_grads
    pcm, logical = _hgp(9, 12)
    g, ei, H = _code(pcm)
    weights = _Case(FIXTURES[1]).weights
    dec = _decoder(weights, 6)
    tr = FusedTrainer(dec, g, logical)
    names = [k for k, _ in dec.named_parameters()]
    shapes = {k: prm.shape for k, prm in dec.named_parameters()}
    sizes = [int(np.prod(shapes[k])) for k in names]
    L = torch.from_numpy(np.asarray(logical, dtype=np.float64))

    def unflat(flat):
        parts = np.split(np.asarray(flat, dtype=np.float64), np.cumsum(sizes)[:-1])
        return {k: torch.from_numpy(np.ascontiguousarray(a).reshape(shapes[k])) for k, a in zip(names, parts)}
    start = np.concatenate([weights[k].double().numpy().reshape(-1) for k in names])
    flat = start.copy()
    adam = AdamOracle(flat.size, dtype=np.float64)
    cond = np.ones(flat.size, dtype=bool)
    for step in range(3):
        x, err = sample_syndromes(g, 64, [0.03, 0.06, 0.1], noise=1, seed=40 + step)
        tr.sync_module()
        train_step_grads(dec, g, x, err, logical)
        g_fused = torch.cat([prm.grad.reshape(-1).float() for _, prm in dec.named_parameters()])
        tr.step(x, err)
        assert torch.equal(tr.grad, g_fused), step
        yd = err.cpu().double()
        _, gr, _ = restate.decode_grad("v2_4", ei, g.V, g.C, x.cpu().double(), unflat(flat),
                                       lambda prob: restate.loss_v2_4(prob, yd, H, L), T=6, dtype=torch.float64)
        g_ref = np.concatenate([gr[k].numpy().reshape(-1) for k in names])
        off = 0
        for n in sizes:
            sl = slice(off, off + n)
            cond[sl] &= np.abs(g_ref[sl]) >= 5e-2 * np.abs(g_ref[sl]).max()
            off += n
        flat = adam.step(flat, g_ref)
    got = tr.w.double().cpu().numpy()
    lr = 3e-4
    assert np.abs(flat - start).max() > lr                     # the steps did move the weights
    assert cond.sum() > 0
    assert np.abs(got - flat)[cond].max() <= 0.1 * lr, np.abs(got - flat)[cond].max()
    assert np.abs(got - flat).max() <= 6 * lr


def test_refusals():
    """A permuted edge order on HGP [[1600,64]]: the streamed training forward needs the canonical order."""
    from gnn_decode_b200 import _cabi, codes
    from gnn_decode_b200.graph import TannerGraph
    pcm = codes.hgp_pcm()
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    perm = torch.from_numpy(np.random.RandomState(0).permutation(ei.size(1)))
    C, V = pcm.shape
    g = TannerGraph(ei[:, perm], V, C, DEV)
    dec = _decoder(_Case(FIXTURES[1]).weights, 3)
    x = torch.zeros((2, g.N), device=DEV)
    x[:, :V] = 3.0
    x[:, V:] = 1.0
    with pytest.raises(_cabi.GdError, match="canonical"):
        dec.decode(x, graph=g)
    torch.cuda.synchronize()

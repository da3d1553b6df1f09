"""The "next" update programs of SURVEY.md 8(f)-3 -- quantum/neural_BP.py (per-edge learned weights,
un-tied layers, gated residual) and quantum/QGNNNI_ca.py (GRUCell(1,1) updates, one prediction per
iteration).  CPU part: the oracle restatement against the fixtures written by the reference's own
classes (bit-exact) and against the reference run live; GPU part: the CUDA kernels against both."""
import numpy as np
import pytest
import torch

from conftest import Golden
from oracle import ref_loader, restate

CASES = {"ext_neural_bp_toricL4": "quantum.neural_BP", "ext_gru_ca_toricL4": "quantum.QGNNNI_ca"}
RTOL, LOGIT_TIE = 1e-4, 1e-3
pytestmark = pytest.mark.usefixtures("one_cpu_thread")


def _all_prob(name):
    z = np.load(__file__.rsplit("/", 1)[0] + "/golden/" + name + ".npz")
    return torch.from_numpy(z["all_prob"]) if "all_prob" in z.files else None


def _make(g, name):
    import importlib
    mod = importlib.import_module("gnn_decode_b200." + CASES[name])
    dec = mod.GNNI(g.T, n_edges=g.E) if g.program == "neural_bp" else mod.GNNI(g.T)
    dec.load_state_dict(g.weights, strict=True)
    return mod, dec


@pytest.mark.parametrize("name", sorted(CASES))
def test_restatement_matches_golden_bit_exact(name):
    g = Golden(name)
    out = restate.decode(g.program, g.edge_index, g.V, g.C, g.x, g.weights, T=g.T, dtype=g.dtype)
    assert out["prob"].dtype == g.dtype and torch.equal(out["prob"], g.prob)
    if g.program == "gru_ca":
        assert torch.equal(out["all_prob"], _all_prob(name))          # every iteration's prediction


MORE = {"ext_v3_0_toricL4": "quantum.decoder_v3_0", "ext_v1_2_2_toricL4": "quantum.decoder_v1_2_2", "ext_v2_4_1_toricL4": "quantum.decoder_v2_4_1"}


@pytest.mark.parametrize("name", sorted(CASES) + sorted(MORE))
def test_state_dict_and_weight_count(name):
    """The drop-in modules carry the reference's state_dict keys in the reference's order (the fixtures hold what the reference's own
    classes saved), and the packed weight buffer has the size the C ABI expects."""
    import ctypes as C
    import importlib
    from gnn_decode_b200 import _cabi
    g = Golden(name)
    if name in MORE:
        dec = importlib.import_module("gnn_decode_b200." + MORE[name]).GNNI(g.T)
        dec.load_state_dict(g.weights, strict=True)
    else:
        mod, dec = _make(g, name)
    assert list(dec.state_dict().keys()) == list(g.weights.keys())
    assert sum(p.numel() for p in dec._gd_params()) == _cabi.lib().gd_weights_size(C.byref(dec.gd_model()))


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference tree not mounted")
@pytest.mark.parametrize("script,program", [("quantum/neural_BP.py", "neural_bp"), ("quantum/QGNNNI_ca.py", "gru_ca")])
def test_restatement_matches_live_reference(script, program):
    with ref_loader.reference_session("quantum"):
        ns = ref_loader.load_reference(script, consts={"BATCH_SIZE": "6", "run1": "6", "run2": "6", "L": "4"}, seed=7)
        torch.manual_seed(3)
        dec = ns.GNNI(3)
        with torch.no_grad():
            for n_, p_ in dec.named_parameters():
                p_.copy_(torch.rand_like(p_) + 0.25 if program == "neural_bp" else p_ * 2)
        batch = next(iter(ns.train_loader))
        batch.x = batch.x.to(next(dec.parameters()).dtype)     # QGNNNI_ca is fp32, gen_syn emits fp64 (input cast only)
        with torch.no_grad():
            want = dec(batch)
        rows, cols = int(ns.rows), int(ns.cols)
        ei = batch.edge_index[:, : batch.edge_index.size(1) // 6]
        got = restate.decode(program, ei, rows, cols, batch.x.reshape(6, rows + cols), dec.state_dict(), T=3)
    if program == "gru_ca":
        assert len(want) == 3
        for i in range(3):
            assert torch.equal(got["all_prob"][i].reshape(-1, 1), want[i])
    else:
        assert torch.equal(got["prob"].reshape(-1, 1), want)


def test_v2_4_1_restatement_matches_golden_and_types():
    """quantum/decoder_v2_4_1.py (un-tied layers, one-hot edge types, gated residual): the restatement reproduces the fixture
    the reference's own classes wrote, bit for bit, and derives the same edge types from the graph alone."""
    g = Golden("ext_v2_4_1_toricL4")
    z = np.load(__file__.rsplit("/", 1)[0] + "/golden/ext_v2_4_1_toricL4.npz")
    assert torch.equal(restate.edge_types_v2_4_1(g.edge_index, g.C), torch.from_numpy(z["edge_types"]))
    out = restate.decode("v2_4_1", g.edge_index, g.V, g.C, g.x, g.weights, T=g.T, dtype=g.dtype)
    assert torch.equal(out["prob"], g.prob)
    from gnn_decode_b200.quantum import decoder_v2_4_1
    dec = decoder_v2_4_1.GNNI(g.T)
    assert list(dec.state_dict().keys()) == list(g.weights.keys())
    dec.load_state_dict(g.weights, strict=True)
    assert torch.equal(decoder_v2_4_1.edge_types(g.edge_index, g.C), torch.from_numpy(z["edge_types"]))


@pytest.mark.skipif(not ref_loader.reference_available(), reason="reference tree not mounted")
def test_v2_4_1_restatement_matches_live_reference():
    with ref_loader.reference_session("quantum"):
        ns = ref_loader.load_reference("quantum/decoder_v2_4_1.py", consts={"BATCH_SIZE": "6", "run1": "6", "run2": "6", "L": "4"}, seed=7,
                                       raw_subs=[("import decoder_v2_4\n", "\n")], truncate_at="'''\nload pretrained model")
        torch.manual_seed(3)
        dec = ns.GNNI(3)
        with torch.no_grad():
            for n_, p_ in dec.named_parameters():
                if n_.endswith("W") or n_.endswith("W_p"):
                    p_.copy_(torch.rand_like(p_) * 0.8 + 0.5)
        batch = next(iter(ns.train_loader))
        with torch.no_grad():
            want = dec(batch)
        rows, cols = int(ns.rows), int(ns.cols)
        ei = batch.edge_index[:, : batch.edge_index.size(1) // 6]
        got = restate.decode("v2_4_1", ei, rows, cols, batch.x.reshape(6, rows + cols), dec.state_dict(), T=3)
    assert torch.equal(got["prob"].reshape(-1, 1), want)


# ------------------------------------------------------------------------------------------ GPU
def _close(got, want, rtol):
    from conftest import logit_worst
    return logit_worst(got, want, rtol)


class _Data(object):
    def __init__(self, g, dev):
        self.x = g.x.reshape(-1, 1).to(dev, g.dtype)
        self.edge_index = g.batched_edge_index().to(dev)


def _graph(g, dev):
    from gnn_decode_b200.graph import TannerGraph
    return TannerGraph(g.edge_index, g.V, g.C, dev)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_fused_decoder_matches_reference(name):
    from gnn_decode_b200.graph import TannerGraph
    g = Golden(name)
    dev = torch.device("cuda", 0)
    mod, dec = _make(g, name)
    dec = dec.to(dev).eval()
    ref = restate.decode(g.program, g.edge_index, g.V, g.C, g.x, g.weights, T=g.T, dtype=torch.float64)
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    prob, logit, hard = dec.decode(g.x.to(dev), graph=tg, return_logits=True, return_hard=True)
    bp = g.program == "neural_bp"
    worst, max_err = _close(logit, ref["logit"], 2e-3 if bp else RTOL)      # sum-product bar: tests/test_parity_gpu.py
    assert worst <= 1.0, "logit mismatch: %.3g x bound (max abs err %.3g)" % (worst, max_err)
    assert (prob.double().cpu() - g.prob.double()).abs().max().item() <= (2e-3 if bp else 1e-5)
    decided = ref["logit"].abs() > LOGIT_TIE
    assert torch.equal(hard.cpu().bool()[decided], (g.prob > 0.5)[decided])
    with torch.no_grad():
        pred = dec(_Data(g, dev))                                          # the reference's entry point
    if g.program == "gru_ca":
        assert isinstance(pred, list) and len(pred) == g.T
        allp, alll = dec.decode_all(g.x.to(dev), graph=tg, return_logits=True)
        assert torch.equal(allp[-1], prob) and torch.equal(pred[-1].reshape(g.B, g.V), prob)
        worst, max_err = _close(alll, ref["all_logit"], RTOL)
        assert worst <= 1.0, "per-iteration logits: %.3g x bound (max abs %.3g)" % (worst, max_err)
        assert (allp.double().cpu() - _all_prob(name).double()).abs().max().item() <= 1e-5
    else:
        assert pred.shape == (g.B * g.V, 1) and pred.dtype == g.dtype
        assert torch.equal(pred.reshape(g.B, g.V).float(), prob)
    # deterministic, independent of the tiling
    x5 = g.x.repeat(5, 1).to(dev)
    p5 = dec.decode(x5, graph=tg)
    assert torch.equal(p5, dec.decode(x5, graph=tg)) and torch.equal(p5[:g.B], prob) and torch.equal(p5[-g.B:], prob)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_single_layer_matches_reference(name):
    """GraphConv.forward / GatedGraphConv.forward == propagate + update (+ GRUCell) through gd_propagate_fwd."""
    g = Golden(name)
    dev = torch.device("cuda", 0)
    mod, dec = _make(g, name)
    dec = dec.to(dev).eval()
    dec.bind_code(g.V, g.C)
    ei = g.batched_edge_index().to(dev)
    ei[1] += g.V
    x = g.x.reshape(-1, 1).to(dev, g.dtype)
    m0 = g.m0.reshape(-1, 1).to(dev, g.dtype)
    with torch.no_grad():
        if g.program == "neural_bp":
            got_var, got_chk = dec.layers[0](m0, ei, x), dec.layers[1](m0, ei, x)
        else:
            got_var, got_chk = dec.ggc1(m0, ei, x, [])[0], dec.ggc2(m0, ei, x, [])[0]
    for got, want, rtol in ((got_var, g.phase_var, RTOL), (got_chk, g.phase_chk, 2e-3 if g.program == "neural_bp" else RTOL)):
        assert got.shape == (g.B * g.E, 1) and got.dtype == g.dtype
        worst, max_err = _close(got.reshape(g.B, g.E), want, rtol)
        assert worst <= 1.0, "phase mismatch %.3g x bound (max abs %.3g)" % (worst, max_err)


@pytest.mark.gpu
def test_ext_programs_reject_what_they_do_not_support():
    from gnn_decode_b200 import _cabi, codes
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.quantum import neural_BP, QGNNNI_ca
    dev = torch.device("cuda", 0)
    g = Golden("ext_neural_bp_toricL4")
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    bad = neural_BP.GNNI(2, n_edges=g.E + 1).to(dev).eval()
    with pytest.raises(ValueError):
        bad.decode(g.x.to(dev), graph=tg)                                  # per-edge weight count != E
    big = TannerGraph.from_pcm(codes.hgp_pcm(), dev)                       # too large for the resident kernel
    dec = QGNNNI_ca.GNNI(2).to(dev).eval()
    with pytest.raises(_cabi.GdError):
        dec.decode(torch.zeros(8, big.N, device=dev), graph=big)


# ---- quantum/decoder_v1_1.py: neural BP with weights shared per edge type (one-hot feat_onehot) ----------------------
def _v1_1_fixture():
    z = np.load(__file__.rsplit("/", 1)[0] + "/golden/ext_v1_1_onehot_toricL4.npz")
    g = Golden("ext_v1_1_onehot_toricL4")
    types = torch.from_numpy(z["edge_types"])
    return g, types, int(z["nb_digits"])


def _expand_v1_1(w, types, T):
    """Per-edge weight vectors of the neural_bp program from decoder_v1_1's type tables: matmul(m * onehot, W) == m * W[type]."""
    out = {}
    for l in range(T):
        out["layers.%d.W" % (2 * l)] = w["layers.%d.W" % (2 * l)][types]
        out["layers.%d.W_p" % (2 * l)] = w["layers.%d.W_p" % (2 * l)][types]
    out["W"], out["W_p"], out["alpha"] = w["W"][types], w["W_p"][types], w["alpha"]
    return out


def test_v1_1_onehot_restatement_matches_golden_bit_exact():
    g, types, nb = _v1_1_fixture()
    out = restate.decode("neural_bp", g.edge_index, g.V, g.C, g.x, _expand_v1_1(g.weights, types, g.T), T=g.T, dtype=g.dtype)
    assert torch.equal(out["prob"], g.prob)


def test_v1_1_state_dict_keys():
    from gnn_decode_b200.quantum import decoder_v1_1
    g, types, nb = _v1_1_fixture()
    dec = decoder_v1_1.GNNI(g.T, edge_types=types, nb_digits=nb)
    assert list(dec.state_dict().keys()) == list(g.weights.keys())          # target_to_source layers own no parameters
    dec.load_state_dict(g.weights, strict=True)
    assert sum(p.numel() for p in dec._gd_params()) == (2 * g.T + 2) * g.E + 1


@pytest.mark.gpu
def test_v1_1_onehot_decoder_matches_reference():
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.quantum import decoder_v1_1
    g, types, nb = _v1_1_fixture()
    dev = torch.device("cuda", 0)
    dec = decoder_v1_1.GNNI(g.T, edge_types=types, nb_digits=nb)
    dec.load_state_dict(g.weights, strict=True)
    dec = dec.to(dev).eval()
    ref = restate.decode("neural_bp", g.edge_index, g.V, g.C, g.x, _expand_v1_1(g.weights, types, g.T), T=g.T, dtype=torch.float64)
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    prob, logit, hard = dec.decode(g.x.to(dev), graph=tg, return_logits=True, return_hard=True)
    worst, max_err = _close(logit, ref["logit"], 2e-3)
    assert worst <= 1.0, "logit mismatch: %.3g x bound (max abs err %.3g)" % (worst, max_err)
    assert (prob.double().cpu() - g.prob.double()).abs().max().item() <= 2e-3
    decided = ref["logit"].abs() > LOGIT_TIE
    assert torch.equal(hard.cpu().bool()[decided], (g.prob > 0.5)[decided])
    with torch.no_grad():
        pred = dec(_Data(g, dev))
    assert pred.shape == (g.B * g.V, 1) and torch.equal(pred.reshape(g.B, g.V).float(), prob)
    # a weight update is picked up by the next call (type tables are re-gathered)
    with torch.no_grad():
        dec.W.mul_(1.5)
    assert not torch.equal(dec.decode(g.x.to(dev), graph=tg), prob)


@pytest.mark.gpu
def test_v2_4_1_fused_and_per_layer_match_reference_fixture():
    """decoder_v2_4_1: (a) GNNI.forward = the fused kernel (GD_PROG_V2_4_1: un-tied layers re-staged per iteration, edge types derived
    in the kernel), (b) forward_layers = every layer's propagate() on the CUDA propagate kernel with the script's own update()s in
    torch -- both against the probabilities the reference itself produced and the fp64 restatement's logits."""
    from gnn_decode_b200.quantum import decoder_v2_4_1
    g = Golden("ext_v2_4_1_toricL4")
    dev = torch.device("cuda", 0)
    dec = decoder_v2_4_1.GNNI(g.T)
    dec.load_state_dict(g.weights, strict=True)
    dec = dec.to(dev).eval()
    d = _Data(g, dev)
    ref = restate.decode("v2_4_1", g.edge_index, g.V, g.C, g.x, g.weights, T=g.T)
    assert torch.equal(ref["prob"], g.prob)
    with torch.no_grad():
        outs = {"fused": dec(d), "fused again": dec(d), "layers": dec.forward_layers(d)}
    assert torch.equal(outs["fused"], outs["fused again"])
    for name, prob in outs.items():
        assert prob.shape == (g.B * g.V, 1) and prob.dtype == torch.float64, name
        logit = -torch.log(prob / (1 - prob)).reshape(g.B, g.V)
        worst, max_err = _close(logit, ref["logit"], RTOL)
        assert worst <= 1.0, "%s logits: %.3g x the bar (max abs err %.3g)" % (name, worst, max_err)
        assert (prob.reshape(g.B, g.V).cpu() - g.prob).abs().max().item() < 1e-5, name
    # logits straight from the kernel (no sigmoid round trip), hard decisions
    tg = _graph(g, dev)
    prob, logit, hard = dec.decode(g.x.to(dev), graph=tg, return_logits=True, return_hard=True)
    worst, max_err = _close(logit, ref["logit"], RTOL)
    assert worst <= 1.0, (worst, max_err)
    decided = ref["logit"].abs() > LOGIT_TIE
    assert torch.equal(hard.cpu().bool()[decided], (ref["logit"] < 0)[decided])
    # a code whose checks do not all have four edges is refused, as the reference's feat_onehot construction would fail on it
    from gnn_decode_b200 import codes
    from gnn_decode_b200.graph import TannerGraph
    rot = TannerGraph.from_pcm(codes.rotated_surface_pcm(3), dev)
    with pytest.raises(ValueError, match="exactly 4 edges"):
        dec.decode(torch.ones(4, rot.N, device=dev), graph=rot)


@pytest.mark.parametrize("name,prog", [("ext_v3_0_toricL4", "v3_0"), ("ext_v1_2_2_toricL4", "v1_2_2")])
def test_v3_0_and_v1_2_2_restatements_match_golden(name, prog):
    """quantum/decoder_v3_0.py (2-input ReLU MLPs + GRUCell per phase, two read-outs over all V+C nodes) and
    quantum/decoder_v1_2_2.py (Tanh MLP variable phase, sum-product check phase, a prediction per iteration): the restatements
    reproduce what the reference's own classes produced, bit for bit."""
    g = Golden(name)
    z = np.load(__file__.rsplit("/", 1)[0] + "/golden/%s.npz" % name)
    out = restate.decode(prog, g.edge_index, g.V, g.C, g.x, g.weights, T=g.T, dtype=g.dtype)
    if prog == "v3_0":
        assert torch.equal(out["prob_all"], torch.from_numpy(z["prob_all"])) and torch.equal(out["prob_p_all"], torch.from_numpy(z["prob_p_all"]))
        assert torch.equal(out["prob"], g.prob)
    else:
        assert torch.equal(out["all_prob"], torch.from_numpy(z["all_prob"])) and out["all_prob"].shape == (g.T, g.B, g.V)


@pytest.mark.parametrize("script,prog,T", [("quantum/decoder_v3_0.py", "v3_0", 3), ("quantum/decoder_v1_2_2.py", "v1_2_2", 3)])
def test_v3_0_and_v1_2_2_restatements_match_live_reference(script, prog, T):
    if not ref_loader.reference_available():
        pytest.skip("reference tree not mounted")
    consts = {"BATCH_SIZE": "6", "run1": "6", "run2": "6", "L": "4"}
    if prog == "v3_0":
        consts["Nc"] = str(T)                                  # the script compares the loop index with its GLOBAL Nc (:267)
    with ref_loader.reference_session("quantum"):
        ns = ref_loader.load_reference(script, consts=consts, seed=11)
        torch.manual_seed(12)
        dec = ns.GNNI(T)
        with torch.no_grad():
            for n_, p_ in dec.named_parameters():
                if "bias" in n_:
                    p_.add_(0.3 * torch.randn_like(p_))
        batch = next(iter(ns.train_loader))
        with torch.no_grad():
            pred = dec(batch)
        rows, cols = int(ns.rows), int(ns.cols)
        E = batch.edge_index.size(1) // 6
        got = restate.decode(prog, batch.edge_index[:, :E].clone(), rows, cols, batch.x.reshape(6, rows + cols), dec.state_dict(), T=T)
        if prog == "v3_0":
            assert torch.equal(got["prob_all"].reshape(-1, 1), pred[0]) and torch.equal(got["prob_p_all"].reshape(-1, 1), pred[1])
        else:
            assert len(pred) == T
            for i in range(T):
                assert torch.equal(got["all_prob"][i].reshape(-1, 1), pred[i])


@pytest.mark.gpu
def test_v1_2_2_fused_decoder_matches_reference_fixture():
    """decoder_v1_2_2 through the drop-in GNNI (fused kernel, GD_PROG_V1_2_2 with a read-out per iteration): the list of predictions
    against what the reference itself produced, logits against the fp64 restatement."""
    from gnn_decode_b200.quantum import decoder_v1_2_2
    g = Golden("ext_v1_2_2_toricL4")
    z = np.load(__file__.rsplit("/", 1)[0] + "/golden/ext_v1_2_2_toricL4.npz")
    dev = torch.device("cuda", 0)
    dec = decoder_v1_2_2.GNNI(g.T)
    dec.load_state_dict(g.weights, strict=True)
    dec = dec.to(dev).eval()
    with torch.no_grad():
        preds = dec(_Data(g, dev))
    assert isinstance(preds, list) and len(preds) == g.T and preds[0].shape == (g.B * g.V, 1) and preds[0].dtype == torch.float64
    ref = restate.decode("v1_2_2", g.edge_index, g.V, g.C, g.x, g.weights, T=g.T)
    _, logits = dec.decode_all(g.x.to(dev), graph=_graph(g, dev), return_logits=True)
    for i in range(g.T):
        worst, max_err = _close(logits[i], ref["all_logit"][i], RTOL)
        assert worst <= 1.0, "iteration %d logits: %.3g x the bar (max abs err %.3g)" % (i, worst, max_err)
        assert (preds[i].reshape(g.B, g.V).cpu() - torch.from_numpy(z["all_prob"][i])).abs().max().item() < 2e-5
    assert torch.equal(dec.decode(g.x.to(dev), graph=_graph(g, dev)), dec.decode_all(g.x.to(dev), graph=_graph(g, dev))[-1])


@pytest.mark.gpu
def test_v1_2_2_layers_run_the_propagate_kernel():
    """The per-layer classes (the reference's plugin API): ggc1 = propagate kernel + this script's Tanh MLP in torch, ggc2 = the
    sum-product check rule in the kernel; iterated by hand as GNNI.forward does (:264-267), the messages match the restatement."""
    from gnn_decode_b200.quantum import decoder_v1_2_2
    g = Golden("ext_v1_2_2_toricL4")
    dev = torch.device("cuda", 0)
    dec = decoder_v1_2_2.GNNI(g.T)
    dec.load_state_dict(g.weights, strict=True)
    dec = dec.to(dev).eval().bind_code(g.V, g.C)
    d = _Data(g, dev)
    ei = torch.cat([d.edge_index[0].unsqueeze(0), d.edge_index[1].unsqueeze(0).add(g.V)], 0)
    m = torch.zeros((ei.size(1), 1), dtype=torch.float64, device=dev)
    with torch.no_grad():
        for _ in range(g.T):
            m_p = m.clone()
            m = dec.ggc1(m, ei, d.x)
            m = dec.ggc2(m, ei, d.x) + m_p
    ref = restate.decode("v1_2_2", g.edge_index, g.V, g.C, g.x, g.weights, T=g.T)["m"]
    err = (m.reshape(g.B, g.E).cpu() - ref).abs()
    assert float((err / ref.abs().clamp_min(1.0)).max()) <= 1e-4, err.max().item()


@pytest.mark.gpu
def test_v3_0_fused_decoder_matches_reference_fixture():
    """decoder_v3_0 through the drop-in GNNI (fused kernel GD_PROG_V3_0 + its second read-out): the reference's two [B*(V+C), 1]
    outputs, logits of both read-outs against the fp64 restatement; the per-layer classes (propagate kernel + torch MLP + GRUCell)
    reproduce the messages."""
    from gnn_decode_b200.quantum import decoder_v3_0
    g = Golden("ext_v3_0_toricL4")
    z = np.load(__file__.rsplit("/", 1)[0] + "/golden/ext_v3_0_toricL4.npz")
    dev = torch.device("cuda", 0)
    dec = decoder_v3_0.GNNI(g.T)
    dec.load_state_dict(g.weights, strict=True)
    dec = dec.to(dev).eval()
    d = _Data(g, dev)
    with torch.no_grad():
        out = dec(d)
    N = g.V + g.C
    assert isinstance(out, list) and len(out) == 2 and out[0].shape == (g.B * N, 1) and out[0].dtype == torch.float64
    assert (out[0].reshape(g.B, N).cpu() - torch.from_numpy(z["prob_all"])).abs().max().item() < 1e-5
    assert (out[1].reshape(g.B, N).cpu() - torch.from_numpy(z["prob_p_all"])).abs().max().item() < 1e-5
    ref = restate.decode("v3_0", g.edge_index, g.V, g.C, g.x, g.weights, T=g.T)
    tg = _graph(g, dev)
    prob, prob_c, logit, logit_c = dec.decode_aux(g.x.to(dev), graph=tg, return_logits=True)
    for got, want in ((logit, ref["logit"]), (logit_c, ref["logit_chk"])):
        worst, max_err = _close(got, want, RTOL)
        assert worst <= 1.0, "logits: %.3g x the bar (max abs err %.3g)" % (worst, max_err)
    assert torch.equal(dec.decode(g.x.to(dev), graph=tg), prob)
    # per-layer classes, iterated as GNNI.forward does (:264-270)
    ei = torch.cat([d.edge_index[0].unsqueeze(0), d.edge_index[1].unsqueeze(0).add(g.V)], 0)
    m = torch.zeros((ei.size(1), 1), dtype=torch.float64, device=dev)
    dec.bind_code(g.V, g.C)
    with torch.no_grad():
        for _ in range(g.T):
            m = dec.ggc1(m, ei, d.x)
            m = dec.ggc2(m, ei, d.x)
    err = (m.reshape(g.B, g.E).cpu() - ref["m"]).abs()
    assert float((err / ref["m"].abs().clamp_min(1.0)).max()) <= 1e-4, err.max().item()

"""GPU suite: the CUDA path, called through the C ABI, against the oracle and the golden vectors.

Bars (BASELINE.json north_star):
  * graph / index tables: bit-exact;
  * hard decisions: bit-exact wherever the reference's own logit is not within LOGIT_TIE of 0;
  * soft logits: |cuda_fp32 - reference| <= RTOL * max(|reference|, 1), RTOL = 1e-4 (conftest.logit_bound: relative
    above |logit| = 1, the same number absolute below it).
    The sum-product (BP) programs are ill-conditioned in the saturated regime (the fp32 reference
    itself is ~1e-2 away from the fp64 evaluation of its own formulas there), so for them the bar is
    RTOL_BP against the fp64 oracle plus hard-decision equality.
"""
import numpy as np
import pytest
import torch

from conftest import Golden, golden_cases, logit_worst, make_decoder
from oracle import restate

pytestmark = pytest.mark.gpu

RTOL, RTOL_BP, LOGIT_TIE = 1e-4, 5e-4, 1e-3     # measured: v2_4 <= 0.08 x, sum-product <= 0.05 x these bars (profiles/r02_parity_envelope.txt)


def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda", 0)


def _logit_close(got, want, rtol):
    return logit_worst(got, want, rtol)


class _Data(object):
    def __init__(self, g, dev, dtype=None):
        self.x = g.x.reshape(-1, 1).to(dev, dtype or g.dtype)
        self.edge_index = g.batched_edge_index().to(dev)


@pytest.mark.parametrize("name", golden_cases())
def test_graph_tables_bit_exact(name):
    from gnn_decode_b200.graph import TannerGraph
    g = Golden(name)
    tg = TannerGraph(g.edge_index, g.V, g.C, _dev())
    t = tg.tables()
    ei = g.edge_index.numpy()
    assert np.array_equal(t["edge_var"], ei[0]) and np.array_equal(t["edge_chk"], ei[1])
    for ptr, ids, key, n in ((t["var_ptr"], t["var_edges"], ei[0], g.V), (t["chk_ptr"], t["chk_edges"], ei[1], g.C)):
        order = np.argsort(key, kind="stable")            # destination-sorted, ascending edge id inside
        assert np.array_equal(ids, order.astype(np.int32))
        assert np.array_equal(ptr, np.concatenate([[0], np.cumsum(np.bincount(key, minlength=n))]).astype(np.int32))
    # H.to_sparse()._indices() route gives the same graph
    tg2 = TannerGraph.from_H(g.H, _dev())
    assert torch.equal(tg2.edge_index, g.edge_index)


def test_batched_edge_index_check():
    from gnn_decode_b200.graph import TannerGraph
    g = Golden("v2_4_toricL4_epoch1")
    dev = _dev()
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    ei = g.batched_edge_index().to(dev)
    assert tg.check_batched(ei, g.B, 0) == 0
    ei2 = ei.clone()
    ei2[1] += g.V
    assert tg.check_batched(ei2, g.B, g.V) == 0
    ei2[0, 5] += 1
    assert tg.check_batched(ei2, g.B, g.V) == 1
    dec = make_decoder(g)[1].to(dev)
    d = _Data(g, dev)
    d.edge_index = ei2 - torch.tensor([[0], [g.V]], device=dev)
    with pytest.raises(ValueError):
        dec(d)


@pytest.mark.parametrize("name", golden_cases())
def test_fused_decoder_matches_reference(name):
    g = Golden(name)
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    ref = restate.decode(g.program, g.edge_index, g.V, g.C, g.x, g.weights, T=g.T, dtype=torch.float64)
    with torch.no_grad():
        pred = dec(_Data(g, dev))                                   # the reference's entry point
    assert pred.shape == (g.B * g.V, 1) and pred.dtype == g.dtype
    from gnn_decode_b200.graph import TannerGraph
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    prob, logit, hard = dec.decode(g.x.to(dev), graph=tg, return_logits=True, return_hard=True)
    assert torch.equal(pred.reshape(g.B, g.V).float(), prob)
    bp = g.program.startswith("bp")
    worst, max_err = _logit_close(logit, ref["logit"], RTOL_BP if bp else RTOL)
    assert worst <= 1.0, "logit mismatch: %.3g x bound (max abs err %.3g)" % (worst, max_err)
    # probabilities against the golden output of the reference's own code (its dtype)
    perr = (prob.double().cpu() - g.prob.double()).abs().max().item()
    # 5e-5: the collapsed epoch67 checkpoint (|logit| up to ~600) sits at 1.8e-5 with every MLP tabulated, 90x inside the logit bar
    assert perr <= (2e-3 if bp else 5e-5), "prob mismatch %.3g (logit: %.3g x bound, max abs err %.3g)" % (perr, worst, max_err)
    # hard decisions bit-exact away from ties
    want_hard = (g.prob > 0.5)
    decided = ref["logit"].abs() > LOGIT_TIE
    assert torch.equal(hard.cpu().bool()[decided], want_hard[decided])
    assert torch.equal(hard.bool(), prob > 0.5)


@pytest.mark.parametrize("name", golden_cases())
def test_single_propagate_matches_reference(name):
    """GraphConv.forward == propagate + update, through gd_propagate_fwd."""
    g = Golden(name)
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    dec.bind_code(g.V, g.C)
    ei = g.batched_edge_index().to(dev)
    ei[1] += g.V                                                    # what GNNI.forward hands to GraphConv
    x = g.x.reshape(-1, 1).to(dev, g.dtype)
    m0 = g.m0.reshape(-1, 1).to(dev, g.dtype)
    bp = g.program.startswith("bp")
    with torch.no_grad():
        got_var = dec.ggc1(m0, ei, x)
        got_chk = dec.ggc2(m0, ei) if g.program in ("cgnni", "bp_classical") else dec.ggc2(m0, ei, x)
    for got, want in ((got_var, g.phase_var), (got_chk, g.phase_chk)):
        assert got.shape == (g.B * g.E, 1) and got.dtype == g.dtype
        worst, max_err = _logit_close(got.reshape(g.B, g.E), want, RTOL_BP if bp else RTOL)
        assert worst <= 1.0, "phase mismatch %.3g x bound (max abs %.3g)" % (worst, max_err)


def test_custom_update_override_runs_unfused():
    """A user subclass overriding update() gets the reference's pre/reduce/post tensor."""
    from gnn_decode_b200.quantum import decoder_v2_4 as q
    g = Golden("v2_4_toricL4_epoch1")
    dev = _dev()
    seen = {}

    class MyConv(q.GraphConv):
        def update(self, aggr_out):
            seen["shape"] = tuple(aggr_out.shape)
            return aggr_out[:, :1] * 2 + aggr_out[:, 1:]

    conv = MyConv("target_to_source").to(dev)
    ei = g.batched_edge_index().to(dev)
    ei[1] += g.V
    x = g.x.reshape(-1, 1).to(dev)
    m0 = g.m0.reshape(-1, 1).to(dev)
    out = conv(m0, ei, x)
    assert seen["shape"] == (g.B * g.E, 2)
    t = torch.tanh(g.m0.double() / 2)
    chk = g.edge_index[1]
    S = torch.zeros(g.B, g.C, dtype=torch.float64).index_add_(1, chk, t)
    want = (S[:, chk] - t) * 2 + g.x[:, g.V:][:, chk]
    assert (out.reshape(g.B, g.E).double().cpu() - want).abs().max().item() < 1e-5


def test_deterministic_and_partial_tiles():
    """Bit-repeatable (atomic-free reductions) and independent of how the batch is tiled."""
    g = Golden("v2_4_toricL5_epoch3")
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    from gnn_decode_b200.graph import TannerGraph
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    gen = torch.Generator().manual_seed(5)
    reps = 37                                                       # 37*16 = 592 syndromes: ragged last tile
    x = g.x.repeat(reps, 1).to(dev)
    a = dec.decode(x, graph=tg)
    b = dec.decode(x, graph=tg)
    assert torch.equal(a, b)
    small = dec.decode(g.x.to(dev), graph=tg)
    assert torch.equal(a.reshape(reps, g.B, g.V), small.unsqueeze(0).expand(reps, -1, -1))
    one = dec.decode(g.x[3:4].to(dev), graph=tg)                     # B = 1
    assert torch.equal(one, small[3:4])
    empty = dec.decode(g.x[:0].to(dev), graph=tg)                    # B = 0
    assert empty.shape == (0, g.V)


def test_decode_host_matches_device_path():
    g = Golden("v2_4_toricL4_epoch1")
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    from gnn_decode_b200.graph import TannerGraph
    dec.bind_graph(TannerGraph(g.edge_index, g.V, g.C, dev))
    reps = 1100                                                      # 17600 syndromes: several chunks
    xh = g.x.float().repeat(reps, 1).contiguous().pin_memory()
    prob_h = torch.empty(xh.size(0), g.V, dtype=torch.float32).pin_memory()
    hard_h = torch.empty(xh.size(0), g.V, dtype=torch.uint8).pin_memory()
    dec.decode_host(xh, prob_h, hard_h)
    prob_d, hard_d = dec.decode(xh.to(dev), return_hard=True)
    assert torch.equal(prob_h, prob_d.cpu()) and torch.equal(hard_h, hard_d.cpu())


def test_fp32_and_fp64_inputs_agree():
    g = Golden("qgnni_toricL4_seeded")
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    p64 = dec(_Data(g, dev, torch.float64))
    p32 = dec(_Data(g, dev, torch.float32))
    assert p64.dtype == torch.float64 and p32.dtype == torch.float32
    assert torch.equal(p64.float(), p32)


@pytest.mark.parametrize("name", ["v2_4_toricL4_epoch1", "qgnni_toricL4_seeded", "cgnni_bch_seeded", "cgnni_ldpc_epoch18",
                                  "bp_quantum_toricL4", "bp_classical_bch"])
def test_streamed_kernel_matches_resident_and_reference(name, gd_opt):
    """The global-memory (streamed) kernel used for codes too large for shared memory, forced on
    a small code: same logits as the oracle (same bar) and hard decisions identical to the
    resident kernel."""
    g = Golden(name)
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    from gnn_decode_b200.graph import TannerGraph
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    x = g.x.repeat(5, 1).to(dev)                                   # 80..160 syndromes: ragged tiles
    p_res, l_res, h_res = dec.decode(x, graph=tg, return_logits=True, return_hard=True)
    gd_opt.set("GD_FORCE_STREAMED")
    assert tg.launch_info(dec.gd_model(), x.size(0))["resident"] == 0
    p_str, l_str, h_str = dec.decode(x, graph=tg, return_logits=True, return_hard=True)
    p_str2 = dec.decode(x, graph=tg)
    gd_opt.unset("GD_FORCE_STREAMED")
    assert torch.equal(p_str, p_str2)                               # deterministic
    ref = restate.decode(g.program, g.edge_index, g.V, g.C, g.x, g.weights, T=g.T, dtype=torch.float64)
    bp = g.program.startswith("bp")
    worst, max_err = _logit_close(l_str[:g.B], ref["logit"], RTOL_BP if bp else RTOL)
    assert worst <= 1.0, "streamed logit mismatch: %.3g x bound (max abs %.3g)" % (worst, max_err)
    decided = (ref["logit"].abs() > LOGIT_TIE).repeat(5, 1)
    assert torch.equal(h_str.cpu()[decided], h_res.cpu()[decided])


def test_hgp_1600_streamed_matches_oracle():
    """BASELINE config 5 shape: hypergraph-product [[1600,64]] (E = 10752) takes the streamed path."""
    from gnn_decode_b200 import codes
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.quantum import QGNNI, BP
    from gnn_decode_b200.sampler import sample_syndromes
    dev = _dev()
    pcm = codes.hgp_pcm()
    tg = TannerGraph.from_pcm(pcm, dev)
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    x, _ = sample_syndromes(tg, 40, [0.02, 0.05], noise=1, seed=9)
    torch.manual_seed(0)
    dec = QGNNI.GNNI(6).to(dev).eval()
    assert tg.launch_info(dec.gd_model(), 40)["resident"] == 0
    prob, logit = dec.decode(x, graph=tg, return_logits=True)
    ref = restate.decode("qgnni", ei, tg.V, tg.C, x.cpu().double(), {k: v.cpu() for k, v in dec.state_dict().items()}, T=6)
    worst, max_err = _logit_close(logit, ref["logit"], RTOL)
    assert worst <= 1.0, "HGP qgnni: %.3g x bound (max abs %.3g)" % (worst, max_err)
    bpd = BP.GNNI(8).to(dev).eval()
    prob, logit, hard = bpd.decode(x, graph=tg, return_logits=True, return_hard=True)
    ref = restate.decode("bp_quantum", ei, tg.V, tg.C, x.cpu().double(), {}, T=8)
    worst, max_err = _logit_close(logit, ref["logit"], 2e-3)      # degree-7 checks, saturated messages: the round-1 sum-product bar
    assert worst <= 1.0, "HGP bp: %.3g x bound (max abs %.3g)" % (worst, max_err)
    decided = ref["logit"].abs() > LOGIT_TIE
    assert torch.equal(hard.cpu().bool()[decided], (ref["prob"] > 0.5)[decided])


@pytest.mark.parametrize("scale,T", [(1.0, 15), (6.0, 4), (1.0, 60)])
def test_v2_4_tabulated_mlps_match_direct_evaluation_and_oracle(scale, T, gd_opt):
    """decoder_v2_4's 1->128->1 check-phase and read-out MLPs run from per-launch cubic tables when the
    in-kernel error bound allows (DESIGN.md 4.1).  (a) tabulated == direct evaluation (GD_NO_CTAB) far inside
    the logit tolerance; (b) with first-layer weights scaled up the bound fails and the kernel must fall back
    by itself -- results still match the oracle; (c) a long run (T = 60) widens the read-out domain."""
    from gnn_decode_b200.graph import TannerGraph
    g = Golden("v2_4_toricL5_epoch3")
    dev = _dev()
    w = {k: v.clone() for k, v in g.weights.items()}
    for k in ("ggc2.mlp.0.weight", "mlp.0.weight"):
        w[k] = w[k] * scale
    mod, dec = make_decoder(g)
    dec.Nc = T
    dec.load_state_dict(w)
    dec = dec.to(dev).eval()
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    x = g.x.repeat(9, 1).to(dev)
    _, l_tab, h_tab = dec.decode(x, graph=tg, return_logits=True, return_hard=True)
    gd_opt.set("GD_NO_CTAB")
    _, l_dir, h_dir = dec.decode(x, graph=tg, return_logits=True, return_hard=True)
    gd_opt.unset("GD_NO_CTAB")
    ref = restate.decode("v2_4", g.edge_index, g.V, g.C, g.x, w, T=T, dtype=torch.float64)
    for l in (l_tab, l_dir):
        worst, max_err = _logit_close(l[:g.B], ref["logit"], RTOL)
        assert worst <= 1.0, "logit mismatch: %.3g x bound (max abs err %.3g)" % (worst, max_err)
    rms = ref["logit"].pow(2).mean().sqrt().item()
    assert (l_tab - l_dir).abs().max().item() <= 2e-5 * (1.0 + rms)
    decided = (ref["logit"].abs() > LOGIT_TIE).repeat(9, 1)
    assert torch.equal(h_tab.cpu()[decided], h_dir.cpu()[decided])


def test_autotuned_geometry_gives_identical_results():
    """gd_decode_autotune times candidate (tile, R, EB) geometries and pins the fastest for (graph, model, B): the
    arithmetic per syndrome does not depend on the geometry, so results stay bit-identical, and other batch sizes
    keep the planner's choice."""
    from gnn_decode_b200.graph import TannerGraph
    g = Golden("v2_4_toricL5_epoch3")
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    x = g.x.repeat(300, 1).to(dev)                                   # 4800 syndromes
    before = dec.decode(x, graph=tg)
    info0 = tg.launch_info(dec.gd_model(), x.size(0))
    info = dec.autotune(x, graph=tg, max_candidates=6)
    assert info["resident"] == 1 and info["tile"] > 0
    assert tg.launch_info(dec.gd_model(), x.size(0)) == info        # the tuned geometry is what later launches use
    assert torch.equal(dec.decode(x, graph=tg), before)
    assert tg.launch_info(dec.gd_model(), x.size(0) + 8) == tg.launch_info(dec.gd_model(), x.size(0) + 8)
    other = dec.decode(x[:1000].contiguous(), graph=tg)             # a different B: untouched by the cache
    assert torch.equal(other, before[:1000])
    assert isinstance(info0, dict)


def test_decode_host_pipeline(gd_opt):
    """gd_decode_host (chunks through the graph's internal gd_pipeline): bit-identical to the device path on ragged batch
    sizes, repeated and changing batch sizes, either output alone, pageable input, a fresh graph context, the edge-owner
    kernel, the streamed kernel (one chunk), and a second decoder with another T on the same graph (a new pipeline)."""
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.sampler import sample_syndromes
    g = Golden("v2_4_toricL4_epoch1")
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    dec.bind_graph(tg)
    x_all, _ = sample_syndromes(tg, 40000, [0.01, 0.04, 0.08, 0.12], noise=0, seed=77)     # every syndrome different
    ref_p, ref_h = dec.decode(x_all, return_hard=True)
    ref_p, ref_h = ref_p.cpu(), ref_h.cpu()
    xh_all = x_all.cpu().pin_memory()

    def both(dec, B, graph=None):
        prob_h = torch.zeros(B, g.V, dtype=torch.float32).pin_memory()
        hard_h = torch.full((B, g.V), 7, dtype=torch.uint8).pin_memory()
        dec.decode_host(xh_all[:B], prob_h, hard_h, graph=graph)
        return prob_h, hard_h

    for B in (40000, 16384, 20001, 33333, 40000):
        prob_h, hard_h = both(dec, B)
        assert torch.equal(prob_h, ref_p[:B]) and torch.equal(hard_h, ref_h[:B]), B
    only_h = dec.decode_host(xh_all, hard_out=torch.empty(40000, g.V, dtype=torch.uint8).pin_memory())
    assert torch.equal(only_h, ref_h)
    only_p = dec.decode_host(xh_all)
    assert torch.equal(only_p, ref_p)
    pageable = dec.decode_host(x_all.cpu()[:17000].clone())                                # pageable host memory works too
    assert torch.equal(pageable, ref_p[:17000])
    tg2 = TannerGraph(g.edge_index, g.V, g.C, dev)                                         # a fresh graph context
    p2 = dec.decode_host(xh_all, graph=tg2)
    assert torch.equal(p2, ref_p)
    for opt, B in (("GD_NO_LEAN", 40000), ("GD_FORCE_STREAMED", 20001)):                   # edge-owner; streamed: one chunk
        gd_opt.set(opt)
        p_d, h_d = dec.decode(x_all[:B], return_hard=True)
        prob_h, hard_h = both(dec, B)
        gd_opt.unset(opt)
        assert torch.equal(prob_h, p_d.cpu()) and torch.equal(hard_h, h_d.cpu()), opt
    dec_t = mod.GNNI(g.T + 2)                                                              # another model on the same graph
    dec_t.load_state_dict(g.weights, strict=True)
    dec_t = dec_t.to(dev).eval()
    p_t, h_t = dec_t.decode(x_all, graph=tg, return_hard=True)
    prob_h, hard_h = both(dec_t, 40000, graph=tg)
    assert torch.equal(prob_h, p_t.cpu()) and torch.equal(hard_h, h_t.cpu())
    assert not torch.equal(p_t.cpu(), ref_p)


@pytest.mark.parametrize("name", ["qgnni_toricL4_seeded", "cgnni_bch_seeded", "bp_quantum_toricL4", "cgnni_ldpc_epoch18"])
def test_decode_host_pipeline_light_programs(name):
    """gd_decode_host through the node-owner (light) kernels: same bits as the device path."""
    from gnn_decode_b200.graph import TannerGraph
    g = Golden(name)
    dev = _dev()
    mod, dec = make_decoder(g)
    dec = dec.to(dev).eval()
    tg = TannerGraph(g.edge_index, g.V, g.C, dev)
    dec.bind_graph(tg)
    B = 36001
    gen = torch.Generator().manual_seed(9)
    reps = (B + g.B - 1) // g.B
    x = g.x.float().repeat(reps, 1)[:B].clone()
    x[:, :g.V] *= 0.25 + 1.5 * torch.rand(B, 1, generator=gen)            # every syndrome different
    xh = x.contiguous().pin_memory()
    ref_p, ref_h = dec.decode(xh.to(dev), return_hard=True)
    for nb in (B, 16384, B):
        prob_h = torch.zeros(nb, g.V, dtype=torch.float32).pin_memory()
        hard_h = torch.full((nb, g.V), 9, dtype=torch.uint8).pin_memory()
        dec.decode_host(xh[:nb], prob_h, hard_h)
        if nb == B:
            assert torch.equal(prob_h, ref_p.cpu()) and torch.equal(hard_h, ref_h.cpu())
        else:
            p2, h2 = dec.decode(xh[:nb].to(dev), return_hard=True)
            assert torch.equal(prob_h, p2.cpu()) and torch.equal(hard_h, h2.cpu())

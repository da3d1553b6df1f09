"""Neural BP (quantum/neural_BP.py) and decoder_v1_1 on the TMA-staged streamed kernel: codes whose edge state does not fit
shared memory (the hypergraph-product [[1600,64]] code), and any code under GD_FORCE_STREAMED.  Against the fp64 oracle, the
resident kernels and themselves; the routes that must refuse still refuse, without launching anything.

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
from conftest import Golden, logit_worst  # noqa: E402
from gnn_decode_b200 import _cabi, codes, options  # noqa: E402
from gnn_decode_b200.graph import TannerGraph  # noqa: E402
from gnn_decode_b200.sampler import sample_syndromes  # noqa: E402
from oracle import restate  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
SP_RTOL, SP_SATURATED, LOGIT_TIE = 2e-3, 30.0, 1e-3      # the sum-product bar of tests/test_random_graphs_gpu.py


def _kernels(fn):
    """Runs fn once under torch.profiler; returns the names of the library's kernels it launched."""
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


SLICE = 2048          # toric L = 5 batches this small leave the node-owner kernel out: the edge-owner kernel decodes them


def _probe_cases():
    """name -> fn() run under the profiler in the child; fn may raise GdError (its message is reported)."""
    def hgp_decoder(program):
        tg = TannerGraph.from_pcm(codes.hgp_pcm(), DEV)
        x, _ = sample_syndromes(tg, 40, [0.02, 0.05], noise=1, seed=9)
        dec = _seeded_neural_bp(6, tg.E) if program == "neural_bp" else _seeded_v1_1(6, tg.E)[0]
        dec = dec.to(DEV).eval()
        return lambda: dec.decode(x, graph=tg)

    def permuted(pcm):
        tg = _permuted(TannerGraph.from_pcm(pcm, DEV))
        dec = _seeded_neural_bp(4, tg.E).to(DEV).eval()
        x = torch.zeros((300, tg.N), device=DEV)
        x[:, tg.V:] = 1.0
        return lambda: dec.decode(x, graph=tg)

    def toric5_slices():
        tg = TannerGraph.from_pcm(codes.toric_pcm(5), DEV)
        dec = _seeded_neural_bp(8, tg.E, seed=5).to(DEV).eval()
        x, _ = sample_syndromes(tg, 3 * SLICE, [0.03, 0.08], noise=1, seed=31)
        return lambda: [dec.decode(x[i:i + SLICE], graph=tg) for i in range(0, x.size(0), SLICE)]

    return {"hgp-neural_bp": (lambda: hgp_decoder("neural_bp"), False), "hgp-v1_1": (lambda: hgp_decoder("v1_1"), False),
            "permuted-toric5-forced": (lambda: permuted(codes.toric_pcm(5)), True),
            "permuted-hgp": (lambda: permuted(codes.hgp_pcm()), False), "toric5-slices": (toric5_slices, False)}


def _probe_main():
    out = {}
    for name, (make, forced) in _probe_cases().items():
        fn = make()
        if forced:
            options.set_option("GD_FORCE_STREAMED")
        err = []

        def run():
            try:
                fn()
            except _cabi.GdError as e:
                err.append(str(e))
        out[name] = {"kernels": _kernels(run), "error": err[0] if err else None}
        if forced:
            options.unset_option("GD_FORCE_STREAMED")
    print(json.dumps(out))


@pytest.fixture(scope="module")
def launched():
    """The kernels each probe launched, read in a child process."""
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def _seeded_neural_bp(T, E, seed=0):
    """Non-trivial weights: W, W_p uniform in [0.6, 1.2], alpha = 0.25."""
    from gnn_decode_b200.quantum import neural_BP
    torch.manual_seed(seed)
    dec = neural_BP.GNNI(T, n_edges=E)
    with torch.no_grad():
        for n_, p_ in dec.named_parameters():
            p_.copy_(torch.full_like(p_, 0.25) if n_ == "alpha" else torch.rand_like(p_) * 0.6 + 0.6)
    return dec


def _seeded_v1_1(T, E, seed=0):
    """decoder_v1_1 with random edge types in [0, 32) and the same weight ranges; also returns the per-edge weights the
    oracle's neural_bp program takes (matmul(m * onehot, W) == m * W[type])."""
    from gnn_decode_b200.quantum import decoder_v1_1
    g = torch.Generator().manual_seed(seed)
    types = torch.randint(0, 32, (E,), generator=g)
    dec = decoder_v1_1.GNNI(T, edge_types=types, nb_digits=32)
    with torch.no_grad():
        for n_, p_ in dec.named_parameters():
            p_.copy_(torch.full_like(p_, 0.25) if n_ == "alpha" else torch.rand(p_.shape, generator=g, dtype=p_.dtype) * 0.6 + 0.6)
    return dec, _expand_types(dec.state_dict(), types, T)


def _expand_types(w, types, T):
    out = {}
    for l in range(T):
        out["layers.%d.W" % (2 * l)] = w["layers.%d.W" % (2 * l)][types]
        out["layers.%d.W_p" % (2 * l)] = w["layers.%d.W_p" % (2 * l)][types]
    out["W"], out["W_p"], out["alpha"] = w["W"][types], w["W_p"][types], w["alpha"]
    return {k: v.detach().cpu() for k, v in out.items()}


def _weights(dec):
    return {k: v.detach().cpu() for k, v in dec.state_dict().items()}


def _oracle(tg, x, w, T):
    return restate.decode("neural_bp", tg.edge_index, tg.V, tg.C, x.double().cpu(), w, T=T, dtype=torch.float64)["logit"]


def _assert_sum_product_bar(logit, ref, what):
    got = logit.double().cpu()
    err = (got - ref).abs()
    ok = (err <= SP_RTOL * ref.abs().clamp_min(1.0)) | (ref.abs() > SP_SATURATED)
    assert bool(ok.all()), "%s: max abs err %.3g where the oracle is not saturated" % (what, err[ref.abs() <= SP_SATURATED].max().item())


def _assert_hard_matches_oracle(hard, ref, what):
    decided = ref.abs() > LOGIT_TIE
    assert torch.equal(hard.cpu().bool()[decided], (ref < 0)[decided]), what


def _streamed(tg, dec, B):
    info = tg.launch_info(dec.gd_model(), B)
    return info["resident"] == 0


# ---- 1. golden fixtures under GD_FORCE_STREAMED ------------------------------------------------------------------------
def _golden_decoder(name):
    g = Golden(name)
    if name == "ext_neural_bp_toricL4":
        from gnn_decode_b200.quantum import neural_BP
        dec = neural_BP.GNNI(g.T, n_edges=g.E)
        dec.load_state_dict(g.weights, strict=True)
        return g, dec, g.weights
    from gnn_decode_b200.quantum import decoder_v1_1
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", name + ".npz"))
    types = torch.from_numpy(z["edge_types"])
    dec = decoder_v1_1.GNNI(g.T, edge_types=types, nb_digits=int(z["nb_digits"]))
    dec.load_state_dict(g.weights, strict=True)
    return g, dec, _expand_types(g.weights, types, g.T)


@pytest.mark.parametrize("name", ["ext_neural_bp_toricL4", "ext_v1_1_onehot_toricL4"])
def test_golden_fixture_on_the_streamed_kernel(name, gd_opt):
    g, dec, w = _golden_decoder(name)
    dec = dec.to(DEV).eval()
    tg = TannerGraph(g.edge_index, g.V, g.C, DEV)
    x5 = g.x.repeat(5, 1)                                   # ragged tiles
    ref = restate.decode("neural_bp", g.edge_index, g.V, g.C, x5, w, T=g.T, dtype=torch.float64)["logit"]
    _, _, hard_res = dec.decode(x5.to(DEV), graph=tg, return_logits=True, return_hard=True)
    gd_opt.set("GD_FORCE_STREAMED")
    assert _streamed(tg, dec, x5.size(0))
    _, logit, hard = dec.decode(x5.to(DEV), graph=tg, return_logits=True, return_hard=True)
    worst, max_err = logit_worst(logit, ref, SP_RTOL)        # the bar the resident kernel meets on this fixture
    assert worst <= 1.0, "logit mismatch: %.3g x bound (max abs err %.3g)" % (worst, max_err)
    decided = ref.abs() > LOGIT_TIE
    assert torch.equal(hard.cpu()[decided], hard_res.cpu()[decided])
    _, logit2, hard2 = dec.decode(x5.to(DEV), graph=tg, return_logits=True, return_hard=True)
    assert torch.equal(logit2, logit) and torch.equal(hard2, hard)


# ---- 2. HGP [[1600,64]] by default routing -----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def hgp():
    tg = TannerGraph.from_pcm(codes.hgp_pcm(), DEV)
    assert (tg.V, tg.C, tg.E) == (3200, 1536, 10752)
    x, _ = sample_syndromes(tg, 40, [0.02, 0.05], noise=1, seed=9)
    return tg, x


@pytest.mark.parametrize("program", ["neural_bp", "v1_1"])
def test_hgp_takes_the_streamed_kernel_and_matches_the_oracle(program, hgp, launched):
    tg, x = hgp
    T = 6
    if program == "neural_bp":
        dec = _seeded_neural_bp(T, tg.E)
        w = _weights(dec)
    else:
        dec, w = _seeded_v1_1(T, tg.E)
    dec = dec.to(DEV).eval()
    assert _streamed(tg, dec, x.size(0))
    probe = launched["hgp-" + program]
    assert probe["error"] is None and set(probe["kernels"]) == {"decode_streamed_tma_kernel"}, probe
    _, logit, hard = dec.decode(x, graph=tg, return_logits=True, return_hard=True)
    ref = _oracle(tg, x, w, T)
    _assert_sum_product_bar(logit, ref, program + " HGP")
    _assert_hard_matches_oracle(hard, ref, program + " HGP")


# ---- 3. random irregular graphs under GD_FORCE_STREAMED ----------------------------------------------------------------
def _random_pcm(rng, C, V, max_row):
    pcm = np.zeros((C, V), dtype=np.uint8)
    for c in range(C):
        d = rng.randint(1, max_row + 1)
        pcm[c, rng.choice(V, size=min(d, V), replace=False)] = 1
    pcm[:, rng.randint(0, V)] = 0            # at least one isolated variable
    if pcm.sum() == 0:
        pcm[0, 0] = 1
    return pcm


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_random_irregular_graph_matches_the_oracle(seed, gd_opt):
    rng = np.random.RandomState(100 * seed + 11)
    C, V = rng.randint(3, 14), rng.randint(6, 40)
    pcm = _random_pcm(rng, C, V, max_row=(12 if seed >= 2 else 6))     # check degrees past the unrolled 1..8
    tg = TannerGraph.from_pcm(pcm, DEV)
    B, T = 70 + 13 * seed, 5
    torch.manual_seed(seed)
    x = torch.randn(B, V + C, dtype=torch.float64) * 1.5 + 1.0
    x[:, V:] = torch.sign(torch.randn(B, C, dtype=torch.float64))
    dec = _seeded_neural_bp(T, tg.E, seed).to(DEV).eval()
    gd_opt.set("GD_FORCE_STREAMED")
    assert _streamed(tg, dec, B)
    _, logit, hard = dec.decode(x.to(DEV), graph=tg, return_logits=True, return_hard=True)
    ref = _oracle(tg, x, _weights(dec), T)
    _assert_sum_product_bar(logit, ref, "random graph seed %d (max check degree %d)" % (seed, tg.max_chk_deg))
    _assert_hard_matches_oracle(hard, ref, "random graph seed %d" % seed)


# ---- 4. batch shapes on toric L = 5 under GD_FORCE_STREAMED -----------------------------------------------------------
@pytest.fixture(scope="module")
def toric5():
    tg = TannerGraph.from_pcm(codes.toric_pcm(5), DEV)
    dec = _seeded_neural_bp(8, tg.E, seed=5).to(DEV).eval()
    return tg, dec


@pytest.mark.parametrize("B", [1, 3, 5, 129, 200])
def test_every_row_equals_decoding_it_alone(B, toric5):
    tg, dec = toric5
    x, _ = sample_syndromes(tg, B, [0.03, 0.08], noise=1, seed=20 + B)
    with options.option("GD_FORCE_STREAMED"):
        info = tg.launch_info(dec.gd_model(), B)
        assert info["resident"] == 0
        if B > 5:
            assert B % info["tile"] != 0                       # a partial last tile
        _, logit, hard = dec.decode(x, graph=tg, return_logits=True, return_hard=True)
        for i in range(B):
            _, li, hi = dec.decode(x[i:i + 1].clone(), graph=tg, return_logits=True, return_hard=True)
            assert torch.equal(li[0], logit[i]) and torch.equal(hi[0], hard[i]), "row %d of %d" % (i, B)


def test_several_tile_rounds_agree_with_the_edge_owner_kernel(toric5, launched):
    tg, dec = toric5
    B = 40000
    x, _ = sample_syndromes(tg, B, [0.03, 0.08], noise=1, seed=31)
    with options.option("GD_FORCE_STREAMED"):
        info = tg.launch_info(dec.gd_model(), B)
        assert info["resident"] == 0 and info["n_tiles"] > 2 * info["grid"]
        _, logit, hard = dec.decode(x, graph=tg, return_logits=True, return_hard=True)
    # the edge-owner kernel: slices too small for the node-owner kernel to fill the GPU
    assert set(launched["toric5-slices"]["kernels"]) == {"decode_kernel"}, launched["toric5-slices"]
    parts = [dec.decode(x[i:i + SLICE], graph=tg, return_logits=True, return_hard=True) for i in range(0, B, SLICE)]
    ref_logit = torch.cat([p[1] for p in parts])
    ref_hard = torch.cat([p[2] for p in parts])
    decided = ref_logit.abs() > LOGIT_TIE
    assert torch.equal(hard[decided], ref_hard[decided])
    print("neural BP, toric L = 5, T = 8, B = %d: max |dlogit| streamed vs edge-owner = %.3g" %
          (B, (logit - ref_logit).abs().max().item()))


# ---- 5. repeated launches ---------------------------------------------------------------------------------------------
def test_repeated_launches_are_bit_identical(gd_opt):
    tg = TannerGraph.from_pcm(codes.toric_pcm(4), DEV)
    dec = _seeded_neural_bp(7, tg.E, seed=2).to(DEV).eval()
    x, _ = sample_syndromes(tg, 1203, [0.03, 0.08], noise=1, seed=4)
    gd_opt.set("GD_FORCE_STREAMED")
    first = dec.decode(x, graph=tg, return_logits=True)[1].clone()
    outs = [dec.decode(x, graph=tg, return_logits=True)[1] for _ in range(25)]   # one stream: the slab is per graph
    torch.cuda.synchronize()
    for o in outs:
        assert torch.equal(o, first)


# ---- 6. refusals ------------------------------------------------------------------------------------------------------
def _permuted(tg, seed=0):
    perm = torch.from_numpy(np.random.RandomState(seed).permutation(tg.E))
    return TannerGraph(tg.edge_index[:, perm], tg.V, tg.C, DEV)


@pytest.mark.parametrize("code", ["toric5-forced", "hgp"])
def test_permuted_edge_order_is_refused_without_a_launch(code, gd_opt, launched):
    probe = launched["permuted-" + code]
    assert probe["kernels"] == [] and probe["error"] and "canonical" in probe["error"], probe
    pcm = codes.toric_pcm(5) if code.startswith("toric") else codes.hgp_pcm()
    tg = _permuted(TannerGraph.from_pcm(pcm, DEV))
    dec = _seeded_neural_bp(4, tg.E).to(DEV).eval()
    x = torch.zeros((300, tg.N), device=DEV)
    x[:, tg.V:] = 1.0
    if code.endswith("forced"):
        gd_opt.set("GD_FORCE_STREAMED")
    with pytest.raises(_cabi.GdError, match="canonical"):
        dec.decode(x, graph=tg)


def test_hidden_not_E_is_still_invalid_on_the_streamed_route(gd_opt):
    lib = _cabi.lib()
    for pcm, forced in ((codes.hgp_pcm(), False), (codes.toric_pcm(5), True)):
        tg = TannerGraph.from_pcm(pcm, DEV)
        x = torch.zeros((8, tg.N), device=DEV)
        prob = torch.empty((8, tg.V), device=DEV)
        model = _cabi.GdModel(_cabi.PROG_NEURAL_BP, int(tg.E) + 1, 5, 0)
        w = torch.zeros(lib.gd_weights_size(ct.byref(model)), device=DEV)
        if forced:
            gd_opt.set("GD_FORCE_STREAMED")
        rc = lib.gd_decode_fwd(tg.handle, ct.byref(model), ct.c_void_p(w.data_ptr()), ct.c_void_p(x.data_ptr()),
                               ct.c_void_p(prob.data_ptr()), None, None, 8, None)
        assert rc == _cabi.GD_ERR_INVALID
        info = _cabi.GdLaunchInfo()
        assert lib.gd_decode_launch_info(tg.handle, ct.byref(model), 8, ct.byref(info)) == _cabi.GD_ERR_INVALID


def test_packed_call_is_still_refused_on_the_streamed_route(hgp):
    from gnn_decode_b200 import packing
    from gnn_decode_b200.quantum import decoder_v2_4
    tg, x = hgp
    prior, bits = packing.pack_x(x, tg.V)
    for dec in (_seeded_neural_bp(4, tg.E), decoder_v2_4.GNNI(4)):
        dec = dec.to(DEV).eval()
        with pytest.raises(_cabi.GdError):
            dec.decode_packed(prior, bits, graph=tg)


# ---- 7. host pipeline -------------------------------------------------------------------------------------------------
def test_decode_host_equals_the_device_path(hgp):
    tg, x = hgp
    dec = _seeded_neural_bp(6, tg.E, seed=3).to(DEV).eval()
    prob, hard = dec.decode(x, graph=tg, return_hard=True)
    x_host = x.cpu().pin_memory()
    prob_h = torch.empty((x.size(0), tg.V), dtype=torch.float32).pin_memory()
    hard_h = torch.empty((x.size(0), tg.V), dtype=torch.uint8).pin_memory()
    dec.decode_host(x_host, prob_out=prob_h, hard_out=hard_h, graph=tg)
    assert torch.equal(prob_h, prob.cpu()) and torch.equal(hard_h, hard.cpu())


if __name__ == "__main__":
    _probe_main()

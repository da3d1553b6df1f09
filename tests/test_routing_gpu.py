"""Which kernel family serves a call (csrc/gd_decode.cu: route_decode; DESIGN.md §4): the kernels one call launches, the launch
geometry gd_decode_launch_info reports for them, the refusals, and that the caller's current device survives a refused call."""
import contextlib
import ctypes as ct
import json
import os
import re
import tempfile

import pytest
import torch

from conftest import Golden
from gnn_decode_b200 import _cabi, codes, options, packing
from gnn_decode_b200.graph import TannerGraph
from gnn_decode_b200.sampler import sample_syndromes

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
P10 = [0.01, 0.02, 0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.09, 0.1]
FAMILY = {
    "lean_prep_kernel": "lean", "lean_tables_kernel": "lean", "lean_decode_kernel": "lean", "lean_unpack_kernel": "lean",
    "lean_bwd_kernel": "lean", "lean_contract_kernel": "lean",
    "decode_kernel": "edge", "decode_bwd_kernel": "edge", "reduce_partials_kernel": "edge",
    "decode_light_kernel": "light", "decode_light_ext_kernel": "light", "cgnni_bwd_light_kernel": "light",
    "cgnni_contract_kernel": "light",
    "decode_streamed_tma_kernel": "streamed_tma", "decode_streamed_kernel": "streamed",
}


def _kernels(fn):
    """Runs fn once under torch.profiler; returns the decode-family kernels it launched as (name, grid, block), in order."""
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
        if ev.get("cat") != "kernel" or "gd::" not in ev.get("name", ""):
            continue
        m = re.search(r"(\w+)\s*(?:<|\()", ev["name"].split("gd::", 1)[1])
        if m and m.group(1) in FAMILY:
            out.append((m.group(1), tuple(ev["args"]["grid"]), tuple(ev["args"]["block"])))
    return out


def _names(ks):
    return {k[0] for k in ks}


def _check_geometry(ks, main, info):
    launches = [k for k in ks if k[0] == main]
    assert launches, (main, ks)
    for _, grid, block in launches:
        assert grid == (info["grid"], 1, 1) and block == (info["threads"], 1, 1), (main, grid, block, info)


def _v2_4(pcm, T=15):
    from gnn_decode_b200.quantum import decoder_v2_4
    g = TannerGraph.from_pcm(pcm, DEV)
    dec = decoder_v2_4.GNNI(T)
    dec.load_state_dict(Golden("v2_4_toricL5_epoch3").weights)
    return g, dec.to(DEV).eval().bind_graph(g)


def _qgnni(pcm, T=10):
    from gnn_decode_b200.quantum import QGNNI
    g = TannerGraph.from_pcm(pcm, DEV)
    torch.manual_seed(0)
    return g, QGNNI.GNNI(T).to(DEV).eval().bind_graph(g)


V2_4_CASES = [
    (None, {"lean_prep_kernel", "lean_tables_kernel", "lean_decode_kernel", "decode_kernel"}, "lean_decode_kernel"),
    ("GD_NO_LEAN", {"decode_kernel"}, "decode_kernel"),
    ("GD_FORCE_STREAMED", {"decode_streamed_tma_kernel"}, "decode_streamed_tma_kernel"),
]


@pytest.mark.parametrize("opt,expected,main", V2_4_CASES, ids=["default", "no_lean", "force_streamed"])
def test_v2_4_rotated_d5(opt, expected, main):
    g, dec = _v2_4(codes.rotated_surface_pcm(5))
    B = 32768                          # enough syndromes for the TMA-staged streamed kernel (>= 128 per SM) under GD_FORCE_STREAMED
    x, _ = sample_syndromes(g, B, P10, noise=1, seed=3)
    with options.option(opt) if opt else contextlib.nullcontext():
        info = g.launch_info(dec.gd_model(), B)
        ks = _kernels(lambda: dec.decode(x))
    assert _names(ks) == expected, ks
    _check_geometry(ks, main, info)


def test_v2_4_toric_L11_takes_the_table_kernel_per_component():
    g, dec = _v2_4(codes.toric_pcm(11))
    B = 9000
    x, _ = sample_syndromes(g, B, P10[:5], noise=0, seed=5)
    info = g.launch_info(dec.gd_model(), B)
    ks = _kernels(lambda: dec.decode(x))
    assert [k[0] for k in ks].count("lean_decode_kernel") == 2, ks
    assert {FAMILY[k[0]] for k in ks} == {"lean", "edge"}, ks       # (edge: the deferred pass)
    _check_geometry(ks, "lean_decode_kernel", info)


@pytest.mark.parametrize("pcm,B,expected", [
    ("toric5", 65536, "decode_light_kernel"),
    ("toric5", 1024, "decode_kernel"),
    ("hgp", 256, "decode_streamed_tma_kernel"),
])
def test_qgnni(pcm, B, expected):
    g, dec = _qgnni(codes.toric_pcm(5) if pcm == "toric5" else codes.hgp_pcm())
    x, _ = sample_syndromes(g, B, [0.02, 0.05], noise=1, seed=9)
    info = g.launch_info(dec.gd_model(), B)
    ks = _kernels(lambda: dec.decode(x))
    assert _names(ks) == {expected}, ks
    _check_geometry(ks, expected, info)


def _train_step(dec, g, x):
    prob = dec.decode(x, graph=g)
    prob.sum().backward()


def test_v2_4_training_step_runs_the_table_family_both_ways():
    g, dec = _v2_4(codes.rotated_surface_pcm(5))
    dec.train()
    x, _ = sample_syndromes(g, 4096, P10, noise=1, seed=7)
    ks = _kernels(lambda: _train_step(dec, g, x))
    assert _names(ks) == {"lean_prep_kernel", "lean_tables_kernel", "lean_decode_kernel", "decode_kernel",
                          "lean_bwd_kernel", "lean_contract_kernel", "decode_bwd_kernel", "reduce_partials_kernel"}, ks


def test_cgnni_training_step_runs_the_node_owner_family_both_ways():
    from gnn_decode_b200.classical import CGNNI
    case = Golden("cgnni_bch_seeded")
    g = TannerGraph(case.edge_index, case.V, case.C, DEV)
    dec = CGNNI.GNNI(case.T)
    dec.load_state_dict(case.weights)
    dec = dec.to(DEV).train()
    x = case.x.to(DEV, torch.float32).repeat(8, 1)
    ks = _kernels(lambda: _train_step(dec, g, x))
    assert _names(ks) == {"decode_light_kernel", "cgnni_bwd_light_kernel", "cgnni_contract_kernel"}, ks


def test_packed_call_refuses_the_streamed_route():
    g, dec = _v2_4(codes.rotated_surface_pcm(5))
    x, _ = sample_syndromes(g, 3000, P10, noise=1, seed=13)
    prior, bits = packing.pack_x(x, g.V)
    with options.option("GD_FORCE_STREAMED"):
        with pytest.raises(_cabi.GdError):
            dec.decode_packed(prior, bits)
    hb = dec.decode_packed(prior, bits)
    _, hard = dec.decode(x, return_hard=True)
    assert torch.equal(packing.unpack_bits(hb, g.V), hard)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_refused_calls_leave_the_callers_device_current():
    """Argument errors found after the switch to the graph's device (no kernel is launched) give the caller's device back."""
    dev1 = torch.device("cuda", 1)
    torch.cuda.set_device(0)
    try:
        lib = _cabi.lib()
        # NEURAL_BP with hidden != E
        g = TannerGraph.from_pcm(codes.toric_pcm(5), dev1)
        x = torch.zeros((8, g.N), device=dev1)
        prob = torch.empty((8, g.V), device=dev1)
        model = _cabi.GdModel(_cabi.PROG_NEURAL_BP, int(g.E) + 1, 5, 0)
        w = torch.zeros(lib.gd_weights_size(ct.byref(model)), device=dev1)
        rc = lib.gd_decode_fwd(g.handle, ct.byref(model), ct.c_void_p(w.data_ptr()), ct.c_void_p(x.data_ptr()),
                               ct.c_void_p(prob.data_ptr()), None, None, 8, None)
        assert rc == _cabi.GD_ERR_INVALID
        assert torch.cuda.current_device() == 0
        # V2_4_1 on a graph whose checks do not all have 4 edges
        g = TannerGraph.from_pcm(codes.rotated_surface_pcm(5), dev1)
        x = torch.zeros((8, g.N), device=dev1)
        prob = torch.empty((8, g.V), device=dev1)
        model = _cabi.GdModel(_cabi.PROG_V2_4_1, 16, 5, 0)
        w = torch.zeros(lib.gd_weights_size(ct.byref(model)), device=dev1)
        rc = lib.gd_decode_fwd(g.handle, ct.byref(model), ct.c_void_p(w.data_ptr()), ct.c_void_p(x.data_ptr()),
                               ct.c_void_p(prob.data_ptr()), None, None, 8, None)
        assert rc == _cabi.GD_ERR_INVALID
        assert torch.cuda.current_device() == 0
    finally:
        torch.cuda.set_device(0)

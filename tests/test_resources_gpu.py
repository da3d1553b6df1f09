"""Device resources of graphs and pipelines are released when they are destroyed: graphs whose lazily made state has been
filled (the table kernel's cache and memory pool, the streamed kernels' slab, gd_decode_host's internal pipeline, the training
path's table sets) and standalone pipelines are created, used and destroyed over and over, and the device's free memory comes
back.  A graph made after the cycles still decodes as the oracle does."""
import gc
import math

import pytest
import torch

from conftest import Golden, logit_worst, make_decoder
from gnn_decode_b200 import codes, packing
from gnn_decode_b200.graph import TannerGraph
from gnn_decode_b200.pipeline import DecodePipeline
from gnn_decode_b200.quantum import decoder_v2_4
from gnn_decode_b200.sampler import sample_syndromes
from oracle import restate

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
P10 = [0.01, 0.02, 0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.09, 0.1]
# Free device memory may move by this much while a test runs for reasons of its own: other work on a shared GPU.  Each test
# repeats its cycle often enough that one leaked cycle per iteration would cost at least 8 times this.
MARGIN = 64 << 20
PCM = codes.rotated_surface_pcm(5)


def _decoder(T=15):
    dec = decoder_v2_4.GNNI(T)
    dec.load_state_dict(Golden("v2_4_toricL5_epoch3").weights)
    return dec.to(DEV).eval()


def _free():
    gc.collect()
    torch.cuda.synchronize()                 # nothing is destroyed with work still queued on it
    torch.cuda.empty_cache()                 # torch's cached blocks would hide what the library gives back
    return torch.cuda.mem_get_info(DEV)[0]


def _cycle(run):
    """run() makes a graph, uses it and returns the objects that own library state; they are destroyed here, after a
    synchronisation.  Returns the device memory their destruction gave back."""
    held = run()
    finalizers = [o._finalizer for o in held]
    before = _free()
    del held[:]
    after = _free()
    assert not any(f.alive for f in finalizers)
    return after - before


def _no_leak(run):
    freed = _cycle(run)                      # also loads the modules and fills torch's cache
    assert freed >= MARGIN // 16, "the cycle held only %.1f MB of its own" % (freed / 2**20)
    cycles = min(128, max(4, math.ceil(8 * MARGIN / freed)))
    base = _free()
    for _ in range(cycles):
        _cycle(run)
    lost = base - _free()
    assert lost <= MARGIN, "%d cycles that each held %.1f MB lost %.1f MB" % (cycles, freed / 2**20, lost / 2**20)


def _golden_on_a_fresh_graph():
    """(decoder, new graph, x, prob) for the golden toric L = 4 case, decoded on the device and checked against the oracle."""
    g = Golden("v2_4_toricL4_epoch1")
    _, dec = make_decoder(g)
    dec = dec.to(DEV).eval()
    tg = TannerGraph(g.edge_index, g.V, g.C, DEV)
    x = g.x.float().to(DEV)
    prob, logit = dec.decode(x, graph=tg, return_logits=True)
    ref = restate.decode(g.program, g.edge_index, g.V, g.C, g.x, g.weights, T=g.T, dtype=torch.float64)
    worst, err = logit_worst(logit, ref["logit"])
    assert worst <= 1.0, "logits differ from the oracle: %.3g x bound (max abs %.3g)" % (worst, err)
    return dec, tg, x, prob


def test_graph_after_table_kernel_inference():
    """The table kernel's cache: metadata, table sets, and the memory pool whose workspace holds the unpacked inputs of a
    large packed call."""
    dec = _decoder()
    g0 = TannerGraph.from_pcm(PCM, DEV)
    x, _ = sample_syndromes(g0, 4096, P10, noise=1, seed=1)
    prior, synd = packing.pack_x(sample_syndromes(g0, 1 << 20, P10, noise=1, seed=2)[0], g0.V)
    ref = dec.decode(x, graph=g0)
    del g0

    def run():
        g = TannerGraph.from_pcm(PCM, DEV)
        assert torch.equal(dec.decode(x, graph=g), ref)
        dec.decode_packed(prior, synd, graph=g)
        return [g]

    _no_leak(run)
    _golden_on_a_fresh_graph()


def test_graph_after_streamed_decode(gd_opt):
    """The per-graph edge-state slab of the streamed kernels."""
    dec = _decoder()
    gd_opt.set("GD_FORCE_STREAMED")
    g0 = TannerGraph.from_pcm(PCM, DEV)
    x, _ = sample_syndromes(g0, 32768, P10, noise=1, seed=3)
    assert g0.launch_info(dec.gd_model(), x.size(0))["resident"] == 0
    ref = dec.decode(x, graph=g0)
    del g0

    def run():
        g = TannerGraph.from_pcm(PCM, DEV)
        assert torch.equal(dec.decode(x, graph=g), ref)
        return [g]

    _no_leak(run)
    _golden_on_a_fresh_graph()


def test_graph_after_decode_host():
    """gd_decode_host's internal pipeline: streams, events and the buffers of its slots."""
    dec = _decoder()
    g0 = TannerGraph.from_pcm(PCM, DEV)
    x, _ = sample_syndromes(g0, 1 << 19, P10, noise=1, seed=4)
    ref = dec.decode(x, graph=g0).cpu()
    xh = x.cpu().pin_memory()
    del g0, x

    def run():
        g = TannerGraph.from_pcm(PCM, DEV)
        assert torch.equal(dec.decode_host(xh, graph=g), ref)
        return [g]

    _no_leak(run)
    dec, tg, x, prob = _golden_on_a_fresh_graph()
    assert torch.equal(dec.decode_host(x.cpu(), graph=tg), prob.cpu())


def test_graph_after_training_step():
    """decoder_v2_4's training forward (with stash) and backward: the table sets and metadata of the training path."""
    dec = _decoder().train()
    g0 = TannerGraph.from_pcm(PCM, DEV)
    x, _ = sample_syndromes(g0, 16384, P10, noise=1, seed=5)
    del g0

    def run():
        g = TannerGraph.from_pcm(PCM, DEV)
        dec.zero_grad()
        dec.decode(x, graph=g).sum().backward()
        assert all(torch.isfinite(p.grad).all() for p in dec.parameters())
        return [g]

    _no_leak(run)
    _golden_on_a_fresh_graph()


def test_standalone_pipeline():
    """gd_pipeline_create / gd_pipeline_destroy with batches submitted in both input forms."""
    dec = _decoder()
    g0 = TannerGraph.from_pcm(PCM, DEV)
    x, _ = sample_syndromes(g0, 1 << 17, P10, noise=1, seed=6)
    ref_p, ref_h = (t.cpu() for t in dec.decode(x, graph=g0, return_hard=True))
    prior, synd = (t.cpu().pin_memory() for t in packing.pack_x(x, g0.V))
    xh = x.cpu().pin_memory()
    prob_out = torch.empty(ref_p.shape, dtype=torch.float32).pin_memory()
    bits_out = torch.empty((x.size(0), (g0.V + 31) // 32), dtype=torch.int32).pin_memory()
    del g0, x

    def run():
        g = TannerGraph.from_pcm(PCM, DEV)
        pipe = DecodePipeline(dec, g, max_B=1 << 15, depth=3)
        prob_out.zero_()
        bits_out.zero_()
        for lo in range(0, xh.size(0), 1 << 15):
            hi = lo + (1 << 15)
            pipe.submit(xh[lo:hi], prob_out=prob_out[lo:hi])
        pipe.drain()
        assert torch.equal(prob_out, ref_p)
        for lo in range(0, xh.size(0), 1 << 15):
            hi = lo + (1 << 15)
            pipe.submit_packed(prior[lo:hi], synd[lo:hi], hard_bits_out=bits_out[lo:hi])
        pipe.drain()
        assert torch.equal(packing.unpack_bits(bits_out, ref_h.size(1)), ref_h)
        return [pipe, g]

    _no_leak(run)
    dec, tg, x, prob = _golden_on_a_fresh_graph()
    pipe = DecodePipeline(dec, tg, max_B=x.size(0), depth=2)
    out = torch.empty(prob.shape, dtype=torch.float32).pin_memory()
    pipe.wait(pipe.submit(x.cpu().pin_memory(), prob_out=out))
    assert torch.equal(out, prob.cpu())

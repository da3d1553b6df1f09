"""Tiny run of every kernel family, meant to be executed under compute-sanitizer (memcheck / racecheck / synccheck):
    compute-sanitizer --tool racecheck python scripts/sanitize_smoke.py
Sizes are small; each launch still covers ragged tiles and every phase.  300 syndromes cannot fill the GPU, so the light
programs take the edge-owner kernel unless GD_FORCE_LIGHT is set, and decoder_v2_4 (below 128 syndromes per SM) takes the
register-batched streamed kernel under GD_FORCE_STREAMED."""
import os, sys, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gnn_decode_b200 import codes, options
from gnn_decode_b200.evaluate import count_failures
from gnn_decode_b200.graph import TannerGraph
from gnn_decode_b200.quantum import decoder_v2_4, QGNNI, BP, neural_BP, QGNNNI_ca
from gnn_decode_b200.classical import CGNNI
from gnn_decode_b200.sampler import sample_syndromes
from gnn_decode_b200.train import train_step_grads

dev = torch.device("cuda", 0)
which = sys.argv[1:] or ["resident", "light", "streamed", "train", "misc"]
Hz, Hx = codes.rotated_surface_checks(3)
pcm = codes.css_pcm(Hz, Hx)
g = TannerGraph.from_pcm(pcm, dev)
x, err = sample_syndromes(g, 300, [0.05, 0.1], noise=1, seed=1)
gt = TannerGraph.from_pcm(codes.toric_pcm(3), dev)
xt, _ = sample_syndromes(gt, 300, [0.05], noise=0, seed=2)
torch.manual_seed(0)
progs = [decoder_v2_4.GNNI(3), QGNNI.GNNI(3), BP.GNNI(3), neural_BP.GNNI(3, n_edges=int(pcm.sum())), QGNNNI_ca.GNNI(3)]
if "resident" in which:
    for d in progs:
        d.to(dev).eval().decode(x, graph=g, return_hard=True)
    CGNNI.GNNI(3).to(dev).eval().decode(xt, graph=gt)
    print("resident ok", flush=True)
if "light" in which:
    with options.option("GD_FORCE_LIGHT"):
        for d in (QGNNI.GNNI(3), BP.GNNI(3)):
            d.to(dev).eval().decode(x, graph=g, return_logits=True)
        CGNNI.GNNI(3).to(dev).eval().decode(xt, graph=gt)
    print("light ok", flush=True)
if "streamed" in which:
    with options.option("GD_FORCE_STREAMED"):
        for d in (QGNNI.GNNI(3), BP.GNNI(3)):
            d.to(dev).eval().decode(x, graph=g, return_hard=True)
        CGNNI.GNNI(3).to(dev).eval().decode(xt, graph=gt)
        print("streamed (TMA) ok", flush=True)
        decoder_v2_4.GNNI(2).to(dev).eval().decode(x, graph=g, return_hard=True)
        print("streamed (register-batched) ok", flush=True)
if "train" in which:
    dec = decoder_v2_4.GNNI(3).to(dev).train()
    train_step_grads(dec, g, x, err, codes.css_logicals(Hz, Hx))
    print("train ok", flush=True)
if "misc" in which:
    hard = decoder_v2_4.GNNI(2).to(dev).eval().decode(x, graph=g, return_hard=True)[1]
    print("failures", count_failures(g, err, hard, codes.css_logicals(Hz, Hx)).tolist(), flush=True)
    conv = decoder_v2_4.GraphConv("target_to_source").to(dev)
    ei = torch.from_numpy(codes.edge_index_of(pcm)).to(dev)
    ei2 = torch.stack([ei[0], ei[1] + g.V])
    conv.bind_code(g.V, g.C)
    conv(torch.randn(ei.size(1), 1, device=dev, dtype=torch.float64), ei2, x[0].double().reshape(-1, 1))
    print("misc ok", flush=True)
torch.cuda.synchronize()
print("all done")

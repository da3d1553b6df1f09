"""Developer check: decoder_v2_4 on the hypergraph-product [[1600,64]] code (streamed kernels), B syndromes: throughput of the
TMA-staged kernel with / without its cubic tables, and of the register-batched kernel (which decoder_v2_4 takes below 128
syndromes per SM); agreement with the fp64 oracle on a subset."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gnn_decode_b200 import codes, options  # noqa: E402
from gnn_decode_b200.graph import TannerGraph  # noqa: E402
from gnn_decode_b200.quantum import decoder_v2_4  # noqa: E402
from gnn_decode_b200.sampler import sample_syndromes  # noqa: E402
from oracle import restate  # noqa: E402

DEV = torch.device("cuda", 0)


def timed(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 32768
    pcm = codes.hgp_pcm()
    g = TannerGraph.from_pcm(pcm, DEV)
    z = np.load(os.path.join(ROOT, "tests", "golden", "v2_4_toricL5_epoch3.npz"))
    w = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
    dec = decoder_v2_4.GNNI(15)
    dec.load_state_dict(w)
    dec = dec.to(DEV).eval().bind_graph(g)
    x, _ = sample_syndromes(g, B, [0.01, 0.02, 0.03, 0.04, 0.05], noise=1, seed=3)
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    ref = restate.decode("v2_4", ei, g.V, g.C, x[:8].double().cpu(), w, T=15)["logit"]
    small = min(B, 64 * torch.cuda.get_device_properties(DEV).multi_processor_count)
    for tag, opts, nb in (("TMA kernel, tables", [], B), ("TMA kernel, direct", ["GD_NO_CTAB"], B),
                          ("register-batched kernel", [], small)):
        for o in opts:
            options.set_option(o, 1)
        xb = x[:nb]
        print("launch:", g.launch_info(dec.gd_model(), nb))
        _, logit = dec.decode(xb, return_logits=True)
        err = (logit[:8].double().cpu() - ref).abs()
        ms = timed(lambda: dec.decode(xb))
        print("%-26s B = %6d %8.2f ms  %8.1f k syndromes/s   worst |d| / (1e-4 max(|ref|, 1)) = %.3f" %
              (tag, nb, ms, nb / ms, (err / (1e-4 * ref.abs().clamp_min(1.0))).max().item()))
        for o in opts:
            options.unset_option(o)


if __name__ == "__main__":
    main()

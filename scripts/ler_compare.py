"""Hard-decision agreement and logical error rate of the tabulated (default) vs direct (GD_NO_CTAB=1 GD_NO_VSKIP=1)
evaluation paths of the decoder_v2_4 kernel on 2^20 sampled syndromes (rotated d=5, depolarizing)."""
import os, sys, subprocess, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if len(sys.argv) > 1:
    from gnn_decode_b200 import codes
    from gnn_decode_b200.evaluate import count_failures
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.quantum import decoder_v2_4
    from gnn_decode_b200.sampler import sample_syndromes
    dev = torch.device("cuda", 0)
    Hz, Hx = codes.rotated_surface_checks(5)
    g = TannerGraph.from_pcm(codes.css_pcm(Hz, Hx), dev)
    z = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "v2_4_toricL5_epoch3.npz"))
    dec = decoder_v2_4.GNNI(15)
    dec.load_state_dict({k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")})
    dec = dec.to(dev).eval()
    B = 1 << 20
    x, err = sample_syndromes(g, B, [0.01, 0.03, 0.05, 0.08], noise=1, seed=2024)
    prob, logit, hard = dec.decode(x, graph=g, return_logits=True, return_hard=True)
    cnt = count_failures(g, err, hard, codes.css_logicals(Hz, Hx)).tolist()
    torch.save({"hard": hard.cpu(), "logit": logit.cpu(), "cnt": cnt}, sys.argv[1])
else:
    env_b = dict(os.environ, GD_NO_CTAB="1", GD_NO_VSKIP="1")
    subprocess.run([sys.executable, __file__, "/tmp/ler_a.pt"], check=True)
    subprocess.run([sys.executable, __file__, "/tmp/ler_b.pt"], check=True, env=env_b)
    a, b = torch.load("/tmp/ler_a.pt"), torch.load("/tmp/ler_b.pt")
    n = a["hard"].numel()
    diff = int((a["hard"] != b["hard"]).sum())
    dl = (a["logit"] - b["logit"]).abs()
    rel = (dl / (1e-4 * a["logit"].abs() + 1e-4 * (1 + a["logit"].pow(2).mean().sqrt()))).max().item()
    print("2^20 syndromes x 50 bits: differing hard decisions %d of %d; max |dlogit| %.3g (%.3f of the 1e-4 parity bound)" % (diff, n, dl.max().item(), rel))
    print("failure counts [syndrome, logical, total]: tabulated %s   direct %s   (B = %d)" % (a["cnt"], b["cnt"], a["hard"].size(0)))

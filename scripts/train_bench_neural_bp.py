"""Neural BP (quantum/neural_BP.py) training-step timing: the TMA-staged streamed forward with stash (gd_decode_fwd_train) and
the per-edge-weight backward (gd_decode_bwd: nbp_bwd_kernel + its fixed-order reduction), on the hypergraph-product
[[1600,64]] code (V = 3200, C = 1536, E = 10752) at T = 15, B = 1024 and 4096, and on toric L = 5 at B = 65 536.  Weights
uniform in [0.6, 1.2], alpha = 0.25, depolarizing syndromes (gd_sample noise 1).  Per workload, CUDA-event times with L2
flushed before every timed call (a 512 MB write between calls, outside the events):
  fwd_stash_ms  gd_decode_fwd_train,
  bwd_ms        gd_decode_bwd,
  step_ms       the drop-in step: decoder.decode(x) in train mode, a weighted sum of prob, loss.backward();
syndromes/s of the step, and each kernel's algorithmic HBM bytes over the device-to-device copy peak measured in the same run:
  forward  per syndrome T E (20 B of m / t traffic + 4 B of stash) + E 4 B read-out + N 4 B input + V 8 B prob / logit;
  backward per syndrome T E 64 B (stash -> m rows 8, L recompute 12, dS / dL 12, du / dq / g 32) + E 16 B read-out + N 4 + V 8.
Also the CPU fp64 oracle step (restate + autograd) at a small B on HGP, for scale.  One JSON line per workload, with the GPU's
name and power limit read in the same run.
  python scripts/train_bench_neural_bp.py [--reps 5] [--out FILE]"""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gnn_decode_b200 import _cabi, codes  # noqa: E402
from gnn_decode_b200.graph import TannerGraph  # noqa: E402
from gnn_decode_b200.quantum import neural_BP  # noqa: E402
from gnn_decode_b200.sampler import sample_syndromes  # noqa: E402
from oracle import restate  # noqa: E402

T = 15
P = [0.01, 0.03, 0.05, 0.08]
WORKLOADS = [("hgp_1600_64", 1024), ("hgp_1600_64", 4096), ("toric_L5", 65536)]


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001 -- no nvidia-smi: say so in the record
        power = None
    return name, power


def pcm_of(code):
    return codes.hgp_pcm() if code == "hgp_1600_64" else codes.toric_pcm(5)


def decoder(E):
    g = torch.Generator().manual_seed(0)
    dec = neural_BP.GNNI(T, n_edges=E)
    with torch.no_grad():
        for n_, p_ in dec.named_parameters():
            p_.copy_(torch.full_like(p_, 0.25) if n_ == "alpha" else torch.rand(p_.shape, generator=g, dtype=p_.dtype) * 0.6 + 0.6)
    return dec


class Flushed(object):
    """Per-call CUDA-event times with L2 overwritten before every call (outside the events)."""

    def __init__(self, dev):
        self.buf = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def time(self, fn, reps):
        fn()                                                  # warm-up of this shape
        ms = []
        for _ in range(reps):
            self.buf.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return sorted(ms)[len(ms) // 2]


def copy_peak(dev):
    """Device-to-device copy bandwidth (read + write bytes per second), 1 GiB each way."""
    a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2.0 * a.numel() * 10 / (e0.elapsed_time(e1) * 1e-3)


def bench_gpu(code, B, reps, dev, fl, peak):
    g = TannerGraph.from_pcm(pcm_of(code), dev)
    dec = decoder(g.E).to(dev).train()
    x, _ = sample_syndromes(g, B, P, noise=1, seed=1)
    lib = _cabi.lib()
    model = dec.gd_model()
    w = torch.cat([q.detach().reshape(-1).float() for q in dec._gd_params()]).to(dev)
    prob = torch.empty((B, g.V), device=dev)
    logit = torch.empty((B, g.V), device=dev)
    stash = torch.empty(lib.gd_stash_floats(g.handle, ct.byref(model), B), device=dev)
    ws = torch.empty(lib.gd_bwd_workspace_floats(g.handle, ct.byref(model), B), device=dev)
    gw = torch.empty(w.numel(), device=dev)
    dlogit = torch.randn((B, g.V), device=dev) * 0.01
    c = torch.randn((B, g.V), device=dev)
    st = ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: ct.c_void_p(t.data_ptr())   # noqa: E731

    def fwd():
        _cabi.check(lib.gd_decode_fwd_train(g.handle, ct.byref(model), p(w), p(x), p(prob), p(logit), p(stash), B, st))

    def bwd():
        _cabi.check(lib.gd_decode_bwd(g.handle, ct.byref(model), p(w), p(x), p(stash), p(dlogit), p(gw), p(ws), 0, B, st))

    def step():
        dec.zero_grad(set_to_none=True)
        (dec.decode(x, graph=g) * c).sum().backward()

    fwd_ms, bwd_ms, step_ms = fl.time(fwd, reps), fl.time(bwd, reps), fl.time(step, reps)
    E, V, N = g.E, g.V, g.N
    fwd_bytes = B * (T * E * 24 + E * 4 + N * 4 + V * 8)
    bwd_bytes = B * (T * E * 64 + E * 16 + N * 4 + V * 8)
    return {"fwd_stash_ms": round(fwd_ms, 3), "bwd_ms": round(bwd_ms, 3), "step_ms": round(step_ms, 3),
            "syndromes_per_s": round(B * 1e3 / step_ms, 1),
            "fwd_hbm_bytes": fwd_bytes, "bwd_hbm_bytes": bwd_bytes, "copy_peak_bytes_per_s": round(peak),
            "fwd_share_of_copy_peak": round(fwd_bytes / (fwd_ms * 1e-3) / peak, 4),
            "bwd_share_of_copy_peak": round(bwd_bytes / (bwd_ms * 1e-3) / peak, 4),
            "stash_bytes": stash.numel() * 4, "workspace_bytes": ws.numel() * 4}


def bench_cpu(B, reps):
    pcm = pcm_of("hgp_1600_64")
    dev = torch.device("cuda", 0)
    g = TannerGraph.from_pcm(pcm, dev)
    x, _ = sample_syndromes(g, B, P, noise=1, seed=1)
    x = x.cpu().double()
    w = {k: v.detach() for k, v in decoder(g.E).state_dict().items()}
    c = torch.randn((B, g.V), dtype=torch.float64)
    t0 = time.perf_counter()
    for _ in range(reps):
        restate.decode_grad("neural_bp", g.edge_index.cpu(), g.V, g.C, x, w, lambda prob: (prob * c).sum(), T=T,
                            dtype=torch.float64)
    ms = (time.perf_counter() - t0) * 1e3 / reps
    return {"step_ms": round(ms, 1), "syndromes_per_s": round(B * 1e3 / ms, 3), "cpu_threads": torch.get_num_threads()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cpu-B", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("train_bench_neural_bp.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    name, power = gpu_info()
    peak = copy_peak(dev)
    fl = Flushed(dev)
    lines = []
    for code, B in WORKLOADS:
        r = {"code": code, "arm": "gpu", "B": B, "T": T}
        r.update(bench_gpu(code, B, a.reps, dev, fl, peak))
        r.update({"gpu": name, "power_limit_w": power})
        lines.append(r)
        print(json.dumps(r), flush=True)
        torch.cuda.empty_cache()
    if a.cpu_B > 0:
        r = {"code": "hgp_1600_64", "arm": "cpu_oracle_fp64_autograd", "B": a.cpu_B, "T": T}
        r.update(bench_cpu(a.cpu_B, 1))
        lines.append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()

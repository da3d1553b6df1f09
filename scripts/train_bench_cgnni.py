"""CGNNI training-step timing: BCH(63,45) and the 4x8 LDPC of classical/CGNNI.py, T = 25, the shipped epoch-18 weights, AWGN
inputs (gd_sample noise 2, SNR 1..6 dB).  Per code and batch size, CUDA-event times of
  fwd_stash_ms  gd_decode_fwd_train (node-owner forward writing the m stash),
  bwd_ms        gd_decode_bwd (node-owner backward + bin contraction),
  step_ms       the public path: decoder(datas) in train() -> F.binary_cross_entropy -> backward -> torch.optim.Adam.step,
and a CPU arm: the oracle's eager fp32 restatement of the forward + autograd (restate.decode_grad) at B = 1024.
One JSON line per (code, arm, B), with the GPU's name and power limit read in the same run.
  python scripts/train_bench_cgnni.py [--sizes 1024,16384,65536] [--out FILE] [--profile DIR]
--profile DIR: instead, a torch.profiler kernel table of three BCH steps at the largest size (a separate run: tracing slows
the host)."""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gnn_decode_b200 import _cabi, codes  # noqa: E402
from gnn_decode_b200.classical import CGNNI  # noqa: E402
from gnn_decode_b200.graph import TannerGraph  # noqa: E402
from gnn_decode_b200.sampler import sample_syndromes  # noqa: E402
from oracle import restate  # noqa: E402

T = 25
SNR = [1.0, 2.0, 3.0, 4.0, 5.0, 6.0]
CODES = {"bch": (codes.bch_63_45_pcm, "cgnni_bch_epoch18"), "ldpc": (codes.ldpc_toy_pcm, "cgnni_ldpc_epoch18")}


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001 -- no nvidia-smi: say so in the record
        power = None
    return name, power


def load(code):
    make_pcm, golden = CODES[code]
    pcm = make_pcm()
    z = np.load(os.path.join(ROOT, "tests", "golden", golden + ".npz"))
    weights = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
    return pcm, weights


def timed(fn, reps):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    fn()                                                   # warm-up of this shape
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(reps):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / reps


def bench_gpu(code, B, reps, dev):
    pcm, weights = load(code)
    g = TannerGraph.from_pcm(pcm, dev)
    dec = CGNNI.GNNI(T)
    dec.load_state_dict(weights)
    dec = dec.to(dev).train().bind_graph(g)
    x, err = sample_syndromes(g, B, SNR, noise=2, seed=1)
    y = err.float()
    lib = _cabi.lib()
    model = dec.gd_model()
    w = dec.packed_weights(dev)
    stash = torch.empty(lib.gd_stash_floats(g.handle, ct.byref(model), B), device=dev)
    prob = torch.empty((B, g.V), device=dev)
    logit = torch.empty((B, g.V), device=dev)
    gl = torch.randn((B, g.V), device=dev) * 1e-3
    ws = torch.empty(lib.gd_bwd_workspace_floats(g.handle, ct.byref(model), B), device=dev)
    gw = torch.empty(w.numel(), device=dev)
    st = ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: ct.c_void_p(t.data_ptr())   # noqa: E731

    def fwd():
        _cabi.check(lib.gd_decode_fwd_train(g.handle, ct.byref(model), p(w), p(x), p(prob), p(logit), p(stash), B, st))

    def bwd():
        _cabi.check(lib.gd_decode_bwd(g.handle, ct.byref(model), p(w), p(x), p(stash), p(gl), p(gw), p(ws), 0, B, st))

    opt = torch.optim.Adam(dec.parameters(), 1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = F.binary_cross_entropy(dec.decode(x), y)
        loss.backward()
        opt.step()

    fwd_ms = timed(fwd, reps)
    bwd_ms = timed(bwd, reps)
    step_ms = timed(step, reps)
    return {"fwd_stash_ms": round(fwd_ms, 4), "bwd_ms": round(bwd_ms, 4), "bwd_over_fwd": round(bwd_ms / fwd_ms, 3),
            "step_ms": round(step_ms, 4), "steps_per_s": round(1e3 / step_ms, 2), "syndromes_per_s": round(B * 1e3 / step_ms, 1),
            "stash_bytes": stash.numel() * 4}


def bench_cpu(code, B, reps):
    pcm, weights = load(code)
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    C, V = pcm.shape
    dev = "cuda:0"
    g = TannerGraph.from_pcm(pcm, dev)
    x, err = sample_syndromes(g, B, SNR, noise=2, seed=1)
    x, y = x.cpu(), err.float().cpu()

    def loss_fn(prob):
        return F.binary_cross_entropy(prob, y)
    restate.decode_grad("cgnni", ei, V, C, x, weights, loss_fn, T=T, dtype=torch.float32)      # warm-up
    t0 = time.perf_counter()
    for _ in range(reps):
        restate.decode_grad("cgnni", ei, V, C, x, weights, loss_fn, T=T, dtype=torch.float32)
    ms = (time.perf_counter() - t0) * 1e3 / reps
    return {"step_ms": round(ms, 2), "steps_per_s": round(1e3 / ms, 3), "syndromes_per_s": round(B * 1e3 / ms, 1),
            "cpu_threads": torch.get_num_threads()}


def profile(outdir, B):
    from torch.profiler import ProfilerActivity, profile as tprof
    pcm, weights = load("bch")
    dev = torch.device("cuda", 0)
    g = TannerGraph.from_pcm(pcm, dev)
    dec = CGNNI.GNNI(T)
    dec.load_state_dict(weights)
    dec = dec.to(dev).train().bind_graph(g)
    x, err = sample_syndromes(g, B, SNR, noise=2, seed=1)
    y = err.float()
    opt = torch.optim.Adam(dec.parameters(), 1e-4)

    def step():
        opt.zero_grad(set_to_none=True)
        F.binary_cross_entropy(dec.decode(x), y).backward()
        opt.step()
    step()
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            step()
        torch.cuda.synchronize()
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=15)
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, "cgnni_train_profile_B%d.txt" % B), "w") as f:
        f.write(table)
    print(table)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1024,16384,65536")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--cpu-B", type=int, default=1024)
    ap.add_argument("--cpu-reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("train_bench_cgnni.py needs a CUDA device")
    sizes = [int(s) for s in a.sizes.split(",")]
    if a.profile:
        profile(a.profile, max(sizes))
        return
    name, power = gpu_info()
    lines = []
    for code in ("bch", "ldpc"):
        for B in sizes:
            r = {"code": code, "arm": "gpu", "B": B, "T": T}
            r.update(bench_gpu(code, B, a.reps, torch.device("cuda", 0)))
            r.update({"gpu": name, "power_limit_w": power})
            lines.append(r)
            print(json.dumps(r), flush=True)
        r = {"code": code, "arm": "cpu_oracle_fp32", "B": a.cpu_B, "T": T}
        r.update(bench_cpu(code, a.cpu_B, a.cpu_reps))
        lines.append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()

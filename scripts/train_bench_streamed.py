"""decoder_v2_4 training-step timing on the hypergraph-product [[1600,64]] code (BASELINE config 5: V = 3200, C = 1536,
E = 10752), whose training state does not fit shared memory: the TMA-staged streamed forward with stash and the backward
with its work arrays in global memory.  T = 15, depolarizing noise (gd_sample noise 1), the toric L = 5 fixture's weights
(h = 128), FusedTrainer (forward -> gd_loss_v2_4 with the code's logicals -> backward -> Adam).  Per batch size, CUDA-event
times of
  fwd_stash_ms  gd_decode_fwd_train,
  loss_ms       gd_loss_v2_4,
  bwd_ms        gd_decode_bwd (backward + the fixed-order partial reduction),
  step_ms       FusedTrainer.step (all of the above + Adam),
the share of the MUFU bound -- the variable-phase MLP's E T h (2 + 3) MUFU operations per syndrome (forward ex2 + lg2,
backward ex2, lg2, rcp) over the ex2 rate gd_microbench measures in the same run -- and a CPU arm: the oracle's fp64
restatement + autograd (restate.decode_grad).  One JSON line per (arm, B), with the GPU's name and power limit.
  python scripts/train_bench_streamed.py [--sizes 1024,4096] [--out FILE] [--profile DIR]
--profile DIR: instead, a torch.profiler kernel table of three steps at the largest size (a separate run: tracing slows the
host)."""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gnn_decode_b200 import _cabi, codes  # noqa: E402
from gnn_decode_b200.graph import TannerGraph  # noqa: E402
from gnn_decode_b200.quantum import decoder_v2_4  # noqa: E402
from gnn_decode_b200.sampler import sample_syndromes  # noqa: E402
from gnn_decode_b200.train import FusedTrainer  # noqa: E402
from oracle import restate  # noqa: E402

T = 15
P = [0.01, 0.03, 0.05, 0.08]
MUFU_PER_UNIT = 2 + 3          # per variable-phase hidden unit and item: forward ex2 + lg2, backward ex2 + lg2 + rcp


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001 -- no nvidia-smi: say so in the record
        power = None
    return name, power


def setup(dev):
    Hz, Hx = codes.hgp_checks(codes.regular_ldpc(24, 32, 3, 4, 1234))
    pcm = codes.css_pcm(Hz, Hx)
    z = np.load(os.path.join(ROOT, "tests", "golden", "grad_v2_4_toricL5_epoch3_T6.npz"))
    weights = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
    g = TannerGraph.from_pcm(pcm, dev) if dev is not None else None
    return pcm, codes.css_logicals(Hz, Hx), weights, g


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


def mufu_rate():
    r = (ct.c_double * 2)()
    _cabi.check(_cabi.lib().gd_microbench(0, 4096, 0, r))      # ex2 instructions x lanes per second
    return r[0]


def bench_gpu(B, reps, dev, rate):
    pcm, logical, weights, g = setup(dev)
    dec = decoder_v2_4.GNNI(T)
    dec.load_state_dict(weights)
    dec = dec.to(dev).train()
    x, err = sample_syndromes(g, B, P, noise=1, seed=1)
    tr = FusedTrainer(dec, g, logical)
    lib = _cabi.lib()
    model = dec.gd_model()
    b = tr._buffers(B)
    ldev = torch.from_numpy(np.ascontiguousarray(logical, dtype=np.uint8)).to(dev)
    st = ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: ct.c_void_p(t.data_ptr())   # noqa: E731

    def fwd():
        _cabi.check(lib.gd_decode_fwd_train(g.handle, ct.byref(model), p(tr.w), p(x), p(b["prob"]), p(b["logit"]), p(b["stash"]),
                                            B, st))

    def loss():
        _cabi.check(lib.gd_loss_v2_4(g.handle, p(ldev), ldev.size(0), p(b["prob"]), p(err), p(b["per"]), None, p(b["gl"]), B, st))

    def bwd():
        _cabi.check(lib.gd_decode_bwd(g.handle, ct.byref(model), p(tr.w), p(x), p(b["stash"]), p(b["gl"]), p(tr.grad), p(b["ws"]),
                                      0, B, st))

    fwd_ms = timed(fwd, reps)
    loss_ms = timed(loss, reps)
    bwd_ms = timed(bwd, reps)
    step_ms = timed(lambda: tr.step(x, err), reps)
    mufu_ops = float(g.E) * T * dec.gd_model().hidden * MUFU_PER_UNIT * B
    return {"fwd_stash_ms": round(fwd_ms, 3), "loss_ms": round(loss_ms, 4), "bwd_ms": round(bwd_ms, 3),
            "step_ms": round(step_ms, 3), "syndromes_per_s": round(B * 1e3 / step_ms, 1),
            "mufu_ops_per_step": mufu_ops, "mufu_rate_per_s": rate,
            "mufu_share_of_step": round(mufu_ops / rate / (step_ms * 1e-3), 4),
            "stash_bytes": b["stash"].numel() * 4, "workspace_bytes": b["ws"].numel() * 4}


def bench_cpu(B, reps):
    pcm, logical, weights, _ = setup(None)
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    C, V = pcm.shape
    H = torch.from_numpy(pcm.T.astype(np.float64))
    L = torch.from_numpy(logical.astype(np.float64))
    dev = torch.device("cuda", 0)
    g = TannerGraph.from_pcm(pcm, dev)
    x, err = sample_syndromes(g, B, P, noise=1, seed=1)
    x, y = x.cpu().double(), err.cpu().double()

    def loss_fn(prob):
        return restate.loss_v2_4(prob, y, H, L)
    t0 = time.perf_counter()
    for _ in range(reps):
        restate.decode_grad("v2_4", ei, V, C, x, weights, loss_fn, T=T, dtype=torch.float64)
    ms = (time.perf_counter() - t0) * 1e3 / reps
    return {"step_ms": round(ms, 1), "syndromes_per_s": round(B * 1e3 / ms, 3), "cpu_threads": torch.get_num_threads()}


def profile(outdir, B):
    from torch.profiler import ProfilerActivity, profile as tprof
    dev = torch.device("cuda", 0)
    pcm, logical, weights, g = setup(dev)
    dec = decoder_v2_4.GNNI(T)
    dec.load_state_dict(weights)
    dec = dec.to(dev).train()
    x, err = sample_syndromes(g, B, P, noise=1, seed=1)
    tr = FusedTrainer(dec, g, logical)
    tr.step(x, err)
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            tr.step(x, err)
        torch.cuda.synchronize()
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=15)
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, "v2_4_hgp_train_profile_B%d.txt" % B), "w") as f:
        f.write("%s\n%s" % (json.dumps(dict(zip(("gpu", "power_limit_w"), gpu_info()))), table))
    print(table)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1024,4096")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cpu-B", type=int, default=4, help="fp64 autograd keeps ~1.3 GB per syndrome at T = 15")
    ap.add_argument("--cpu-reps", type=int, default=1)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("train_bench_streamed.py needs a CUDA device")
    sizes = [int(s) for s in a.sizes.split(",")]
    if a.profile:
        profile(a.profile, max(sizes))
        return
    name, power = gpu_info()
    rate = mufu_rate()
    lines = []
    for B in sizes:
        r = {"code": "hgp_1600_64", "arm": "gpu_fused_trainer", "B": B, "T": T}
        r.update(bench_gpu(B, a.reps, torch.device("cuda", 0), rate))
        r.update({"gpu": name, "power_limit_w": power})
        lines.append(r)
        print(json.dumps(r), flush=True)
    if a.cpu_B > 0:
        r = {"code": "hgp_1600_64", "arm": "cpu_oracle_fp64_autograd", "B": a.cpu_B, "T": T}
        r.update(bench_cpu(a.cpu_B, a.cpu_reps))
        lines.append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()

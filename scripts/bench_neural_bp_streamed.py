"""Neural BP decode throughput on the hypergraph-product [[1600,64]] code (BASELINE config 5: V = 3200, C = 1536, E = 10752),
whose edge state does not fit shared memory: the TMA-staged streamed kernel.  B = 16 384, T = 50, depolarizing noise (gd_sample
noise 1), seeded weights (W, W_p uniform in [0.6, 1.2], alpha = 0.25).  QGNNI (T = 50, the same kernel, the same 20 B per edge
and iteration) decodes the same batch in the same process, alternating step by step with neural BP, so both rates and both
shares of peak come from one run.

Per arm: CUDA-event time of each step (3 warm-up steps, then --steps timed ones; L2 flushed with a 256 MiB write before every
step), syndromes/s, and the share of the HBM peak measured in the same call (best of several >= 2 GB device-to-device copies,
read + write counted).  Algorithmic bytes per call: B (4N + 4V + V) (inputs, prob, hard) + B E (20 T - 8) (streamed edge state;
the first iteration fetches no m).  One JSON line per arm, with the GPU's name and power limit.
  python scripts/bench_neural_bp_streamed.py [--steps 10] [--out FILE]
  python scripts/bench_neural_bp_streamed.py --profile DIR     (a torch.profiler kernel table instead: tracing slows the host)"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gnn_decode_b200 import codes  # noqa: E402
from gnn_decode_b200.graph import TannerGraph  # noqa: E402
from gnn_decode_b200.quantum import QGNNI, neural_BP  # noqa: E402
from gnn_decode_b200.sampler import sample_syndromes  # noqa: E402

B, T = 16384, 50
P = [0.01, 0.03, 0.05, 0.08]
WARMUP = 3
COPY_BYTES = 2 << 30          # per side of the peak copy


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(out.splitlines()[0])
    except Exception:  # noqa: BLE001 -- no nvidia-smi: say so in the record
        power = None
    return name, power


def algorithmic_bytes(g):
    return B * (4 * g.N + 4 * g.V + g.V) + B * g.E * (20 * T - 8)


def hbm_peak_gbs(dev, reps=5):
    """Best of `reps` device-to-device copies of COPY_BYTES: (read + write) bytes / time."""
    src = torch.empty(COPY_BYTES, dtype=torch.uint8, device=dev).fill_(1)
    dst = torch.empty_like(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dst.copy_(src)
    best = 1e30
    for _ in range(reps):
        e0.record()
        dst.copy_(src)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del src, dst
    torch.cuda.empty_cache()
    return 2 * COPY_BYTES / (best * 1e-3) / 1e9


def setup(dev):
    g = TannerGraph.from_pcm(codes.hgp_pcm(), dev)
    x, _ = sample_syndromes(g, B, P, noise=1, seed=2024)
    torch.manual_seed(0)
    nbp = neural_BP.GNNI(T, n_edges=g.E)
    with torch.no_grad():
        for n_, p_ in nbp.named_parameters():
            p_.copy_(torch.full_like(p_, 0.25) if n_ == "alpha" else torch.rand_like(p_) * 0.6 + 0.6)
    torch.manual_seed(1)
    arms = {"neural_bp": nbp.to(dev).eval(), "qgnni": QGNNI.GNNI(T).to(dev).eval()}
    for name, dec in arms.items():
        info = g.launch_info(dec.gd_model(), B)
        if info["resident"] != 0:
            raise RuntimeError("%s did not take the streamed kernel: %s" % (name, info))
    return g, x, arms


def profile(out_dir, dev):
    g, x, arms = setup(dev)
    for dec in arms.values():
        for _ in range(WARMUP):
            dec.decode(x, graph=g)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for dec in arms.values():
            dec.decode(x, graph=g)
        torch.cuda.synchronize()
    os.makedirs(out_dir, exist_ok=True)
    table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=15)
    name, power = gpu_info()
    with open(os.path.join(out_dir, "neural_bp_streamed_profile.txt"), "w") as f:
        f.write("%s\n%s" % (json.dumps({"gpu": name, "power_limit_w": power, "B": B, "T": T}), table))
    print(table)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None, metavar="DIR")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    if a.profile:
        profile(a.profile, dev)
        return
    steps = max(10, a.steps)
    g, x, arms = setup(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for dec in arms.values():
        for _ in range(WARMUP):
            dec.decode(x, graph=g)
    torch.cuda.synchronize()
    peaks = [hbm_peak_gbs(dev)]
    times = {k: [] for k in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(steps):
        for name, dec in arms.items():                    # alternate the arms step by step
            flush.fill_(1)                                # evict the inputs and the slab from L2 (untimed)
            e0.record()
            dec.decode(x, graph=g)
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1))
    peaks.append(hbm_peak_gbs(dev))
    peak = max(peaks)
    gpu, power = gpu_info()
    nbytes = algorithmic_bytes(g)
    lines = []
    for name, ts in times.items():
        ts = sorted(ts)
        med = ts[len(ts) // 2]
        gbs = nbytes / (med * 1e-3) / 1e9
        lines.append({"arm": name, "code": "hgp_1600_64", "V": g.V, "C": g.C, "E": g.E, "B": B, "T": T, "noise": "depolarizing",
                      "steps": steps, "median_ms": med, "min_ms": ts[0], "max_ms": ts[-1], "syndromes_per_s": B / (med * 1e-3),
                      "algorithmic_bytes": nbytes, "achieved_gbs": gbs, "hbm_peak_gbs": peak, "hbm_peak_runs_gbs": peaks,
                      "frac_of_peak": gbs / peak, "l2": "flushed (256 MiB write) before every step",
                      "peak_source": "best device-to-device copy of 2 GiB in this run, read + write", "gpu": gpu,
                      "power_limit_w": power})
    for r in lines:
        print(json.dumps(r))
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in lines))


if __name__ == "__main__":
    main()

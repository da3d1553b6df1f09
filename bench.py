#!/usr/bin/env python
"""bench.py -- decoded syndromes/s of the fused message-passing decoder (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one pass of the hot path (GNNI.forward: T message-passing iterations + read-out +
hard decision) over one batch of synthetic syndromes.  N = 1 workload = BASELINE.json configs[1]:
the decoder_v2_4 program (hidden 128 Softplus, T = 15) on the rotated surface code d = 5 under
depolarizing noise, batch 65536 per GPU, sampled on the GPU by the Philox sampler before the timed
region.  N > 1 (torchrun, one rank per GPU): every rank decodes its own shard of the batch, no
data-path collective (SURVEY.md section 8e) -> "scaling": "weak".

`value`  : syndromes/s with inputs resident in HBM (CUDA events around each step, L2 flushed
           between steps, max over ranks).
`e2e`    : the same metric through the reference-facing call with HOST buffers
           (decoder.decode_host -> C ABI gd_decode_host): pinned host x -> device, kernel,
           prob + hard bits -> pinned host, all inside the timed region.
`roofline`: HBM roofline of the decode kernel (algorithmic bytes / measured duration vs
           MEASURED_PEAKS.json) -- tiny by construction, the fused kernel moves ~0.8 KB per
           syndrome -- plus `pipe`: the pipe that actually binds it (MUFU ex2+lg2 for Softplus),
           with its peak measured live by gd_microbench.
`cpu_baseline` / `--impl reference`: the oracle port of the reference's CPU path (same ATen op
           sequence, torch threads = all host cores) on a bounded sample of the same workload.
`--dump-outputs DIR`: the headline workload's prob and hard decisions from the last timed step, as float32 .npy files.  The
           inputs are a function of the arguments alone (seeded sampler, shipped weights), so the files of two builds compare
           output for output.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

_P10 = [0.01, 0.02, 0.03, 0.04, 0.05, 0.06, 0.07, 0.08, 0.09, 0.1]
_P5 = [0.01, 0.02, 0.03, 0.04, 0.05]
_SNR = [1.0, 2.0, 3.0, 4.0, 5.0, 6.0]
WORKLOADS = {
    # name: (program, code builder, T, per-GPU batch, noise, p list / SNR list)
    # BASELINE.json configs[1] -- the N = 1 default:
    "v2_4_rotated_d5_depol_B65536": ("v2_4", ("rotated", 5), 15, 65536, 1, _P10),
    "v2_4_toric_L5_iidxz_B65536": ("v2_4", ("toric", 5), 15, 65536, 0, _P10),
    # configs[2]: d = 11, batch sharded over the GPUs
    "v2_4_toric_L11_iidxz_B65536": ("v2_4", ("toric", 11), 15, 65536, 0, _P5),
    "v2_4_rotated_d11_depol_B65536": ("v2_4", ("rotated", 11), 15, 65536, 1, _P5),
    # configs[0]: classical decoder on the smallest bundled code (and BCH(63,45)), B = 1024
    "cgnni_ldpc_awgn_B1024": ("cgnni", ("ldpc", 8), 25, 1024, 2, _SNR),
    "cgnni_bch_awgn_B1024": ("cgnni", ("bch", 63), 25, 1024, 3, _SNR),
    "cgnni_bch_awgn_B65536": ("cgnni", ("bch", 63), 25, 65536, 3, _SNR),
    # configs[4]: hypergraph-product [[1600,64]], many iterations, streamed global-memory path
    "qgnni_hgp1600_depol_B16384_T50": ("qgnni", ("hgp", 1600), 50, 16384, 1, _P5),
    "bp_hgp1600_depol_B16384_T50": ("bp_quantum", ("hgp", 1600), 50, 16384, 1, _P5),
    "v2_4_hgp1600_depol_B8192": ("v2_4", ("hgp", 1600), 15, 8192, 1, _P5),
}
DEFAULT_WORKLOAD = "v2_4_rotated_d5_depol_B65536"
PROGRAM_NAMES = {"v2_4": "quantum/decoder_v2_4.GNNI (h=128 Softplus)", "qgnni": "quantum/QGNNI.GNNI (h=10 ReLU)",
                 "bp_quantum": "quantum/BP.GNNI (sum-product)", "cgnni": "classical/CGNNI.GNNI (h=10 ReLU)"}


def build_pcm(spec):
    from gnn_decode_b200 import codes
    kind, size = spec
    if kind == "rotated":
        return codes.rotated_surface_pcm(size)
    if kind == "toric":
        return codes.toric_pcm(size)
    if kind == "hgp":
        return codes.hgp_pcm()
    if kind == "ldpc":
        return codes.ldpc_toy_pcm()
    return codes.bch_63_45_pcm()


def _golden_weights(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", name))
    return {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}


def load_weights(program):
    """Weights as a reference state_dict: the shipped checkpoints (carried in the golden fixtures) for
    decoder_v2_4 (quantum/new_model/epoch3) and CGNNI (classical/model/epoch18); the reference ships no
    QGNNI checkpoint, so that program runs its own seeded default initialisation; BP has none."""
    if program == "v2_4":
        return _golden_weights("v2_4_toricL5_epoch3.npz"), "reference checkpoint quantum/new_model epoch3"
    if program == "cgnni":
        return _golden_weights("cgnni_ldpc_epoch18.npz"), "reference checkpoint classical/model epoch18"
    if program == "qgnni":
        from gnn_decode_b200.quantum import QGNNI
        torch.manual_seed(1234)
        return {k: v.detach().clone() for k, v in QGNNI.GNNI(1).state_dict().items()}, "seeded default init (no shipped checkpoint)"
    return {}, "none (parameter-free)"


def make_decoder(program, T, weights):
    from gnn_decode_b200.quantum import decoder_v2_4, QGNNI, BP
    from gnn_decode_b200.classical import CGNNI
    dec = {"v2_4": decoder_v2_4.GNNI, "qgnni": QGNNI.GNNI, "bp_quantum": BP.GNNI, "cgnni": CGNNI.GNNI}[program](T)
    if weights:
        dec.load_state_dict(weights)
    return dec


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed regions (B200_PROFILING.md recipe).
    The sampler process is started before warm-up (it takes ~0.3 s to produce its first line); only
    samples that arrive inside a marked window [begin(), end()] are reported."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.windows, self._t0 = index, None, [], [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.monotonic(), line.strip()))

    def begin(self):
        self._t0 = time.monotonic()

    def end(self):
        self.windows.append((self._t0, time.monotonic()))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for t, ln in self.lines:
            if not any(a - 0.02 <= t <= b + 0.03 for a, b in self.windows):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples inside the timed windows"],
                    "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(power),
                "window_s": round(sum(b - a for a, b in self.windows), 4)}


# ---------------------------------------------------------------------------------------------
_ALLOCATOR_WARM = False


def _warm_cpu_allocator():
    """Be fair to the CPU reference: its intermediates are ~10 MB tensors, exactly at glibc's dynamic mmap threshold
    in a fresh process, so every ATen op would mmap + page-fault + munmap its output (measured on the GPU box: 2.5 k
    syndromes/s cold vs 8.3 k once any larger block has been freed, which raises the threshold and keeps those
    tensors on the heap).  A long-running reference process is in the fast state; put this one there too."""
    global _ALLOCATOR_WARM
    if not _ALLOCATOR_WARM:
        t = torch.empty(30 << 20, dtype=torch.uint8)   # < glibc's 32 MB cap: freeing it raises the mmap threshold to 30 MB
        t.fill_(1)
        del t
        _ALLOCATOR_WARM = True


def cpu_reference_rate(program, pcm, T, weights, x_sample, chunk, budget_s, threads):
    """Time the oracle port (the reference's CPU arithmetic) on a bounded sample; returns
    (syndromes/s, syndromes timed, seconds)."""
    from gnn_decode_b200 import codes
    from oracle import restate
    torch.set_num_threads(threads)
    _warm_cpu_allocator()
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    C_, V = pcm.shape
    done, t_used = 0, 0.0
    restate.decode(program, ei, V, C_, x_sample[:min(chunk, 8)], weights, T=T)     # warm-up
    i = 0
    while done < x_sample.size(0) and t_used < budget_s:
        xb = x_sample[i:i + chunk]
        if xb.size(0) == 0:
            break
        t0 = time.perf_counter()
        restate.decode(program, ei, V, C_, xb, weights, T=T)
        t_used += time.perf_counter() - t0
        done += xb.size(0)
        i += chunk
    return done / t_used, done, t_used


DUMP_BUDGET = 63 * 10 ** 6      # bytes of array data written by --dump-outputs: with the .npy headers, under 64 MB


def dump_outputs(path, arrays):
    """Write each [B, ...] output as path/<name>.npy in float32, so that two builds can be compared output for output.  When they
    exceed DUMP_BUDGET together, the same fixed, seeded sample of rows is kept from each, and its row indices go to rows.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {k: v.cpu().numpy().astype(np.float32) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes for a in arrays.values()) // max(n, 1)
    if n * row_bytes > DUMP_BUDGET:
        rows = np.sort(np.random.RandomState(1234).choice(n, DUMP_BUDGET // (row_bytes + 8), replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-autotune", action="store_true", help="keep the planner's model geometry (skip gd_decode_autotune)")
    ap.add_argument("--no-extras", action="store_true", help="headline workload only (skip the short passes over the other BASELINE configs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the headline workload returned (prob, hard) as DIR/<name>.npy "
                         "(rank 0's shard under torchrun)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    program, code_spec, T, B, noise, p_list = WORKLOADS[args.workload]
    pcm = build_pcm(code_spec)
    Cn, V = pcm.shape
    N = V + Cn
    E = int(pcm.sum())
    weights, weights_src = load_weights(program)
    cores = os.cpu_count() or 1
    config = {"workload": args.workload, "program": PROGRAM_NAMES[program], "code": "%s-%d" % code_spec,
              "V": V, "C": Cn, "E": E, "T": T, "batch_per_gpu": B,
              "noise": ["iid-xz", "depolarizing", "awgn (all-zero codeword)", "awgn (all-one codeword)"][noise],
              "l2": "L2 flushed (256 MiB write) between timed steps", "weights": weights_src}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        from gnn_decode_b200 import codes  # noqa: F401  (host-side code builders only)
        rng = np.random.RandomState(1234)
        # bounded sample of the same workload: synthetic syndromes with the same layout/statistics
        est_rate, _, _ = cpu_reference_rate(program, pcm, T, weights, _host_sample(pcm, noise, p_list, 128, rng), 128, 5.0, cores)
        total_budget = 150.0
        per_step = int(max(128, min(4096, est_rate * total_budget / max(1, args.steps + args.warmup))) // 128 * 128)
        xs = _host_sample(pcm, noise, p_list, per_step, rng)
        for _ in range(args.warmup):
            cpu_reference_rate(program, pcm, T, weights, xs, 128, 1e9, cores)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_reference_rate(program, pcm, T, weights, xs, 128, 1e9, cores)
        dt = time.perf_counter() - t0
        value = per_step * args.steps / dt
        line = {"impl": "reference", "metric": "decoded syndromes/sec", "value": value, "unit": "syndromes/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if program == "cgnni" else "f64", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": value, "unit": "syndromes/s", "cores": cores, "kind": "port",
                                 "sample": "%d syndromes per step in chunks of 128 (the reference's BATCH_SIZE), reference dtype, "
                                           "torch CPU %d threads, oracle/restate.py" % (per_step, cores)},
                "e2e": {"value": value, "unit": "syndromes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _pin_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    line = run_workload(args.workload, args, dev, rank, world, clocks, headline=True)
    extras = []
    if not args.no_extras:
        for name in EXTRA_WORKLOADS:
            if name == args.workload:
                continue
            try:
                extras.append(run_workload(name, args, dev, rank, world, None, headline=False))
            except Exception as ex:  # noqa: BLE001  (an extra must never cost the headline line)
                extras.append({"workload": name, "error": "%s: %s" % (type(ex).__name__, ex)})
        try:
            extras.append(run_training(args, dev, rank, world))
        except Exception as ex:  # noqa: BLE001
            extras.append({"workload": TRAIN_WORKLOAD, "error": "%s: %s" % (type(ex).__name__, ex)})
    if rank == 0:
        clk = clocks.stop()
        if line.get("_clock_probe_s"):
            clk["load_probe_s"] = line.pop("_clock_probe_s")
        line.pop("_clock_probe_s", None)
        line["clocks"] = clk
        if extras:
            line["extra_workloads"] = extras
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


# the other BASELINE.json configs, run short after the headline and embedded as `extra_workloads`
EXTRA_WORKLOADS = ["cgnni_ldpc_awgn_B1024", "cgnni_bch_awgn_B1024", "v2_4_toric_L11_iidxz_B65536", "v2_4_rotated_d11_depol_B65536",
                   "qgnni_hgp1600_depol_B16384_T50", "bp_hgp1600_depol_B16384_T50"]
TRAIN_WORKLOAD = "train_v2_4_rotated_d7_B4096"


def _pin_to_gpu_numa_node(index):
    """Run this rank (and first-touch its pinned buffers) on the CPUs next to its GPU.  No-op when the topology is not exposed."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:  # noqa: BLE001
        pass


def lean_wavefronts_per_syndrome(pcm, T):
    """Algorithmic shared-memory wavefronts (128 B each) per syndrome of the check-owner table kernel (DESIGN.md 4.0): per
    iteration and edge one message read, one message write and one 128-bit check-table look-up (4 wavefronts per warp),
    plus, where the variable has a second edge, one sibling read and one 128-bit variable-table look-up; the first
    iteration (all messages zero) is one look-up per check; the read-out is one read + one look-up per edge and a staged
    logit per variable.  Counted per warp of 32 syndromes, conflict-free, metadata broadcasts not counted."""
    deg = pcm.sum(0)
    E = int(pcm.sum())
    E_sib = int(deg[deg >= 2].sum())
    Cn, V = pcm.shape
    per_warp = (T - 1) * (6 * E + 5 * E_sib) + (E + 4 * Cn) + 5 * E + 2 * V
    return per_warp / 32.0


def run_workload(name, args, dev, rank, world, clocks, headline):
    from gnn_decode_b200 import _cabi, options, packing
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.pipeline import DecodePipeline
    from gnn_decode_b200.sampler import sample_syndromes
    program, code_spec, T, B, noise, p_list = WORKLOADS[name]
    pcm = build_pcm(code_spec)
    Cn, V = pcm.shape
    N = V + Cn
    E = int(pcm.sum())
    weights, weights_src = load_weights(program)
    cores = os.cpu_count() or 1
    steps = args.steps if headline else max(3, min(args.steps, 10))
    warmup = args.warmup if headline else 3
    local_rank = dev.index
    g = TannerGraph.from_pcm(pcm, dev)
    dec = make_decoder(program, T, weights).to(dev).eval()
    dec.bind_graph(g)
    model = dec.gd_model()
    info = g.launch_info(model, B)
    x, err = sample_syndromes(g, B, p_list, noise=noise, seed=1234, first_sample=rank * B)
    lean = False
    if program == "v2_4":
        with options.option("GD_NO_LEAN"):
            lean = g.launch_info(model, B) != info
    if not args.no_autotune and not lean:
        dec.autotune(x)                      # edge-owner kernel only: one-time geometry measurement, outside every timed region
        info = g.launch_info(model, B)
    prob = torch.empty((B, V), dtype=torch.float32, device=dev)
    hard = torch.empty((B, V), dtype=torch.uint8, device=dev)
    wdev = dec.packed_weights(dev)
    wptr = C.c_void_p(wdev.data_ptr()) if wdev is not None else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lib = _cabi.lib()
    stream = torch.cuda.current_stream(dev)

    def step(xx=x):
        _cabi.check(lib.gd_decode_fwd(g.handle, C.byref(model), wptr, C.c_void_p(xx.data_ptr()),
                                      C.c_void_p(prob.data_ptr()), None, C.c_void_p(hard.data_ptr()), xx.size(0),
                                      C.c_void_p(stream.cuda_stream)))

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(dev)

    def allmax(v):
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    for _ in range(warmup):
        flush.fill_(1)
        step()
    barrier()
    if clocks is not None and rank == 0:
        clocks.begin()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for e0, e1 in evs:
        flush.fill_(1)                       # evict the inputs from L2 (untimed)
        e0.record(stream)
        step()
        e1.record(stream)
    barrier()
    if clocks is not None and rank == 0:
        clocks.end()
    prob_ref, hard_ref = prob.cpu(), hard.cpu()             # what the last timed step returned
    if headline and rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"prob": prob_ref, "hard": hard_ref})
    clock_probe_s = 0.0
    # The timed region can be shorter than the clock sampler's period (nvidia-smi reports every 20 ms): keep exactly the same
    # step running, untimed, for 0.3 s more so the clocks / throttle reasons are sampled under this load.
    if clocks is not None and rank == 0 and clocks.windows[-1][1] - clocks.windows[-1][0] < 0.3:
        clocks.begin()
        t_probe = time.monotonic()
        while time.monotonic() - t_probe < 0.3:
            for _ in range(8):
                step()
            torch.cuda.synchronize(dev)
        clocks.end()
        clock_probe_s = round(time.monotonic() - t_probe, 3)
    kernel_ms = [e0.elapsed_time(e1) for e0, e1 in evs]
    total_ms_max = allmax(sum(kernel_ms))
    ms_per_step = total_ms_max / steps
    value = world * B * steps / (total_ms_max * 1e-3)

    # ---- end to end: pinned host buffers -> device -> decode -> host, every step, through the asynchronous pipeline ----
    depth = 3
    pipe = DecodePipeline(dec, g, max_B=B, depth=depth)
    xh = x.cpu().pin_memory()
    e2e = {}
    if program == "v2_4" and g.launch_info(dec.gd_model(), B)["resident"]:       # (gd_decode_packed_fwd: resident codes only)
        # packed form: what x carries per syndrome is one prior float + C check-sign bits; V hard-decision bits come back
        prior_d, synd_d = packing.pack_x(x, V)
        prior_h, synd_h = prior_d.cpu().pin_memory(), synd_d.cpu().pin_memory()
        bits_h = [torch.empty((B, (V + 31) // 32), dtype=torch.int32).pin_memory() for _ in range(depth)]
        for i in range(depth):
            pipe.submit_packed(prior_h, synd_h, hard_bits_out=bits_h[i])
        pipe.drain()
        barrier()
        if clocks is not None and rank == 0:
            clocks.begin()
        t0 = time.perf_counter()
        for i in range(steps):
            pipe.submit_packed(prior_h, synd_h, hard_bits_out=bits_h[i % depth])   # H2D of this step's inputs + decode + D2H of its result
        pipe.drain()
        dt = allmax(time.perf_counter() - t0)
        if clocks is not None and rank == 0:
            clocks.end()
        same_bits = bool(torch.equal(packing.unpack_bits(bits_h[(steps - 1) % depth], V), hard_ref))
        e2e = {"value": world * B * steps / dt, "unit": "syndromes/s",
               "h2d_bytes_per_step": B * (4 + 4 * ((Cn + 31) // 32)), "d2h_bytes_per_step": B * 4 * ((V + 31) // 32),
               "api": "DecodePipeline.submit_packed -> gd_pipeline_submit_packed (pinned host buffers; prior float + check-sign bits "
                      "in, hard-decision bits out; %d batches in flight)" % depth,
               "matches_device_path": same_bits}
    # the reference's own layout: x [B, V+C] fp32 in, prob fp32 + hard bytes out
    prob_h = [torch.empty((B, V), dtype=torch.float32).pin_memory() for _ in range(depth)]
    hard_h = [torch.empty((B, V), dtype=torch.uint8).pin_memory() for _ in range(depth)]
    n_e2e = steps if headline else max(3, steps // 2)
    for i in range(depth):
        pipe.submit(xh, prob_out=prob_h[i], hard_out=hard_h[i])
    pipe.drain()
    barrier()
    t0 = time.perf_counter()
    for i in range(n_e2e):
        pipe.submit(xh, prob_out=prob_h[i % depth], hard_out=hard_h[i % depth])
    pipe.drain()
    dt = allmax(time.perf_counter() - t0)
    same = bool(torch.equal(prob_h[(n_e2e - 1) % depth], prob_ref) and torch.equal(hard_h[(n_e2e - 1) % depth], hard_ref))
    fp32_form = {"value": world * B * n_e2e / dt, "unit": "syndromes/s", "h2d_bytes_per_step": B * N * 4, "d2h_bytes_per_step": B * V * 5,
                 "api": "DecodePipeline.submit -> gd_pipeline_submit (x [B, V+C] fp32 in, prob fp32 + hard uint8 out; %d batches in flight)" % depth,
                 "matches_device_path": same}
    if e2e:
        e2e["fp32_form"] = fp32_form
    else:
        e2e = fp32_form
    if headline:
        # the blocking single call of round 1, for continuity
        dec.decode_host(xh, prob_h[0], hard_h[0])
        barrier()
        t0 = time.perf_counter()
        for _ in range(max(3, steps // 3)):
            dec.decode_host(xh, prob_h[0], hard_h[0])
        dt = allmax(time.perf_counter() - t0)
        e2e["blocking_call"] = {"value": world * B * max(3, steps // 3) / dt, "unit": "syndromes/s",
                                "api": "GNNI.decode_host -> gd_decode_host (one synchronous call per batch, fp32 layout)",
                                "matches_device_path": bool(torch.equal(prob_h[0], prob_ref))}
    del pipe

    out = {"metric": "decoded syndromes/sec", "value": value, "unit": "syndromes/s", "n_gpus": world,
           "steps": steps, "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    if rank != 0:
        return out
    config = {"workload": name, "program": PROGRAM_NAMES[program], "code": "%s-%d" % code_spec,
              "V": V, "C": Cn, "E": E, "T": T, "batch_per_gpu": B,
              "noise": ["iid-xz", "depolarizing", "awgn (all-zero codeword)", "awgn (all-one codeword)"][noise],
              "l2": "L2 flushed (256 MiB write) between timed steps", "weights": weights_src, "launch": info,
              "parallelism": "batch-sharded x%d, no collective" % world}
    # ---- rooflines ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        hbm_peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    else:
        hbm_peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    io_bytes = B * (4 * N + 4 * V + V)                       # x in, prob + hard out, per launch
    med_ms = statistics.median(kernel_ms)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_decode_kernel_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(name)
    n_kernels = 1
    if info["resident"]:
        alg_bytes = io_bytes
        kname = "gd::lean_decode_kernel (+ prep / tables / deferred-pass launches)" if lean else "gd::decode_kernel<%s, resident>" % program
        n_kernels = 4 if lean else 1
        note = "fused resident kernel: ~%d B/syndrome of HBM traffic, so HBM is not the binding resource; see pipe" % (alg_bytes // B)
    else:
        # streamed path (DESIGN.md 4.2): per edge and iteration m: R,R,W  t: W,R = 20 B for the learned programs, 16 B for
        # sum-product (sign rides in t); the first iteration reads no m (m == 0).
        per_edge = (16 * T - 4) if program.startswith("bp") else (20 * T - 8)
        alg_bytes = io_bytes + B * E * max(per_edge, 0)
        kname = "gd::decode_streamed_tma_kernel<%s>" % program
        note = "streamed global-memory path: %.2f MB of edge-state traffic per syndrome" % (E * per_edge / 1e6)
    achieved = alg_bytes / (med_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "peak_source": peak_src, "kernel": kname,
                "kernel_ms": med_ms, "algorithmic_bytes_per_launch": alg_bytes, "note": note}
    if lean:
        r = (C.c_double * 2)()
        _cabi.check(lib.gd_microbench(7, 4096, local_rank, r))    # conflict-free 128-bit shared-memory loads: wavefronts / s
        wf_peak = r[0]
        wf = lean_wavefronts_per_syndrome(pcm, T) * B
        measured = None
        mpath = os.path.join(ROOT, "profiles", "r02_lean_kernel_ncu.json")
        if os.path.exists(mpath):
            measured = json.load(open(mpath)).get(name)
        roofline["pipe"] = {
            "name": "shared-memory data pipe (l1tex LSU wavefronts, 128 B per cycle per SM): the decoder evaluates nothing but table "
                    "look-ups -- all three Softplus MLPs and the tanh are cubic tables built in double precision once per weight "
                    "set (DESIGN.md 4.0) -- so 128-bit table loads and the message reads / writes are the whole kernel",
            "achieved": wf / (med_ms * 1e-3) / 1e12, "peak": wf_peak / 1e12, "unit": "T wavefronts/s",
            "frac": wf / (med_ms * 1e-3) / wf_peak,
            "what": "ALGORITHMIC (conflict-free) wavefronts per launch = %.0f per syndrome x %d syndromes, over the time of the WHOLE "
                    "step (4 launches: hash check + input packing, table refresh + sort by prior, decode, deferred pass); the decode "
                    "kernel alone is ~85%% of it" % (wf / B, B),
            "peak_source": "gd_microbench kind=7 (conflict-free LDS.128 stream), measured live on this GPU",
            "ncu": measured}
    elif program == "v2_4":
        r = (C.c_double * 2)()
        _cabi.check(lib.gd_microbench(1, 4096, local_rank, r))   # ex2+lg2 pairs / s: the Softplus unit rate
        deg = pcm.sum(0)
        n_vact = int(deg[deg >= 2].sum())
        hid = dec.mlp[0].out_features
        units = B * hid * (T * n_vact + (E - n_vact)) if info["resident"] else B * hid * T * E
        roofline["pipe"] = {"name": "xu (MUFU): Softplus hidden units of the 2-input variable-phase MLP evaluated directly (check-phase and "
                                    "read-out MLPs are cubic tables); peak = the 2-MUFU-per-unit (ex2+lg2) rate",
                            "achieved": units / (med_ms * 1e-3) / 1e12, "peak": r[0] / 1e12, "unit": "T Softplus units/s",
                            "frac": units / (med_ms * 1e-3) / r[0],
                            "peak_source": "gd_microbench kind=1 (ex2+lg2 pairs/s), measured live on this GPU", "units_per_launch": units}
    out.update({"config": config, "e2e": e2e, "gpu_launches": steps * n_kernels, "roofline": roofline})
    if headline and lean:
        # the general path beside the fast one: the same batch with per-variable priors (no syndrome is table-eligible, every
        # one is decoded by the edge-owner kernel's direct evaluation)
        xg = x.clone()
        xg[:, :V] += 1e-3 * torch.arange(V, device=dev, dtype=torch.float32)
        for _ in range(2):
            step(xg)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(3):
            step(xg)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        out["general_path"] = {"value": 3 * B / (e0.elapsed_time(e1) * 1e-3), "unit": "syndromes/s (1 GPU)",
                               "what": "same batch with per-variable priors: nothing is table-eligible, every syndrome takes the "
                                       "edge-owner kernel's direct (MUFU) evaluation of the variable-phase MLP"}
    if headline:
        out["_clock_probe_s"] = clock_probe_s
    if headline and not args.no_cpu_baseline and world == 1:
        rng = np.random.RandomState(1234)  # noqa: F841
        # bounded sample: this workload's own syndromes (cycled if the batch is small), stop after ~15 s of CPU work
        n_s = max(128, min(131072, int(5e7 // N)))           # <= 400 MB of fp64 inputs
        reps = max(1, -(-n_s // B))
        xs_cpu = x[:n_s].cpu().double().repeat(reps, 1)[:n_s]
        rate, n_done, secs = cpu_reference_rate(program, pcm, T, weights, xs_cpu, 128, 15.0, cores)
        out["cpu_baseline"] = {"value": rate, "unit": "syndromes/s", "cores": cores, "kind": "port",
                               "sample": "%d syndromes of this workload in chunks of 128 (the reference's BATCH_SIZE), "
                                         "fp64, %.1f s, oracle/restate.py on %d torch threads" % (n_done, secs, cores)}
    if not headline:
        out = {"workload": name, "value": out["value"], "unit": "syndromes/s", "ms_per_step": ms_per_step, "steps": steps,
               "n_gpus": world, "e2e": e2e, "roofline": {k: roofline[k] for k in ("bound", "achieved", "peak", "unit", "frac", "kernel")},
               "config": {k: config[k] for k in ("program", "code", "V", "C", "E", "T", "batch_per_gpu", "noise", "launch")}}
        if "pipe" in roofline:
            out["roofline"]["pipe"] = {k: roofline["pipe"][k] for k in ("achieved", "peak", "unit", "frac")}
    return out


def run_training(args, dev, rank, world):
    """BASELINE configs[3]: one training step of the decoder_v2_4 program on the rotated surface code d = 7, B = 4096 per GPU:
    forward with stash, sparse loss, hand-written backward, gradient all-reduce (one peer-memory kernel with Adam fused in;
    NCCL when symmetric memory is unavailable), Adam."""
    import torch.distributed as dist
    from gnn_decode_b200 import codes
    from gnn_decode_b200.graph import TannerGraph
    from gnn_decode_b200.quantum import decoder_v2_4
    from gnn_decode_b200.sampler import sample_syndromes
    from gnn_decode_b200.train import FusedTrainer
    d, B, T = 7, 4096, 15
    Hz, Hx = codes.rotated_surface_checks(d)
    pcm = codes.css_pcm(Hz, Hx)
    logical = codes.css_logicals(Hz, Hx)
    g = TannerGraph.from_pcm(pcm, dev)
    torch.manual_seed(0)
    dec = decoder_v2_4.GNNI(T).to(dev).train().bind_graph(g)
    p2p, how = None, "none (1 GPU)"
    if world > 1:
        how = "NCCL all-reduce of the flat gradient (1 283 floats)"
        try:
            from gnn_decode_b200.dist import P2PAllReduce
            p2p = P2PAllReduce(sum(p.numel() for p in dec._gd_params()), dev)
            how = "peer-memory kernel over NVLink (gd_p2p_allreduce_adam: exchange + Adam in one launch)"
        except Exception as ex:  # noqa: BLE001
            how += " [peer-memory kernel unavailable: %s]" % type(ex).__name__
    trainer = FusedTrainer(dec, g, logical, lr=3e-4, weight_decay=1e-9, p2p=p2p)
    x, err = sample_syndromes(g, B, [0.01, 0.03, 0.05, 0.08], noise=1, seed=1, first_sample=rank * B)
    for _ in range(3):
        trainer.step(x, err)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    n = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        loss = trainer.step(x, err)
    e1.record()
    torch.cuda.synchronize(dev)
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item() / n
    ar_us = None
    if world > 1:
        flat = torch.zeros(trainer.w.numel(), dtype=torch.float32, device=dev)
        fn = (lambda: p2p(flat)) if p2p is not None else (lambda: dist.all_reduce(flat))
        for _ in range(5):
            fn()
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(50):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        ar_us = e0.elapsed_time(e1) / 50 * 1e3
        if p2p is not None:
            p2p.check()
    return {"workload": TRAIN_WORKLOAD, "value": world * B / (ms * 1e-3), "unit": "syndromes/s", "ms_per_step": ms,
            "steps_per_s": 1e3 / ms, "steps": n, "n_gpus": world, "loss": float(loss.item()),
            "gradient_allreduce": how, "allreduce_us": ar_us,
            "config": {"program": PROGRAM_NAMES["v2_4"], "code": "rotated-7", "V": g.V, "C": g.C, "E": g.E, "T": T, "batch_per_gpu": B,
                       "step": "forward(+stash) + loss + backward + all-reduce + Adam(lr 3e-4, wd 1e-9), fp32 master weights"}}


def _host_sample(pcm, noise, p_list, n, rng):
    """Host-side synthetic syndromes with gen_syn's layout (quantum/error_generate.py:252-278), or the
    classical AWGN LLRs of classical/CGNNI.py:125-147,159 for noise 2 / 3."""
    Cn, V = pcm.shape
    if noise >= 2:
        snr = np.asarray(p_list)[rng.randint(0, len(p_list), n)]
        sigma = np.sqrt(1.0 / 10.0 ** (snr / 10.0))[:, None]
        y = (1.0 if noise == 2 else -1.0) + sigma * rng.standard_normal((n, V))
        return torch.from_numpy(np.concatenate([2.0 * y / sigma ** 2, np.zeros((n, Cn))], 1))
    p = np.asarray(p_list)[rng.randint(0, len(p_list), n)]
    if noise == 0:
        err = (rng.random_sample((n, V)) < p[:, None]).astype(np.uint8)
        pm = p
    else:
        nq = V // 2
        u = rng.random_sample((n, nq))
        err = np.concatenate([(u < 2 * p[:, None] / 3), (u >= p[:, None] / 3) & (u < p[:, None])], 1).astype(np.uint8)
        pm = 2 * p / 3
    syn = (err.astype(np.int64) @ pcm.T.astype(np.int64)) % 2
    x = np.concatenate([np.repeat(np.log((1 - pm) / pm)[:, None], V, 1), 1.0 - 2.0 * syn], 1)
    return torch.from_numpy(x)


if __name__ == "__main__":
    sys.exit(main())

"""bench.py's output contract: the reference arm (`--impl reference`, the oracle port on the host cores) runs without a
GPU and prints the agreed JSON line; bad arguments are refused; --dump-outputs stays inside its size budget; the roofline numerator
of the table kernel is what DESIGN.md says it is.  (The GPU arm's
line is checked where a GPU exists: tests/test_bench_gpu.py.)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def _check_common(d):
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["metric"] == "decoded syndromes/sec" and d["unit"] == "syndromes/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["data"] == "synthetic" and "workload" in d["config"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["ms_per_step"] > 0


def test_reference_arm_runs_on_cpu_and_prints_the_contract_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    _check_common(d)
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"] == "v2_4_rotated_d5_depol_B65536"        # BASELINE.json configs[1]


def test_bench_rejects_zero_steps_and_reference_dumps():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, cwd=ROOT, env=env, capture_output=True,
                             text=True, timeout=300)
        assert out.returncode == 2 and "error:" in out.stderr, (extra, out.stderr[-2000:])
    assert not os.path.exists(os.path.join(ROOT, "unused"))


def test_dump_outputs_keeps_a_fixed_sample_of_rows_within_the_budget(tmp_path, monkeypatch):
    """An output pair larger than the budget is written as the same seeded sample of rows from each array, with the row indices
    (at a 1 MB budget here; the same rule keeps e.g. the HGP workload's 210 MB of prob + hard inside 64 MB)."""
    import numpy as np
    import torch
    monkeypatch.syspath_prepend(ROOT)
    import bench
    budget = 10 ** 6
    monkeypatch.setattr(bench, "DUMP_BUDGET", budget)
    B, V = 2048, 300                                     # 4.9 MB of prob + hard as float32
    prob = torch.rand(B, V, generator=torch.Generator().manual_seed(0))
    hard = (prob > 0.5).to(torch.uint8)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), {"prob": prob, "hard": hard})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["hard.npy", "prob.npy", "rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= budget + 3 * 128       # + one .npy header per file
    rows = np.load(tmp_path / "a" / "rows.npy")
    assert rows.dtype == np.float64 and len(rows) == budget // (8 * V + 8) and (np.diff(rows) > 0).all()
    p, h = np.load(tmp_path / "a" / "prob.npy"), np.load(tmp_path / "a" / "hard.npy")
    assert p.dtype == h.dtype == np.float32 and p.shape == h.shape == (len(rows), V)
    assert np.array_equal(p, prob.numpy()[rows.astype(np.int64)]) and np.array_equal(h, hard.numpy()[rows.astype(np.int64)])
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


def test_wavefront_count_of_the_table_kernel():
    """bench.py's algorithmic shared-memory wavefront count (the roofline numerator of the check-owner table kernel) on the
    headline code: rotated d = 5 has 80 edges, 60 of them on variables with a second edge, 24 checks, 50 variables."""
    sys.path.insert(0, ROOT)
    import bench
    from gnn_decode_b200 import codes
    pcm = codes.rotated_surface_pcm(5)
    assert bench.lean_wavefronts_per_syndrome(pcm, 15) == (14 * (6 * 80 + 5 * 60) + (80 + 4 * 24) + 5 * 80 + 2 * 50) / 32.0

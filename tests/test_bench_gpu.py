"""The GPU arm of bench.py prints the contract line (run short, headline workload only)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(dump_dir):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "3", "--no-extras", "--no-cpu-baseline",
                          "--dump-outputs", str(dump_dir)],
                         cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_gpu_arm_prints_the_contract_line(tmp_path):
    d = _bench(tmp_path / "a")
    assert d["steps"] == 3
    # the last timed step's outputs, whole (the headline's 65536 x 50 pair is inside the size budget)
    prob, hard = np.load(tmp_path / "a" / "prob.npy"), np.load(tmp_path / "a" / "hard.npy")
    assert sorted(os.listdir(tmp_path / "a")) == ["hard.npy", "prob.npy"]
    assert prob.shape == hard.shape == (65536, 50) and prob.dtype == hard.dtype == np.float32
    assert ((prob >= 0) & (prob <= 1)).all() and set(np.unique(hard)) <= {0.0, 1.0}
    decided = np.abs(prob - 0.5) > 1e-3
    assert np.array_equal(hard[decided], (prob[decided] > 0.5).astype(np.float32))
    # the same arguments give the same inputs, so a second run dumps the same outputs
    _bench(tmp_path / "b")
    for f in ("prob.npy", "hard.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "clocks", "gpu_launches", "roofline"):
        assert k in d, k
    assert d["config"]["workload"] == "v2_4_rotated_d5_depol_B65536" and d["n_gpus"] == 1 and d["gpu_launches"] > 0
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert 0 < r["pipe"]["frac"] < 1.2 and r["pipe"]["unit"] == "T wavefronts/s"
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["matches_device_path"] is True
    assert e["fp32_form"]["matches_device_path"] is True and e["blocking_call"]["matches_device_path"] is True
    assert e["value"] > 0 and e["fp32_form"]["value"] < d["value"]   # (the packed form skips the 19 MB input scan: it may beat `value`)
    assert d["general_path"]["value"] < d["value"]

import glob
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    """`gpu`-marked tests need a CUDA device: skip (not fail) them on a box without one."""
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class _GdOptions(object):
    """Set / unset library tunables (gnn_decode_b200.options) for one test; everything touched is unset again afterwards."""

    def __init__(self):
        self.touched = set()

    def set(self, name, value=1):
        from gnn_decode_b200 import options
        options.set_option(name, value)
        self.touched.add(name)

    def unset(self, name):
        from gnn_decode_b200 import options
        options.unset_option(name)

    def restore(self):
        from gnn_decode_b200 import options
        for name in self.touched:
            options.unset_option(name)


@pytest.fixture
def gd_opt():
    o = _GdOptions()
    yield o
    o.restore()


@pytest.fixture
def one_cpu_thread():
    """Run the test's CPU arithmetic on one thread.  How torch's CPU matmuls and reductions split their rows over threads sets
    the order of floating-point sums, so the bit-exact comparisons with the golden fixtures hold at one thread, on a host with
    any number of cores, and not at every thread count (at 3, 5 or 7 threads some fixtures differ in the last bit)."""
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def logit_bound(ref, rtol=1e-4):
    """The parity bar on soft logits (BASELINE.json north_star: "within 1e-4 relative in fp32"): |got - ref| <= rtol * max(|ref|, 1),
    i.e. rtol relative for |logit| >= 1 and rtol ABSOLUTE below (a logit is a sum of fp32 terms of magnitude ~10-100, so its
    rounding error does not shrink with the logit; measured worst cases over the suite: 4e-5 absolute, 5e-5 relative on
    |logit| > 0.1 -- scripts/lean_check.py, profiles/r02_parity_envelope.txt).  Round 1 used a floor of 1e-4 (1 + rms) ~ 5e-3."""
    return rtol * ref.abs().clamp_min(1.0)


def logit_worst(got, ref, rtol=1e-4):
    """(max of |got - ref| / bound, max |got - ref|) in double on the CPU."""
    ref = ref.double().cpu()
    err = (got.double().cpu() - ref).abs()
    return (err / logit_bound(ref, rtol)).max().item(), err.max().item()


def golden_cases():
    return sorted(os.path.basename(f)[:-4] for f in glob.glob(os.path.join(GOLDEN, "*.npz"))
                  if not f.endswith("codes.npz") and not os.path.basename(f).startswith(("grad_", "ext_")))


class Golden(object):
    """One fixture produced by oracle/make_golden.py from the reference's own classes."""

    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN, name + ".npz"))
        self.name = name
        self.program = str(z["program"])
        self.V, self.C, self.E, self.B, self.T = (int(z[k]) for k in ("V", "C", "E", "B", "T"))
        self.dtype = getattr(torch, str(z["dtype"]))
        self.edge_index = torch.from_numpy(z["edge_index"])
        self.x = torch.from_numpy(z["x"])
        self.y = torch.from_numpy(z["y"])
        self.prob = torch.from_numpy(z["prob"])
        self.m0 = torch.from_numpy(z["m0"])
        self.phase_var = torch.from_numpy(z["phase_var"])
        self.phase_chk = torch.from_numpy(z["phase_chk"])
        self.weights = {k[2:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("w:")}
        self.logical = torch.from_numpy(z["logical"]) if "logical" in z.files else None
        self.H = torch.from_numpy(z["H"])

    def batched_edge_index(self):
        """data.edge_index as the PyG DataLoader would deliver it (check ids un-offset)."""
        N = self.V + self.C
        off = (torch.arange(self.B) * N).repeat_interleave(self.E)
        return self.edge_index.repeat(1, self.B) + off


@pytest.fixture(scope="session")
def codes_npz():
    return np.load(os.path.join(GOLDEN, "codes.npz"))


def make_decoder(g):
    """Instantiate the drop-in decoder matching a golden case and load its weights."""
    import importlib
    modname = {"v2_4": "quantum.decoder_v2_4", "qgnni": "quantum.QGNNI", "bp_quantum": "quantum.BP",
               "cgnni": "classical.CGNNI", "bp_classical": "classical.BP"}[g.program]
    mod = importlib.import_module("gnn_decode_b200." + modname)
    dec = mod.GNNI(g.T)
    if g.weights:
        dec.load_state_dict(g.weights, strict=True)
    return mod, dec

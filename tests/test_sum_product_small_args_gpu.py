"""Sum-product inference with small message arguments, on every kernel that runs it, against the fp64 oracle (oracle/restate.py).

Priors of magnitude 1e-4 .. 0.1 (p close to 0.5) keep every variable-to-check argument |a| below ~0.1 and many below 1e-3,
where log|tanh(a/2)| = log(1 - q) - log(1 + q), q = e^-|a|, cancels unless 1 - q is formed without subtraction
(gd_math.cuh, bp_one_minus_exp).  No message reaches a clamp (|a| >> 2e-20, |o| << 1 - eps2), so the learned programs' bar
applies: |got - ref| <= 1e-4 max(|ref|, 1) (conftest.logit_bound), not the saturated regime's 2e-3 / 5e-4.

The logits are a poor witness of that cancellation: tanh(a/2) itself is only off by ~1e-7 absolute, so the logits move by
~1e-7.  The check phase's output m = 2 atanh(o), o = prod tanh(a'/2) over the siblings, carries log|tanh|'s absolute error as
a relative one, so gd_propagate_fwd's check phase is held to 1e-4 of |m| itself on inputs down to |a| = 1e-4.

Kernels: the edge-owner kernel (a batch too small for the node-owner planner), the node-owner kernel (GD_FORCE_LIGHT on a
batch that fills the GPU), the TMA-staged streamed kernel (GD_FORCE_STREAMED, canonical edge order), the register-batched
streamed kernel (GD_FORCE_STREAMED on a permuted edge order; the sum-product programs only) and gd_propagate_fwd.  Which
kernel each case launches is read with torch.profiler in a child process (this file run as a script; profiler sessions early
in a pytest process make later sessions of other test files miss kernels) and asserted, so a planner change cannot move a case
to another kernel unnoticed."""
import json
import math
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

if __name__ == "__main__":
    _ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [_ROOT, os.path.join(_ROOT, "tests")]
from conftest import logit_worst  # noqa: E402
from gnn_decode_b200 import codes, options  # noqa: E402
from gnn_decode_b200.graph import TannerGraph  # noqa: E402
from oracle import restate  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
RTOL = 1e-4
KERNELS = {"edge_owner": (False, 300, None), "node_owner": (False, 4096, "GD_FORCE_LIGHT"),
           "streamed_tma": (False, 300, "GD_FORCE_STREAMED"), "streamed": (True, 300, "GD_FORCE_STREAMED")}
CASES = [(p, k) for p in ("bp_quantum", "bp_classical") for k in KERNELS] + \
        [("neural_bp", k) for k in ("edge_owner", "node_owner", "streamed_tma")] + [("v1_2_2", "edge_owner")]
# decode kernels by family (gd::<name>); a case must launch its own family's kernel and no other family's
FAMILY = {"decode_kernel": "edge_owner", "decode_light_kernel": "node_owner", "decode_light_ext_kernel": "node_owner",
          "decode_streamed_tma_kernel": "streamed_tma", "decode_streamed_kernel": "streamed", "lean_decode_kernel": "lean"}


def _small_priors(B, V, C, classical, seed):
    gen = torch.Generator().manual_seed(seed)
    mag = torch.exp(torch.empty((B, V), dtype=torch.float64).uniform_(np.log(1e-4), np.log(0.1), generator=gen))
    x = torch.zeros((B, V + C), dtype=torch.float64)
    x[:, :V] = mag * torch.where(torch.rand((B, V), generator=gen) < 0.5, -1.0, 1.0)
    if not classical:
        x[:, V:] = torch.where(torch.rand((B, C), generator=gen) < 0.3, -1.0, 1.0)
    return x.float()


def _decoder(program, T, E):
    from gnn_decode_b200.quantum import BP, decoder_v1_2_2, neural_BP
    from gnn_decode_b200.classical import BP as CBP
    torch.manual_seed(5)
    if program == "neural_bp":
        dec = neural_BP.GNNI(T, n_edges=E)
        with torch.no_grad():
            for n_, p_ in dec.named_parameters():
                p_.copy_(torch.full_like(p_, 0.25) if n_ == "alpha" else torch.rand_like(p_) * 0.6 + 0.6)
        return dec
    if program == "v1_2_2":
        dec = decoder_v1_2_2.GNNI(T)
        with torch.no_grad():                 # the variable-phase MLP's output is the check phase's argument: make it small
            dec.ggc1.mlp[2].weight.mul_(1e-2)
            dec.ggc1.mlp[2].bias.mul_(1e-2)
        return dec
    return {"bp_quantum": BP.GNNI, "bp_classical": CBP.GNNI}[program](T)


def _case(program, kernel):
    """(edge_index, V, C, T, graph, decoder, x, option) of one case."""
    permuted, B, opt = KERNELS[kernel]
    pcm = codes.toric_pcm(5)
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    if permuted:
        ei = ei[:, torch.from_numpy(np.random.RandomState(1).permutation(ei.size(1)))]
    C, V = pcm.shape
    T = 5
    x = _small_priors(B, V, C, program == "bp_classical", seed=B)
    dec = _decoder(program, T, ei.size(1)).to(DEV).eval()
    return ei, V, C, T, TannerGraph(ei, V, C, DEV), dec, x, opt


def _families(fn):
    """The decode-kernel families fn launches, read from one torch.profiler session."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    out = set()
    for ev in events:
        if ev.get("cat") == "kernel" and "gd::" in ev.get("name", ""):
            m = re.search(r"(\w+)\s*(?:<|\()", ev["name"].split("gd::", 1)[1])
            if m and m.group(1) in FAMILY:
                out.add(FAMILY[m.group(1)])
    return out


def _launched_main():
    out = {}
    for program, kernel in CASES:
        _, _, _, _, g, dec, x, opt = _case(program, kernel)
        xd = x.to(DEV)
        if opt:
            options.set_option(opt, 1)
        try:
            with torch.no_grad():
                out["%s-%s" % (program, kernel)] = sorted(_families(lambda: dec.decode(xd, graph=g, return_logits=True)))
        finally:
            if opt:
                options.unset_option(opt)
    print(json.dumps(out))


@pytest.fixture(scope="module")
def launched():
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("program,kernel", CASES)
def test_each_case_runs_its_kernel(program, kernel, launched):
    assert launched["%s-%s" % (program, kernel)] == [kernel]


@pytest.mark.parametrize("program,kernel", CASES)
def test_small_arguments_match_fp64(program, kernel, gd_opt):
    ei, V, C, T, g, dec, x, opt = _case(program, kernel)
    w = {k: v.detach().cpu() for k, v in dec.state_dict().items()}
    ref = restate.decode(program, ei, V, C, x.double(), w, T=T, dtype=torch.float64)["logit"]
    if opt:
        gd_opt.set(opt)
    with torch.no_grad():
        _, logit = dec.decode(x.to(DEV), graph=g, return_logits=True)
    worst, max_err = logit_worst(logit, ref, RTOL)
    print("%s %s: worst %.3g x bar, max abs err %.3g, max |logit| %.3g" % (program, kernel, worst, max_err, ref.abs().max()))
    assert worst <= 1.0, "%s %s: %.3g x bar (max abs err %.3g)" % (program, kernel, worst, max_err)


def _check_phase_fp64(m, x, ei, V, C, classical):
    """The sum-product check phase in fp64 with the output as 2 atanh(o): restate's log(1 + o) - log(1 - o) keeps only
    ~1e-16 / |o| of relative accuracy, 4e-4 at the smallest outputs here.  No clamp binds on these inputs."""
    mm = m.double()
    a = mm.abs()
    lt = torch.log(-torch.expm1(-a)) - torch.log1p(torch.exp(-a))                  # log|tanh(m/2)|
    neg = (mm < 0).double()
    chk = ei[1]
    S = torch.zeros((m.size(0), C), dtype=torch.float64).index_add_(1, chk, lt)[:, chk] - lt
    n = torch.zeros((m.size(0), C), dtype=torch.float64).index_add_(1, chk, neg)[:, chk] - neg
    if not classical:
        n = n + (1 - x[:, V:].double()[:, chk]) / 2
    return 2.0 * torch.atanh(torch.cos(math.pi * n) * torch.exp(S))


@pytest.mark.parametrize("program", ["bp_quantum", "bp_classical"])
def test_propagate_check_phase_small_arguments_relative(program):
    """gd_propagate_fwd's check phase on messages of magnitude 1e-4 .. 1: each output within 1e-4 of its own magnitude."""
    from gnn_decode_b200.quantum import BP
    from gnn_decode_b200.classical import BP as CBP
    pcm = codes.toric_pcm(5)
    ei = torch.from_numpy(codes.edge_index_of(pcm))
    C, V = pcm.shape
    E, B = ei.size(1), 64
    classical = program == "bp_classical"
    x = _small_priors(B, V, C, classical, seed=7)
    gen = torch.Generator().manual_seed(8)
    m = torch.exp(torch.empty((B, E), dtype=torch.float64).uniform_(np.log(1e-4), 0.0, generator=gen))
    m = (m * torch.where(torch.rand((B, E), generator=gen) < 0.5, -1.0, 1.0)).float()
    ref = _check_phase_fp64(m, x, ei, V, C, classical)
    oracle_ref = restate.propagate(program, "chk", ei, V, C, m.double(), x.double(), dtype=torch.float64)
    assert ((ref - oracle_ref).abs() <= 1e-12).all()             # the same function (restate loses ~1e-16 / |o| relative)
    dec = (CBP.GNNI(1) if classical else BP.GNNI(1)).to(DEV).eval()
    dec.bind_code(V, C)
    bei = restate.batched_edge_index(ei, V, C, B).to(DEV)        # check ids offset by V: what GNNI.forward hands to GraphConv
    with torch.no_grad():
        mf, xf = m.reshape(-1, 1).to(DEV), x.reshape(-1, 1).to(DEV)
        got = (dec.ggc2(mf, bei) if classical else dec.ggc2(mf, bei, xf)).reshape(B, E).double().cpu()
    rel = (got - ref).abs() / ref.abs()
    print("%s check phase: max relative error %.3g, min |m| %.3g" % (program, rel.max().item(), ref.abs().min().item()))
    assert ref.abs().min().item() < 1e-9                        # outputs far below fp32's 2^-24 next to 1 are in the sweep
    assert rel.max().item() <= RTOL


if __name__ == "__main__":
    _launched_main()

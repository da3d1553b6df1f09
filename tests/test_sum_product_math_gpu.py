"""The sum-product device primitives (gnn_decode_b200/csrc/gd_math.cuh, gd_nodemath.cuh) against fp64 (oracle/sp_math.py) at the
same fp32 arguments: log-spaced magnitudes from 1e-30 to 120 of both signs, +-0, and +-64 ulps around every branch point and
clamp.  Every sum-product kernel (edge-owner, node-owner, both streamed kernels, propagate, the neural BP backward) inlines
these functions, so an inaccuracy here is one in all of them.

A probe (tests/csrc/sp_math_probe.cu) evaluates each primitive elementwise exactly as the kernels inline it; it is compiled
once per module with the library's own nvcc and flags and loaded with ctypes, so the library's ABI carries no test hooks.

Bars:
  * values: |got - ref| <= 1e-6 max(|ref|, 1).  fp32 rounding and the MUFU approximations (ex2 / lg2 / rcp, each within a few
    1e-7 relative or absolute) put the worst of a correct evaluation at a few 1e-7 of the value, or of 1 below |value| = 1;
    what remains is headroom, not error that is allowed to grow.  A formula that cancels (1 - q at small |a| with q from
    ex2.approx) misses by orders of magnitude.
  * check outputs also relative to themselves (they are the next layer's messages, small ones included): 1e-6 |ref| plus
    2^-23 u |ref| for the fp32 rounding of the exponent -u log2 e.
  * derivatives: |got - ref| <= 1e-6 |ref| wherever ref is a normal fp32 number (1 / sinhf: libm's sinhf is within 2 ulp),
    and within FLT_MIN where ref is below the normal range (subnormal or past sinhf's overflow); arguments inside the clamp
    band (below) are left to the clamp checks.
  * clamp decisions: a derivative is 0 exactly where its forward value sits at its clamp, and the device decides a clamp as
    fp64 does wherever the fp64 value is off the clamp by more than CLAMP_BAND (relative): inside that band fp32 rounding of
    the argument decides, and the value there equals the clamp to within the value bar."""
import ctypes as ct
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from oracle import sp_math

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
PROBE_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "sp_math_probe.cu")
VALUE_BAR, DERIV_BAR, CLAMP_BAND = 1e-6, 1e-6, 1e-6
FN = {"log_abs_tanh_half_clamped": 0, "log_abs_tanh_half": 1, "nbp_t": 2, "one_minus_exp": 3, "check_out": 4, "dcheck_out": 5,
      "dlog_abs_tanh_half": 6}


class Probe(object):
    def __init__(self, path):
        self.lib = ct.CDLL(path)
        self.lib.sp_math_probe.restype = ct.c_int
        self.lib.sp_math_probe.argtypes = [ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_float, ct.c_int]

    def __call__(self, fn, a, param=0.0, odd=False):
        x = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(DEV)
        out = torch.empty_like(x)
        torch.cuda.synchronize()
        rc = self.lib.sp_math_probe(FN[fn], ct.c_void_p(x.data_ptr()), ct.c_void_p(out.data_ptr()), x.numel(), param, int(odd))
        assert rc == 0, "probe launch failed: cudaError %d" % rc
        torch.cuda.synchronize()
        return out.cpu().numpy().astype(np.float64)


def compile_probe(include_dir, out_dir):
    from gnn_decode_b200 import build
    so = os.path.join(out_dir, "sp_math_probe.so")
    cmd = [build._nvcc()] + build.NVCC_FLAGS + ["-I", include_dir, PROBE_SRC, "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, "nvcc failed:\n%s\n%s" % (" ".join(cmd), r.stdout + r.stderr)
    return Probe(so)


@pytest.fixture(scope="module")
def probe():
    from gnn_decode_b200 import build
    with tempfile.TemporaryDirectory() as d:
        yield compile_probe(build.CSRC, d)


def _value_check(what, a, got, ref):
    """Assert the value bar; print the worst err / bar and where it sits (the record of the measured envelope)."""
    assert np.isfinite(got).all(), "%s: non-finite at %s" % (what, a[~np.isfinite(got)][:8])
    ratio = np.abs(got - ref) / (VALUE_BAR * np.maximum(np.abs(ref), 1.0))
    i = int(np.argmax(ratio))
    print("%s: worst |got - ref| = %.3g x bar at %.9g (got %.9g, ref %.9g)" % (what, ratio[i], a[i], got[i], ref[i]))
    bad = ratio > 1.0
    assert not bad.any(), "%s: %d arguments off the bar, |a| in [%.3g, %.3g], worst %.3g x bar at %.9g" % (
        what, bad.sum(), np.abs(a[bad]).min(), np.abs(a[bad]).max(), ratio[i], a[i])


def _deriv_check(what, a, got, ref, skip):
    """skip: arguments inside the clamp band, where rounding decides the clamp (the clamp checks cover those)."""
    got, ref, a = got[~skip], ref[~skip], a[~skip]
    normal = np.abs(ref) >= sp_math.FLT_MIN
    assert np.isfinite(got).all(), "%s: non-finite at %s" % (what, a[~np.isfinite(got)][:8])
    ratio = np.where(normal, np.abs(got - ref) / (DERIV_BAR * np.where(normal, np.abs(ref), 1.0)), 0.0)
    i = int(np.argmax(ratio))
    print("%s: worst relative |got - ref| = %.3g x bar at %.9g (got %.9g, ref %.9g)" % (what, ratio[i], a[i], got[i], ref[i]))
    bad = ratio > 1.0
    assert not bad.any(), "%s: %d arguments off the bar, |a| in [%.3g, %.3g], worst %.3g x bar at %.9g" % (
        what, bad.sum(), np.abs(a[bad]).min(), np.abs(a[bad]).max(), ratio[i], a[i])
    tiny = ~normal & (np.abs(got - ref) > sp_math.FLT_MIN)
    assert not tiny.any(), "%s: below the normal range, off by more than FLT_MIN at %s" % (what, a[tiny][:8])


# ---- log|tanh(a/2)|, both input-clamp variants, both lower clamps -----------------------------------------------------------
@pytest.mark.parametrize("log_eps1", sp_math.LOG_EPS1)
@pytest.mark.parametrize("clamp_in", [True, False])
def test_log_abs_tanh_half(probe, clamp_in, log_eps1):
    a = sp_math.signed_sweep()
    got = probe("log_abs_tanh_half_clamped" if clamp_in else "log_abs_tanh_half", a, log_eps1)
    ref = sp_math.log_abs_tanh_half(a, log_eps1, clamp_in)
    _value_check("log|tanh(a/2)| clamp_in=%s log_eps1=%.6g" % (clamp_in, log_eps1), a, got, ref)
    assert (got >= log_eps1).all() and (got <= 0.0).all()
    # the lower clamp: decided as fp64 decides it away from the crossover
    raw = sp_math.log_abs_tanh_half_raw(a, clamp_in)
    far = np.abs(raw - log_eps1) > CLAMP_BAND * abs(log_eps1)
    assert np.array_equal((got == np.float32(log_eps1))[far], (raw <= log_eps1)[far])


# ---- neural BP's variable output: sign in the sign bit, never 0 -------------------------------------------------------------
def test_nbp_t(probe):
    a = sp_math.signed_sweep()
    got = probe("nbp_t", a)
    ref = sp_math.nbp_t(a)
    _value_check("nbp_t", a, got, ref)
    # > 0 exactly where u < 0 (-0 counts as non-negative), and |t| >= FLT_MIN everywhere: past |a| ~ 87 ex2 underflows and
    # log|tanh| would be 0, which carries no sign
    assert np.array_equal(np.signbit(got), ~(a < 0))
    assert (np.abs(got) >= sp_math.FLT_MIN).all()
    past = np.abs(a) > 87.0
    assert past.any() and (got[past & (a > 0)] <= -sp_math.FLT_MIN).all() and (got[past & (a < 0)] >= sp_math.FLT_MIN).all()


# ---- 1 - e^-u ---------------------------------------------------------------------------------------------------------------
def test_one_minus_exp(probe):
    u = sp_math.magnitudes()
    got = probe("one_minus_exp", u)
    ref = sp_math.one_minus_exp(u)
    _value_check("1 - e^-u", u, got, ref)
    # the log of it is taken (bp_check_out): below the series threshold it must be accurate relative to itself
    s = (u > 0) & (u < sp_math.SERIES)
    rel = np.abs(got[s] - ref[s]) / ref[s]
    print("1 - e^-u, u < %.3g: worst relative error %.3g" % (sp_math.SERIES, rel.max()))
    assert rel.max() <= VALUE_BAR


# ---- the check output and its derivative ------------------------------------------------------------------------------------
def _ext():
    return np.concatenate([-sp_math.magnitudes(), np.zeros(1, np.float32)]).astype(np.float32)   # ext <= 0, with -0 and +0


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("eps2", sp_math.EPS2)
def test_check_out(probe, eps2, odd):
    ext = _ext()
    got = probe("check_out", ext, eps2, odd)
    ref = sp_math.check_out(ext, odd, eps2)
    _value_check("check_out eps2=%.3g odd=%d" % (eps2, odd), ext, got, ref)
    assert np.array_equal(np.signbit(got), np.full(got.shape, odd))
    # m is the next layer's message and enters sums with terms of any size: it must keep its digits when it is small too.
    # Relative bar: VALUE_BAR, plus 2^-23 u for the rounding of the exponent -u log2 e to fp32 (2^-24 u relative in e^-u).
    # Past u ~ 87 ex2.approx.ftz returns 0 and so does m: within 2^-124 absolute there.
    u = -ext.astype(np.float64)
    rel_bar = VALUE_BAR + 2.0 ** -23 * u
    big = np.abs(ref) >= 2.0 ** -124
    ratio = np.abs(got - ref)[big] / (rel_bar[big] * np.abs(ref[big]))
    i = int(np.argmax(ratio))
    print("check_out eps2=%.3g odd=%d: worst relative |got - ref| = %.3g x bar at %.9g" % (eps2, odd, ratio[i], ext[big][i]))
    assert ratio[i] <= 1.0, "check_out: relative error %.3g x bar at ext = %.9g" % (ratio[i], ext[big][i])
    assert (np.abs(got - ref)[~big] <= 2.0 ** -124).all()


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("eps2", sp_math.EPS2)
def test_dcheck_out(probe, eps2, odd):
    ext = _ext()
    got = probe("dcheck_out", ext, eps2, odd)
    ref = sp_math.dcheck_out(ext, odd, eps2)
    one = sp_math.one_minus_exp(-ext.astype(np.float64))
    far = np.abs(one - eps2) > CLAMP_BAND * eps2
    _deriv_check("dcheck_out eps2=%.3g odd=%d" % (eps2, odd), ext, got, ref, ~far)
    # 0 exactly where the forward sits at its clamp: there its value is the one at ext = 0
    val = probe("check_out", ext, eps2, odd)
    at_clamp = np.abs(val - val[-1]) <= VALUE_BAR * abs(val[-1])
    overflow = -ext.astype(np.float64) > 89.0                     # 1 / sinhf(u) underflows to 0 there, unclamped
    assert (at_clamp | overflow)[got == 0.0].all()
    assert np.array_equal((got == 0.0)[far & ~overflow], sp_math.check_out_clamped(ext, eps2)[far & ~overflow])


@pytest.mark.parametrize("log_eps1", sp_math.LOG_EPS1)
def test_dlog_abs_tanh_half(probe, log_eps1):
    a = sp_math.signed_sweep()
    got = probe("dlog_abs_tanh_half", a, log_eps1)
    ref = sp_math.dlog_abs_tanh_half(a, log_eps1)
    raw = sp_math.log_abs_tanh_half_raw(a, False)
    far = np.abs(raw - log_eps1) > CLAMP_BAND * abs(log_eps1)
    _deriv_check("dlog|tanh(a/2)| log_eps1=%.6g" % log_eps1, a, got, ref, ~far)
    lv = probe("log_abs_tanh_half", a, log_eps1)
    overflow = np.abs(a.astype(np.float64)) > 89.0
    at_clamp = lv == np.float32(log_eps1)
    assert np.array_equal((got == 0.0)[~overflow], at_clamp[~overflow])
    assert np.array_equal((got == 0.0)[far & ~overflow], (raw <= log_eps1)[far & ~overflow])

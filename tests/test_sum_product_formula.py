"""The near branch of bp_log_abs_tanh_half (gnn_decode_b200/csrc/gd_math.cuh), restated in fp32 numpy, against fp64 over the
argument sweep of tests/test_sum_product_math_gpu.py (oracle/sp_math.py), at that file's value bar, 1e-6 max(|ref|, 1).

The MUFU approximations are drawn at their worst instead of emulated bit for bit: q = ex2.approx(-|a| log2 e) off by
+-2^-22 relative (the PTX ISA gives ex2.approx.f32 a maximum error of 2 ulp; relative to q in [0.5, 1) that is at most
2^-22), lg2.approx off by +-2^-22 absolute (the PTX ISA: 2^-22.6 absolute on the mantissa) and rcp.approx off by
+-2^-23 relative (1 ulp); every sign combination is evaluated and the worst is kept.  The other operations are IEEE fp32.

With 1 - q formed by subtraction, q's error is an absolute error of ~2.4e-7 in 1 - q, i.e. ~2.4e-7 / |a| in log|tanh(a/2)|:
the check must fail for that formula, and pass for the one the kernels use (1 - q from the series of bp_one_minus_exp
below |a| = 0.25).  This pins the algorithm without a GPU, as tests/test_tables.py pins the cubic tables."""
import itertools

import numpy as np
import pytest

from oracle import sp_math

VALUE_BAR = 1e-6
F = np.float32
LOG2E, LN2 = F(1.4426950408889634), F(0.6931471805599453)


def _fma(a, b, c):
    return (a.astype(np.float64) * b + c).astype(np.float32)


def _ex2(x, rel):
    """ex2.approx.ftz.f32 at its worst: 2^x (0 below the normal range) times (1 + rel)."""
    y = np.exp2(x.astype(np.float64))
    y = np.where(y < sp_math.FLT_MIN, 0.0, y)
    return (y * (1.0 + rel)).astype(np.float32)


def _lg2(x, err):
    with np.errstate(divide="ignore"):
        return (np.log2(np.where(x < sp_math.FLT_MIN, 0.0, x).astype(np.float64)) + err).astype(np.float32)


def _one_minus_exp(u, p, series):
    """bp_one_minus_exp: u (1 - u/2 + u^2/6 - u^3/24 + u^4/120 - u^5/720) below `series`, 1 - p above."""
    ser = _fma(u, F(-1.0 / 720.0), F(1.0 / 120.0))
    ser = _fma(-ser, u, F(1.0 / 24.0))
    ser = _fma(-ser, u, F(1.0 / 6.0))
    ser = _fma(-ser, u, F(0.5))
    ser = _fma(-ser, u, F(1.0))
    return np.where(u < F(series), u * ser, F(1.0) - p)


def log_abs_tanh_half_fp32(a, log_eps1, series, e_q, e_lg2, e_rcp):
    """bp_log_abs_tanh_half<false> in fp32, 1 - q from the series below |a| = series and by subtraction above."""
    aa = np.abs(a).astype(np.float32)
    q = _ex2(-aa * LOG2E, e_q)
    q2 = q * q
    ser = _fma(q2, F(1.0 / 9.0), F(1.0 / 7.0))
    ser = _fma(ser, q2, F(0.2))
    ser = _fma(ser, q2, F(1.0 / 3.0))
    ser = _fma(ser, q2, F(1.0))
    far = F(-2.0) * q * ser
    one_minus = _one_minus_exp(aa, q, series)
    rcp = (1.0 / (F(1.0) + q).astype(np.float64) * (1.0 + e_rcp)).astype(np.float32)
    near = LN2 * _lg2(one_minus * rcp, e_lg2)
    return np.maximum(np.where(aa < F(1.4), near, far), F(log_eps1))


def _worst(series, log_eps1):
    a = sp_math.magnitudes()
    ref = sp_math.log_abs_tanh_half(a, log_eps1, False)
    worst = np.zeros(a.shape)
    for e_q, e_lg2, e_rcp in itertools.product((-2.0 ** -22, 2.0 ** -22), (-2.0 ** -22, 2.0 ** -22), (-2.0 ** -23, 2.0 ** -23)):
        got = log_abs_tanh_half_fp32(a, log_eps1, series, e_q, e_lg2, e_rcp).astype(np.float64)
        worst = np.maximum(worst, np.abs(got - ref) / (VALUE_BAR * np.maximum(np.abs(ref), 1.0)))
    return a, worst


@pytest.mark.parametrize("log_eps1", sp_math.LOG_EPS1)
def test_near_branch_as_the_kernels_form_it_meets_the_value_bar(log_eps1):
    """1 - q from the series below |a| = 0.25: the subtraction above it loses at most q / (1 - q) 2^-22 <= 3.6 2^-22 relative."""
    a, worst = _worst(sp_math.SERIES, log_eps1)
    i = int(np.argmax(worst))
    print("series below %.3g: worst %.3g x bar at |a| = %.9g" % (sp_math.SERIES, worst[i], a[i]))
    assert worst[i] <= 1.0, "worst %.3g x bar at |a| = %.9g" % (worst[i], a[i])


@pytest.mark.parametrize("log_eps1", sp_math.LOG_EPS1)
def test_near_branch_by_subtraction_fails_the_value_bar(log_eps1):
    """1 - q by subtraction everywhere: off the bar by orders of magnitude at small |a| (~2.4e-7 / |a| absolute)."""
    a, worst = _worst(0.0, log_eps1)
    assert worst[(a > 1e-5) & (a < 1e-3)].min() > 10.0
    assert worst[(a > 1e-5) & (a < 1e-4)].min() > 100.0


@pytest.mark.parametrize("log_eps1", sp_math.LOG_EPS1)
def test_series_only_below_0_1_leaves_the_subtraction_off_the_bar(log_eps1):
    """Why the series reaches 0.25: handing over at 0.1 leaves q / (1 - q) ~ 9.5 on q's error just above it, and the worst case
    there is past the bar (the five-term series is accurate enough up to 0.1; the sixth term carries it to 0.25)."""
    a, worst = _worst(0.1, log_eps1)
    assert worst[(a >= 0.1) & (a < 0.11)].max() > 1.0
    assert worst[a < 0.1].max() <= 1.0

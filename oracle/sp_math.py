"""fp64 references of the sum-product device primitives (gnn_decode_b200/csrc/gd_math.cuh, gd_nodemath.cuh) and the fp32
argument sweep they are checked on: log-spaced magnitudes from 1e-30 to 120 of both signs, +-0, and +-64 ulps around every
point where a primitive changes branch or clamps.

Each reference takes the fp32 argument the device sees (as float64) and the fp32 values of the constants the kernels use, and
forms every difference that cancels with expm1 / log1p, so it is accurate to fp64 rounding at every argument."""
import numpy as np

FLT_MIN = float(np.finfo(np.float32).tiny)
LOG_EPS1 = (float(np.float32(-46.0517019)), float(np.float32(-16.1180957)))   # log 1e-20 (BP_QUANTUM, neural BP), log 1e-7
EPS2 = (float(np.float32(1e-15)), float(np.float32(1e-12)), float(np.float32(1e-7)))   # neural BP, BP_QUANTUM, BP_CLASSICAL
NEAR_FAR = 1.4            # bp_log_abs_tanh_half: near branch below, series in q = e^-|a| above
SERIES = 0.25             # bp_one_minus_exp: series below, 1 - e^-u above
CLAMP_IN = 10.0           # bp_log_abs_tanh_half<true>: |a| clamped to 10


def ulps_around(x, n=64):
    """The fp32 values within n ulps of fp32(x), both sides, x included."""
    i = np.array([x], dtype=np.float32).view(np.int32)[0]
    return (np.arange(-n, n + 1, dtype=np.int64) + int(i)).astype(np.int32).view(np.float32)


def branch_points():
    """Magnitudes where a primitive changes branch or clamps."""
    pts = [0.1, SERIES, NEAR_FAR, CLAMP_IN]                # 0.1: where a five-term series would hand over
    pts += [2.0 * np.exp(le) for le in LOG_EPS1]           # log|tanh(a/2)| = log eps1 at a ~ 2 eps1 (2e-20, 2e-7)
    pts += [126.0 * np.log(2.0), 128.0 * np.log(2.0)]      # ex2.approx.ftz: 2^-|a| log2 e leaves the normal range, then 0
    pts += [float(np.arcsinh(np.finfo(np.float32).max))]   # sinhf overflows: the derivatives become 0
    pts += list(EPS2)                                      # bp_check_out: 1 - e^-u = eps2
    pts += [float(-np.log1p(-e)) for e in EPS2]            # bp_check_out: e^-u = 1 - eps2
    return pts


def magnitudes():
    """Non-negative fp32 arguments: log-spaced 1e-30 .. 120, 0, and +-64 ulps around every branch point."""
    parts = [np.geomspace(1e-30, 120.0, 4001).astype(np.float32), np.zeros(1, np.float32)]
    parts += [ulps_around(p) for p in branch_points()]
    a = np.unique(np.concatenate(parts))
    return a[a >= 0]


def signed_sweep():
    """magnitudes() with both signs, -0 included."""
    m = magnitudes()
    return np.concatenate([m, -m]).astype(np.float32)


def one_minus_exp(u):
    """1 - e^-u."""
    return -np.expm1(-np.asarray(u, np.float64))


def log_abs_tanh_half_raw(a, clamp_in):
    """log|tanh(a/2)| = log(1 - q) - log(1 + q), q = e^-|a|, after the +-10 input clamp if clamp_in; -inf at 0."""
    aa = np.abs(np.asarray(a, np.float64))
    if clamp_in:
        aa = np.minimum(aa, CLAMP_IN)
    with np.errstate(divide="ignore"):
        return np.log(-np.expm1(-aa)) - np.log1p(np.exp(-aa))


def log_abs_tanh_half(a, log_eps1, clamp_in):
    return np.maximum(log_abs_tanh_half_raw(a, clamp_in), log_eps1)


def nbp_t(a, log_eps1=LOG_EPS1[0]):
    """Neural BP's variable output: log|tanh(a/2)| (no input clamp), at most -FLT_MIN, negated where a < 0."""
    a = np.asarray(a, np.float64)
    tv = np.minimum(log_abs_tanh_half(a, log_eps1, False), -FLT_MIN)
    return np.where(a < 0, -tv, tv)


def check_out(ext, odd, eps2):
    """log((1 + o) / (1 - o)), o = (-1)^odd e^ext with |o| clamped to 1 - eps2, ext <= 0 (u = -ext).  log(1 - p) is formed
    from 1 - p = -expm1(-u) up to u = 1 and as log1p(-p) beyond (where 1 - p rounds p's digits away once p < 1e-16)."""
    u = np.maximum(-np.asarray(ext, np.float64), 0.0)
    p = np.minimum(np.exp(-u), 1.0 - eps2)
    with np.errstate(divide="ignore"):
        log_one_minus = np.where(u > 1.0, np.log1p(-p), np.log(np.maximum(one_minus_exp(u), eps2)))
    mag = np.log1p(p) - log_one_minus
    return -mag if odd else mag


def check_out_clamped(ext, eps2):
    """Where check_out's clamp of |o| at 1 - eps2 binds."""
    return one_minus_exp(np.maximum(-np.asarray(ext, np.float64), 0.0)) < eps2


def dcheck_out(ext, odd, eps2):
    """d check_out / d ext = +-1 / sinh(u), 0 where the clamp binds."""
    u = np.maximum(-np.asarray(ext, np.float64), 0.0)
    with np.errstate(divide="ignore", over="ignore"):
        r = np.where(check_out_clamped(ext, eps2), 0.0, 1.0 / np.sinh(u))
    return -r if odd else r


def dlog_abs_tanh_half(a, log_eps1):
    """d/da log|tanh(a/2)| = 1 / sinh(a), 0 where the lower clamp binds."""
    a = np.asarray(a, np.float64)
    with np.errstate(divide="ignore", over="ignore"):
        return np.where(log_abs_tanh_half_raw(a, False) <= log_eps1, 0.0, 1.0 / np.sinh(a))

"""CPU model of the weight gradient of a 1 -> h -> 1 ReLU MLP taken through per-segment bins, as the CGNNI backward kernel
(gnn_decode_b200/csrc/gd_backward_light.cu) takes it.

f(x) = b2 + sum_u c_u relu(a_u x + b_u) is one line between two consecutive breakpoints t_u = -b_u / a_u, with a fixed set of
active units.  For a loss sum_i g_i f(x_i), the gradient w.r.t. (a, b, c, b2) is therefore fixed by Sg_j = sum g_i and
Sgx_j = sum g_i x_i over the items x_i of segment j:
    dW1_u = c_u sum_{j active} Sgx_j,  db1_u = c_u sum_{j active} Sg_j,  dW2_u = sum_{j active} (a_u Sgx_j + b_u Sg_j),  db2 = sum_j Sg_j.
Breakpoints, their order and the active sets follow pwl_build (csrc/gd_math.cuh): breakpoints rounded to fp32, ties ordered by
unit index, a unit with a_u = 0 active everywhere iff b_u > 0; segment j of x = the number of breakpoints < x."""
import numpy as np


def breakpoints(w1, b1):
    """fp32 breakpoints -b/a (+inf where a == 0) and each unit's rank in the sorted list."""
    a, b = np.asarray(w1, np.float64).reshape(-1), np.asarray(b1, np.float64).reshape(-1)
    h = a.size
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(a != 0, (-b / np.where(a != 0, a, 1.0)).astype(np.float32), np.float32(np.inf)).astype(np.float32)
    rank = np.array([sum(1 for v in range(h) if t[v] < t[u] or (t[v] == t[u] and v < u)) for u in range(h)])
    return t, rank


def segments(w1, b1, x):
    """Segment index of every fp32 input x."""
    t, _ = breakpoints(w1, b1)
    x32 = np.asarray(x, np.float32).reshape(-1)
    return (t[None, :] < x32[:, None]).sum(1)


def bins(w1, b1, x, g, npad=16):
    """(Sg, Sgx) per segment, in float64."""
    j = segments(w1, b1, x)
    x64, g64 = np.asarray(x, np.float64).reshape(-1), np.asarray(g, np.float64).reshape(-1)
    return np.bincount(j, g64, npad), np.bincount(j, g64 * x64, npad)


def contract(w1, b1, w2, Sg, Sgx):
    """The bins -> weight-gradient contraction.  Returns (dW1 [h], db1 [h], dW2 [h], db2)."""
    a, b = np.asarray(w1, np.float64).reshape(-1), np.asarray(b1, np.float64).reshape(-1)
    c = np.asarray(w2, np.float64).reshape(-1)
    _, rank = breakpoints(w1, b1)
    j = np.arange(len(Sg))
    dW1, db1, dW2 = np.zeros_like(a), np.zeros_like(a), np.zeros_like(a)
    for u in range(a.size):
        if a[u] == 0:
            act = np.full(j.shape, b[u] > 0)
        else:
            act = rank[u] < j if a[u] > 0 else rank[u] >= j
        G, GX = Sg[act].sum(), Sgx[act].sum()
        dW1[u], db1[u], dW2[u] = c[u] * GX, c[u] * G, a[u] * GX + b[u] * G
    return dW1, db1, dW2, Sg.sum()

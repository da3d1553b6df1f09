"""fp64 restatement of the neural BP training backward (gnn_decode_b200/csrc/gd_backward_nbp.cu): the hand-derived recurrence
that kernel implements, written out on [B, E] tensors, so that it can be pinned against torch autograd through
oracle/restate.py::_forward_neural_bp on the CPU.

Forward (quantum/neural_BP.py GNNI.forward), per syndrome, layer l, edge e = (v, c), s_c the check input, pi_v the prior:
    q_e = W_l[e] m^l_e,   u_e = sum_{e' in v, e' != e} q_e' + W_p,l[e] pi_v,
    a_e = tanh(u_e / 2),  L_e = log clamp(|a_e|, 1e-20, 1e10),  n_e = [a_e < 0],
    S_e = sum_{e' in c, e' != e} L_e',  sigma_e = cos(pi (sum_{e' in c, e' != e} n_e' + (1 - s_c) / 2)),
    o_e = clamp(sigma_e exp(S_e), -1 + 1e-15, 1 - 1e-15),  m^{l+1}_e = log(1 + o_e) - log(1 - o_e) + alpha m^l_e,
    logit_v = sum_{e in v} (W[e] m^T_e + W_p[e] pi_v).
Backward, g = dL/dm^{l+1}, l = T-1 .. 0, from g_e = dlogit_v W[e]:
    dW[e] = sum_b dlogit_v m^T_e,  dW_p[e] = sum_b dlogit_v pi_v,
    dalpha += sum_b sum_e g_e m^l_e,
    dS_e = g_e sigma_e / sinh(-S_e) where the o-clamp does not bind, else 0,   dL_e = sum_{e' in c, e' != e} dS_e',
    du_e = dL_e / sinh(u_e) where |a_e| >= 1e-20, else 0,   dW_p,l[e] += sum_b du_e pi_v,
    dq_e = sum_{e' in v, e' != e} du_e',  dW_l[e] += sum_b dq_e m^l_e,  g_e <- alpha g_e + W_l[e] dq_e.
The sign count sigma carries no gradient.

Everything is evaluated so that fp64 keeps the digits of saturated messages that torch's op sequence loses:
  * log|tanh(u/2)| as log1p(-q) - log1p(q), q = e^-|u| (tanh(u/2), and 1 - q, round to 1 and lose q's digits past |u| ~ 20);
  * 1 -+ o from S with expm1 (exp(S) rounds to 1 when S ~ -1e-14, and 1 - o then keeps two digits);
  * every "sum over the node's other edges" (S, dL, u, dq) as prefix + suffix sums, never the node's total minus the edge's own
    term: a saturated message's log|tanh| (down to -46) or a near-clamp edge's dS (up to ~1e15 g) would swamp its siblings'
    terms in the total, and those terms are what the difference is.
In the unsaturated range this is the same function to rounding."""
import math

import torch

EPS1, EPS2 = 1e-20, 1e-15


def _excl(val, idx, n):
    """sum over the OTHER edges of the same node (idx: the node of every edge): [B, E] -> [B, E], as the sum of the edges before
    it plus the sum of the edges after it in a dense [B, n, max degree] layout (no subtraction)."""
    E = idx.numel()
    order = torch.argsort(idx, stable=True)
    deg = torch.bincount(idx, minlength=n)
    start = torch.cumsum(deg, 0) - deg
    pos = torch.empty(E, dtype=torch.long)
    pos[order] = torch.arange(E) - start[idx[order]]
    D = max(int(deg.max()), 1)
    dense = torch.zeros((val.size(0), n, D), dtype=val.dtype)
    dense[:, idx, pos] = val
    zero = torch.zeros((val.size(0), n, 1), dtype=val.dtype)
    before = torch.cat([zero, torch.cumsum(dense, 2)[:, :, :-1]], 2)
    after = torch.cat([torch.cumsum(dense.flip(2), 2).flip(2)[:, :, 1:], zero], 2)
    return (before + after)[:, idx, pos]


def grads(edge_index, V, C, x, w, T, dlogit, info=None):
    """edge_index [2, E] (variable, check), x [B, V+C] (prior | check sign), w: neural BP state dict (layers.{2l}.W / W_p
    [E, 1], W, W_p [E, 1], alpha [1, 1]), dlogit [B, V].  Returns (logit [B, V], {name: dL/dname}) in float64.
    info (a dict, optional) receives max |u|, how many (syndrome, edge, layer) items the o-clamp bound, and how many have
    1e-20 < |u| < 1e-3 (small messages off the log clamp, where log|tanh(u/2)| is hardest to form in fp32)."""
    ev, ec = edge_index[0].long(), edge_index[1].long()
    x = x.double()
    B = x.size(0)
    pi = x[:, :V][:, ev]                                  # [B, E] prior of each edge's variable
    s = x[:, V:][:, ec]                                   # [B, E] sign of each edge's check
    W = {k: v.double().reshape(-1) for k, v in w.items()}
    alpha = float(W["alpha"][0])
    E = ev.numel()
    m = torch.zeros((B, E), dtype=torch.float64)
    saved = []
    for l in range(T):
        Wl, Wpl = W["layers.%d.W" % (2 * l)], W["layers.%d.W_p" % (2 * l)]
        u = _excl(Wl * m, ev, V) + Wpl * pi
        q = torch.exp(-u.abs())
        log_abs_a = torch.log1p(-q) - torch.log1p(q)                           # log|tanh(u/2)|
        pass_l = log_abs_a >= math.log(EPS1)
        L = torch.where(pass_l, log_abs_a, torch.full_like(u, math.log(EPS1)))
        S = _excl(L, ec, C)
        cnt = _excl((u < 0).double(), ec, C)
        sigma = torch.cos(math.pi * (cnt + (1 - s) / 2))
        one_minus = -torch.expm1(S)                                            # 1 - |o| before the clamp
        pass_o = one_minus >= EPS2
        mag = torch.where(pass_o, torch.log1p(torch.exp(S)) - torch.log(one_minus.clamp_min(EPS2)),
                          torch.full_like(S, math.log((2 - EPS2) / EPS2)))
        if info is not None:
            info["max_abs_u"] = max(info.get("max_abs_u", 0.0), u.abs().max().item())
            info["o_clamped"] = info.get("o_clamped", 0) + int((~pass_o).sum())
            info["small_u"] = info.get("small_u", 0) + int(((u.abs() < 1e-3) & (u.abs() > 1e-20)).sum())
        saved.append((m, u, pass_l, S, sigma, pass_o))
        m = sigma * mag + alpha * m
    logit = torch.zeros((B, V), dtype=torch.float64).index_add_(1, ev, W["W"] * m + W["W_p"] * pi)
    dl = dlogit.double()[:, ev]                           # [B, E] dL/dlogit of each edge's variable
    out = {"W": (dl * m).sum(0), "W_p": (dl * pi).sum(0)}
    g = dl * W["W"]
    dalpha = 0.0
    zero = torch.zeros((), dtype=torch.float64)
    for l in range(T - 1, -1, -1):
        ml, u, pass_l, S, sigma, pass_o = saved[l]
        dalpha += float((g * ml).sum())
        dS = torch.where(pass_o, g * sigma / torch.sinh(-S), zero)
        dL = _excl(dS, ec, C)
        du = torch.where(pass_l, dL / torch.sinh(u), zero)
        out["layers.%d.W_p" % (2 * l)] = (du * pi).sum(0)
        dq = _excl(du, ev, V)
        Wl = W["layers.%d.W" % (2 * l)]
        out["layers.%d.W" % (2 * l)] = (dq * ml).sum(0)
        g = alpha * g + Wl * dq
    out["alpha"] = torch.tensor([dalpha], dtype=torch.float64)
    return logit, {k: v.reshape(w[k].shape) for k, v in out.items()}

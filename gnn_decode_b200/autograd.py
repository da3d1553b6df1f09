"""Training path: torch.autograd.Function around the hand-written forward-with-stash and backward
kernels (gd_decode_fwd_train / gd_decode_bwd) of decoder_v2_4, CGNNI and neural BP (quantum/neural_BP.py,
and decoder_v1_1, whose per-edge weights are gathered from its type tables).  Gradients flow to the
decoder's parameters (the reference never differentiates w.r.t. its inputs).  Neural BP trains on the
TMA-staged streamed kernel on every code; a graph outside the canonical edge order (H.to_sparse()) is
refused with GdError."""
import ctypes as ct

import torch

from . import _cabi


def _ptr(t):
    return ct.c_void_p(t.data_ptr()) if t is not None else None


class _DecodeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, decoder, graph, x32, *params):
        lib = _cabi.lib()
        dev = x32.device
        B = x32.size(0)
        model = decoder.gd_model()
        with torch.no_grad():
            w = torch.cat([p.detach().reshape(-1).to(torch.float32) for p in params]).contiguous()
        n_stash = lib.gd_stash_floats(graph.handle, ct.byref(model), B)
        if n_stash < 0:
            _cabi.check(_cabi.GD_ERR_INVALID, "gd_stash_floats")
        stash = torch.empty(max(n_stash, 1), dtype=torch.float32, device=dev)
        prob = torch.empty((B, graph.V), dtype=torch.float32, device=dev)
        logit = torch.empty((B, graph.V), dtype=torch.float32, device=dev)
        st = ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        with torch.cuda.device(dev):
            _cabi.check(lib.gd_decode_fwd_train(graph.handle, ct.byref(model), _ptr(w), _ptr(x32), _ptr(prob),
                                                _ptr(logit), _ptr(stash), B, st), "gd_decode_fwd_train")
        ctx.decoder, ctx.graph, ctx.model = decoder, graph, model
        ctx.save_for_backward(x32, w, stash, prob, logit)
        ctx.shapes = [(p.shape, p.dtype) for p in params]
        ctx.mark_non_differentiable(logit)
        return prob, logit

    @staticmethod
    def backward(ctx, grad_prob, _grad_logit_unused):
        lib = _cabi.lib()
        x32, w, stash, prob, logit = ctx.saved_tensors
        graph, model = ctx.graph, ctx.model
        dev = x32.device
        B = x32.size(0)
        g = grad_prob.to(torch.float32)
        if model.program == _cabi.PROG_CGNNI:
            # prob = clamp(s, 1e-7, 1 - 1e-7), s = sigmoid(-logit) (CGNNI.py:282): torch.clamp's gradient mask is inclusive,
            # so clamped outputs pass nothing; dL/dlogit = -dL/dprob * s * (1 - s) on the rest
            s = torch.sigmoid(-logit)
            grad_logit = torch.where((s >= 1e-7) & (s <= 1.0 - 1e-7), -g * s * (1.0 - s), torch.zeros_like(s)).contiguous()
        else:
            # prob = sigmoid(-logit) (decoder_v2_4, neural BP: no clamp)  ->  dL/dlogit = -dL/dprob * prob * (1 - prob)
            grad_logit = (-g * prob * (1.0 - prob)).contiguous()
        n_ws = lib.gd_bwd_workspace_floats(graph.handle, ct.byref(model), B)
        if n_ws < 0:
            _cabi.check(_cabi.GD_ERR_UNSUPPORTED, "gd_bwd_workspace_floats")
        ws = torch.empty(n_ws, dtype=torch.float32, device=dev)
        gw = torch.empty(w.numel(), dtype=torch.float32, device=dev)
        st = ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        with torch.cuda.device(dev):
            _cabi.check(lib.gd_decode_bwd(graph.handle, ct.byref(model), _ptr(w), _ptr(x32), _ptr(stash), _ptr(grad_logit),
                                          _ptr(gw), _ptr(ws), 0, B, st), "gd_decode_bwd")
        grads, off = [], 0
        for shape, dtype in ctx.shapes:
            n = 1
            for d in shape:
                n *= d
            grads.append(gw[off:off + n].view(shape).to(dtype))
            off += n
        return (None, None, None) + tuple(grads)


def decode_with_grad(decoder, graph, x, return_logits=False, return_hard=False):
    if decoder._gd_program not in (_cabi.PROG_V2_4, _cabi.PROG_CGNNI, _cabi.PROG_NEURAL_BP):
        raise _cabi.GdError("training (backward) kernels exist for the decoder_v2_4, CGNNI and neural BP programs only; "
                            "call .eval() or wrap inference in torch.no_grad()")
    x32 = x.detach().to(torch.float32).contiguous()
    if x32.data_ptr() % 16:
        x32 = x32.clone()
    prob, logit = _DecodeFn.apply(decoder, graph, x32, *decoder._gd_params())
    out = [prob]
    if return_logits:
        out.append(logit)
    if return_hard:
        out.append((prob.detach() > 0.5).to(torch.uint8))
    return out[0] if len(out) == 1 else tuple(out)

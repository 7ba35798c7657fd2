"""Tensor-level wrappers and torch.autograd.Functions over the C ABI (include/acr_b200.h).

PyTorch is used here for device memory, streams and autograd bookkeeping only; every computation
below is one of the hand-written sm_100a kernels in acr_wsss_b200/csrc.  No CPU fallback exists:
CPU tensors raise.
"""
import ctypes

import numpy as np
import torch

from . import _lib

_GETAM_FUNCS = {"grad": 0, "grad_s": 1, "cam_grad": 2, "cam_grad_s": 3}


class _Profile:
    """Optional per-entry-point timing (CUDA events on the launching stream) and launch counting.
    Off by default; bench.py switches it on for the timed region."""

    def __init__(self):
        self.reset(False)

    def reset(self, enabled=False):
        self.enabled = enabled
        self.events = {}     # name -> list of (start, end)
        self.launches = 0

    def summary(self):
        torch.cuda.synchronize()
        kernels = {}
        for name, evs in self.events.items():
            kernels[name] = {"name": name, "calls": len(evs), "ms": sum(a.elapsed_time(b) for a, b in evs)}
        return {"launches": self.launches, "kernels": kernels}


PROFILE = _Profile()

# Direct accumulation into preallocated fp32 .grad buffers (weight gradients by the GEMM itself, bias / LayerNorm gradients by
# this repo's kernels) is an optimisation of the TRAINING step only: Trainer switches it on around its forward+backward.
# Everything else (CAM inference on a Trainer-attached model, autograd.grad for activations, user code) gets ordinary
# autograd-returned gradients, whatever the parameters' .grad happen to hold.
DIRECT_GRADS = False


class direct_grads:
    """Context manager: with ops.direct_grads(): loss = ...; loss.backward()"""

    def __enter__(self):
        global DIRECT_GRADS
        self.prev, DIRECT_GRADS = DIRECT_GRADS, True

    def __exit__(self, *exc):
        global DIRECT_GRADS
        DIRECT_GRADS = self.prev


def _call(name, nlaunch, *args):
    """Invoke C-ABI entry `name`; raises on failure.  `nlaunch` = kernels this call launches (for gpu_launches)."""
    fn = getattr(_lib.lib(), name)
    if PROFILE.enabled:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = fn(*args)
        b.record()
        PROFILE.events.setdefault(name, []).append((a, b))
        PROFILE.launches += nlaunch
    else:
        rc = fn(*args)
    _lib.check(rc, name)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("acr_wsss_b200 ops need CUDA tensors: there is no CPU fallback")


def _alias(t):
    """A fresh (non-view) tensor sharing t's memory, so autograd treats it as a new output."""
    return torch.empty(0, device=t.device, dtype=t.dtype).set_(t.untyped_storage(), t.storage_offset(), t.shape, t.stride())


def _dense_map(t):
    """A [B,N,N] map with dense rows; returns (tensor, batch_stride_in_elements)."""
    if t.stride(-1) != 1 or t.stride(-2) != t.shape[-1]:
        t = t.contiguous()
    return t, t.stride(0)


def _strided_map(t):
    """A [B,N,N] map with unit column stride (rows may be padded); returns (tensor, batch stride, row stride)."""
    if t.stride(-1) != 1:
        t = t.contiguous()
    return t, t.stride(0), t.stride(1)


# ----------------------------------------------------------------------------------------------
# (a1) attention core
# ----------------------------------------------------------------------------------------------
class _AttnCoreF32(torch.autograd.Function):
    """softmax(QK^T*scale) V with materialised P (reference data flow, vision_transformer.py:198-214)."""

    @staticmethod
    def forward(ctx, qkv, num_heads, scale, mean_slot, state):
        _need_cuda(qkv)
        B, N, E3 = qkv.shape
        E = E3 // 3
        D = E // num_heads
        qkv = qkv.contiguous().float()
        P = torch.empty(B, num_heads, N, N, device=qkv.device, dtype=torch.float32)
        out = torch.empty(B, N, E, device=qkv.device, dtype=torch.float32)
        if mean_slot is None:
            mean_slot = torch.empty(B, N, N, device=qkv.device, dtype=torch.float32)
        assert mean_slot.stride(-1) == 1 and mean_slot.stride(-2) == N
        _call("acr_attn_fwd_f32", 4, _p(qkv), B, N, num_heads, D, scale, _p(P), _p(out),
                                               _p(mean_slot), mean_slot.stride(0), _stream())
        ctx.save_for_backward(qkv, P)
        ctx.dims = (B, N, num_heads, D, scale)
        ctx.state = state
        if state is not None:
            state["attn"] = P
            state["row0"] = None
        ctx.set_materialize_grads(False)
        return out, _alias(mean_slot)

    @staticmethod
    def backward(ctx, d_out, g_mean):
        qkv, P = ctx.saved_tensors
        B, N, H, D, scale = ctx.dims
        d_out = torch.zeros(B, N, H * D, device=qkv.device) if d_out is None else d_out.contiguous().float()
        gs = 0
        if g_mean is not None:
            g_mean, gs = _dense_map(g_mean.float())
        dP = torch.empty_like(P)
        dS = torch.empty_like(P)
        d_qkv = torch.empty_like(qkv)
        _call("acr_attn_bwd_f32", 5, _p(qkv), _p(P), _p(d_out), B, N, H, D, scale,
                                               _p(g_mean), gs, _p(dP), _p(dS), _p(d_qkv), _stream())
        if ctx.state is not None and ctx.state.get("capture_grad", True):
            ctx.state["attn_grad"] = dP          # what save_attn_gradients keeps (vision_transformer.py:192-193)
        return d_qkv, None, None, None, None


class _AttnCoreBF16(torch.autograd.Function):
    """Fused tcgen05 path: bf16 operands, fp32 accumulate, P never written to HBM."""

    @staticmethod
    def forward(ctx, qkv, num_heads, scale, mean_slot, state):
        _need_cuda(qkv)
        B, N, E3 = qkv.shape
        E = E3 // 3
        D = E // num_heads
        qkv = qkv.contiguous().to(torch.bfloat16)
        out = torch.empty(B, N, E, device=qkv.device, dtype=torch.bfloat16)
        lse = torch.empty(B, num_heads, N, device=qkv.device, dtype=torch.float32)
        p_row0 = torch.empty(B, num_heads, N, device=qkv.device, dtype=torch.float32) if state is not None else None
        if mean_slot is None:
            mean_slot = torch.empty(B, N, N, device=qkv.device, dtype=torch.float32)
        assert mean_slot.stride(-1) == 1 and mean_slot.stride(-2) == N
        _call("acr_attn_fwd_bf16", 2, _p(qkv), B, N, num_heads, D, scale, _p(out), _p(lse),
                                                _p(mean_slot), mean_slot.stride(0), _p(p_row0), _stream())
        ctx.save_for_backward(qkv, out, lse)
        ctx.dims = (B, N, num_heads, D, scale)
        ctx.state = state
        if state is not None:
            state["attn"] = None
            state["row0"] = p_row0
            state["qkv"] = qkv
            state["fused"] = True       # lets consistency_loss hand its gradient over as sign codes
        ctx.set_materialize_grads(False)
        return out, _alias(mean_slot)

    @staticmethod
    def backward(ctx, d_out, g_mean):
        qkv, out, lse = ctx.saved_tensors
        B, N, H, D, scale = ctx.dims
        d_out = (torch.zeros(B, N, H * D, device=qkv.device, dtype=torch.bfloat16) if d_out is None
                 else d_out.contiguous().to(torch.bfloat16))
        gs, gl = 0, 0
        code, cbs, cld, w_cls, w_aff, g_scale = None, 0, 0, 0.0, 0.0, None
        if ctx.state is not None and ctx.state.get("g_code") is not None:
            # always consumed (popped), whatever else arrives: a stale slice must never leak into a later backward
            code = ctx.state.pop("g_code")                      # [B,N,ld] uint8 view of the [B,L,N,ld] code tensor
            w_cls, w_aff = ctx.state.pop("g_w")
            g_scale = ctx.state.pop("g_scale")
            if g_mean is not None:
                # a dense gradient reached the same stack through autograd (an extra loss on attn1 / attn2): the kernel takes
                # ONE form of G, so the codes are decoded into the dense map (rare path, one elementwise pass)
                g_mean = g_mean.float() + decode_sign_codes(code, N, w_cls, w_aff, g_scale)
                code, w_cls, w_aff, g_scale = None, 0.0, 0.0, None
            else:
                cbs, cld = code.stride(0), code.stride(1)
        if g_mean is not None:
            g_mean, gs, gl = _strided_map(g_mean.float())
        d_qkv = torch.empty_like(qkv)
        want_row0 = ctx.state is not None and ctx.state.get("capture_grad", True)
        g_row0 = torch.empty(B, H, N, device=qkv.device, dtype=torch.float32) if want_row0 else None
        wsb = _lib.lib().acr_attn_bwd_bf16_workspace(B, N, H, D)
        ws = torch.empty(wsb, device=qkv.device, dtype=torch.uint8)
        _call("acr_attn_bwd_bf16", 4, _p(qkv), _p(out), _p(lse), _p(d_out), B, N, H, D, scale,
              _p(g_mean), gs, gl, _p(code), cbs, cld, w_cls, w_aff, _p(g_scale),
              _p(d_qkv), _p(g_row0), _p(ws), wsb, _stream())
        if want_row0:
            ctx.state["grad_row0"] = g_row0
            # what Attention.get_attn_gradients() needs to rebuild the full dP on demand (accessor protocol; 2 B x N x E bytes)
            ctx.state["d_out"] = d_out
            ctx.state["g_dense"] = (g_mean if g_mean is not None else
                                    (decode_sign_codes(code, N, w_cls, w_aff, g_scale) if code is not None else None))
        return d_qkv, None, None, None, None


def decode_sign_codes(code, N, w_cls, w_aff, g_scale=None):
    """Sign codes [B,N,ld] (0x00 / 0x3F / 0xBF) -> the dense gradient they stand for, [B,N,N] fp32: +-w (w_cls on the cls row,
    w_aff elsewhere), times the upstream scalar."""
    c = code[..., :N]
    g = (c == 0x3F).float() - (c == 0xBF).float()
    w = torch.full((N, 1), float(w_aff), device=code.device)
    w[0, 0] = float(w_cls)
    g = g * w
    return g * g_scale.reshape(()) if g_scale is not None else g


def attention_core(qkv, num_heads, scale, mean_slot=None, state=None, precision="fp32"):
    """qkv [B,N,3E] (output of the qkv Linear) -> (out [B,N,E], head-mean attention [B,N,N] fp32).

    `mean_slot`, when given, is the [B,N,N] view of slot l of a preallocated [B,L,N,N] stack; the
    kernel writes into it directly and the returned map aliases it (no stack copy).
    """
    fn = _AttnCoreBF16 if precision == "bf16" else _AttnCoreF32
    return fn.apply(qkv, num_heads, float(scale), mean_slot, state)


class _StackViews(torch.autograd.Function):
    """Zero-copy replacement for torch.stack(attn_list, dim=1) (DPT/ACR.py:112): the per-block maps
    already live in the slots of `stack`; backward hands each block its slice of the incoming gradient."""

    @staticmethod
    def forward(ctx, stack, *maps):
        ctx.n = len(maps)
        ctx.set_materialize_grads(False)
        return _alias(stack)

    @staticmethod
    def backward(ctx, g):
        if g is None:
            return (None,) * (ctx.n + 1)
        return (None,) + tuple(g[:, l] for l in range(ctx.n))


class _StackViewsSplit(torch.autograd.Function):
    """stack_views for a batch that holds the two views back to back ([2B,L,N,N]): returns the two halves as separate
    autograd outputs (attn1, attn2), still without copying the stack."""

    @staticmethod
    def forward(ctx, stack, *maps):
        ctx.n = len(maps)
        ctx.set_materialize_grads(False)
        B = stack.shape[0] // 2
        return _alias(stack[:B]), _alias(stack[B:])

    @staticmethod
    def backward(ctx, g1, g2):
        if g1 is None and g2 is None:
            return (None,) * (ctx.n + 1)
        # dense-gradient fallback (e.g. the reference's inline loss): one concatenation per step
        if g1 is None:
            g1 = torch.zeros_like(g2)
        if g2 is None:
            g2 = torch.zeros_like(g1)
        g = torch.cat([g1, g2], dim=0)
        return (None,) + tuple(g[:, l] for l in range(ctx.n))


def stack_views_split(stack, maps, states=None):
    a1, a2 = _StackViewsSplit.apply(stack, *maps)
    if states is not None:
        a1._acr_states = a2._acr_states = list(states)
        a1._acr_half, a2._acr_half = 0, 1
    return a1, a2


def stack_views(stack, maps, states=None):
    out = _StackViews.apply(stack, *maps)
    if states is not None:
        out._acr_states = list(states)      # per-block state dicts of the forward pass that produced this stack
    return out


# ----------------------------------------------------------------------------------------------
# Linear with a cached bf16 copy of the fp32 master weight (library GEMM; only the cast / accumulate traffic changes)
# ----------------------------------------------------------------------------------------------
class _LinearCachedBF16(torch.autograd.Function):
    """y = x W^T + b with bf16 operands taken from a persistent bf16 copy of the master weights (refreshed once per
    optimiser step) instead of autocast's per-call casts; the weight / bias gradients are accumulated straight into the
    fp32 .grad buffers (one mixed-precision add instead of cast + add).  The GEMMs themselves stay cuBLAS."""

    @staticmethod
    def forward(ctx, x, weight, bias, w16, b16, skip_bias_grad=False):
        x2 = x.reshape(-1, x.shape[-1])
        y = torch.nn.functional.linear(x2, w16, b16)      # (torch.addmm with a 1-D bf16 bias takes a 60x slower path)
        ctx.save_for_backward(x2, w16)
        ctx.params = (weight, None if skip_bias_grad else bias)      # skipped: add_layer_norm's backward owns the bias gradient
        ctx.in_shape = x.shape
        return y.view(*x.shape[:-1], w16.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, w16 = ctx.saved_tensors
        weight, bias = ctx.params
        dy2 = dy.reshape(-1, dy.shape[-1])
        dx = (dy2 @ w16).view(ctx.in_shape) if ctx.needs_input_grad[0] else None
        gw = gb = None
        if not ctx.needs_input_grad[1]:
            pass                                    # e.g. the truncated GETAM backward: only the activations' gradient is wanted
        elif DIRECT_GRADS and weight.grad is not None and weight.grad.dtype == torch.float32 and dy2.is_cuda and dy2.dtype == torch.bfloat16:
            # dW accumulated by the GEMM itself: bf16 operands, fp32 accumulator written in place (no bf16 dW, no add kernel)
            torch.addmm(weight.grad, dy2.t(), x2, out_dtype=torch.float32, out=weight.grad)
        else:
            gw = (dy2.t() @ x2).float()
        if bias is not None and ctx.needs_input_grad[2]:
            if DIRECT_GRADS and bias.grad is not None and dy2.is_cuda and dy2.dtype == torch.bfloat16 and dy2.is_contiguous() and dy2.shape[1] % 2 == 0:
                colsum_bf16(dy2, bias.grad, accumulate=True)       # db accumulated straight into the fp32 .grad
            else:
                gb = dy2.sum(0, dtype=torch.float32)
        return dx, gw, gb, None, None, None


def augment_batch(src_u8, offsets, params, B, crop_size, want_ori=True):
    """get_data_from_chunk_v2's per-image pixel work (myTool.py:1171-1196) for B decoded images packed in `src_u8`
    (device uint8); params int32 [B,12] from data.augment_params.  Returns (images [B,3,dim,dim] fp32, ori uint8 or None)."""
    _need_cuda(src_u8, offsets, params)
    out = torch.empty(B, 3, crop_size, crop_size, device=src_u8.device, dtype=torch.float32)
    ori = torch.empty(B, 3, crop_size, crop_size, device=src_u8.device, dtype=torch.uint8) if want_ori else None
    _call("acr_augment_batch", 1, _p(src_u8), _p(offsets), _p(params), int(B), int(crop_size), _p(out), _p(ori), _stream())
    return out, ori


def sgd_momentum_step(param, grad, buf, param_bf16, momentum, neg_lr):
    """buf = momentum*buf + grad ; param += neg_lr*buf ; param_bf16 = bf16(param) on flat fp32 buffers, one pass
    (neg_lr: device scalar).  tool/torchutils.py:10-31 as it really runs (SURVEY Q2)."""
    _need_cuda(param, grad, buf, neg_lr)
    _call("acr_sgd_momentum_step", 1, _p(param), _p(grad), _p(buf), _p(param_bf16), param.numel(), float(momentum), _p(neg_lr), _stream())


def colsum_bf16(x, out, accumulate=False):
    """out[F] (+)= x.sum(0) for a contiguous bf16 [M,F] matrix; fp32 accumulation, deterministic."""
    M, F = x.shape
    wsb = _lib.lib().acr_colsum_workspace(F)
    ws = torch.empty(wsb, device=x.device, dtype=torch.uint8)
    _call("acr_colsum_bf16", 2, _p(x), M, F, _p(out), int(accumulate), _p(ws), wsb, _stream())
    return out


def linear_cached_bf16(x, weight, bias, w16, b16, skip_bias_grad=False):
    return _LinearCachedBF16.apply(x, weight, bias, w16, b16, skip_bias_grad)


class _LinearGeluCachedBF16(torch.autograd.Function):
    """fc1 + exact GELU of the MLP (models/vision_transformer.py:158-160) on the cached-bf16 path: the GELU runs in this
    repo's kernels and its backward also produces fc1's bias gradient, so the [M,4E] gradient is read once."""

    @staticmethod
    def forward(ctx, x, weight, bias, w16, b16):
        x2 = x.reshape(-1, x.shape[-1])
        f = torch.nn.functional.linear(x2, w16, b16)
        y = torch.empty_like(f)
        _call("acr_gelu_fwd_bf16", 1, _p(f), _p(y), f.numel(), _stream())
        ctx.save_for_backward(x2, w16, f)
        ctx.params = (weight, bias)
        ctx.in_shape = x.shape
        return y.view(*x.shape[:-1], w16.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, w16, f = ctx.saved_tensors
        weight, bias = ctx.params
        M, F = f.shape
        dy2 = dy.reshape(M, F).contiguous()
        df = torch.empty_like(f)
        want_w, want_b = ctx.needs_input_grad[1], bias is not None and ctx.needs_input_grad[2]
        fused_bias = DIRECT_GRADS and want_b and bias.grad is not None and bias.grad.dtype == torch.float32
        gb = None
        if fused_bias:
            wsb = _lib.lib().acr_gelu_bwd_workspace(F)
            ws = torch.empty(wsb, device=f.device, dtype=torch.uint8)
            _call("acr_gelu_bwd_bf16", 2, _p(f), _p(dy2), _p(df), M, F, _p(bias.grad), 1, _p(ws), wsb, _stream())
        else:
            _call("acr_gelu_bwd_bf16", 1, _p(f), _p(dy2), _p(df), M, F, None, 0, None, 0, _stream())
            if want_b:
                gb = df.sum(0, dtype=torch.float32)
        dx = (df @ w16).view(ctx.in_shape) if ctx.needs_input_grad[0] else None
        gw = None
        if not want_w:
            pass
        elif DIRECT_GRADS and weight.grad is not None and weight.grad.dtype == torch.float32:
            torch.addmm(weight.grad, df.t(), x2, out_dtype=torch.float32, out=weight.grad)
        else:
            gw = (df.t() @ x2).float()
        return dx, gw, gb, None, None


def linear_gelu_cached_bf16(x, weight, bias, w16, b16):
    _need_cuda(x)
    return _LinearGeluCachedBF16.apply(x, weight, bias, w16, b16)


# ----------------------------------------------------------------------------------------------
# LayerNorm around the attention core (writes the following Linear's bf16 operand directly)
# ----------------------------------------------------------------------------------------------
class _LayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps, out_bf16):
        _need_cuda(x)
        E = x.shape[-1]
        x2 = x.contiguous().view(-1, E)
        if x2.dtype not in (torch.bfloat16, torch.float32):
            x2 = x2.float()
        xb = int(x2.dtype == torch.bfloat16)
        M = x2.shape[0]
        y = torch.empty(M, E, device=x.device, dtype=torch.bfloat16 if out_bf16 else torch.float32)
        mean = torch.empty(M, device=x.device, dtype=torch.float32)
        rstd = torch.empty(M, device=x.device, dtype=torch.float32)
        w, b = weight.contiguous().float(), bias.contiguous().float()
        _call("acr_layernorm_fwd", 1, _p(x2), xb, None, None, _p(w), _p(b), M, E, float(eps), _p(y), int(out_bf16), _p(mean), _p(rstd), _stream())
        ctx.save_for_backward(x2, mean, rstd, w)
        ctx.shape = x.shape
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, mean, rstd, w = ctx.saved_tensors
        M, E = x2.shape
        dy2 = dy.contiguous().view(M, E)
        if dy2.dtype not in (torch.bfloat16, torch.float32):
            dy2 = dy2.float()
        dx = torch.empty_like(x2)
        dg = torch.empty(E, device=x2.device, dtype=torch.float32)
        db = torch.empty(E, device=x2.device, dtype=torch.float32)
        wsb = _lib.lib().acr_layernorm_bwd_workspace(E)
        ws = torch.empty(wsb, device=x2.device, dtype=torch.uint8)
        _call("acr_layernorm_bwd", 2, _p(dy2), int(dy2.dtype == torch.bfloat16), None, _p(x2), int(x2.dtype == torch.bfloat16), _p(mean), _p(rstd), _p(w), M, E,
              _p(dx), _p(dg), _p(db), None, 0, _p(ws), wsb, _stream())
        return dx.view(ctx.shape), dg, db, None, None


class _AddLayerNorm(torch.autograd.Function):
    """s = x + branch ; y = LayerNorm(s)  (Block.forward, models/vision_transformer.py:230-233: the residual add and the norm
    that follows it) in one pass over the residual stream; returns (s, y).  Backward adds the gradient arriving at s over
    the skip connection to the LayerNorm input gradient inside the kernel (no separate accumulation pass)."""

    @staticmethod
    def forward(ctx, x, branch, weight, bias, eps, out_bf16, branch_bias):
        _need_cuda(x, branch)
        ctx.branch_bias = branch_bias
        E = x.shape[-1]
        x2 = x.contiguous().view(-1, E)
        r2 = branch.contiguous().view(-1, E)
        if r2.dtype != x2.dtype:
            r2 = r2.to(x2.dtype)
        xb = int(x2.dtype == torch.bfloat16)
        M = x2.shape[0]
        ssum = torch.empty_like(x2)
        y = torch.empty(M, E, device=x.device, dtype=torch.bfloat16 if out_bf16 else torch.float32)
        mean = torch.empty(M, device=x.device, dtype=torch.float32)
        rstd = torch.empty(M, device=x.device, dtype=torch.float32)
        w, b = weight.contiguous().float(), bias.contiguous().float()
        _call("acr_layernorm_fwd", 1, _p(x2), xb, _p(r2), _p(ssum), _p(w), _p(b), M, E, float(eps), _p(y), int(out_bf16), _p(mean), _p(rstd), _stream())
        ctx.norm_params = (weight, bias)
        ctx.save_for_backward(ssum, mean, rstd, w)
        ctx.shape = x.shape
        return ssum.view(x.shape), y.view(x.shape)

    @staticmethod
    def backward(ctx, ds, dy):
        s2, mean, rstd, w = ctx.saved_tensors
        M, E = s2.shape
        bb = ctx.branch_bias
        if dy is None:
            if bb is not None:
                raise RuntimeError("add_layer_norm: branch_bias given but the normalised output received no gradient")
            return ds, ds, None, None, None, None, None
        dy2 = dy.contiguous().view(M, E)
        if dy2.dtype not in (torch.bfloat16, torch.float32):
            dy2 = dy2.float()
        ds2 = None
        if ds is not None:
            ds2 = ds.contiguous().view(M, E)
            if ds2.dtype != s2.dtype:
                ds2 = ds2.to(s2.dtype)
        dx = torch.empty_like(s2)
        wsb = _lib.lib().acr_layernorm_bwd_workspace(E)
        ws = torch.empty(wsb, device=s2.device, dtype=torch.uint8)
        # bias gradient of the Linear that produced `branch` = column sums of dx, taken in the same pass
        col = bb.grad if bb is not None else None
        nw, nb = ctx.norm_params
        direct = DIRECT_GRADS and all(p_.grad is not None and p_.grad.dtype == torch.float32 and p_.grad.is_contiguous() for p_ in (nw, nb))
        if direct:          # d-gamma / d-beta added straight into the fp32 .grad buffers by the finish kernel
            dg, db = nw.grad, nb.grad
        else:
            dg = torch.empty(E, device=s2.device, dtype=torch.float32)
            db = torch.empty(E, device=s2.device, dtype=torch.float32)
            if col is not None:
                dg.zero_()
                db.zero_()
        acc = int(direct or col is not None)
        _call("acr_layernorm_bwd", 2, _p(dy2), int(dy2.dtype == torch.bfloat16), _p(ds2), _p(s2), int(s2.dtype == torch.bfloat16), _p(mean), _p(rstd),
              _p(w), M, E, _p(dx), _p(dg), _p(db), _p(col), acc, _p(ws), wsb, _stream())
        dx = dx.view(ctx.shape)
        if direct:
            return dx, dx, None, None, None, None, None
        return dx, dx, dg, db, None, None, None


def add_layer_norm(x, branch, weight, bias, eps=1e-6, out_bf16=False, branch_bias=None):
    """(x + branch, LayerNorm(x + branch)) with the add fused into the LayerNorm kernels (forward and backward).
    branch_bias: the bias Parameter of the Linear that produced `branch` (via linear_cached_bf16(..., skip_bias_grad=True));
    its fp32 .grad is incremented by the column sums of the branch gradient inside the backward kernel."""
    if branch_bias is not None and not (DIRECT_GRADS and branch_bias.grad is not None and branch_bias.grad.dtype == torch.float32
                                        and x.dtype == torch.bfloat16 and out_bf16):
        raise RuntimeError("add_layer_norm: branch_bias needs ops.direct_grads(), a preallocated fp32 .grad and the bf16 stream")
    return _AddLayerNorm.apply(x, branch, weight, bias, eps, out_bf16, branch_bias)


def layer_norm(x, weight, bias, eps=1e-6, out_bf16=False):
    """nn.LayerNorm(eps) over the last dimension of an fp32 or bf16 tensor; output fp32 or (out_bf16) bf16."""
    return _LayerNorm.apply(x, weight, bias, eps, out_bf16)


# ----------------------------------------------------------------------------------------------
# (a7) consistency loss
# ----------------------------------------------------------------------------------------------
def consistency_codes(attn1, attn2, p, one_buffer=False, swapped=False):
    """loss2 plus the gradient as SIGN CODES: uint8 [B,L,N,ld] (ld = N padded to 128), 0x00 / 0x3F (+) / 0xBF (-).
    one_buffer: c1/c2 are the two halves of a single [2B,L,N,ld] tensor (views batched through the trunk together);
    swapped: attn1 is the SECOND half of that batch (consistency_loss(attn2, attn1)), so c1 must land in rows [B:]."""
    _need_cuda(attn1, attn2)
    B, L, N, _ = attn1.shape
    a1 = attn1.contiguous().float()
    a2 = attn2.contiguous().float()
    ld = (N + 127) // 128 * 128
    loss2 = torch.empty(2, device=a1.device, dtype=torch.float32)
    if one_buffer:
        c = torch.empty(2 * B, L, N, ld, device=a1.device, dtype=torch.uint8)
        c1, c2 = (c[B:], c[:B]) if swapped else (c[:B], c[B:])
    else:
        c1 = torch.empty(B, L, N, ld, device=a1.device, dtype=torch.uint8)
        c2 = torch.empty(B, L, N, ld, device=a1.device, dtype=torch.uint8)
    wsb = _lib.lib().acr_consistency_workspace(B, L, N)
    ws = torch.empty(wsb, device=a1.device, dtype=torch.uint8)
    _call("acr_consistency_fwd_bwd", 2, _p(a1), _p(a2), B, L, N, int(p), 1.0, 1.0, _p(loss2), None, None, 0,
          _p(c1), _p(c2), ld, _p(ws), wsb, _stream())
    return loss2, c1, c2


def consistency_fwd_bwd(attn1, attn2, p, alpha_cls=1.0, alpha_aff=1.0, need_grad=True):
    """Returns (loss2 [2] = (cls_align, aff_align), g1, g2); g = alpha_cls*dcls/dA + alpha_aff*daff/dA."""
    _need_cuda(attn1, attn2)
    assert attn1.shape == attn2.shape and attn1.dim() == 4
    B, L, N, _ = attn1.shape
    a1 = attn1.contiguous().float()
    a2 = attn2.contiguous().float()
    loss2 = torch.empty(2, device=a1.device, dtype=torch.float32)
    # gradient rows are padded to a multiple of 4 floats (16-byte aligned rows for the attention backward's
    # 128-bit loads); callers see the dense [B,L,N,N] view
    Np = (N + 3) // 4 * 4
    g1 = torch.empty(B, L, N, Np, device=a1.device, dtype=torch.float32) if need_grad else None
    g2 = torch.empty(B, L, N, Np, device=a1.device, dtype=torch.float32) if need_grad else None
    wsb = _lib.lib().acr_consistency_workspace(B, L, N)
    ws = torch.empty(wsb, device=a1.device, dtype=torch.uint8)
    _call("acr_consistency_fwd_bwd", 2, _p(a1), _p(a2), B, L, N, int(p), float(alpha_cls), float(alpha_aff),
                                             _p(loss2), _p(g1), _p(g2), Np, None, None, 0, _p(ws), wsb, _stream())
    if need_grad:
        g1, g2 = g1[..., :N], g2[..., :N]
    return loss2, g1, g2


class _ConsistencyLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, attn1, attn2, p, alpha):
        need = attn1.requires_grad or attn2.requires_grad
        loss2, g1, g2 = consistency_fwd_bwd(attn1.detach(), attn2.detach(), p, alpha, alpha, need_grad=need)
        if need:
            ctx.save_for_backward(g1, g2)
        ctx.need = need
        total = alpha * (loss2[0] + loss2[1])
        ctx.mark_non_differentiable(loss2)
        return total, loss2

    @staticmethod
    def backward(ctx, g_total, _g_loss2):
        if not ctx.need:
            return None, None, None, None
        g1, g2 = ctx.saved_tensors
        # g1/g2 already carry alpha/count; scale by the incoming scalar (1.0 in the training step)
        return g1.mul_(g_total), g2.mul_(g_total), None, None


class _ConsistencyLossCodes(torch.autograd.Function):
    """Same loss, but the gradient never exists as fp32 [B,L,N,N]: backward hands each attention block its slice of the
    sign-code tensor (plus the two weights and autograd's upstream scalar, kept on the device) through the block's
    state dict, and returns no tensor gradient.  The fused attention backward picks the codes up (autograd runs it
    after this node because the stack it produced feeds this loss)."""

    @staticmethod
    def forward(ctx, attn1, attn2, p, alpha, states1, states2, swapped):
        B, L, N, _ = attn1.shape
        merged = states1 is states2 or (len(states1) == len(states2) and all(a is b for a, b in zip(states1, states2)))
        loss2, c1, c2 = consistency_codes(attn1.detach(), attn2.detach(), p, merged, swapped and merged)
        if merged:      # both views went through the trunk as one batch of 2B: c1/c2 are the halves of one buffer
            ctx.codes = (c1._base if c1._base is not None else c1,)
            ctx.states = (states1,)
        else:
            ctx.codes = (c1, c2)
            ctx.states = (states1, states2)
        ctx.w = (alpha / (B * L * (N - 1)), alpha / (B * L * float(N - 1) ** 2))
        total = alpha * (loss2[0] + loss2[1])
        ctx.mark_non_differentiable(loss2)
        return total, loss2

    @staticmethod
    def backward(ctx, g_total, _g_loss2):
        scale = g_total.detach().reshape(1).float().contiguous()
        for codes, states in zip(ctx.codes, ctx.states):
            for l, st in enumerate(states):
                if st.get("g_code") is not None:
                    # a second loss on the same stacks: codes cannot be summed byte-wise
                    raise RuntimeError("consistency_loss was applied twice to the same attention stacks; its sign-code gradient "
                                       "cannot be accumulated -- combine the terms into one call, or detach the stacks' "
                                       "_acr_states attribute to use the dense-gradient path")
                st["g_code"] = codes[:, l]
                st["g_w"] = ctx.w
                st["g_scale"] = scale
        return None, None, None, None, None, None, None


def consistency_loss(attn1, attn2, p, alpha):
    """alpha*(cls_align + aff_align) with its gradient fused; also returns the two components (detached).

    When both stacks come straight from the fused attention path (ops.stack_views with per-block states), the gradient
    travels as one sign byte per element instead of dense fp32 maps (4x less HBM traffic in the loss kernel and in
    every attention backward); otherwise dense fp32 gradients flow through autograd as usual."""
    st1, st2 = getattr(attn1, "_acr_states", None), getattr(attn2, "_acr_states", None)
    if (st1 is not None and st2 is not None and attn1.requires_grad and attn2.requires_grad
            and all(s is not None and s.get("fused") for s in st1 + st2)):
        h1, h2 = getattr(attn1, "_acr_half", None), getattr(attn2, "_acr_half", None)
        merged = len(st1) == len(st2) and all(a is b for a, b in zip(st1, st2))
        if not merged or (h1, h2) in ((0, 1), (1, 0)):         # (the same half twice would need two code slices per block)
            return _ConsistencyLossCodes.apply(attn1, attn2, int(p), float(alpha), st1, st2, (h1, h2) == (1, 0))
    return _ConsistencyLoss.apply(attn1, attn2, int(p), float(alpha))


# ----------------------------------------------------------------------------------------------
# (a8) GETAM, (a9) refine
# ----------------------------------------------------------------------------------------------
def getam_row0(p_row0, g_row0, start_layer=0, func="grad", skip=1, want_rows=False):
    """p_row0/g_row0 [L,H,N] -> cls_cam [1,N-skip] (and per-block rows [L,N] if want_rows)."""
    _need_cuda(p_row0, g_row0)
    L, H, N = p_row0.shape
    p_row0 = p_row0.contiguous().float()
    g_row0 = g_row0.contiguous().float()
    cam = torch.empty(1, N - skip, device=p_row0.device, dtype=torch.float32)
    rows = torch.empty(L, N, device=p_row0.device, dtype=torch.float32) if want_rows else None
    _call("acr_getam_row0", 1, _p(p_row0), _p(g_row0), L, H, N, int(start_layer), _GETAM_FUNCS[func], int(skip),
                                         _p(cam), _p(rows), _stream())
    return (cam, rows) if want_rows else cam


def getam_row0_batch(p_row0, g_row0, start_layer=0, func="grad", skip=1):
    """p_row0/g_row0 [L,S,H,N] (S samples stacked over the L used blocks) -> cls_cam [S,N-skip]."""
    _need_cuda(p_row0, g_row0)
    L, S, H, N = p_row0.shape
    p_row0 = p_row0.contiguous().float()
    g_row0 = g_row0.contiguous().float()
    cam = torch.empty(S, N - skip, device=p_row0.device, dtype=torch.float32)
    _call("acr_getam_row0_batch", 1, _p(p_row0), _p(g_row0), S, L, H, N, int(start_layer), _GETAM_FUNCS[func], int(skip), _p(cam), _stream())
    return cam


def affinity_sum(attn, normalize=False):
    """attn [B,L,N,N] -> A [B,N-1,N-1] = sum_l attn[:,l,1:,1:] (infer_cam.py:164-165)."""
    _need_cuda(attn)
    B, L, N, _ = attn.shape
    attn = attn.contiguous().float()
    A = torch.empty(B, N - 1, N - 1, device=attn.device, dtype=torch.float32)
    _call("acr_affinity_sum", 1, _p(attn), B, L, N, int(bool(normalize)), _p(A), _stream())
    return A


def affinity_apply(A, cam, t=1):
    """A [B,Np,Np], cam [B,Np,C] -> A^t cam (infer_cam.py:184, all classes in one contraction)."""
    _need_cuda(A, cam)
    B, Np, _ = A.shape
    C = cam.shape[-1]
    A = A.contiguous().float()
    cam = cam.contiguous().float()
    out = torch.empty_like(cam)
    tmp = torch.empty_like(cam) if t > 1 else None
    _call("acr_affinity_refine", 1, _p(A), _p(cam), B, Np, C, int(t), _p(out), _p(tmp), _stream())
    return out


def affinity_refine_tc(attn, cam, t=1, normalize=False):
    """attn [B,L,N,N], cam [B,N-1,C] -> (sum_l attn[:,l,1:,1:])^t cam on the tensor cores (infer_cam.py:164-165,184): the block sum,
    the contraction for all classes and the row normalisation in one tcgen05 kernel per power (csrc/refine_tc.cu)."""
    _need_cuda(attn, cam)
    B, L, N, _ = attn.shape
    C = cam.shape[-1]
    attn = attn.contiguous().float()
    cam = cam.contiguous().float()
    out = torch.empty_like(cam)
    nbytes = _lib.lib().acr_affinity_refine_tc_workspace(B, N, C, int(t))
    ws = torch.empty(nbytes, device=attn.device, dtype=torch.uint8) if nbytes else None
    _call("acr_affinity_refine_tc", int(t), _p(attn), B, L, N, _p(cam), C, int(t), int(bool(normalize)), _p(out), _p(ws), nbytes, _stream())
    return out


def cam_finish(cams, patches, grids, labels, planes, total):
    """Finish of batched CAM inference for every plane of a batch in one launch (csrc/cam_finish.cu, infer_cam.py:153-215).
    cams / patches: per scale [2M, ph*pw, n] GETAM maps and [2M, ph*pw, C] patch CAMs (batch index v*M+m, view 0 = flipped
    input); grids: per scale (ph, pw); labels [M, C]; planes: rows {offset, image, channel, kind (0 GETAM, 1 patch CAM),
    rows, cols}, see acr_cam_finish in include/acr_b200.h.  Returns the packed fp32 buffer of `total` elements."""
    _need_cuda(labels, *cams, *patches)
    ns = len(grids)
    assert len(cams) == ns and len(patches) == ns
    cams = [c.contiguous().float() for c in cams]
    patches = [c.contiguous().float() for c in patches]
    labels = labels.contiguous().float()
    M, C = labels.shape
    table = np.ascontiguousarray(np.asarray(planes, dtype=np.int64).reshape(-1, 6))
    out = torch.empty(total, device=labels.device, dtype=torch.float32)
    ws = torch.empty(table.nbytes, device=labels.device, dtype=torch.uint8)
    _call("acr_cam_finish", 1 if len(table) else 0,
          (ctypes.c_void_p * ns)(*[c.data_ptr() for c in cams]), (ctypes.c_void_p * ns)(*[c.data_ptr() for c in patches]),
          (ctypes.c_int * (2 * ns))(*[int(v) for g in grids for v in g]), ns, M, cams[0].shape[-1], C, _p(labels),
          table.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)), len(table), _p(out), int(total), _p(ws), table.nbytes, _stream())
    return out


class _PatchCam(torch.autograd.Function):
    """relu(tokens . W^T + b) through acr_patch_cam_tc; the backward (nobody on the reference path uses it: infer_cam.py:158
    detaches the result at once) is the plain closed form."""

    @staticmethod
    def forward(ctx, tokens, weight, bias):
        B, M, E = tokens.shape
        C = weight.shape[0]
        out = torch.empty(B, M, C, device=tokens.device, dtype=torch.float32)
        w = weight.detach().contiguous().float()
        bv = None if bias is None else bias.detach().contiguous().float()
        _call("acr_patch_cam_tc", 1, _p(tokens), tokens.stride(0), tokens.stride(1), B, M, E, _p(w), _p(bv), C, 1, _p(out), _stream())
        ctx.save_for_backward(tokens, weight, out)
        ctx.has_bias = bias is not None
        return out

    @staticmethod
    def backward(ctx, dy):
        tokens, weight, out = ctx.saved_tensors
        dz = dy * (out > 0)
        dx = dz @ weight.float()
        dw = dz.flatten(0, 1).t() @ tokens.flatten(0, 1)
        return dx, dw.to(weight.dtype), (dz.sum((0, 1)) if ctx.has_bias else None)


def patch_cam(tokens, weight, bias):
    """DPT/ACR.py:133-134: x_patch_cam = relu(cls_head(x_patch)), tokens [B,M,E] fp32 (any batch / row strides, unit inner stride)."""
    _need_cuda(tokens, weight)
    assert tokens.dtype == torch.float32 and tokens.stride(2) == 1
    return _PatchCam.apply(tokens, weight, bias)


class _CrfHead(torch.autograd.Function):
    """Patch-token logits [B,P*P,C] -> probabilities [B,C+1,S/2,S/2] the dense-CRF term filters (csrc/crf_head.cu): bilinear
    up-sampling to SxS, softmax over [background = 0, classes], bilinear down-sampling by 0.5, fused."""

    @staticmethod
    def forward(ctx, logits, S):
        B, PP, C = logits.shape
        P = int(round(PP ** 0.5))
        assert P * P == PP and S % 2 == 0
        logits = logits.contiguous().float()
        seg = torch.empty(B, C + 1, S // 2, S // 2, device=logits.device, dtype=torch.float32)
        _call("acr_crf_head_fwd", 1, _p(logits), B, P, C, S, _p(seg), _stream())
        ctx.save_for_backward(logits)
        ctx.dims = (B, P, C, S)
        return seg

    @staticmethod
    def backward(ctx, g_seg):
        (logits,) = ctx.saved_tensors
        B, P, C, S = ctx.dims
        d_up = torch.empty(B, C, S, S, device=logits.device, dtype=torch.float32)
        _call("acr_crf_head_bwd", 1, _p(logits), _p(g_seg.contiguous().float()), B, P, C, S, _p(d_up), _stream())
        if S <= 512:      # gather form of the bilinear backward (the library's scatters with atomics: 16.6 ms at [8,80,448,448])
            d_patch = torch.empty(B, C, P, P, device=logits.device, dtype=torch.float32)
            _call("acr_bilinear_up_bwd", 1, _p(d_up), B * C, P, S, _p(d_patch), _stream())
        else:
            d_patch = torch.ops.aten.upsample_bilinear2d_backward(d_up, [S, S], [B, C, P, P], False, None, None)
        return d_patch.flatten(2).transpose(1, 2), None


def crf_head(logits, S):
    _need_cuda(logits)
    return _CrfHead.apply(logits, S)


# ----------------------------------------------------------------------------------------------
# (a10) PAMR, (a11) bilateral
# ----------------------------------------------------------------------------------------------
def pamr_forward(x, mask, dilations, num_iter):
    _need_cuda(x, mask)
    B, K, H, W = x.shape
    _, C, mh, mw = mask.shape
    x = x.contiguous().float()
    mask = mask.contiguous().float()
    nd = len(dilations)
    dil = (ctypes.c_int * nd)(*[int(d) for d in dilations])
    out = torch.empty(B, C, H, W, device=x.device, dtype=torch.float32)
    wsb = _lib.lib().acr_pamr_workspace(B, K, C, H, W, nd)
    ws = torch.empty(wsb, device=x.device, dtype=torch.uint8)
    _call("acr_pamr_fwd", 3, _p(x), _p(mask), B, K, C, H, W, mh, mw, dil, nd, int(num_iter),
                                       _p(out), _p(ws), wsb, _stream())
    return out


def bilateral_filter(images, ins, sigmargb, sigmaxy, return_lattice_size=False):
    """Device-tensor form of bilateralfilter_batch: images [N,3,H,W] (0..255), ins [N,K,H,W] -> outs."""
    _need_cuda(images, ins)
    N, K, H, W = ins.shape
    assert images.shape == (N, 3, H, W)
    images = images.contiguous().float()
    ins = ins.contiguous().float()
    outs = torch.empty_like(ins)
    wsb = _lib.lib().acr_bilateral_workspace(N, K, H, W)
    ws = torch.empty(wsb + 256, device=ins.device, dtype=torch.uint8)
    off = (-ws.data_ptr()) % 256
    msz = (ctypes.c_int * N)() if return_lattice_size else None
    _call("acr_bilateral_batch", 11 * ((N + 7) // 8), _p(images), _p(ins), _p(outs), N, K, H, W, float(sigmargb), float(sigmaxy),
                                              ctypes.c_void_p(ws.data_ptr() + off), wsb, msz, _stream())
    if return_lattice_size:
        return outs, list(msz)
    return outs


def dense_crf(images, probs, n_iter=10, sxy_g=3.0, compat_g=3.0, sxy_b=80.0, srgb=13.0, compat_b=10.0, clip=1e-5):
    """Dense-CRF mean-field inference (densecrf 2.x, Potts over a Gaussian and a bilateral kernel; acr_dense_crf):
    images [N,3,H,W] (0..255), probs [N,C,H,W] scores (unary -log(max(P, clip)); they need not sum to 1) -> Q [N,C,H,W],
    the marginals after n_iter iterations.  Deterministic; capturable in a CUDA graph (the workspace is allocated here)."""
    _need_cuda(images, probs)
    N, C, H, W = probs.shape
    assert images.shape == (N, 3, H, W)
    images = images.contiguous().float()
    probs = probs.contiguous().float()
    q = torch.empty_like(probs)
    wsb = _lib.lib().acr_dense_crf_workspace(N, C, H, W)
    ws = torch.empty(wsb + 256, device=probs.device, dtype=torch.uint8)
    off = (-ws.data_ptr()) % 256
    _call("acr_dense_crf", (11 + 8 * int(n_iter)) * ((N + 7) // 8), _p(images), _p(probs), _p(q), N, C, H, W, int(n_iter),
          float(sxy_g), float(compat_g), float(sxy_b), float(srgb), float(compat_b), float(clip),
          ctypes.c_void_p(ws.data_ptr() + off), wsb, _stream())
    return q

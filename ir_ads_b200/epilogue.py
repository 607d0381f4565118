"""Fused residual add + LayerNorm: the epilogue that follows every MSDeformAttn call and every FFN in the reference's
transformer layers (``x = x + identity; x = norm(x)``: detrex/layers/transformer.py:152-192 with the residuals added at
multi_scale_deform_attn.py:363 and detrex/layers/mlp.py:127-132).  One sm_100a kernel forward (reads both addends,
writes the normalised row; the sum is never stored), one backward (recomputes the sum, writes ONE gradient that serves
both addends, reduces weight / bias gradients in a fixed order) -- ir_ads_b200/csrc/msda_epilogue.cu, bound through the
same C ABI (include/msda.h: msda_add_layernorm_forward / _backward).  CUDA only, float32 / bfloat16 / float16.

Under autocast the attention / FFN output is 16-bit while the residual stays float32; ``add_layer_norm`` then takes the
mixed form (``msda_add_layernorm_mixed_*``): the 16-bit addend is widened inside the kernel, the result is float32 --
what ``norm(a + b)`` gives with torch's type promotion -- and the backward writes the float32 gradient and its 16-bit
rounding (the 16-bit addend's gradient, as autograd's cast would round it) in one pass.
"""
from __future__ import annotations

import ctypes

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib
from .functional import _VALUE_TAG, _aligned, _ptr, _require

_LN_DTYPES = (torch.float32, torch.bfloat16, torch.float16)
_HALF_DTYPES = (torch.bfloat16, torch.float16)


def add_layer_norm_supported(x: torch.Tensor) -> bool:
    c = x.shape[-1] if x.dim() else 0
    return x.is_cuda and x.dtype in _LN_DTYPES and c > 0 and c % 4 == 0 and c <= 1024


class AddLayerNormFunction(Function):
    """``apply(a, b, weight, bias, eps)`` -> ``LayerNorm(a + b)`` over the last dimension."""

    @staticmethod
    def forward(ctx, a, b, weight, bias, eps):
        y, saved = _same_forward(a, b, weight, bias, eps)
        ctx.save_for_backward(*saved)
        ctx.param_dtypes = (weight.dtype, bias.dtype)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y):
        dx, dgamma, dbeta = _same_backward(grad_y, *ctx.saved_tensors)
        wd, bd = ctx.param_dtypes
        return (dx if ctx.needs_input_grad[0] else None, dx if ctx.needs_input_grad[1] else None,
                dgamma.to(wd) if ctx.needs_input_grad[2] else None, dbeta.to(bd) if ctx.needs_input_grad[3] else None,
                None)


class AddLayerNormMixedFunction(Function):
    """``apply(a, b, weight, bias, eps)`` -> ``LayerNorm(a + b)`` in float32 for a bfloat16 / float16 ``a`` and a
    float32 ``b``: one kernel each way, no widened copy of ``a`` and no cast of its gradient."""

    @staticmethod
    def forward(ctx, a, b, weight, bias, eps):
        y, saved = _mixed_forward(a, b, weight, bias, eps)
        ctx.save_for_backward(*saved)
        ctx.param_dtypes = (weight.dtype, bias.dtype)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_y):
        da, db, dgamma, dbeta = _mixed_backward(grad_y, *ctx.saved_tensors)
        wd, bd = ctx.param_dtypes
        return (da if ctx.needs_input_grad[0] else None, db if ctx.needs_input_grad[1] else None,
                dgamma.to(wd) if ctx.needs_input_grad[2] else None, dbeta.to(bd) if ctx.needs_input_grad[3] else None,
                None)


# The bodies of the two Functions, shared with the ir_ads_b200::add_layer_norm ops (ir_ads_b200/ops.py).  The forwards
# return the output and what the backward reads: (a, b, float32 weight, mean, rstd).
def _same_forward(a, b, weight, bias, eps):
    _require(a.is_cuda, "add_layer_norm: Not implemented on the CPU")
    _require(a.shape == b.shape and a.dtype == b.dtype and b.device == a.device, "a and b must match")
    _require(a.dtype in _LN_DTYPES, f"unsupported dtype {a.dtype} (float32, bfloat16, float16)")
    C = a.shape[-1]
    _require(tuple(weight.shape) == (C,) and tuple(bias.shape) == (C,), "weight / bias must be [C]")
    a, b = _aligned(a.contiguous()), _aligned(b.contiguous())
    w32, b32 = _aligned(weight.float().contiguous()), _aligned(bias.float().contiguous())
    rows = a.numel() // C if C else 0
    y = torch.empty_like(a)
    mean = torch.empty(rows, dtype=torch.float32, device=a.device)
    rstd = torch.empty(rows, dtype=torch.float32, device=a.device)
    stream = torch.cuda.current_stream(a.device).cuda_stream
    status = _lib.lib().msda_add_layernorm_forward(ctypes.c_void_p(stream), _ptr(a), _ptr(b), _ptr(w32), _ptr(b32),
                                                   rows, C, float(eps), _ptr(y), _ptr(mean), _ptr(rstd),
                                                   _VALUE_TAG[a.dtype])
    _lib.check(status, "msda_add_layernorm_forward")
    return y, (a, b, w32, mean, rstd)


def _same_backward(grad_y, a, b, w32, mean, rstd):
    """``(grad of a + b in a's dtype, float32 grad_weight, float32 grad_bias)``."""
    C = a.shape[-1]
    rows = a.numel() // C
    grad_y = _aligned(grad_y.contiguous())
    _require(grad_y.dtype == a.dtype and grad_y.shape == a.shape, "grad_output must match the output")
    dx = torch.empty_like(a)
    dgamma = torch.empty(C, dtype=torch.float32, device=a.device)
    dbeta = torch.empty(C, dtype=torch.float32, device=a.device)
    handle = _lib.lib()
    ws_bytes = int(handle.msda_add_layernorm_workspace_bytes(rows, C))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=a.device)
    stream = torch.cuda.current_stream(a.device).cuda_stream
    status = handle.msda_add_layernorm_backward(ctypes.c_void_p(stream), _ptr(grad_y), _ptr(a), _ptr(b), _ptr(w32),
                                                _ptr(mean), _ptr(rstd), rows, C, _ptr(dx), _ptr(dgamma), _ptr(dbeta),
                                                _ptr(ws), ws_bytes, _VALUE_TAG[a.dtype])
    _lib.check(status, "msda_add_layernorm_backward")
    return dx, dgamma, dbeta


def _mixed_forward(a, b, weight, bias, eps):
    _require(a.is_cuda, "add_layer_norm: Not implemented on the CPU")
    _require(a.shape == b.shape and b.device == a.device, "a and b must match")
    _require(a.dtype in _HALF_DTYPES and b.dtype == torch.float32,
             f"mixed add_layer_norm: a bfloat16 / float16, b float32 (got {a.dtype}, {b.dtype})")
    C = a.shape[-1]
    _require(tuple(weight.shape) == (C,) and tuple(bias.shape) == (C,), "weight / bias must be [C]")
    a, b = _aligned(a.contiguous()), _aligned(b.contiguous())
    w32, b32 = _aligned(weight.float().contiguous()), _aligned(bias.float().contiguous())
    rows = a.numel() // C if C else 0
    y = torch.empty_like(b)
    mean = torch.empty(rows, dtype=torch.float32, device=a.device)
    rstd = torch.empty(rows, dtype=torch.float32, device=a.device)
    stream = torch.cuda.current_stream(a.device).cuda_stream
    status = _lib.lib().msda_add_layernorm_mixed_forward(ctypes.c_void_p(stream), _ptr(a), _ptr(b), _ptr(w32),
                                                         _ptr(b32), rows, C, float(eps), _ptr(y), _ptr(mean),
                                                         _ptr(rstd), _VALUE_TAG[a.dtype])
    _lib.check(status, "msda_add_layernorm_mixed_forward")
    return y, (a, b, w32, mean, rstd)


def _mixed_backward(grad_y, a, b, w32, mean, rstd):
    """``(16-bit grad_a, float32 grad_b, float32 grad_weight, float32 grad_bias)``."""
    C = a.shape[-1]
    rows = a.numel() // C
    grad_y = _aligned(grad_y.float().contiguous())
    _require(grad_y.shape == b.shape, "grad_output must match the output")
    da = torch.empty_like(a)
    db = torch.empty_like(b)
    dgamma = torch.empty(C, dtype=torch.float32, device=a.device)
    dbeta = torch.empty(C, dtype=torch.float32, device=a.device)
    handle = _lib.lib()
    ws_bytes = int(handle.msda_add_layernorm_workspace_bytes(rows, C))
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=a.device)
    stream = torch.cuda.current_stream(a.device).cuda_stream
    status = handle.msda_add_layernorm_mixed_backward(ctypes.c_void_p(stream), _ptr(grad_y), _ptr(a), _ptr(b),
                                                      _ptr(w32), _ptr(mean), _ptr(rstd), rows, C, _ptr(da),
                                                      _ptr(db), _ptr(dgamma), _ptr(dbeta), _ptr(ws), ws_bytes,
                                                      _VALUE_TAG[a.dtype])
    _lib.check(status, "msda_add_layernorm_mixed_backward")
    return da, db, dgamma, dbeta


def add_layer_norm(a: torch.Tensor, b: torch.Tensor, norm: torch.nn.LayerNorm) -> torch.Tensor:
    """``norm(a + b)``: the fused kernel where it applies (CUDA, C % 4 == 0, C <= 1024, affine LayerNorm over the last
    dimension; a and b both float32 / bfloat16 / float16, or -- under autocast -- one of them bfloat16 / float16 and the
    other float32, in either order, with a float32 result), otherwise the two PyTorch ops it replaces.  Two float16
    addends under autocast also take the PyTorch ops: autocast runs the LayerNorm in float32 on their float16 sum and
    returns float32, which the same-dtype kernel (float16 result) would not reproduce.  (Two bfloat16 addends keep the
    kernel and its bfloat16 result under autocast, as before float16 was supported.)"""
    if not (add_layer_norm_supported(a) and add_layer_norm_supported(b) and a.shape == b.shape
            and norm.elementwise_affine and norm.bias is not None and tuple(norm.normalized_shape) == (a.shape[-1],)):
        return norm(a + b)
    if a.dtype == b.dtype == torch.float16 and torch.is_autocast_enabled(a.device.type):
        return norm(a + b)
    if a.dtype == b.dtype:
        if torch.compiler.is_compiling():
            return torch.ops.ir_ads_b200.add_layer_norm(a, b, norm.weight, norm.bias, norm.eps)[0]
        return AddLayerNormFunction.apply(a, b, norm.weight, norm.bias, norm.eps)
    if a.dtype == torch.float32:
        a, b = b, a                                   # float addition commutes: the 16-bit addend goes first
    if b.dtype == torch.float32:
        if torch.compiler.is_compiling():
            return torch.ops.ir_ads_b200.add_layer_norm(a, b, norm.weight, norm.bias, norm.eps)[0]
        return AddLayerNormMixedFunction.apply(a, b, norm.weight, norm.bias, norm.eps)
    return norm(a + b)

"""Operator boundary of the B200-native MSDeformAttn: the two functions the reference exposes as
``detrex._C.ms_deform_attn_forward / ms_deform_attn_backward``
(/root/reference/detrex/layers/csrc/vision.cpp:54-59, ms_deform_attn.h:21-62) and the autograd
``MultiScaleDeformableAttnFunction`` built on them
(/root/reference/detrex/layers/multi_scale_deform_attn.py:44-93), with the same names, argument
order and error behaviour -- bound to libmsda_b200.so through ctypes instead of pybind11.

Differences from the reference, all documented in SURVEY.md appendix B and DESIGN.md:
  * bf16 ``value`` is supported (locations / weights stay float32, fp32 accumulate); the reference
    dispatches float and double only (ms_deform_attn_cuda.cu:65).  float16 is refused here as there; the fused
    module path (MSDeformAttnFusedFunction) takes it natively;
  * ``im2col_step`` is accepted and ignored: one launch covers the batch, so the reference's
    ``batch % im2col_step == 0`` assert (ms_deform_attn_cuda.cu:53) has nothing to protect;
  * a non-contiguous ``grad_output`` is made contiguous instead of asserting (cu:99);
  * CPU tensors raise (as ms_deform_attn.h:39 does) -- there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import contextlib
import ctypes
from typing import List

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib

# value dtypes of the public operator (the reference's _C dispatches float / double only; bf16 is an extension)
_DTYPE_TAG = {torch.float32: _lib.MSDA_F32, torch.float64: _lib.MSDA_F64, torch.bfloat16: _lib.MSDA_BF16}
# value dtypes of the fused module path and of the library-internal calls: float16 as well (MSDA_F16: every kernel
# widens it exactly and accumulates in float32).  The public operator keeps refusing float16, as the reference's does.
_VALUE_TAG = {**_DTYPE_TAG, torch.float16: _lib.MSDA_F16}
_FUSED_DTYPES = (torch.float32, torch.bfloat16, torch.float16)
# the fused paths' autocast tags: 16-bit value AND 16-bit offsets / logits (the Linear outputs as autocast produces them)
_AUX16_TAG = {torch.bfloat16: _lib.MSDA_BF16_AUX16, torch.float16: _lib.MSDA_F16_AUX16}


def _aux_tag(value_dtype, aux_dtype, what):
    """The dtype tag of a fused call: the value's tag with float32 offsets / logits, its autocast tag when they are in
    the value's own 16-bit type; any other mix is refused."""
    if aux_dtype == torch.float32:
        return _VALUE_TAG[value_dtype]
    _require(aux_dtype == value_dtype and value_dtype in _AUX16_TAG,
             f"{what} must be float32, or in the value's dtype when that is float16 / bfloat16 "
             f"(got {aux_dtype} with a {value_dtype} value)")
    return _AUX16_TAG[value_dtype]

_state = {"deterministic": False, "flags": 0}


def set_deterministic(enabled: bool) -> None:
    """Select the bit-reproducible backward (also implied by torch.use_deterministic_algorithms): MSDeformAttn, the fused
    module path and DCNv3 (``dcnv3_backward``, ``DCNv3Function``, the ``DCNv3`` module) then compute every gradient in a
    fixed order, so two runs on the same inputs give the same bits."""
    _state["deterministic"] = bool(enabled)


@contextlib.contextmanager
def kernel_flags(flags: int):
    """Temporarily OR extra MSDA_FLAG_* bits into every call (tests / benchmarks)."""
    old = _state["flags"]
    _state["flags"] = old | int(flags)
    try:
        yield
    finally:
        _state["flags"] = old


def _flags(backward: bool) -> int:
    f = _state["flags"]
    if backward and (_state["deterministic"] or torch.are_deterministic_algorithms_enabled()):
        f |= _lib.FLAG_DETERMINISTIC
    return f


def _deterministic() -> bool:
    """Whether backward passes take the bit-reproducible route.  The custom ops (ir_ads_b200/ops.py) take it as an
    argument, read here while the graph is built, so that the compiler guards on it."""
    return bool(_flags(True) & _lib.FLAG_DETERMINISTIC)


def _ptr(t: torch.Tensor) -> ctypes.c_void_p:
    return ctypes.c_void_p(t.data_ptr())


def _require(cond: bool, msg: str) -> None:
    if not cond:
        raise RuntimeError(msg)


def _aligned(t):
    """The kernels use 128-bit accesses (include/msda.h): a contiguous tensor whose storage offset leaves it off a
    16-byte boundary (a slice of a flat buffer, say) is copied into a fresh allocation.  Never the case for tensors
    that own their storage; the reference's scalar kernels had no such requirement, so the wrappers hide it."""
    if t is None or t.numel() == 0 or t.data_ptr() % 16 == 0:
        return t
    return t.clone(memory_format=torch.contiguous_format)


def _check_inputs(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, tags=_DTYPE_TAG):
    # mirrors the AT_ASSERTM block of ms_deform_attn_cuda.cu:29-39
    _require(value.is_cuda, "Not implemented on the CPU")  # ms_deform_attn.h:39
    for name, t in (("value", value), ("spatial_shapes", spatial_shapes),
                    ("level_start_index", level_start_index), ("sampling_loc", sampling_loc),
                    ("attn_weight", attn_weight)):
        _require(t.is_cuda, f"{name} must be a CUDA tensor")
        _require(t.is_contiguous(), f"{name} tensor has to be contiguous")
        _require(t.device == value.device, f"{name} must be on {value.device}")
    _require(value.dim() == 4, "value must be [B, S, H, D]")
    _require(sampling_loc.dim() == 6 and sampling_loc.shape[-1] == 2, "sampling_loc must be [B, Q, H, L, P, 2]")
    _require(attn_weight.dim() == 5, "attn_weight must be [B, Q, H, L, P]")
    _require(spatial_shapes.dtype == torch.int64 and level_start_index.dtype == torch.int64,
             "spatial_shapes / level_start_index must be int64")
    B, S, H, D = value.shape
    Bq, Q, Hq, L, P, _ = sampling_loc.shape
    _require(Bq == B and Hq == H, "sampling_loc batch / heads do not match value")
    _require(tuple(attn_weight.shape) == (B, Q, H, L, P), "attn_weight shape does not match sampling_loc")
    _require(spatial_shapes.shape == (L, 2) and level_start_index.shape == (L,),
             "spatial_shapes must be [L, 2] and level_start_index [L]")
    names = ", ".join(str(t).replace("torch.", "") for t in tags)
    _require(value.dtype in tags, f"unsupported value dtype {value.dtype} ({names})")
    aux = torch.float64 if value.dtype == torch.float64 else torch.float32
    _require(sampling_loc.dtype == aux and attn_weight.dtype == aux,
             f"sampling_loc / attn_weight must be {aux} when value is {value.dtype}")
    return B, S, H, D, L, Q, P


def ms_deform_attn_forward(value: torch.Tensor, spatial_shapes: torch.Tensor, level_start_index: torch.Tensor,
                           sampling_loc: torch.Tensor, attn_weight: torch.Tensor, im2col_step: int = 64) -> torch.Tensor:
    """``detrex._C.ms_deform_attn_forward`` (vision.cpp:55): returns ``[B, Q, H*D]`` in value's dtype."""
    B, S, H, D, L, Q, P = _check_inputs(value, spatial_shapes, level_start_index, sampling_loc, attn_weight)
    value, sampling_loc, attn_weight = _aligned(value), _aligned(sampling_loc), _aligned(attn_weight)
    out = torch.empty((B, Q, H * D), dtype=value.dtype, device=value.device)
    stream = torch.cuda.current_stream(value.device).cuda_stream
    status = _lib.lib().msda_forward(ctypes.c_void_p(stream), _ptr(value), _ptr(spatial_shapes), _ptr(level_start_index),
                                     _ptr(sampling_loc), _ptr(attn_weight), B, S, H, D, L, Q, P, _ptr(out),
                                     _DTYPE_TAG[value.dtype], _flags(False))
    _lib.check(status, "ms_deform_attn_forward")
    return out


def ms_deform_attn_backward(value: torch.Tensor, spatial_shapes: torch.Tensor, level_start_index: torch.Tensor,
                            sampling_loc: torch.Tensor, attn_weight: torch.Tensor, grad_output: torch.Tensor,
                            im2col_step: int = 64) -> List[torch.Tensor]:
    """``detrex._C.ms_deform_attn_backward`` (vision.cpp:56): ``[grad_value, grad_sampling_loc, grad_attn_weight]``."""
    return _backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output, True)


def _backward(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, grad_output,
              need_grad_value: bool, tags=_DTYPE_TAG, flags=None) -> List[torch.Tensor]:
    """The backward behind ms_deform_attn_backward.  ``need_grad_value=False`` (the autograd Function passes it when
    ``value`` does not require grad, e.g. a frozen memory branch) returns ``None`` for ``grad_value`` and, on the
    shapes the fast kernels cover, skips its scatter -- the dominant cost of the backward -- altogether.  ``tags``:
    the accepted value dtypes (library-internal callers pass _VALUE_TAG to hand float16 over natively).  ``flags``:
    the MSDA_FLAG_* bits, ``_flags(True)`` when not given."""
    B, S, H, D, L, Q, P = _check_inputs(value, spatial_shapes, level_start_index, sampling_loc, attn_weight, tags)
    _require(grad_output.is_cuda and grad_output.device == value.device, "grad_output must be a CUDA tensor")
    _require(grad_output.dtype == value.dtype, "grad_output dtype must match value")
    _require(grad_output.numel() == B * Q * H * D, "grad_output must be [B, Q, H*D]")
    grad_output = _aligned(grad_output.contiguous())
    value, sampling_loc, attn_weight = _aligned(value), _aligned(sampling_loc), _aligned(attn_weight)
    grad_loc = torch.empty_like(sampling_loc)
    grad_w = torch.empty_like(attn_weight)
    flags = _flags(True) if flags is None else flags
    tag = tags[value.dtype]
    handle = _lib.lib()
    skip_scatter = (not need_grad_value and B * S * D > 0 and Q * L * P > 0
                    and b"_fast_" in handle.msda_dispatch_name(D, L, P, S, H, tag, flags, 1))
    if skip_scatter:
        status = handle.msda_backward(
            ctypes.c_void_p(torch.cuda.current_stream(value.device).cuda_stream), _ptr(grad_output), _ptr(value),
            _ptr(spatial_shapes), _ptr(level_start_index), _ptr(sampling_loc), _ptr(attn_weight), B, S, H, D, L, Q, P,
            ctypes.c_void_p(0), _ptr(grad_loc), _ptr(grad_w), ctypes.c_void_p(0), 0, tag,
            flags | _lib.FLAG_NO_GRAD_VALUE)
        _lib.check(status, "ms_deform_attn_backward")
        return [None, grad_loc, grad_w]
    grad_value = torch.empty_like(value)
    ws_bytes = int(handle.msda_backward_workspace_bytes(B, S, H, D, L, Q, P, tag, flags))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=value.device) if ws_bytes else None
    stream = torch.cuda.current_stream(value.device).cuda_stream
    status = handle.msda_backward(ctypes.c_void_p(stream), _ptr(grad_output), _ptr(value), _ptr(spatial_shapes),
                                  _ptr(level_start_index), _ptr(sampling_loc), _ptr(attn_weight), B, S, H, D, L, Q, P,
                                  _ptr(grad_value), _ptr(grad_loc), _ptr(grad_w),
                                  _ptr(ws) if ws is not None else ctypes.c_void_p(0), ws_bytes, tag, flags)
    _lib.check(status, "ms_deform_attn_backward")
    return [grad_value if need_grad_value else None, grad_loc, grad_w]


class MultiScaleDeformableAttnFunction(Function):
    """Same six-argument ``apply`` as the reference (multi_scale_deform_attn.py:44-54)."""

    @staticmethod
    def forward(ctx, value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights,
                im2col_step):
        ctx.im2col_step = im2col_step
        output = ms_deform_attn_forward(value, value_spatial_shapes, value_level_start_index, sampling_locations,
                                        attention_weights, ctx.im2col_step)
        ctx.save_for_backward(value, value_spatial_shapes, value_level_start_index, sampling_locations,
                              attention_weights)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights = ctx.saved_tensors
        grad_value, grad_sampling_loc, grad_attn_weight = _backward(
            value, value_spatial_shapes, value_level_start_index, sampling_locations, attention_weights, grad_output,
            need_grad_value=ctx.needs_input_grad[0])
        return grad_value, None, None, grad_sampling_loc, grad_attn_weight, None


def multi_scale_deformable_attn_pytorch(value: torch.Tensor, value_spatial_shapes: torch.Tensor,
                                        sampling_locations: torch.Tensor, attention_weights: torch.Tensor) -> torch.Tensor:
    """Same name, arguments and result as the reference's grid_sample formulation
    (/root/reference/detrex/layers/multi_scale_deform_attn.py:96-136), computed by the CUDA kernels: callers that
    import this function (the reference's tests do, tests/test_ms_deform_attn.py:20) keep working, differentiably.
    There is still no CPU path: CPU tensors raise.  ``level_start_index`` is derived on the device (no sync)."""
    _require(value.is_cuda, "Not implemented on the CPU")
    shapes = value_spatial_shapes.to(device=value.device, dtype=torch.int64).contiguous()
    sizes = shapes[:, 0] * shapes[:, 1]
    level_start_index = torch.cat((sizes.new_zeros((1,)), sizes.cumsum(0)[:-1]))
    return MultiScaleDeformableAttnFunction.apply(value.contiguous(), shapes, level_start_index,
                                                  sampling_locations.contiguous(), attention_weights.contiguous(), 64)


# ------------------------------------------------------------------------------------------------
# fused module path (SURVEY.md section 8f-1): softmax + sampling-location arithmetic inside the kernels
# ------------------------------------------------------------------------------------------------
def fused_supported(value: torch.Tensor, num_levels: int, num_points: int) -> bool:
    """True when the fused kernels cover this problem (fast-kernel shapes, float32 / bfloat16 / float16 value);
    otherwise the module composes the pre-op chain in PyTorch."""
    if not value.is_cuda or value.dtype not in _FUSED_DTYPES or value.dim() != 4:
        return False
    _, S, H, D = value.shape
    if not isinstance(S, int):
        # a dynamic value length under torch.compile: asked as 0, which leaves the 32-bit offset bound on S to the
        # kernels' entry points (they refuse a problem past it)
        S = 0
    return _fused_supported_dims(D, num_levels, num_points, S, H, _VALUE_TAG[value.dtype], _flags(False))


@torch.compiler.assume_constant_result
def _fused_supported_dims(D, L, P, S, H, tag, flags) -> bool:
    """Under torch.compile the answer is taken while the graph is built, for the traced shapes."""
    return bool(_lib.lib().msda_fused_supported(D, L, P, S, H, tag, flags))


def _mask_ptr(mask) -> ctypes.c_void_p:
    return _ptr(mask) if mask is not None else ctypes.c_void_p(0)


def _check_fused_inputs(value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, reference_points,
                        key_padding_mask):
    """Everything the kernels trust (they read the shapes as int64 and index with B/H/Q/L/P as given): the same
    checks _check_inputs makes for the plain operator (ms_deform_attn_cuda.cu:29-39), for the fused argument list."""
    _require(value.is_cuda, "Not implemented on the CPU")
    for name, t in (("value", value), ("sampling_offsets", sampling_offsets), ("attn_logits", attn_logits),
                    ("reference_points", reference_points), ("spatial_shapes", spatial_shapes),
                    ("level_start_index", level_start_index)):
        _require(t.is_cuda and t.device == value.device, f"{name} must be a CUDA tensor on {value.device}")
        _require(t.is_contiguous(), f"{name} tensor has to be contiguous")
    _require(value.dim() == 4, "value must be [B, S, H, D]")
    _require(value.dtype in _FUSED_DTYPES, f"unsupported value dtype {value.dtype} (float32, bfloat16, float16)")
    _require(sampling_offsets.dim() == 6 and sampling_offsets.shape[-1] == 2, "sampling_offsets must be [B, Q, H, L, P, 2]")
    B, S, H, D = value.shape
    Bq, Q, Hq, L, P, _ = sampling_offsets.shape
    _require(Bq == B and Hq == H, "sampling_offsets batch / heads do not match value")
    _require(spatial_shapes.dtype == torch.int64 and level_start_index.dtype == torch.int64,
             "spatial_shapes / level_start_index must be int64")
    _require(tuple(spatial_shapes.shape) == (L, 2) and tuple(level_start_index.shape) == (L,),
             "spatial_shapes must be [L, 2] and level_start_index [L]")
    _require(sampling_offsets.dtype == attn_logits.dtype, "sampling_offsets / attn_logits must share a dtype")
    tag = _aux_tag(value.dtype, sampling_offsets.dtype, "sampling_offsets / attn_logits")
    _require(reference_points.dtype == torch.float32, "reference_points must be float32")
    _require(tuple(attn_logits.shape) == (B, Q, H, L * P), "attn_logits must be [B, Q, H, L*P]")
    ref_dim = reference_points.shape[-1]
    _require(tuple(reference_points.shape) == (B, Q, L, ref_dim) and ref_dim in (2, 4),
             "reference_points must be [B, Q, L, 2 or 4]")
    mask = None
    if key_padding_mask is not None:
        _require(key_padding_mask.dtype in (torch.bool, torch.uint8), "key_padding_mask must be bool or uint8")
        _require(tuple(key_padding_mask.shape) == (B, S), "key_padding_mask must be [B, S]")
        _require(key_padding_mask.is_cuda and key_padding_mask.device == value.device,
                 f"key_padding_mask must be a CUDA tensor on {value.device}")
        mask = key_padding_mask.contiguous()   # one byte per pixel either way; non-zero = padded
    return (B, S, H, D, L, Q, P, ref_dim), mask, tag


def _fused_pre_ops(spatial_shapes, sampling_offsets, attn_logits, reference_points):
    """The module's own composition (multi_scale_deform_attn.py:300-332): softmax over L*P and the location affine."""
    B, Q, H, L, P, _ = sampling_offsets.shape
    weights = attn_logits.softmax(-1).view(B, Q, H, L, P)
    if reference_points.shape[-1] == 2:
        normalizer = torch.stack([spatial_shapes[..., 1], spatial_shapes[..., 0]], -1)
        loc = reference_points[:, :, None, :, None, :] + sampling_offsets / normalizer[None, None, None, :, None, :]
    else:
        loc = (reference_points[:, :, None, :, None, :2]
               + sampling_offsets / P * reference_points[:, :, None, :, None, 2:] * 0.5)
    return loc.contiguous(), weights.contiguous()


class MSDeformAttnFusedFunction(Function):
    """``apply(value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, reference_points,
    key_padding_mask=None)`` -> ``[B, Q, H*D]``.  ``sampling_offsets [B,Q,H,L,P,2]`` and ``attn_logits
    [B,Q,H,L*P]`` are the raw outputs of the module's two Linear layers: float32, or -- as autocast produces them --
    in value's dtype when that is bfloat16 / float16, and then their gradients come back in that dtype too (the float32
    gradients rounded once inside the kernel: the bits of the float32 route followed by a cast).  ``value`` is
    float32, bfloat16 or float16 (the output and ``grad_value`` share its dtype, accumulation is float32); ``reference_points
    [B,Q,L,2|4]`` float32.  Equivalent to softmax + location affine (multi_scale_deform_attn.py:300-332)
    followed by MultiScaleDeformableAttnFunction, without materialising locations / weights or their
    gradients.  With ``key_padding_mask [B,S]`` (bool or uint8, True = padded) it is additionally equivalent
    to ``value.masked_fill(key_padding_mask[..., None, None], 0)`` in front of that (py:291-292): ``value`` is
    passed unmasked, masked pixels read as zeros inside the kernels and receive a zero ``grad_value``.

    Deterministic mode (set_deterministic / torch.use_deterministic_algorithms): the forward is the same fused
    kernel (it has no atomics); the backward materialises locations / weights with the module's own PyTorch
    composition, runs the bit-reproducible unfused backward (MSDA_FLAG_DETERMINISTIC) and applies the chain
    rule through softmax / affine in PyTorch -- every step run-to-run reproducible."""

    @staticmethod
    def forward(ctx, value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, reference_points,
                key_padding_mask=None):
        out, saved, mask = _fused_forward(value, spatial_shapes, level_start_index, sampling_offsets, attn_logits,
                                          reference_points, key_padding_mask)
        ctx.save_for_backward(*saved)
        ctx.value_mask = mask
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        grad_value, grad_off, grad_logits, grad_ref = _fused_backward(
            grad_output, *ctx.saved_tensors, ctx.value_mask, _flags(True), ctx.needs_input_grad[0],
            ctx.needs_input_grad[5])
        return grad_value, None, None, grad_off, grad_logits, grad_ref, None


def _fused_forward(value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, reference_points,
                   key_padding_mask):
    """MSDeformAttnFusedFunction's forward (also the body of the ``ir_ads_b200::msda_fused`` op): the output, the
    aligned tensors its backward reads and the contiguous padding mask."""
    (B, S, H, D, L, Q, P, ref_dim), mask, tag = _check_fused_inputs(
        value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, reference_points, key_padding_mask)
    value, sampling_offsets, attn_logits, reference_points = (
        _aligned(value), _aligned(sampling_offsets), _aligned(attn_logits), _aligned(reference_points))
    out = torch.empty((B, Q, H * D), dtype=value.dtype, device=value.device)
    stream = torch.cuda.current_stream(value.device).cuda_stream
    status = _lib.lib().msda_fused_forward(
        ctypes.c_void_p(stream), _ptr(value), _ptr(spatial_shapes), _ptr(level_start_index), _ptr(sampling_offsets),
        _ptr(attn_logits), _ptr(reference_points), ref_dim, _mask_ptr(mask), B, S, H, D, L, Q, P, _ptr(out),
        tag, _flags(False))
    _lib.check(status, "msda_fused_forward")
    return out, (value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, reference_points), mask


def _fused_backward(grad_output, value, spatial_shapes, level_start_index, sampling_offsets, attn_logits,
                    reference_points, mask, flags, need_value, need_ref):
    """MSDeformAttnFusedFunction's backward (also the body of ``ir_ads_b200::msda_fused_backward``) under the
    MSDA_FLAG_* bits ``flags``: ``[grad_value, grad_offsets, grad_logits, grad_reference_points]``.  ``grad_value`` may
    be None when ``need_value`` is False; ``grad_reference_points`` is None unless ``need_ref``."""
    B, S, H, D = value.shape
    _, Q, _, L, P, _ = sampling_offsets.shape
    ref_dim = reference_points.shape[-1]
    _require(grad_output.is_cuda and grad_output.device == value.device, "grad_output must be a CUDA tensor")
    _require(grad_output.dtype == value.dtype, "grad_output dtype must match value")
    _require(grad_output.numel() == B * Q * H * D, "grad_output must be [B, Q, H*D]")
    grad_output = _aligned(grad_output.contiguous())
    value, sampling_offsets, attn_logits, reference_points = (
        _aligned(value), _aligned(sampling_offsets), _aligned(attn_logits), _aligned(reference_points))
    if (flags & _lib.FLAG_DETERMINISTIC) or need_ref:
        # Composition around the unfused backward: the deterministic mode, and the rare case of reference points
        # that require grad (DINO detaches them) -- d loc / d ref is the identity on (x, y) and off / P * 0.5 on
        # (w, h), taken from grad_sampling_loc itself so that boxes with w == 0 or h == 0 keep their (x, y) grad.
        # 16-bit offsets / logits are widened (exact) and the final gradients cast: the float32 route's bits.
        aux_dtype = sampling_offsets.dtype
        sampling_offsets, attn_logits = sampling_offsets.float(), attn_logits.float()
        loc, weights = _fused_pre_ops(spatial_shapes, sampling_offsets, attn_logits, reference_points)
        v = value if mask is None else value.masked_fill(mask.bool()[..., None, None], 0)
        grad_value, g_loc, g_w = _backward(v, spatial_shapes, level_start_index, loc, weights, grad_output,
                                           need_grad_value=need_value, tags=_VALUE_TAG, flags=flags)
        if grad_value is not None and mask is not None:
            grad_value = grad_value.masked_fill(mask.bool()[..., None, None], 0)
        g_w = g_w.view(B, Q, H, L * P)
        w_flat = weights.view(B, Q, H, L * P)
        grad_logits = w_flat * (g_w - (g_w * w_flat).sum(-1, keepdim=True))
        if ref_dim == 2:
            normalizer = torch.stack([spatial_shapes[..., 1], spatial_shapes[..., 0]], -1).to(g_loc.dtype)
            grad_off = g_loc / normalizer[None, None, None, :, None, :]
        else:
            grad_off = g_loc * (reference_points[:, :, None, :, None, 2:] * (0.5 / P))
        grad_ref = None
        if need_ref:
            g_xy = g_loc.sum(dim=(2, 4))
            grad_ref = g_xy if ref_dim == 2 else torch.cat(
                [g_xy, (g_loc * sampling_offsets * (0.5 / P)).sum(dim=(2, 4))], -1)
        return grad_value, grad_off.to(aux_dtype), grad_logits.to(aux_dtype), grad_ref
    grad_value = torch.empty_like(value)
    grad_off = torch.empty_like(sampling_offsets)
    grad_logits = torch.empty_like(attn_logits)
    tag = _aux_tag(value.dtype, sampling_offsets.dtype, "sampling_offsets / attn_logits")
    handle = _lib.lib()
    ws_bytes = int(handle.msda_backward_workspace_bytes(B, S, H, D, L, Q, P, tag, flags))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=value.device) if ws_bytes else None
    stream = torch.cuda.current_stream(value.device).cuda_stream
    status = handle.msda_fused_backward(
        ctypes.c_void_p(stream), _ptr(grad_output), _ptr(value), _ptr(spatial_shapes), _ptr(level_start_index),
        _ptr(sampling_offsets), _ptr(attn_logits), _ptr(reference_points), ref_dim, _mask_ptr(mask),
        B, S, H, D, L, Q, P, _ptr(grad_value), _ptr(grad_off), _ptr(grad_logits),
        _ptr(ws) if ws is not None else ctypes.c_void_p(0), ws_bytes, tag, flags)
    _lib.check(status, "msda_fused_backward")
    return grad_value, grad_off, grad_logits, None


def debug_bookkeeping(sampling_loc: torch.Tensor, spatial_shapes: torch.Tensor, level_start_index: torch.Tensor,
                      spatial_size: int, channels: int):
    """Integer bookkeeping of the float kernels (test hook, see include/msda.h)."""
    B, Q, H, L, P, _ = sampling_loc.shape
    n = B * Q * H * L * P
    offs = torch.empty((n, 4), dtype=torch.int64, device=sampling_loc.device)
    frac = torch.empty((n, 2), dtype=torch.float32, device=sampling_loc.device)
    stream = torch.cuda.current_stream(sampling_loc.device).cuda_stream
    status = _lib.lib().msda_debug_bookkeeping(ctypes.c_void_p(stream), _ptr(sampling_loc.contiguous()),
                                               _ptr(spatial_shapes), _ptr(level_start_index), B, spatial_size, H,
                                               channels, L, Q, P, _ptr(offs), _ptr(frac))
    _lib.check(status, "msda_debug_bookkeeping")
    return offs, frac


# ------------------------------------------------------------------------------------------------
# packed (padding-free) batches of the fused module path: ir_ads_b200/packing.py, include/msda.h msda_packed_*
# ------------------------------------------------------------------------------------------------
def _check_packed_inputs(value, sampling_offsets, attn_logits, reference_points, packing):
    _require(value.is_cuda, "Not implemented on the CPU")
    for name, t in (("value", value), ("sampling_offsets", sampling_offsets), ("attn_logits", attn_logits),
                    ("reference_points", reference_points), ("packing.meta", packing.meta),
                    ("packing.spatial_shapes", packing.spatial_shapes)):
        _require(t.is_cuda and t.device == value.device, f"{name} must be a CUDA tensor on {value.device}")
        _require(t.is_contiguous(), f"{name} tensor has to be contiguous")
    _require(value.dim() == 3, "value must be [T_v, H, D]")
    _require(value.dtype in _FUSED_DTYPES, f"unsupported value dtype {value.dtype} (float32, bfloat16, float16)")
    T_v, H, D = value.shape
    L = packing.num_levels
    _require(T_v == packing.total_value, f"value has {T_v} rows, the packing {packing.total_value}")
    _require(sampling_offsets.dim() == 5 and sampling_offsets.shape[-1] == 2, "sampling_offsets must be [T_q, H, L, P, 2]")
    T_q, Hq, Lq, P, _ = sampling_offsets.shape
    _require(Hq == H and Lq == L, "sampling_offsets heads / levels do not match value / packing")
    _require(T_q == packing.total_query, f"{T_q} query rows, the packing has {packing.total_query}")
    _require(sampling_offsets.dtype == attn_logits.dtype, "sampling_offsets / attn_logits must share a dtype")
    tag = _aux_tag(value.dtype, sampling_offsets.dtype, "sampling_offsets / attn_logits")
    _require(tuple(attn_logits.shape) == (T_q, H, L * P), "attn_logits must be [T_q, H, L*P]")
    _require(reference_points.dtype == torch.float32, "reference_points must be float32")
    ref_dim = reference_points.shape[-1]
    _require(tuple(reference_points.shape) == (T_q, L, ref_dim) and ref_dim in (2, 4),
             "reference_points must be [T_q, L, 2 or 4]")
    return (T_v, H, D, L, T_q, P, ref_dim), tag


class MSDeformAttnPackedFunction(Function):
    """``apply(value, sampling_offsets, attn_logits, reference_points, packing)`` -> ``[T_q, H*D]``: the fused module
    path over a packed batch (``packing``: an ``ir_ads_b200.packing.PackedLevels``).  ``value [T_v, H, D]``,
    ``sampling_offsets [T_q, H, L, P, 2]``, ``attn_logits [T_q, H, L*P]``, ``reference_points [T_q, L, 2|4]``, dtypes
    as MSDeformAttnFusedFunction.  Every query row gets the bits MSDeformAttnFusedFunction gives for the padded batch
    with ``packing.padding_mask`` as key_padding_mask (output, offset and logit gradients); ``grad_value`` equals its
    valid rows up to the order of the float reds.

    Two cases leave the packed kernels: deterministic mode and ``reference_points`` that require grad.  Their backward
    unpacks into the padded layout, runs MSDeformAttnFusedFunction's backward there and packs the gradients -- the bits
    of the padded route (padding query rows get a zero output gradient)."""

    @staticmethod
    def forward(ctx, value, sampling_offsets, attn_logits, reference_points, packing):
        out, saved = _packed_forward(value, sampling_offsets, attn_logits, reference_points, packing)
        ctx.save_for_backward(*saved)
        ctx.packing = packing
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        return _packed_backward(grad_output, *ctx.saved_tensors, ctx.packing, _flags(True), ctx.needs_input_grad[:4])


def _packed_forward(value, sampling_offsets, attn_logits, reference_points, packing):
    """MSDeformAttnPackedFunction's forward (also the body of ``ir_ads_b200::msda_packed``): the output and the
    aligned tensors its backward reads."""
    (T_v, H, D, L, T_q, P, ref_dim), tag = _check_packed_inputs(value, sampling_offsets, attn_logits,
                                                                reference_points, packing)
    value, sampling_offsets, attn_logits, reference_points = (
        _aligned(value), _aligned(sampling_offsets), _aligned(attn_logits), _aligned(reference_points))
    out = torch.empty((T_q, H * D), dtype=value.dtype, device=value.device)
    stream = torch.cuda.current_stream(value.device).cuda_stream
    status = _lib.lib().msda_packed_forward(
        ctypes.c_void_p(stream), _ptr(value), _ptr(packing.spatial_shapes), _ptr(packing.meta),
        _ptr(sampling_offsets), _ptr(attn_logits), _ptr(reference_points), ref_dim, packing.batch, T_v, H, D, L,
        T_q, P, packing.max_value, packing.max_query, _ptr(out), tag, _flags(False))
    _lib.check(status, "msda_packed_forward")
    return out, (value, sampling_offsets, attn_logits, reference_points)


def _packed_backward(grad_output, value, sampling_offsets, attn_logits, reference_points, packing, flags, needs):
    """MSDeformAttnPackedFunction's backward (also the body of ``ir_ads_b200::msda_packed_backward``) under the
    MSDA_FLAG_* bits ``flags``; ``needs``: which of value, offsets, logits and reference points want a gradient.
    Returns ``(grad_value, grad_offsets, grad_logits, grad_reference_points, None)``."""
    T_v, H, D = value.shape
    T_q, _, L, P, _ = sampling_offsets.shape
    ref_dim = reference_points.shape[-1]
    _require(grad_output.is_cuda and grad_output.device == value.device, "grad_output must be a CUDA tensor")
    _require(grad_output.dtype == value.dtype, "grad_output dtype must match value")
    _require(grad_output.numel() == T_q * H * D, "grad_output must be [T_q, H*D]")
    grad_output = _aligned(grad_output.contiguous())
    value, sampling_offsets, attn_logits, reference_points = (
        _aligned(value), _aligned(sampling_offsets), _aligned(attn_logits), _aligned(reference_points))
    if (flags & _lib.FLAG_DETERMINISTIC) or needs[3]:
        return _packed_backward_padded(value, sampling_offsets, attn_logits, reference_points, grad_output,
                                       packing, flags, needs)
    grad_value = torch.empty_like(value)
    grad_off = torch.empty_like(sampling_offsets)
    grad_logits = torch.empty_like(attn_logits)
    tag = _aux_tag(value.dtype, sampling_offsets.dtype, "sampling_offsets / attn_logits")
    handle = _lib.lib()
    ws_bytes = int(handle.msda_packed_backward_workspace_bytes(T_v, H, D, tag, flags))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=value.device) if ws_bytes else None
    stream = torch.cuda.current_stream(value.device).cuda_stream
    status = handle.msda_packed_backward(
        ctypes.c_void_p(stream), _ptr(grad_output), _ptr(value), _ptr(packing.spatial_shapes), _ptr(packing.meta),
        _ptr(sampling_offsets), _ptr(attn_logits), _ptr(reference_points), ref_dim, packing.batch, T_v, H, D, L,
        T_q, P, packing.max_value, packing.max_query, _ptr(grad_value), _ptr(grad_off), _ptr(grad_logits),
        _ptr(ws) if ws is not None else ctypes.c_void_p(0), ws_bytes, tag, flags)
    _lib.check(status, "msda_packed_backward")
    return grad_value, grad_off, grad_logits, None, None


def _packed_backward_padded(value, sampling_offsets, attn_logits, reference_points, grad_output, packing, flags,
                            needs):
    """Backward of MSDeformAttnPackedFunction through the padded layout: unpack, MSDeformAttnFusedFunction's own
    backward (deterministic composition, reference-point gradient), pack the gradients."""
    from .packing import unpack_tokens
    v, mask = unpack_tokens(value, packing)
    off = unpack_tokens(sampling_offsets, packing, queries=True)[0]
    lg = unpack_tokens(attn_logits, packing, queries=True)[0]
    ref = unpack_tokens(reference_points, packing, queries=True)[0]
    go = unpack_tokens(grad_output, packing, queries=True)[0]
    got = _fused_backward(go, v, packing.spatial_shapes, packing.level_start_index, off, lg, ref, mask, flags,
                          bool(needs[0]), bool(needs[3]))

    def pack(g, index, need):
        return None if g is None or not need else g.reshape((-1,) + tuple(g.shape[2:])).index_select(0, index)

    return (pack(got[0], packing.value_index, needs[0]), pack(got[1], packing.query_index, needs[1]),
            pack(got[2], packing.query_index, needs[2]), pack(got[3], packing.query_index, needs[3]), None)

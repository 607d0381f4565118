"""DCNv3 core op on the sm_100a gather/scatter kernels (SURVEY.md section 8f-4).

Mirrors the reference's ``DCNv3Function`` and the ``detrex._C.dcnv3_forward / dcnv3_backward`` pair
(/root/reference/detrex/layers/dcn_v3.py:21-65, detrex/layers/csrc/vision.cpp:57-58,
detrex/layers/csrc/DCNv3/dcnv3_cuda.cu): same argument order, channels-last tensors, autograd for
input / offset / mask.  DCNv3 is MSDeformAttn with one level, K = kernel_h*kernel_w points whose
positions come from a convolution-style grid, and groups in the role of heads -- so it runs on the
same kernels with a different record-building phase (ir_ads_b200/csrc/msda_fast.cuh, PRE == 2).

Fast path: group_channels in {16, 32, 64, 128}, K <= 64, float32 / bfloat16 / float16 input (float16 and bfloat16
are widened exactly inside the kernels, accumulation is float32).  Every other shape / dtype the reference dispatches
(any channel count, float64: detrex/layers/csrc/DCNv3/dcnv3_cuda.cu:66-80 uses AT_DISPATCH_FLOATING_TYPES_AND_HALF)
runs as a composition on the GENERIC MSDeformAttn kernels (csrc/msda_generic.cuh, any D, float32 / float64): the convolution-grid sampling positions
are formed with the reference kernel's arithmetic in PyTorch, normalised, and handed to
MultiScaleDeformableAttnFunction with one level -- still CUDA only, still no CPU path.

The ``DCNv3`` module runs its mask softmax inside the kernels on the fast shapes (``DCNv3FusedFunction``, PRE == 3):
the kernels take the mask Linear's raw logits, so the mask and its gradient never reach HBM.  Elsewhere it composes
``F.softmax`` and ``DCNv3Function`` as the reference does.
"""
from __future__ import annotations

import ctypes
from typing import List

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib
from . import functional
from .functional import _aligned, _ptr, _require

_DCN_TAG = {torch.float32: _lib.MSDA_F32, torch.bfloat16: _lib.MSDA_BF16, torch.float16: _lib.MSDA_F16}


def _declare(handle):
    if getattr(handle, "_dcn_declared", False):
        return handle
    vp, i, u, sz, f = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint, ctypes.c_size_t, ctypes.c_float
    handle.msda_dcnv3_forward.restype = i
    handle.msda_dcnv3_forward.argtypes = [vp, vp, vp, vp] + [i] * 10 + [f] + [i] * 5 + [vp, i, u]
    handle.msda_dcnv3_backward.restype = i
    handle.msda_dcnv3_backward.argtypes = [vp, vp, vp, vp, vp] + [i] * 10 + [f] + [i] * 5 + [vp, vp, vp, vp, sz, i, u]
    handle.msda_dcnv3_backward_workspace_bytes.restype = sz
    handle.msda_dcnv3_backward_workspace_bytes.argtypes = [i] * 10 + [u]
    # fused module path: the same signatures, mask logits in place of the mask
    handle.msda_dcnv3_fused_forward.restype = i
    handle.msda_dcnv3_fused_forward.argtypes = handle.msda_dcnv3_forward.argtypes
    handle.msda_dcnv3_fused_backward.restype = i
    handle.msda_dcnv3_fused_backward.argtypes = handle.msda_dcnv3_backward.argtypes
    handle._dcn_declared = True
    return handle


def _geometry(input, offset, mask, kernel_h, kernel_w, group, group_channels, aux_checked=False):
    _require(input.is_cuda, "Not implemented on the CPU")
    for name, t in (("input", input), ("offset", offset), ("mask", mask)):
        _require(t.is_cuda and t.device == input.device, f"{name} must be a CUDA tensor on {input.device}")
        _require(t.is_contiguous(), f"{name} tensor has to be contiguous")
    _require(input.dim() == 4 and offset.dim() == 4 and mask.dim() == 4, "input / offset / mask must be 4-d (N,H,W,C)")
    N, H_in, W_in, C = input.shape
    _, H_out, W_out, _ = offset.shape
    K = kernel_h * kernel_w
    _require(C == group * group_channels, f"input channels {C} != group*group_channels {group * group_channels}")
    _require(tuple(offset.shape) == (N, H_out, W_out, group * K * 2), "offset must be [N, H_out, W_out, group*K*2]")
    _require(tuple(mask.shape) == (N, H_out, W_out, group * K), "mask must be [N, H_out, W_out, group*K]")
    _require(input.dtype in _DCN_TAG, f"unsupported input dtype {input.dtype}")
    # float16 offset / mask as well: the reference's _C takes them in the input's dtype (dcnv3_cuda.cu:66-80)
    _require(aux_checked or (offset.dtype in (torch.float32, torch.float16) and mask.dtype in (torch.float32, torch.float16)),
             "offset / mask must be float32 or float16")
    return N, H_in, W_in, H_out, W_out


def dcnv3_forward(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                  group, group_channels, offset_scale, im2col_step=256) -> torch.Tensor:
    """``detrex._C.dcnv3_forward``: returns ``[N, H_out, W_out, group*group_channels]``."""
    N, H_in, W_in, H_out, W_out = _geometry(input, offset, mask, kernel_h, kernel_w, group, group_channels)
    input, offset, mask = _aligned(input), _aligned(offset.float()), _aligned(mask.float())
    out = torch.empty((N, H_out, W_out, group * group_channels), dtype=input.dtype, device=input.device)
    stream = torch.cuda.current_stream(input.device).cuda_stream
    status = _declare(_lib.lib()).msda_dcnv3_forward(
        ctypes.c_void_p(stream), _ptr(input), _ptr(offset), _ptr(mask), kernel_h, kernel_w, stride_h, stride_w, pad_h,
        pad_w, dilation_h, dilation_w, group, group_channels, float(offset_scale), N, H_in, W_in, H_out, W_out,
        _ptr(out), _DCN_TAG[input.dtype], 0)
    _lib.check(status, "dcnv3_forward")
    return out


def dcnv3_backward(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                   group, group_channels, offset_scale, grad_output, im2col_step=256) -> List[torch.Tensor]:
    """``detrex._C.dcnv3_backward``: ``[grad_input, grad_offset, grad_mask]``, each in the dtype of its input (the
    offset / mask gradients are computed in float32).  Under ``set_deterministic(True)`` or
    ``torch.use_deterministic_algorithms(True)`` grad_input is bit-reproducible (MSDA_FLAG_DETERMINISTIC); grad_offset
    and grad_mask are the same bits either way."""
    return _dcnv3_backward(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                           dilation_w, group, group_channels, offset_scale, grad_output, functional._flags(True))


def _dcnv3_backward(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                    group, group_channels, offset_scale, grad_output, flags) -> List[torch.Tensor]:
    """dcnv3_backward under the MSDA_FLAG_* bits ``flags``."""
    N, H_in, W_in, H_out, W_out = _geometry(input, offset, mask, kernel_h, kernel_w, group, group_channels)
    _require(grad_output.is_cuda and grad_output.dtype == input.dtype, "grad_output must match input's device / dtype")
    grad_output = _aligned(grad_output.contiguous())
    off_dtype, mask_dtype = offset.dtype, mask.dtype
    input, offset, mask = _aligned(input), _aligned(offset.float()), _aligned(mask.float())
    grad_input = torch.empty_like(input)
    grad_offset = torch.empty_like(offset)
    grad_mask = torch.empty_like(mask)
    tag = _DCN_TAG[input.dtype]
    handle = _declare(_lib.lib())
    ws_bytes = handle.msda_dcnv3_backward_workspace_bytes(kernel_h, kernel_w, group, group_channels, N, H_in, W_in,
                                                          H_out, W_out, tag, flags)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=input.device) if ws_bytes else None
    stream = torch.cuda.current_stream(input.device).cuda_stream
    status = handle.msda_dcnv3_backward(
        ctypes.c_void_p(stream), _ptr(grad_output), _ptr(input), _ptr(offset), _ptr(mask), kernel_h, kernel_w,
        stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels, float(offset_scale), N, H_in,
        W_in, H_out, W_out, _ptr(grad_input), _ptr(grad_offset), _ptr(grad_mask),
        _ptr(ws) if ws is not None else ctypes.c_void_p(0), ws_bytes, tag, flags)
    _lib.check(status, "dcnv3_backward")
    return [grad_input, grad_offset.to(off_dtype), grad_mask.to(mask_dtype)]


def fast_supported(input: torch.Tensor, kernel_h: int, kernel_w: int, group_channels: int) -> bool:
    """The shapes / dtypes the DCN record mode of the fast kernels covers."""
    return (group_channels in (16, 32, 64, 128) and 1 <= kernel_h * kernel_w <= 64
            and input.dtype in (torch.float32, torch.bfloat16, torch.float16))


def dcnv3_composed(input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                   group, group_channels, offset_scale) -> torch.Tensor:
    """DCNv3 as ONE-LEVEL MSDeformAttn on the generic kernels, differentiable through autograd.  Sampling position of
    kernel point (i, j) for output pixel (ho, wo), in input-pixel units (dcnv3_im2col_cuda.cuh:232-260):
        x = (cw - pad_w + wo*stride_w) - cw*scale + (i*dil_w + off_x)*scale,   cw = dil_w*(kernel_w-1)//2   (y alike)
    MSDeformAttn samples at loc*size - 0.5, so loc = (x + 0.5) / W_in."""
    from .functional import MultiScaleDeformableAttnFunction
    _require(input.is_cuda, "Not implemented on the CPU")
    N, H_in, W_in, C = input.shape
    _, H_out, W_out, _ = offset.shape
    K = kernel_h * kernel_w
    _require(C == group * group_channels, f"input channels {C} != group*group_channels {group * group_channels}")
    _require(tuple(offset.shape) == (N, H_out, W_out, group * K * 2), "offset must be [N, H_out, W_out, group*K*2]")
    _require(tuple(mask.shape) == (N, H_out, W_out, group * K), "mask must be [N, H_out, W_out, group*K]")
    cdt = torch.float64 if input.dtype == torch.float64 else torch.float32
    dev = input.device
    value = input.to(cdt).reshape(N, H_in * W_in, group, group_channels)
    off = offset.to(cdt).reshape(N, H_out, W_out, group, K, 2)
    cw, ch = (dilation_w * (kernel_w - 1)) // 2, (dilation_h * (kernel_h - 1)) // 2
    pt = torch.arange(K, device=dev)
    i, j = (pt // kernel_h).to(cdt), (pt % kernel_h).to(cdt)                 # point index = i*kernel_h + j, i over kernel_w
    wo = torch.arange(W_out, device=dev, dtype=cdt).view(1, 1, W_out, 1, 1)
    ho = torch.arange(H_out, device=dev, dtype=cdt).view(1, H_out, 1, 1, 1)
    x = (cw - pad_w + wo * stride_w) - cw * offset_scale + (i * dilation_w + off[..., 0]) * offset_scale
    y = (ch - pad_h + ho * stride_h) - ch * offset_scale + (j * dilation_h + off[..., 1]) * offset_scale
    loc = torch.stack([(x + 0.5) / W_in, (y + 0.5) / H_in], -1).reshape(N, H_out * W_out, group, 1, K, 2)
    w = mask.to(cdt).reshape(N, H_out * W_out, group, 1, K)
    shapes = torch.tensor([[H_in, W_in]], dtype=torch.long, device=dev)
    lsi = torch.zeros(1, dtype=torch.long, device=dev)
    out = MultiScaleDeformableAttnFunction.apply(value.contiguous(), shapes, lsi, loc.contiguous(), w.contiguous(), 64)
    return out.reshape(N, H_out, W_out, C).to(input.dtype)


class DCNv3Function(Function):
    """Same 15-argument ``apply`` as the reference (dcn_v3.py:21-65)."""

    @staticmethod
    def forward(ctx, input, offset, mask, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w,
                group, group_channels, offset_scale, im2col_step):
        ctx.args = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels,
                    offset_scale)
        ctx.im2col_step = im2col_step
        ctx.composed = None
        if not fast_supported(input, kernel_h, kernel_w, group_channels):
            # any other channel count / float64: the composition on the generic kernels, graph kept for backward
            with torch.enable_grad():
                leaves = [t.detach().requires_grad_(True) for t in (input, offset, mask)]
                out = dcnv3_composed(*leaves, *ctx.args)
            ctx.composed = (leaves, out)
            return out.detach()
        output = dcnv3_forward(input, offset.float(), mask.float(), *ctx.args, im2col_step)
        ctx.save_for_backward(input, offset, mask)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        if ctx.composed is not None:
            leaves, out = ctx.composed
            ctx.composed = None
            return tuple(torch.autograd.grad(out, leaves, grad_output.to(out.dtype))) + (None,) * 12
        input, offset, mask = ctx.saved_tensors
        gi, go, gm = dcnv3_backward(input, offset.float(), mask.float(), *ctx.args, grad_output.to(input.dtype),
                                    ctx.im2col_step)
        return (gi, go.to(offset.dtype), gm.to(mask.dtype)) + (None,) * 12


# ------------------------------------------------------------------------------------------------
# fused module path: the DCNv3 module's mask softmax inside the kernels (csrc/msda_fast.cuh, PRE == 3)
# ------------------------------------------------------------------------------------------------
def _fused_geometry(input, offset, mask_logits, kernel_h, kernel_w, group, group_channels):
    """The problem's dimensions and its dtype tag: offset / mask_logits float32, or both in the input's own 16-bit
    type (the module's Linear outputs under autocast; MSDA_*_AUX16)."""
    _require(input.dtype in _DCN_TAG, f"unsupported input dtype {input.dtype}")
    _require(offset.dtype == mask_logits.dtype, "offset / mask_logits must share a dtype")
    tag = functional._aux_tag(input.dtype, offset.dtype, "offset / mask_logits")
    dims = _geometry(input, offset, mask_logits, kernel_h, kernel_w, group, group_channels, aux_checked=True)
    _require(fast_supported(input, kernel_h, kernel_w, group_channels),
             f"fused DCNv3 needs group_channels in {{16, 32, 64, 128}}, kernel_h*kernel_w <= 64 and a float32 / "
             f"bfloat16 / float16 input (got {group_channels}, {kernel_h * kernel_w}, {input.dtype})")
    return dims, tag


def dcnv3_fused_forward(input, offset, mask_logits, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                        dilation_w, group, group_channels, offset_scale) -> torch.Tensor:
    """``dcnv3_forward`` with ``mask = softmax(mask_logits)`` over each (pixel, group) row of K, the softmax done inside
    the kernel (``msda_dcnv3_fused_forward``).  ``offset`` / ``mask_logits`` are float32, or both in the input's
    16-bit dtype."""
    (N, H_in, W_in, H_out, W_out), tag = _fused_geometry(input, offset, mask_logits, kernel_h, kernel_w, group,
                                                         group_channels)
    input, offset, mask_logits = _aligned(input), _aligned(offset), _aligned(mask_logits)
    out = torch.empty((N, H_out, W_out, group * group_channels), dtype=input.dtype, device=input.device)
    stream = torch.cuda.current_stream(input.device).cuda_stream
    status = _declare(_lib.lib()).msda_dcnv3_fused_forward(
        ctypes.c_void_p(stream), _ptr(input), _ptr(offset), _ptr(mask_logits), kernel_h, kernel_w, stride_h, stride_w,
        pad_h, pad_w, dilation_h, dilation_w, group, group_channels, float(offset_scale), N, H_in, W_in, H_out, W_out,
        _ptr(out), tag, 0)
    _lib.check(status, "dcnv3_fused_forward")
    return out


def dcnv3_fused_backward(input, offset, mask_logits, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                         dilation_w, group, group_channels, offset_scale, grad_output) -> List[torch.Tensor]:
    """``[grad_input, grad_offset, grad_mask_logits]`` of ``dcnv3_fused_forward``: float reds, the softmax's chain rule
    inside the kernel (``msda_dcnv3_fused_backward``).  There is no deterministic form; ``DCNv3FusedFunction``
    composes one.  The offset / logit gradients come back in the dtype of offset / mask_logits."""
    (N, H_in, W_in, H_out, W_out), tag = _fused_geometry(input, offset, mask_logits, kernel_h, kernel_w, group,
                                                         group_channels)
    _require(grad_output.is_cuda and grad_output.dtype == input.dtype, "grad_output must match input's device / dtype")
    grad_output = _aligned(grad_output.contiguous())
    input, offset, mask_logits = _aligned(input), _aligned(offset), _aligned(mask_logits)
    grad_input = torch.empty_like(input)
    grad_offset = torch.empty_like(offset)
    grad_logits = torch.empty_like(mask_logits)
    handle = _declare(_lib.lib())
    ws_bytes = handle.msda_dcnv3_backward_workspace_bytes(kernel_h, kernel_w, group, group_channels, N, H_in, W_in,
                                                          H_out, W_out, tag, 0)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=input.device) if ws_bytes else None
    stream = torch.cuda.current_stream(input.device).cuda_stream
    status = handle.msda_dcnv3_fused_backward(
        ctypes.c_void_p(stream), _ptr(grad_output), _ptr(input), _ptr(offset), _ptr(mask_logits), kernel_h, kernel_w,
        stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels, float(offset_scale), N, H_in,
        W_in, H_out, W_out, _ptr(grad_input), _ptr(grad_offset), _ptr(grad_logits),
        _ptr(ws) if ws is not None else ctypes.c_void_p(0), ws_bytes, tag, 0)
    _lib.check(status, "dcnv3_fused_backward")
    return [grad_input, grad_offset, grad_logits]


class DCNv3FusedFunction(Function):
    """``apply(input, offset, mask_logits, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
    dilation_w, group, group_channels, offset_scale, im2col_step)``: ``DCNv3Function`` with the mask replaced by its
    pre-softmax logits ``[N, H_out, W_out, group*K]`` -- the DCNv3 module's ``softmax(mask(x1).reshape(..., group,
    K), -1)`` runs inside the kernels, so the mask and its gradient never reach HBM.  Gradients for ``input``,
    ``offset`` and ``mask_logits``.  ``offset`` / ``mask_logits`` are float32, or -- as autocast produces them -- both
    in the input's dtype when that is bfloat16 / float16, and their gradients then come back in that dtype (the
    float32 gradients rounded once inside the kernel); ``input`` is float32, bfloat16 or float16 on the fast-kernel
    shapes (``fast_supported``) -- anything else raises, the module composes instead.

    Deterministic mode (set_deterministic / torch.use_deterministic_algorithms), as MSDeformAttnFusedFunction: the
    forward is the same fused kernel (it has no atomics); the backward forms the mask with torch.softmax, runs the
    bit-reproducible ``dcnv3_backward`` and applies the softmax's chain rule with torch's own softmax backward -- the
    same bits as ``torch.softmax`` followed by ``DCNv3Function`` in deterministic mode."""

    @staticmethod
    def forward(ctx, input, offset, mask_logits, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h,
                dilation_w, group, group_channels, offset_scale, im2col_step):
        ctx.args = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels,
                    offset_scale)
        ctx.im2col_step = im2col_step
        output = dcnv3_fused_forward(input, offset, mask_logits, *ctx.args)
        ctx.save_for_backward(input, offset, mask_logits)
        return output

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_output):
        input, offset, mask_logits = ctx.saved_tensors
        return tuple(_dcnv3_fused_backward_route(input, offset, mask_logits, ctx.args, grad_output,
                                                 functional._flags(True))) + (None,) * 12


def _dcnv3_fused_backward_route(input, offset, mask_logits, args, grad_output, flags):
    """DCNv3FusedFunction's backward (also the body of ``ir_ads_b200::dcnv3_fused_backward``) under the MSDA_FLAG_*
    bits ``flags``; ``args``: the eleven geometry arguments.  ``[grad_input, grad_offset, grad_mask_logits]``."""
    grad_output = grad_output.to(input.dtype)
    if not flags & _lib.FLAG_DETERMINISTIC:
        return dcnv3_fused_backward(input, offset, mask_logits, *args, grad_output)
    # 16-bit offset / logits are widened (exact) and the final gradients cast: the float32 route's bits
    # The softmax's chain rule is the kernel autograd's SoftmaxBackward runs, called directly: inside a custom op
    # (ir_ads_b200/ops.py) autograd is switched off below the dispatcher, and torch.enable_grad does not restore it.
    aux_dtype = offset.dtype
    N, H_out, W_out, _ = mask_logits.shape
    mask = torch.softmax(mask_logits.detach().float().view(N, H_out, W_out, args[8], -1), -1)
    gi, go, gm = _dcnv3_backward(input, offset.float(), mask.view(N, H_out, W_out, -1), *args, grad_output, flags)
    g_logits = torch._softmax_backward_data(gm.view_as(mask), mask, -1, torch.float32)
    return [gi, go.to(aux_dtype), g_logits.view_as(mask_logits).to(aux_dtype)]


# ------------------------------------------------------------------------------------------------
# the DCNv3 operator module (InternImage), same constructor / parameter names as the reference
# (/root/reference/detrex/layers/dcn_v3.py:373-500) so InternImage checkpoints load
# ------------------------------------------------------------------------------------------------
import torch.nn as nn  # noqa: E402
import torch.nn.functional as F  # noqa: E402


class _Permute(nn.Module):
    def __init__(self, *dims):
        super().__init__()
        self.dims = dims

    def forward(self, x):
        return x.permute(*self.dims)


def _norm_layer(dim, kind, in_format, out_format, eps=1e-6):
    """Sequential with the reference's slot layout (dcn_v3.py:192-214), so ``dw_conv.1.<k>.weight`` keys match."""
    layers = []
    if kind == "BN":
        if in_format == "channels_last":
            layers.append(_Permute(0, 3, 1, 2))
        layers.append(nn.BatchNorm2d(dim))
        if out_format == "channels_last":
            layers.append(_Permute(0, 2, 3, 1))
    elif kind == "LN":
        if in_format == "channels_first":
            layers.append(_Permute(0, 2, 3, 1))
        layers.append(nn.LayerNorm(dim, eps=eps))
        if out_format == "channels_first":
            layers.append(_Permute(0, 3, 1, 2))
    else:
        raise NotImplementedError(f"norm layer {kind!r}")
    return nn.Sequential(*layers)


def _act_layer(kind):
    if kind == "ReLU":
        return nn.ReLU(inplace=True)
    if kind == "SiLU":
        return nn.SiLU(inplace=True)
    if kind == "GELU":
        return nn.GELU()
    raise NotImplementedError(f"activation {kind!r}")


class DCNv3(nn.Module):
    """input (N, H, W, C) -> output (N, H, W, C): input projection, depth-wise conv branch producing offsets and
    softmax-normalised masks per group, the DCNv3 core op, optional centre-feature blending, output projection."""

    def __init__(self, channels=64, kernel_size=3, dw_kernel_size=None, stride=1, pad=1, dilation=1, group=4,
                 offset_scale=1.0, act_layer="GELU", norm_layer="LN", center_feature_scale=False):
        super().__init__()
        if channels % group != 0:
            raise ValueError(f"channels must be divisible by group, but got {channels} and {group}")
        dw_kernel_size = dw_kernel_size if dw_kernel_size is not None else kernel_size
        self.offset_scale = offset_scale
        self.channels = channels
        self.kernel_size = kernel_size
        self.dw_kernel_size = dw_kernel_size
        self.stride = stride
        self.dilation = dilation
        self.pad = pad
        self.group = group
        self.group_channels = channels // group
        self.center_feature_scale = center_feature_scale
        self.dw_conv = nn.Sequential(
            nn.Conv2d(channels, channels, kernel_size=dw_kernel_size, stride=1, padding=(dw_kernel_size - 1) // 2,
                      groups=channels),
            _norm_layer(channels, norm_layer, "channels_first", "channels_last"),
            _act_layer(act_layer))
        self.offset = nn.Linear(channels, group * kernel_size * kernel_size * 2)
        self.mask = nn.Linear(channels, group * kernel_size * kernel_size)
        self.input_proj = nn.Linear(channels, channels)
        self.output_proj = nn.Linear(channels, channels)
        self._reset_parameters()
        if center_feature_scale:
            self.center_feature_scale_proj_weight = nn.Parameter(torch.zeros((group, channels), dtype=torch.float))
            self.center_feature_scale_proj_bias = nn.Parameter(torch.zeros((group,), dtype=torch.float))

    def _reset_parameters(self):
        for lin in (self.offset, self.mask):
            nn.init.constant_(lin.weight.data, 0.0)
            nn.init.constant_(lin.bias.data, 0.0)
        for lin in (self.input_proj, self.output_proj):
            nn.init.xavier_uniform_(lin.weight.data)
            nn.init.constant_(lin.bias.data, 0.0)

    def forward(self, input):
        N, H, W, _ = input.shape
        x = self.input_proj(input)
        x_proj = x
        dtype = x.dtype
        x1 = self.dw_conv(input.permute(0, 3, 1, 2))
        offset = self.offset(x1)
        geometry = (self.kernel_size, self.kernel_size, self.stride, self.stride, self.pad, self.pad, self.dilation,
                    self.dilation, self.group, self.group_channels, self.offset_scale, 256)
        if fast_supported(x, self.kernel_size, self.kernel_size, self.group_channels):
            # fused: the mask softmax runs inside the kernels on float32 logits (under autocast the mask is therefore
            # not rounded to the input dtype, as the composition below rounds it).  16-bit Linear outputs in the
            # input's dtype (autocast) go in as they are: the kernels widen them exactly and round their gradients.
            mask_logits = self.mask(x1)
            if not (offset.dtype == mask_logits.dtype == dtype and dtype in (torch.float16, torch.bfloat16)):
                offset, mask_logits = offset.float(), mask_logits.float()
            if torch.compiler.is_compiling():
                x = torch.ops.ir_ads_b200.dcnv3_fused(x.contiguous(), offset.contiguous(),
                                                      mask_logits.reshape(N, H, W, -1).contiguous(), *geometry[:11],
                                                      functional._deterministic())
            else:
                x = DCNv3FusedFunction.apply(x.contiguous(), offset.contiguous(),
                                             mask_logits.reshape(N, H, W, -1).contiguous(), *geometry)
        else:
            mask = F.softmax(self.mask(x1).reshape(N, H, W, self.group, -1), -1).reshape(N, H, W, -1).type(dtype)
            x = DCNv3Function.apply(x.contiguous(), offset.contiguous(), mask.contiguous(), *geometry)
        if self.center_feature_scale:
            scale = F.linear(x1, weight=self.center_feature_scale_proj_weight,
                             bias=self.center_feature_scale_proj_bias).sigmoid()
            scale = scale[..., None].repeat(1, 1, 1, 1, self.channels // self.group).flatten(-2)
            x = x * (1 - scale) + x_proj * scale
        return self.output_proj(x)

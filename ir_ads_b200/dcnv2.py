"""Deformable convolution v1 / v2: detectron2's ``deform_conv`` / ``modulated_deform_conv`` functions and its
``DeformConv`` / ``ModulatedDeformConv`` modules (detectron2/layers/deform_conv.py), with the same arguments,
parameters and initialisation, so configs and checkpoints work unchanged.

The sampling runs in libmsda_b200's kernels (include/msda.h, ``msda_dcnv2_im2col`` / ``msda_dcnv2_col2im``); the
products with the weight are cuBLAS GEMMs through torch:

  forward   input rows (NHWC) -> im2col -> columns [pixels, groups, K * C/groups] -> columns @ W^T (+ bias) -> output
  backward  grad_columns = grad_out @ W -> col2im (grad_input, grad_offset, grad_mask); the columns are recomputed
            (saving them would cost K times the input's memory) for grad_W += grad_out^T @ columns; grad_bias.

The column order makes each conv group's weight matrix a plain reshape of ``weight.permute(0, 2, 3, 1)`` (``_wmat``);
only this module and the kernels know it.  Columns are built for whole images at a time, at most ``im2col_step``
images and at most ``MAX_COLUMN_ELEMENTS`` elements a chunk (a single image may exceed it); any batch size works.

Memory format: the output (and grad_input) has the input's memory format.  A ``channels_last`` input costs no copy; a
contiguous NCHW input costs one transpose in and one out.  ``offset`` / ``mask`` may be in either format and are
copied at most once.  Under autocast the op runs in the autocast dtype, as ``conv2d`` does: 16-bit columns and GEMMs
with float32 accumulation; offsets and mask then go in float32 when both are float32, else in the 16-bit type.

There is no CPU path.  The backward's grad_input is accumulated with float atomics: with ``set_deterministic(True)``
or ``torch.use_deterministic_algorithms(True)`` it raises, as PyTorch's CUDA ops without a deterministic
implementation do (a warning under ``warn_only=True``).  grad_offset / grad_mask / grad_weight are reproducible.
"""
from __future__ import annotations

import ctypes
import warnings
from typing import Tuple

import torch
from torch import nn
from torch.nn.modules.utils import _pair

from . import _lib
from . import functional as _functional
from .functional import _aligned, _ptr, _require

_TAG = {torch.float32: _lib.MSDA_F32, torch.float64: _lib.MSDA_F64, torch.bfloat16: _lib.MSDA_BF16,
        torch.float16: _lib.MSDA_F16}
_AUX16_TAG = {torch.bfloat16: _lib.MSDA_BF16_AUX16, torch.float16: _lib.MSDA_F16_AUX16}
# Column elements per chunk: 256 Mi (512 MiB of bf16 columns).  The backward holds two such buffers.
MAX_COLUMN_ELEMENTS = 1 << 28


class _Geom:
    """Shapes of one call: input [B, C, H, W], weight [C_out, C/groups, kh, kw], output [B, C_out, Ho, Wo]."""

    def __init__(self, input, weight, stride_h, stride_w, pad_h, pad_w, dil_h, dil_w, groups, deformable_groups,
                 im2col_step):
        self.B, self.C, self.H, self.W = input.shape
        self.C_out, _, self.kh, self.kw = weight.shape
        self.K = self.kh * self.kw
        self.Ho = (self.H + 2 * pad_h - (dil_h * (self.kh - 1) + 1)) // stride_h + 1
        self.Wo = (self.W + 2 * pad_w - (dil_w * (self.kw - 1) + 1)) // stride_w + 1
        self.P = self.Ho * self.Wo
        self.groups, self.dg = groups, deformable_groups
        per_image = max(1, self.P * self.K * self.C)
        self.step = max(1, min(im2col_step, self.B, MAX_COLUMN_ELEMENTS // per_image))
        self.ints = [self.C, self.H, self.W, self.Ho, self.Wo, self.kh, self.kw, stride_h, stride_w, pad_h, pad_w,
                     dil_h, dil_w, groups, deformable_groups]

    def abi(self, batch):   # batch, channels, ..., deformable_groups as the C ABI takes them
        return [batch] + self.ints


def _channels_last(t: torch.Tensor) -> bool:
    return not t.is_contiguous() and t.is_contiguous(memory_format=torch.channels_last)


def _nhwc(t: torch.Tensor) -> torch.Tensor:
    """[B, C, H, W] -> contiguous [B, H, W, C]: a view of a channels_last tensor, one copy otherwise."""
    return t.permute(0, 2, 3, 1).contiguous()


def _nchw(rows: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
    """Contiguous [B, H, W, C] -> [B, C, H, W] in ``like``'s memory format (a view for channels_last)."""
    t = rows.permute(0, 3, 1, 2)
    return t if _channels_last(like) else t.contiguous()


def _wmat(weight: torch.Tensor, groups: int) -> torch.Tensor:
    """[C_out, C/groups, kh, kw] -> [groups, C_out/groups, kh*kw*C/groups] in the columns' (k, c) order."""
    return weight.permute(0, 2, 3, 1).reshape(groups, weight.shape[0] // groups, -1)


def _check(input, offset, mask, weight, bias, g: _Geom):
    _require(input.is_cuda, "Not implemented on the CPU")
    for name, t in (("offset", offset), ("mask", mask), ("weight", weight), ("bias", bias)):
        if t is not None:
            _require(t.is_cuda and t.device == input.device, f"{name} must be a CUDA tensor on {input.device}")
    _require(input.dim() == 4 and weight.dim() == 4, "input must be [B, C, H, W] and weight [C_out, C/groups, kh, kw]")
    _require(input.dtype in _TAG, f"unsupported input dtype {input.dtype}")
    _require(weight.dtype == input.dtype and (bias is None or bias.dtype == input.dtype),
             f"weight / bias must have the input's dtype {input.dtype}")
    _require(g.groups >= 1 and g.dg >= 1 and g.C % g.groups == 0 and g.C % g.dg == 0 and g.C_out % g.groups == 0,
             f"channels ({g.C} in, {g.C_out} out) must be divisible by groups ({g.groups}) and the input channels by "
             f"deformable_groups ({g.dg})")
    _require(weight.shape[1] * g.groups == g.C, f"weight {tuple(weight.shape)} does not fit {g.C} input channels")
    _require(g.Ho >= 1 and g.Wo >= 1, "the input is smaller than the kernel")
    _require(tuple(offset.shape) == (g.B, g.dg * g.K * 2, g.Ho, g.Wo),
             f"offset must be [{g.B}, {g.dg * g.K * 2}, {g.Ho}, {g.Wo}], got {tuple(offset.shape)}")
    if mask is not None:
        _require(tuple(mask.shape) == (g.B, g.dg * g.K, g.Ho, g.Wo),
                 f"mask must be [{g.B}, {g.dg * g.K}, {g.Ho}, {g.Wo}], got {tuple(mask.shape)}")
    _require(bias is None or tuple(bias.shape) == (g.C_out,), f"bias must be [{g.C_out}]")
    aux = offset.dtype
    _require(mask is None or mask.dtype == aux, "offset and mask must share a dtype")
    if aux == input.dtype and input.dtype in _AUX16_TAG:
        return _AUX16_TAG[input.dtype]
    _require(aux == (torch.float64 if input.dtype == torch.float64 else torch.float32),
             f"offset / mask must be float32 (float64 for a float64 input) or the input's 16-bit dtype, got {aux}")
    return _TAG[input.dtype]


def _stream(t: torch.Tensor) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _im2col(x, off, msk, cols, g: _Geom, tag: int) -> None:
    nb = x.shape[0]
    handle = _lib.lib()
    _lib.check(handle.msda_dcnv2_im2col(_stream(x), _ptr(x), _ptr(off), None if msk is None else _ptr(msk),
                                        *g.abi(nb), _ptr(cols), tag, _functional._flags(False)), "msda_dcnv2_im2col")


def _chunks(g: _Geom):
    for b0 in range(0, g.B, g.step):
        yield b0, min(g.step, g.B - b0)


def _prepare(input, offset, mask):
    x = _aligned(_nhwc(input))
    off = _aligned(_nhwc(offset))
    msk = None if mask is None else _aligned(_nhwc(mask))
    return x, off, msk


def _forward(input, offset, mask, weight, bias, g: _Geom) -> torch.Tensor:
    tag = _check(input, offset, mask, weight, bias, g)
    x, off, msk = _prepare(input, offset, mask)
    wm = _wmat(weight, g.groups)
    out = torch.empty((g.B * g.P, g.C_out), dtype=input.dtype, device=input.device)
    cols = torch.empty((g.step * g.P, g.groups, g.K * g.C // g.groups), dtype=input.dtype, device=input.device)
    for b0, nb in _chunks(g):
        c = cols[:nb * g.P]
        sl = slice(b0, b0 + nb)
        _im2col(_aligned(x[sl]), _aligned(off[sl]), None if msk is None else _aligned(msk[sl]), c, g, tag)
        rows = out[b0 * g.P:(b0 + nb) * g.P]
        if g.groups == 1:
            if bias is None:
                torch.mm(c.view(nb * g.P, -1), wm[0].t(), out=rows)
            else:
                torch.addmm(bias, c.view(nb * g.P, -1), wm[0].t(), out=rows)
        else:
            rows.copy_(torch.bmm(c.transpose(0, 1), wm.transpose(1, 2)).transpose(0, 1).reshape(nb * g.P, -1))
            if bias is not None:
                rows += bias
    return _nchw(out.view(g.B, g.Ho, g.Wo, g.C_out), input)


def _alert_not_deterministic() -> None:
    msg = ("deformable convolution backward (msda_dcnv2_col2im) does not have a deterministic implementation: its "
           "grad_input is accumulated with float atomics")
    if _functional._state["deterministic"] or not torch.is_deterministic_algorithms_warn_only_enabled():
        raise RuntimeError(msg + ", but deterministic algorithms were requested (set_deterministic / "
                                 "torch.use_deterministic_algorithms)")
    warnings.warn(msg + ".")


def _backward(grad_out, input, offset, mask, weight, bias, g: _Geom, need: Tuple[bool, ...]):
    """(grad_input, grad_offset, grad_mask or None, grad_weight or None, grad_bias or None)."""
    if _functional._deterministic():
        _alert_not_deterministic()
    tag = _check(input, offset, mask, weight, bias, g)
    _require(grad_out.is_cuda and grad_out.dtype == input.dtype and
             tuple(grad_out.shape) == (g.B, g.C_out, g.Ho, g.Wo), "grad_output must match the output")
    x, off, msk = _prepare(input, offset, mask)
    go = _nhwc(grad_out).view(g.B * g.P, g.C_out)
    wm = _wmat(weight, g.groups)
    dev, dt = input.device, input.dtype
    KCg = g.K * g.C // g.groups
    gcols = torch.empty((g.step * g.P, g.groups, KCg), dtype=dt, device=dev)
    cols = torch.empty_like(gcols) if need[3] else None
    ws = torch.empty(max(1, _lib.lib().msda_dcnv2_col2im_workspace_bytes(*g.abi(g.step), tag, 0)), dtype=torch.uint8,
                     device=dev)
    gx_parts, goff_parts, gmsk_parts = [], [], []
    gw = None
    multi = g.step < g.B
    handle = _lib.lib()
    for b0, nb in _chunks(g):
        sl = slice(b0, b0 + nb)
        go_c = go[b0 * g.P:(b0 + nb) * g.P]
        gc = gcols[:nb * g.P]
        if g.groups == 1:
            torch.mm(go_c, wm[0], out=gc.view(nb * g.P, -1))
        else:
            gc.copy_(torch.bmm(go_c.view(nb * g.P, g.groups, -1).transpose(0, 1), wm).transpose(0, 1))
        xc, offc = _aligned(x[sl]), _aligned(off[sl])
        mc = None if msk is None else _aligned(msk[sl])
        gx = torch.empty_like(xc)
        goff = torch.empty_like(offc)
        gm = None if mc is None else torch.empty_like(mc)
        _lib.check(handle.msda_dcnv2_col2im(_stream(x), _ptr(gc), _ptr(xc), _ptr(offc),
                                            None if mc is None else _ptr(mc), *g.abi(nb), _ptr(gx), _ptr(goff),
                                            None if gm is None else _ptr(gm), _ptr(ws), ws.numel(), tag,
                                            _functional._flags(False)), "msda_dcnv2_col2im")
        gx_parts.append(gx)
        goff_parts.append(goff)
        gmsk_parts.append(gm)
        if need[3]:
            c = cols[:nb * g.P]
            _im2col(xc, offc, mc, c, g, tag)
            if g.groups == 1:
                part = torch.mm(go_c.t(), c.view(nb * g.P, -1)).unsqueeze(0)
            else:
                part = torch.bmm(go_c.view(nb * g.P, g.groups, -1).permute(1, 2, 0), c.transpose(0, 1))
            if multi:   # chunks are summed in float32
                part = part.float()
            gw = part if gw is None else gw.add_(part)

    def join(parts):
        return parts[0] if len(parts) == 1 else torch.cat(parts)

    grad_input = _nchw(join(gx_parts), input) if need[0] else None
    grad_offset = _nchw(join(goff_parts), offset) if need[1] else None
    grad_mask = _nchw(join(gmsk_parts), mask) if (mask is not None and need[2]) else None
    grad_weight = None
    if need[3]:
        grad_weight = gw.to(dt).view(g.C_out, g.kh, g.kw, -1).permute(0, 3, 1, 2).contiguous()
    grad_bias = go.sum(0, dtype=torch.float32).to(dt) if (bias is not None and need[4]) else None
    return grad_input, grad_offset, grad_mask, grad_weight, grad_bias


class DCNv2Function(torch.autograd.Function):
    """``apply(input, offset, mask, weight, bias, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, groups,
    deformable_groups, im2col_step)``; ``mask`` None is DCNv1, ``bias`` may be None.  No autocast handling: use
    ``deform_conv`` / ``modulated_deform_conv``."""

    @staticmethod
    def forward(ctx, input, offset, mask, weight, bias, *ints):
        g = _Geom(input, weight, *ints)
        ctx.save_for_backward(input, offset, mask, weight, bias)
        ctx.ints = ints
        return _forward(input, offset, mask, weight, bias, g)

    @staticmethod
    def backward(ctx, grad_out):
        input, offset, mask, weight, bias = ctx.saved_tensors
        g = _Geom(input, weight, *ctx.ints)
        grads = _backward(grad_out, input, offset, mask, weight, bias, g, ctx.needs_input_grad[:5])
        return grads + (None,) * len(ctx.ints)


def _call(input, offset, mask, weight, bias, stride, padding, dilation, groups, deformable_groups, im2col_step):
    ints = (*_pair(stride), *_pair(padding), *_pair(dilation), int(groups), int(deformable_groups), int(im2col_step))
    if input.is_cuda and input.dtype != torch.float64 and torch.is_autocast_enabled("cuda"):
        dt = torch.get_autocast_dtype("cuda")
        input, weight = input.to(dt), weight.to(dt)
        bias = None if bias is None else bias.to(dt)
        if not (offset.dtype == torch.float32 and (mask is None or mask.dtype == torch.float32)):
            offset = offset.to(dt)
            mask = None if mask is None else mask.to(dt)
        with torch.autocast("cuda", enabled=False):
            return _dispatch(input, offset, mask, weight, bias, ints)
    return _dispatch(input, offset, mask, weight, bias, ints)


def _dispatch(input, offset, mask, weight, bias, ints):
    if torch.compiler.is_compiling():
        from . import ops
        return ops.dcnv2(input, offset, mask, weight, bias, *ints)
    return DCNv2Function.apply(input, offset, mask, weight, bias, *ints)


def deform_conv(input, offset, weight, stride=1, padding=0, dilation=1, groups=1, deformable_groups=1,
                im2col_step=64):
    """DCNv1 (detectron2's ``deform_conv``): input [B, C, H, W], offset [B, dg*kh*kw*2, Ho, Wo] as (dy, dx) pairs,
    weight [C_out, C/groups, kh, kw].  ``im2col_step`` bounds the images per column chunk; any batch size works."""
    return _call(input, offset, None, weight, None, stride, padding, dilation, groups, deformable_groups, im2col_step)


def modulated_deform_conv(input, offset, mask, weight, bias=None, stride=1, padding=0, dilation=1, groups=1,
                          deformable_groups=1, im2col_step=64):
    """DCNv2 (detectron2's ``modulated_deform_conv``): as ``deform_conv`` plus mask [B, dg*kh*kw, Ho, Wo] and an
    optional bias [C_out]."""
    return _call(input, offset, mask, weight, bias, stride, padding, dilation, groups, deformable_groups, im2col_step)


class _DeformConvBase(nn.Module):
    def __init__(self, in_channels, out_channels, kernel_size, stride, padding, dilation, groups, deformable_groups,
                 bias, norm, activation):
        super().__init__()
        assert in_channels % groups == 0, f"in_channels {in_channels} cannot be divisible by groups {groups}"
        assert out_channels % groups == 0, f"out_channels {out_channels} cannot be divisible by groups {groups}"
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _pair(kernel_size)
        self.stride = _pair(stride)
        self.padding = _pair(padding)
        self.dilation = _pair(dilation)
        self.groups = groups
        self.deformable_groups = deformable_groups
        self.with_bias = bias
        self.norm = norm
        self.activation = activation
        self.weight = nn.Parameter(torch.Tensor(out_channels, in_channels // groups, *self.kernel_size))
        self.bias = nn.Parameter(torch.Tensor(out_channels)) if bias else None
        nn.init.kaiming_uniform_(self.weight, nonlinearity="relu")
        if self.bias is not None:
            nn.init.constant_(self.bias, 0)

    def _finish(self, x):
        if self.norm is not None:
            x = self.norm(x)
        if self.activation is not None:
            x = self.activation(x)
        return x

    def extra_repr(self):
        return (f"in_channels={self.in_channels}, out_channels={self.out_channels}, kernel_size={self.kernel_size}, "
                f"stride={self.stride}, padding={self.padding}, dilation={self.dilation}, groups={self.groups}, "
                f"deformable_groups={self.deformable_groups}, bias={self.with_bias}")


class DeformConv(_DeformConvBase):
    """detectron2's ``DeformConv`` (DCNv1): ``forward(x, offset)``; no bias (``bias=True`` is refused, as there)."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 deformable_groups=1, bias=False, norm=None, activation=None):
        assert not bias
        super().__init__(in_channels, out_channels, kernel_size, stride, padding, dilation, groups, deformable_groups,
                         False, norm, activation)

    def forward(self, x, offset):
        x = deform_conv(x, offset, self.weight, self.stride, self.padding, self.dilation, self.groups,
                        self.deformable_groups)
        return self._finish(x)


class ModulatedDeformConv(_DeformConvBase):
    """detectron2's ``ModulatedDeformConv`` (DCNv2): ``forward(x, offset, mask)``."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 deformable_groups=1, bias=True, norm=None, activation=None):
        super().__init__(in_channels, out_channels, kernel_size, stride, padding, dilation, groups, deformable_groups,
                         bias, norm, activation)

    def forward(self, x, offset, mask):
        x = modulated_deform_conv(x, offset, mask, self.weight, self.bias, self.stride, self.padding, self.dilation,
                                  self.groups, self.deformable_groups)
        return self._finish(x)


__all__ = ["DeformConv", "ModulatedDeformConv", "deform_conv", "modulated_deform_conv", "DCNv2Function",
           "MAX_COLUMN_ELEMENTS"]

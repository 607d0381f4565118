"""The module paths' kernels as ``torch.library`` custom ops, for ``torch.compile`` and ``torch.export``.

Every kernel is reached through ``ctypes``, which the compiler cannot trace, so each autograd Function the modules call
would split the graph.  The ops below wrap those Functions' bodies (the argument checks, alignment, workspace sizing
and error checks stay in functional.py, epilogue.py and dcnv3.py) behind a schema, a fake kernel and an autograd
formula:

  ir_ads_b200::msda_fused / msda_fused_backward      MSDeformAttnFusedFunction
  ir_ads_b200::msda_packed / msda_packed_backward    MSDeformAttnPackedFunction
  ir_ads_b200::add_layer_norm / _backward            AddLayerNormFunction and AddLayerNormMixedFunction
  ir_ads_b200::dcnv3_fused / dcnv3_fused_backward    DCNv3FusedFunction

``MultiScaleDeformableAttention``, ``epilogue.add_layer_norm`` and the ``DCNv3`` module call them only while
``torch.compiler.is_compiling()``; eager code keeps calling the Functions.

Choices the backward makes are op arguments, fixed when the graph is built: ``deterministic`` (read from
``set_deterministic`` / ``torch.use_deterministic_algorithms`` by the caller, so the compiler guards on it and
recompiles when it changes) and which inputs need a gradient.  Bits set with ``kernel_flags`` (a test and benchmark
hook) are still read when the op runs.  Workspaces are allocated inside the ops with ``torch.empty``.  No op writes
into an input.  The fake kernels only allocate: registering or tracing the ops never loads libmsda_b200.so.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib
from . import dcnv3 as _dcnv3
from . import epilogue as _epilogue
from . import functional as _functional


def _flags(deterministic: bool) -> int:
    return _functional._flags(False) | (_lib.FLAG_DETERMINISTIC if deterministic else 0)


# ------------------------------------------------------------------------------------------------
# msda_fused: MSDeformAttnFusedFunction
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("ir_ads_b200::msda_fused", mutates_args=())
def msda_fused(value: torch.Tensor, spatial_shapes: torch.Tensor, level_start_index: torch.Tensor,
               sampling_offsets: torch.Tensor, attn_logits: torch.Tensor, reference_points: torch.Tensor,
               key_padding_mask: Optional[torch.Tensor], deterministic: bool) -> torch.Tensor:
    """MSDeformAttnFusedFunction's forward: ``[B, Q, H*D]`` in value's dtype.  ``deterministic`` selects the route
    of the backward only."""
    return _functional._fused_forward(value, spatial_shapes, level_start_index, sampling_offsets, attn_logits,
                                      reference_points, key_padding_mask)[0]


@msda_fused.register_fake
def _(value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, reference_points, key_padding_mask,
      deterministic):
    B, _, H, D = value.shape
    return value.new_empty((B, sampling_offsets.shape[1], H * D))


@torch.library.custom_op(
    "ir_ads_b200::msda_fused_backward", mutates_args=(),
    schema="(Tensor grad_output, Tensor value, Tensor spatial_shapes, Tensor level_start_index, "
           "Tensor sampling_offsets, Tensor attn_logits, Tensor reference_points, Tensor? key_padding_mask, "
           "bool deterministic, bool need_value, bool need_ref) -> (Tensor?, Tensor, Tensor, Tensor?)")
def msda_fused_backward(grad_output, value, spatial_shapes, level_start_index, sampling_offsets, attn_logits,
                        reference_points, key_padding_mask, deterministic, need_value, need_ref):
    """``(grad_value or None, grad_offsets, grad_logits, grad_reference_points or None)``: the routes of
    MSDeformAttnFusedFunction's backward (float reds, or the deterministic / reference-point composition)."""
    mask = None if key_padding_mask is None else key_padding_mask.contiguous()
    gv, go, gl, gr = _functional._fused_backward(grad_output, value, spatial_shapes, level_start_index,
                                                 sampling_offsets, attn_logits, reference_points, mask,
                                                 _flags(deterministic), need_value, need_ref)
    return (gv if need_value else None), go, gl, gr


@msda_fused_backward.register_fake
def _(grad_output, value, spatial_shapes, level_start_index, sampling_offsets, attn_logits, reference_points,
      key_padding_mask, deterministic, need_value, need_ref):
    return (torch.empty_like(value) if need_value else None, torch.empty_like(sampling_offsets),
            torch.empty_like(attn_logits), torch.empty_like(reference_points) if need_ref else None)


def _msda_fused_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs[:7])
    ctx.deterministic = inputs[7]


def _msda_fused_grad(ctx, grad_output):
    need = ctx.needs_input_grad
    gv, go, gl, gr = msda_fused_backward(grad_output, *ctx.saved_tensors, ctx.deterministic, need[0], need[5])
    return gv, None, None, go, gl, gr, None, None


msda_fused.register_autograd(_msda_fused_grad, setup_context=_msda_fused_setup)


# ------------------------------------------------------------------------------------------------
# msda_packed: MSDeformAttnPackedFunction
# ------------------------------------------------------------------------------------------------
class _PackedTables:
    """What MSDeformAttnPackedFunction's kernels and its padded backward read of a ``PackedLevels``, from the op's
    arguments: its device tables and host ints (the counts are their shapes, so nothing syncs)."""

    def __init__(self, meta, spatial_shapes, level_start_index, value_index, query_index, padding_mask, max_value,
                 max_query, query_pad):
        self.meta, self.spatial_shapes, self.level_start_index = meta, spatial_shapes, level_start_index
        self.value_index, self.query_index, self.padding_mask = value_index, query_index, padding_mask
        self.batch, self.padded_len = padding_mask.shape
        self.num_levels = spatial_shapes.shape[0]
        self.total_value, self.total_query = value_index.shape[0], query_index.shape[0]
        self.max_value, self.max_query, self.query_pad = max_value, max_query, query_pad
        self.num_queries = query_pad   # query rows unpack to [B, query_pad]; their mask is never read


@torch.library.custom_op("ir_ads_b200::msda_packed", mutates_args=())
def msda_packed(value: torch.Tensor, sampling_offsets: torch.Tensor, attn_logits: torch.Tensor,
                reference_points: torch.Tensor, meta: torch.Tensor, spatial_shapes: torch.Tensor,
                level_start_index: torch.Tensor, value_index: torch.Tensor, query_index: torch.Tensor,
                padding_mask: torch.Tensor, max_value: int, max_query: int, query_pad: int,
                deterministic: bool) -> torch.Tensor:
    """MSDeformAttnPackedFunction's forward: ``[T_q, H*D]``.  The ``PackedLevels`` arrives as its tables (``meta``
    for the kernels; the padded layout's shapes, level starts, token rows and mask for the backward's padded route)
    and host ints."""
    packing = _PackedTables(meta, spatial_shapes, level_start_index, value_index, query_index, padding_mask, max_value,
                            max_query, query_pad)
    return _functional._packed_forward(value, sampling_offsets, attn_logits, reference_points, packing)[0]


@msda_packed.register_fake
def _(value, sampling_offsets, attn_logits, reference_points, meta, spatial_shapes, level_start_index, value_index,
      query_index, padding_mask, max_value, max_query, query_pad, deterministic):
    _, H, D = value.shape
    return value.new_empty((sampling_offsets.shape[0], H * D))


@torch.library.custom_op(
    "ir_ads_b200::msda_packed_backward", mutates_args=(),
    schema="(Tensor grad_output, Tensor value, Tensor sampling_offsets, Tensor attn_logits, Tensor reference_points, "
           "Tensor meta, Tensor spatial_shapes, Tensor level_start_index, Tensor value_index, Tensor query_index, "
           "Tensor padding_mask, SymInt max_value, SymInt max_query, SymInt query_pad, bool deterministic, "
           "bool need_value, bool need_ref) -> (Tensor?, Tensor, Tensor, Tensor?)")
def msda_packed_backward(grad_output, value, sampling_offsets, attn_logits, reference_points, meta, spatial_shapes,
                         level_start_index, value_index, query_index, padding_mask, max_value, max_query, query_pad,
                         deterministic, need_value, need_ref):
    """``(grad_value or None, grad_offsets, grad_logits, grad_reference_points or None)``: the routes of
    MSDeformAttnPackedFunction's backward (packed float reds, or the padded route in deterministic mode and for
    reference points that need a gradient)."""
    packing = _PackedTables(meta, spatial_shapes, level_start_index, value_index, query_index, padding_mask, max_value,
                            max_query, query_pad)
    gv, go, gl, gr, _ = _functional._packed_backward(grad_output, value, sampling_offsets, attn_logits,
                                                     reference_points, packing, _flags(deterministic),
                                                     (need_value, True, True, need_ref))
    return (gv if need_value else None), go, gl, (gr if need_ref else None)


@msda_packed_backward.register_fake
def _(grad_output, value, sampling_offsets, attn_logits, reference_points, meta, spatial_shapes, level_start_index,
      value_index, query_index, padding_mask, max_value, max_query, query_pad, deterministic, need_value, need_ref):
    return (torch.empty_like(value) if need_value else None, torch.empty_like(sampling_offsets),
            torch.empty_like(attn_logits), torch.empty_like(reference_points) if need_ref else None)


def _msda_packed_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs[:10])
    ctx.ints = inputs[10:13]
    ctx.deterministic = inputs[13]


def _msda_packed_grad(ctx, grad_output):
    need = ctx.needs_input_grad
    gv, go, gl, gr = msda_packed_backward(grad_output, *ctx.saved_tensors, *ctx.ints, ctx.deterministic, need[0],
                                          need[3])
    return (gv, go, gl, gr) + (None,) * 10


msda_packed.register_autograd(_msda_packed_grad, setup_context=_msda_packed_setup)


# ------------------------------------------------------------------------------------------------
# add_layer_norm: AddLayerNormFunction (a and b in one dtype) and AddLayerNormMixedFunction (16-bit a, float32 b)
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("ir_ads_b200::add_layer_norm", mutates_args=())
def add_layer_norm(a: torch.Tensor, b: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor,
                   eps: float) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """``(LayerNorm(a + b), mean, rstd)`` over the last dimension: the same-dtype form when a and b share a dtype
    (result in it), else the mixed form (a bfloat16 / float16, b float32, float32 result)."""
    fwd = _epilogue._same_forward if a.dtype == b.dtype else _epilogue._mixed_forward
    y, (_, _, _, mean, rstd) = fwd(a, b, weight, bias, eps)
    return y, mean, rstd


@add_layer_norm.register_fake
def _(a, b, weight, bias, eps):
    rows = a.numel() // a.shape[-1] if a.shape[-1] else 0
    stats = a.new_empty((rows,), dtype=torch.float32)
    return (torch.empty_like(a if a.dtype == b.dtype else b, memory_format=torch.contiguous_format), stats,
            torch.empty_like(stats))


@torch.library.custom_op(
    "ir_ads_b200::add_layer_norm_backward", mutates_args=(),
    schema="(Tensor grad_y, Tensor a, Tensor b, Tensor weight, Tensor mean, Tensor rstd) "
           "-> (Tensor, Tensor?, Tensor, Tensor)")
def add_layer_norm_backward(grad_y, a, b, weight, mean, rstd):
    """``(grad_b, grad_a or None, grad_weight, grad_bias)``, weight / bias gradients in float32.  In the same-dtype
    form one gradient serves both addends and ``grad_a`` is None; in the mixed form ``grad_a`` is its 16-bit rounding."""
    a, b = _functional._aligned(a.contiguous()), _functional._aligned(b.contiguous())
    w32 = _functional._aligned(weight.float().contiguous())
    if a.dtype == b.dtype:
        dx, dgamma, dbeta = _epilogue._same_backward(grad_y, a, b, w32, mean, rstd)
        return dx, None, dgamma, dbeta
    da, db, dgamma, dbeta = _epilogue._mixed_backward(grad_y, a, b, w32, mean, rstd)
    return db, da, dgamma, dbeta


@add_layer_norm_backward.register_fake
def _(grad_y, a, b, weight, mean, rstd):
    C = a.shape[-1]
    grad_a = None if a.dtype == b.dtype else torch.empty_like(a, memory_format=torch.contiguous_format)
    return (torch.empty_like(b, memory_format=torch.contiguous_format), grad_a,
            weight.new_empty((C,), dtype=torch.float32), weight.new_empty((C,), dtype=torch.float32))


def _add_layer_norm_setup(ctx, inputs, output):
    a, b, weight, _, _ = inputs
    ctx.save_for_backward(a, b, weight, output[1], output[2])
    ctx.mark_non_differentiable(output[1], output[2])
    ctx.param_dtypes = (inputs[2].dtype, inputs[3].dtype)


def _add_layer_norm_grad(ctx, grad_y, grad_mean, grad_rstd):
    a, b, weight, mean, rstd = ctx.saved_tensors
    grad_b, grad_a, dgamma, dbeta = add_layer_norm_backward(grad_y, a, b, weight, mean, rstd)
    wd, bd = ctx.param_dtypes
    return grad_b if grad_a is None else grad_a, grad_b, dgamma.to(wd), dbeta.to(bd), None


add_layer_norm.register_autograd(_add_layer_norm_grad, setup_context=_add_layer_norm_setup)


# ------------------------------------------------------------------------------------------------
# dcnv3_fused: DCNv3FusedFunction
# ------------------------------------------------------------------------------------------------
@torch.library.custom_op("ir_ads_b200::dcnv3_fused", mutates_args=())
def dcnv3_fused(input: torch.Tensor, offset: torch.Tensor, mask_logits: torch.Tensor, kernel_h: int, kernel_w: int,
                stride_h: int, stride_w: int, pad_h: int, pad_w: int, dilation_h: int, dilation_w: int, group: int,
                group_channels: int, offset_scale: float, deterministic: bool) -> torch.Tensor:
    """DCNv3FusedFunction's forward: ``[N, H_out, W_out, group*group_channels]`` in input's dtype."""
    return _dcnv3.dcnv3_fused_forward(input, offset, mask_logits, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                                      dilation_h, dilation_w, group, group_channels, offset_scale)


@dcnv3_fused.register_fake
def _(input, offset, mask_logits, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group,
      group_channels, offset_scale, deterministic):
    N, H_out, W_out, _ = offset.shape
    return input.new_empty((N, H_out, W_out, group * group_channels))


@torch.library.custom_op(
    "ir_ads_b200::dcnv3_fused_backward", mutates_args=(),
    schema="(Tensor grad_output, Tensor input, Tensor offset, Tensor mask_logits, SymInt kernel_h, SymInt kernel_w, "
           "SymInt stride_h, SymInt stride_w, SymInt pad_h, SymInt pad_w, SymInt dilation_h, SymInt dilation_w, "
           "SymInt group, SymInt group_channels, float offset_scale, bool deterministic) -> (Tensor, Tensor, Tensor)")
def dcnv3_fused_backward(grad_output, input, offset, mask_logits, kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w,
                         dilation_h, dilation_w, group, group_channels, offset_scale, deterministic):
    """``(grad_input, grad_offset, grad_mask_logits)``: the routes of DCNv3FusedFunction's backward."""
    args = (kernel_h, kernel_w, stride_h, stride_w, pad_h, pad_w, dilation_h, dilation_w, group, group_channels,
            offset_scale)
    return tuple(_dcnv3._dcnv3_fused_backward_route(input, offset, mask_logits, args, grad_output,
                                                     _flags(deterministic)))


@dcnv3_fused_backward.register_fake
def _(grad_output, input, offset, mask_logits, *args):
    return (torch.empty_like(input, memory_format=torch.contiguous_format),
            torch.empty_like(offset, memory_format=torch.contiguous_format),
            torch.empty_like(mask_logits, memory_format=torch.contiguous_format))


def _dcnv3_fused_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs[:3])
    ctx.args = inputs[3:15]


def _dcnv3_fused_grad(ctx, grad_output):
    gi, go, gm = dcnv3_fused_backward(grad_output, *ctx.saved_tensors, *ctx.args)
    return (gi, go, gm) + (None,) * 12


dcnv3_fused.register_autograd(_dcnv3_fused_grad, setup_context=_dcnv3_fused_setup)

"""``MultiScaleDeformableAttention`` -- drop-in for the reference module
(/root/reference/detrex/layers/multi_scale_deform_attn.py:139-363): same constructor, same
``forward`` signature (extra keyword arguments from ``BaseTransformerLayer`` are swallowed,
detrex/layers/transformer.py:155-165), same sub-module / parameter names (``sampling_offsets``,
``attention_weights``, ``value_proj``, ``output_proj``) and the same initialisation, so DINO /
vCLR checkpoints load unchanged.  The four projections stay cuBLAS through ``nn.Linear``; the
core op runs on the sm_100a kernels through :class:`MultiScaleDeformableAttnFunction`.

What differs from the reference module:
  * no device->host synchronisation per call: the reference asserts
    ``(spatial_shapes[:,0]*spatial_shapes[:,1]).sum() == num_value`` on the device tensor every
    forward (py:286), which blocks the host 12 times per step; here the check runs on a HOST copy of the shapes
    when the caller has one (``level_shapes=[(H_l, W_l), ...]``, what ``encoder.flatten_levels`` returns: free),
    otherwise once per live shapes tensor OBJECT (keyed by the object, dropped when it dies -- never by address);
  * bfloat16 and float16 activations (autocast) go to the bf16 / f16-value kernels with float32 sampling
    locations / weights and float32 accumulation instead of failing in the float-only dispatch.  The reference
    widens float16 to float32 around the op (py:343, :355-356); here the fused path takes the float16 value as it is,
    with the same output (the kernels widen exactly, so only the final rounding to float16 remains) and half the
    value bytes read and saved for backward.  The 16-bit sampling offsets / attention logits that autocast's Linears
    produce go into the fused kernels as they are too (no float32 copy, no cast kernel either way; the same bits as
    widening them).  Only the unfused fallback (``fuse_pre_ops = False`` or shapes the
    fused kernels do not cover) still widens float16, since the plain op, like the reference's, has no float16 form;
  * there is no CPU branch (py:350-353): a CPU tensor raises;
  * ``add_identity=False`` (keyword, default True) returns ``dropout(output_proj(...))`` WITHOUT the residual
    (py:363), for callers that fuse ``+ identity`` into the LayerNorm that follows (ir_ads_b200/epilogue.py);
  * ``packing=PackedLevels`` (keyword, ir_ads_b200/packing.py): a padding-free batch -- 2-D ``[T_q, C]`` query and
    ``[T_v, C]`` value, ``reference_points [T_q, L, 2|4]``, no ``key_padding_mask`` -- through the packed fused
    kernels (MSDeformAttnPackedFunction); the result is ``[T_q, C]``.
"""
from __future__ import annotations

import math
import warnings
import weakref
from typing import Optional

import torch
import torch.nn as nn

from .functional import (MSDeformAttnFusedFunction, MSDeformAttnPackedFunction, MultiScaleDeformableAttnFunction,
                         _deterministic, fused_supported)


# shapes tensors already validated: id(tensor) -> (version, num_value); entries die with their tensor
_SHAPE_CHECKS: dict = {}


def _is_power_of_2(n: int) -> bool:
    if not isinstance(n, int) or n < 0:
        raise ValueError(f"invalid input for _is_power_of_2: {n} (type: {type(n)})")
    return n != 0 and (n & (n - 1)) == 0


class MultiScaleDeformableAttention(nn.Module):
    """Multi-scale deformable attention (Deformable DETR, arXiv:2010.04159).

    Args mirror the reference: embed_dim=256, num_heads=8, num_levels=4, num_points=4,
    img2col_step=64 (kept for compatibility, unused by the kernels), dropout=0.1,
    batch_first=False (``(n, bs, embed_dim)`` tensors).
    """

    def __init__(self, embed_dim: int = 256, num_heads: int = 8, num_levels: int = 4, num_points: int = 4,
                 img2col_step: int = 64, dropout: float = 0.1, batch_first: bool = False):
        super().__init__()
        if embed_dim % num_heads != 0:
            raise ValueError(f"embed_dim must be divisible by num_heads, but got {embed_dim} and {num_heads}")
        if not _is_power_of_2(embed_dim // num_heads):
            warnings.warn("MultiScaleDeformableAttention: a power-of-two head dimension is more efficient "
                          "(head dims 16/32/64/128 use the vectorised sm_100a kernels).")
        self.dropout = nn.Dropout(dropout)
        self.batch_first = batch_first
        self.im2col_step = img2col_step
        self.embed_dim = embed_dim
        self.num_heads = num_heads
        self.num_levels = num_levels
        self.num_points = num_points
        # construction order == the reference's (py:193-196) so a seeded run draws the same numbers
        self.sampling_offsets = nn.Linear(embed_dim, num_heads * num_levels * num_points * 2)
        self.attention_weights = nn.Linear(embed_dim, num_heads * num_levels * num_points)
        self.value_proj = nn.Linear(embed_dim, embed_dim)
        self.output_proj = nn.Linear(embed_dim, embed_dim)
        # fused pre-op chain (softmax + sampling-location arithmetic inside the kernels); set False to
        # run the reference's step-by-step composition around the core op instead
        self.fuse_pre_ops = True
        self.init_weights()

    def init_weights(self) -> None:
        """Reference initialisation (py:200-223): zero offset weights, per-head unit directions scaled
        by the point index as offset bias, uniform attention, Xavier projections."""
        nn.init.constant_(self.sampling_offsets.weight.data, 0.0)
        thetas = torch.arange(self.num_heads, dtype=torch.float32) * (2.0 * math.pi / self.num_heads)
        directions = torch.stack([thetas.cos(), thetas.sin()], -1)
        directions = directions / directions.abs().max(-1, keepdim=True)[0]
        grid = directions.view(self.num_heads, 1, 1, 2).repeat(1, self.num_levels, self.num_points, 1)
        grid = grid * torch.arange(1, self.num_points + 1, dtype=torch.float32).view(1, 1, -1, 1)
        with torch.no_grad():
            self.sampling_offsets.bias = nn.Parameter(grid.reshape(-1))
        nn.init.constant_(self.attention_weights.weight.data, 0.0)
        nn.init.constant_(self.attention_weights.bias.data, 0.0)
        nn.init.xavier_uniform_(self.value_proj.weight.data)
        nn.init.constant_(self.value_proj.bias.data, 0.0)
        nn.init.xavier_uniform_(self.output_proj.weight.data)
        nn.init.constant_(self.output_proj.bias.data, 0.0)

    @staticmethod
    def _check_shapes(spatial_shapes: torch.Tensor, num_value: int, level_shapes=None) -> None:
        """sum(H_l * W_l) == num_value (py:286).  The fast kernels' 32-bit offsets and the deterministic path's
        workspace bound rely on it."""
        if level_shapes is not None:
            total = sum(int(h) * int(w) for h, w in level_shapes)
            if total != num_value or len(level_shapes) != spatial_shapes.shape[0]:
                raise AssertionError(f"sum(H_l*W_l) = {total} does not match the value length {num_value}")
            return
        key = id(spatial_shapes)
        hit = _SHAPE_CHECKS.get(key)
        if hit is not None and hit == (spatial_shapes._version, num_value):
            return
        if spatial_shapes.is_cuda and torch.cuda.is_current_stream_capturing():
            return                                   # cannot sync inside a capture; the warm-up pass checked
        total = int((spatial_shapes[:, 0] * spatial_shapes[:, 1]).sum())   # one sync per live tensor object
        if total != num_value:
            raise AssertionError(f"sum(H_l*W_l) = {total} does not match the value length {num_value}")
        if hit is None:
            weakref.finalize(spatial_shapes, _SHAPE_CHECKS.pop, key, None)   # the id may be re-used after death
        _SHAPE_CHECKS[key] = (spatial_shapes._version, num_value)

    def _forward_packed(self, query, value, identity, reference_points, key_padding_mask, packing, add_identity):
        if key_padding_mask is not None:
            raise ValueError("a packed batch has no padding: key_padding_mask must be None")
        if query.dim() != 2 or value.dim() != 2:
            raise ValueError("with packing=, query and value are 2-D [T, C] token rows")
        if value.shape[0] != packing.total_value or query.shape[0] != packing.total_query:
            raise AssertionError(f"{value.shape[0]} value / {query.shape[0]} query rows, the packing has "
                                 f"{packing.total_value} / {packing.total_query}")
        H, L, P = self.num_heads, self.num_levels, self.num_points
        if packing.num_levels != L:
            raise AssertionError(f"the packing has {packing.num_levels} levels, the module {L}")
        if reference_points.shape[-1] not in (2, 4):
            raise ValueError(
                f"Last dim of reference_points must be 2 or 4, but get {reference_points.shape[-1]} instead.")
        T_q = query.shape[0]
        value = self.value_proj(value)
        io_dtype = value.dtype
        value = value.view(value.shape[0], H, -1)
        if not (self.fuse_pre_ops and fused_supported(value.unsqueeze(0), L, P)):
            raise RuntimeError("packed batches run on the fused kernels only (fuse_pre_ops, CUDA, float32 / bfloat16 / "
                               "float16, head dim 16/32/64/128, L <= 16, L*P <= 64)")
        offsets = self.sampling_offsets(query).view(T_q, H, L, P, 2)
        logits = self.attention_weights(query).view(T_q, H, L * P)
        if not (offsets.dtype == logits.dtype == value.dtype and value.dtype in (torch.float16, torch.bfloat16)):
            offsets, logits = offsets.float(), logits.float()
        if torch.compiler.is_compiling():
            output = torch.ops.ir_ads_b200.msda_packed(
                value.contiguous(), offsets.contiguous(), logits.contiguous(), reference_points.float().contiguous(),
                packing.meta, packing.spatial_shapes, packing.level_start_index, packing.value_index,
                packing.query_index, packing.padding_mask, packing.max_value, packing.max_query, packing.query_pad,
                _deterministic())
        else:
            output = MSDeformAttnPackedFunction.apply(value.contiguous(), offsets.contiguous(), logits.contiguous(),
                                                      reference_points.float().contiguous(), packing)
        if output.dtype != io_dtype:
            output = output.to(io_dtype)
        output = self.dropout(self.output_proj(output))
        return output + identity if add_identity else output

    def forward(self, query: torch.Tensor, key: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None,
                identity: Optional[torch.Tensor] = None, query_pos: Optional[torch.Tensor] = None,
                key_padding_mask: Optional[torch.Tensor] = None, reference_points: Optional[torch.Tensor] = None,
                spatial_shapes: Optional[torch.Tensor] = None, level_start_index: Optional[torch.Tensor] = None,
                **kwargs) -> torch.Tensor:
        if value is None:
            value = query
        if identity is None:
            identity = query
        if query_pos is not None:
            query = query + query_pos
        packing = kwargs.get("packing")
        if packing is not None:
            return self._forward_packed(query, value, identity, reference_points, key_padding_mask, packing,
                                        kwargs.get("add_identity", True))
        if not self.batch_first:
            query = query.permute(1, 0, 2)
            value = value.permute(1, 0, 2)

        bs, num_query, _ = query.shape
        _, num_value, _ = value.shape
        self._check_shapes(spatial_shapes, num_value, kwargs.get("level_shapes"))
        H, L, P = self.num_heads, self.num_levels, self.num_points

        value = self.value_proj(value)
        if not value.is_cuda:
            raise RuntimeError("MultiScaleDeformableAttention: Not implemented on the CPU "
                               "(the B200 build has no PyTorch fallback)")
        if reference_points.shape[-1] not in (2, 4):
            raise ValueError(
                f"Last dim of reference_points must be 2 or 4, but get {reference_points.shape[-1]} instead.")
        offsets = self.sampling_offsets(query).view(bs, num_query, H, L, P, 2)
        logits = self.attention_weights(query).view(bs, num_query, H, L * P)

        io_dtype = value.dtype
        value = value.view(bs, num_value, H, -1)
        fused = self.fuse_pre_ops and fused_supported(value, L, P)
        if io_dtype == torch.float16 and not fused:
            value = value.float()                         # the plain op has no float16 form (py:343)
        if key_padding_mask is not None and not fused:
            value = value.masked_fill(key_padding_mask[..., None, None], float(0))
        if fused:
            # the padding mask goes into the kernels (masked pixels read as zeros, zero grad_value): the masked
            # copy of value (py:291-292) and its backward never exist.  16-bit offsets / logits in value's dtype (the
            # Linear outputs under autocast) go in as they are: the kernels widen them exactly and round their
            # gradients, so neither a float32 copy nor a cast kernel exists in either direction.
            if not (offsets.dtype == logits.dtype == value.dtype and value.dtype in (torch.float16, torch.bfloat16)):
                offsets, logits = offsets.float(), logits.float()
            if torch.compiler.is_compiling():
                output = torch.ops.ir_ads_b200.msda_fused(
                    value.contiguous(), spatial_shapes, level_start_index, offsets.contiguous(), logits.contiguous(),
                    reference_points.float().contiguous(), key_padding_mask, _deterministic())
            else:
                output = MSDeformAttnFusedFunction.apply(
                    value.contiguous(), spatial_shapes, level_start_index, offsets.contiguous(),
                    logits.contiguous(), reference_points.float().contiguous(), key_padding_mask)
            if output.dtype != io_dtype:
                output = output.to(io_dtype)
            output = self.output_proj(output)
            if not self.batch_first:
                output = output.permute(1, 0, 2)
            if not kwargs.get("add_identity", True):      # the caller fuses the residual into its LayerNorm (epilogue.py)
                return self.dropout(output)
            return self.dropout(output) + identity

        weights = logits.softmax(-1).view(bs, num_query, H, L, P)

        if reference_points.shape[-1] == 2:
            normalizer = torch.stack([spatial_shapes[..., 1], spatial_shapes[..., 0]], -1)
            locations = reference_points[:, :, None, :, None, :] + offsets / normalizer[None, None, None, :, None, :]
        elif reference_points.shape[-1] == 4:
            locations = (reference_points[:, :, None, :, None, :2]
                         + offsets / P * reference_points[:, :, None, :, None, 2:] * 0.5)
        else:
            raise ValueError(
                f"Last dim of reference_points must be 2 or 4, but get {reference_points.shape[-1]} instead.")

        aux = torch.float64 if value.dtype == torch.float64 else torch.float32
        output = MultiScaleDeformableAttnFunction.apply(
            value.contiguous(), spatial_shapes, level_start_index, locations.to(aux).contiguous(),
            weights.to(aux).contiguous(), self.im2col_step)
        if output.dtype != io_dtype:
            output = output.to(io_dtype)

        output = self.output_proj(output)
        if not self.batch_first:
            output = output.permute(1, 0, 2)
        if not kwargs.get("add_identity", True):
            return self.dropout(output)
        return self.dropout(output) + identity

"""Callers of the op on the encoder side (SURVEY.md section 8f-2 / 8f-3): the glue that produces the op's
inputs and the encoder layer / stack that wraps it.  PyTorch code (the GEMMs, LayerNorm and FFN stay
library kernels); what changes relative to the reference is host behaviour: level shapes are kept on
the host as well as on the device, so nothing here synchronises, and a whole stack is CUDA-graph
capturable (tests/test_module_gpu.py).

Mirrors, with the same sub-module names so DINO / vCLR checkpoints load:
  flatten_levels        DINOTransformer.forward, projects/vCLR_deformable_mask/modeling/dino_transformer.py:372-398
  get_valid_ratio       dino_transformer.py:353-361
  get_reference_points  dino_transformer.py:322-351
  DeformableEncoderLayer  BaseTransformerLayer with ("self_attn","norm","ffn","norm")
                          (detrex/layers/transformer.py:29-192, detrex/layers/mlp.py:58-132), as built by
                          DINOTransformerEncoder (dino_transformer.py:46-65)
  DeformableEncoder     DINOTransformerEncoder (dino_transformer.py:32-106)
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn as nn

from .epilogue import add_layer_norm, add_layer_norm_supported
from .module import MultiScaleDeformableAttention


def get_valid_ratio(mask: torch.Tensor) -> torch.Tensor:
    """mask [B, H, W] (True = padding) -> [B, 2] (valid_w / W, valid_h / H)."""
    _, H, W = mask.shape
    valid_h = torch.sum(~mask[:, :, 0], 1)
    valid_w = torch.sum(~mask[:, 0, :], 1)
    return torch.stack([valid_w.float() / W, valid_h.float() / H], -1)


def get_reference_points(level_shapes: Sequence[Tuple[int, int]], valid_ratios: torch.Tensor, device) -> torch.Tensor:
    """Pixel-centre reference points of every level, [B, sum(H_l*W_l), L, 2].  `level_shapes` is the HOST list
    of (H_l, W_l): the reference iterates the device tensor (one sync per level)."""
    refs = []
    for lvl, (H, W) in enumerate(level_shapes):
        ys = torch.linspace(0.5, H - 0.5, H, dtype=torch.float32, device=device)
        xs = torch.linspace(0.5, W - 0.5, W, dtype=torch.float32, device=device)
        ref_y, ref_x = torch.meshgrid(ys, xs, indexing="ij")
        ref_y = ref_y.reshape(-1)[None] / (valid_ratios[:, None, lvl, 1] * H)
        ref_x = ref_x.reshape(-1)[None] / (valid_ratios[:, None, lvl, 0] * W)
        refs.append(torch.stack((ref_x, ref_y), -1))
    reference_points = torch.cat(refs, 1)
    return reference_points[:, :, None] * valid_ratios[:, None]


def flatten_levels(feats: Sequence[torch.Tensor], masks: Sequence[torch.Tensor], pos_embeds: Sequence[torch.Tensor],
                   level_embeds: Optional[torch.Tensor] = None):
    """[B,C,H_l,W_l] feature maps -> the flattened tensors the encoder consumes.
    Returns (feat [B,S,C], mask [B,S], pos [B,S,C], spatial_shapes [L,2] int64 on device,
    level_start_index [L] int64 on device, level_shapes host list, valid_ratios [B,L,2])."""
    feat_flat, mask_flat, pos_flat, shapes = [], [], [], []
    for lvl, (feat, mask, pos) in enumerate(zip(feats, masks, pos_embeds)):
        _, _, h, w = feat.shape
        shapes.append((h, w))
        pos = pos.flatten(2).transpose(1, 2)
        if level_embeds is not None:
            pos = pos + level_embeds[lvl].view(1, 1, -1)
        feat_flat.append(feat.flatten(2).transpose(1, 2))
        mask_flat.append(mask.flatten(1))
        pos_flat.append(pos)
    dev = feats[0].device
    spatial_shapes = torch.as_tensor(shapes, dtype=torch.long, device=dev)
    starts = [0]
    for h, w in shapes[:-1]:
        starts.append(starts[-1] + h * w)
    level_start_index = torch.as_tensor(starts, dtype=torch.long, device=dev)    # host arithmetic: no cumsum kernel
    valid_ratios = torch.stack([get_valid_ratio(m) for m in masks], 1)
    return (torch.cat(feat_flat, 1), torch.cat(mask_flat, 1), torch.cat(pos_flat, 1), spatial_shapes,
            level_start_index, shapes, valid_ratios)


class FFN(nn.Module):
    """Two-layer feed-forward block with identity connection; parameter names as detrex/layers/mlp.py:58-132
    (``layers.0.0`` and ``layers.1``)."""

    def __init__(self, embed_dim=256, feedforward_dim=1024, ffn_drop=0.0):
        super().__init__()
        self.embed_dim = embed_dim
        self.feedforward_dim = feedforward_dim
        self.layers = nn.Sequential(
            nn.Sequential(nn.Linear(embed_dim, feedforward_dim), nn.ReLU(inplace=True), nn.Dropout(ffn_drop)),
            nn.Linear(feedforward_dim, embed_dim),
            nn.Dropout(ffn_drop),
        )

    def forward(self, x, identity=None):
        return (x if identity is None else identity) + self.layers(x)


class DeformableEncoderLayer(nn.Module):
    """self_attn (MSDeformAttn) -> norm -> ffn -> norm, post-norm, batch-first
    (BaseTransformerLayer with operation_order ("self_attn", "norm", "ffn", "norm"), detrex/layers/transformer.py:152-192).
    Both ``x + identity; norm(x)`` epilogues run as ONE fused kernel each (ir_ads_b200/epilogue.py) where it applies
    (CUDA, float32 / bfloat16); ``fuse_epilogue = False`` restores the op-by-op composition.
    ``packing=PackedLevels`` (ir_ads_b200/packing.py): ``query`` / ``query_pos`` are packed ``[T, C]`` rows and
    ``reference_points`` ``[T, L, 2]`` (packed_reference_points); every step after the op works row by row."""

    def __init__(self, embed_dim=256, num_heads=8, feedforward_dim=1024, attn_dropout=0.1, ffn_dropout=0.1,
                 num_feature_levels=4, num_points=4):
        super().__init__()
        self.embed_dim = embed_dim
        self.pre_norm = False
        self.attentions = nn.ModuleList([MultiScaleDeformableAttention(
            embed_dim=embed_dim, num_heads=num_heads, num_levels=num_feature_levels, num_points=num_points,
            dropout=attn_dropout, batch_first=True)])
        self.ffns = nn.ModuleList([FFN(embed_dim, feedforward_dim, ffn_dropout)])
        self.norms = nn.ModuleList([nn.LayerNorm(embed_dim), nn.LayerNorm(embed_dim)])
        self.fuse_epilogue = True

    def forward(self, query, query_pos=None, query_key_padding_mask=None, reference_points=None,
                spatial_shapes=None, level_start_index=None, **kwargs):
        # self_attn: key = value = query, key_padding_mask = query_key_padding_mask (transformer.py:152-167)
        if self.fuse_epilogue and add_layer_norm_supported(query):
            attn = self.attentions[0](query, None, None, None, query_pos=query_pos,
                                      key_padding_mask=query_key_padding_mask, reference_points=reference_points,
                                      spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                                      level_shapes=kwargs.get("level_shapes"), packing=kwargs.get("packing"),
                                      add_identity=False)
            query = add_layer_norm(attn, query, self.norms[0])                    # norm(attn + identity)
            return add_layer_norm(self.ffns[0].layers(query), query, self.norms[1])   # norm(ffn(x) + x)
        query = self.attentions[0](query, None, None, None, query_pos=query_pos,
                                   key_padding_mask=query_key_padding_mask, reference_points=reference_points,
                                   spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                                   level_shapes=kwargs.get("level_shapes"), packing=kwargs.get("packing"))
        query = self.norms[0](query)
        query = self.ffns[0](query)
        return self.norms[1](query)


class DeformableEncoder(nn.Module):
    """num_layers x DeformableEncoderLayer (+ optional final LayerNorm), DINOTransformerEncoder's contract.
    ``packing=`` is handed to every layer (a packed batch, see DeformableEncoderLayer)."""

    def __init__(self, embed_dim=256, num_heads=8, feedforward_dim=1024, attn_dropout=0.1, ffn_dropout=0.1,
                 num_layers=6, post_norm=False, num_feature_levels=4, num_points=4):
        super().__init__()
        self.num_layers = num_layers
        self.embed_dim = embed_dim
        self.layers = nn.ModuleList([
            DeformableEncoderLayer(embed_dim, num_heads, feedforward_dim, attn_dropout, ffn_dropout,
                                   num_feature_levels, num_points) for _ in range(num_layers)])
        self.post_norm_layer = nn.LayerNorm(embed_dim) if post_norm else None

    def forward(self, query, key=None, value=None, query_pos=None, query_key_padding_mask=None, **kwargs):
        for layer in self.layers:
            query = layer(query, query_pos=query_pos, query_key_padding_mask=query_key_padding_mask, **kwargs)
        if self.post_norm_layer is not None:
            query = self.post_norm_layer(query)
        return query


# ------------------------------------------------------------------------------------------------
# decoder side (SURVEY 8f-3): what DINOTransformerDecoder feeds the cross-attention op
# ------------------------------------------------------------------------------------------------
def decoder_reference_points_input(reference_points: torch.Tensor, valid_ratios: torch.Tensor) -> torch.Tensor:
    """Per-level reference boxes / points for the decoder's MSDeformAttn cross-attention
    (dino_transformer.py:186-194): ``[B, Q, 4]`` boxes are scaled by ``cat(valid_ratios, valid_ratios)``,
    ``[B, Q, 2]`` points by ``valid_ratios``; result ``[B, Q, L, 4 | 2]`` -- the module's ``reference_points``."""
    if reference_points.shape[-1] == 4:
        return reference_points[:, :, None] * torch.cat([valid_ratios, valid_ratios], -1)[:, None]
    if reference_points.shape[-1] == 2:
        return reference_points[:, :, None] * valid_ratios[:, None]
    raise ValueError(f"reference_points last dim must be 2 or 4, got {reference_points.shape[-1]}")


class DeformableCrossAttentionBlock(nn.Module):
    """The MSDeformAttn cross-attention + norm step of a DINO decoder layer (``cross_attn`` then ``norm`` in
    the layer's operation order, dino_transformer.py:124-150): queries attend to the encoder memory through
    per-level reference boxes.  The decoder's self-attention (nn.MultiheadAttention) and FFN stay PyTorch.
    ``packing=PackedLevels``: ``memory`` is the packed ``[T_v, C]`` encoder output of that batch (no key_padding_mask);
    queries stay ``[B, Q, C]`` and attend to their own image's rows (``packing.cross(Q)``).  ``level_shapes``: the host
    ``(H_l, W_l)`` list, handed to the module's shape check (no device read; what torch.compile needs)."""

    def __init__(self, embed_dim=256, num_heads=8, attn_dropout=0.1, num_feature_levels=4, num_points=4):
        super().__init__()
        self.attn = MultiScaleDeformableAttention(embed_dim=embed_dim, num_heads=num_heads,
                                                  num_levels=num_feature_levels, num_points=num_points,
                                                  dropout=attn_dropout, batch_first=True)
        self.norm = nn.LayerNorm(embed_dim)

    def forward(self, query, memory, query_pos, reference_points, valid_ratios, spatial_shapes, level_start_index,
                key_padding_mask=None, packing=None, level_shapes=None):
        ref_in = decoder_reference_points_input(reference_points, valid_ratios)
        if packing is not None:
            B, Q, C = query.shape
            cross = packing.cross(Q)
            rows = (query.reshape(B * Q, C), None if query_pos is None else query_pos.reshape(B * Q, C))
            ref_rows = ref_in.reshape(B * Q, ref_in.shape[2], ref_in.shape[3])
            if add_layer_norm_supported(query):
                out = self.attn(rows[0], None, memory, None, query_pos=rows[1], key_padding_mask=key_padding_mask,
                                reference_points=ref_rows, packing=cross, add_identity=False)
                return add_layer_norm(out, rows[0], self.norm).view(B, Q, -1)
            out = self.attn(rows[0], None, memory, None, query_pos=rows[1], key_padding_mask=key_padding_mask,
                            reference_points=ref_rows, packing=cross)
            return self.norm(out).view(B, Q, -1)
        if add_layer_norm_supported(query):
            out = self.attn(query, None, memory, None, query_pos=query_pos, key_padding_mask=key_padding_mask,
                            reference_points=ref_in, spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                            level_shapes=level_shapes, add_identity=False)
            return add_layer_norm(out, query, self.norm)
        out = self.attn(query, None, memory, None, query_pos=query_pos, key_padding_mask=key_padding_mask,
                        reference_points=ref_in, spatial_shapes=spatial_shapes, level_start_index=level_start_index,
                        level_shapes=level_shapes)
        return self.norm(out)

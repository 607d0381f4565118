"""Padding-free ("packed") batches for the encoder and the decoder's cross-attention.

A detection batch pads every image to the largest height and width in the batch, and ``flatten_levels`` hands the
encoder ``[B, S, C]`` tensors in which every padded pixel is a query row that runs through the op, the four
projections, both LayerNorms and the FFN of every layer -- work that cannot reach a valid token.  A packed batch keeps
the valid pixels only, the equivalent of FlashAttention's "varlen" interface:

  * image ``b``'s pixels of level ``l`` are its valid top-left rectangle ``h_v[b,l] x w_v[b,l]`` of the padded level
    ``(H_l, W_l)``, row-major with row pitch ``w_v``; levels follow each other, images are concatenated: ``[T_v, C]``;
  * DETR-family masks come from nearest-interpolating the image mask (``F.interpolate(mask, size)``), so they are
    always such rectangles; :func:`valid_extents` computes them on the host, so no step syncs to count tokens;
  * queries come in per-image ranges: the value tokens themselves (encoder self-attention) or ``Q`` per image
    (decoder cross-attention over packed memory, :meth:`PackedLevels.cross`).

Every valid token gets the result of the padded route with the padding mask (include/msda.h, msda_packed_*).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from .encoder import get_reference_points

_META_FIXED = 4   # per image {value_start, value_count, query_start, query_count}, then L x {h_v, w_v, level start}


def _nearest_valid(valid: int, in_size: int, out_size: int) -> int:
    """How many of ``out_size`` nearest-interpolated positions read one of the first ``valid`` of ``in_size`` input
    positions: ATen's nearest source index (upsample nearest, no explicit scale) in its float32 arithmetic,
    ``min(floor(i * (float(in) / out)), in - 1)``, which is non-decreasing in ``i``."""
    if out_size == in_size:
        return valid
    if out_size == 2 * in_size:
        return min(2 * valid, out_size)
    scale = np.float32(in_size) / np.float32(out_size)
    src = np.floor(np.arange(out_size, dtype=np.float32) * scale).astype(np.int64)
    return int(np.count_nonzero(np.minimum(src, in_size - 1) < valid))


def valid_extents(image_sizes: Sequence[Tuple[int, int]], padded_hw: Tuple[int, int],
                  level_shapes: Sequence[Tuple[int, int]]) -> List[List[Tuple[int, int]]]:
    """Host integers ``[b][l] = (h_v, w_v)``: the valid rectangle of image ``b`` (``image_sizes[b] = (h, w)``, its
    top-left corner of the ``padded_hw`` batch tensor) on level ``l`` of shape ``level_shapes[l] = (H_l, W_l)`` --
    exactly the un-masked region of ``F.interpolate(mask[None].float(), size=(H_l, W_l)).bool()`` for the image mask
    ``mask[y, x] = y >= h or x >= w``."""
    Hp, Wp = int(padded_hw[0]), int(padded_hw[1])
    out = []
    for h, w in image_sizes:
        if not (0 <= h <= Hp and 0 <= w <= Wp):
            raise ValueError(f"image size {(h, w)} outside the padded size {(Hp, Wp)}")
        out.append([(_nearest_valid(int(h), Hp, int(H)), _nearest_valid(int(w), Wp, int(W))) for H, W in level_shapes])
    return out


class PackedLevels:
    """Host counts and device metadata of one packed batch.

    ``extents[b][l] = (h_v, w_v)`` (from :func:`valid_extents`), ``level_shapes`` the padded ``(H_l, W_l)``.  Queries
    are the value tokens (encoder form); :meth:`cross` gives the decoder form.  Build it once per batch: the
    constructor copies its small tables to ``device`` once, and nothing that uses it syncs or copies from the host, so
    a packed encoder forward + backward is CUDA-graph capturable.

    Host attributes: ``batch``, ``num_levels``, ``level_shapes``, ``extents``, ``value_counts``, ``query_counts``,
    ``total_value``, ``total_query``, ``max_value``, ``max_query``, ``padded_len`` (``S = sum H_l*W_l``).
    Device tensors: ``spatial_shapes [L, 2]``, ``level_start_index [L]`` (padded layout), ``meta`` (the kernels'
    per-image table), ``value_index [T_v]`` / ``query_index [T_q]`` (row of every token in the padded
    ``[B * S]`` / ``[B * query_pad]`` layout), ``padding_mask [B, S]`` (True = padded) and ``valid_ratios [B, L, 2]``
    (``get_valid_ratio`` of the interpolated masks, bit for bit)."""

    def __init__(self, extents: Sequence[Sequence[Tuple[int, int]]], level_shapes: Sequence[Tuple[int, int]],
                 device, num_queries: Optional[int] = None, _tables=None):
        self.level_shapes = [(int(h), int(w)) for h, w in level_shapes]
        self.extents = [[(int(h), int(w)) for h, w in img] for img in extents]
        self.batch, self.num_levels = len(self.extents), len(self.level_shapes)
        self.device = torch.device(device)
        L = self.num_levels
        for img in self.extents:
            if len(img) != L or any(not (0 <= hv <= H and 0 <= wv <= W)
                                    for (hv, wv), (H, W) in zip(img, self.level_shapes)):
                raise ValueError("every image needs one valid rectangle inside each padded level")
        starts = [0]
        for H, W in self.level_shapes:
            starts.append(starts[-1] + H * W)
        self.padded_len = starts[-1]
        self.value_counts = [sum(hv * wv for hv, wv in img) for img in self.extents]
        self.num_queries = num_queries
        self.query_counts = list(self.value_counts) if num_queries is None else [int(num_queries)] * self.batch
        self.query_pad = self.padded_len if num_queries is None else int(num_queries)
        self.total_value, self.total_query = sum(self.value_counts), sum(self.query_counts)
        self.max_value = max(self.value_counts, default=0)
        self.max_query = max(self.query_counts, default=0)

        meta, v0, q0 = [], 0, 0
        for img, nv, nq in zip(self.extents, self.value_counts, self.query_counts):
            row, inner = [v0, nv, q0, nq], 0
            for hv, wv in img:
                row += [hv, wv, inner]
                inner += hv * wv
            meta.append(row)
            v0, q0 = v0 + nv, q0 + nq
        dev = self.device
        self.meta = torch.tensor(meta, dtype=torch.int64).reshape(self.batch, _META_FIXED + 3 * L).to(dev)
        if _tables is not None:   # the decoder form shares the value-side tables of its encoder form
            (self.spatial_shapes, self.level_start_index, self.value_index, self.padding_mask,
             self.valid_ratios) = _tables
        else:
            self.spatial_shapes = torch.tensor(self.level_shapes, dtype=torch.int64).reshape(L, 2).to(dev)
            self.level_start_index = torch.tensor(starts[:-1], dtype=torch.int64).to(dev)
            index, mask = [], np.ones((self.batch, self.padded_len), dtype=bool)
            for b, img in enumerate(self.extents):
                for (hv, wv), (H, W), s in zip(img, self.level_shapes, starts):
                    rows = (s + np.arange(hv)[:, None] * W + np.arange(wv)[None, :]).reshape(-1)
                    mask[b, rows] = False
                    index.append(b * self.padded_len + rows)
            self.value_index = torch.from_numpy(np.concatenate(index) if index else np.zeros(0, np.int64)).to(dev)
            self.padding_mask = torch.from_numpy(mask).to(dev)
            # get_valid_ratio: (count of valid columns / W, count of valid rows / H) as a float32 division
            ratios = [[(np.float32(wv) / np.float32(W), np.float32(hv) / np.float32(H))
                       for (hv, wv), (H, W) in zip(img, self.level_shapes)] for img in self.extents]
            self.valid_ratios = torch.tensor(np.asarray(ratios, dtype=np.float32).reshape(self.batch, L, 2)).to(dev)
        if num_queries is None:
            self.query_index = self.value_index
        else:
            self.query_index = torch.arange(self.total_query, dtype=torch.int64, device=dev)
        self._cross = {}

    def cross(self, num_queries: int) -> "PackedLevels":
        """The decoder form over this packed memory: ``num_queries`` queries per image, rows ``b*Q .. (b+1)*Q``
        (cached per ``num_queries``)."""
        hit = self._cross.get(int(num_queries))
        if hit is None:
            hit = PackedLevels(self.extents, self.level_shapes, self.device, num_queries=int(num_queries),
                               _tables=(self.spatial_shapes, self.level_start_index, self.value_index,
                                        self.padding_mask, self.valid_ratios))
            self._cross[int(num_queries)] = hit
        return hit

    def padded_fraction(self) -> float:
        """Share of the padded ``[B, S]`` tokens that are padding."""
        full = self.batch * self.padded_len
        return 1.0 - self.total_value / full if full else 0.0


def pack_levels(feats: Sequence[torch.Tensor], packing: PackedLevels,
                pos_embeds: Optional[Sequence[torch.Tensor]] = None, level_embeds: Optional[torch.Tensor] = None):
    """Packed twin of ``encoder.flatten_levels``: ``[B, C, H_l, W_l]`` maps (padded as the batch is) -> ``feat
    [T_v, C]`` and, with ``pos_embeds``, ``pos [T_v, C]`` (plus ``level_embeds[l]`` as flatten_levels adds it) -- the
    rows of flatten_levels' ``[B, S, C]`` tensors at the valid pixels, in packed order."""
    def flat(maps, add_level):
        parts = []
        for lvl, m in enumerate(maps):
            t = m.flatten(2).transpose(1, 2)
            if add_level and level_embeds is not None:
                t = t + level_embeds[lvl].view(1, 1, -1)
            parts.append(t)
        x = torch.cat(parts, 1)
        return x.reshape(-1, x.shape[-1]).index_select(0, packing.value_index)

    feat = flat(feats, False)
    if pos_embeds is None:
        return feat
    return feat, flat(pos_embeds, True)


def packed_reference_points(packing: PackedLevels) -> torch.Tensor:
    """The encoder's reference points ``[T_v, L, 2]``: the valid rows of ``get_reference_points(level_shapes,
    valid_ratios)`` bit for bit (computed that way, on the device)."""
    ref = get_reference_points(packing.level_shapes, packing.valid_ratios, packing.device)
    return ref.reshape(-1, packing.num_levels, 2).index_select(0, packing.value_index)


def unpack_tokens(x: torch.Tensor, packing: PackedLevels, queries: bool = False):
    """``[T, C]`` packed rows -> ``([B, S, C]`` zero-padded, ``mask [B, S]`` True = padded) for code that wants the
    padded layout (two-stage proposals, say).  Differentiable.  ``queries=True`` unpacks query rows of a decoder
    form (``[B, Q, C]``, no padding)."""
    index, length = (packing.query_index, packing.query_pad) if queries else (packing.value_index, packing.padded_len)
    out = x.new_zeros((packing.batch * length,) + tuple(x.shape[1:])).index_copy(0, index, x)
    out = out.view((packing.batch, length) + tuple(x.shape[1:]))
    if queries and packing.num_queries is not None:
        return out, torch.zeros((packing.batch, length), dtype=torch.bool, device=x.device)
    return out, packing.padding_mask

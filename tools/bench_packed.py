"""Packed (padding-free) against padded batches: the fused MSDeformAttn op and the 6-layer encoder (fused add + LayerNorm
epilogues on), float32 and bf16 autocast, forward + backward, on 2-image batches.

Mixes: seeded draws from a detrex-like augmentation model -- shorter side from 480..800 step 32, longer side
capped at 1333, aspect ratios 1, 4:3, 3:2, 16:9 with both images of a batch in the same orientation (aspect-ratio
grouping), the batch padded to the largest height / width rounded up to 32 -- plus one mix of two equal images (no
padding: packed must not be slower there).  DINO-R50 levels: strides 8 / 16 / 32 / 64, 256 channels, 8 heads, 4
points.  Padded and packed alternate in one process; every timed pass reads one of several input sets, together
larger than the 126 MB L2.  Times are CUDA-event medians.  One JSON line per (workload, dtype, mix).

  python tools/bench_packed.py [--iters 20] [--warmup 3] [--mixes 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import random
import sys
from functools import partial

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ir_ads_b200.encoder import DeformableEncoder, get_reference_points  # noqa: E402
from ir_ads_b200.functional import MSDeformAttnFusedFunction, MSDeformAttnPackedFunction  # noqa: E402
from ir_ads_b200.packing import PackedLevels, packed_reference_points, valid_extents  # noqa: E402
from timing import card, timed  # noqa: E402

C, HEADS, L, P = 256, 8, 4, 4
DEV = torch.device("cuda")


def draw_mix(rng):
    aspect = rng.choice((1.0, 4 / 3, 3 / 2, 16 / 9))
    landscape = rng.random() < 0.5
    sizes = []
    for _ in range(2):
        s = rng.randrange(480, 801, 32)
        l = min(1333, int(round(s * aspect)))
        sizes.append((s, l) if landscape else (l, s))
    return sizes


def levels_of(padded):
    Hp, Wp = padded
    shapes = [(-(-Hp // s), -(-Wp // s)) for s in (8, 16, 32)]
    shapes.append((-(-shapes[-1][0] // 2), -(-shapes[-1][1] // 2)))   # the extra stride-2 conv of the last level
    return shapes


def make_packing(sizes):
    padded = (-(-max(h for h, _ in sizes) // 32) * 32, -(-max(w for _, w in sizes) // 32) * 32)
    shapes = levels_of(padded)
    return PackedLevels(valid_extents(sizes, padded, shapes), shapes, DEV)


def op_sets(pk, vdt, n, gen):
    """n input sets of the fused op, padded and packed (packed = the valid rows of the padded set)"""
    B, S, D = pk.batch, pk.padded_len, C // HEADS
    adt = torch.float32 if vdt == torch.float32 else vdt
    pad, packed = [], []
    for _ in range(n):
        v = torch.randn(B, S, HEADS, D, generator=gen).to(DEV, vdt)
        off = torch.randn(B, S, HEADS, L, P, 2, generator=gen).to(DEV, adt)
        lg = torch.randn(B, S, HEADS, L * P, generator=gen).to(DEV, adt)
        ref = get_reference_points(pk.level_shapes, pk.valid_ratios, DEV).contiguous()
        go = torch.randn(B, S, HEADS * D, generator=gen).to(DEV, vdt)
        flat = lambda t: t.reshape((B * S,) + tuple(t.shape[2:]))[pk.value_index].contiguous()  # noqa: E731
        packed.append([t.requires_grad_(i < 3) for i, t in enumerate(map(flat, (v, off, lg, ref)))] + [flat(go)])
        pad.append([t.requires_grad_(i < 3) for i, t in enumerate((v, off, lg, ref))] + [go])
    return pad, packed


def enc_sets(pk, n, gen):
    B, S = pk.batch, pk.padded_len
    ref_pad = get_reference_points(pk.level_shapes, pk.valid_ratios, DEV)
    ref_pk = packed_reference_points(pk)
    pad, packed = [], []
    for _ in range(n):
        x = torch.randn(B, S, C, generator=gen).to(DEV)
        pos = torch.randn(B, S, C, generator=gen).to(DEV)
        flat = lambda t: t.reshape(B * S, C)[pk.value_index].contiguous()  # noqa: E731
        packed.append((flat(x).requires_grad_(True), flat(pos), ref_pk))
        pad.append((x.requires_grad_(True), pos, ref_pad))
    return pad, packed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--mixes", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rng = random.Random(a.seed)
    mixes = [("model%d" % i, draw_mix(rng)) for i in range(a.mixes)] + [("equal", [(800, 1066), (800, 1066)])]
    gen = torch.Generator().manual_seed(a.seed)
    torch.manual_seed(a.seed)
    enc = DeformableEncoder(C, HEADS, 1024, 0.0, 0.0, num_layers=6, num_feature_levels=L, num_points=P).to(DEV)
    lines = []

    def emit(rec):
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))

    emit(card())
    for name, sizes in mixes:
        pk = make_packing(sizes)
        base = dict(mix=name, sizes=sizes, level_shapes=pk.level_shapes, tokens_padded=pk.batch * pk.padded_len,
                    tokens_packed=pk.total_value, padded_fraction=round(pk.padded_fraction(), 4))
        # ---- the op ----
        for vdt in (torch.float32, torch.bfloat16):
            pad, packed = op_sets(pk, vdt, 3, gen)

            def run_pad(s):
                out = MSDeformAttnFusedFunction.apply(s[0], pk.spatial_shapes, pk.level_start_index, s[1], s[2], s[3],
                                                      pk.padding_mask)
                out.backward(s[4])

            def run_pk(s):
                MSDeformAttnPackedFunction.apply(s[0], s[1], s[2], s[3], pk).backward(s[4])

            t = timed({"padded": [(partial(run_pad, s),) for s in pad],
                       "packed": [(partial(run_pk, s),) for s in packed]}, a.iters, a.warmup)
            (mp,), (mk,) = t["padded"], t["packed"]
            emit(dict(base, workload="op_fwd_bwd", dtype=str(vdt).replace("torch.", ""), padded_ms=mp, packed_ms=mk,
                      speedup=round(mp / mk, 3)))
            del pad, packed
        # ---- the 6-layer encoder ----
        pad, packed = enc_sets(pk, 2, gen)
        for amp in (False, True):
            def run_enc(s, packing):
                kw = dict(query_pos=s[1], reference_points=s[2], spatial_shapes=pk.spatial_shapes,
                          level_start_index=pk.level_start_index, level_shapes=pk.level_shapes)
                if packing:
                    kw["packing"] = pk
                else:
                    kw["query_key_padding_mask"] = pk.padding_mask
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
                    out = enc(s[0], **kw)
                out.float().sum().backward()

            t = timed({"padded": [(partial(run_enc, s, False),) for s in pad],
                       "packed": [(partial(run_enc, s, True),) for s in packed]}, a.iters, a.warmup)
            (mp,), (mk,) = t["padded"], t["packed"]
            emit(dict(base, workload="encoder6_fwd_bwd", dtype="bf16_autocast" if amp else "float32",
                      padded_ms=round(mp, 3), packed_ms=round(mk, 3), speedup=round(mp / mk, 3)))
        del pad, packed
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

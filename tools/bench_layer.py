#!/usr/bin/env python
"""Encoder-layer timing (SURVEY 8f-2): DeformableEncoderLayer forward+backward at the DINO-R50 encoder shape,
fused `add + LayerNorm` epilogues (ir_ads_b200/epilogue.py) vs the op-by-op composition.
Usage: python tools/bench_layer.py [--batch 8] [--iters 10]"""
import argparse
import json
import os
import sys
from functools import partial

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ir_ads_b200.encoder import DeformableEncoderLayer  # noqa: E402
from ir_ads_b200.workloads import LEVELS, _pixel_centres, level_tensors  # noqa: E402
from timing import card, timed  # noqa: E402


def run(batch, iters, fused, amp, dev="cuda:0"):
    levels = LEVELS["dino_r50"]
    shapes, lsi = level_tensors(levels, dev)
    S = sum(h * w for h, w in levels)
    torch.manual_seed(0)
    layer = DeformableEncoderLayer(attn_dropout=0.0, ffn_dropout=0.0).to(dev)
    layer.fuse_epilogue = fused
    ref = _pixel_centres(levels, dev)[None, :, None, :].expand(batch, S, 4, 2).contiguous()
    sets = [(torch.randn(batch, S, 256, device=dev, requires_grad=True), torch.randn(batch, S, 256, device=dev) * 0.1,
             torch.randn(batch, S, 256, device=dev)) for _ in range(3)]
    ctx = torch.autocast("cuda", dtype=torch.bfloat16) if amp else torch.autocast("cuda", enabled=False)

    def step(x, pos, go):
        with ctx:
            out = layer(x, query_pos=pos, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi,
                        level_shapes=levels)
        out.backward(go.to(out.dtype))
    return timed({"layer": [(partial(step, *s),) for s in sets]}, iters, 3)["layer"][0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    print(json.dumps(card()), flush=True)
    res = {"what": "DeformableEncoderLayer fwd+bwd, DINO-R50 800x1333 encoder shape, ms (median)", "batch": a.batch}
    for amp in (False, True):
        for fused in (True, False):
            res[f"{'bf16_autocast' if amp else 'fp32'}_{'fused_epilogue' if fused else 'op_by_op'}"] = round(
                run(a.batch, a.iters, fused, amp), 3)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

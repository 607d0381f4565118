#!/usr/bin/env python
"""DCNv3 backward: default route (float reds) vs the bit-reproducible one (MSDA_FLAG_DETERMINISTIC), on the
InternImage-T-like stages of tools/bench_dcnv3.py.  One process; per shape both are warmed up, then timed alternately
with CUDA events, median of --iters calls each.  The dense 3x3 stride-1 problems take the cell reduce.  Prints the card
name and power limit first, then one JSON line per shape (and dtype)."""
import argparse
import json
import os
import sys
from functools import partial

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ir_ads_b200 import _lib, dcnv3_backward, functional  # noqa: E402
from timing import card, timed  # noqa: E402

SHAPES = ((16, 200, 336, 4, 16), (16, 100, 168, 8, 16), (16, 50, 84, 16, 16), (16, 25, 42, 32, 16), (8, 100, 168, 8, 32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=25)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--dtypes", default="float32,bfloat16")
    a = ap.parse_args()
    print(json.dumps(card()), flush=True)
    dev = "cuda:0"
    for dname in a.dtypes.split(","):
        dtype = getattr(torch, dname)
        for (N, H, W, G, C) in SHAPES:
            g = torch.Generator(device=dev).manual_seed(0)
            inp = torch.randn(N, H, W, G * C, device=dev, generator=g).to(dtype)
            off = torch.randn(N, H, W, G * 18, device=dev, generator=g)
            mask = torch.softmax(torch.randn(N, H, W, G, 9, device=dev, generator=g), -1).reshape(N, H, W, G * 9)
            go = torch.randn(N, H, W, G * C, device=dev, generator=g).to(dtype)
            args = (3, 3, 1, 1, 1, 1, 1, 1, G, C, 1.0)

            def call(flags):
                with functional.kernel_flags(flags):
                    return dcnv3_backward(inp, off, mask, *args, go)

            modes = {"default": 0, "deterministic": _lib.FLAG_DETERMINISTIC}
            t = timed({k: [(partial(call, f),)] for k, f in modes.items()}, a.iters, a.warmup)
            # the two routes agree to float-summation accuracy (and the deterministic one with itself, bit for bit)
            d0, d1, d2 = call(0)[0].float(), call(modes["deterministic"])[0], call(modes["deterministic"])[0]
            row = {"shape": [N, H, W, G, C], "dtype": dname, "points": N * H * W * G * 9, "iters": a.iters,
                   "default_bwd_ms": t["default"][0], "det_bwd_ms": t["deterministic"][0],
                   "det_reproducible": bool(torch.equal(d1, d2)),
                   "det_vs_default_max_rel": float((d1.float() - d0).abs().max() / d0.abs().max().clamp_min(1e-30))}
            row["det_over_default"] = round(row["det_bwd_ms"] / row["default_bwd_ms"], 3)
            print(json.dumps(row), flush=True)
            del inp, off, mask, go
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

"""Eager against torch.compile (default mode and reduce-overhead) for the 6-layer encoder, forward + backward.

Workloads: cfg2 (DINO-R50 levels at 800x1333, B=8) and cfg4 (VOC-shape levels, B=2), unpadded, float32 and bf16
autocast, fused add + LayerNorm epilogues on.  The three variants are compiled and warmed up first, then timed in
alternating rounds in one process; every timed pass reads one of several input sets, together larger than the 126 MB
L2.  Times are CUDA-event medians of whole steps (forward, backward, gradient accumulation).  One JSON line per
(workload, dtype, variant), the card's name and power limit in each.

  python tools/bench_compile.py [--iters 20] [--warmup 3] [--rounds 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ir_ads_b200.encoder import DeformableEncoder, get_reference_points  # noqa: E402
from ir_ads_b200.workloads import LEVELS  # noqa: E402

C, HEADS = 256, 8
DEV = torch.device("cuda")
WORKLOADS = {"cfg2": ("dino_r50", 8), "cfg4": ("voc", 2)}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else torch.cuda.get_device_name()


def inputs(levels, batch, n_sets, gen):
    S = sum(h * w for h, w in levels)
    ratios = torch.ones(batch, len(levels), 2, device=DEV)
    ref = get_reference_points(levels, ratios, DEV)
    sets = [(torch.randn(batch, S, C, generator=gen).to(DEV).requires_grad_(True),
             torch.randn(batch, S, C, generator=gen).to(DEV)) for _ in range(n_sets)]
    return sets, ref


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--workloads", default="cfg2,cfg4")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = card()
    lines = []
    for name in args.workloads.split(","):
        level_key, batch = WORKLOADS[name]
        levels = [tuple(x) for x in LEVELS[level_key]]
        shapes = torch.tensor(levels, dtype=torch.int64, device=DEV)
        starts = torch.tensor([0] + [sum(h * w for h, w in levels[:i + 1]) for i in range(len(levels) - 1)],
                              dtype=torch.int64, device=DEV)
        gen = torch.Generator().manual_seed(0)
        torch.manual_seed(0)
        enc = DeformableEncoder(C, HEADS, 1024, 0.0, 0.0, num_layers=6).to(DEV)
        # enough sets to exceed L2 with their activations: each set is 2 * B * S * C * 4 bytes
        per_set = 2 * batch * sum(h * w for h, w in levels) * C * 4
        sets, ref = inputs(levels, batch, max(2, -(-256 * 2 ** 20 // per_set)), gen)

        def step(q, pos):
            out = enc(q, query_pos=pos, reference_points=ref, spatial_shapes=shapes, level_start_index=starts,
                      level_shapes=levels)
            out.float().square().mean().backward()
            return out

        for dtype in ("float32", "bf16"):
            ac = dtype == "bf16"

            def wrap(fn):
                def run(s):
                    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac):
                        return fn(*s)
                return run

            variants = {"eager": wrap(step)}
            variants["compile"] = wrap(torch.compile(step))
            ro = torch.compile(step, mode="reduce-overhead")

            def ro_step(s, _ro=ro):
                torch.compiler.cudagraph_mark_step_begin()
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac):
                    return _ro(*s)
            variants["reduce-overhead"] = ro_step
            for fn in variants.values():                 # compile and warm up every variant before timing any
                for i in range(args.warmup):
                    fn(sets[i % len(sets)])
            torch.cuda.synchronize()
            times = {k: [] for k in variants}
            for _ in range(args.rounds):
                for k, fn in variants.items():
                    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.iters + 1)]
                    ev[0].record()
                    for i in range(args.iters):
                        fn(sets[i % len(sets)])
                        ev[i + 1].record()
                    torch.cuda.synchronize()
                    times[k] += [ev[i].elapsed_time(ev[i + 1]) for i in range(args.iters)]
            base = statistics.median(times["eager"])
            for k, t in times.items():
                med = statistics.median(t)
                rec = {"workload": name, "batch": batch, "dtype": dtype, "variant": k, "median_ms": round(med, 3),
                       "p10_ms": round(sorted(t)[len(t) // 10], 3), "p90_ms": round(sorted(t)[len(t) * 9 // 10], 3),
                       "speedup_vs_eager": round(base / med, 3), "samples": len(t), "gpu": gpu}
                print(json.dumps(rec), flush=True)
                lines.append(rec)
            for p in enc.parameters():
                p.grad = None
            torch._dynamo.reset()
    if args.out:
        with open(args.out, "w") as f:
            f.writelines(json.dumps(r) + "\n" for r in lines)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Module-level timing (SURVEY 8d: "module-level (with projections) ... reported separately"):
MultiScaleDeformableAttention forward+backward at the encoder / decoder shapes, fused vs step-by-step
pre-op chain, next to the same module driving the REFERENCE's CUDA kernels (oracle/_ref).
Usage: python tools/bench_module.py [--batch 8] [--iters 10]"""
import argparse
import json
import os
import statistics
import sys
from functools import partial

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ir_ads_b200 import MultiScaleDeformableAttention  # noqa: E402
from ir_ads_b200 import module as msda_module  # noqa: E402
from ir_ads_b200.workloads import LEVELS, level_tensors  # noqa: E402
from timing import card, timed  # noqa: E402


class RefKernelFunction(torch.autograd.Function):
    """The reference's autograd Function (multi_scale_deform_attn.py:44-93) over its own kernels."""

    @staticmethod
    def forward(ctx, value, shapes, lsi, loc, w, step):
        from oracle import ref_cuda
        ctx.save_for_backward(value, shapes, lsi, loc, w)
        return ref_cuda.forward(value, shapes, lsi, loc, w)

    @staticmethod
    def backward(ctx, go):
        from oracle import ref_cuda
        value, shapes, lsi, loc, w = ctx.saved_tensors
        gv, gl, gw = ref_cuda.backward(go.contiguous(), value, shapes, lsi, loc, w)
        return gv, None, None, gl, gw, None


def run(kind, batch, iters, mode, dev="cuda:0", amp=None, masked=False):
    levels = LEVELS["dino_r50"]
    shapes, lsi = level_tensors(levels, dev)
    S = sum(h * w for h, w in levels)
    Q = S if kind == "encoder" else 2000
    torch.manual_seed(0)
    m = MultiScaleDeformableAttention(dropout=0.0, batch_first=True).to(dev)
    with torch.no_grad():
        m.sampling_offsets.weight.normal_(0, 0.02)
        m.attention_weights.weight.normal_(0, 0.1)
    m.fuse_pre_ops = mode == "fused"
    saved = msda_module.MultiScaleDeformableAttnFunction
    if mode == "reference_kernels":
        msda_module.MultiScaleDeformableAttnFunction = RefKernelFunction
    try:
        sets = []
        for i in range(3):
            q = torch.randn(batch, Q, 256, device=dev, requires_grad=True)
            val = None if kind == "encoder" else torch.randn(batch, S, 256, device=dev)
            ref = torch.rand(batch, Q, 4, 2 if kind == "encoder" else 4, device=dev)
            go = torch.randn(batch, Q, 256, device=dev)
            sets.append((q, val, ref, go))
        # batch-padding pattern: the right ~10 % of every level of every second image is padding
        mask = None
        if masked:
            mask = torch.zeros(batch, S, dtype=torch.bool, device=dev)
            start = 0
            for h, w in levels:
                mm = torch.zeros(h, w, dtype=torch.bool, device=dev)
                mm[:, (9 * w) // 10:] = True
                mask[1::2, start:start + h * w] = mm.reshape(-1)
                start += h * w

        def step(q, val, ref, go):
            with torch.autocast("cuda", dtype=amp, enabled=amp is not None):
                out = m(q, value=val, key_padding_mask=mask, reference_points=ref, spatial_shapes=shapes,
                        level_start_index=lsi)
            out.backward(go.to(out.dtype))
            # so that the next call assigns its gradients instead of adding to these; after the launches, so the host
            # work overlaps the backward kernels
            q.grad = None
            m.zero_grad(set_to_none=True)

        t = timed({mode: [(partial(step, *s),) for s in sets]}, iters, 3)[mode][0]
    finally:
        msda_module.MultiScaleDeformableAttnFunction = saved
    pts = batch * Q * 8 * 4 * 4
    return {"kind": kind, "batch": batch, "mode": mode, "amp": str(amp), "key_padding_mask": masked, "ms": round(t, 3),
            "gpts_s": round(pts / t / 1e6, 3)}


def run_stack(batch, iters, graph, amp=None, dev="cuda:0"):
    """6-layer DeformableEncoder (MSDA + LayerNorm + FFN per layer) forward+backward at the DINO-R50 shape."""
    from ir_ads_b200 import encoder
    levels = LEVELS["dino_r50"]
    shapes, lsi = level_tensors(levels, dev)
    S = sum(h * w for h, w in levels)
    torch.manual_seed(0)
    enc = encoder.DeformableEncoder(attn_dropout=0.0, ffn_dropout=0.0).to(dev)
    x = torch.randn(batch, S, 256, device=dev, requires_grad=True)
    pos = torch.randn(batch, S, 256, device=dev)
    ref = encoder.get_reference_points(levels, torch.ones(batch, 4, 2, device=dev), dev)
    go = torch.randn(batch, S, 256, device=dev)

    def step():
        with torch.autocast("cuda", dtype=amp, enabled=amp is not None):
            out = enc(x, query_pos=pos, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi)
        out.backward(go.to(out.dtype))

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    runner = step
    if graph:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step()
        runner = g.replay
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        runner()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    t = statistics.median(times)
    pts = 6 * batch * S * 8 * 4 * 4
    return {"kind": "encoder_stack_6_layers", "batch": batch, "mode": "cuda_graph" if graph else "eager",
            "amp": str(amp), "ms": round(t, 3), "gpts_s": round(pts / t / 1e6, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default="")
    ap.add_argument("--mask-only", action="store_true", help="only the key_padding_mask comparison (fused vs unfused)")
    a = ap.parse_args()
    rows = [card()]
    print(json.dumps(rows[0]), flush=True)
    for kind in ("encoder", "decoder"):
        for mode in ("fused", "unfused"):
            for amp in (None, torch.bfloat16):
                r = run(kind, a.batch, a.iters, mode, amp=amp, masked=True)
                rows.append(r)
                print(json.dumps(r), flush=True)
    if a.mask_only:
        return
    for kind in ("encoder", "decoder"):
        for b in sorted({a.batch, 1}):
            for mode in ("fused", "unfused", "reference_kernels"):
                r = run(kind, b, a.iters, mode)
                rows.append(r)
                print(json.dumps(r), flush=True)
        for mode in ("fused", "unfused"):
            r = run(kind, a.batch, a.iters, mode, amp=torch.bfloat16)
            rows.append(r)
            print(json.dumps(r), flush=True)
    for b in sorted({a.batch, 1}):
        for graph in (False, True):
            for amp in (None, torch.bfloat16):
                r = run_stack(b, a.iters, graph, amp)
                rows.append(r)
                print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()

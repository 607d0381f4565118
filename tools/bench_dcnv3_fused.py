#!/usr/bin/env python
"""Fused DCNv3 module path (mask softmax inside the kernels) against the unfused route, on the InternImage-T-like stages
of tools/bench_dcnv3.py (3x3, stride 1, pad 1).  One process; per shape and measurement both sides are warmed up,
then timed alternately with CUDA events, median of --iters.  Inputs rotate over enough copies that each timed call
reads a working set larger than the 126 MB L2.  Prints the card name and power limit first, then one JSON line per
shape:
  core   fused forward (DCNv3FusedFunction) vs torch.softmax + DCNv3Function forward, and the two backwards
         (fused kernel vs the core backward + softmax backward of autograd), float32 input
  module DCNv3 module forward + backward, fused route vs the composition it replaced, float32 and under float16
         autocast, with the peak memory of each route."""
import argparse
import json
import os
import sys
from functools import partial

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ir_ads_b200 import DCNv3Function, DCNv3FusedFunction  # noqa: E402
from ir_ads_b200.dcnv3 import DCNv3  # noqa: E402
from timing import card, rotations, timed  # noqa: E402

SHAPES = ((16, 200, 336, 4, 16), (16, 100, 168, 8, 16), (16, 50, 84, 16, 16), (16, 25, 42, 32, 16), (8, 100, 168, 8, 32))


def softmax_rows(logits, G):
    N, H, W, _ = logits.shape
    return torch.softmax(logits.view(N, H, W, G, -1), -1).view(N, H, W, -1)


def composed_forward(m, input):
    """the DCNv3 module's forward before the fused route: F.softmax, .type(dtype), DCNv3Function"""
    N, H, W, _ = input.shape
    x = m.input_proj(input)
    x1 = m.dw_conv(input.permute(0, 3, 1, 2))
    offset = m.offset(x1)
    mask = torch.nn.functional.softmax(m.mask(x1).reshape(N, H, W, m.group, -1), -1).reshape(N, H, W, -1).type(x.dtype)
    x = DCNv3Function.apply(x.contiguous(), offset.contiguous(), mask.contiguous(), m.kernel_size, m.kernel_size,
                            m.stride, m.stride, m.pad, m.pad, m.dilation, m.dilation, m.group, m.group_channels,
                            m.offset_scale, 256)
    return m.output_proj(x)


def core(N, H, W, G, C, iters, warmup):
    dev = "cuda:0"
    K, args = 9, (3, 3, 1, 1, 1, 1, 1, 1, G, C, 1.0)
    set_bytes = N * H * W * (G * C * 4 * 2 + G * K * 3 * 4)
    n_rot = rotations(set_bytes, 1, 8)
    g = torch.Generator(device=dev).manual_seed(0)
    sets = []
    for _ in range(n_rot):
        inp = torch.randn(N, H, W, G * C, device=dev, generator=g).requires_grad_(True)
        off = torch.randn(N, H, W, G * K * 2, device=dev, generator=g).requires_grad_(True)
        lg = torch.randn(N, H, W, G * K, device=dev, generator=g).requires_grad_(True)
        go = torch.randn(N, H, W, G * C, device=dev, generator=g)
        sets.append((inp, off, lg, go))
    with torch.no_grad():
        fwd = {k: t for k, (t,) in timed({
            "fused": [(partial(DCNv3FusedFunction.apply, *s[:3], *args, 256),) for s in sets],
            "unfused": [(lambda s=s: DCNv3Function.apply(s[0], s[1], softmax_rows(s[2], G), *args, 256),)
                        for s in sets],
        }, iters, warmup).items()}
    outs = {"fused": [DCNv3FusedFunction.apply(*s[:3], *args, 256) for s in sets],
            "unfused": [DCNv3Function.apply(s[0], s[1], softmax_rows(s[2], G), *args, 256) for s in sets]}
    bwd = {k: t for k, (t,) in timed({k: [(partial(torch.autograd.grad, o, s[:3], s[3], retain_graph=True),)
                                             for o, s in zip(outs[k], sets)] for k in outs}, iters, warmup).items()}
    a = torch.autograd.grad(outs["fused"][0], sets[0][:3], sets[0][3], retain_graph=True)
    b = torch.autograd.grad(outs["unfused"][0], sets[0][:3], sets[0][3], retain_graph=True)
    rel = {k: float((x - y).abs().max() / y.abs().max().clamp_min(1e-30))
           for k, x, y in zip(("grad_input", "grad_offset", "grad_logits"), a, b)}
    o_f, o_u = outs["fused"][0].detach(), outs["unfused"][0].detach()
    rel["out"] = float((o_f - o_u).abs().max() / o_u.abs().max())
    del outs, sets
    torch.cuda.empty_cache()
    return {"rotated_sets": n_rot, "fwd_ms": fwd, "bwd_ms": bwd, "fwd_speedup": round(fwd["unfused"] / fwd["fused"], 3),
            "bwd_speedup": round(bwd["unfused"] / bwd["fused"], 3), "fused_vs_unfused_max_rel": rel}


def module(N, H, W, G, C, iters, warmup, amp):
    dev = "cuda:0"
    torch.manual_seed(0)
    m = DCNv3(channels=G * C, group=G).to(dev)
    with torch.no_grad():
        for lin in (m.offset, m.mask):
            lin.weight.normal_(0.0, 0.2)
            lin.bias.normal_(0.0, 1.0)
    set_bytes = N * H * W * G * C * 4 * 2
    n_rot = rotations(set_bytes, 1, 4)
    g = torch.Generator(device=dev).manual_seed(1)
    xs = [torch.randn(N, H, W, G * C, device=dev, generator=g).requires_grad_(True) for _ in range(n_rot)]
    gos = [torch.randn(N, H, W, G * C, device=dev, generator=g) for _ in range(n_rot)]
    params = list(m.parameters())
    fwds = {"fused": m, "composed": lambda x: composed_forward(m, x)}

    def step(k, i):
        with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
            out = fwds[k](xs[i])
        torch.autograd.grad(out, [xs[i]] + params, gos[i].to(out.dtype))

    ms = {k: t for k, (t,) in timed({k: [(partial(step, k, i),) for i in range(n_rot)] for k in fwds}, iters,
                                    warmup).items()}
    peak = {}
    for k in fwds:
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        step(k, 0)
        torch.cuda.synchronize()
        peak[k] = round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)
    del xs, gos
    torch.cuda.empty_cache()
    return {"amp_f16": amp, "fwd_bwd_ms": ms, "speedup": round(ms["composed"] / ms["fused"], 3), "peak_extra_mib": peak}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=25)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--skip-module", action="store_true")
    a = ap.parse_args()
    print(json.dumps(card()), flush=True)
    for (N, H, W, G, C) in SHAPES:
        row = {"shape": [N, H, W, G, C], "K": 9, "core_f32": core(N, H, W, G, C, a.iters, a.warmup)}
        if not a.skip_module:
            row["module_f32"] = module(N, H, W, G, C, a.iters, a.warmup, False)
            row["module_amp_f16"] = module(N, H, W, G, C, a.iters, a.warmup, True)
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Deformable convolution (ir_ads_b200.dcnv2) on the conv2 of R50-DCN's bottleneck blocks at 800x1333 (3x3, pad 1,
C_in = C_out, deformable_groups 1, modulated): res3 128 ch (stride 2 from 200x334, and stride 1 at 100x167), res4 256
ch at 50x84, res5 512 ch at 25x42, B = 2 and 8; float32 and bfloat16 autocast; forward and forward + backward.

Arms, alternated call by call in one process, CUDA-event medians of --iters after --warmup:
  ours         modulated_deform_conv, channels_last input (no layout copy)
  torchvision  torchvision.ops.deform_conv2d on CUDA, NCHW input (the generic kernel this replaces); left out with the
               reason recorded when its CUDA kernel does not load or run on this GPU
  conv2d       torch conv2d of the same shape, channels_last: what a plain 3x3 convolution costs
Inputs rotate over enough copies that each timed call reads a working set larger than the 126 MB L2.  The split of our
time into im2col, col2im and the cuBLAS GEMMs (forward: columns @ W^T; backward: grad_out @ W and grad_out^T @ columns)
times each piece alone, on the same shapes.  Prints the card name and power limit first, then one JSON line per
(shape, batch, dtype)."""
import argparse
import json
import os
import sys
from functools import partial

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ir_ads_b200 import _lib, modulated_deform_conv  # noqa: E402
from ir_ads_b200 import dcnv2 as _dcnv2  # noqa: E402
from timing import card, rotations, timed  # noqa: E402

# (name, C, H_in, W_in, stride)
SHAPES = (("res3_s2", 128, 200, 334, 2), ("res3", 128, 100, 167, 1), ("res4", 256, 50, 84, 1), ("res5", 512, 25, 42, 1))


def torchvision_status():
    """None when torchvision's CUDA deform_conv2d runs here, else why not."""
    try:
        from torchvision.ops import deform_conv2d
        x = torch.randn(1, 16, 8, 8, device="cuda", requires_grad=True)
        y = deform_conv2d(x, torch.zeros(1, 18, 8, 8, device="cuda"), torch.randn(16, 16, 3, 3, device="cuda"),
                          padding=1, mask=torch.ones(1, 9, 8, 8, device="cuda"))
        y.sum().backward()
        torch.cuda.synchronize()
        return None
    except Exception as e:   # noqa: BLE001 -- any failure to load or run the kernel is the finding
        return f"{type(e).__name__}: {str(e).splitlines()[0][:300]}"


def make_sets(B, C, H, W, s, n_rot, dev):
    Ho, Wo = (H - 1) // s + 1, (W - 1) // s + 1
    g = torch.Generator(device=dev).manual_seed(0)
    sets = []
    for _ in range(n_rot):
        x = torch.randn(B, C, H, W, device=dev, generator=g)
        off = torch.randn(B, 18, Ho, Wo, device=dev, generator=g) * 2.0
        m = torch.rand(B, 9, Ho, Wo, device=dev, generator=g)
        go = torch.randn(B, C, Ho, Wo, device=dev, generator=g)
        sets.append((x, off, m, go))
    return sets, Ho, Wo


def bench_shape(name, C, H, W, s, B, amp, tv_ok, iters, warmup):
    dev = "cuda:0"
    set_bytes = B * C * H * W * 4 * 2
    n_rot = rotations(set_bytes, 2, 8)
    sets, Ho, Wo = make_sets(B, C, H, W, s, n_rot, dev)
    torch.manual_seed(0)
    w = (torch.randn(C, C, 3, 3, device=dev) / (9 * C) ** 0.5).requires_grad_(True)
    cl = [(x.contiguous(memory_format=torch.channels_last).requires_grad_(True), off.requires_grad_(True),
           m.requires_grad_(True), go.contiguous(memory_format=torch.channels_last)) for x, off, m, go in sets]
    nchw = [(x.requires_grad_(True), off, m, go) for x, off, m, go in sets]
    dt = torch.bfloat16 if amp else torch.float32

    def ours(i, bwd):
        x, off, m, go = cl[i]
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            y = modulated_deform_conv(x, off, m, w, None, s, 1)
        if bwd:
            torch.autograd.grad(y, (x, off, m, w), go.to(y.dtype))

    def tv(i, bwd):
        from torchvision.ops import deform_conv2d
        x, off, m, go = nchw[i]
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            y = deform_conv2d(x, off, w, None, stride=s, padding=1, mask=m)
        if bwd:
            torch.autograd.grad(y, (x, off, m, w), go.to(y.dtype))

    def conv(i, bwd):
        x, _, _, go = cl[i]
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            y = torch.nn.functional.conv2d(x, w, None, s, 1)
        if bwd:
            torch.autograd.grad(y, (x, w), go.to(y.dtype))

    arms = {"ours": ours, "conv2d": conv}
    if tv_ok:
        arms["torchvision"] = tv
    row = {"shape": name, "B": B, "C": C, "in": [H, W], "out": [Ho, Wo], "stride": s,
           "dtype": "bf16_autocast" if amp else "f32", "rotated_sets": n_rot,
           "gflop_fwd": round(2 * B * Ho * Wo * 9 * C * C / 1e9, 3)}
    for key, bwd in (("fwd_ms", False), ("fwd_bwd_ms", True)):
        with torch.set_grad_enabled(bwd):
            t = timed({k: [(partial(f, i, bwd),) for i in range(n_rot)] for k, f in arms.items()}, iters, warmup)
        row[key] = {k: ms for k, (ms,) in t.items()}
    for key in ("fwd_ms", "fwd_bwd_ms"):
        t = row[key]
        row[key.replace("_ms", "_ours_vs")] = {k: round(t[k] / t["ours"], 3) for k in t if k != "ours"}
    if tv_ok and not amp:   # same inputs, same answer (float32)
        with torch.no_grad():
            x, off, m, _ = nchw[0]
            from torchvision.ops import deform_conv2d
            a = modulated_deform_conv(cl[0][0], off, m, w, None, s, 1)
            b = deform_conv2d(x, off, w, None, stride=s, padding=1, mask=m)
            row["ours_vs_torchvision_max_rel"] = float((a - b).abs().max() / b.abs().max())
    row["split_ms"] = split(cl, w, B, C, H, W, s, dt, iters, warmup, n_rot)
    del sets, cl, nchw
    torch.cuda.empty_cache()
    return row


def split(cl, w, B, C, H, W, s, dt, iters, warmup, n_rot):
    """im2col, col2im and the GEMMs of one call, each timed alone (16-bit offsets / mask under autocast, as a bf16
    offset conv produces them)."""
    xs = [_dcnv2._nhwc(x.detach().to(dt)) for x, _, _, _ in cl]
    aux = dt if dt != torch.float32 else torch.float32
    offs = [_dcnv2._nhwc(off.detach().to(aux)) for _, off, _, _ in cl]
    ms = [_dcnv2._nhwc(m.detach().to(aux)) for _, _, m, _ in cl]
    wt = w.detach().to(dt)
    g = _dcnv2._Geom(cl[0][0], wt, s, s, 1, 1, 1, 1, 1, 1, B)
    tag = {torch.float32: _lib.MSDA_F32, torch.bfloat16: _lib.MSDA_BF16_AUX16}[dt]
    dev = xs[0].device
    cols = torch.empty((B * g.P, 9 * C), dtype=dt, device=dev)
    gcols = torch.randn((B * g.P, 9 * C), device=dev).to(dt)
    go = torch.randn((B * g.P, C), device=dev).to(dt)
    wm = _dcnv2._wmat(wt, 1)[0]
    gx = torch.empty_like(xs[0])
    goff, gm = torch.empty_like(offs[0]), torch.empty_like(ms[0])
    ws = torch.empty(max(1, _lib.lib().msda_dcnv2_col2im_workspace_bytes(*g.abi(B), tag, 0)), dtype=torch.uint8,
                     device=dev)
    h = _lib.lib()

    def im2col(i):
        _dcnv2._im2col(xs[i], offs[i], ms[i], cols, g, tag)

    def col2im(i):
        _lib.check(h.msda_dcnv2_col2im(_dcnv2._stream(xs[i]), _dcnv2._ptr(gcols), _dcnv2._ptr(xs[i]),
                                       _dcnv2._ptr(offs[i]), _dcnv2._ptr(ms[i]), *g.abi(B), _dcnv2._ptr(gx),
                                       _dcnv2._ptr(goff), _dcnv2._ptr(gm), _dcnv2._ptr(ws), ws.numel(), tag, 0), "col2im")

    fns = {"im2col": im2col, "col2im": col2im,
           "gemm_fwd": lambda i: torch.mm(cols, wm.t()),
           "gemm_bwd": lambda i: (torch.mm(go, wm), torch.mm(go.t(), cols))}
    t = timed({k: [(partial(f, i),) for i in range(n_rot)] for k, f in fns.items()}, iters, warmup)
    return {k: ms for k, (ms,) in t.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batches", default="2,8")
    a = ap.parse_args()
    info = card()
    reason = torchvision_status()
    info["torchvision_cuda_deform_conv2d"] = "runs" if reason is None else f"left out: {reason}"
    print(json.dumps(info), flush=True)
    for B in [int(b) for b in a.batches.split(",")]:
        for (name, C, H, W, s) in SHAPES:
            for amp in (False, True):
                print(json.dumps(bench_shape(name, C, H, W, s, B, amp, reason is None, a.iters, a.warmup)), flush=True)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Autocast-native module paths against the routes they replace, under float16 and bfloat16 autocast.

  native  the modules as they are: the 16-bit offset / logit Linear outputs go into the fused kernels as produced
          (MSDA_*_AUX16), and a 16-bit addend plus a float32 residual take the mixed add + LayerNorm kernel
  widened the previous route, reconstructed in the same process: both Linear outputs widened with .float() in front
          of the fused Function (autograd then rounds their gradients back with a cast), and add + LayerNorm falling
          back to norm(a + b) whenever the addends' dtypes differ

Workloads: the MSDeformAttn module at cfg2 (DINO-R50 encoder, B=8), the DCNv3 module at the five InternImage-T-like
stages of tools/bench_dcnv3_fused.py, and DeformableEncoderLayer at cfg2 B=8.  One process; per workload both routes are
warmed up, then forward + backward is timed alternately with CUDA events, median of --iters.  Inputs rotate over enough
copies that every timed call reads more than the 126 MB L2.  Per route also: the peak memory allocated above the
resting set during one forward + backward, and the CUDA kernels one forward + backward launches (torch.profiler, in a
pass of its own).  Prints the card name and power limit first, then one JSON line per workload."""
import argparse
import contextlib
import json
import os
import sys
from functools import partial

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ir_ads_b200.dcnv3 as dcnv3_mod  # noqa: E402
import ir_ads_b200.encoder as encoder_mod  # noqa: E402
import ir_ads_b200.module as module_mod  # noqa: E402
from bench_dcnv3_fused import SHAPES as DCN_SHAPES  # noqa: E402
from ir_ads_b200 import MultiScaleDeformableAttention  # noqa: E402
from ir_ads_b200.encoder import DeformableEncoderLayer  # noqa: E402
from ir_ads_b200.epilogue import AddLayerNormFunction  # noqa: E402
from ir_ads_b200.workloads import LEVELS, _pixel_centres, level_tensors  # noqa: E402
from timing import card, rotations, timed  # noqa: E402

DEV = "cuda:0"


class _Widened:
    """a fused Function whose offsets / logits arrive widened to float32, as the modules passed them before"""

    def __init__(self, fn, aux):
        self.fn, self.aux = fn, aux

    def apply(self, *args):
        args = list(args)
        for i in self.aux:
            args[i] = args[i].float()
        return self.fn.apply(*args)


def _same_dtype_add_layer_norm(a, b, norm):
    if a.dtype == b.dtype and a.shape == b.shape and norm.bias is not None and a.shape[-1] % 4 == 0:
        return AddLayerNormFunction.apply(a, b, norm.weight, norm.bias, norm.eps)
    return norm(a + b)


@contextlib.contextmanager
def widened_route():
    saved = (module_mod.MSDeformAttnFusedFunction, dcnv3_mod.DCNv3FusedFunction, encoder_mod.add_layer_norm)
    module_mod.MSDeformAttnFusedFunction = _Widened(saved[0], (3, 4))
    dcnv3_mod.DCNv3FusedFunction = _Widened(saved[1], (1, 2))
    encoder_mod.add_layer_norm = _same_dtype_add_layer_norm
    try:
        yield
    finally:
        module_mod.MSDeformAttnFusedFunction, dcnv3_mod.DCNv3FusedFunction, encoder_mod.add_layer_norm = saved


def measure(fwd, xs, gos, params, dtype, iters, warmup):
    """median ms of forward + backward per route (alternated), peak extra MiB, kernels launched per call"""
    routes = {"native": contextlib.nullcontext, "widened": widened_route}

    def step(route, i):
        with routes[route]():
            with torch.autocast("cuda", dtype=dtype):
                out = fwd(xs[i])
            torch.autograd.grad(out, [xs[i]] + params, gos[i].to(out.dtype))

    t = timed({r: [(partial(step, r, i),) for i in range(len(xs))] for r in routes}, iters, warmup)
    ms = {r: v for r, (v,) in t.items()}
    peak, kernels = {}, {}
    for r in routes:
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        step(r, 0)
        torch.cuda.synchronize()
        peak[r] = round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            step(r, 0)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                 and not e.name.startswith("Memset") and not e.name.startswith("Memcpy")]
        kernels[r] = {"total": len(names),
                      "casts": sum(1 for s in names if "copy" in s.lower() or "cast" in s.lower()),
                      "library": sum(1 for s in names if "msda" in s or "layernorm" in s.lower() and "add_" in s)}
    return {"fwd_bwd_ms": ms, "speedup": round(ms["widened"] / ms["native"], 3), "peak_extra_mib": peak,
            "kernels_per_call": kernels}


def msda_module(dtype, iters, warmup):
    torch.manual_seed(0)
    levels = [tuple(l) for l in LEVELS["dino_r50"]]
    shapes, lsi = level_tensors(levels, DEV)
    S, B = sum(h * w for h, w in levels), 8
    m = MultiScaleDeformableAttention(dropout=0.0, batch_first=True).to(DEV)
    with torch.no_grad():
        m.sampling_offsets.weight.normal_(0, 0.05)
        m.attention_weights.weight.normal_(0, 0.2)
    ref = _pixel_centres(levels, DEV)[None, :, None, :].expand(B, S, 4, 2).contiguous()
    n = rotations(B * S * 256 * 4 * 2, 1, 3)
    xs = [torch.randn(B, S, 256, device=DEV).requires_grad_(True) for _ in range(n)]
    gos = [torch.randn(B, S, 256, device=DEV) for _ in range(n)]
    fwd = lambda x: m(x, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi, level_shapes=levels)
    return measure(fwd, xs, gos, list(m.parameters()), dtype, iters, warmup)


def encoder_layer(dtype, iters, warmup):
    torch.manual_seed(0)
    levels = [tuple(l) for l in LEVELS["dino_r50"]]
    shapes, lsi = level_tensors(levels, DEV)
    S, B = sum(h * w for h, w in levels), 8
    layer = DeformableEncoderLayer(attn_dropout=0.0, ffn_dropout=0.0).to(DEV)
    with torch.no_grad():
        layer.attentions[0].sampling_offsets.weight.normal_(0, 0.05)
        layer.attentions[0].attention_weights.weight.normal_(0, 0.2)
    ref = _pixel_centres(levels, DEV)[None, :, None, :].expand(B, S, 4, 2).contiguous()
    pos = torch.randn(B, S, 256, device=DEV) * 0.1
    n = rotations(B * S * 256 * 4 * 2, 1, 3)
    xs = [torch.randn(B, S, 256, device=DEV).requires_grad_(True) for _ in range(n)]
    gos = [torch.randn(B, S, 256, device=DEV) for _ in range(n)]
    fwd = lambda x: layer(x, query_pos=pos, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi,
                          level_shapes=levels)
    return measure(fwd, xs, gos, list(layer.parameters()), dtype, iters, warmup)


def dcn_module(shape, dtype, iters, warmup):
    N, H, W, G, C = shape
    torch.manual_seed(0)
    m = dcnv3_mod.DCNv3(channels=G * C, group=G).to(DEV)
    with torch.no_grad():
        for lin in (m.offset, m.mask):
            lin.weight.normal_(0.0, 0.2)
            lin.bias.normal_(0.0, 1.0)
    n = rotations(N * H * W * G * C * 4 * 2, 1, 4)
    xs = [torch.randn(N, H, W, G * C, device=DEV).requires_grad_(True) for _ in range(n)]
    gos = [torch.randn(N, H, W, G * C, device=DEV) for _ in range(n)]
    return measure(m, xs, gos, list(m.parameters()), dtype, iters, warmup)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    a = ap.parse_args()
    print(json.dumps(card()), flush=True)
    for name in ("f16", "bf16"):
        dtype = torch.float16 if name == "f16" else torch.bfloat16
        print(json.dumps({"workload": "msda_module_cfg2_B8", "autocast": name,
                          **msda_module(dtype, a.iters, a.warmup)}), flush=True)
        print(json.dumps({"workload": "encoder_layer_cfg2_B8", "autocast": name,
                          **encoder_layer(dtype, a.iters, a.warmup)}), flush=True)
        for shape in DCN_SHAPES:
            print(json.dumps({"workload": "dcnv3_module", "shape": list(shape), "autocast": name,
                              **dcn_module(shape, dtype, a.iters, a.warmup)}), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

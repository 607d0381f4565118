#!/usr/bin/env python
"""float16 value timing on one GPU, in one process (tools/sweep.py's method: CUDA events, three rotating input sets
larger than L2, median over iterations; the variants of a row are alternated iteration by iteration):
  op      the plain operator through the C ABI with float32 / bfloat16 / float16 value at the cfg2 and cfg3 shapes and
          cfg5 with the deterministic backward (preallocated outputs and workspace: kernel time only);
  module  MultiScaleDeformableAttention forward+backward at the encoder shape under float16 autocast: the module as it
          is (float16 value to the fused kernels) against the widening route it replaced (value.float() in front of
          the fused Function, output.half() behind it);
  dcnv3   tools/bench_dcnv3.py's stages, float16 against float32 input.
The first line names the card and its power limit.
Usage: python tools/bench_fp16.py [--iters 10] [--out profiles/x.jsonl]"""
import argparse
import copy
import ctypes
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ir_ads_b200 import MultiScaleDeformableAttention, _lib, dcnv3_backward, dcnv3_forward  # noqa: E402
from ir_ads_b200.functional import _VALUE_TAG, MSDeformAttnFusedFunction  # noqa: E402
from ir_ads_b200.workloads import LEVELS, WORKLOADS, level_tensors, make_workload_inputs  # noqa: E402
from timing import card, timed  # noqa: E402

DEV = "cuda:0"
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


class PlainOp:
    """One input set in one value dtype with its preallocated outputs; fwd() / bwd() enqueue one C-ABI call each."""

    def __init__(self, base, dtype, flags):
        value, shapes, lsi, loc, w, go = base
        self.v, self.go = value.to(dtype), go.to(dtype)
        self.shapes, self.lsi, self.loc, self.w, self.flags = shapes, lsi, loc, w, flags
        self.tag = _VALUE_TAG[dtype]
        self.dims = (*value.shape[:3], value.shape[3], loc.shape[3], loc.shape[1], loc.shape[4])   # B S H D L Q P
        B, S, H, D, L, Q, P = self.dims
        self.out = torch.empty(B, Q, H * D, dtype=dtype, device=DEV)
        self.gv, self.gl, self.gw = torch.empty_like(self.v), torch.empty_like(loc), torch.empty_like(w)
        self.ws_bytes = int(_lib.lib().msda_backward_workspace_bytes(B, S, H, D, L, Q, P, self.tag, flags))
        self.ws = torch.empty(max(self.ws_bytes, 16), dtype=torch.uint8, device=DEV)

    def fwd(self):
        B, S, H, D, L, Q, P = self.dims
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(_lib.lib().msda_forward(st, _p(self.v), _p(self.shapes), _p(self.lsi), _p(self.loc), _p(self.w), B,
                                           S, H, D, L, Q, P, _p(self.out), self.tag, 0), "msda_forward")

    def bwd(self):
        B, S, H, D, L, Q, P = self.dims
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(_lib.lib().msda_backward(st, _p(self.go), _p(self.v), _p(self.shapes), _p(self.lsi), _p(self.loc),
                                            _p(self.w), B, S, H, D, L, Q, P, _p(self.gv), _p(self.gl), _p(self.gw),
                                            _p(self.ws), self.ws_bytes, self.tag, self.flags), "msda_backward")


def bench_op(iters):
    rows = []
    for cfg, det in (("cfg2", False), ("cfg3_f32", False), ("cfg5", True)):
        wl = WORKLOADS[cfg]
        flags = _lib.FLAG_DETERMINISTIC if det else 0
        sets = []
        for seed in range(3):
            value, shapes, lsi, loc, w = make_workload_inputs(wl, "model", seed, DEV)
            go = torch.randn(wl.batch, wl.queries, wl.num_heads * wl.head_dim, device=DEV)
            sets.append((value, shapes, lsi, loc, w, go))
        ops = {dt: [PlainOp(s, DTYPES[dt], flags) for s in sets] for dt in DTYPES}
        res = timed({dt: [(o.fwd, o.bwd) for o in ops[dt]] for dt in DTYPES}, iters, 3)
        for dt, (f, b) in res.items():
            rows.append({"section": "op", "workload": cfg.replace("_f32", ""), "det": det, "value": dt,
                         "fwd_ms": f, "bwd_ms": b})
        del ops, sets
        torch.cuda.empty_cache()
    return rows


def bench_module(iters, batch=8):
    """Encoder shape (DINO-R50 levels, Q = S), float16 autocast, forward + backward with the projections."""
    shapes, lsi = level_tensors(LEVELS["dino_r50"], DEV)
    S = sum(h * w for h, w in LEVELS["dino_r50"])
    torch.manual_seed(0)
    m = MultiScaleDeformableAttention(dropout=0.0, batch_first=True).to(DEV)
    m_old = copy.deepcopy(m)
    H, L, P = m.num_heads, m.num_levels, m.num_points
    qs = [torch.randn(batch, S, 256, device=DEV, requires_grad=True) for _ in range(3)]
    refs = [torch.rand(batch, S, L, 2, device=DEV) for _ in range(3)]

    def new(i):
        with torch.autocast("cuda", dtype=torch.float16):
            return m(qs[i], reference_points=refs[i], spatial_shapes=shapes, level_start_index=lsi)

    def old(i):
        q = qs[i]
        with torch.autocast("cuda", dtype=torch.float16):
            value = m_old.value_proj(q).view(batch, S, H, -1).float()
            off = m_old.sampling_offsets(q).view(batch, S, H, L, P, 2)
            logits = m_old.attention_weights(q).view(batch, S, H, L * P)
            out = MSDeformAttnFusedFunction.apply(value.contiguous(), shapes, lsi, off.float().contiguous(),
                                                  logits.float().contiguous(), refs[i].contiguous(), None)
            return m_old.output_proj(out.half()) + q

    def step(route, i):
        box = {}

        def fwd():
            box["out"] = route(i)

        def bwd():
            box["out"].float().sum().backward()
        return fwd, bwd

    res = timed({"fp16_native": [step(new, i) for i in range(3)], "fp16_widened": [step(old, i) for i in range(3)]},
                iters, 3)
    return [{"section": "module", "shape": "encoder", "batch": batch, "route": k, "fwd_ms": f, "bwd_ms": b}
            for k, (f, b) in res.items()]


def bench_dcnv3(iters):
    rows = []
    for (N, H, W, G, C) in ((16, 200, 336, 4, 16), (16, 100, 168, 8, 16), (16, 50, 84, 16, 16), (16, 25, 42, 32, 16),
                            (8, 100, 168, 8, 32)):
        args = (3, 3, 1, 1, 1, 1, 1, 1, G, C, 1.0)
        sets = []
        for _ in range(3):
            inp = torch.randn(N, H, W, G * C, device=DEV)
            off = torch.randn(N, H, W, G * 18, device=DEV)
            mask = torch.softmax(torch.randn(N, H, W, G, 9, device=DEV), -1).reshape(N, H, W, G * 9)
            go = torch.randn(N, H, W, G * C, device=DEV)
            sets.append((inp, off, mask, go))

        def stages(s, dt):
            inp, off, mask, go = s[0].to(dt), s[1], s[2], s[3].to(dt)
            return (lambda: dcnv3_forward(inp, off, mask, *args), lambda: dcnv3_backward(inp, off, mask, *args, go))

        res = timed({dt: [stages(s, DTYPES[dt]) for s in sets] for dt in ("f32", "f16")}, iters, 3)
        for dt, (f, b) in res.items():
            rows.append({"section": "dcnv3", "shape": [N, H, W, G, C], "input": dt, "fwd_ms": f, "bwd_ms": b})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--sections", default="op,module,dcnv3")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    rows = [card()]
    print(json.dumps(rows[0]), flush=True)
    for sec in a.sections.split(","):
        for r in {"op": bench_op, "module": bench_module, "dcnv3": bench_dcnv3}[sec](a.iters):
            rows.append(r)
            print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in rows) + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Kernel-variant sweep on one GPU: times the core op's forward and backward per launch
(CUDA events, 3 rotating input sets > L2, median of N) for a list of (workload, dist, flags).
Usage: python tools/sweep.py [--workloads cfg2,cfg3] [--flags 0,4,65536] [--iters 10]"""
import argparse
import json
import os
import sys
from functools import partial

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ir_ads_b200  # noqa: E402
from ir_ads_b200 import functional  # noqa: E402
from ir_ads_b200.workloads import WORKLOADS, make_workload_inputs  # noqa: E402
from timing import card, timed  # noqa: E402


def hbm_peak_gbs():
    """The roofline denominator bench.py uses: MEASURED_PEAKS.json hbm_gbs, else B200_PROFILING.md's fallback."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"])
    except Exception:
        return 6650.0


def time_variant(wl, dist, flags, iters, sets=3, dev="cuda:0", deterministic=False):
    data = []
    odt = torch.bfloat16 if wl.value_dtype == "bf16" else torch.float32
    for i in range(sets):
        value, shapes, lsi, loc, w = make_workload_inputs(wl, dist, seed=i, device=dev)
        go = torch.randn(wl.batch, wl.queries, wl.num_heads * wl.head_dim, device=dev).to(odt)
        data.append((value, shapes, lsi, loc, w, go))
    functional.set_deterministic(deterministic)
    with functional.kernel_flags(flags):
        f, b = timed({"op": [(partial(ir_ads_b200.ms_deform_attn_forward, value, shapes, lsi, loc, w, 64),
                              partial(ir_ads_b200.ms_deform_attn_backward, value, shapes, lsi, loc, w, go, 64))
                             for value, shapes, lsi, loc, w, go in data]}, iters, 3)["op"]
    functional.set_deterministic(False)
    fb, bb = wl.algorithmic_bytes()
    peak = hbm_peak_gbs()
    return {"workload": wl.name, "dist": dist, "flags": flags, "det": deterministic, "fwd_ms": f, "bwd_ms": b,
            "gpts_s": round(wl.points / (f + b) / 1e6, 3),
            "fwd_frac_hbm": round(fb / f / 1e6 / peak, 4), "bwd_frac_hbm": round(bb / b / 1e6 / peak, 4),
            "fb_frac_hbm": round((fb + bb) / (f + b) / 1e6 / peak, 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="cfg2")
    ap.add_argument("--dists", default="model")
    ap.add_argument("--flags", default="0")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--det", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    rows = [card()]
    print(json.dumps(rows[0]), flush=True)
    for name in a.workloads.split(","):
        for dist in a.dists.split(","):
            for fl in a.flags.split(","):
                r = time_variant(WORKLOADS[name], dist, int(fl), a.iters, deterministic=a.det)
                rows.append(r)
                print(json.dumps(r), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()

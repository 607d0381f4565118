#!/usr/bin/env python
"""DCNv3 core op timing next to the reference's own kernels on the same GPU (InternImage-T-like stages)."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ir_ads_b200 import dcnv3_backward, dcnv3_forward  # noqa: E402
from oracle import ref_cuda  # noqa: E402
from timing import card, timed  # noqa: E402


def main():
    argparse.ArgumentParser(description=__doc__).parse_args()
    print(json.dumps(card()), flush=True)
    dev = "cuda:0"
    for (N, H, W, G, C) in ((16, 200, 336, 4, 16), (16, 100, 168, 8, 16), (16, 50, 84, 16, 16), (16, 25, 42, 32, 16),
                            (8, 100, 168, 8, 32)):
        k, s, p, d, scale = 3, 1, 1, 1, 1.0
        inp = torch.randn(N, H, W, G * C, device=dev)
        off = torch.randn(N, H, W, G * 18, device=dev)
        mask = torch.softmax(torch.randn(N, H, W, G, 9, device=dev), -1).reshape(N, H, W, G * 9)
        go = torch.randn(N, H, W, G * C, device=dev)
        args = (k, k, s, s, p, p, d, d, G, C, scale)
        arms = {"b200": [(lambda: dcnv3_forward(inp, off, mask, *args),
                          lambda: dcnv3_backward(inp, off, mask, *args, go))]}
        if ref_cuda.dcn_available():
            arms["reference"] = [(lambda: ref_cuda.dcnv3_forward_backward(inp, off, mask, go, *args, backward=False),
                                  lambda: ref_cuda.dcnv3_forward_backward(inp, off, mask, go, *args))]
        res = timed(arms, 5, 3)
        row = {"shape": [N, H, W, G, C], "points": N * H * W * G * 9,
               "b200_fwd_ms": res["b200"][0], "b200_bwd_ms": res["b200"][1]}
        if "reference" in res:
            # the reference backward timing above includes a second forward; subtract it
            row["ref_fwd_ms"] = res["reference"][0]
            row["ref_bwd_ms"] = round(res["reference"][1] - res["reference"][0], 4)
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()

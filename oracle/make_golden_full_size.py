"""Writes tests/golden/full_size_golden.npz: what tests/test_parity_gpu.py's BASELINE-shape comparisons check against.

The reference kernels (ms_deform_im2col_cuda.cuh) are a restatement away here: oracle/msda_oracle.c follows them
line by line -- in float64 the reference expressions, in float32 the reference kernel's own rounding (coordinate
h_im = loc*H - 0.5 as cuh:284-285 rounds it, every product and sum rounded to float).  For every case below, on
inputs made on the CPU from fixed seeds (make_case_inputs), this stores
  <case>/check                  float64 sums of value and sampling_loc (the inputs the data belongs to)
  <case>/<tensor>/sample        the float64 result at SAMPLE flat indices drawn by sample_index()
  <case>/<tensor>/absmax        max |float64 result| over the whole tensor
and for float32 cases what the float32 restatement of the reference arithmetic costs against it, whole tensor:
  <case>/<tensor>/err32         max |float32 - float64|
  <case>/<tensor>/viol32        elements with |float32 - float64| > ATOL + RTOL * |float64|
grad_sampling_loc is taken times smooth_mask(band 1e-4) throughout (it is discontinuous at cell boundaries).

(The restatement rounds every product and sum separately, in sequence; the reference kernels as compiled contract to
FMAs and accumulate in other orders, and their measured float32 cost is larger -- tests/golden/
full_size_reference_fp32.json -- so the restatement's is the stricter bar.)

  python oracle/make_golden_full_size.py        # ~1 minute on 8 cores
"""
from __future__ import annotations

import os
import sys
from multiprocessing import Pool

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

OUT = os.path.join(ROOT, "tests", "golden", "full_size_golden.npz")
TENSORS = ("out", "grad_value", "grad_sampling_loc", "grad_attn_weight")
SAMPLE = 256
RTOL, ATOL, BAND = 1e-5, 1e-6, 1e-4
# (workload, dist, batch): the cases of tests/test_parity_gpu.py::test_against_reference_at_baseline_shapes
CASES = [("cfg1", "model", 2), ("cfg1", "edge", 2), ("cfg2", "model", 2), ("cfg2", "test", 1), ("cfg3_f32", "model", 8),
         ("cfg4", "model", 2), ("cfg5", "model", 1)]


def case_key(cfg, dist, batch):
    return f"{cfg}/{dist}/B{batch}"


def make_case_inputs(cfg, dist, batch):
    """(value, shapes, lsi, loc, w, grad_out) on the CPU; grad_out in value's dtype."""
    from ir_ads_b200.workloads import WORKLOADS, make_workload_inputs
    wl = WORKLOADS[cfg]
    value, shapes, lsi, loc, w = make_workload_inputs(wl, dist, 5, "cpu", batch=batch)
    go = torch.randn(batch, wl.queries, wl.num_heads * wl.head_dim, generator=torch.Generator().manual_seed(6))
    return value, shapes, lsi, loc, w, go.to(value.dtype)


def sample_index(numel):
    return torch.randint(numel, (SAMPLE,), generator=torch.Generator().manual_seed(numel)).sort()[0]


def load(cfg, dist, batch):
    """The stored data of one case: {"check", "<tensor>/sample", "<tensor>/absmax", ...}."""
    blob = np.load(OUT)
    key = case_key(cfg, dist, batch) + "/"
    return {k[len(key):]: blob[k] for k in blob.files if k.startswith(key)}


def check_inputs(stored, value, loc):
    """The inputs are the ones the stored data was made from (same seeds, same generator)."""
    got = np.array([value.double().sum().item(), loc.double().sum().item()])
    assert np.allclose(got, stored["check"], rtol=1e-9, atol=1e-6), (got, stored["check"])


def sampled(t):
    """float64 numpy values of tensor `t` at the stored sample's flat indices."""
    idx = sample_index(t.numel())
    return t.reshape(-1)[idx.to(t.device)].double().cpu().numpy()


def smooth_mask(loc, shapes, band=BAND):
    wh = np.array([[w, h] for h, w in shapes], dtype=np.float64)[None, None, None, :, None, :]
    px = loc.astype(np.float64) * wh - 0.5
    return (np.abs(px - np.round(px)) > band).all(-1, keepdims=True)


def _image(task):
    """One image of one case: per-tensor float64 samples falling in it, absmax, and the float32 statistics."""
    (cfg, dist, batch), b = task
    from oracle import msda_c
    value, shapes, lsi, loc, w, go = make_case_inputs(cfg, dist, batch)
    f32 = value.dtype == torch.float32
    a = [value[b:b + 1].float().numpy(), shapes.numpy(), lsi.numpy(), loc[b:b + 1].numpy(), w[b:b + 1].numpy()]
    g = go[b:b + 1].float().numpy()
    m = smooth_mask(a[3], a[1])
    truth = [msda_c.forward(*a, np.float64)] + list(msda_c.backward(g, *a, np.float64))
    ref32 = None
    if f32:
        ref32 = [msda_c.forward(*a, np.float32, coord_mode=msda_c.COORD_REFERENCE)] + \
                list(msda_c.backward(g, *a, np.float32, coord_mode=msda_c.COORD_REFERENCE))
    res = {}
    for k, name in enumerate(TENSORS):
        mk = m if name == "grad_sampling_loc" else 1.0
        t = (truth[k] * mk).reshape(-1)
        per = t.size
        idx = sample_index(per * batch).numpy()
        mine = idx[(idx >= b * per) & (idx < (b + 1) * per)] - b * per
        res[name] = {"sample": t[mine], "absmax": float(np.abs(t).max())}
        if ref32 is not None:
            d = np.abs((ref32[k].astype(np.float64) * mk).reshape(-1) - t)
            res[name]["err32"] = float(d.max())
            res[name]["viol32"] = int((d > ATOL + RTOL * np.abs(t)).sum())
    return (cfg, dist, batch), b, res


def main():
    tasks = [(c, b) for c in CASES for b in range(c[2])]
    tasks.sort(key=lambda t: -t[0][2])                   # the large cases first
    with Pool(os.cpu_count()) as pool:
        done = pool.map(_image, tasks, chunksize=1)
    blob = {}
    for c in CASES:
        key = case_key(*c)
        value, _, _, loc, _, _ = make_case_inputs(*c)
        blob[f"{key}/check"] = np.array([value.double().sum().item(), loc.double().sum().item()])
        parts = sorted(((b, r) for cc, b, r in done if cc == c), key=lambda p: p[0])
        for name in TENSORS:
            blob[f"{key}/{name}/sample"] = np.concatenate([r[name]["sample"] for _, r in parts])
            blob[f"{key}/{name}/absmax"] = np.array(max(r[name]["absmax"] for _, r in parts))
            if "err32" in parts[0][1][name]:
                blob[f"{key}/{name}/err32"] = np.array(max(r[name]["err32"] for _, r in parts))
                blob[f"{key}/{name}/viol32"] = np.array(sum(r[name]["viol32"] for _, r in parts))
    np.savez_compressed(OUT, **blob)
    print(f"wrote {OUT} ({os.path.getsize(OUT)} bytes, {len(blob)} arrays)")


if __name__ == "__main__":
    main()

"""Full-size parity at the sizes BASELINE.json quotes -- every tensor, forward AND backward.

The CPU oracle cannot reach these sizes within a test, so the yardstick is the reference's own formulation,
multi_scale_deformable_attn_pytorch (restated in oracle/msda_torch.py and pinned to reference-made vectors by
test_oracle.py), run on the same GPU in FLOAT64 on the same inputs: an fp32 tensor widens to fp64 exactly, and so does
a bf16 one, so "the reference on identical inputs" is well defined for both.  What the reference's own CUDA kernels in
float32 cost against their float64 result on these very inputs (seeded, generated on cuda:0) was measured on a B200
and is stored in tests/golden/full_size_reference_fp32.json.

Two criteria are evaluated for every tensor and PRINTED (pytest -s / the captured log shows them):
  * max-norm:    max|got - ref| <= rtol * max|ref| + atol          (asserted; the tolerance of the north_star:
                 fp32 1e-5 / 1e-6, bf16 value 1e-2)
  * per-element: |got - ref| <= atol + rtol * |ref| element by element, the literal reading of torch.allclose that
                 the reference's own test uses (tests/test_ms_deform_attn.py:127): the number of violating elements
                 is reported for this repo AND for the reference's float32 kernels (stored), and this repo must not
                 have more violations than those did (+ a small slack), since a sum of 64 float32 products that
                 cancels to ~0 has no per-element relative accuracy in ANY float32 implementation.
"""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
REFERENCE_FP32 = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "full_size_reference_fp32.json")


def _mods():
    import ir_ads_b200
    from ir_ads_b200 import _lib, functional, workloads
    from oracle import msda_torch
    return ir_ads_b200, _lib, functional, workloads, msda_torch


def smooth_mask_t(loc, shapes, band):
    """torch twin of test_oracle.smooth_mask: [B,Q,H,L,P,1] bool, True where no pixel coordinate is within `band` of
    an integer (grad_sampling_loc is discontinuous there)."""
    wh = torch.stack([shapes[:, 1], shapes[:, 0]], -1).double()[None, None, None, :, None, :]
    px = loc.double() * wh - 0.5
    return ((px - px.round()).abs() > band).all(-1, keepdim=True)


def report(name, got, ref, rtol, atol, mask=None, worst32=float("nan"), viol32=-1):
    """Returns (max-norm ok, violations of got, n) and prints one line; worst32 / viol32: the reference's float32
    kernels on the same inputs, stored."""
    got, ref = got.double(), ref.double()
    if mask is not None:
        got, ref = got * mask, ref * mask
    diff = (got - ref).abs()
    bound = rtol * ref.abs().max().item() + atol
    worst = diff.max().item()
    viol = int((diff > atol + rtol * ref.abs()).sum().item())
    print(f"[full-size parity] {name:38s} max|err| {worst:.3e} (bound {bound:.3e}; reference fp32 kernels {worst32:.3e})  "
          f"per-element allclose(rtol={rtol:g}, atol={atol:g}) violations: {viol} of {diff.numel()} "
          f"(reference fp32 kernels: {viol32})")
    return worst <= bound, viol, diff.numel()


def run_ours(value, shapes, lsi, loc, w, go, flags=0):
    ir, _lib, functional, *_ = _mods()
    v = value.detach().clone().requires_grad_(True)
    lo = loc.detach().clone().requires_grad_(True)
    ww = w.detach().clone().requires_grad_(True)
    with functional.kernel_flags(flags):
        out = ir.MultiScaleDeformableAttnFunction.apply(v, shapes, lsi, lo, ww, 64)
        out.backward(go)
    torch.cuda.synchronize()
    return out.detach(), v.grad, lo.grad, ww.grad


def run_reference_f64(value, shapes, loc, w, go):
    """The reference formulation in float64 on the inputs' device, one image at a time (images are independent)
    to bound the memory its stacked per-level samples take."""
    msda_torch = _mods()[4]
    parts = [msda_torch.forward_backward_f64(value[b:b + 1], shapes, loc[b:b + 1], w[b:b + 1], go[b:b + 1])
             for b in range(value.shape[0])]
    return [torch.cat(t) for t in zip(*parts)]


CASES = [
    # name, workload, batch, dist, flags name
    ("cfg2_B8_default", "cfg2", 8, "model", "default"),
    ("cfg2_B8_fold", "cfg2", 8, "model", "fold"),
    ("cfg2_B8_nofold", "cfg2", 8, "model", "nofold"),
    ("cfg2_B8_test_dist", "cfg2", 8, "test", "default"),
    ("cfg3_bf16_B8", "cfg3", 8, "model", "default"),
    ("cfg3_bf16_B8_edge", "cfg3", 8, "edge", "default"),
    ("cfg2_bf16_B8", "cfg2_bf16", 8, "model", "default"),
    ("cfg3_f32_B8", "cfg3_f32", 8, "model", "default"),
    ("cfg4_B2", "cfg4", 2, "model", "default"),
    ("cfg5_det_B8", "cfg5", 8, "model", "deterministic"),
    ("cfg5_B8_fold", "cfg5", 8, "model", "fold"),
]


@pytest.mark.parametrize("name,cfg,batch,dist,mode", CASES, ids=[c[0] for c in CASES])
def test_full_size_all_tensors(name, cfg, batch, dist, mode):
    ir, _lib, functional, workloads, _ = _mods()
    if mode == "fold" and not _lib.has_experiments():
        pytest.skip("product library: the folding backward is compiled into experiment builds only")
    wl = workloads.WORKLOADS[cfg]
    value, shapes, lsi, loc, w = workloads.make_workload_inputs(wl, dist, 5, DEV, batch=batch)
    bf16 = value.dtype == torch.bfloat16
    go = torch.randn(batch, wl.queries, wl.num_heads * wl.head_dim, device=DEV,
                     generator=torch.Generator(device=DEV).manual_seed(6)).to(value.dtype)
    with open(REFERENCE_FP32) as f:
        ref32 = json.load(f)["cases"][name]
    flags = {"default": 0, "fold": _lib.FLAG_FOLD_ON, "nofold": _lib.FLAG_FOLD_OFF,
             "deterministic": _lib.FLAG_DETERMINISTIC}[mode]
    got = run_ours(value, shapes, lsi, loc, w, go, flags)
    if mode == "deterministic":
        again = run_ours(value, shapes, lsi, loc, w, go, flags)
        assert all(torch.equal(a, b) for a, b in zip(got, again)), "deterministic backward is not bit-reproducible"
        del again
    # the reference formulation in float64 on the same (exactly widened) inputs
    truth = run_reference_f64(value, shapes, loc, w, go)
    m = smooth_mask_t(loc, shapes, 1e-4).double()
    masked_pts = int((1 - m).sum().item())
    print(f"[full-size parity] {name}: B={batch} Q={wl.queries} points={wl.points // wl.batch * batch} "
          f"grad_loc points within 1e-4 px of a cell boundary (left out): {masked_pts}")
    rt = 1e-2 if bf16 else 1e-5
    # fp32 outputs of the bf16 problem (grad_loc, grad_w) see only fp32-accumulate error
    rt_aux = 1e-4 if bf16 else 1e-5
    ok = True
    slack = 1e-6
    for (tn, g, t, rtol, msk) in (("out", got[0], truth[0], rt, None),
                                  ("grad_value", got[1], truth[1], rt, None),
                                  ("grad_sampling_loc", got[2], truth[2], rt_aux, m),
                                  ("grad_attn_weight", got[3], truth[3], rt_aux, None)):
        viol32 = ref32[tn]["viol32"]
        good, viol, n = report(f"{name}/{tn}", g, t, rtol, 1e-6, msk, ref32[tn]["err32"], viol32)
        ok = ok and good
        assert n == ref32[tn]["n"], (tn, n)
        if not bf16:
            # never worse than the reference's own float32 kernels element by element (slack: 1e-6 of the elements)
            assert viol <= viol32 + slack * n + 16, (tn, viol, viol32)
    assert ok, "max-norm tolerance exceeded (see the printed lines)"


@pytest.mark.parametrize("cfg,batch", [("cfg2", 4), ("cfg3", 8), ("cfg3_f32", 8)])
def test_full_size_fused_path_with_padding_mask(cfg, batch):
    """The module's fused path (softmax + location affine + key_padding_mask inside the kernels) at full size
    against the step-by-step composition the reference module performs (masked_fill, softmax, location arithmetic:
    multi_scale_deform_attn.py:289-332) around the reference formulation in float64."""
    ir, _lib, functional, workloads, msda_torch = _mods()
    from ir_ads_b200.functional import MSDeformAttnFusedFunction
    wl = workloads.WORKLOADS[cfg]
    torch.manual_seed(3)
    shapes, lsi = workloads.level_tensors(wl.levels, DEV)
    S, Q, H, D, L, P = wl.spatial_size, wl.queries, wl.num_heads, wl.head_dim, wl.num_levels, wl.num_points
    vdt = torch.bfloat16 if wl.value_dtype == "bf16" else torch.float32
    value = torch.randn(batch, S, H, D, device=DEV).to(vdt)
    # offsets as the module's init pattern + noise (pixels), logits ~ N(0, 1)
    steps = torch.arange(1, P + 1, device=DEV, dtype=torch.float32)
    off = workloads._head_directions(H, DEV)[None, None, :, None, None, :] * steps[None, None, None, None, :, None]
    off = (off + 2.0 * torch.randn(batch, Q, H, L, P, 2, device=DEV)).contiguous()
    logits = torch.randn(batch, Q, H, L * P, device=DEV)
    if wl.kind == "encoder":
        ref = workloads._pixel_centres(wl.levels, DEV)[None, :, None, :].expand(batch, Q, L, 2).contiguous()
    else:
        ref = torch.cat([torch.rand(batch, Q, 1, 2, device=DEV), 0.02 + 0.48 * torch.rand(batch, Q, 1, 2, device=DEV)],
                        -1).expand(batch, Q, L, 4).contiguous()
    # batch-padding pattern: the right / bottom margins of every level of every second image
    mask = torch.zeros(batch, S, dtype=torch.bool, device=DEV)
    start = 0
    for h, wd in wl.levels:
        mm = torch.zeros(h, wd, dtype=torch.bool, device=DEV)
        mm[:, (4 * wd) // 5:] = True
        mm[(5 * h) // 6:, :] = True
        mask[1::2, start:start + h * wd] = mm.reshape(-1)
        start += h * wd
    go = torch.randn(batch, Q, H * D, device=DEV).to(vdt)

    leaves = [t.clone().requires_grad_(True) for t in (value, off, logits)]
    out = MSDeformAttnFusedFunction.apply(leaves[0], shapes, lsi, leaves[1], leaves[2], ref, mask)
    out.backward(go)
    torch.cuda.synchronize()

    # reference composition in float64, autograd through the reference formulation
    v64 = value.double().requires_grad_(True)
    o64 = off.double().requires_grad_(True)
    l64 = logits.double().requires_grad_(True)
    vm = v64.masked_fill(mask[..., None, None], 0.0)                                   # py:291-292
    ww = l64.softmax(-1).view(batch, Q, H, L, P)                                       # py:303-310
    r64 = ref.double()
    if ref.shape[-1] == 2:                                                             # py:313-324
        norm = torch.stack([shapes[..., 1], shapes[..., 0]], -1).double()
        lo = r64[:, :, None, :, None, :] + o64 / norm[None, None, None, :, None, :]
    else:                                                                              # py:325-332
        lo = r64[:, :, None, :, None, :2] + o64 / P * r64[:, :, None, :, None, 2:] * 0.5
    want = msda_torch.forward(vm, shapes, lo, ww)
    want.backward(go.double())
    torch.cuda.synchronize()

    bf16 = vdt == torch.bfloat16
    rt = 1e-2 if bf16 else 1e-5
    # the kernels form loc in float32 (the module's arithmetic): a location moves by ~1e-7 relative to the float64
    # composition, which moves a sample across a cell boundary only inside the masked band
    m = smooth_mask_t(lo.detach(), shapes, 2e-4).double()
    ok = True
    for tn, g, t, rtol, msk in (("out", out.detach(), want.detach(), rt if bf16 else 2e-5, None),
                                ("grad_value", leaves[0].grad, v64.grad, rt if bf16 else 2e-5, None),
                                ("grad_offsets", leaves[1].grad, o64.grad, 1e-4, m),
                                ("grad_logits", leaves[2].grad, l64.grad, 1e-4, None)):
        good, *_ = report(f"{cfg}_fused_mask/{tn}", g, t, rtol, 1e-6, msk)
        ok = ok and good
    assert ok
    assert float(leaves[0].grad[mask].abs().max()) == 0.0       # masked pixels receive no gradient

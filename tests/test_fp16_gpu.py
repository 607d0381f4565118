"""float16 value (MSDA_F16) on the sm_100a kernels.

A float16 number widens exactly to float32 and every kernel computes in float32 from widened values, so the float16
kernels must give the float32 kernels' numbers on ``value.float()`` / ``grad_out.float()`` with only the final stores
rounded: the output equal to ``out32.half()``, the float32 gradients (locations, weights, the fused path's offsets /
logits, DCNv3's offset / mask) equal bit for bit, and grad_value equal to ``gv32.half()`` under
MSDA_FLAG_DETERMINISTIC.  With float reds grad_value is a float32 sum in an order that changes from run to run, for
float32 as well: there it is checked to one float16 ulp plus that run-to-run spread, which is bounded by
64 float32 ulps of the sum of the contributions' magnitudes (the same backward with |grad_out|).  The public reference-signature op refuses
float16 (as the reference's does), so the plain op is driven through the C ABI here.
"""
import copy
import ctypes

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES  # noqa: F401  (same golden file)
from test_oracle import smooth_mask

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _p(t):
    return ctypes.c_void_p(t.data_ptr() if t is not None else 0)


def c_op(value, shapes, lsi, loc, w, go, flags=0):
    """msda_forward + msda_backward through the C ABI for any value dtype: (out, grad_value, grad_loc, grad_w)."""
    from ir_ads_b200 import _lib, functional
    tag = functional._VALUE_TAG[value.dtype]
    B, S, H, D = value.shape
    _, Q, _, L, P, _ = loc.shape
    h = _lib.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.empty(B, Q, H * D, dtype=value.dtype, device=value.device)
    _lib.check(h.msda_forward(st, _p(value), _p(shapes), _p(lsi), _p(loc), _p(w), B, S, H, D, L, Q, P, _p(out), tag,
                              flags), "msda_forward")
    gv, gl, gw = torch.empty_like(value), torch.empty_like(loc), torch.empty_like(w)
    ws_bytes = int(h.msda_backward_workspace_bytes(B, S, H, D, L, Q, P, tag, flags))
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=value.device)
    _lib.check(h.msda_backward(st, _p(go.contiguous()), _p(value), _p(shapes), _p(lsi), _p(loc), _p(w), B, S, H, D, L, Q,
                               P, _p(gv), _p(gl), _p(gw), _p(ws), ws_bytes, tag, flags), "msda_backward")
    return out, gv, gl, gw


def f16_ulp(x):
    """Spacing of float16 at |x| (x float32): 2^(e-11) for x = m * 2^e, m in [0.5, 1); 2^-24 in the subnormal range."""
    _, e = torch.frexp(x.abs().float())
    return torch.clamp(torch.ldexp(torch.ones_like(x, dtype=torch.float32), (e - 11).to(torch.int32)), min=2.0 ** -24)


def assert_within_one_ulp(got16, want32, gv_abs, what):
    """|got16 - want32.half()| <= one float16 ulp + 64 float32 ulps of gv_abs (sum of |contributions|: red order)."""
    a, b = got16.float(), want32.half().float()
    bound = f16_ulp(torch.maximum(a.abs(), b.abs())) + 64 * 2.0 ** -24 * gv_abs.float()
    bad = ((a - b).abs() > bound) | (torch.isnan(a) != torch.isnan(b))
    assert not bad.any(), f"{what}: {int(bad.sum())} elements more than one float16 ulp (+ red-order spread) apart"


def assert_identity(r16, r32, what, det=False, gv_abs=None):
    out16, gv16, gl16, gw16 = r16
    out32, gv32, gl32, gw32 = r32
    assert out16.dtype == torch.float16 and gv16.dtype == torch.float16
    assert torch.equal(out16, out32.half()), f"{what}: out"
    assert torch.equal(gl16, gl32), f"{what}: grad_loc"
    assert torch.equal(gw16, gw32), f"{what}: grad_w"
    if det:
        assert torch.equal(gv16, gv32.half()), f"{what}: grad_value (deterministic)"
    else:
        assert_within_one_ulp(gv16, gv32, gv_abs, f"{what}: grad_value")


def _inputs(levels, B, Q, H, D, P, kind="decoder", dist="edge", seed=7):
    from ir_ads_b200.workloads import make_inputs
    value, shapes, lsi, loc, w = make_inputs(levels, B, Q, H, D, P, kind, dist, seed, DEV)
    Qr = loc.shape[1]
    go = torch.randn(B, Qr, H * D, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 1))
    return value.half(), shapes, lsi, loc, w, go.half()


def assert_close(got, ref, rtol, atol, what):
    got = got.detach().double().cpu().numpy() if torch.is_tensor(got) else got
    bound = rtol * np.abs(ref).max() + atol
    worst = np.abs(got - ref).max()
    assert worst <= bound, f"{what}: max abs err {worst:.3e} > {bound:.3e}"


# ------------------------------------------------------------------------------------------------
# 1. golden cases against the float64 oracle on the float16-rounded inputs
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["d32", "d64", "edge_d32", "enc_mini", "dec_mini", "stress_mini"])
def test_f16_value_matches_reference_golden(golden, name):
    from oracle import msda_c
    c = golden(name)
    v16 = torch.as_tensor(c["value"]).half()
    go16 = torch.as_tensor(c["grad_out"]).half()
    v, go = v16.float().numpy(), go16.float().numpy()
    ref_out = msda_c.forward(v, c["shapes"], c["lsi"], c["loc"], c["w"], np.float64)
    rgv, rgl, rgw = msda_c.backward(go, v, c["shapes"], c["lsi"], c["loc"], c["w"], np.float64)
    dev = lambda a, dt=None: torch.as_tensor(a).to(DEV, dt) if dt else torch.as_tensor(a).to(DEV)
    out, gv, gl, gw = c_op(dev(v16), dev(c["shapes"]), dev(c["lsi"]), dev(c["loc"], torch.float32),
                           dev(c["w"], torch.float32), dev(go16))
    torch.cuda.synchronize()
    m = smooth_mask(c["loc"], c["shapes"], band=1e-4)
    assert_close(out, ref_out, 1e-3, 0.0, "out")                 # float16 output rounding: 2^-11 relative
    assert_close(gv, rgv, 1e-3, 0.0, "grad_value")
    assert_close(gw, rgw, 1e-5, 1e-6, "grad_w")                  # float32 outputs: the float32 bounds
    assert_close(gl.detach().double().cpu().numpy() * m, rgl * m, 1e-5, 1e-6, "grad_loc")


# ------------------------------------------------------------------------------------------------
# 2. identity with the float32 kernels on widened inputs
# ------------------------------------------------------------------------------------------------
LEVELS = [(9, 7), (5, 4), (3, 2), (2, 2), (1, 1)]


@pytest.mark.parametrize("generic", [False, True])
@pytest.mark.parametrize("D,L,P", [(16, 2, 4), (32, 4, 4), (32, 5, 8), (64, 3, 3), (128, 1, 8), (32, 4, 3),
                                   (16, 5, 8), (64, 4, 4), (128, 2, 3)])
def test_f16_equals_f32_on_widened_inputs(D, L, P, generic):
    from ir_ads_b200 import _lib
    flags = _lib.FLAG_FORCE_GENERIC if generic else 0
    value, shapes, lsi, loc, w, go = _inputs(LEVELS[:L], 2, 37, 4, D, P)
    name = _lib.lib().msda_dispatch_name(D, L, P, value.shape[1], 4, _lib.MSDA_F16, flags, 0).decode()
    assert ("generic" in name) == generic, name
    r16 = c_op(value, shapes, lsi, loc, w, go, flags)
    r32 = c_op(value.float(), shapes, lsi, loc, w, go.float(), flags)
    gv_abs = c_op(value.float(), shapes, lsi, loc, w.abs(), go.float().abs(), flags)[1]
    torch.cuda.synchronize()
    assert_identity(r16, r32, f"D={D} L={L} P={P} {name}", gv_abs=gv_abs)


def test_f16_no_grad_value_route():
    """MSDA_FLAG_NO_GRAD_VALUE (frozen value): the scatter-free kernel gives the same float32 gradients."""
    from ir_ads_b200 import _lib
    value, shapes, lsi, loc, w, go = _inputs(LEVELS[:4], 2, 37, 8, 32, 4, dist="model")
    B, S, H, D = value.shape
    _, Q, _, L, P, _ = loc.shape
    gl, gw = torch.empty_like(loc), torch.empty_like(w)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(_lib.lib().msda_backward(st, _p(go), _p(value), _p(shapes), _p(lsi), _p(loc), _p(w), B, S, H, D, L, Q, P,
                                        _p(None), _p(gl), _p(gw), _p(None), 0, _lib.MSDA_F16, _lib.FLAG_NO_GRAD_VALUE),
               "msda_backward")
    _, _, gl32, gw32 = c_op(value.float(), shapes, lsi, loc, w, go.float())
    torch.cuda.synchronize()
    assert torch.equal(gl, gl32) and torch.equal(gw, gw32)


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("ref_dim,D,L,P", [(2, 32, 4, 4), (4, 32, 4, 4), (2, 64, 3, 8), (4, 16, 2, 3), (2, 128, 1, 5)])
def test_fused_function_f16_equals_f32(ref_dim, D, L, P, masked):
    from ir_ads_b200.functional import MSDeformAttnFusedFunction
    from ir_ads_b200.workloads import level_tensors
    g = torch.Generator(device=DEV).manual_seed(D + L + P + ref_dim)
    levels = [(11, 13), (6, 7), (3, 4), (2, 2)][:L]
    shapes, lsi = level_tensors(levels, DEV)
    S, B, Q, H = sum(h * w for h, w in levels), 2, 29, 4
    value = torch.randn(B, S, H, D, device=DEV, generator=g).half()
    off = torch.randn(B, Q, H, L, P, 2, device=DEV, generator=g) * 2.0
    logits = torch.randn(B, Q, H, L * P, device=DEV, generator=g)
    ref = torch.rand(B, Q, L, ref_dim, device=DEV, generator=g)
    go = torch.randn(B, Q, H * D, device=DEV, generator=g).half()
    mask = (torch.rand(B, S, device=DEV, generator=g) < 0.2) if masked else None

    def run(v, gout):
        leaves = [t.clone().requires_grad_(True) for t in (v, off, logits)]
        out = MSDeformAttnFusedFunction.apply(leaves[0], shapes, lsi, leaves[1], leaves[2], ref, mask)
        out.backward(gout)
        return out.detach(), leaves[0].grad, leaves[1].grad, leaves[2].grad

    r16, r32 = run(value, go), run(value.float(), go.float())
    gv_abs = run(value.float(), go.float().abs())[1]                # softmax weights are positive
    torch.cuda.synchronize()
    assert_identity(r16, r32, f"fused ref_dim={ref_dim} D={D} masked={masked}", gv_abs=gv_abs)


def _dcn_case(stride, pad, dil, scale, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    N, H, W, G, C, k = 2, 48, 64, 8, 32, 3
    Ho = (H + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
    Wo = (W + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
    inp = torch.randn(N, H, W, G * C, device=DEV, generator=g).half()
    off = torch.randn(N, Ho, Wo, G * 9 * 2, device=DEV, generator=g) * 2.0
    mask = torch.softmax(torch.randn(N, Ho, Wo, G, 9, device=DEV, generator=g), -1).reshape(N, Ho, Wo, G * 9)
    go = torch.randn(N, Ho, Wo, G * C, device=DEV, generator=g).half()
    return inp, off, mask, go, (k, k, stride, stride, pad, pad, dil, dil, G, C, scale)


@pytest.mark.parametrize("stride,pad,dil,scale", [(1, 1, 1, 1.0), (2, 1, 1, 2.0), (1, 2, 2, 0.7)])
def test_dcnv3_f16_equals_f32(stride, pad, dil, scale):
    from ir_ads_b200.dcnv3 import DCNv3Function
    inp, off, mask, go, args = _dcn_case(stride, pad, dil, scale)

    def run(x, gout):
        leaves = [t.clone().requires_grad_(True) for t in (x, off, mask)]
        out = DCNv3Function.apply(*leaves, *args, 256)
        out.backward(gout)
        return out.detach(), leaves[0].grad, leaves[1].grad, leaves[2].grad

    r16, r32 = run(inp, go), run(inp.float(), go.float())
    gv_abs = run(inp.float(), go.float().abs())[1]                   # the masks are positive
    torch.cuda.synchronize()
    assert_identity(r16, r32, f"dcnv3 stride={stride} dil={dil}", gv_abs=gv_abs)


# ------------------------------------------------------------------------------------------------
# 3. deterministic backward
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,Q", [(32, 4000), (64, 4000), (32, 4)])
def test_f16_deterministic_backward(D, Q):
    """Contended shape (many queries onto a tiny map: dense, cell-reduce route) and a sparse one (per-pixel gather
    route): three runs bit-identical, the sorted reduction == the fixed-point reds, and each route -- the generic
    kernels too -- equal to the same route's float32 result rounded to float16.  (The generic kernels form their
    fixed-point products in another order than the fast ones, in float32 as well, so they are compared with their own
    float32 twin.)"""
    from ir_ads_b200 import _lib
    det = _lib.FLAG_DETERMINISTIC
    value, shapes, lsi, loc, w, go = _inputs([(5, 7), (3, 4), (2, 2)], 2, Q, 4, D, 4, dist="model", seed=21)
    runs = [c_op(value, shapes, lsi, loc, w, go, det) for _ in range(3)]
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b)
    atomic = c_op(value, shapes, lsi, loc, w, go, det | _lib.FLAG_DET_ATOMIC)
    generic = c_op(value, shapes, lsi, loc, w, go, det | _lib.FLAG_FORCE_GENERIC)
    assert torch.equal(atomic[1], runs[0][1])
    r32 = c_op(value.float(), shapes, lsi, loc, w, go.float(), det)
    g32 = c_op(value.float(), shapes, lsi, loc, w, go.float(), det | _lib.FLAG_FORCE_GENERIC)
    torch.cuda.synchronize()
    assert_identity(runs[0], r32, "deterministic sorted", det=True)
    assert_identity(atomic, r32, "deterministic fixed-point reds", det=True)
    assert_identity(generic, g32, "deterministic generic", det=True)


# ------------------------------------------------------------------------------------------------
# 4. non-finite values
# ------------------------------------------------------------------------------------------------
def test_f16_inf_nan_propagate_like_f32():
    """Inf / NaN in pixels that points sample: the widening (HADD2.F32) keeps them, so every output is what the
    float32 kernel gives on the widened value -- same NaN positions, same infinities, same finite numbers."""
    value, shapes, lsi, loc, w, go = _inputs([(6, 5), (3, 3)], 1, 16, 2, 32, 4, dist="model", seed=5)
    value[0, 3, 0, 5] = float("inf")
    value[0, 7, 1, 9] = float("nan")
    value[0, 12, 0, 0] = -float("inf")
    value[0, 14, 1, 3] = 2.0 ** -20                                # a subnormal float16 stays exact as well
    r16 = c_op(value, shapes, lsi, loc, w, go)
    r32 = c_op(value.float(), shapes, lsi, loc, w, go.float())
    torch.cuda.synchronize()
    same = lambda a, b: torch.equal(torch.nan_to_num(a, nan=7.0), torch.nan_to_num(b, nan=7.0)) and torch.equal(
        torch.isnan(a), torch.isnan(b))
    assert not torch.isfinite(r32[0]).all(), "the non-finite pixels must be sampled for this test to mean anything"
    assert same(r16[0], r32[0].half()), "out"
    assert same(r16[2], r32[2]) and same(r16[3], r32[3]), "grad_loc / grad_w"


def test_f16_unsampled_non_finite_padding_stays_finite():
    """A NaN / Inf in a pixel no point loads (corners outside the map are never read) changes nothing."""
    from ir_ads_b200.workloads import level_tensors
    shapes, lsi = level_tensors([(4, 4)], DEV)
    B, S, H, D, Q, P = 1, 16, 2, 32, 3, 2
    value = torch.randn(B, S, H, D, device=DEV).half()
    loc = torch.tensor([0.30, 0.30], device=DEV).expand(B, Q, H, 1, P, 2).contiguous()   # cell (0..1, 0..1) only
    w = torch.full((B, Q, H, 1, P), 0.5, device=DEV)
    go = torch.randn(B, Q, H * D, device=DEV).half()
    clean = c_op(value, shapes, lsi, loc, w, go)
    dirty_v = value.clone()
    dirty_v[0, 15] = float("nan")                                   # pixel (3, 3): never a corner
    dirty_v[0, 10] = float("inf")                                   # pixel (2, 2): never a corner
    dirty = c_op(dirty_v, shapes, lsi, loc, w, go)
    torch.cuda.synchronize()
    for a, b in zip(clean, dirty):
        assert torch.isfinite(b).all() and torch.equal(a, b)


# ------------------------------------------------------------------------------------------------
# 5. full size
# ------------------------------------------------------------------------------------------------
def _full(cfg):
    from ir_ads_b200.workloads import WORKLOADS, make_workload_inputs
    wl = WORKLOADS[cfg]
    value, shapes, lsi, loc, w = make_workload_inputs(wl, "model", 0, DEV)
    B, Q, H, D = value.shape[0], loc.shape[1], value.shape[2], value.shape[3]
    go = torch.randn(B, Q, H * D, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1)).half()
    return value.half(), shapes, lsi, loc, w, go


def test_f16_full_size_cfg2():
    value, shapes, lsi, loc, w, go = _full("cfg2")
    assert value.shape[0] == 8
    r16 = c_op(value, shapes, lsi, loc, w, go)
    r32 = c_op(value.float(), shapes, lsi, loc, w, go.float())
    gv_abs = c_op(value.float(), shapes, lsi, loc, w, go.float().abs())[1]
    torch.cuda.synchronize()
    assert_identity(r16, r32, "cfg2 B=8", gv_abs=gv_abs)


def test_f16_full_size_cfg5_deterministic():
    from ir_ads_b200 import _lib
    value, shapes, lsi, loc, w, go = _full("cfg5")
    assert value.shape[0] == 8
    r16 = c_op(value, shapes, lsi, loc, w, go, _lib.FLAG_DETERMINISTIC)
    r32 = c_op(value.float(), shapes, lsi, loc, w, go.float(), _lib.FLAG_DETERMINISTIC)
    torch.cuda.synchronize()
    assert torch.equal(r16[1], r32[1].half())
    assert_identity(r16, r32, "cfg5 B=8 deterministic", det=True)


# ------------------------------------------------------------------------------------------------
# 6. module under float16 autocast
# ------------------------------------------------------------------------------------------------
def _module_case():
    from ir_ads_b200 import MultiScaleDeformableAttention
    from ir_ads_b200.workloads import level_tensors
    torch.manual_seed(0)
    levels = [(12, 17), (6, 9), (3, 5), (2, 3)]
    shapes, lsi = level_tensors(levels, DEV)
    S = sum(h * w for h, w in levels)
    m = MultiScaleDeformableAttention(dropout=0.0, batch_first=True).to(DEV)
    with torch.no_grad():
        m.sampling_offsets.weight.normal_(0, 0.05)
        m.attention_weights.weight.normal_(0, 0.2)
    q = torch.randn(2, S, 256, device=DEV)
    ref_pts = torch.rand(2, S, 4, 2, device=DEV)
    return m, q, ref_pts, shapes, lsi


def _widening_route(m, q, ref_pts, shapes, lsi):
    """The module's fused path as it was before the float16 kernels: value widened to float32 in front of the fused
    Function, its output rounded to float16 before output_proj."""
    from ir_ads_b200.functional import MSDeformAttnFusedFunction
    B, Q, _ = q.shape
    H, L, P = m.num_heads, m.num_levels, m.num_points
    value = m.value_proj(q).view(B, Q, H, -1).float()
    offsets = m.sampling_offsets(q).view(B, Q, H, L, P, 2)
    logits = m.attention_weights(q).view(B, Q, H, L * P)
    out = MSDeformAttnFusedFunction.apply(value.contiguous(), shapes, lsi, offsets.float().contiguous(),
                                          logits.float().contiguous(), ref_pts.float().contiguous(), None)
    return m.output_proj(out.half()) + q


def test_module_fp16_autocast_matches_widening_route():
    m, q, ref_pts, shapes, lsi = _module_case()
    m_old = copy.deepcopy(m)
    gout = torch.randn(q.shape, device=DEV)
    with torch.autocast("cuda", dtype=torch.float16):
        new = m(q, reference_points=ref_pts, spatial_shapes=shapes, level_start_index=lsi)
        old = _widening_route(m_old, q, ref_pts, shapes, lsi)
    assert torch.equal(new, old)
    (new * gout).sum().backward()
    (old * gout).sum().backward()
    torch.cuda.synchronize()
    for (k, p), p_old in zip(m.named_parameters(), m_old.parameters()):
        err = (p.grad - p_old.grad).abs().max().item()
        assert err <= 1e-3 * p_old.grad.abs().max().item() + 1e-9, (k, err)


def test_module_fp16_autocast_saves_fp16_value():
    m, q, ref_pts, shapes, lsi = _module_case()
    B, S, _ = q.shape
    saved = []

    def pack(t):
        saved.append((t.dtype, tuple(t.shape)))
        return t

    with torch.autograd.graph.saved_tensors_hooks(pack, lambda t: t):
        with torch.autocast("cuda", dtype=torch.float16):
            m(q, reference_points=ref_pts, spatial_shapes=shapes, level_start_index=lsi)
    value_shape = (B, S, m.num_heads, m.embed_dim // m.num_heads)
    kinds = [dt for dt, shape in saved if shape == value_shape]
    assert kinds == [torch.float16], saved


def test_module_fp16_autocast_cuda_graph():
    m, q, ref_pts, shapes, lsi = _module_case()
    x = q.clone().requires_grad_(True)

    def step():
        with torch.autocast("cuda", dtype=torch.float16, cache_enabled=False):
            out = m(x, reference_points=ref_pts, spatial_shapes=shapes, level_start_index=lsi)
        out.float().square().mean().backward()
        return out

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            m.zero_grad(set_to_none=True); x.grad = None
            step()
    torch.cuda.current_stream().wait_stream(side)
    m.zero_grad(set_to_none=True); x.grad = None
    eager = step().detach().clone()
    eager_grad = x.grad.detach().clone()
    m.zero_grad(set_to_none=True); x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    x.grad.zero_()
    for p in m.parameters():
        p.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert captured.dtype == eager.dtype and torch.equal(captured, eager)
    assert torch.allclose(x.grad, eager_grad, rtol=1e-3, atol=1e-6)     # grad_value reds reorder


# ------------------------------------------------------------------------------------------------
# 7. detrex._C.dcnv3_forward / dcnv3_backward with half tensors
# ------------------------------------------------------------------------------------------------
def test_C_dcnv3_half_input_offset_mask():
    from oracle import dcnv3_torch
    from test_dcnv3 import pixel_smooth_mask

    from ir_ads_b200 import _C
    for stride, pad, dil, scale in ((1, 1, 1, 1.0), (2, 1, 1, 2.0)):
        inp, off, mask, go, args = _dcn_case(stride, pad, dil, scale, seed=3)
        off, mask = off.half(), mask.half()
        out = _C.dcnv3_forward(inp, off, mask, *args, 256)
        gi, goff, gm = _C.dcnv3_backward(inp, off, mask, *args, go, 256)
        torch.cuda.synchronize()
        assert out.dtype == gi.dtype == goff.dtype == gm.dtype == torch.float16
        want = dcnv3_torch.forward_backward(inp.double(), off.double(), mask.double(), go.double(), *args)
        m = torch.from_numpy(pixel_smooth_mask({"offset": off.float().cpu().numpy(), "args": args}, 1e-4)).to(DEV)
        for a, b, key in zip((out, gi, goff, gm), want, ("out", "grad_input", "grad_offset", "grad_mask")):
            mk = m.double() if key == "grad_offset" else 1.0
            err = ((a.double() - b) * mk).abs().max().item()
            assert err <= 2e-3 * b.abs().max().item() + 1e-6, (key, stride, err)


def test_dcnv3_function_f16_has_no_widening_copy():
    from ir_ads_b200 import _lib
    from ir_ads_b200.dcnv3 import DCNv3Function
    inp, off, mask, go, args = _dcn_case(1, 1, 1, 1.0, seed=4)
    x = inp.clone().requires_grad_(True)
    DCNv3Function.apply(x, off, mask, *args, 256).backward(go)            # warm-up
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    out = DCNv3Function.apply(x, off, mask, *args, 256)
    assert _lib.launch_count() - n0 == 1                                  # the fast forward, float16 in and out
    n0 = _lib.launch_count()
    out.backward(go)
    assert _lib.launch_count() - n0 == 2                                  # the fast backward + float -> half cast
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU], record_shapes=True) as prof:
        DCNv3Function.apply(x, off, mask, *args, 256).backward(go)
        torch.cuda.synchronize()
    big = tuple(inp.shape)
    copies = [e for e in prof.events() if e.name == "aten::_to_copy"
              and any(tuple(s) == big for s in (e.input_shapes or []) if isinstance(s, (list, tuple)))]
    assert not copies, [(e.name, e.input_shapes) for e in copies]

"""GPU parity tests proper: the sm_100a kernels, called through the C ABI (ctypes -> libmsda_b200.so
via ir_ads_b200.functional), against the CPU oracle and the reference-made golden vectors.

Tolerances (BASELINE.json north_star): fp32 within 1e-5 relative + 1e-6 absolute, bf16 value with
fp32 accumulate within 1e-2 relative, index bookkeeping bit-exact.  "Relative" is taken against the
largest magnitude of the reference tensor (a sum of 64 products has no meaningful per-element
relative error when it cancels to ~0); where values are small (the reference test's own
distribution) the per-element torch.allclose criterion of the reference test is applied as well.
"""
import ctypes

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES
from test_oracle import smooth_mask

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _mods():
    import ir_ads_b200
    from ir_ads_b200 import _lib, functional, workloads
    from oracle import msda_c, msda_torch
    return ir_ads_b200, _lib, functional, workloads, msda_c, msda_torch


def run_cuda(value, shapes, lsi, loc, w, go, dtype=torch.float32, flags=0):
    ir, _lib, functional, *_ = _mods()
    aux = torch.float64 if dtype == torch.float64 else torch.float32
    v = torch.as_tensor(value).detach().to(DEV, dtype).clone().requires_grad_(True)
    lo = torch.as_tensor(loc).detach().to(DEV, aux).clone().requires_grad_(True)
    ww = torch.as_tensor(w).detach().to(DEV, aux).clone().requires_grad_(True)
    with functional.kernel_flags(flags):
        out = ir.MultiScaleDeformableAttnFunction.apply(v, torch.as_tensor(shapes).to(DEV), torch.as_tensor(lsi).to(DEV),
                                                        lo, ww, 64)
        out.backward(torch.as_tensor(go).to(DEV, dtype))
    torch.cuda.synchronize()
    f = lambda t: t.detach().double().cpu().numpy()
    return f(out), f(v.grad), f(lo.grad), f(ww.grad)


def needs_experiments():
    """The folding backward lives in -DMSDA_EXPERIMENTS builds only (MSDA_B200_LIB=build/variants/lib_exp.so)."""
    if not _mods()[1].has_experiments():
        pytest.skip("product library: experiment kernels not compiled in (tools/build_variant.sh exp -DMSDA_EXPERIMENTS)")


def nerr(a, b):
    """max |a-b| normalised by max |b|."""
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def assert_close(got, ref, rtol, atol, what):
    bound = rtol * np.abs(ref).max() + atol
    worst = np.abs(got - ref).max()
    assert worst <= bound, f"{what}: max abs err {worst:.3e} > {bound:.3e} (ref max {np.abs(ref).max():.3e})"


# ------------------------------------------------------------------------------------------------
# golden vectors made by the reference
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_fp32_matches_reference_golden(golden, name):
    c = golden(name)
    out, gv, gl, gw = run_cuda(c["value"], c["shapes"], c["lsi"], c["loc"], c["w"], c["grad_out"])
    m = smooth_mask(c["loc"], c["shapes"], band=1e-4)
    assert_close(out, c["f64/out"], 1e-5, 1e-6, "out")
    assert_close(gv, c["f64/grad_value"], 1e-5, 1e-6, "grad_value")
    assert_close(gw, c["f64/grad_w"], 1e-5, 1e-6, "grad_w")
    assert_close(gl * m, c["f64/grad_loc"] * m, 1e-5, 1e-6, "grad_loc")
    if name in ("ref_test", "d30", "d32", "d64", "d71", "d1025"):  # the reference test's own criterion and value scale
        assert np.allclose(out, c["f64/out"], rtol=1e-5, atol=1e-8)


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_fp64_matches_reference_golden(golden, name):
    """The reference's own pin (tests/test_ms_deform_attn.py:103-129): double, allclose defaults."""
    c = golden(name)
    out, gv, gl, gw = run_cuda(c["value"], c["shapes"], c["lsi"], c["loc"], c["w"], c["grad_out"], torch.float64)
    m = smooth_mask(c["loc"], c["shapes"])
    assert np.allclose(out, c["f64/out"], rtol=1e-5, atol=1e-8)
    assert nerr(out, c["f64/out"]) < 1e-13
    assert nerr(gv, c["f64/grad_value"]) < 1e-12
    assert nerr(gw, c["f64/grad_w"]) < 1e-12
    assert nerr(gl * m, c["f64/grad_loc"] * m) < 1e-12


@pytest.mark.parametrize("name", ["d32", "d64", "edge_d32", "enc_mini", "dec_mini", "stress_mini"])
def test_bf16_value_matches_reference_golden(golden, name):
    c = golden(name)
    vb = torch.as_tensor(c["value"]).bfloat16()
    gob = torch.as_tensor(c["grad_out"]).bfloat16()
    _, _, _, _, msda_c, _ = _mods()
    # oracle on the SAME (bf16-rounded) inputs, evaluated in fp64
    ref_out = msda_c.forward(vb.float().numpy(), c["shapes"], c["lsi"], c["loc"], c["w"], np.float64)
    rgv, rgl, rgw = msda_c.backward(gob.float().numpy(), vb.float().numpy(), c["shapes"], c["lsi"], c["loc"], c["w"], np.float64)
    out, gv, gl, gw = run_cuda(vb, c["shapes"], c["lsi"], c["loc"], c["w"], gob, torch.bfloat16)
    m = smooth_mask(c["loc"], c["shapes"], band=1e-4)
    assert_close(out, ref_out, 1e-2, 1e-6, "out")          # bf16 output rounding: 2^-9 relative
    assert_close(gv, rgv, 1e-2, 1e-6, "grad_value")
    assert_close(gw, rgw, 1e-4, 1e-6, "grad_w")             # fp32 outputs: only fp32 accumulate error
    assert_close(gl * m, rgl * m, 1e-4, 1e-6, "grad_loc")


# ------------------------------------------------------------------------------------------------
# the channel counts the reference's gradcheck walks, fast vs generic dispatch
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("channels", [30, 32, 64, 71, 1025, 16, 128, 2048])
def test_channels_against_oracle(channels):
    _, _, _, workloads, msda_c, _ = _mods()
    levels = [(6, 4), (3, 2)]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 2, 5, 2, channels, 2, "decoder", "edge", 40 + channels)
    go = torch.randn(2, 5, 2 * channels, generator=torch.Generator().manual_seed(channels))
    a = [t.numpy() for t in (value, shapes, lsi, loc, w)]
    ref_out = msda_c.forward(*a, np.float64)
    rgv, rgl, rgw = msda_c.backward(go.numpy(), *a, np.float64)
    m = smooth_mask(a[3], a[1], band=1e-4)
    for dtype, tol in ((torch.float64, 1e-12), (torch.float32, 1e-5)):
        out, gv, gl, gw = run_cuda(*a, go, dtype)
        assert_close(out, ref_out, tol, tol * 0.1, f"out D={channels} {dtype}")
        assert_close(gv, rgv, tol, tol * 0.1, "grad_value")
        assert_close(gw, rgw, tol, tol * 0.1, "grad_w")
        assert_close(gl * m, rgl * m, tol, tol * 0.1, "grad_loc")


@pytest.mark.parametrize("channels", [30, 32, 64, 71])
def test_gradcheck_double(channels):
    """tests/test_ms_deform_attn.py:131-133 (gradcheck in fp64), same tiny shape."""
    ir, *_ = _mods()
    N, M, Lq, L, P = 1, 2, 2, 2, 2
    shapes = torch.as_tensor([(6, 4), (3, 2)], dtype=torch.long, device=DEV)
    lsi = torch.cat((shapes.new_zeros((1,)), shapes.prod(1).cumsum(0)[:-1]))
    S = 30
    g = torch.Generator(device=DEV).manual_seed(channels)
    value = (torch.rand(N, S, M, channels, device=DEV, generator=g) * 0.01).double().requires_grad_(True)
    loc = torch.rand(N, Lq, M, L, P, 2, device=DEV, generator=g).double().requires_grad_(True)
    w = torch.rand(N, Lq, M, L, P, device=DEV, generator=g) + 1e-5
    w = (w / w.sum(-1, keepdim=True).sum(-2, keepdim=True)).double().requires_grad_(True)
    assert torch.autograd.gradcheck(ir.MultiScaleDeformableAttnFunction.apply, (value, shapes, lsi, loc, w, 2))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("D,L,P", [(32, 4, 4), (32, 5, 8), (64, 3, 4), (16, 2, 3), (128, 1, 5), (32, 4, 1)])
def test_fast_and_generic_kernels_agree(D, L, P, dtype):
    _, _lib, _, workloads, _, _ = _mods()
    levels = [(9, 7), (5, 4), (3, 2), (2, 2), (1, 1)][:L]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 2, 37, 4, D, P, "decoder", "edge", 7, value_dtype=dtype)
    go = torch.randn(2, 37, 4 * D, generator=torch.Generator().manual_seed(1)).to(dtype)
    fast = run_cuda(value, shapes, lsi, loc, w, go, dtype)
    slow = run_cuda(value, shapes, lsi, loc, w, go, dtype, flags=_lib.FLAG_FORCE_GENERIC)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    for f, s, name in zip(fast, slow, ("out", "grad_value", "grad_loc", "grad_w")):
        assert_close(f, s, tol, 1e-6, name)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("D,P", [(32, 4), (64, 4), (16, 8), (128, 2), (32, 3)])
def test_row_orders_agree(D, P, dtype):
    """Row order is a scheduling choice: STRIP, TILE2D (encoder form, Q == S) and the folding backward must give
    the same forward and the same grad_loc / grad_w as the LINEAR order bit for bit (same per-row arithmetic) and
    the same grad_value up to float summation order.  (The product library carries one order per pass and ignores
    the order hints, so there the comparison is trivially true; the experiment build -- the second pytest command of
    tools/gpu_calls/gpu_r02*.sh -- instantiates and honours all of them.)"""
    _, _lib, _, workloads, msda_c, _ = _mods()
    levels = [(21, 37), (11, 19), (6, 10), (3, 5)]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 2, 0, 4, D, P, "encoder", "model", 3, value_dtype=dtype)
    go = torch.randn(2, value.shape[1], 4 * D, generator=torch.Generator().manual_seed(1)).to(dtype)
    linear = run_cuda(value, shapes, lsi, loc, w, go, dtype, flags=_lib.FLAG_ORDER_LINEAR)
    # (FOLD_ON selects the folding backward in experiment builds and is ignored by the product library)
    for flag in (_lib.FLAG_ORDER_STRIP, _lib.FLAG_ORDER_TILE2D, _lib.FLAG_FOLD_ON, _lib.FLAG_FOLD_OFF, 0):
        other = run_cuda(value, shapes, lsi, loc, w, go, dtype, flags=flag)
        assert np.array_equal(other[0], linear[0]) and np.array_equal(other[2], linear[2]) and np.array_equal(other[3], linear[3])
        assert_close(other[1], linear[1], 1e-5 if dtype == torch.float32 else 1e-2, 1e-6, f"grad_value (order flag {flag})")
    if dtype == torch.float32:
        ref = msda_c.forward(value.numpy(), shapes.numpy(), lsi.numpy(), loc.numpy(), w.numpy(), np.float64)
        assert_close(linear[0], ref, 1e-5, 1e-6, "out vs oracle")


def test_tile2d_order_on_a_pathological_pyramid():
    """1-pixel-wide levels make the tile count exceed the launch bound derived from S: the kernels'
    grid-stride step (TILE2D order and the folding backward) must still cover every query."""
    _, _lib, _, workloads, _, _ = _mods()
    levels = [(300, 1), (1, 200), (64, 1), (1, 1)]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 1, 0, 2, 32, 4, "encoder", "model", 3)
    go = torch.randn(1, value.shape[1], 64, generator=torch.Generator().manual_seed(1))
    b = run_cuda(value, shapes, lsi, loc, w, go, flags=_lib.FLAG_ORDER_LINEAR)
    for flag in (_lib.FLAG_ORDER_TILE2D, _lib.FLAG_FOLD_ON):
        a = run_cuda(value, shapes, lsi, loc, w, go, flags=flag)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3])
        assert_close(a[1], b[1], 1e-5, 1e-6, "grad_value")


# ------------------------------------------------------------------------------------------------
# backward: on-SM folding of grad_value (csrc/msda_fold.cuh), encoder form
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("D,L,P,dist", [(32, 4, 4, "model"), (32, 4, 4, "edge"), (32, 4, 4, "test"), (64, 3, 4, "model"),
                                        (32, 5, 8, "model"), (32, 1, 5, "edge"), (64, 4, 6, "test"), (32, 8, 4, "model"),
                                        (32, 16, 4, "edge")])
def test_folding_backward_against_oracle(D, L, P, dist, dtype):
    """grad_value pre-added on the SM == the one-red-per-corner path == the fp64 oracle; grad_loc / grad_w are
    untouched by the fold (bit-identical).  (32, 8, 4) takes the 8x8 tile with a runtime point count, (32, 5, 8)
    the 8x4 tile; (32, 16, 4) has no folding instantiation that fits shared memory and must fall back cleanly."""
    needs_experiments()
    _, _lib, _, workloads, msda_c, _ = _mods()
    levels = [(19, 27), (10, 14), (5, 7), (3, 4), (2, 2), (1, 1), (1, 2), (2, 1), (1, 1), (1, 1), (1, 1), (1, 1), (1, 1),
              (1, 1), (1, 1), (1, 1)][:L]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 2, 0, 4, D, P, "encoder", dist, 11, value_dtype=dtype)
    go = torch.randn(2, value.shape[1], 4 * D, generator=torch.Generator().manual_seed(2)).to(dtype)
    on = run_cuda(value, shapes, lsi, loc, w, go, dtype, flags=_lib.FLAG_FOLD_ON)
    off = run_cuda(value, shapes, lsi, loc, w, go, dtype, flags=_lib.FLAG_FOLD_OFF)
    a = [value.float().numpy(), shapes.numpy(), lsi.numpy(), loc.numpy(), w.numpy()]
    rgv, _, _ = msda_c.backward(go.float().numpy(), *a, np.float64)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    assert_close(on[1], rgv, tol, 1e-6, "grad_value vs oracle")
    assert_close(on[1], off[1], tol, 1e-6, "grad_value vs all-reds path")
    assert np.array_equal(on[2], off[2]) and np.array_equal(on[3], off[3])


def test_folding_backward_table_overflow():
    """Uniformly random locations on two large levels: an 8 x 8 query tile touches ~3800 distinct pixels, more than
    the 2048-slot table holds, so part of the contributions take the direct-red fallback of the filing lane."""
    needs_experiments()
    _, _lib, _, workloads, msda_c, _ = _mods()
    levels = [(64, 64), (48, 48)]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 1, 0, 2, 32, 8, "encoder", "test", 5)
    go = torch.randn(1, value.shape[1], 64, generator=torch.Generator().manual_seed(3))
    a = [t.numpy() for t in (value, shapes, lsi, loc, w)]
    rgv, rgl, rgw = msda_c.backward(go.numpy(), *a, np.float64)
    m = smooth_mask(a[3], a[1], band=1e-4)
    _, gv, gl, gw = run_cuda(*a, go, torch.float32, flags=_lib.FLAG_FOLD_ON)
    assert_close(gv, rgv, 1e-5, 1e-6, "grad_value")
    assert_close(gw, rgw, 1e-5, 1e-6, "grad_w")
    assert_close(gl * m, rgl * m, 1e-5, 1e-6, "grad_loc")


def test_folding_backward_dispatch():
    """The fold is one kernel launch; it applies to the encoder form only (Q == S) and never under an explicit row
    order, the deterministic flag or the generic flag."""
    needs_experiments()
    ir, _lib, functional, workloads, _, _ = _mods()
    h = _lib.lib()
    value, shapes, lsi, loc, w = workloads.make_inputs([(21, 37), (11, 19)], 1, 0, 4, 32, 4, "encoder", "model", 2, DEV)
    go = torch.randn(1, value.shape[1], 128, device=DEV)
    with functional.kernel_flags(_lib.FLAG_FOLD_ON):
        n0 = h.msda_kernel_launch_count()
        gv, gl, gw = ir.ms_deform_attn_backward(value, shapes, lsi, loc, w, go, 64)
        assert h.msda_kernel_launch_count() - n0 == 1
    gv0, gl0, gw0 = ir.ms_deform_attn_backward(value, shapes, lsi, loc, w, go, 64)
    torch.cuda.synchronize()
    assert torch.equal(gl, gl0) and torch.equal(gw, gw0)
    assert_close(gv.double().cpu().numpy(), gv0.double().cpu().numpy(), 1e-5, 1e-6, "grad_value")
    # CUDA-graph capture of the folding backward
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with functional.kernel_flags(_lib.FLAG_FOLD_ON), torch.cuda.stream(side):
        ir.ms_deform_attn_backward(value, shapes, lsi, loc, w, go, 64)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            cgv, cgl, cgw = ir.ms_deform_attn_backward(value, shapes, lsi, loc, w, go, 64)
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(cgl, gl0) and torch.equal(cgw, gw0)
    assert_close(cgv.double().cpu().numpy(), gv0.double().cpu().numpy(), 1e-5, 1e-6, "grad_value (graph replay)")


@pytest.mark.parametrize("dtype,D", [(torch.float32, 32), (torch.bfloat16, 32), (torch.float32, 30), (torch.float64, 32),
                                     (torch.float32, 64)])
def test_deterministic_backward_is_bit_reproducible(dtype, D):
    """MSDA_FLAG_DETERMINISTIC (cfg 5's requirement): grad_value identical bit for bit across runs --
    on a contended shape (many queries onto a tiny map) where float atomics do reorder -- and within
    tolerance of the fp64 oracle.  grad_loc / grad_w are reproducible in both modes."""
    _, _lib, _, workloads, msda_c, _ = _mods()
    levels = [(5, 7), (3, 4), (2, 2)]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 2, 4000, 4, D, 4, "decoder", "model", 21, value_dtype=dtype)
    go = torch.randn(2, 4000, 4 * D, generator=torch.Generator().manual_seed(2)).to(dtype)
    runs = [run_cuda(value, shapes, lsi, loc, w, go, dtype, flags=_lib.FLAG_DETERMINISTIC) for _ in range(3)]
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert np.array_equal(a, b)
    fast = run_cuda(value, shapes, lsi, loc, w, go, dtype)
    assert np.array_equal(fast[2], runs[0][2]) and np.array_equal(fast[3], runs[0][3])
    # the sorted segment reduction (fast shapes) and the fixed-point reds give the same bits
    atomic = run_cuda(value, shapes, lsi, loc, w, go, dtype, flags=_lib.FLAG_DETERMINISTIC | _lib.FLAG_DET_ATOMIC)
    for a, b in zip(runs[0], atomic):
        assert np.array_equal(a, b)
    v64 = value.double().numpy()
    rgv, _, _ = msda_c.backward(go.double().numpy(), v64, shapes.numpy(), lsi.numpy(), loc.numpy(), w.numpy(), np.float64)
    tol = {torch.float32: 1e-5, torch.bfloat16: 1e-2, torch.float64: 1e-9}[dtype]
    assert_close(runs[0][1], rgv, tol, 1e-6, "deterministic grad_value vs oracle")
    assert_close(fast[1], rgv, tol, 1e-6, "atomic grad_value vs oracle")


@pytest.mark.parametrize("cfg", ["enc", "dec", "dec_sparse"])
def test_deterministic_sorted_path_on_pyramids(cfg):
    """Sorted path on multi-level pyramids (encoder and decoder forms, edge locations included): bit-equal to
    the fixed-point red path, reproducible, and within tolerance of the oracle.  "enc" and "dec" are dense
    (>= 4 points per pixel and head: one-pass cell reduce), "dec_sparse" takes the per-pixel gather."""
    _, _lib, _, workloads, msda_c, _ = _mods()
    levels = [(21, 37), (11, 19), (6, 10), (3, 5)]
    kind, Q, dist = {"enc": ("encoder", 0, "model"), "dec": ("decoder", 333, "edge"),
                     "dec_sparse": ("decoder", 40, "edge")}[cfg]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 2, Q, 8, 32, 4, kind, dist, 17)
    go = torch.randn(2, loc.shape[1], 256, generator=torch.Generator().manual_seed(5))
    a = run_cuda(value, shapes, lsi, loc, w, go, flags=_lib.FLAG_DETERMINISTIC)
    b = run_cuda(value, shapes, lsi, loc, w, go, flags=_lib.FLAG_DETERMINISTIC)
    c = run_cuda(value, shapes, lsi, loc, w, go, flags=_lib.FLAG_DETERMINISTIC | _lib.FLAG_DET_ATOMIC)
    for x, y, z in zip(a, b, c):
        assert np.array_equal(x, y) and np.array_equal(x, z)
    rgv, _, _ = msda_c.backward(go.numpy(), value.numpy(), shapes.numpy(), lsi.numpy(), loc.numpy(), w.numpy(), np.float64)
    assert_close(a[1], rgv, 1e-5, 1e-6, "sorted deterministic grad_value vs oracle")


def test_deterministic_backward_scale_extremes():
    """The fixed-point scale follows max|grad_out| * max|w|: tiny and huge gradients keep ~2^-38 relative
    resolution; all-zero gradients give exact zeros."""
    _, _lib, _, workloads, msda_c, _ = _mods()
    levels = [(5, 7), (3, 4)]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 1, 50, 2, 32, 4, "decoder", "model", 5)
    go = torch.randn(1, 50, 64, generator=torch.Generator().manual_seed(2))
    base = run_cuda(value, shapes, lsi, loc, w, go, flags=_lib.FLAG_DETERMINISTIC)[1]
    for factor in (2.0 ** -60, 2.0 ** 40):
        got = run_cuda(value, shapes, lsi, loc, w, go * factor, flags=_lib.FLAG_DETERMINISTIC)[1]
        assert np.array_equal(got, base * factor)          # power-of-two scaling commutes exactly
    zero = run_cuda(value, shapes, lsi, loc, w, go * 0, flags=_lib.FLAG_DETERMINISTIC)[1]
    assert not zero.any()


def test_deterministic_cell_reduce_edge_inputs():
    """Dense deterministic path (one-pass cell reduce) on inputs built to stress its bookkeeping: almost every
    point of an image out of range (entry slices that start in the middle of a cell and runs of empty cells),
    every point in ONE cell (a cell spanning many 64-entry slices), and nothing in range at all."""
    _, _lib, _, workloads, msda_c, _ = _mods()
    levels = [(9, 13), (5, 7), (3, 4)]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 3, 700, 4, 32, 4, "decoder", "test", 29)
    loc = loc.clone()
    loc[0, 5:] = 7.5                                  # image 0: only 5 queries sample anything
    loc[1] = torch.tensor([0.31, 0.62])               # image 1: every point of every level in one cell per level
    go = torch.randn(3, 700, 128, generator=torch.Generator().manual_seed(3))
    a = run_cuda(value, shapes, lsi, loc, w, go, flags=_lib.FLAG_DETERMINISTIC)
    b = run_cuda(value, shapes, lsi, loc, w, go, flags=_lib.FLAG_DETERMINISTIC | _lib.FLAG_DET_ATOMIC)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    rgv, _, _ = msda_c.backward(go.numpy(), value.numpy(), shapes.numpy(), lsi.numpy(), loc.numpy(), w.numpy(), np.float64)
    assert_close(a[1], rgv, 1e-5, 1e-6, "cell-reduce grad_value vs oracle")
    loc[:] = -3.0                                     # nothing in range: no entries at all
    z = run_cuda(value, shapes, lsi, loc, w, go, flags=_lib.FLAG_DETERMINISTIC)
    assert not z[0].any() and not z[1].any() and not z[2].any() and not z[3].any()


def test_backward_skips_the_scatter_when_value_needs_no_grad():
    """autograd tells the Function that `value` needs no gradient (frozen memory branch): the fast path then runs the
    backward kernel with the grad_value scatter compiled out -- same grad_loc / grad_w bits, no grad for value -- and
    the generic path simply drops the gradient."""
    ir, _lib, functional, workloads, _, _ = _mods()
    for D in (32, 30):                                   # fast kernels / generic kernels
        value, shapes, lsi, loc, w = workloads.make_inputs([(9, 13), (5, 7)], 2, 60, 4, D, 4, "decoder", "model", 8)
        go = torch.randn(2, 60, 4 * D, generator=torch.Generator().manual_seed(1)).to(DEV)
        shapes, lsi = shapes.to(DEV), lsi.to(DEV)
        res = {}
        for need in (True, False):
            v = value.to(DEV).requires_grad_(need)
            lo, ww = loc.to(DEV).requires_grad_(True), w.to(DEV).requires_grad_(True)
            out = ir.MultiScaleDeformableAttnFunction.apply(v, shapes, lsi, lo, ww, 64)
            before = _lib.launch_count()
            out.backward(go)
            res[need] = (v.grad, lo.grad.clone(), ww.grad.clone(), _lib.launch_count() - before)
        assert res[True][0] is not None and res[False][0] is None
        assert torch.equal(res[True][1], res[False][1]) and torch.equal(res[True][2], res[False][2])
        assert res[False][3] >= 1                        # the CUDA kernels ran in both cases



# ------------------------------------------------------------------------------------------------
# bookkeeping: bit-exact
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [32, 16, 128, 30])
@pytest.mark.parametrize("dist", ["model", "test", "edge"])
def test_bookkeeping_bit_exact(dist, D):
    """Sampling / index bookkeeping bit-exact (north_star).  For D in {16, 32, 128} the subject is the FAST kernels'
    own per-point record (msda::make_record -- clamped low-corner offset, alias and validity flags), decoded into the
    four corner offsets exactly as their gather / scatter loops decode it; for D = 30 it is the generic kernels'
    coordinate code.  Compared with
      (1) the oracle's EXACT cell (float64 evaluation of loc*size - 0.5, msda_oracle_bookkeeping(is_f32=0)): the
          integers must be identical and the fraction must be the float64 fraction correctly rounded to float32
          (<= 1 ulp) -- independent of how the kernel gets there;
      (2) the oracle's float restatement of the kernel's compensated arithmetic: identical bits."""
    _, _, functional, workloads, msda_c, _ = _mods()
    levels = [(25, 42), (13, 21), (7, 11), (4, 6)]
    value, shapes, lsi, loc, w = workloads.make_inputs(levels, 2, 300, 8, D, 4, "decoder", dist, 11)
    B, S, H, _ = value.shape
    offs, frac = functional.debug_bookkeeping(loc.to(DEV), shapes.to(DEV), lsi.to(DEV), S, D)
    offs, frac = offs.cpu().numpy(), frac.cpu().numpy()
    exact_offs, exact_frac = msda_c.bookkeeping(loc.numpy(), shapes.numpy(), lsi.numpy(), B, S, H, D, False)
    assert np.array_equal(offs, exact_offs)               # the exact (fp64) cell of every point, every corner
    live = (exact_offs >= 0).any(1)
    ulp = np.spacing(np.maximum(np.abs(exact_frac), np.float32(2.0 ** -24)).astype(np.float32))
    # a fraction that rounds up to 1.0 is the same sample as (cell + 1, 0): excluded from the ulp check only
    same_cell = np.abs(frac.astype(np.float64) - exact_frac.astype(np.float64)) < 0.5
    assert (np.abs(frac.astype(np.float64) - exact_frac.astype(np.float64))[live[:, None] & same_cell] <=
            ulp[live[:, None] & same_cell]).all()
    ref_offs, ref_frac = msda_c.bookkeeping(loc.numpy(), shapes.numpy(), lsi.numpy(), B, S, H, D, True,
                                            msda_c.COORD_COMPENSATED)
    assert np.array_equal(offs, ref_offs)
    assert np.array_equal(frac.view(np.uint32), ref_frac.view(np.uint32))   # bit for bit


# ------------------------------------------------------------------------------------------------
# against the reference at the BASELINE shapes
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg,batch,dist", [("cfg1", 2, "model"), ("cfg1", 2, "edge"), ("cfg2", 2, "model"),
                                            ("cfg2", 1, "test"), ("cfg3_f32", 8, "model"), ("cfg4", 2, "model"),
                                            ("cfg5", 1, "model")])
def test_against_reference_at_baseline_shapes(cfg, batch, dist):
    """Whole-tensor comparison at the BASELINE shapes, including the full encoder shape the CPU oracle cannot reach
    within a test.  Stored data (tests/golden/full_size_golden.npz, oracle/make_golden_full_size.py) holds the
    float64 result of the reference kernels' arithmetic at a fixed sample of elements, and what the reference
    kernels' float32 arithmetic costs against it over the whole tensor; the reference's own formulation
    (oracle/msda_torch.py) is evaluated live in float64 on the same GPU for the whole-tensor check."""
    from oracle import make_golden_full_size as fsg
    _, _, _, workloads, _, msda_torch = _mods()
    stored = fsg.load(cfg, dist, batch)
    value, shapes, lsi, loc, w, go = [t.to(DEV) for t in fsg.make_case_inputs(cfg, dist, batch)]
    fsg.check_inputs(stored, value, loc)
    wl = workloads.WORKLOADS[cfg]
    flags = _mods()[1].FLAG_DETERMINISTIC if wl.deterministic else 0      # cfg 5 asks for the deterministic backward
    out, gv, gl, gw = run_cuda(value, shapes, lsi, loc, w, go, flags=flags)
    if wl.deterministic:
        again = run_cuda(value, shapes, lsi, loc, w, go, flags=flags)
        assert all(np.array_equal(a, b) for a, b in zip((out, gv, gl, gw), again))
    f = lambda t: t.double().cpu().numpy()
    # live yardstick over the whole tensor: the reference formulation in float64 on the same float32 inputs
    truth = [f(t) for t in msda_torch.forward_backward_f64(value, shapes, loc, w, go)]
    m = smooth_mask(loc.cpu().numpy(), shapes.cpu().numpy(), band=1e-4)
    for got, tru, mk, name in zip((out, gv, gl, gw), truth, [1.0, 1.0, m, 1.0], fsg.TENSORS):
        got = got * mk
        assert_close(got, tru * mk, 1e-5, 1e-6, f"{name} vs the reference formulation (fp64)")
        # the stored float64 reference result at its sample of elements
        want = stored[f"{name}/sample"]
        worst = np.abs(fsg.sampled(torch.from_numpy(got)) - want).max()
        assert worst <= 1e-5 * stored[f"{name}/absmax"] + 1e-6, (name, worst)
        # at least as accurate as the reference kernels' float32 arithmetic
        mine = np.abs(got - tru * mk).max()
        theirs = float(stored[f"{name}/err32"])
        assert mine <= 1.5 * theirs + 1e-6 * max(1.0, float(stored[f"{name}/absmax"])), (name, mine, theirs)


# ------------------------------------------------------------------------------------------------
# BASELINE configs: cfg1 at full size against the torch port in fp64; big ones through properties
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dist", ["model", "test", "edge"])
def test_cfg1_full_size_against_fp64_port(dist):
    _, _, _, workloads, _, msda_torch = _mods()
    wl = workloads.WORKLOADS["cfg1"]
    value, shapes, lsi, loc, w = workloads.make_workload_inputs(wl, dist, 2)
    go = torch.randn(wl.batch, wl.queries, 256, generator=torch.Generator().manual_seed(3))
    r_out, r_gv, r_gl, r_gw = [t.numpy() for t in msda_torch.forward_backward_f64(value, shapes, loc, w, go)]
    out, gv, gl, gw = run_cuda(value, shapes, lsi, loc, w, go)
    m = smooth_mask(loc.numpy(), shapes.numpy(), band=1e-4)
    assert_close(out, r_out, 1e-5, 1e-6, "out")
    assert_close(gv, r_gv, 1e-5, 1e-6, "grad_value")
    assert_close(gw, r_gw, 1e-5, 1e-6, "grad_w")
    assert_close(gl * m, r_gl * m, 1e-5, 1e-6, "grad_loc")


@pytest.mark.parametrize("cfg", ["cfg2", "cfg3", "cfg5"])
def test_full_size_properties(cfg):
    """Size-independent properties at BASELINE.json's full sizes (the oracle cannot run these):
    (1) constant value => out = sum of in-range bilinear mass per row, grad_loc = 0 inside;
    (2) linearity in value; (3) <out, go> == <value, grad_value> (adjoint identity, the
    'checksum of checksums' of a linear gather/scatter pair); (4) a sampled sub-block of rows
    agrees with the C oracle."""
    ir, _, _, workloads, msda_c, _ = _mods()
    wl = workloads.WORKLOADS[cfg]
    B = 2 if cfg != "cfg3" else wl.batch
    value, shapes, lsi, loc, w = workloads.make_workload_inputs(wl, "model", 1, DEV, batch=B)
    vdt = value.dtype
    Q = wl.queries
    gen = torch.Generator(device=DEV).manual_seed(9)
    go = torch.randn(B, Q, wl.num_heads * wl.head_dim, device=DEV, generator=gen).to(vdt)
    fn = ir.MultiScaleDeformableAttnFunction.apply

    v = value.clone().requires_grad_(True)
    out = fn(v, shapes, lsi, loc, w, 64)
    out.backward(go)
    # (3) adjoint identity in fp64 accumulation
    lhs = (out.double() * go.double()).sum().item()
    rhs = (value.double() * v.grad.double()).sum().item()
    tol = 2e-2 if vdt == torch.bfloat16 else 1e-4
    assert abs(lhs - rhs) <= tol * max(abs(lhs), abs(rhs), 1.0), (lhs, rhs)
    # (2) linearity: f(2v) == 2 f(v) exactly (power-of-two scaling commutes with rounding)
    out2 = fn((value * 2), shapes, lsi, loc, w, 64)
    assert torch.equal(out2, out.detach() * 2)
    # (1) constant value
    ones = torch.ones_like(value)
    lo = loc.clone().requires_grad_(True)
    o1 = fn(ones, shapes, lsi, lo, w, 64)
    assert float(o1.detach().float().max()) <= 1.0 + 1e-2 and float(o1.detach().float().min()) >= -1e-6
    # (4) sampled rows vs the C oracle (fp64) -- first 3 queries of image 0 and last 3 of image B-1
    for b, q0 in ((0, 0), (B - 1, Q - 3)):
        sl = slice(q0, q0 + 3)
        ref = msda_c.forward(value[b:b + 1].float().cpu().numpy(), shapes.cpu().numpy(), lsi.cpu().numpy(),
                             loc[b:b + 1, sl].cpu().numpy(), w[b:b + 1, sl].cpu().numpy(), np.float64)
        got = out[b:b + 1, sl].detach().double().cpu().numpy()
        rt = 1e-2 if vdt == torch.bfloat16 else 1e-5
        assert_close(got, ref, rt, 1e-6, f"{cfg} rows b={b}")


@pytest.mark.parametrize("seed", list(range(24)))
def test_random_problem_shapes_against_oracle(seed):
    """Seeded fuzz over (levels, B, Q, H, D, P, dtype, distribution, flags): forward and all three gradients against the
    fp64 C oracle, through whichever kernels the shape dispatches to (fast, generic, every row order, the folding
    backward, the deterministic paths: fixed-point reds, per-pixel gather, cell reduce)."""
    _, _lib, _, workloads, msda_c, _ = _mods()
    rng = np.random.default_rng(1000 + seed)
    L = int(rng.integers(1, 6))
    levels, h, w = [], int(rng.integers(3, 40)), int(rng.integers(3, 40))
    for _ in range(L):
        levels.append((h, w))
        h, w = max(1, (h + 1) // 2), max(1, (w + 1) // 2)
    B, H = int(rng.integers(1, 4)), int(rng.choice([1, 2, 4, 8]))
    D = int(rng.choice([16, 32, 64, 128, 8, 24, 40]))
    P = int(rng.integers(1, 9))
    encoder = bool(rng.integers(0, 2))
    Q = 0 if encoder else int(rng.integers(1, 200))
    dist = str(rng.choice(["model", "test", "edge"]))
    dtype = torch.bfloat16 if (rng.integers(0, 4) == 0) else torch.float32
    flag_choices = [0, _lib.FLAG_ORDER_LINEAR, _lib.FLAG_ORDER_STRIP, _lib.FLAG_FOLD_OFF, _lib.FLAG_FORCE_GENERIC,
                    _lib.FLAG_DETERMINISTIC, _lib.FLAG_DETERMINISTIC | _lib.FLAG_DET_ATOMIC,
                    _lib.FLAG_DETERMINISTIC | _lib.FLAG_FORCE_GENERIC]
    if encoder:
        flag_choices += [_lib.FLAG_FOLD_ON, _lib.FLAG_FOLD_ON, _lib.FLAG_ORDER_TILE2D]
    flags = int(rng.choice(flag_choices))
    value, shapes, lsi, loc, wgt = workloads.make_inputs(levels, B, Q, H, D, P, "encoder" if encoder else "decoder", dist,
                                                         seed, value_dtype=dtype)
    Qn = loc.shape[1]
    go = torch.randn(B, Qn, H * D, generator=torch.Generator().manual_seed(seed)).to(dtype)
    a = [value.float().numpy(), shapes.numpy(), lsi.numpy(), loc.numpy(), wgt.numpy()]
    ref_out = msda_c.forward(*a, np.float64)
    rgv, rgl, rgw = msda_c.backward(go.float().numpy(), *a, np.float64)
    m = smooth_mask(a[3], a[1], band=1e-4)
    out, gv, gl, gw = run_cuda(value, shapes, lsi, loc, wgt, go, dtype, flags=flags)
    what = f"levels={levels} B={B} Q={Qn} H={H} D={D} P={P} {dist} {dtype} flags={flags}"
    vt = 1e-5 if dtype == torch.float32 else 1e-2
    at = 1e-5 if dtype == torch.float32 else 1e-4
    assert_close(out, ref_out, vt, 1e-6, "out " + what)
    assert_close(gv, rgv, vt, 1e-6, "grad_value " + what)
    assert_close(gw, rgw, at, 1e-6, "grad_w " + what)
    assert_close(gl * m, rgl * m, at, 1e-6, "grad_loc " + what)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("D", [16, 32, 128])
@pytest.mark.parametrize("dist", ["test", "edge"])
def test_degenerate_pyramids_against_oracle(dist, D, dtype):
    """One-pixel, one-row and one-column levels: almost every bilinear cell has padded corners, low corners at -1 and
    unclamped offsets in front of / behind the level (the records' validity bits alone keep the loops inside the map)."""
    _, _, _, workloads, msda_c, _ = _mods()
    levels = [(1, 1), (1, 7), (5, 1), (2, 2)]
    value, shapes, lsi, loc, wgt = workloads.make_inputs(levels, 2, 40, 2, D, 3, "decoder", dist, 21, value_dtype=dtype)
    loc = (loc - 0.5) * 1.6 + 0.5                              # a good share outside [0, 1] on both sides
    go = torch.randn(2, 40, 2 * D, generator=torch.Generator().manual_seed(2)).to(dtype)
    a = [value.float().numpy(), shapes.numpy(), lsi.numpy(), loc.numpy(), wgt.numpy()]
    ref_out = msda_c.forward(*a, np.float64)
    rgv, rgl, rgw = msda_c.backward(go.float().numpy(), *a, np.float64)
    m = smooth_mask(a[3], a[1], band=1e-4)
    out, gv, gl, gw = run_cuda(value, shapes, lsi, loc, wgt, go, dtype)
    vt = 1e-5 if dtype == torch.float32 else 1e-2
    at = 1e-5 if dtype == torch.float32 else 1e-4
    assert_close(out, ref_out, vt, 1e-6, "out")
    assert_close(gv, rgv, vt, 1e-6, "grad_value")
    assert_close(gw, rgw, at, 1e-6, "grad_w")
    assert_close(gl * m, rgl * m, at, 1e-6, "grad_loc")


def test_pytorch_named_entry_point(golden):
    """multi_scale_deformable_attn_pytorch(value, shapes, loc, w) -- the reference's other public function
    (multi_scale_deform_attn.py:96-136) -- runs on the kernels and matches the reference-made vectors."""
    ir, *_ = _mods()
    c = golden("ref_test")
    v = torch.as_tensor(c["value"]).to(DEV, torch.float64).requires_grad_(True)
    out = ir.multi_scale_deformable_attn_pytorch(v, torch.as_tensor(c["shapes"]).to(DEV),
                                                 torch.as_tensor(c["loc"]).to(DEV, torch.float64),
                                                 torch.as_tensor(c["w"]).to(DEV, torch.float64))
    out.backward(torch.as_tensor(c["grad_out"]).to(DEV, torch.float64))
    assert np.allclose(out.detach().cpu().numpy(), c["f64/out"], rtol=1e-5, atol=1e-8)
    assert nerr(v.grad.cpu().numpy(), c["f64/grad_value"]) < 1e-12
    with pytest.raises(RuntimeError, match="CPU"):
        ir.multi_scale_deformable_attn_pytorch(torch.as_tensor(c["value"]), torch.as_tensor(c["shapes"]),
                                               torch.as_tensor(c["loc"]), torch.as_tensor(c["w"]))


# ------------------------------------------------------------------------------------------------
# edge behaviour (SURVEY appendix B)
# ------------------------------------------------------------------------------------------------
def test_empty_and_ragged_inputs():
    ir, *_ = _mods()
    shapes = torch.as_tensor([(3, 4), (1, 2)], dtype=torch.long, device=DEV)
    lsi = torch.as_tensor([0, 12], dtype=torch.long, device=DEV)
    fn = ir.MultiScaleDeformableAttnFunction.apply
    # zero queries
    out = fn(torch.randn(2, 14, 2, 16, device=DEV), shapes, lsi, torch.rand(2, 0, 2, 2, 3, 2, device=DEV),
             torch.rand(2, 0, 2, 2, 3, device=DEV), 64)
    assert out.shape == (2, 0, 32)
    # zero batch
    out = fn(torch.randn(0, 14, 2, 16, device=DEV), shapes, lsi, torch.rand(0, 5, 2, 2, 3, 2, device=DEV),
             torch.rand(0, 5, 2, 2, 3, device=DEV), 64)
    assert out.shape == (0, 5, 32)
    # zero points: empty sum -> zeros, and backward gives zero grad_value
    v = torch.randn(1, 14, 2, 16, device=DEV, requires_grad=True)
    out = fn(v, shapes, lsi, torch.rand(1, 5, 2, 2, 0, 2, device=DEV), torch.rand(1, 5, 2, 2, 0, device=DEV), 64)
    assert out.shape == (1, 5, 32) and float(out.abs().max()) == 0.0
    out.sum().backward()
    assert float(v.grad.abs().max()) == 0.0
    # a batch that the reference's im2col_step assert would reject (B=3, step=2: cu:53)
    v, s2, l2, loc, w = _mods()[3].make_inputs([(3, 4), (1, 2)], 3, 4, 2, 16, 3, "decoder", "test", 0, DEV)
    assert fn(v, s2, l2, loc, w, 2).shape == (3, 4, 32)


def test_nan_and_inf_locations_are_skipped():
    """Kernel semantics of the reference gate (cuh:288): NaN / Inf locations contribute nothing."""
    ir, _, _, workloads, *_ = _mods()
    v, shapes, lsi, loc, w = workloads.make_inputs([(5, 6), (2, 3)], 1, 4, 2, 32, 2, "decoder", "test", 3, DEV)
    base = ir.MultiScaleDeformableAttnFunction.apply(v, shapes, lsi, loc, w, 64)
    loc2, w2 = loc.clone(), w.clone()
    loc2[0, 1, 0, 0, 0, 0] = float("nan")
    loc2[0, 2, 1, 1, 1, 1] = float("inf")
    w_ref = w.clone()
    w_ref[0, 1, 0, 0, 0] = 0
    w_ref[0, 2, 1, 1, 1] = 0
    got = ir.MultiScaleDeformableAttnFunction.apply(v, shapes, lsi, loc2, w2, 64)
    want = ir.MultiScaleDeformableAttnFunction.apply(v, shapes, lsi, loc, w_ref, 64)
    assert torch.isfinite(got).all() and torch.equal(got, want) and not torch.equal(got, base)


def test_non_finite_values_outside_a_points_footprint_do_not_leak():
    """A corner that is zero padding for a point is never LOADED (the reference's per-corner bounds checks, cuh:56-80,
    skip it too), so a NaN / Inf in a pixel no point actually samples -- here the first and last pixel of every level,
    with a third of the points gated out altogether -- leaves the output and every gradient finite and bit-identical
    to the same problem with zeros in those pixels.  (Round 1 clamped padded corners onto the border pixel with weight
    0 and multiplied: 0 * NaN.)"""
    ir, _, _, workloads, *_ = _mods()
    levels = [(14, 20), (9, 12), (5, 7)]
    for dtype in (torch.float32, torch.bfloat16):
        v, shapes, lsi, loc, w = workloads.make_inputs(levels, 2, 60, 4, 32, 4, "decoder", "test", 5, DEV)
        g = torch.Generator(device=DEV).manual_seed(3)
        loc = torch.rand(loc.shape, device=DEV, generator=g) * 0.45 + 0.3          # well inside every level
        gate = torch.rand(loc.shape[:-1], device=DEV, generator=g) < 0.33
        far = torch.where(torch.rand(loc.shape, device=DEV, generator=g) < 0.5, -0.7, 1.6)
        loc = torch.where(gate[..., None], far, loc)
        v = v.to(dtype)
        poisoned = v.clone()
        start = 0
        for h, wd in levels:
            poisoned[:, start] = float("nan")
            poisoned[:, start + h * wd - 1] = float("inf")
            start += h * wd
        go = torch.randn(2, 60, 4 * 32, device=DEV, generator=g).to(dtype)
        res = []
        for val in (poisoned, v):
            vv, lo, ww = val.clone().requires_grad_(True), loc.clone().requires_grad_(True), w.clone().requires_grad_(True)
            out = ir.MultiScaleDeformableAttnFunction.apply(vv, shapes, lsi, lo, ww, 64)
            out.backward(go)
            res.append((out.detach(), vv.grad, lo.grad, ww.grad))
        for a, b in zip(res[0][:1] + res[0][2:], res[1][:1] + res[1][2:]):
            assert torch.isfinite(a).all() and torch.equal(a, b)
        assert torch.isfinite(res[0][1]).all()                 # nothing is scattered from a poisoned row either
        assert (res[0][1].float() - res[1][1].float()).abs().max() <= 1e-2 * res[1][1].float().abs().max()


def test_misaligned_tensors():
    """Rows are read and written with 128-bit accesses, so the C ABI requires 16-byte aligned pointers (include/msda.h)
    and says so instead of faulting; the Python wrappers copy a mis-aligned view (a slice of a flat buffer at an odd
    element offset) into a fresh allocation, as the reference's scalar kernels needed no alignment at all."""
    ir, _lib, functional, workloads, *_ = _mods()
    v, shapes, lsi, loc, w = workloads.make_inputs([(6, 7), (3, 4)], 2, 9, 2, 32, 2, "decoder", "test", 1, DEV)
    go = torch.randn(2, 9, 2 * 32, device=DEV)

    def off_by_one(t):
        flat = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
        view = flat[1:].view(t.shape)
        view.copy_(t)
        assert view.data_ptr() % 16 != 0 and view.is_contiguous()
        return view

    want = ir.ms_deform_attn_forward(v, shapes, lsi, loc, w, 64)
    got = ir.ms_deform_attn_forward(off_by_one(v), shapes, lsi, off_by_one(loc), off_by_one(w), 64)
    assert torch.equal(got, want)
    gw = ir.ms_deform_attn_backward(v, shapes, lsi, loc, w, go, 64)
    gg = ir.ms_deform_attn_backward(off_by_one(v), shapes, lsi, off_by_one(loc), off_by_one(w), off_by_one(go), 64)
    assert torch.equal(gg[1], gw[1]) and torch.equal(gg[2], gw[2])
    assert (gg[0] - gw[0]).abs().max() <= 1e-5 * gw[0].abs().max()
    # the C ABI itself refuses
    bad = off_by_one(v)
    out = torch.empty(2, 9, 64, device=DEV)
    B, S, H, D = v.shape
    status = _lib.lib().msda_forward(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream),
                                     ctypes.c_void_p(bad.data_ptr()), ctypes.c_void_p(shapes.data_ptr()),
                                     ctypes.c_void_p(lsi.data_ptr()), ctypes.c_void_p(loc.data_ptr()),
                                     ctypes.c_void_p(w.data_ptr()), B, S, H, D, 2, 9, 2, ctypes.c_void_p(out.data_ptr()),
                                     _lib.MSDA_F32, 0)
    assert status != 0 and b"16-byte aligned" in _lib.lib().msda_last_error_message()


def test_non_contiguous_grad_output_and_errors():
    ir, _lib, _, workloads, *_ = _mods()
    v, shapes, lsi, loc, w = workloads.make_inputs([(5, 6), (2, 3)], 2, 4, 2, 32, 2, "decoder", "test", 3, DEV)
    v.requires_grad_(True)
    out = ir.MultiScaleDeformableAttnFunction.apply(v, shapes, lsi, loc, w, 64)
    go = torch.randn(64, 4, 2, device=DEV).permute(2, 1, 0)          # non-contiguous [2,4,64]
    out.backward(go)                                                 # reference asserts here (cu:99)
    v2 = v.detach().clone().requires_grad_(True)
    ir.MultiScaleDeformableAttnFunction.apply(v2, shapes, lsi, loc, w, 64).backward(go.contiguous())
    assert torch.allclose(v.grad, v2.grad, rtol=1e-5, atol=1e-6)
    with pytest.raises(RuntimeError, match="contiguous"):
        ir.MultiScaleDeformableAttnFunction.apply(v.detach().transpose(1, 2), shapes, lsi, loc, w, 64)
    with pytest.raises(RuntimeError, match="float32"):
        ir.MultiScaleDeformableAttnFunction.apply(v.detach(), shapes, lsi, loc.double(), w.double(), 64)
    with pytest.raises(RuntimeError, match="dtype"):
        ir.MultiScaleDeformableAttnFunction.apply(v.detach().half(), shapes, lsi, loc, w, 64)


def test_kernels_actually_launch():
    ir, _lib, _, workloads, *_ = _mods()
    v, shapes, lsi, loc, w = workloads.make_inputs([(5, 6), (2, 3)], 2, 4, 2, 32, 2, "decoder", "test", 3, DEV)
    before = _lib.launch_count()
    ir.ms_deform_attn_forward(v, shapes, lsi, loc, w, 64)
    assert _lib.launch_count() == before + 1

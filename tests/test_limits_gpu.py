"""The kernels at the edges of what their dispatch admits, against float64 references.

The rest of the suite samples the middle of the supported range.  This file goes to the limits the fast kernels'
admission rule (``fast_ok``: D in {16, 32, 64, 128}, L <= 16, L*P <= 64, 32-bit element offsets inside one image) and
its neighbours draw, where 32-bit arithmetic, shared-memory sizing and level / bin tables are at their tightest:

  * 16 levels, L*P = 64 (the point-count template PT = 4, 8 and the run-time count 0), and one step past each limit
    (13 x 5, 17 x 1, 1 x 65: the generic kernels);
  * the backward's shared-memory opt-in above 48 KB (D = 16 at L*P = 64);
  * empty levels (H_l = 0 or W_l = 0) on every plain-op route, the sorted deterministic path's bin table included;
  * the 32-bit image-offset gate ``(S + 65536) * H * D < 2^31`` from both sides, with a second image that lies past
    2^31 elements.

Every case asserts which route ran (``msda_dispatch_name``, ``msda_fused_supported``, the deterministic workspace
size), so a moved gate cannot turn a fast-path case into a generic one unnoticed.  References: the float64 C oracle
(oracle/msda_oracle.c) on the inputs as rounded to the dtype under test; for the fused and packed paths its float64
composition (reference points + offsets / normaliser, softmax, oracle); for the 2^31 cases a sparse float64 bilinear
gather / scatter over the touched corners, written here with int64 indices.  Tolerances are test_parity_gpu.py's.
"""
import ctypes

import numpy as np
import pytest
import torch

from test_fp16_gpu import c_op
from test_oracle import smooth_mask
from test_packed_gpu import assert_red_close, padded_inputs, run_packed, run_padded
from test_parity_gpu import assert_close, run_cuda

pytestmark = pytest.mark.gpu

DEV = "cuda:0"

# 16 levels of mixed shapes: 1 x 1, one-row and one-column levels, and levels that do not halve down to 1 x 1
LEVELS16 = [(7, 9), (4, 5), (1, 1), (1, 6), (4, 1), (3, 3), (2, 5), (1, 1), (5, 2), (2, 2), (1, 7), (3, 1), (2, 4),
            (1, 1), (2, 3), (6, 1)]


def pyramid(L):
    if L == 1:
        return [(9, 11)]
    return (LEVELS16 + [(2, 2)])[:L]


# (L, P) the fast kernels take -- PT = 4, PT = 8, and the run-time point count at P = 64, 1 and 3 -- and one step past
# each limit, which the generic kernels take
FAST_LP = {"pt4": (16, 4), "pt8": (8, 8), "pt0": (1, 64), "pt0_p1": (16, 1), "pt0_p3": (16, 3)}
GENERIC_LP = {"lp65": (13, 5), "l17": (17, 1), "p65": (1, 65)}
PT_CLASS = {"pt4": ["pt4"], "pt8": ["pt8"], "pt0": ["pt0", "pt0_p1", "pt0_p3"]}
DI = {16: 0, 32: 1, 64: 2, 128: 3}   # spreads the cases of a parametrize grid over the (L, P) of a class
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


def _lib():
    from ir_ads_b200 import _lib
    return _lib


def route(D, L, P, S, H, dtype, flags=0, backward=1):
    from ir_ads_b200 import functional
    return _lib().lib().msda_dispatch_name(D, L, P, S, H, functional._VALUE_TAG[dtype], flags, backward).decode()


def tolerances(dtype):
    """(values and grad_value, float32 gradients): test_parity_gpu.py's bounds"""
    return (1e-5, 1e-5) if dtype == torch.float32 else (1e-2, 1e-4)


def plain(value, shapes, lsi, loc, w, go, flags=0):
    """(out, grad_value, grad_loc, grad_w) as float64 numpy: the public op for float32 / bfloat16, the C ABI for float16
    (the public op refuses float16, as the reference's does)."""
    if value.dtype == torch.float16:
        r = c_op(*(t.to(DEV) for t in (value, shapes, lsi, loc, w, go)), flags=flags)
        torch.cuda.synchronize()
        return [t.detach().double().cpu().numpy() for t in r]
    return run_cuda(value, shapes, lsi, loc, w, go, value.dtype, flags)


def oracle64(value, shapes, lsi, loc, w, go):
    from oracle import msda_c
    a = [value.double().numpy(), shapes.numpy(), lsi.numpy(), loc.numpy(), w.numpy()]
    out = msda_c.forward(*a, np.float64)
    return [out] + list(msda_c.backward(go.double().numpy(), *a, np.float64))


def check_plain(got, ref, loc, shapes, dtype, what):
    vt, at = tolerances(dtype)
    m = smooth_mask(loc.numpy(), shapes.numpy(), band=1e-4)
    assert_close(got[0], ref[0], vt, 1e-6, "out " + what)
    assert_close(got[1], ref[1], vt, 1e-6, "grad_value " + what)
    assert_close(got[3], ref[3], at, 1e-6, "grad_w " + what)
    assert_close(got[2] * m, ref[2] * m, at, 1e-6, "grad_loc " + what)


def plain_inputs(levels, B, Q, H, D, P, dtype, seed, kind="decoder"):
    from ir_ads_b200.workloads import make_inputs
    value, shapes, lsi, loc, w = make_inputs(levels, B, Q, H, D, P, kind, "edge", seed, value_dtype=dtype)
    go = torch.randn(B, loc.shape[1], H * D, generator=torch.Generator().manual_seed(seed + 1)).to(dtype)
    return value, shapes, lsi, loc, w, go


# ------------------------------------------------------------------------------------------------
# a. levels and points: plain op, forward and backward
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lp", list(FAST_LP))
@pytest.mark.parametrize("D", [16, 32, 64, 128])
@pytest.mark.parametrize("dt", list(DTYPES))
def test_plain_op_at_level_and_point_limits(dt, D, lp):
    """Forward and backward on the fast kernels at L = 16 / L*P = 64 against the oracle; the float32 cases also take
    the generic kernels (FORCE_GENERIC) as a cross-check and the scatter-free backward of a value that needs no
    gradient (same grad_loc / grad_w bits)."""
    dtype, (L, P) = DTYPES[dt], FAST_LP[lp]
    levels = pyramid(L)
    value, shapes, lsi, loc, w, go = plain_inputs(levels, 2, 23, 2, D, P, dtype, seed=D + L * P)
    S = value.shape[1]
    name = route(D, L, P, S, 2, dtype)
    assert "_fast_" in name and route(D, L, P, S, 2, dtype, backward=0).startswith("fwd_fast_"), name
    what = f"{levels} D={D} P={P} {dt}"
    got = plain(value, shapes, lsi, loc, w, go)
    ref = oracle64(value, shapes, lsi, loc, w, go)
    check_plain(got, ref, loc, shapes, dtype, what)
    if dtype == torch.float32:
        flags = _lib().FLAG_FORCE_GENERIC
        assert "_generic_" in route(D, L, P, S, 2, dtype, flags)
        check_plain(plain(value, shapes, lsi, loc, w, go, flags), ref, loc, shapes, dtype, "generic " + what)
    # the scatter-free backward (value needs no gradient): float32 / bfloat16 through the Function's backward route,
    # float16 through the C ABI flag
    from ir_ads_b200 import functional
    if dtype == torch.float16:
        B, _, H, _ = value.shape
        Q = loc.shape[1]
        gl, gw = torch.empty(loc.shape, device=DEV), torch.empty(w.shape, device=DEV)
        p = lambda t: ctypes.c_void_p(t.data_ptr() if t is not None else 0)  # noqa: E731
        dv = [t.to(DEV) for t in (go, value, shapes, lsi, loc, w)]
        _lib().check(_lib().lib().msda_backward(
            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream), *[p(t) for t in dv], B, S, H, D, L, Q, P,
            p(None), p(gl), p(gw), p(None), 0, _lib().MSDA_F16, _lib().FLAG_NO_GRAD_VALUE), "msda_backward")
    else:
        gv, gl, gw = functional._backward(value.to(DEV), shapes.to(DEV), lsi.to(DEV), loc.to(DEV), w.to(DEV),
                                          go.to(DEV), need_grad_value=False)
        assert gv is None
    torch.cuda.synchronize()
    assert np.array_equal(gl.double().cpu().numpy(), got[2]) and np.array_equal(gw.double().cpu().numpy(), got[3])


@pytest.mark.parametrize("lp", list(GENERIC_LP))
@pytest.mark.parametrize("dt", list(DTYPES))
def test_plain_op_one_step_past_the_limits(dt, lp):
    """L*P = 65 and L = 17 leave the fast kernels: the generic ones must take them, and agree with the oracle."""
    dtype, (L, P) = DTYPES[dt], GENERIC_LP[lp]
    D = {"lp65": 32, "l17": 16, "p65": 64}[lp]
    levels = pyramid(L)
    value, shapes, lsi, loc, w, go = plain_inputs(levels, 2, 19, 2, D, P, dtype, seed=L * P)
    assert "_generic_" in route(D, L, P, value.shape[1], 2, dtype)
    got = plain(value, shapes, lsi, loc, w, go)
    check_plain(got, oracle64(value, shapes, lsi, loc, w, go), loc, shapes, dtype, f"{levels} D={D} P={P} {dt}")


def _det_cases():
    cases = []
    for form in ("dense", "sparse"):
        for D in (16, 32, 64, 128):
            for pt in PT_CLASS:
                cases.append(("f32", D, pt, form))
            for i, dt in enumerate(("bf16", "f16")):
                cases.append((dt, D, list(PT_CLASS)[(DI[D] + i) % 3], form))
    return cases


@pytest.mark.parametrize("dt,D,pt,form", _det_cases())
def test_deterministic_routes_at_level_and_point_limits(dt, D, pt, form):
    """MSDA_FLAG_DETERMINISTIC on the fast shapes: the sorted segment reduction -- the cell reduce for the encoder
    form (Q == S, dense), the per-pixel gather for few queries (sparse) -- bit-equal to the fixed-point reds
    (DET_ATOMIC) and within tolerance of the oracle."""
    dtype = DTYPES[dt]
    lp = PT_CLASS[pt][DI[D] % len(PT_CLASS[pt])]
    L, P = FAST_LP[lp]
    levels = pyramid(L)
    S = sum(h * w for h, w in levels)
    Q = 0 if form == "dense" else 3
    value, shapes, lsi, loc, w, go = plain_inputs(levels, 2, Q, 2, D, P, dtype, seed=7 * D + L,
                                                  kind="encoder" if form == "dense" else "decoder")
    n_points = loc[..., 0].numel()
    assert (n_points >= 4 * 2 * S * 2) == (form == "dense")              # kDetDenseRatio: the cell reduce or the gather
    det = _lib().FLAG_DETERMINISTIC
    assert "_fast_" in route(D, L, P, S, 2, dtype, det)                   # fast shapes: the sorted route
    a = plain(value, shapes, lsi, loc, w, go, det)
    b = plain(value, shapes, lsi, loc, w, go, det | _lib().FLAG_DET_ATOMIC)
    for x, y, name in zip(a, b, ("out", "grad_value", "grad_loc", "grad_w")):
        assert np.array_equal(x, y), name
    check_plain(a, oracle64(value, shapes, lsi, loc, w, go), loc, shapes, dtype, f"{levels} D={D} P={P} {dt} {form}")


# ------------------------------------------------------------------------------------------------
# a. levels and points: fused and packed module paths
# ------------------------------------------------------------------------------------------------
# (value dtype, offsets / logits dtype): float32 offsets with every value dtype, and the two autocast tags
FUSED_TAGS = {"f32": (torch.float32, torch.float32), "bf16": (torch.bfloat16, torch.float32),
              "f16": (torch.float16, torch.float32), "bf16_aux16": (torch.bfloat16, torch.bfloat16),
              "f16_aux16": (torch.float16, torch.float16)}


def fused_case(levels, B, Q, H, D, P, vdt, adt, ref_dim, masked, seed):
    from ir_ads_b200.workloads import level_tensors
    g = torch.Generator().manual_seed(seed)
    shapes, lsi = level_tensors(levels)
    S, L = sum(h * w for h, w in levels), len(levels)
    value = torch.randn(B, S, H, D, generator=g).to(vdt)
    off = (torch.randn(B, Q, H, L, P, 2, generator=g) * 3.0).to(adt)
    logits = (torch.randn(B, Q, H, L * P, generator=g) * 2.0).to(adt)
    ref = torch.rand(B, Q, L, ref_dim, generator=g)
    mask = (torch.rand(B, S, generator=g) < 0.2) if masked else None
    go = torch.randn(B, Q, H * D, generator=g).to(vdt)
    return value, shapes, lsi, off, logits, ref, mask, go


def fused_reference(value, shapes, lsi, off, logits, ref, mask, go):
    """The module's composition in float64 on the rounded inputs (multi_scale_deform_attn.py:291-332): masked value,
    softmax over L*P, reference points + offsets / normaliser (ref_dim 2) or + offsets / P * wh / 2 (ref_dim 4), then
    the oracle; the offset / logit gradients by the chain rule.  (out, grad_value, grad_off, grad_logits, loc)."""
    B, Q, H, L, P, _ = off.shape
    v = value.double()
    if mask is not None:
        v = v.masked_fill(mask[..., None, None], 0)
    o, r = off.double(), ref.double()
    w = torch.softmax(logits.double(), -1).view(B, Q, H, L, P)
    norm = torch.stack([shapes[:, 1], shapes[:, 0]], -1).double()[None, None, None, :, None, :]
    if ref.shape[-1] == 2:
        loc = r[:, :, None, :, None, :] + o / norm
    else:
        loc = r[:, :, None, :, None, :2] + o / P * r[:, :, None, :, None, 2:] * 0.5
    out, gv, gl, gw = oracle64(v, shapes, lsi, loc, w, go)
    if mask is not None:
        gv[mask.numpy()] = 0
    gw = torch.from_numpy(gw).view(B, Q, H, L * P)
    wf = w.view(B, Q, H, L * P)
    g_logits = wf * (gw - (gw * wf).sum(-1, keepdim=True))
    gl = torch.from_numpy(gl)
    g_off = gl / norm if ref.shape[-1] == 2 else gl * r[:, :, None, :, None, 2:] * (0.5 / P)
    return out, gv, g_off.numpy(), g_logits.numpy(), loc.numpy()


def check_fused(got, want, shapes, vdt, adt, what):
    vt, at = tolerances(vdt)
    if adt != torch.float32:
        at = 1e-2                       # offset / logit gradients rounded to the 16-bit type
    f = lambda t: t.detach().double().cpu().numpy()  # noqa: E731
    m = smooth_mask(want[4], shapes.numpy(), band=1e-4)
    assert_close(f(got[0]), want[0], vt, 1e-6, "out " + what)
    assert_close(f(got[1]), want[1], vt, 1e-6, "grad_value " + what)
    assert_close(f(got[2]) * m, want[2] * m, at, 1e-6, "grad_offsets " + what)
    assert_close(f(got[3]), want[3], at, 1e-6, "grad_logits " + what)


def test_fused_supported_at_the_point_limit():
    """The fused kernels take L*P = 64 and refuse 65 (the module then composes the pre-ops around the plain op)."""
    h = _lib().lib()
    for tag in (_lib().MSDA_F32, _lib().MSDA_BF16, _lib().MSDA_F16, _lib().MSDA_BF16_AUX16, _lib().MSDA_F16_AUX16):
        for D in (16, 32, 64, 128):
            for (L, P), ok in (((16, 4), 1), ((8, 8), 1), ((1, 64), 1), ((13, 5), 0), ((1, 65), 0), ((17, 1), 0)):
                assert h.msda_fused_supported(D, L, P, 100, 2, tag, 0) == ok, (tag, D, L, P)


@pytest.mark.parametrize("pt", list(PT_CLASS))
@pytest.mark.parametrize("D", [16, 32, 64, 128])
@pytest.mark.parametrize("tag", list(FUSED_TAGS))
def test_fused_function_at_level_and_point_limits(tag, D, pt):
    """MSDeformAttnFusedFunction (softmax and location affine inside the kernels), forward and backward, against its
    float64 composition; ref_dim 2 / 4 and the padding mask alternate over the cases."""
    from ir_ads_b200.functional import MSDeformAttnFusedFunction, _aux_tag
    vdt, adt = FUSED_TAGS[tag]
    lp = PT_CLASS[pt][DI[D] % len(PT_CLASS[pt])]
    L, P = FAST_LP[lp]
    i = list(FUSED_TAGS).index(tag) + DI[D] + list(PT_CLASS).index(pt)
    ref_dim, masked = (2, 4)[i % 2], bool((i // 2) % 2)
    levels = pyramid(L)
    case = fused_case(levels, 2, 21, 2, D, P, vdt, adt, ref_dim, masked, seed=D + L + P + ref_dim)
    value, shapes, lsi, off, logits, ref, mask, go = case
    S = value.shape[1]
    assert _lib().lib().msda_fused_supported(D, L, P, S, 2, _aux_tag(vdt, adt, "offsets"), 0) == 1
    assert "_fast_" in route(D, L, P, S, 2, vdt)
    leaves = [t.to(DEV).requires_grad_(True) for t in (value, off, logits)]
    dev = lambda t: None if t is None else t.to(DEV)  # noqa: E731
    out = MSDeformAttnFusedFunction.apply(leaves[0], dev(shapes), dev(lsi), leaves[1], leaves[2], dev(ref), dev(mask))
    out.backward(go.to(DEV))
    torch.cuda.synchronize()
    assert out.dtype == vdt and leaves[1].grad.dtype == adt
    check_fused([out] + [t.grad for t in leaves], fused_reference(*case), shapes, vdt, adt,
                f"{levels} D={D} P={P} {tag} ref_dim={ref_dim} masked={masked}")


@pytest.mark.parametrize("lp", list(FAST_LP))
@pytest.mark.parametrize("tag", list(FUSED_TAGS))
def test_packed_at_level_and_point_limits(tag, lp):
    """MSDeformAttnPackedFunction on 16-level pyramids and L*P = 64: the padded fused path's bits (output, offset and
    logit gradients; grad_value up to the red order), and the float64 composition on the padded layout."""
    from ir_ads_b200.packing import PackedLevels, unpack_tokens
    vdt, adt = FUSED_TAGS[tag]
    L, P = FAST_LP[lp]
    D = (16, 32, 64, 128)[(list(FUSED_TAGS).index(tag) + list(FAST_LP).index(lp)) % 4]
    ref_dim = 2 + 2 * (list(FAST_LP).index(lp) % 2)
    shapes = pyramid(L)
    ext = [shapes[:], [(1, 1)] * L, [(max(1, h * 2 // 3), max(1, w // 2)) for h, w in shapes]]
    packing = PackedLevels(ext, shapes, DEV)
    gen = torch.Generator().manual_seed(D + L * P)
    packed, padded, go = padded_inputs(packing, 2, D, P, ref_dim, vdt, adt, gen)
    out, g = run_packed(packed, go, packing)
    ref_out, rg = run_padded(padded, go, packing)
    assert torch.equal(out, ref_out)
    assert torch.equal(g[1], rg[1]) and torch.equal(g[2], rg[2])
    assert_red_close(g[0], rg[0], vdt)
    # float64 composition on the padded layout, read back at the packed rows
    B, Qp = packing.batch, packing.query_pad
    go_pad = unpack_tokens(go, packing, queries=True)[0].view(B, Qp, 2 * D)
    cpu = [t.detach().cpu() for t in (*padded, go_pad)]
    want = fused_reference(cpu[0], packing.spatial_shapes.cpu(), packing.level_start_index.cpu(), cpu[1], cpu[2],
                           cpu[3], packing.padding_mask.cpu(), cpu[4])
    qi, vi = packing.query_index.cpu().numpy(), packing.value_index.cpu().numpy()
    rows = lambda a, idx: a.reshape((-1,) + a.shape[2:])[idx]  # noqa: E731
    want = [rows(want[0], qi), rows(want[1], vi), rows(want[2], qi), rows(want[3], qi), rows(want[4], qi)]
    m = smooth_mask(want[4][:, None], np.asarray(shapes), band=1e-4)[:, 0]
    vt, at = tolerances(vdt)
    at = 1e-2 if adt != torch.float32 else at
    f = lambda t: t.detach().double().cpu().numpy()  # noqa: E731
    assert_close(f(out), want[0], vt, 1e-6, "packed out")
    assert_close(f(g[0]), want[1], vt, 1e-6, "packed grad_value")
    assert_close(f(g[1]) * m, want[2] * m, at, 1e-6, "packed grad_offsets")
    assert_close(f(g[2]), want[3], at, 1e-6, "packed grad_logits")


# ------------------------------------------------------------------------------------------------
# b. empty levels
# ------------------------------------------------------------------------------------------------
# Each pyramid has sum_l (H_l - 1)(W_l - 1) < 0: counting (H_l + 1)(W_l + 1) bins for the empty level would overrun the
# deterministic workspace's B*H*(2S + 2L) bins.
EMPTY_PYRAMIDS = {"first": [(0, 100), (2, 2)], "three": [(3, 0), (1, 1), (0, 5)],
                  "middle": [(9, 11), (5, 6), (0, 200), (3, 3), (2, 2)]}


def empty_level_inputs(levels, B, Q, H, D, P, dtype, seed):
    from ir_ads_b200.workloads import level_tensors
    g = torch.Generator().manual_seed(seed)
    shapes, lsi = level_tensors(levels)
    S, L = sum(h * w for h, w in levels), len(levels)
    Q = Q or S
    value = torch.randn(B, S, H, D, generator=g).to(dtype)
    loc = torch.rand(B, Q, H, L, P, 2, generator=g) * 1.4 - 0.2
    w = torch.softmax(torch.randn(B, Q, H, L * P, generator=g), -1).view(B, Q, H, L, P)
    go = torch.randn(B, Q, H * D, generator=g).to(dtype)
    return value, shapes, lsi, loc.contiguous(), w.contiguous(), go


@pytest.mark.parametrize("form", ["dense", "sparse"])
@pytest.mark.parametrize("dt,D", [("f32", 32), ("bf16", 16)])
@pytest.mark.parametrize("pyr", list(EMPTY_PYRAMIDS))
def test_empty_levels_on_every_route(pyr, dt, D, form):
    """A level of size 0 x W or H x 0 holds no pixel: its points sample zeros and get zero gradients.  Fast, generic,
    both sorted deterministic reductions (cell reduce: encoder form; gather: few queries), the fixed-point reds and the
    scatter-free backward against the oracle, and the sorted routes bit-equal to DET_ATOMIC."""
    from ir_ads_b200 import functional
    dtype = DTYPES[dt]
    levels = EMPTY_PYRAMIDS[pyr]
    S, L = sum(h * w for h, w in levels), len(levels)
    assert sum((h - 1) * (w - 1) for h, w in levels) < 0
    P, Q = (4, 0) if form == "dense" else (1, 1)
    value, shapes, lsi, loc, w, go = empty_level_inputs(levels, 2, Q, 2, D, P, dtype, seed=S + L + D)
    assert (loc[..., 0].numel() >= 4 * 2 * S * 2) == (form == "dense")
    what = f"{levels} {dt} D={D} {form}"
    ref = oracle64(value, shapes, lsi, loc, w, go)
    lib = _lib()
    assert "_fast_" in route(D, L, P, S, 2, dtype)
    fast = plain(value, shapes, lsi, loc, w, go)
    check_plain(fast, ref, loc, shapes, dtype, "fast " + what)
    check_plain(plain(value, shapes, lsi, loc, w, go, lib.FLAG_FORCE_GENERIC), ref, loc, shapes, dtype, "generic " + what)
    sorted_ = plain(value, shapes, lsi, loc, w, go, lib.FLAG_DETERMINISTIC)
    atomic = plain(value, shapes, lsi, loc, w, go, lib.FLAG_DETERMINISTIC | lib.FLAG_DET_ATOMIC)
    for x, y, name in zip(sorted_, atomic, ("out", "grad_value", "grad_loc", "grad_w")):
        assert np.array_equal(x, y), name
    check_plain(sorted_, ref, loc, shapes, dtype, "deterministic " + what)
    generic_det = plain(value, shapes, lsi, loc, w, go, lib.FLAG_DETERMINISTIC | lib.FLAG_FORCE_GENERIC)
    check_plain(generic_det, ref, loc, shapes, dtype, "generic deterministic " + what)
    gv, gl, gw = functional._backward(value.to(DEV), shapes.to(DEV), lsi.to(DEV), loc.to(DEV), w.to(DEV), go.to(DEV),
                                      need_grad_value=False)
    assert gv is None
    assert np.array_equal(gl.double().cpu().numpy(), fast[2]) and np.array_equal(gw.double().cpu().numpy(), fast[3])
    # the empty level's points: zero gradients on every route
    for l, (h, wd) in enumerate(levels):
        if h * wd == 0:
            for r in (fast, sorted_, generic_det):
                assert not r[2][:, :, :, l].any() and not r[3][:, :, :, l].any()


# ------------------------------------------------------------------------------------------------
# c. the 32-bit image-offset gate: (S + 65536) * H * D < 2^31, H = 1, D = 16, bfloat16 value, B = 2
# ------------------------------------------------------------------------------------------------
S_FAST = (1 << 27) - 65536 - 1          # (S + 65536) * 16 == 2^31 - 16: the fast kernels' last S
BIG_PYRAMIDS = {
    # a wide, tall level and a one-row filler that makes S exact
    "tall": lambda S: [(8192, 16375), (1, S - 8192 * 16375)],
    # one row spanning most of the image: W * H * D > 2^31, so the y+1 corner offset overflows int (predicated off)
    "row": lambda S: [(1, S - 64), (8, 8)],
}


F32_EXACT = 1 << 24


def f32(n):
    """A level size as the kernels scale by it: rounded to float32 (the reference does the same, cuh:284)."""
    return float(np.float32(n))


def big_points(levels, B, Q, P):
    """float32 locations [B, Q, 1, L, P, 2]: per level the first pixel, the bottom-right corner, the last column,
    the last row and the cells next to both, the same in every image (Q * P == 6).  Along an axis longer than 2^24
    pixels float32 coordinates no longer resolve single pixels, so there the points stay within the first 2^24."""
    L = len(levels)
    loc = np.zeros((B, Q, 1, L, P, 2), np.float32)
    for l, (h, w) in enumerate(levels):
        def at(cx, cy):   # the location of pixel coordinate (cx, cy) in the kernels' loc * size - 0.5 convention
            return ((cx + 0.5) / f32(w), (cy + 0.5) / f32(h))
        if w <= F32_EXACT and h <= F32_EXACT:
            pts = [(0.0, 0.0), (1.0, 1.0), (1.0, 0.3), (0.6, 1.0), at(0.25, 0.375), at(w - 1.75, h - 1.625)]
        else:
            we, he = min(w, F32_EXACT), min(h, F32_EXACT)
            pts = [(0.0, 0.0), at(we - 1.25, he - 0.5), at(we - 0.75, 0.3 * he), at(0.6 * we, he - 0.5),
                   at(0.25, 0.375), at(we - 1.75, he - 1.625)]
        loc[:, :, 0, l] = np.asarray(pts, np.float32).reshape(Q, P, 2)[None]
    return loc


def sparse_reference(value_rows, row_of, levels, lsi, S, loc, w, go):
    """float64 bilinear gather / scatter over the touched corners only, with int64 value rows.  ``value_rows[i]`` is
    the value row ``row_of[i]`` (= b*S + s).  Pixel coordinates are loc * size - 0.5 with the size rounded to float32,
    as the kernels (and the reference's) scale.  Returns out, {row: grad_value row}, grad_loc, grad_w."""
    B, Q, _, L, P, _ = loc.shape
    D = go.shape[-1]
    index = {int(r): i for i, r in enumerate(row_of)}
    out = np.zeros((B, Q, D))
    gvals = {}
    gl = np.zeros(loc.shape)
    gw = np.zeros(w.shape)
    for b in range(B):
        for q in range(Q):
            for l, (hl, wl) in enumerate(levels):
                for p in range(P):
                    cx = float(loc[b, q, 0, l, p, 0]) * f32(wl) - 0.5   # exact: a product of two float32
                    cy = float(loc[b, q, 0, l, p, 1]) * f32(hl) - 0.5
                    if not (-1 < cx < wl and -1 < cy < hl):
                        continue
                    x0, y0 = int(np.floor(cx)), int(np.floor(cy))
                    lw, lh = cx - x0, cy - y0
                    aw = float(w[b, q, 0, l, p])
                    corners = [(y0, x0, (1 - lh) * (1 - lw), -(1 - lh), -(1 - lw)),
                               (y0, x0 + 1, (1 - lh) * lw, 1 - lh, -lw),
                               (y0 + 1, x0, lh * (1 - lw), -lh, 1 - lw),
                               (y0 + 1, x0 + 1, lh * lw, lh, lw)]
                    val, dx, dy = np.zeros(D), np.zeros(D), np.zeros(D)
                    for y, x, cw, cdx, cdy in corners:
                        if 0 <= y < hl and 0 <= x < wl:
                            r = b * S + int(lsi[l]) + y * wl + x
                            v = value_rows[index[r]]
                            val += cw * v
                            dx += cdx * v
                            dy += cdy * v
                            gvals[r] = gvals.get(r, 0.0) + cw * aw * go[b, q]
                    out[b, q] += aw * val
                    gw[b, q, 0, l, p] = float(go[b, q] @ val)
                    gl[b, q, 0, l, p] = (wl * aw * (go[b, q] @ dx), hl * aw * (go[b, q] @ dy))
    return out, gvals, gl, gw


def touched_rows(levels, lsi, S, loc):
    rows = set()
    B, Q, _, L, P, _ = loc.shape
    for b in range(B):
        for l, (hl, wl) in enumerate(levels):
            for c in loc[b, :, 0, l].reshape(-1, 2):
                cx, cy = float(c[0]) * f32(wl) - 0.5, float(c[1]) * f32(hl) - 0.5
                if -1 < cx < wl and -1 < cy < hl:
                    x0, y0 = int(np.floor(cx)), int(np.floor(cy))
                    for y in (y0, y0 + 1):
                        for x in (x0, x0 + 1):
                            if 0 <= y < hl and 0 <= x < wl:
                                rows.add(b * S + int(lsi[l]) + y * wl + x)
    return np.array(sorted(rows), dtype=np.int64)


@pytest.mark.parametrize("side", ["fast", "generic"])
@pytest.mark.parametrize("pyr", list(BIG_PYRAMIDS))
def test_image_offset_gate_at_2_31(pyr, side):
    """S on both sides of (S + 65536) * H * D = 2^31 with H = 1, D = 16, a bfloat16 value (4.3 GB per image) and two
    images, so the second one ends past 2^31 elements.  Forward, default backward and deterministic backward (on the
    fast side the sparse sorted path) against a float64 gather / scatter over the touched corners; every other element
    of grad_value must be zero."""
    from ir_ads_b200 import MultiScaleDeformableAttnFunction, functional
    lib = _lib()
    S = S_FAST + (0 if side == "fast" else 1)
    B, H, D, Q, P = 2, 1, 16, 3, 2
    levels = BIG_PYRAMIDS[pyr](S)
    L = len(levels)
    assert sum(h * w for h, w in levels) == S and all(h > 0 and w > 0 for h, w in levels)
    assert ((S + 65536) * H * D < (1 << 31)) == (side == "fast")
    name = route(D, L, P, S, H, torch.bfloat16)
    assert (f"_{side}_" in name), name
    n_value = B * S * H * D
    det = lib.FLAG_DETERMINISTIC
    h = lib.lib()
    ws_default = int(h.msda_backward_workspace_bytes(B, S, H, D, L, Q, P, lib.MSDA_BF16, 0))
    ws_det = int(h.msda_backward_workspace_bytes(B, S, H, D, L, Q, P, lib.MSDA_BF16, det))
    # the sorted path's workspace is bins + entries; the fixed-point reds need 8 bytes per value element
    assert (ws_det < n_value * 8) == (side == "fast"), ws_det
    need = 56 << 30   # measured peak of these cases on a B200: 52 GiB (value, grad_value, workspace, the checks' temporaries)
    free = torch.cuda.mem_get_info()[0]
    if free < need:
        pytest.skip(f"needs {need / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")

    shapes = torch.tensor(levels, dtype=torch.int64)
    lsi = torch.cat((shapes.new_zeros(1), (shapes[:, 0] * shapes[:, 1]).cumsum(0)[:-1]))
    loc = big_points(levels, B, Q, P)
    g = torch.Generator().manual_seed(5)
    w = torch.softmax(torch.randn(B, Q, H, L * P, generator=g), -1).view(B, Q, H, L, P).numpy()
    go = torch.randn(B, Q, H * D, generator=g).bfloat16()
    rows = touched_rows(levels, lsi.numpy(), S, loc)
    assert rows.max() >= S and rows.max() * D >= (1 << 31)                # image 1 reaches past 2^31 elements
    torch.cuda.reset_peak_memory_stats()
    value = torch.zeros(B, S, H, D, dtype=torch.bfloat16, device=DEV)
    rows_dev = torch.from_numpy(rows).to(DEV)
    value.view(B * S, H * D)[rows_dev] = torch.randn(len(rows), H * D, generator=g).bfloat16().to(DEV)
    value_rows = value.view(B * S, H * D)[rows_dev].double().cpu().numpy()
    ref_out, ref_gv, ref_gl, ref_gw = sparse_reference(value_rows, rows, levels, lsi.numpy(), S, loc, w,
                                                       go.double().numpy())
    ref_gv = np.stack([ref_gv.get(int(r), np.zeros(D)) for r in rows])
    m = smooth_mask(loc, shapes.numpy(), band=1e-4)
    dev = [t.to(DEV) for t in (shapes, lsi, torch.from_numpy(loc), torch.from_numpy(w))]

    def check(out, grads, what):
        f = lambda t: t.detach().double().cpu().numpy()  # noqa: E731
        if out is not None:
            assert_close(f(out), ref_out.reshape(B, Q, H * D), 1e-2, 1e-6, "out " + what)
        gv, gl, gw = grads
        flat = gv.view(B * S, H * D)
        assert_close(f(flat[rows_dev]), ref_gv, 1e-2, 1e-6, "grad_value " + what)
        flat.index_fill_(0, rows_dev, 0)
        assert int(torch.count_nonzero(flat)) == 0, "grad_value outside the touched rows " + what
        assert_close(f(gw), ref_gw, 1e-4, 1e-6, "grad_w " + what)
        assert_close(f(gl) * m, ref_gl * m, 1e-4, 1e-6, "grad_loc " + what)

    vv = value.requires_grad_(True)
    lo, ww = dev[2].clone().requires_grad_(True), dev[3].clone().requires_grad_(True)
    out = MultiScaleDeformableAttnFunction.apply(vv, dev[0], dev[1], lo, ww, 64)
    out.backward(go.to(DEV))
    torch.cuda.synchronize()
    check(out, (vv.grad, lo.grad, ww.grad), f"{pyr} {side} default")
    vv.grad = None
    del out
    with functional.kernel_flags(det):
        grads = functional._backward(value.detach(), dev[0], dev[1], dev[2], dev[3], go.to(DEV), True)
    torch.cuda.synchronize()
    check(None, grads, f"{pyr} {side} deterministic")
    del grads
    print(f"\n[2^31 {pyr} {side}] peak device memory {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")

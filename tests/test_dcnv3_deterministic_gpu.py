"""Bit-reproducible DCNv3 backward (MSDA_FLAG_DETERMINISTIC) on the fast shapes.

grad_input is summed in 64-bit fixed point -- by the sorted segment reduction (entries filed by the DCNv3 backward,
per-pixel gather for sparse problems, cell reduce + finalize for dense ones) or by integer reds -- and converted once,
so it does not depend on arrival order.  grad_offset / grad_mask never did; they must stay the default route's bits.
Every test restores the global switches it touches.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import dcnv3_torch
from test_dcnv3 import CASES

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def _flagbits():
    from ir_ads_b200 import _lib
    return _lib.FLAG_DETERMINISTIC, _lib.FLAG_DET_ATOMIC, _lib.FLAG_DET_SEPARATE_FILL


def _out_size(H, k, stride, pad, dil):
    return (H + 2 * pad - (dil * (k - 1) + 1)) // stride + 1


def make_case(N, H, W, G, C, k=3, stride=1, pad=1, dil=1, scale=1.0, dtype=torch.float32, seed=0, contention=False,
              off_mag=1.5):
    """Inputs on the device.  contention: the offsets send every sample of a map into one of four cells (fractions kept
    away from the cell edges), so thousands of contributions meet in a few grad_input rows and float reds reorder."""
    g = torch.Generator().manual_seed(seed)
    Ho, Wo = _out_size(H, k, stride, pad, dil), _out_size(W, k, stride, pad, dil)
    K = k * k
    inp = torch.randn(N, H, W, G * C, generator=g)
    mask = torch.softmax(torch.randn(N, Ho, Wo, G, K, generator=g), -1).reshape(N, Ho, Wo, G * K)
    go = torch.randn(N, Ho, Wo, G * C, generator=g)
    if contention:
        cw, ch = (dil * (k - 1)) // 2, (dil * (k - 1)) // 2
        i = (torch.arange(K) // k).double().view(1, 1, 1, 1, K)
        j = (torch.arange(K) % k).double().view(1, 1, 1, 1, K)
        wo = torch.arange(Wo).double().view(1, 1, Wo, 1, 1)
        ho = torch.arange(Ho).double().view(1, Ho, 1, 1, 1)
        cells = torch.tensor([[2, 3], [2, 4], [W // 2, H // 2], [W - 3, H - 2]], dtype=torch.float64)
        pick = torch.randint(0, 4, (N, Ho, Wo, G, K), generator=g)
        frac = 0.1 + 0.8 * torch.rand(N, Ho, Wo, G, K, 2, generator=g, dtype=torch.float64)
        tx = cells[pick][..., 0] + frac[..., 0]
        ty = cells[pick][..., 1] + frac[..., 1]
        ox = (tx - (cw - pad + wo * stride - cw * scale)) / scale - i * dil
        oy = (ty - (ch - pad + ho * stride - ch * scale)) / scale - j * dil
        off = torch.stack([ox, oy], -1).float().reshape(N, Ho, Wo, G * K * 2)
    else:
        off = torch.randn(N, Ho, Wo, G * K * 2, generator=g) * off_mag
    args = (k, k, stride, stride, pad, pad, dil, dil, G, C, scale)
    return inp.to(DEV, dtype), off.to(DEV), mask.to(DEV), go.to(DEV, dtype), args


def bwd(inp, off, mask, go, args, flags):
    """dcnv3_backward with `flags` ORed into the call (the kernel_flags hook)."""
    from ir_ads_b200 import dcnv3_backward, functional
    with functional.kernel_flags(flags):
        r = dcnv3_backward(inp, off, mask, *args, go)
    torch.cuda.synchronize()
    return r


def assert_bits(a, b, what):
    for x, y, name in zip(a, b, ("grad_input", "grad_offset", "grad_mask")):
        assert x.dtype == y.dtype and torch.equal(x, y), (what, name, (x.double() - y.double()).abs().max().item())


# ------------------------------------------------------------------------------------------------
# 1. bit-reproducible under contention
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("C", [16, 32, 64, 128])
def test_reproducible_under_contention(C, dtype):
    DET, _, _ = _flagbits()
    case = make_case(2, 24, 40, 4 if C < 128 else 2, C, dtype=dtype, seed=C, contention=True)
    runs = [bwd(*case, DET) for _ in range(3)]
    for r in runs[1:]:
        assert_bits(runs[0], r, f"C={C} {dtype}")
    assert runs[0][0].dtype == dtype and torch.isfinite(runs[0][0].float()).all()
    assert runs[0][0].abs().max() > 0


# ------------------------------------------------------------------------------------------------
# 2. three routes, one answer
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("k,stride,pad,kind", [(3, 1, 1, "dense"), (3, 2, 1, "sparse"), (1, 1, 0, "sparse")])
def test_emit_separate_fill_and_atomic_agree(k, stride, pad, kind, dtype):
    DET, ATOMIC, SEP = _flagbits()
    N, H, W, G, C = 2, 30, 44, 4, 32
    Ho, Wo = _out_size(H, k, stride, pad, 1), _out_size(W, k, stride, pad, 1)
    assert (Ho * Wo * k * k >= 4 * H * W) == (kind == "dense")   # the cell reduce vs the per-pixel gather
    for contention in (False, True):
        case = make_case(N, H, W, G, C, k, stride, pad, dtype=dtype, seed=k + stride, contention=contention)
        emit = bwd(*case, DET)
        assert_bits(emit, bwd(*case, DET | SEP), f"separate fill {kind}")
        assert_bits(emit, bwd(*case, DET | ATOMIC), f"fixed-point reds {kind}")


# ------------------------------------------------------------------------------------------------
# 3. the other gradients are untouched
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("k,stride", [(3, 1), (3, 2), (5, 1)])
def test_offset_and_mask_gradients_equal_default_route(k, stride, dtype):
    DET, ATOMIC, SEP = _flagbits()
    case = make_case(2, 28, 36, 4, 16, k, stride, k // 2, dtype=dtype, seed=5)
    _, goff0, gm0 = bwd(*case, 0)
    for flags in (DET, DET | SEP, DET | ATOMIC):
        _, goff, gm = bwd(*case, flags)
        assert torch.equal(goff, goff0) and torch.equal(gm, gm0), flags


# ------------------------------------------------------------------------------------------------
# 4. accurate
# ------------------------------------------------------------------------------------------------
def _check_against_port(inp, off, mask, go, args, gi, what):
    want = dcnv3_torch.forward_backward(inp.double(), off.double(), mask.double(), go.double(), *args)[1]
    err = (gi.double() - want).abs().max().item()
    assert err <= 1e-5 * want.abs().max().item() + 1e-6, (what, err)


@pytest.fixture(scope="module")
def golden():
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    blob = np.load(os.path.join(root, "tests", "golden", "dcnv3_golden.npz"))

    def case(name):
        c = {k[len(name) + 1:]: blob[k] for k in blob.files if k.startswith(name + "/")}
        N, H, W, G, C, k, s, p, d = [int(x) for x in c["geom"]]
        c["args"] = (k, k, s, s, p, p, d, d, G, C, float(c["scale"][0]))
        return c

    return case


@pytest.mark.parametrize("name", CASES)
def test_golden_geometries_against_port(golden, name):
    DET, ATOMIC, _ = _flagbits()
    c = golden(name)
    t = lambda key: torch.from_numpy(c[key]).to(DEV, torch.float32)
    inp, off, mask, go = t("input"), t("offset"), t("mask"), t("grad_out")
    gi = bwd(inp, off, mask, go, c["args"], DET)[0]
    assert np.abs(gi.double().cpu().numpy() - c["grad_input"]).max() <= 1e-5 * np.abs(c["grad_input"]).max() + 1e-6
    _check_against_port(inp, off, mask, go, c["args"], gi, name)
    assert torch.equal(gi, bwd(inp, off, mask, go, c["args"], DET | ATOMIC)[0])


@pytest.mark.parametrize("stride,pad,dil,scale", [(1, 1, 1, 1.0), (2, 1, 1, 2.0), (1, 2, 2, 0.7)])
def test_reference_formulation_sets_against_port_and_default(stride, pad, dil, scale):
    """The stride / pad / dilation / scale sets of test_against_reference_dcnv3_formulation."""
    DET, _, _ = _flagbits()
    case = make_case(2, 48, 64, 8, 32, 3, stride, pad, dil, scale, seed=11, off_mag=2.0)
    gi = bwd(*case, DET)[0]
    _check_against_port(*case, gi, (stride, pad, dil, scale))
    gi0 = bwd(*case, 0)[0]
    err = (gi - gi0).abs().max().item()
    assert err <= 1e-5 * gi0.abs().max().item() + 1e-6, err


# ------------------------------------------------------------------------------------------------
# 5. 2-byte identity
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("k,stride,C", [(3, 1, 16), (3, 1, 64), (3, 2, 32), (1, 1, 128)])
def test_two_byte_equals_f32_on_widened_inputs_rounded_once(k, stride, C, dtype):
    DET, ATOMIC, _ = _flagbits()
    inp, off, mask, go, args = make_case(2, 20, 28, 2, C, k, stride, k // 2, dtype=dtype, seed=C + k)
    for flags in (DET, DET | ATOMIC):
        gi16, goff16, gm16 = bwd(inp, off, mask, go, args, flags)
        gi32, goff32, gm32 = bwd(inp.float(), off, mask, go.float(), args, flags)
        assert torch.equal(gi16, gi32.to(dtype)), flags
        assert torch.equal(goff16, goff32) and torch.equal(gm16, gm32), flags


# ------------------------------------------------------------------------------------------------
# 6. scale extremes, zero grad_output, every sample outside the map
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,stride", [(3, 1), (3, 2)])
def test_power_of_two_scaling_is_exact(k, stride):
    DET, ATOMIC, _ = _flagbits()
    inp, off, mask, go, args = make_case(2, 24, 32, 4, 32, k, stride, 1, seed=3)
    for flags in (DET, DET | ATOMIC):
        base = bwd(inp, off, mask, go, args, flags)[0]
        for e in (-60, 40):
            f = 2.0 ** e
            got = bwd(inp, off, mask, go * f, args, flags)[0]
            assert torch.equal(got, base * f), (flags, e)


def _c_backward(inp, off, mask, go, args, flags):
    """msda_dcnv3_backward through the C ABI with a workspace the caller keeps: (grad_input, grad_offset, grad_mask,
    workspace)."""
    from ir_ads_b200 import _lib
    from ir_ads_b200.dcnv3 import _DCN_TAG, _declare
    h = _declare(_lib.lib())
    k, _, s, _, p, _, d, _, G, C, scale = args
    N, H, W, _ = inp.shape
    _, Ho, Wo, _ = off.shape
    tag = _DCN_TAG[inp.dtype]
    nbytes = h.msda_dcnv3_backward_workspace_bytes(k, k, G, C, N, H, W, Ho, Wo, tag, flags)
    ws = torch.full((nbytes,), 0x5A, dtype=torch.uint8, device=DEV)
    gi, goff, gm = torch.empty_like(inp), torch.empty_like(off), torch.empty_like(mask)
    p_ = lambda t: ctypes.c_void_p(t.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(h.msda_dcnv3_backward(st, p_(go), p_(inp), p_(off), p_(mask), k, k, s, s, p, p, d, d, G, C, scale, N, H,
                                     W, Ho, Wo, p_(gi), p_(goff), p_(gm), p_(ws), nbytes, tag, flags), "dcnv3_backward")
    # one byte less is refused before anything is launched
    assert h.msda_dcnv3_backward(st, p_(go), p_(inp), p_(off), p_(mask), k, k, s, s, p, p, d, d, G, C, scale, N, H, W, Ho,
                                 Wo, p_(gi), p_(goff), p_(gm), p_(ws), nbytes - 1, tag, flags) == 3   # MSDA_ERR_WORKSPACE
    torch.cuda.synchronize()
    return gi, goff, gm, ws


def test_zero_grad_output_and_samples_outside_the_map():
    DET, ATOMIC, _ = _flagbits()
    N, H, W, G, C = 2, 16, 20, 4, 16
    inp, off, mask, go, args = make_case(N, H, W, G, C, seed=9)
    for flags in (DET, DET | ATOMIC):
        gi, goff, gm = bwd(inp, off, mask, torch.zeros_like(go), args, flags)
        assert not gi.any() and not goff.any() and not gm.any()
    far = torch.full_like(off, -1000.0)
    for flags in (DET, DET | ATOMIC):
        gi, goff, gm = bwd(inp, far, mask, go, args, flags)
        assert not gi.any() and not goff.any() and not gm.any()
    # sorted route: the bin starts (the exclusive scan of the per-cell counts, bins + 1 ints after the 256-byte level
    # table) are all zero, i.e. no entry was filed
    gi, goff, gm, ws = _c_backward(inp, far, mask, go, args, DET)
    assert not gi.any() and not goff.any() and not gm.any()
    bins = N * G * (2 * H * W + 2)
    starts = ws[256:256 + 4 * (bins + 1)]
    assert not starts.any()
    table = ws[:24].cpu().numpy().view(np.int64)
    assert table.tolist() == [H, W, 0]


# ------------------------------------------------------------------------------------------------
# 7. switches
# ------------------------------------------------------------------------------------------------
def test_switches_give_the_same_bits_through_function_and_C():
    from ir_ads_b200 import _C, functional, set_deterministic
    from ir_ads_b200.dcnv3 import DCNv3Function
    DET, _, _ = _flagbits()
    inp, off, mask, go, args = make_case(2, 24, 32, 4, 16, seed=13, contention=True)
    want = bwd(inp, off, mask, go, args, DET)

    def through_function():
        leaves = [t.clone().requires_grad_(True) for t in (inp, off, mask)]
        DCNv3Function.apply(*leaves, *args, 256).backward(go)
        torch.cuda.synchronize()
        return [t.grad for t in leaves]

    def through_C():
        r = _C.dcnv3_backward(inp, off, mask, *args, go, 256)
        torch.cuda.synchronize()
        return r

    for switch in ("set_deterministic", "torch", "flag"):
        old_torch = torch.are_deterministic_algorithms_enabled()
        try:
            if switch == "set_deterministic":
                set_deterministic(True)
            elif switch == "torch":
                torch.use_deterministic_algorithms(True)
            with functional.kernel_flags(DET if switch == "flag" else 0):
                assert_bits(through_function(), want, switch + " / DCNv3Function")
                assert_bits(through_C(), want, switch + " / _C")
        finally:
            set_deterministic(False)
            torch.use_deterministic_algorithms(old_torch)


def test_module_twice_gives_identical_gradients():
    from ir_ads_b200 import set_deterministic
    from ir_ads_b200.dcnv3 import DCNv3
    torch.manual_seed(0)
    m = DCNv3(channels=64, group=4).to(DEV)
    with torch.no_grad():   # non-trivial offsets / masks (the reference initialises both layers to zero)
        for lin in (m.offset, m.mask):
            lin.weight.normal_(0.0, 0.2)
            lin.bias.normal_(0.0, 1.0)
    x0 = torch.randn(2, 28, 36, 64, device=DEV)
    gout = torch.randn(2, 28, 36, 64, device=DEV)
    old_cudnn = torch.backends.cudnn.deterministic
    try:
        set_deterministic(True)
        torch.backends.cudnn.deterministic = True
        grads = []
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            x = x0.clone().requires_grad_(True)
            m(x).backward(gout)
            torch.cuda.synchronize()
            grads.append([x.grad.clone()] + [p.grad.clone() for p in m.parameters()])
        for a, b in zip(*grads):
            assert torch.equal(a, b)
    finally:
        set_deterministic(False)
        torch.backends.cudnn.deterministic = old_cudnn


# ------------------------------------------------------------------------------------------------
# 8. graph capture
# ------------------------------------------------------------------------------------------------
def test_forward_backward_captured_as_one_graph():
    from ir_ads_b200 import set_deterministic
    from ir_ads_b200.dcnv3 import DCNv3Function
    inp, off, mask, go, args = make_case(2, 24, 32, 4, 32, seed=17)
    x, o, mk = (t.clone().requires_grad_(True) for t in (inp, off, mask))

    def step():
        out = DCNv3Function.apply(x, o, mk, *args, 256)
        return [out] + list(torch.autograd.grad(out, (x, o, mk), go))

    try:
        set_deterministic(True)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                step()
        torch.cuda.current_stream().wait_stream(side)
        eager = [t.detach().clone() for t in step()]
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            captured = step()
        for t in captured:
            t.zero_()
        graph.replay()
        torch.cuda.synchronize()
        for a, b in zip(captured, eager):
            assert torch.equal(a, b)
    finally:
        set_deterministic(False)


# ------------------------------------------------------------------------------------------------
# 9. realistic size: InternImage-T stage 1
# ------------------------------------------------------------------------------------------------
def test_internimage_t_stage1():
    DET, _, _ = _flagbits()
    case = make_case(16, 200, 336, 4, 16, seed=21)
    a = bwd(*case, DET)
    b = bwd(*case, DET)
    assert_bits(a, b, "stage 1")
    gi0, goff0, gm0 = bwd(*case, 0)
    assert torch.equal(a[1], goff0) and torch.equal(a[2], gm0)
    err = (a[0] - gi0).abs().max().item()
    assert err <= 1e-5 * gi0.abs().max().item() + 1e-6, err

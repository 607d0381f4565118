"""Deformable convolution (ir_ads_b200.dcnv2) on the GPU against torchvision.ops.deform_conv2d in float64 on the CPU
(detectron2's semantics: (dy, dx) offset pairs laid out [dg][K][2], mask [dg*K], zero outside the map), on inputs
widened from the dtype under test: forward and every gradient over kernel / stride / padding / dilation / groups /
deformable groups / channel counts (fast and generic kernels), with and without mask and bias, offsets that leave the
map; bfloat16 / float16 and autocast; float64 gradcheck; memory formats; reproducibility of grad_offset / grad_mask;
the deterministic switch; CUDA-graph capture; torch.compile; a DeformBottleneckBlock-style block at full size."""
import warnings

import pytest
import torch

from ir_ads_b200 import DeformConv, ModulatedDeformConv, _lib, deform_conv, kernel_flags, modulated_deform_conv
from ir_ads_b200 import set_deterministic

tv_ops = pytest.importorskip("torchvision.ops")

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")


@pytest.fixture(autouse=True)
def _fresh():
    set_deterministic(False)
    yield
    set_deterministic(False)


def out_size(n, k, s, p, d):
    return (n + 2 * p - (d * (k - 1) + 1)) // s + 1


def make(B, C, H, W, Cout, k, s=1, p=0, d=1, groups=1, dg=1, mask=True, bias=True, leave=False, dtype=torch.float32,
         seed=0):
    """Inputs in `dtype` (float32 / bfloat16 / float16 / float64); offsets ~ N(0, 2) px, with `leave` a quarter of them
    pushed a map size out."""
    kh, kw = (k, k) if isinstance(k, int) else k
    ph, pw = (p, p) if isinstance(p, int) else p
    Ho, Wo = out_size(H, kh, s, ph, d), out_size(W, kw, s, pw, d)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, C, H, W, generator=g)
    off = torch.randn(B, dg * kh * kw * 2, Ho, Wo, generator=g) * 2.0
    if leave:
        far = torch.rand(off.shape, generator=g) < 0.25
        off = torch.where(far, off + torch.sign(off) * max(H, W), off)
    if dtype in (torch.bfloat16, torch.float16):
        # 16-bit offsets are coarse: keep every sampling position off the integer grid (fraction 3/8 is exact for
        # |offset| < 32), where the bilinear sample has kinks and, at exactly -1, detectron2's gate and torchvision's
        # coordinate gradient disagree
        off = off.floor() + 0.375
    m = torch.rand(B, dg * kh * kw, Ho, Wo, generator=g) if mask else None
    w = torch.randn(Cout, C // groups, kh, kw, generator=g) / (C // groups * kh * kw) ** 0.5
    b = torch.randn(Cout, generator=g) if bias else None
    cast = (lambda t: None if t is None else t.to(dtype))
    return dict(x=cast(x), off=cast(off), m=cast(m), w=cast(w), b=cast(b), stride=s, padding=(ph, pw), dilation=d,
                groups=groups, dg=dg, out_shape=(B, Cout, Ho, Wo))


def snap(off, kernel, stride, padding, dilation):
    """float64 offsets whose sampling positions are exactly the kernels' float32 ones, fl32(base + offset): the oracle
    then picks the same bilinear cell (a float64 position a rounding away from an integer may pick the next one,
    where the offset gradient jumps -- on the 150k points of a res3 map that happens a few times)."""
    (kh, kw), (ph, pw) = kernel, padding
    B, _, Ho, Wo = off.shape
    K = kh * kw
    o = off.detach().float().cpu().view(B, -1, K, 2, Ho, Wo)
    i, j = torch.arange(K) // kw, torch.arange(K) % kw
    by = (torch.arange(Ho).view(1, 1, 1, Ho, 1) * stride - ph + (i * dilation).view(1, 1, K, 1, 1)).expand(1, 1, K, Ho, Wo)
    bx = (torch.arange(Wo).view(1, 1, 1, 1, Wo) * stride - pw + (j * dilation).view(1, 1, K, 1, 1)).expand(1, 1, K, Ho, Wo)
    y = (by.float() + o[:, :, :, 0]).double() - by.double()
    x = (bx.float() + o[:, :, :, 1]).double() - bx.double()
    return torch.stack((y, x), 3).view(off.shape)


def oracle(case, go, device="cpu"):
    """torchvision in float64 (on the CPU unless `device` says otherwise), at the kernels' float32 sampling positions:
    (out, {name: grad})."""
    t = {n: (None if case[n] is None else case[n].detach().double().to(device).requires_grad_(True))
         for n in ("x", "off", "m", "w", "b")}
    kernel = tuple(case["w"].shape[2:])
    stride = case["stride"]
    t["off"] = snap(case["off"], kernel, stride, case["padding"], case["dilation"]).to(device).requires_grad_(True)
    out = tv_ops.deform_conv2d(t["x"], t["off"], t["w"], t["b"], stride=case["stride"], padding=case["padding"],
                               dilation=case["dilation"], mask=t["m"])
    out.backward(go.double().to(device))
    return out.detach(), {n: t[n].grad for n in t if t[n] is not None}


def ours(case, go, fmt=torch.contiguous_format, step=64):
    t = {n: (None if case[n] is None else case[n].detach().to(DEV).requires_grad_(True))
         for n in ("x", "off", "m", "w", "b")}
    x = t["x"].contiguous(memory_format=fmt)
    if t["m"] is None:
        out = deform_conv(x, t["off"], t["w"], case["stride"], case["padding"], case["dilation"], case["groups"],
                          case["dg"], im2col_step=step)
    else:
        out = modulated_deform_conv(x, t["off"], t["m"], t["w"], t["b"], case["stride"], case["padding"],
                                    case["dilation"], case["groups"], case["dg"], im2col_step=step)
    out.backward(go.to(DEV, out.dtype).contiguous(memory_format=fmt))
    return out.detach(), {n: t[n].grad for n in t if t[n] is not None}


def nerr(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def check(case, tol, fmt=torch.contiguous_format, step=64):
    go = torch.randn(case["out_shape"], generator=torch.Generator().manual_seed(7)).to(case["x"].dtype)
    ref_out, ref_g = oracle(case, go)
    out, g = ours(case, go, fmt, step)
    assert out.shape == ref_out.shape
    errs = {"out": nerr(out, ref_out)}
    errs.update({n: nerr(g[n], ref_g[n]) for n in ref_g})
    assert all(e < tol for e in errs.values()), errs
    return errs


# (C, Cout, k, stride, pad, dil, groups, dg, mask, bias, H, W): channel counts per deformable group 16 .. 512 (fast
# kernels) and odd ones (generic kernels)
SWEEP = [
    (16, 16, 3, 1, 1, 1, 1, 1, True, True, 11, 13),
    (32, 24, 1, 1, 0, 1, 1, 1, True, False, 9, 10),
    (64, 32, 5, 2, 2, 1, 2, 2, True, True, 13, 12),
    (128, 32, (3, 1), 1, (1, 0), 1, 1, 1, False, False, 9, 11),
    (256, 16, 3, 2, 1, 2, 1, 1, True, True, 11, 9),
    (512, 16, 3, 1, 2, 2, 1, 1, True, False, 7, 8),
    (64, 32, 3, 1, 1, 1, 1, 4, True, True, 9, 9),
    (128, 64, 3, 2, 0, 1, 2, 4, False, False, 12, 13),
    (96, 32, 3, 1, 1, 1, 2, 2, True, True, 8, 10),       # C/groups 48, C/dg 48: D = 16
    (24, 16, 3, 1, 1, 1, 1, 2, True, True, 9, 8),        # C/dg = 12: generic
    (7, 5, 3, 1, 1, 1, 1, 1, True, True, 8, 9),          # odd channels: generic
    (30, 12, 3, 2, 2, 2, 2, 1, False, False, 12, 11),    # generic, DCNv1, groups
]


@pytest.mark.parametrize("leave", [False, True])
@pytest.mark.parametrize("cfg", SWEEP, ids=[f"C{c[0]}-k{c[2]}-s{c[3]}-g{c[6]}-dg{c[7]}" for c in SWEEP])
def test_float32_against_torchvision(cfg, leave):
    C, Cout, k, s, p, d, groups, dg, mask, bias, H, W = cfg
    case = make(2, C, H, W, Cout, k, s, p, d, groups, dg, mask, bias, leave=leave, seed=C + s)
    check(case, 5e-5)


@pytest.mark.parametrize("cfg", [SWEEP[0], SWEEP[2], SWEEP[6]], ids=["C16", "C64-g2-dg2", "C64-dg4"])
def test_generic_kernels_on_fast_shapes(cfg):
    C, Cout, k, s, p, d, groups, dg, mask, bias, H, W = cfg
    case = make(2, C, H, W, Cout, k, s, p, d, groups, dg, mask, bias, leave=True, seed=3)
    n0 = _lib.launch_count()
    with kernel_flags(_lib.FLAG_FORCE_GENERIC):
        check(case, 5e-5)
    assert _lib.launch_count() > n0


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("cfg", [SWEEP[0], SWEEP[4], SWEEP[8], SWEEP[10]], ids=["C16", "C256", "C96", "C7"])
def test_16_bit_within_1e_2(cfg, dtype):
    C, Cout, k, s, p, d, groups, dg, mask, bias, H, W = cfg
    case = make(2, C, H, W, Cout, k, s, p, d, groups, dg, mask, bias, leave=True, dtype=dtype, seed=11)
    check(dict(case, off=case["off"].float(), m=case["m"].float()), 1e-2)     # float32 offsets / mask


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_16_bit_offsets_and_mask(dtype):
    """offset / mask in the input's 16-bit type (MSDA_*_AUX16): gradients come back in that type."""
    case = make(2, 64, 10, 11, 32, 3, 1, 1, 1, 1, 2, True, True, leave=True, dtype=dtype, seed=5)
    check(case, 1e-2)
    case32 = dict(case, off=case["off"].float(), m=case["m"].float())
    _, g = ours(case32, torch.randn(2, 32, 10, 11))
    assert g["off"].dtype == torch.float32 and g["x"].dtype == dtype


def test_autocast_runs_in_the_autocast_dtype():
    case = make(2, 128, 12, 14, 64, 3, 1, 1, 1, 1, 1, True, True, seed=9)
    x = case["x"].to(DEV).requires_grad_(True)
    w = case["w"].to(DEV).requires_grad_(True)
    off, m = case["off"].to(DEV), case["m"].to(DEV)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y = modulated_deform_conv(x, off, m, w, case["b"].to(DEV), 1, 1)
    assert y.dtype == torch.bfloat16
    y.float().square().sum().backward()
    assert x.grad.dtype == torch.float32 and w.grad.dtype == torch.float32
    ref = tv_ops.deform_conv2d(case["x"].double(), case["off"].double(), case["w"].double(), case["b"].double(),
                               padding=1, mask=case["m"].double())
    assert nerr(y, ref) < 1e-2


def test_float64_gradcheck():
    case = make(1, 5, 5, 6, 3, 3, 1, 1, 1, 1, 1, True, True, seed=2)
    args = [case[n].double().to(DEV).requires_grad_(True) for n in ("x", "off", "m", "w", "b")]

    def fn(x, off, m, w, b):
        return modulated_deform_conv(x, off, m, w, b, 1, 1)

    assert torch.autograd.gradcheck(fn, args, eps=1e-6, atol=1e-5, rtol=1e-4, nondet_tol=1e-12)


def test_memory_formats_give_identical_bits():
    """channels_last costs no copy and NCHW one transpose each way; both run the same kernels and GEMMs.  grad_input is
    accumulated with float reds whose order is not fixed, so it is compared to float rounding only."""
    case = make(2, 64, 14, 15, 48, 3, 2, 1, 1, 1, 2, True, True, leave=True, seed=4)
    go = torch.randn(2, 48, 7, 8)
    a_out, a = ours(case, go, torch.contiguous_format)
    b_out, b = ours(case, go, torch.channels_last)
    assert torch.equal(a_out, b_out)
    for n in ("off", "m", "w", "b"):
        assert torch.equal(a[n], b[n]), n
    assert torch.allclose(a["x"], b["x"], rtol=1e-5, atol=1e-6)
    x = case["x"].to(DEV).contiguous(memory_format=torch.channels_last)
    y = modulated_deform_conv(x, case["off"].to(DEV), case["m"].to(DEV), case["w"].to(DEV), None, 2, 1, 1, 1, 2)
    assert y.is_contiguous(memory_format=torch.channels_last)
    assert modulated_deform_conv(x.contiguous(), case["off"].to(DEV), case["m"].to(DEV), case["w"].to(DEV), None, 2,
                                 1, 1, 1, 2).is_contiguous()


@pytest.mark.parametrize("force_generic", [False, True])
def test_offset_and_mask_gradients_are_bit_reproducible(force_generic):
    case = make(2, 128, 16, 17, 64, 3, 1, 1, 1, 1, 2, True, True, leave=True, seed=8)
    go = torch.randn(2, 64, 16, 17)
    with kernel_flags(_lib.FLAG_FORCE_GENERIC if force_generic else 0):
        runs = [ours(case, go)[1] for _ in range(3)]
    for r in runs[1:]:
        assert torch.equal(r["off"], runs[0]["off"]) and torch.equal(r["m"], runs[0]["m"])


def test_chunks_of_images_match_one_chunk():
    """im2col_step splits the batch into chunks of images; any batch size works (5 images, chunks of 2)."""
    case = make(5, 32, 9, 10, 16, 3, 1, 1, 1, 1, 1, True, True, seed=12)
    go = torch.randn(5, 16, 9, 10)
    a_out, a = ours(case, go, step=64)
    b_out, b = ours(case, go, step=2)
    assert torch.equal(a_out, b_out)
    for n in ("off", "m"):
        assert torch.equal(a[n], b[n])
    # grad_weight: one GEMM against per-chunk GEMMs summed; grad_input: float reds
    assert torch.allclose(a["w"], b["w"], rtol=1e-4, atol=1e-4) and torch.allclose(a["x"], b["x"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("B", [65535, 65536])
def test_batch_at_the_grid_y_limit(B):
    """The fast im2col / col2im launches put the images of a chunk on grid.y, so they take at most 65535; a larger chunk
    (im2col_step >= B hands the whole batch to one launch) goes to the generic kernels.  Both sides of that gate against
    torchvision in float64 (on the GPU: 65536 tiny images).  At 65535 the offset gradients differ in their bits from the
    generic kernels' (another summation order: the fast kernels ran); at 65536 both runs are the generic kernels."""
    case = make(B, 16, 5, 5, 16, 3, 1, 1, 1, 1, 1, True, True, leave=True, seed=13)
    go = torch.randn(case["out_shape"], generator=torch.Generator().manual_seed(7))
    ref_out, ref_g = oracle(case, go, DEV)
    # 3.3 million sampling positions: a few lie within float32 rounding of an integer, where the offset gradient jumps
    # and either one-sided derivative is right -- those offsets are left out of the grad_offset comparison
    s = snap(case["off"], (3, 3), 1, case["padding"], 1)
    smooth = ((s - s.round()).abs() > 1e-4).view(B, 9, 2, 5, 5).all(2, keepdim=True).expand(B, 9, 2, 5, 5)
    ref_g["off"] = ref_g["off"].cpu() * smooth.reshape(s.shape)
    res = {}
    for flags in (0, _lib.FLAG_FORCE_GENERIC):
        n0 = _lib.launch_count()
        with kernel_flags(flags):
            out, g = ours(case, go, step=B)
        assert _lib.launch_count() > n0
        errs = {"out": nerr(out, ref_out)}
        errs.update({n: nerr(g[n].cpu() * smooth.reshape(s.shape) if n == "off" else g[n], ref_g[n]) for n in ref_g})
        assert all(e < 5e-5 for e in errs.values()), (flags, errs)
        res[flags] = (out, g)
    (out, g), (gout, gg) = res[0], res[_lib.FLAG_FORCE_GENERIC]
    if B <= 65535:
        assert not torch.equal(g["off"], gg["off"])
    else:
        assert torch.equal(out, gout) and torch.equal(g["off"], gg["off"]) and torch.equal(g["m"], gg["m"])


def test_deterministic_mode_raises_and_warns():
    case = make(1, 16, 6, 6, 8, 3, 1, 1, 1, 1, 1, True, True, seed=1)
    go = torch.randn(1, 8, 6, 6)
    set_deterministic(True)
    with pytest.raises(RuntimeError, match="deterministic"):
        ours(case, go)
    set_deterministic(False)
    old, old_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        with pytest.raises(RuntimeError, match="deterministic"):
            ours(case, go)
        torch.use_deterministic_algorithms(True, warn_only=True)
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            _, g = ours(case, go)
        assert any("deterministic" in str(w.message) for w in caught)
        assert g["x"] is not None
    finally:
        torch.use_deterministic_algorithms(old, warn_only=old_warn)


def test_cuda_graph_capture_of_module_forward_backward():
    torch.manual_seed(0)
    mod = ModulatedDeformConv(64, 64, 3, padding=1).to(DEV)
    case = make(2, 64, 12, 13, 64, 3, 1, 1, 1, 1, 1, True, True, seed=6)
    x = case["x"].to(DEV).requires_grad_(True)
    off, m = case["off"].to(DEV).requires_grad_(True), case["m"].to(DEV).requires_grad_(True)

    def step():
        y = mod(x, off, m)
        y.square().mean().backward()
        return y

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            mod.zero_grad(set_to_none=True); x.grad = off.grad = m.grad = None
            step()
    torch.cuda.current_stream().wait_stream(side)
    mod.zero_grad(set_to_none=True); x.grad = off.grad = m.grad = None
    eager = step().detach().clone()
    eager_g = [t.grad.detach().clone() for t in (off, m, mod.weight, mod.bias, x)]
    mod.zero_grad(set_to_none=True); x.grad = off.grad = m.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    for t in (off, m, mod.weight, mod.bias, x):
        t.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, eager)
    got = [t.grad for t in (off, m, mod.weight, mod.bias, x)]
    for a, b in zip(got[:4], eager_g[:4]):
        assert torch.equal(a, b)
    assert torch.allclose(got[4], eager_g[4], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("with_mask", [True, False])
def test_torch_compile_fullgraph_matches_eager(with_mask):
    torch._dynamo.reset()
    torch.manual_seed(0)
    mod = (ModulatedDeformConv(32, 32, 3, padding=1) if with_mask else DeformConv(32, 32, 3, padding=1)).to(DEV)
    case = make(2, 32, 10, 11, 32, 3, 1, 1, 1, 1, 1, True, False, seed=13)
    x = case["x"].to(DEV).requires_grad_(True)
    off, m = case["off"].to(DEV), case["m"].to(DEV)

    def fn(x, off, m):
        return mod(x, off, m) if with_mask else mod(x, off)

    compiled = torch.compile(fn, fullgraph=True, backend="aot_eager")
    y_c = compiled(x, off, m)
    y_c.square().sum().backward()
    gx_c, gw_c = x.grad.clone(), mod.weight.grad.clone()
    x.grad = None; mod.weight.grad = None
    y_e = fn(x, off, m)
    y_e.square().sum().backward()
    assert torch.equal(y_c, y_e)
    assert torch.equal(gw_c, mod.weight.grad)
    assert torch.allclose(gx_c, x.grad, rtol=1e-5, atol=1e-5)    # float reds
    torch._dynamo.reset()


def test_opcheck_dcnv2():
    case = make(2, 32, 8, 9, 16, 3, 1, 1, 1, 1, 1, True, True, seed=14)
    args = (case["x"].to(DEV).requires_grad_(True), case["off"].to(DEV).requires_grad_(True),
            case["m"].to(DEV).requires_grad_(True), case["w"].to(DEV).requires_grad_(True),
            case["b"].to(DEV).requires_grad_(True), 1, 1, 1, 1, 1, 1, 1, 1, 64)
    torch.library.opcheck(torch.ops.ir_ads_b200.dcnv2.default, args,
                          test_utils=("test_schema", "test_autograd_registration", "test_faketensor"))


def test_deform_bottleneck_block_at_res3_full_size():
    """detectron2's DeformBottleneckBlock conv2 (modulated): offset conv -> chunk -> sigmoid -> ModulatedDeformConv, at
    res3 of an 800x1333 image (stride 2 from 200x334, 128 channels, channels_last), against the same composition with
    torchvision's deform_conv2d in float64 on the CPU (offset conv included, on the same widened parameters)."""
    torch.manual_seed(0)
    B, C, H, W = 1, 128, 200, 334
    conv_offset = torch.nn.Conv2d(C, 27, 3, stride=2, padding=1).to(DEV)
    torch.nn.init.normal_(conv_offset.weight, std=0.01)
    torch.nn.init.normal_(conv_offset.bias, std=0.5)
    dcn = ModulatedDeformConv(C, C, 3, stride=2, padding=1, bias=False).to(DEV)
    x = torch.randn(B, C, H, W, device=DEV).contiguous(memory_format=torch.channels_last).requires_grad_(True)

    def block(x, conv_offset, conv):
        o1, o2, mk = torch.chunk(conv_offset(x), 3, dim=1)
        return conv(x, torch.cat((o1, o2), dim=1), mk.sigmoid())

    old_tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False     # the offset conv in float32, as the oracle's in float64
    try:
        out = block(x, conv_offset, dcn)
        go = torch.randn_like(out)
        out.backward(go)
        with torch.no_grad():
            om32 = conv_offset(x.detach())      # the float32 offsets the kernels sampled at
    finally:
        torch.backends.cudnn.allow_tf32 = old_tf32
    assert out.shape == (B, C, 100, 167) and out.is_contiguous(memory_format=torch.channels_last)
    conv_d = torch.nn.Conv2d(C, 27, 3, stride=2, padding=1).double()
    conv_d.load_state_dict({k: v.cpu().double() for k, v in conv_offset.state_dict().items()})
    xd = x.detach().cpu().double().requires_grad_(True)
    wd = dcn.weight.detach().cpu().double().requires_grad_(True)
    target = snap(torch.cat(torch.chunk(om32, 3, dim=1)[:2], dim=1), (3, 3), 2, (1, 1), 1)

    def tv_at_float32_positions(x, off, m):   # the value of the snapped offsets, the gradient of the float64 ones
        return tv_ops.deform_conv2d(x, off + (target - off).detach(), wd, None, stride=2, padding=1, mask=m)

    ref = block(xd, conv_d, tv_at_float32_positions)
    ref.backward(go.cpu().double())
    assert nerr(out, ref) < 2e-5
    assert nerr(dcn.weight.grad, wd.grad) < 2e-5
    assert nerr(x.grad, xd.grad) < 1e-4

"""Fused DCNv3 module path on the sm_100a kernels: ``DCNv3FusedFunction`` / ``msda_dcnv3_fused_*`` take the mask
logits and run the module's softmax over K inside the kernels (record mode kPreDcnSoftmax).

Contract: the result of ``torch.softmax`` followed by ``DCNv3Function`` (the unfused route) up to the softmax's float
rounding, and of the float64 port ``oracle/dcnv3_torch.py`` behind a float64 softmax; float16 equal to the float32
kernels on widened input (output rounded once, offset / logit gradients bit for bit); the ``DCNv3`` module equal to
its old composition (and, under autocast, within the bound that the unrounded mask explains)."""
import pytest
import torch

from oracle import dcnv3_torch
from test_dcnv3 import pixel_smooth_mask
from test_fp16_gpu import assert_within_one_ulp

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


def out_size(H, k, s, p, d):
    return (H + 2 * p - (d * (k - 1) + 1)) // s + 1


def make_case(N, H, W, G, C, k, s, p, d, scale, seed=0, logit_scale=2.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    Ho, Wo, K = out_size(H, k, s, p, d), out_size(W, k, s, p, d), k * k
    inp = torch.randn(N, H, W, G * C, device=DEV, generator=g)
    off = torch.randn(N, Ho, Wo, G * K * 2, device=DEV, generator=g) * 1.5
    logits = torch.randn(N, Ho, Wo, G * K, device=DEV, generator=g) * logit_scale
    go = torch.randn(N, Ho, Wo, G * C, device=DEV, generator=g)
    return inp, off, logits, go, (k, k, s, s, p, p, d, d, G, C, scale)


def softmax_rows(logits, G):
    N, Ho, Wo, _ = logits.shape
    return torch.softmax(logits.view(N, Ho, Wo, G, -1), -1).view(N, Ho, Wo, -1)


def fused(inp, off, logits, go, args):
    """(out, grad_input, grad_offset, grad_logits) through DCNv3FusedFunction"""
    from ir_ads_b200 import DCNv3FusedFunction
    leaves = [t.clone().requires_grad_(True) for t in (inp, off, logits)]
    out = DCNv3FusedFunction.apply(*leaves, *args, 256)
    out.backward(go)
    return [out.detach()] + [t.grad for t in leaves]


def unfused(inp, off, logits, go, args):
    """the same through torch.softmax + DCNv3Function (the route the module took before)"""
    from ir_ads_b200 import DCNv3Function
    leaves = [t.clone().requires_grad_(True) for t in (inp, off, logits)]
    out = DCNv3Function.apply(leaves[0], leaves[1], softmax_rows(leaves[2], args[8]), *args, 256)
    out.backward(go)
    return [out.detach()] + [t.grad for t in leaves]


def port(inp, off, logits, go, args):
    """float64 softmax + the float64 port of the reference's dcnv3_core_pytorch, differentiated by autograd"""
    leaves = [t.double().clone().requires_grad_(True) for t in (inp, off, logits)]
    out = dcnv3_torch.forward(leaves[0], leaves[1], softmax_rows(leaves[2], args[8]), *args)
    out.backward(go.double())
    return [out.detach()] + [t.grad for t in leaves]


KEYS = ("out", "grad_input", "grad_offset", "grad_logits")


def assert_close(got, want, off, args, what, rtol=1e-5):
    """test_dcnv3's bars: |err| <= rtol * max|want| + 1e-6, grad_offset away from bilinear cell boundaries"""
    m = torch.from_numpy(pixel_smooth_mask({"offset": off.cpu().numpy(), "args": args}, 1e-4)).to(DEV).double()
    for a, b, key in zip(got, want, KEYS):
        mk = m if key == "grad_offset" else 1.0
        err = ((a.double() - b.double()) * mk).abs().max().item()
        assert err <= rtol * b.double().abs().max().item() + 1e-6, (what, key, err)


GEOMS = [(3, 1, 1, 1, 1.0), (3, 2, 1, 1, 2.0), (3, 1, 2, 2, 0.7), (5, 1, 2, 1, 1.3)]


# ------------------------------------------------------------------------------------------------
# 1. float32: fused == unfused == float64 port
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [16, 32, 64, 128])
@pytest.mark.parametrize("k,s,p,d,scale", GEOMS)
def test_f32_matches_unfused_and_port(C, k, s, p, d, scale):
    case = make_case(2, 13, 17, 3, C, k, s, p, d, scale, seed=C + k + s)
    got = fused(*case)
    assert_close(got, unfused(*case), case[1], case[4], "vs unfused")
    assert_close(got, port(*case), case[1], case[4], "vs port")


@pytest.mark.parametrize("k", [1, 7, 8])
def test_f32_point_counts(k):
    """K = 1, 49 and 64 (the most the fast kernels take), besides the 9 and 25 above"""
    case = make_case(2, 12, 15, 2, 32, k, 1, k // 2, 1, 1.0, seed=k)
    got = fused(*case)
    assert_close(got, unfused(*case), case[1], case[4], f"K={k * k} vs unfused")
    assert_close(got, port(*case), case[1], case[4], f"K={k * k} vs port")


# ------------------------------------------------------------------------------------------------
# 2. float16 / bfloat16
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [16, 32, 64, 128])
@pytest.mark.parametrize("k,s,p,d,scale", [GEOMS[0], GEOMS[2]])
def test_f16_equals_f32_on_widened_input(C, k, s, p, d, scale):
    inp, off, logits, go, args = make_case(2, 13, 17, 3, C, k, s, p, d, scale, seed=C)
    inp, go = inp.half(), go.half()
    r16 = fused(inp, off, logits, go, args)
    r32 = fused(inp.float(), off, logits, go.float(), args)
    gi_abs = fused(inp.float(), off, logits, go.float().abs(), args)[1]   # softmax weights are positive
    assert r16[0].dtype == torch.float16 and r16[1].dtype == torch.float16
    assert torch.equal(r16[0], r32[0].half())
    assert torch.equal(r16[2], r32[2]) and torch.equal(r16[3], r32[3])
    assert_within_one_ulp(r16[1], r32[1], gi_abs, f"fused dcnv3 f16 C={C}")


@pytest.mark.parametrize("C", [16, 32, 64, 128])
def test_bf16_close_to_f32(C):
    inp, off, logits, go, args = make_case(2, 13, 17, 3, C, 3, 1, 1, 1, 1.0, seed=5 + C)
    inp, go = inp.bfloat16(), go.bfloat16()
    rb = fused(inp, off, logits, go, args)
    r32 = fused(inp.float(), off, logits, go.float(), args)
    assert rb[0].dtype == torch.bfloat16 and rb[1].dtype == torch.bfloat16
    for a, b, key, tol in zip(rb, r32, KEYS, (1e-2, 1e-2, 1e-5, 1e-5)):
        err = (a.float() - b).abs().max().item()
        assert err <= tol * b.abs().max().item() + 1e-6, (key, err)


# ------------------------------------------------------------------------------------------------
# 3. non-finite and extreme logits: what the unfused route makes of torch.softmax's output
# ------------------------------------------------------------------------------------------------
def test_extreme_logits_follow_torch_softmax():
    inp, off, logits, go, args = make_case(2, 10, 12, 2, 32, 3, 1, 1, 1, 1.0, seed=9)
    G = args[8]
    lg = logits.view(2, 10, 12, G, 9)
    lg[0, 1, 2, 0, 3] = 1e4
    lg[0, 1, 2, 1, :] = -1e4
    lg[0, 1, 2, 1, 5] = 1e4
    lg[1, 3, :, 0, 0] = -float("inf")             # some points switched off
    lg[1, 4, 5, 1, :] = -float("inf")             # a whole row: torch.softmax gives NaN
    got, want = fused(inp, off, logits, go, args), unfused(inp, off, logits, go, args)
    for a, b, key in zip(got, want, KEYS):
        assert torch.equal(torch.isnan(a), torch.isnan(b)), key
        fin = ~torch.isnan(b)
        err = (a[fin] - b[fin]).abs().max().item()
        assert err <= 1e-5 * b[fin].abs().max().item() + 1e-6, (key, err)
    assert torch.isnan(got[3].view(2, 10, 12, G, 9)[1, 4, 5, 1]).all()
    assert (got[3].view(2, 10, 12, G, 9)[1, 3, :, 0, 0] == 0).all()      # weight 0 -> logit gradient 0
    assert torch.isfinite(got[0][0]).all()


# ------------------------------------------------------------------------------------------------
# 4. the DCNv3 module: fused route against the old composition
# ------------------------------------------------------------------------------------------------
def composed_forward(m, input):
    """the DCNv3 module's forward before the fused route (the reference's composition)"""
    from ir_ads_b200 import DCNv3Function
    N, H, W, _ = input.shape
    x = m.input_proj(input)
    x_proj = x
    x1 = m.dw_conv(input.permute(0, 3, 1, 2))
    offset = m.offset(x1)
    mask = torch.nn.functional.softmax(m.mask(x1).reshape(N, H, W, m.group, -1), -1).reshape(N, H, W, -1).type(x.dtype)
    x = DCNv3Function.apply(x.contiguous(), offset.contiguous(), mask.contiguous(), m.kernel_size, m.kernel_size,
                            m.stride, m.stride, m.pad, m.pad, m.dilation, m.dilation, m.group, m.group_channels,
                            m.offset_scale, 256)
    if m.center_feature_scale:
        scale = torch.nn.functional.linear(x1, weight=m.center_feature_scale_proj_weight,
                                           bias=m.center_feature_scale_proj_bias).sigmoid()
        scale = scale[..., None].repeat(1, 1, 1, 1, m.channels // m.group).flatten(-2)
        x = x * (1 - scale) + x_proj * scale
    return m.output_proj(x)


def make_module(channels=64, group=4, cfs=False, seed=0):
    from ir_ads_b200.dcnv3 import DCNv3
    torch.manual_seed(seed)
    m = DCNv3(channels=channels, group=group, center_feature_scale=cfs).to(DEV)
    with torch.no_grad():   # non-trivial offsets / masks (the reference initialises both layers to zero)
        for lin in (m.offset, m.mask):
            lin.weight.normal_(0.0, 0.2)
            lin.bias.normal_(0.0, 1.0)
        if cfs:
            m.center_feature_scale_proj_weight.normal_(0.0, 0.1)
    return m


def module_grads(m, forward, x0, gout, dtype=None):
    x = x0.clone().requires_grad_(True)
    params = [p for p in m.parameters()]
    if dtype is None:
        out = forward(x)
    else:
        with torch.autocast("cuda", dtype=dtype):
            out = forward(x)
    grads = torch.autograd.grad(out, [x] + params, gout.to(out.dtype))
    return out.detach(), grads


@pytest.mark.parametrize("cfs", [False, True])
@pytest.mark.parametrize("dtype,tol", [(None, 1e-5), (torch.float16, 1e-2), (torch.bfloat16, 5e-2)])
def test_module_fused_matches_composition(cfs, dtype, tol):
    """float32: the softmax rounding only.  Under autocast the composition rounds the mask (and its gradient) to the
    autocast dtype and the fused route does not: bounded at 1e-2 (float16) / 5e-2 (bfloat16) of the largest value."""
    m = make_module(cfs=cfs, seed=1)
    x0 = torch.randn(2, 20, 24, 64, device=DEV)
    gout = torch.randn(2, 20, 24, 64, device=DEV)
    out_f, g_f = module_grads(m, m, x0, gout, dtype)
    out_c, g_c = module_grads(m, lambda x: composed_forward(m, x), x0, gout, dtype)
    assert out_f.dtype == out_c.dtype
    names = ["out", "input"] + [n for n, _ in m.named_parameters()]
    for a, b, name in zip([out_f] + list(g_f), [out_c] + list(g_c), names):
        err = (a.float() - b.float()).abs().max().item()
        assert err <= tol * b.float().abs().max().item() + 1e-6, (name, err)


def test_module_graph_has_no_softmax_node_and_one_kernel_forward():
    from ir_ads_b200 import DCNv3FusedFunction, _lib
    m = make_module()
    x = torch.randn(2, 16, 16, 64, device=DEV, requires_grad=True)

    def names(out):
        seen, stack, found = set(), [out.grad_fn], []
        while stack:
            f = stack.pop()
            if f is None or f in seen:
                continue
            seen.add(f)
            found.append(type(f).__name__)
            stack.extend(nf for nf, _ in f.next_functions)
        return found

    fused_names = names(m(x))
    assert "SoftmaxBackward0" not in fused_names and any("DCNv3FusedFunction" in n for n in fused_names)
    assert "SoftmaxBackward0" in names(composed_forward(m, x))
    for dtype in (torch.float32, torch.bfloat16, torch.float16):
        inp, off, logits, go, args = make_case(2, 12, 14, 4, 16, 3, 1, 1, 1, 1.0, seed=3)
        inp, go = inp.to(dtype).requires_grad_(True), go.to(dtype)
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        out = DCNv3FusedFunction.apply(inp, off, logits, *args, 256)
        assert _lib.launch_count() - n0 == 1, dtype                  # softmax and core op in one kernel
        n0 = _lib.launch_count()
        out.backward(go)
        assert _lib.launch_count() - n0 == (1 if dtype == torch.float32 else 2), dtype   # + float -> 2-byte cast


# ------------------------------------------------------------------------------------------------
# 5. deterministic mode
# ------------------------------------------------------------------------------------------------
def test_deterministic_route_is_the_composed_route_bit_for_bit():
    from ir_ads_b200 import set_deterministic
    case = make_case(2, 24, 28, 4, 32, 3, 1, 1, 1, 1.0, seed=11)
    try:
        set_deterministic(True)
        a, b = fused(*case), fused(*case)
        want = unfused(*case)
    finally:
        set_deterministic(False)
    for x, y, z, key in zip(a[1:], b[1:], want[1:], KEYS[1:]):
        assert torch.equal(x, y), key
        assert torch.equal(x, z), key


def test_module_twice_gives_identical_gradients():
    from ir_ads_b200 import set_deterministic
    m = make_module(cfs=True, seed=2)
    x0 = torch.randn(2, 28, 36, 64, device=DEV)
    gout = torch.randn(2, 28, 36, 64, device=DEV)
    old_cudnn = torch.backends.cudnn.deterministic
    try:
        set_deterministic(True)
        torch.backends.cudnn.deterministic = True
        runs = [module_grads(m, m, x0, gout)[1] for _ in range(2)]
    finally:
        set_deterministic(False)
        torch.backends.cudnn.deterministic = old_cudnn
    for a, b in zip(*runs):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------
# 6. CUDA-graph capture of the module, forward + backward
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("det", [False, True])
def test_module_forward_backward_captured(det):
    from ir_ads_b200 import set_deterministic
    m = make_module(cfs=True, seed=4)
    x = torch.randn(2, 20, 24, 64, device=DEV, requires_grad=True)
    gout = torch.randn(2, 20, 24, 64, device=DEV)
    params = list(m.parameters())

    def step():
        out = m(x)
        return [out] + list(torch.autograd.grad(out, [x] + params, gout))

    old_cudnn = torch.backends.cudnn.deterministic
    try:
        set_deterministic(det)
        torch.backends.cudnn.deterministic = True
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
        # (float reds, and the library-external layers of the module, may sum in another order from run to run)
        for a, b in zip(captured, eager):
            assert (a - b).abs().max().item() <= 1e-5 * b.abs().max().item() + 1e-6
    finally:
        set_deterministic(False)
        torch.backends.cudnn.deterministic = old_cudnn


# ------------------------------------------------------------------------------------------------
# 7. shapes the fused kernels do not take: the module composes, as before
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("channels,group,kernel_size,dtype", [(96, 4, 3, torch.float32), (64, 4, 9, torch.float32),
                                                              (64, 4, 3, torch.float64)])
def test_unsupported_shapes_fall_back(channels, group, kernel_size, dtype):
    from ir_ads_b200 import DCNv3FusedFunction
    from ir_ads_b200.dcnv3 import DCNv3
    torch.manual_seed(0)
    m = DCNv3(channels=channels, group=group, kernel_size=kernel_size, pad=kernel_size // 2).to(DEV, dtype)
    with torch.no_grad():
        for lin in (m.offset, m.mask):
            lin.weight.normal_(0.0, 0.2)
    x0 = torch.randn(2, 11, 13, channels, device=DEV, dtype=dtype)
    gout = torch.randn(2, 11, 13, channels, device=DEV, dtype=dtype)
    out_f, g_f = module_grads(m, m, x0, gout)
    out_c, g_c = module_grads(m, lambda x: composed_forward(m, x), x0, gout)
    assert torch.equal(out_f, out_c)
    for a, b in zip(g_f, g_c):
        assert (a - b).abs().max().item() <= 1e-5 * b.abs().max().item() + 1e-6
    # the Function itself refuses them: a missing kernel is an error, not a silent fallback
    K = kernel_size * kernel_size
    with pytest.raises(RuntimeError, match="fused DCNv3 needs|unsupported input dtype"):
        DCNv3FusedFunction.apply(torch.zeros(1, 4, 4, channels, device=DEV, dtype=dtype),
                                 torch.zeros(1, 4, 4, group * K * 2, device=DEV),
                                 torch.zeros(1, 4, 4, group * K, device=DEV), kernel_size, kernel_size, 1, 1,
                                 kernel_size // 2, kernel_size // 2, 1, 1, group, channels // group, 1.0, 256)


# ------------------------------------------------------------------------------------------------
# 8. realistic size: InternImage-T stage 1
# ------------------------------------------------------------------------------------------------
def test_internimage_t_stage1():
    case = make_case(16, 200, 336, 4, 16, 3, 1, 1, 1, 1.0, seed=21)
    got, want = fused(*case), unfused(*case)
    # both routes sample at the same float32 locations (dcn_location): grad_offset needs no cell-boundary mask here
    for a, b, key in zip(got, want, KEYS):
        err = (a - b).abs().max().item()
        assert err <= 1e-5 * b.abs().max().item() + 1e-6, (key, err)

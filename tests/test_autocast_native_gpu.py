"""Autocast-native module paths on the B200: 16-bit offsets / logits in the fused MSDeformAttn and DCNv3 kernels
(MSDA_BF16_AUX16 / MSDA_F16_AUX16) and the mixed-dtype add + LayerNorm epilogue.

Contract: widening f16 / bf16 to float is exact and the kernels compute in float32, so the 16-bit route gives the
`.float()` route's output bits, and its offset / logit gradients are that route's float32 gradients rounded once (what
autograd's cast gives).  grad_value differs by the float-red order only, and not at all in deterministic mode."""
import pytest
import torch

from test_dcnv3_fused_gpu import make_case

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
HALVES = [torch.float16, torch.bfloat16]


def same_bits(a, b):
    """torch.equal, NaN-aware: NaN where the other is NaN (payloads are not promised), equal bits elsewhere"""
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a.masked_fill(na, 0), b.masked_fill(nb, 0))


def assert_red_spread(got, want, what):
    """grad_value of two float-red runs: one rounding of the 16-bit result apart at most"""
    err = (got.double() - want.double()).abs()
    ulp = want.double().abs() * (2.0 ** -7 if want.dtype == torch.bfloat16 else 2.0 ** -10) * 2
    assert bool((err <= ulp + 1e-6 * want.double().abs().max()).all()), (what, float(err.max()))


@pytest.fixture
def deterministic():
    from ir_ads_b200 import set_deterministic
    set_deterministic(True)
    yield
    set_deterministic(False)


# ------------------------------------------------------------------------------------------------
# 1. MSDeformAttnFusedFunction: 16-bit offsets / logits against the .float() route
# ------------------------------------------------------------------------------------------------
def msda_case(D, dtype, ref_dim, masked, seed=0, levels=((12, 17), (6, 9), (3, 5), (2, 3)), B=2, Q=37, H=4, P=4):
    from ir_ads_b200.workloads import level_tensors
    g = torch.Generator(device=DEV).manual_seed(seed)
    shapes, lsi = level_tensors(list(levels), DEV)
    S, L = sum(h * w for h, w in levels), len(levels)
    value = torch.randn(B, S, H, D, device=DEV, generator=g).to(dtype)
    off = (torch.randn(B, Q, H, L, P, 2, device=DEV, generator=g) * 3.0).to(dtype)
    logits = (torch.randn(B, Q, H, L * P, device=DEV, generator=g) * 2.0).to(dtype)
    ref = torch.rand(B, Q, L, ref_dim, device=DEV, generator=g)
    mask = (torch.rand(B, S, device=DEV, generator=g) < 0.2) if masked else None
    go = torch.randn(B, Q, H * D, device=DEV, generator=g).to(dtype)
    return value, shapes, lsi, off, logits, ref, mask, go


def msda_run(value, shapes, lsi, off, logits, ref, mask, go, widen):
    from ir_ads_b200.functional import MSDeformAttnFusedFunction
    v = value.clone().requires_grad_(True)
    o = (off.float() if widen else off).clone().requires_grad_(True)
    lg = (logits.float() if widen else logits).clone().requires_grad_(True)
    out = MSDeformAttnFusedFunction.apply(v, shapes, lsi, o, lg, ref, mask)
    out.backward(go)
    return out.detach(), v.grad, o.grad, lg.grad


LEVELS4 = ((12, 17), (6, 9), (3, 5), (2, 3))
# (levels, P): the three point-count specialisations of the fused kernels -- P = 4, P = 8 and a runtime P (here 3) --
# and an odd L*P = 9, which writes each row's gradients point by point instead of two points per store
LP_CASES = [(LEVELS4, 4), (LEVELS4, 8), (LEVELS4[:3], 3)]


@pytest.mark.parametrize("lp", LP_CASES, ids=["L4P4", "L4P8", "L3P3"])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("ref_dim", [2, 4])
@pytest.mark.parametrize("dtype", HALVES)
@pytest.mark.parametrize("D", [16, 32, 64, 128])
def test_msda_function_16bit_route(D, dtype, ref_dim, masked, lp):
    levels, P = lp
    case = msda_case(D, dtype, ref_dim, masked, seed=D + ref_dim + P, levels=levels, P=P)
    new = msda_run(*case, widen=False)
    old = msda_run(*case, widen=True)
    assert new[0].dtype == dtype and torch.equal(new[0], old[0])
    assert new[2].dtype == dtype and same_bits(new[2], old[2].to(dtype))
    assert new[3].dtype == dtype and same_bits(new[3], old[3].to(dtype))
    assert_red_spread(new[1], old[1], "grad_value")


@pytest.mark.parametrize("dtype", HALVES)
def test_msda_function_16bit_route_deterministic(dtype, deterministic):
    case = msda_case(32, dtype, 4, True, seed=7)
    new = msda_run(*case, widen=False)
    old = msda_run(*case, widen=True)
    assert torch.equal(new[0], old[0]) and torch.equal(new[1], old[1])
    assert same_bits(new[2], old[2].to(dtype)) and same_bits(new[3], old[3].to(dtype))


def test_msda_function_reference_points_requiring_grad():
    from ir_ads_b200.functional import MSDeformAttnFusedFunction
    value, shapes, lsi, off, logits, ref, mask, go = msda_case(32, torch.bfloat16, 4, False, seed=3)
    res = []
    for widen in (False, True):
        o = (off.float() if widen else off).clone().requires_grad_(True)
        lg = (logits.float() if widen else logits).clone().requires_grad_(True)
        r = ref.clone().requires_grad_(True)
        out = MSDeformAttnFusedFunction.apply(value, shapes, lsi, o, lg, r, mask)
        out.backward(go)
        res.append((out.detach(), o.grad, lg.grad, r.grad))
    (n_out, n_o, n_lg, n_r), (o_out, o_o, o_lg, o_r) = res
    assert torch.equal(n_out, o_out) and torch.equal(n_r, o_r)
    assert same_bits(n_o, o_o.bfloat16()) and same_bits(n_lg, o_lg.bfloat16())


def test_msda_function_refuses_other_mixes():
    from ir_ads_b200.functional import MSDeformAttnFusedFunction
    value, shapes, lsi, off, logits, ref, mask, go = msda_case(32, torch.float16, 2, False)
    with pytest.raises(RuntimeError, match="value's dtype"):
        MSDeformAttnFusedFunction.apply(value, shapes, lsi, off.bfloat16(), logits.bfloat16(), ref, None)
    with pytest.raises(RuntimeError, match="share a dtype"):
        MSDeformAttnFusedFunction.apply(value, shapes, lsi, off, logits.float(), ref, None)
    with pytest.raises(RuntimeError, match="value's dtype"):
        MSDeformAttnFusedFunction.apply(value.float(), shapes, lsi, off, logits, ref, None)


def test_msda_extreme_logits_f16():
    """+-inf, NaN, 65504 and all -inf rows behave as the .float() route (NaN-aware)"""
    value, shapes, lsi, off, logits, ref, mask, go = msda_case(32, torch.float16, 2, False, seed=11)
    lg = logits.clone()
    lg[0, 0, 0, 3] = float("inf")
    lg[0, 1, 1, 5] = float("nan")
    lg[0, 2, 2, :] = 65504.0
    lg[0, 3, 3, 1] = -65504.0
    lg[1, 4, 0, :] = float("-inf")
    lg[1, 5, 1, 2:] = float("-inf")
    new = msda_run(value, shapes, lsi, off, lg, ref, None, go, widen=False)
    old = msda_run(value, shapes, lsi, off, lg, ref, None, go, widen=True)
    assert same_bits(new[0], old[0])
    assert same_bits(new[2], old[2].half()) and same_bits(new[3], old[3].half())
    assert torch.isnan(new[3][1, 4, 0]).all() and not torch.isnan(new[3][1, 5, 1, :2]).any()


# ------------------------------------------------------------------------------------------------
# 2. DCNv3FusedFunction: 16-bit offset / mask logits against the .float() route
# ------------------------------------------------------------------------------------------------
def dcn_run(inp, off, lg, go, args, widen):
    from ir_ads_b200 import DCNv3FusedFunction
    i = inp.clone().requires_grad_(True)
    o = (off.float() if widen else off).clone().requires_grad_(True)
    m = (lg.float() if widen else lg).clone().requires_grad_(True)
    out = DCNv3FusedFunction.apply(i, o, m, *args, 256)
    out.backward(go)
    return out.detach(), i.grad, o.grad, m.grad


DCN_CASES = [  # N, H, W, G, C, k, stride, pad, dilation, offset_scale
    (2, 9, 11, 4, 16, 3, 1, 1, 1, 1.0), (2, 10, 9, 2, 32, 3, 2, 1, 1, 2.0), (1, 12, 10, 2, 64, 5, 1, 2, 2, 0.7),
    (1, 8, 7, 1, 128, 3, 1, 0, 1, 1.3), (1, 12, 12, 2, 16, 8, 1, 3, 1, 1.0)]


@pytest.mark.parametrize("dtype", HALVES)
@pytest.mark.parametrize("case", DCN_CASES, ids=lambda c: "C%d_k%d_s%d_p%d_d%d" % (c[4], c[5], c[6], c[7], c[8]))
def test_dcn_function_16bit_route(case, dtype):
    inp, off, lg, go, args = make_case(*case, seed=case[4])
    inp, off, lg, go = inp.to(dtype), off.to(dtype), lg.to(dtype), go.to(dtype)
    new = dcn_run(inp, off, lg, go, args, widen=False)
    old = dcn_run(inp, off, lg, go, args, widen=True)
    assert new[0].dtype == dtype and torch.equal(new[0], old[0])
    assert new[2].dtype == dtype and same_bits(new[2], old[2].to(dtype))
    assert new[3].dtype == dtype and same_bits(new[3], old[3].to(dtype))
    assert_red_spread(new[1], old[1], "grad_input")


@pytest.mark.parametrize("dtype", HALVES)
def test_dcn_function_16bit_route_deterministic(dtype, deterministic):
    inp, off, lg, go, args = make_case(2, 10, 9, 4, 32, 3, 1, 1, 1, 1.0, seed=5)
    inp, off, lg, go = inp.to(dtype), off.to(dtype), lg.to(dtype), go.to(dtype)
    new = dcn_run(inp, off, lg, go, args, widen=False)
    old = dcn_run(inp, off, lg, go, args, widen=True)
    assert torch.equal(new[0], old[0]) and torch.equal(new[1], old[1])
    assert same_bits(new[2], old[2].to(dtype)) and same_bits(new[3], old[3].to(dtype))


def test_dcn_extreme_logits_f16():
    inp, off, lg, go, args = make_case(1, 8, 8, 2, 16, 3, 1, 1, 1, 1.0, seed=2)
    inp, off, lg, go = inp.half(), off.half(), lg.half(), go.half()
    lg[0, 0, 0, 2] = float("inf")
    lg[0, 1, 1, 4] = float("nan")
    lg[0, 2, 2, :9] = 65504.0
    lg[0, 3, 3, 9:] = float("-inf")
    lg[0, 4, 4, 1:9] = float("-inf")
    new = dcn_run(inp, off, lg, go, args, widen=False)
    old = dcn_run(inp, off, lg, go, args, widen=True)
    assert same_bits(new[0], old[0])
    assert same_bits(new[2], old[2].half()) and same_bits(new[3], old[3].half())


# ------------------------------------------------------------------------------------------------
# 3. both modules under autocast, against a reconstruction of the .float() route
# ------------------------------------------------------------------------------------------------
def msda_module(seed=0, levels=((12, 17), (6, 9), (3, 5), (2, 3)), B=2):
    from ir_ads_b200 import MultiScaleDeformableAttention
    from ir_ads_b200.workloads import level_tensors
    torch.manual_seed(seed)
    shapes, lsi = level_tensors(list(levels), DEV)
    S = sum(h * w for h, w in levels)
    m = MultiScaleDeformableAttention(dropout=0.0, batch_first=True).to(DEV)
    with torch.no_grad():
        m.sampling_offsets.weight.normal_(0, 0.05)
        m.attention_weights.weight.normal_(0, 0.2)
    q = torch.randn(B, S, 256, device=DEV)
    ref = torch.rand(B, S, len(levels), 2, device=DEV)
    return m, q, ref, shapes, lsi


def msda_widening_route(m, q, ref, shapes, lsi):
    """the module's fused branch before 16-bit offsets / logits: both Linear outputs widened with .float()"""
    from ir_ads_b200.functional import MSDeformAttnFusedFunction
    B, Q, _ = q.shape
    H, L, P = m.num_heads, m.num_levels, m.num_points
    value = m.value_proj(q).view(B, Q, H, -1)
    offsets = m.sampling_offsets(q).view(B, Q, H, L, P, 2)
    logits = m.attention_weights(q).view(B, Q, H, L * P)
    out = MSDeformAttnFusedFunction.apply(value.contiguous(), shapes, lsi, offsets.float().contiguous(),
                                          logits.float().contiguous(), ref.float().contiguous(), None)
    return m.output_proj(out) + q


def dcn_module(seed=0, N=2, H=12, W=14, G=4, C=16):
    from ir_ads_b200.dcnv3 import DCNv3
    torch.manual_seed(seed)
    m = DCNv3(channels=G * C, group=G).to(DEV)
    with torch.no_grad():
        for lin in (m.offset, m.mask):
            lin.weight.normal_(0.0, 0.2)
            lin.bias.normal_(0.0, 1.0)
    return m, torch.randn(N, H, W, G * C, device=DEV)


def dcn_widening_route(m, input):
    """the DCNv3 module's fused branch before 16-bit offset / logits: both Linear outputs widened with .float()"""
    from ir_ads_b200 import DCNv3FusedFunction
    N, H, W, _ = input.shape
    x = m.input_proj(input)
    x1 = m.dw_conv(input.permute(0, 3, 1, 2))
    offset = m.offset(x1)
    x = DCNv3FusedFunction.apply(x.contiguous(), offset.float().contiguous(),
                                 m.mask(x1).float().reshape(N, H, W, -1).contiguous(), m.kernel_size, m.kernel_size,
                                 m.stride, m.stride, m.pad, m.pad, m.dilation, m.dilation, m.group, m.group_channels,
                                 m.offset_scale, 256)
    return m.output_proj(x)


def _modules():
    def msda(seed):
        m, q, ref, shapes, lsi = msda_module(seed)
        return m, q, (lambda mm, x: mm(x, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi)), \
            (lambda mm, x: msda_widening_route(mm, x, ref, shapes, lsi))

    def dcn(seed):
        m, x = dcn_module(seed)
        return m, x, (lambda mm, xx: mm(xx)), dcn_widening_route
    return {"msda": msda, "dcn": dcn}


def _run_module(m, x, fwd, dtype, gout):
    m.zero_grad(set_to_none=True)
    xx = x.clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=dtype):
        out = fwd(m, xx)
    (out.float() * gout).sum().backward()
    return [out.detach(), xx.grad] + [p.grad.clone() for p in m.parameters()]


@pytest.mark.parametrize("dtype", HALVES)
@pytest.mark.parametrize("kind", ["msda", "dcn"])
def test_module_autocast_matches_widening_route(kind, dtype, deterministic):
    import copy
    m, x, new_fwd, old_fwd = _modules()[kind](1)
    m_old = copy.deepcopy(m)
    gout = torch.randn(x.shape, device=DEV)
    new = _run_module(m, x, new_fwd, dtype, gout)
    old = _run_module(m_old, x, old_fwd, dtype, gout)
    for i, (a, b) in enumerate(zip(new, old)):
        assert torch.equal(a, b), (kind, i)


@pytest.mark.parametrize("dtype", HALVES)
@pytest.mark.parametrize("kind", ["msda", "dcn"])
def test_module_autocast_outputs_equal_default_mode(kind, dtype):
    m, x, new_fwd, old_fwd = _modules()[kind](2)
    with torch.autocast("cuda", dtype=dtype):
        assert torch.equal(new_fwd(m, x), old_fwd(m, x))


def _fused_node(out):
    seen, stack = set(), [out.grad_fn]
    while stack:
        n = stack.pop()
        if n is None or n in seen:
            continue
        seen.add(n)
        if "FusedFunction" in type(n).__name__:
            return n
        stack.extend(f for f, _ in n.next_functions)
    raise AssertionError("no fused node in the graph")


def _casts_below(node, stop=("AddmmBackward0", "MmBackward0", "BmmBackward0", "LinearBackward0", "AddBackward0",
                              "AccumulateGrad")):
    """node types between `node` and the Linear layers that feed it"""
    found, stack = [], [node]
    while stack:
        n = stack.pop()
        if n is None:
            continue
        name = type(n).__name__
        if name in stop:
            continue
        found.append(name)
        stack.extend(f for f, _ in n.next_functions)
    return found


@pytest.mark.parametrize("dtype", HALVES)
@pytest.mark.parametrize("kind", ["msda", "dcn"])
def test_module_autocast_saves_16bit_projections_and_has_no_casts(kind, dtype):
    m, x, new_fwd, _ = _modules()[kind](3)
    saved = []
    with torch.autograd.graph.saved_tensors_hooks(lambda t: saved.append(t) or t, lambda t: t):
        with torch.autocast("cuda", dtype=dtype):
            out = new_fwd(m, x)
    node = _fused_node(out)
    idx = (3, 4) if kind == "msda" else (1, 2)
    for i in idx:
        names = _casts_below(node.next_functions[i][0])
        assert "ToCopyBackward0" not in names, (kind, names)
    # the fused node's saved offsets / logits are 16-bit, and no float32 tensor of their shape is saved anywhere
    if kind == "msda":
        B, S, _ = x.shape
        shapes = [(B, S, m.num_heads, m.num_levels, m.num_points, 2), (B, S, m.num_heads, m.num_levels * m.num_points)]
    else:
        N, H, W, _ = x.shape
        K = m.kernel_size ** 2
        shapes = [(N, H, W, m.group * K * 2), (N, H, W, m.group * K)]
    for shp in shapes:
        kinds = [t.dtype for t in saved if tuple(t.shape) == shp]
        assert dtype in kinds and torch.float32 not in kinds, (shp, kinds)


@pytest.mark.parametrize("kind", ["msda", "dcn"])
def test_module_autocast_cuda_graph(kind):
    m, x, new_fwd, _ = _modules()[kind](4)
    xin = x.clone().requires_grad_(True)

    def step():
        with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
            out = new_fwd(m, xin)
        out.float().square().mean().backward()
        return out

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            m.zero_grad(set_to_none=False)
            xin.grad = None
            step()
    torch.cuda.current_stream().wait_stream(side)
    eager = step().detach().clone()
    m.zero_grad(set_to_none=False)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


# ------------------------------------------------------------------------------------------------
# 4. epilogue: float16 same-dtype form and the mixed form
# ------------------------------------------------------------------------------------------------
def _ln_fp64(a, b, w, bias, go):
    ref = [t.double().clone().requires_grad_(True) for t in (a, b, w, bias)]
    want = torch.nn.functional.layer_norm(ref[0] + ref[1], (a.shape[-1],), ref[2], ref[3], 1e-5)
    want.backward(go.double())
    return [want.detach()] + [t.grad for t in ref]


def _close(got, exp, tol, what):
    got, exp = got.double(), exp.double()
    err = (got - exp).abs().max().item()
    assert err <= tol * exp.abs().max().item() + 1e-6, (what, err)


@pytest.mark.parametrize("swap", [False, True])
@pytest.mark.parametrize("dtype", HALVES)
@pytest.mark.parametrize("rows,C", [((7, 33), 256), ((5000,), 64), ((3, 5), 100), ((2, 9), 1024), ((0,), 256),
                                    ((100000,), 256), ((3, 7), 200), ((5, 3), 516), ((9,), 772), ((4, 4), 1020)])
def test_mixed_epilogue(rows, C, dtype, swap):
    from ir_ads_b200.epilogue import add_layer_norm
    torch.manual_seed(C)
    a = (torch.randn(*rows, C, device=DEV) * 2.0 + 0.3).to(dtype)
    b = torch.randn(*rows, C, device=DEV)
    norm = torch.nn.LayerNorm(C).to(DEV)
    with torch.no_grad():
        norm.weight.normal_(1.0, 0.5)
        norm.bias.normal_(0.0, 0.1)
    go = torch.randn(*rows, C, device=DEV)
    res = []
    for _ in range(2):
        norm.zero_grad(set_to_none=True)
        la, lb = a.clone().requires_grad_(True), b.clone().requires_grad_(True)
        y = add_layer_norm(lb, la, norm) if swap else add_layer_norm(la, lb, norm)
        node = type(y.grad_fn).__name__
        y.backward(go)
        res.append([y.detach(), la.grad, lb.grad, norm.weight.grad.clone(), norm.bias.grad.clone()])
    y, ga, gb, gw, gbias = res[0]
    assert y.dtype == torch.float32 and ga.dtype == dtype and gb.dtype == torch.float32
    assert all(torch.equal(p, q) for p, q in zip(res[0], res[1]))       # bit-reproducible, parameters included
    assert torch.equal(ga, gb.to(dtype))                                 # grad_a is grad_b rounded once
    if a.numel() == 0:
        return
    assert "AddLayerNormMixedFunction" in node
    want = _ln_fp64(a, b, norm.weight.detach(), norm.bias.detach(), go)
    for got, exp, what in zip((y, gb, gw, gbias), (want[0], want[2], want[3], want[4]), ("y", "grad_b", "dw", "db")):
        _close(got, exp, 1e-5, what)


@pytest.mark.parametrize("rows,C", [((7, 33), 256), ((5000,), 64), ((2, 9), 1024), ((100000,), 256), ((3, 7), 200),
                                    ((5, 3), 516), ((9,), 772), ((4, 4), 1020)])
def test_f16_epilogue(rows, C):
    from ir_ads_b200.epilogue import AddLayerNormFunction
    torch.manual_seed(C)
    a = (torch.randn(*rows, C, device=DEV) * 2.0 + 0.3).half()
    b = torch.randn(*rows, C, device=DEV).half()
    w = torch.randn(C, device=DEV) * 0.5 + 1.0
    bias = torch.randn(C, device=DEV) * 0.1
    go = torch.randn(*rows, C, device=DEV).half()
    leaves = [t.clone().requires_grad_(True) for t in (a, b, w, bias)]
    y = AddLayerNormFunction.apply(*leaves, 1e-5)
    y.backward(go)
    want = _ln_fp64(a, b, w, bias, go)
    assert y.dtype == torch.float16
    _close(y, want[0], 2e-3, "y")
    _close(leaves[0].grad, want[1], 2e-3, "grad_a")
    assert torch.equal(leaves[0].grad, leaves[1].grad)
    _close(leaves[2].grad, want[3], 2e-3, "dw")
    _close(leaves[3].grad, want[4], 2e-3, "db")
    leaves2 = [t.clone().requires_grad_(True) for t in (a, b, w, bias)]
    AddLayerNormFunction.apply(*leaves2, 1e-5).backward(go)
    assert all(torch.equal(p.grad, q.grad) for p, q in zip(leaves, leaves2))


def test_f16_addends_under_autocast_keep_the_float32_result():
    """Two float16 addends under autocast: norm(a + b) as before float16 was supported (float32 LayerNorm, float32
    result); without autocast the float16 kernel runs and returns float16."""
    from ir_ads_b200 import _lib
    from ir_ads_b200.epilogue import add_layer_norm
    torch.manual_seed(9)
    a, b = torch.randn(64, 256, device=DEV).half(), torch.randn(64, 256, device=DEV).half()
    norm = torch.nn.LayerNorm(256).to(DEV)
    with torch.autocast("cuda", dtype=torch.float16):
        n0 = _lib.launch_count()
        y = add_layer_norm(a, b, norm)
        assert _lib.launch_count() == n0
        want = norm(a + b)
    assert y.dtype == torch.float32 and torch.equal(y, want)
    n0 = _lib.launch_count()
    y16 = add_layer_norm(a, b, norm)
    assert y16.dtype == torch.float16 and _lib.launch_count() == n0 + 1


def _layer_case(kind, seed=2):
    from ir_ads_b200.encoder import DeformableCrossAttentionBlock, DeformableEncoderLayer
    from ir_ads_b200.workloads import _pixel_centres, level_tensors
    torch.manual_seed(seed)
    levels = [(12, 17), (6, 9), (3, 5), (2, 3)]
    shapes, lsi = level_tensors(levels, DEV)
    S = sum(h * w for h, w in levels)
    if kind == "encoder":
        layer = DeformableEncoderLayer(attn_dropout=0.0, ffn_dropout=0.0).to(DEV)
        attn, norms = layer.attentions[0], list(layer.norms)
    else:
        layer = DeformableCrossAttentionBlock(attn_dropout=0.0).to(DEV)
        attn, norms = layer.attn, [layer.norm]
    with torch.no_grad():
        attn.sampling_offsets.weight.normal_(0, 0.05)
        attn.attention_weights.weight.normal_(0, 0.2)
        for n in norms:
            n.weight.normal_(1.0, 0.2)
            n.bias.normal_(0.0, 0.1)
    if kind == "encoder":
        x = torch.randn(2, S, 256, device=DEV)
        pos = torch.randn(2, S, 256, device=DEV) * 0.1
        ref = _pixel_centres(levels, DEV)[None, :, None, :].expand(2, S, 4, 2).contiguous()
        fwd = lambda xx: layer(xx, query_pos=pos, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi,
                               level_shapes=levels)
    else:
        x = torch.randn(2, 50, 256, device=DEV)
        memory = torch.randn(2, S, 256, device=DEV)
        pos = torch.randn(2, 50, 256, device=DEV) * 0.1
        boxes = torch.rand(2, 50, 4, device=DEV) * 0.5 + 0.25
        ratios = torch.ones(2, 4, 2, device=DEV)
        fwd = lambda xx: layer(xx, memory, pos, boxes, ratios, shapes, lsi)
    return layer, x, fwd


@pytest.mark.parametrize("dtype", HALVES)
@pytest.mark.parametrize("kind", ["encoder", "cross"])
def test_layer_blocks_fuse_the_epilogue_under_autocast(kind, dtype):
    """Fused epilogue vs op by op (add + LayerNorm in PyTorch) under autocast.  The fused kernel's LayerNorm differs
    from torch's in float rounding only, but a 16-bit Linear downstream can round that difference up to one 16-bit ulp,
    so the bound is the 16-bit type's, not the float32 test's 3e-5."""
    from ir_ads_b200 import _lib
    from ir_ads_b200.epilogue import add_layer_norm
    import ir_ads_b200.encoder as enc
    layer, x, fwd = _layer_case(kind)
    res, launches = {}, {}
    for fused in (True, False):
        layer.zero_grad(set_to_none=True)
        xx = x.clone().requires_grad_(True)
        enc.add_layer_norm = add_layer_norm if fused else (lambda a, b, norm: norm(a + b))
        try:
            n0 = _lib.launch_count()
            with torch.autocast("cuda", dtype=dtype):
                out = fwd(xx)
            torch.cuda.synchronize()
            launches[fused] = _lib.launch_count() - n0
        finally:
            enc.add_layer_norm = add_layer_norm
        if fused:
            assert "AddLayerNormMixedFunction" in type(out.grad_fn).__name__
        out.float().square().mean().backward()
        res[fused] = [out.detach().float(), xx.grad] + [p.grad.clone() for p in layer.parameters()]
    n_epilogues = 2 if kind == "encoder" else 1
    assert launches[True] == launches[False] + n_epilogues        # one fused kernel per epilogue ran
    tol = 3e-2 if dtype == torch.bfloat16 else 5e-3
    for i, (a, b) in enumerate(zip(res[True], res[False])):
        err = float((a.double() - b.double()).abs().max())
        assert err <= tol * float(b.double().abs().max()) + 1e-6, (kind, i, err)


# ------------------------------------------------------------------------------------------------
# 5. full size
# ------------------------------------------------------------------------------------------------
def test_full_size_cfg2_encoder_module_bf16_deterministic(deterministic):
    """cfg2 (DINO-R50 encoder, B=8): deterministic bits of the module under bf16 autocast equal the .float() route"""
    import copy
    from ir_ads_b200.workloads import LEVELS, _pixel_centres
    levels = [tuple(l) for l in LEVELS["dino_r50"]]
    m, q, _, shapes, lsi = msda_module(5, levels=levels, B=8)
    ref = _pixel_centres(levels, DEV)[None, :, None, :].expand(8, q.shape[1], 4, 2).contiguous()
    m_old = copy.deepcopy(m)
    gout = torch.randn(q.shape, device=DEV)
    new = _run_module(m, q, lambda mm, x: mm(x, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi,
                                             level_shapes=levels), torch.bfloat16, gout)
    old = _run_module(m_old, q, lambda mm, x: msda_widening_route(mm, x, ref, shapes, lsi), torch.bfloat16, gout)
    for i, (a, b) in enumerate(zip(new, old)):
        assert torch.equal(a, b), i


def test_full_size_dcn_stage1_f16():
    """InternImage-T stage 1 (16 x 200 x 336, G = 4, group_channels 16) under float16 autocast"""
    import copy
    m, x = dcn_module(6, N=16, H=200, W=336, G=4, C=16)
    m_old = copy.deepcopy(m)
    gout = torch.randn(x.shape, device=DEV)
    new = _run_module(m, x, lambda mm, xx: mm(xx), torch.float16, gout)
    old = _run_module(m_old, x, dcn_widening_route, torch.float16, gout)
    assert torch.equal(new[0], old[0])
    for i, (a, b) in enumerate(zip(new[1:], old[1:])):   # float reds: the order of the grad_input sums differs
        err = float((a.double() - b.double()).abs().max())
        assert err <= 1e-2 * float(b.double().abs().max()) + 1e-6, (i, err)

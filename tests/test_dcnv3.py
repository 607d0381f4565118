"""DCNv3 core op (SURVEY 8f-4): oracle port pinned to reference-made vectors (CPU), sm_100a kernels vs those
vectors (GPU).  Golden: tests/golden/dcnv3_golden.npz from /root/reference/detrex/layers/dcn_v3.py:121-166."""
import os

import numpy as np
import pytest
import torch

from oracle import dcnv3_torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = ["k3_s1", "k3_s2", "k3_d2", "k5", "k1"]


@pytest.fixture(scope="module")
def golden():
    blob = np.load(os.path.join(ROOT, "tests", "golden", "dcnv3_golden.npz"))

    def case(name):
        c = {k[len(name) + 1:]: blob[k] for k in blob.files if k.startswith(name + "/")}
        N, H, W, G, C, k, s, p, d = [int(x) for x in c["geom"]]
        c["args"] = (k, k, s, s, p, p, d, d, G, C, float(c["scale"][0]))
        return c

    return case


def pixel_smooth_mask(c, band):
    """[N,Ho,Wo,G*K*2] mask: False where a sampling coordinate is within `band` px of an integer (bilinear cell
    boundary, where grad_offset is discontinuous)."""
    k, _, s, _, p, _, d, _, G, C, scale = c["args"]
    off = c["offset"].astype(np.float64)
    N, Ho, Wo, _ = off.shape
    K = k * k
    off = off.reshape(N, Ho, Wo, G, K, 2)
    centre = (d * (k - 1)) // 2
    i = (np.arange(K) // k)[None, None, None, None, :]
    j = (np.arange(K) % k)[None, None, None, None, :]
    wo = np.arange(Wo)[None, None, :, None, None]
    ho = np.arange(Ho)[None, :, None, None, None]
    px = centre - p + wo * s - centre * scale + (i * d + off[..., 0]) * scale
    py = centre - p + ho * s - centre * scale + (j * d + off[..., 1]) * scale
    ok = (np.abs(px - np.round(px)) > band) & (np.abs(py - np.round(py)) > band)
    return np.repeat(ok[..., None], 2, -1).reshape(N, Ho, Wo, G * K * 2)


@pytest.mark.parametrize("name", CASES)
def test_port_matches_reference_golden(golden, name):
    c = golden(name)
    t = lambda k: torch.from_numpy(c[k]).double()
    out, gi, go, gm = dcnv3_torch.forward_backward(t("input"), t("offset"), t("mask"), t("grad_out"), *c["args"])
    for got, key in ((out, "out"), (gi, "grad_input"), (go, "grad_offset"), (gm, "grad_mask")):
        assert np.abs(got.numpy() - c[key]).max() <= 1e-12 * max(1.0, np.abs(c[key]).max()), key


def test_cpu_tensors_raise():
    from ir_ads_b200.dcnv3 import DCNv3Function
    x = torch.randn(1, 4, 4, 32)
    with pytest.raises(RuntimeError, match="CPU"):
        DCNv3Function.apply(x, torch.zeros(1, 4, 4, 2 * 9 * 2), torch.ones(1, 4, 4, 18), 3, 3, 1, 1, 1, 1, 1, 1, 2, 16, 1.0, 256)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("name", CASES)
def test_kernels_match_reference_golden(golden, name, dtype):
    from ir_ads_b200.dcnv3 import DCNv3Function
    c = golden(name)
    dev = "cuda:0"
    inp = torch.from_numpy(c["input"]).to(dev, dtype)
    go = torch.from_numpy(c["grad_out"]).to(dev, dtype)
    if dtype == torch.bfloat16:     # yardstick on the same rounded inputs
        ref = dcnv3_torch.forward_backward(inp.double().cpu(), torch.from_numpy(c["offset"]).double(),
                                           torch.from_numpy(c["mask"]).double(), go.double().cpu(), *c["args"])
        want = [r.numpy() for r in ref]
    else:
        want = [c["out"], c["grad_input"], c["grad_offset"], c["grad_mask"]]
    leaves = [inp.clone().requires_grad_(True), torch.from_numpy(c["offset"]).to(dev).requires_grad_(True),
              torch.from_numpy(c["mask"]).to(dev).requires_grad_(True)]
    out = DCNv3Function.apply(*leaves, *c["args"], 256)
    out.backward(go)
    got = [out] + [t.grad for t in leaves]
    m = pixel_smooth_mask(c, 1e-4)
    tol = 1e-5 if dtype == torch.float32 else 1e-2
    for g, w, key in zip(got, want, ("out", "grad_input", "grad_offset", "grad_mask")):
        g = g.detach().double().cpu().numpy()
        mk = m if key == "grad_offset" else 1.0
        t = tol if key in ("out", "grad_input") else max(tol, 1e-4) if dtype == torch.bfloat16 else tol
        assert np.abs(g * mk - w * mk).max() <= t * np.abs(w).max() + 1e-6, (key, float(np.abs(g * mk - w * mk).max()))


@pytest.mark.gpu
def test_dcnv3_larger_shape_and_unsupported():
    """InternImage-like stage (56x56, 4 groups x 16 channels, 3x3) against the port in float64."""
    from ir_ads_b200.dcnv3 import DCNv3Function
    dev = "cuda:0"
    g = torch.Generator().manual_seed(0)
    N, H, W, G, C, k = 2, 56, 56, 4, 16, 3
    inp = torch.randn(N, H, W, G * C, generator=g)
    off = torch.randn(N, H, W, G * 9 * 2, generator=g)
    mask = torch.softmax(torch.randn(N, H, W, G, 9, generator=g), -1).reshape(N, H, W, G * 9)
    go = torch.randn(N, H, W, G * C, generator=g)
    args = (k, k, 1, 1, 1, 1, 1, 1, G, C, 1.0)
    want = dcnv3_torch.forward_backward(inp.double(), off.double(), mask.double(), go.double(), *args)
    leaves = [t.to(dev).requires_grad_(True) for t in (inp, off, mask)]
    out = DCNv3Function.apply(*leaves, *args, 256)
    out.backward(go.to(dev))
    for gt, w, key in zip([out, leaves[0].grad, leaves[2].grad], [want[0], want[1], want[3]], ("out", "grad_input", "grad_mask")):
        err = (gt.detach().double().cpu() - w).abs().max().item()
        assert err <= 1e-5 * w.abs().max().item() + 1e-6, (key, err)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.float16])
@pytest.mark.parametrize("C,k,stride,pad,dil,scale", [(24, 3, 1, 1, 1, 1.0), (8, 3, 2, 1, 1, 2.0), (40, 5, 1, 2, 1, 0.7),
                                                      (12, 3, 1, 2, 2, 1.0), (16, 9, 1, 4, 1, 1.0)])
def test_dcnv3_generic_shapes_against_port(C, k, stride, pad, dil, scale, dtype):
    """Channel counts outside {16,32,64,128}, K > 64 (9x9 = 81 points) and float64 -- everything else the reference
    dispatches (dcnv3_cuda.cu:66-80) -- run as a one-level MSDeformAttn composition on the generic kernels; checked
    against the float64 port of dcnv3_core_pytorch, all four tensors."""
    from ir_ads_b200.dcnv3 import DCNv3Function, fast_supported
    dev = "cuda:0"
    g = torch.Generator().manual_seed(C + k)
    N, H, W, G = 2, 13, 17, 3
    K = k * k
    Ho = (H + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
    Wo = (W + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
    inp = torch.randn(N, H, W, G * C, generator=g)
    off = torch.randn(N, Ho, Wo, G * K * 2, generator=g) * 1.5
    mask = torch.softmax(torch.randn(N, Ho, Wo, G, K, generator=g), -1).reshape(N, Ho, Wo, G * K)
    go = torch.randn(N, Ho, Wo, G * C, generator=g)
    args = (k, k, stride, stride, pad, pad, dil, dil, G, C, scale)
    if dtype == torch.float16:
        inp, go = inp.half().float(), go.half().float()       # yardstick on the same rounded inputs
    assert dtype == torch.float64 or not fast_supported(inp.to(dtype), k, k, C)
    want = dcnv3_torch.forward_backward(inp.double(), off.double(), mask.double(), go.double(), *args)
    aux = torch.float64 if dtype == torch.float64 else torch.float32
    leaves = [inp.to(dev, dtype).requires_grad_(True), off.to(dev, aux).requires_grad_(True),
              mask.to(dev, aux).requires_grad_(True)]
    out = DCNv3Function.apply(*leaves, *args, 256)
    assert out.dtype == dtype and tuple(out.shape) == (N, Ho, Wo, G * C)
    out.backward(go.to(dev, dtype))
    c = {"offset": off.numpy(), "args": args}
    m = torch.from_numpy(pixel_smooth_mask(c, 1e-4)).double()
    # (the port, like the reference function it restates, builds its reference points and dilation grid in float32 --
    # dcn_v3.py:74-118 -- so even the float64 run agrees with it to float32 location accuracy only)
    tol = {torch.float64: 1e-5, torch.float32: 1e-5, torch.float16: 2e-3}[dtype]
    for gt, w, key in zip([out, leaves[0].grad, leaves[1].grad, leaves[2].grad], want, ("out", "grad_input", "grad_offset", "grad_mask")):
        gt = gt.detach().double().cpu()
        mk = m if key == "grad_offset" else 1.0
        err = ((gt - w) * mk).abs().max().item()
        assert err <= tol * w.abs().max().item() + 1e-6, (key, err, w.abs().max().item())


@pytest.mark.gpu
def test_against_reference_dcnv3_formulation():
    """Whole-tensor comparison with the reference's own formulation (dcnv3_core_pytorch as restated in
    oracle/dcnv3_torch.py, pinned to reference-made vectors above) in float64 on the same GPU."""
    from ir_ads_b200.dcnv3 import DCNv3Function
    dev = "cuda:0"
    g = torch.Generator(device=dev).manual_seed(0)
    N, H, W, G, C, k = 2, 48, 64, 8, 32, 3
    for stride, pad, dil, scale in ((1, 1, 1, 1.0), (2, 1, 1, 2.0), (1, 2, 2, 0.7)):
        Ho = (H + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
        Wo = (W + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
        inp = torch.randn(N, H, W, G * C, device=dev, generator=g)
        off = torch.randn(N, Ho, Wo, G * 9 * 2, device=dev, generator=g) * 2.0
        mask = torch.softmax(torch.randn(N, Ho, Wo, G, 9, device=dev, generator=g), -1).reshape(N, Ho, Wo, G * 9)
        go = torch.randn(N, Ho, Wo, G * C, device=dev, generator=g)
        args = (k, k, stride, stride, pad, pad, dil, dil, G, C, scale)
        want = dcnv3_torch.forward_backward(inp.double(), off.double(), mask.double(), go.double(), *args)
        leaves = [t.clone().requires_grad_(True) for t in (inp, off, mask)]
        out = DCNv3Function.apply(*leaves, *args, 256)
        out.backward(go)
        got = [out.detach()] + [t.grad for t in leaves]
        # grad_offset is discontinuous where a sampling coordinate crosses a bilinear cell boundary, and the float64
        # yardstick may pick the other cell within float32 location accuracy: those points are left out
        m = torch.from_numpy(pixel_smooth_mask({"offset": off.cpu().numpy(), "args": args}, 1e-4)).to(dev).double()
        for a, b, key in zip(got, want, ("out", "grad_input", "grad_offset", "grad_mask")):
            mk = m if key == "grad_offset" else 1.0
            err = ((a.double() - b) * mk).abs().max().item()
            assert err <= 1e-5 * b.abs().max().item() + 1e-6, (key, stride, err)


def test_dcnv3_module_parameter_layout():
    from ir_ads_b200.dcnv3 import DCNv3
    m = DCNv3(channels=64, group=4, center_feature_scale=True)
    keys = list(m.state_dict())
    for k in ("dw_conv.0.weight", "dw_conv.1.1.weight", "offset.weight", "mask.bias", "input_proj.weight",
              "output_proj.bias", "center_feature_scale_proj_weight", "center_feature_scale_proj_bias"):
        assert k in keys, k
    assert m.offset.weight.abs().sum() == 0 and m.mask.bias.abs().sum() == 0
    with pytest.raises(ValueError):
        DCNv3(channels=30, group=4)


@pytest.mark.gpu
def test_dcnv3_module_matches_port_composition():
    """Module on the GPU vs the same parameters around the oracle port on the CPU in float64."""
    from ir_ads_b200.dcnv3 import DCNv3
    torch.manual_seed(0)
    m = DCNv3(channels=64, group=4, center_feature_scale=True)
    with torch.no_grad():
        m.offset.weight.normal_(0, 0.3)
        m.mask.weight.normal_(0, 0.3)
        m.center_feature_scale_proj_weight.normal_(0, 0.1)
    x = torch.randn(2, 11, 13, 64)
    md = m.double()
    xd = x.double()
    x1 = md.dw_conv(xd.permute(0, 3, 1, 2))
    off = md.offset(x1)
    mask = torch.softmax(md.mask(x1).reshape(2, 11, 13, 4, -1), -1).reshape(2, 11, 13, -1)
    xp = md.input_proj(xd)
    core = dcnv3_torch.forward(xp, off, mask, 3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0)
    sc = torch.nn.functional.linear(x1, md.center_feature_scale_proj_weight, md.center_feature_scale_proj_bias).sigmoid()
    sc = sc[..., None].repeat(1, 1, 1, 1, 16).flatten(-2)
    want = md.output_proj(core * (1 - sc) + xp * sc).detach()
    got = m.float().to("cuda:0")(x.to("cuda:0")).detach().cpu().double()
    assert (got - want).abs().max() <= 2e-5 * want.abs().max() + 1e-6

"""Fused residual add + LayerNorm (ir_ads_b200/epilogue.py, csrc/msda_epilogue.cu) against torch's own
``F.layer_norm(a + b)`` evaluated in float64 -- the two ops it replaces in the reference's transformer layers
(/root/reference/detrex/layers/transformer.py:152-192)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
# 100 000 rows: more than the 148 * 8 CTAs of 8 warps (9472 rows), so every warp loops over rows and carries its
# dgamma / dbeta partials; C = 200, 516, 772, 1020: the two- and eight-wide vector widths with predicated tail chunks
@pytest.mark.parametrize("rows,C", [((7, 33), 256), ((1,), 4), ((5000,), 64), ((3, 5), 100), ((2, 9), 1024), ((11,), 384),
                                    ((0,), 256), ((100000,), 256), ((3, 7), 200), ((5, 3), 516), ((9,), 772),
                                    ((4, 4), 1020)])
def test_add_layer_norm_matches_torch_fp64(rows, C, dtype):
    from ir_ads_b200.epilogue import AddLayerNormFunction
    torch.manual_seed(C + len(rows))
    a = (torch.randn(*rows, C, device=DEV) * 2.0 + 0.3).to(dtype)
    b = torch.randn(*rows, C, device=DEV).to(dtype)
    w = torch.randn(C, device=DEV) * 0.5 + 1.0
    bias = torch.randn(C, device=DEV) * 0.1
    go = torch.randn(*rows, C, device=DEV).to(dtype)
    leaves = [t.clone().requires_grad_(True) for t in (a, b, w, bias)]
    y = AddLayerNormFunction.apply(leaves[0], leaves[1], leaves[2], leaves[3], 1e-5)
    y.backward(go)
    ref = [t.double().clone().requires_grad_(True) for t in (a, b, w, bias)]
    want = F.layer_norm(ref[0] + ref[1], (C,), ref[2], ref[3], 1e-5)
    want.backward(go.double())
    tol = 2e-6 if dtype == torch.float32 else 1e-2
    assert y.dtype == dtype and y.shape == a.shape
    if a.numel() == 0:
        assert float(leaves[2].grad.abs().max()) == 0.0
        return

    def close(got, exp, what, t=tol):
        got, exp = got.double(), exp.double()
        assert (got - exp).abs().max() <= t * exp.abs().max() + 1e-6, (what, float((got - exp).abs().max()), float(exp.abs().max()))

    close(y, want, "y")
    close(leaves[0].grad, ref[0].grad, "grad_a")
    assert torch.equal(leaves[0].grad, leaves[1].grad)           # one gradient serves both addends
    n_rows = a.numel() // C
    close(leaves[2].grad, ref[2].grad, "grad_weight", max(tol, 1e-5) if dtype == torch.float32 else 2e-2)
    close(leaves[3].grad, ref[3].grad, "grad_bias", max(tol, 1e-5) if dtype == torch.float32 else 2e-2)
    # fixed reduction order: bit-reproducible
    leaves2 = [t.clone().requires_grad_(True) for t in (a, b, w, bias)]
    AddLayerNormFunction.apply(*leaves2, 1e-5).backward(go)
    assert all(torch.equal(p.grad, q.grad) for p, q in zip(leaves, leaves2)), n_rows


def test_add_layer_norm_errors_and_fallback():
    from ir_ads_b200.epilogue import AddLayerNormFunction, add_layer_norm
    norm = torch.nn.LayerNorm(6).to(DEV)                      # 6 % 4 != 0: the PyTorch composition
    a, b = torch.randn(3, 6, device=DEV), torch.randn(3, 6, device=DEV)
    assert torch.allclose(add_layer_norm(a, b, norm), norm(a + b))
    norm64 = torch.nn.LayerNorm(8).to(DEV).double()           # float64: the PyTorch composition
    a, b = torch.randn(3, 8, device=DEV).double(), torch.randn(3, 8, device=DEV).double()
    assert torch.allclose(add_layer_norm(a, b, norm64), norm64(a + b))
    with pytest.raises(RuntimeError, match="CPU"):
        AddLayerNormFunction.apply(torch.randn(2, 8), torch.randn(2, 8), torch.ones(8), torch.zeros(8), 1e-5)
    with pytest.raises(RuntimeError):
        AddLayerNormFunction.apply(torch.randn(2, 6, device=DEV), torch.randn(2, 6, device=DEV), torch.ones(6, device=DEV),
                                   torch.zeros(6, device=DEV), 1e-5)


def test_encoder_layer_fused_epilogue_matches_composition():
    """DeformableEncoderLayer with the fused epilogues == the op-by-op composition (add, LayerNorm, FFN identity)."""
    from ir_ads_b200.encoder import DeformableEncoderLayer
    from ir_ads_b200.workloads import _pixel_centres, level_tensors
    torch.manual_seed(2)
    levels = [(12, 17), (6, 9), (3, 5), (2, 3)]
    shapes, lsi = level_tensors(levels, DEV)
    S = sum(h * w for h, w in levels)
    layer = DeformableEncoderLayer(attn_dropout=0.0, ffn_dropout=0.0).to(DEV)
    with torch.no_grad():
        layer.attentions[0].sampling_offsets.weight.normal_(0, 0.05)
        layer.attentions[0].attention_weights.weight.normal_(0, 0.2)
        for n in layer.norms:
            n.weight.normal_(1.0, 0.2)
            n.bias.normal_(0.0, 0.1)
    x = torch.randn(2, S, 256, device=DEV)
    pos = torch.randn(2, S, 256, device=DEV) * 0.1
    ref = _pixel_centres(levels, DEV)[None, :, None, :].expand(2, S, 4, 2).contiguous()
    res = {}
    for fused in (True, False):
        layer.fuse_epilogue = fused
        layer.zero_grad(set_to_none=True)
        xx = x.clone().requires_grad_(True)
        out = layer(xx, query_pos=pos, reference_points=ref, spatial_shapes=shapes, level_start_index=lsi, level_shapes=levels)
        out.square().mean().backward()
        res[fused] = [out.detach(), xx.grad] + [p.grad.clone() for p in layer.parameters()]
    for a, b in zip(res[True], res[False]):
        assert (a - b).abs().max() <= 3e-5 * b.abs().max() + 1e-7, float((a - b).abs().max() / b.abs().max())

"""Packed (padding-free) batches on the GPU: MSDeformAttnPackedFunction against the padded fused path with the
rectangle mask (same bits for the output and the offset / logit gradients, grad_value within the float-red spread,
equal in deterministic mode), the decoder form, reference points that require grad, the encoder layer / 6-layer
encoder / cross-attention block packed against padded, one kernel per forward, CUDA-graph capture, and non-finite
values between images."""
import copy

import pytest
import torch

from ir_ads_b200 import _lib
from ir_ads_b200.encoder import (DeformableCrossAttentionBlock, DeformableEncoder, DeformableEncoderLayer,
                                 get_reference_points)
from ir_ads_b200.functional import MSDeformAttnFusedFunction, MSDeformAttnPackedFunction, set_deterministic
from ir_ads_b200.packing import PackedLevels, pack_levels, packed_reference_points, unpack_tokens

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
SHAPES4 = [(12, 17), (6, 9), (3, 5), (2, 3)]


def mixes(L):
    """[B][L] (h_v, w_v): B = 3 with an unpadded image and a 1 x 1 one, and B = 1 (one padded image)"""
    shapes = SHAPES4[:L]
    return shapes, [
        [shapes[:], [(1, 1)] * L, [(max(1, H * 2 // 3), max(1, W // 2)) for H, W in shapes]],
        [[(max(1, H - 1), max(1, W - 2)) for H, W in shapes]],
    ]


def padded_inputs(packing, H, D, P, ref_dim, vdt, adt, gen):
    """random padded tensors (zeros at padded rows of value and at padding query rows) and their packed rows"""
    B, S, L = packing.batch, packing.padded_len, packing.num_levels
    Qp = packing.query_pad
    value = torch.randn(B * S, H, D, generator=gen).to(DEV, vdt)
    off = (torch.randn(B * Qp, H, L, P, 2, generator=gen) * 3).to(DEV, adt)
    lg = torch.randn(B * Qp, H, L * P, generator=gen).to(DEV, adt)
    ref = torch.rand(B * Qp, L, ref_dim, generator=gen).to(DEV)
    go = torch.randn(packing.total_query, H * D, generator=gen).to(DEV, vdt)
    packed = (value[packing.value_index], off[packing.query_index], lg[packing.query_index], ref[packing.query_index])
    pv = unpack_tokens(packed[0], packing)[0].view(B, S, H, D)
    pq = [unpack_tokens(t, packing, queries=True)[0] for t in packed[1:]]
    return packed, (pv, *pq), go


def run_packed(packed, go, packing, need_ref=False):
    xs = [t.clone().requires_grad_(True) for t in packed[:3]] + [packed[3].clone().requires_grad_(need_ref)]
    out = MSDeformAttnPackedFunction.apply(*xs, packing)
    out.backward(go)
    return out, [x.grad for x in xs]


def run_padded(padded, go, packing, need_ref=False):
    xs = [t.clone().requires_grad_(True) for t in padded[:3]] + [padded[3].clone().requires_grad_(need_ref)]
    mask = packing.padding_mask
    out = MSDeformAttnFusedFunction.apply(xs[0], packing.spatial_shapes, packing.level_start_index, xs[1], xs[2], xs[3],
                                          mask)
    out.backward(unpack_tokens(go, packing, queries=True)[0].view(out.shape))
    q = packing.query_index
    flat = lambda t: t.reshape((-1,) + tuple(t.shape[2:]))  # noqa: E731
    grads = [flat(xs[0].grad)[packing.value_index]] + [flat(x.grad)[q] if x.grad is not None else None for x in xs[1:]]
    return flat(out)[q], grads


def assert_red_close(a, b, vdt):
    """grad_value: the same contributions summed in another order (and, for 16-bit values, rounded once)"""
    if vdt == torch.float32:
        torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-5 * float(b.abs().max()))
    else:
        torch.testing.assert_close(a.float(), b.float(), rtol=1.6e-2, atol=1e-2 * float(b.float().abs().max()))


CASES = [(vdt, adt) for vdt in (torch.float32, torch.bfloat16, torch.float16)
         for adt in ((torch.float32,) if vdt == torch.float32 else (torch.float32, vdt))]


@pytest.mark.parametrize("LP", [(4, 4), (4, 8), (3, 3)])
@pytest.mark.parametrize("ref_dim", [2, 4])
@pytest.mark.parametrize("vdt,adt", CASES)
@pytest.mark.parametrize("D", [16, 32, 64, 128])
def test_packed_equals_padded_fused(D, vdt, adt, ref_dim, LP):
    L, P = LP
    shapes, mix_list = mixes(L)
    gen = torch.Generator().manual_seed(D * 7 + L * 3 + P + ref_dim)
    for ext in mix_list:
        packing = PackedLevels(ext, shapes, DEV)
        packed, padded, go = padded_inputs(packing, 4, D, P, ref_dim, vdt, adt, gen)
        out, g = run_packed(packed, go, packing)
        ref_out, rg = run_padded(padded, go, packing)
        assert out.dtype == vdt and g[1].dtype == adt
        assert torch.equal(out, ref_out)
        assert torch.equal(g[1], rg[1]) and torch.equal(g[2], rg[2])
        assert_red_close(g[0], rg[0], vdt)


@pytest.mark.parametrize("vdt", [torch.float32, torch.bfloat16])
def test_deterministic_mode_is_bit_equal(vdt):
    shapes, mix_list = mixes(4)
    gen = torch.Generator().manual_seed(11)
    packing = PackedLevels(mix_list[0], shapes, DEV)
    packed, padded, go = padded_inputs(packing, 8, 32, 4, 2, vdt, torch.float32, gen)
    set_deterministic(True)
    try:
        n0 = _lib.launch_count()
        out, g = run_packed(packed, go, packing)
        assert _lib.launch_count() > n0
        ref_out, rg = run_padded(padded, go, packing)
        out2, g2 = run_packed(packed, go, packing)
    finally:
        set_deterministic(False)
    assert torch.equal(out, ref_out)
    for a, b, c in zip(g[:3], rg[:3], g2[:3]):
        assert torch.equal(a, b) and torch.equal(a, c)


@pytest.mark.parametrize("vdt,adt", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16)])
def test_decoder_form(vdt, adt):
    """q_start = b*Q over packed memory: a plain [B*Q] query set"""
    shapes, mix_list = mixes(4)
    gen = torch.Generator().manual_seed(12)
    packing = PackedLevels(mix_list[0], shapes, DEV).cross(30)
    assert packing.total_query == 90 and packing.meta[:, 2].tolist() == [0, 30, 60]
    packed, padded, go = padded_inputs(packing, 8, 32, 4, 4, vdt, adt, gen)
    out, g = run_packed(packed, go, packing)
    ref_out, rg = run_padded(padded, go, packing)
    assert torch.equal(out, ref_out) and torch.equal(g[1], rg[1]) and torch.equal(g[2], rg[2])
    assert_red_close(g[0], rg[0], vdt)


def test_reference_points_requiring_grad():
    shapes, mix_list = mixes(4)
    gen = torch.Generator().manual_seed(13)
    packing = PackedLevels(mix_list[0], shapes, DEV).cross(20)
    packed, padded, go = padded_inputs(packing, 8, 32, 4, 4, torch.float32, torch.float32, gen)
    out, g = run_packed(packed, go, packing, need_ref=True)
    ref_out, rg = run_padded(padded, go, packing, need_ref=True)
    assert torch.equal(out, ref_out)
    assert g[3] is not None and torch.equal(g[3], rg[3])
    assert torch.equal(g[1], rg[1]) and torch.equal(g[2], rg[2])
    assert_red_close(g[0], rg[0], torch.float32)


def test_one_kernel_per_forward():
    shapes, mix_list = mixes(4)
    packing = PackedLevels(mix_list[0], shapes, DEV)
    packed, _, _ = padded_inputs(packing, 8, 32, 4, 2, torch.float32, torch.float32, torch.Generator().manual_seed(1))
    n0 = _lib.launch_count()
    MSDeformAttnPackedFunction.apply(*packed, packing)
    assert _lib.launch_count() - n0 == 1


def test_non_finite_values_between_images_do_not_leak():
    """Rows between two images' value ranges (NaN / Inf) are never read: every corner is bounded by its own image's
    valid rectangle; their grad_value stays zero."""
    shapes, mix_list = mixes(4)
    gen = torch.Generator().manual_seed(14)
    packing = PackedLevels(mix_list[0], shapes, DEV)
    packed, _, go = padded_inputs(packing, 8, 32, 4, 2, torch.float32, torch.float32, gen)
    out, g = run_packed(packed, go, packing)
    gap = 5
    gapped = copy.copy(packing)
    meta = packing.meta.clone()
    meta[:, 0] += torch.arange(packing.batch, device=DEV) * gap
    gapped.meta, gapped.total_value = meta, packing.total_value + gap * (packing.batch - 1)
    gapped.max_value = packing.max_value
    value = torch.full((gapped.total_value,) + tuple(packed[0].shape[1:]), float("nan"), device=DEV)
    keep = torch.cat([torch.arange(int(s), int(s) + int(n), device=DEV) for s, n in meta[:, :2].tolist()])
    value[keep] = packed[0]
    value[keep[:1] + packing.value_counts[0]] = float("inf")
    out2, g2 = run_packed((value,) + packed[1:], go, gapped)
    assert torch.isfinite(out2).all() and torch.equal(out, out2)
    assert torch.equal(g[1], g2[1]) and torch.equal(g[2], g2[2])
    gap_rows = torch.ones(gapped.total_value, dtype=torch.bool, device=DEV)
    gap_rows[keep] = False
    assert (g2[0][gap_rows] == 0).all()
    assert_red_close(g2[0][keep], g[0], torch.float32)


# ---- encoder / decoder callers --------------------------------------------------------------------------------
def _batch(ext, shapes, C, gen):
    packing = PackedLevels(ext, shapes, DEV)
    B, S = packing.batch, packing.padded_len
    feats = [torch.randn(B, C, H, W, generator=gen).to(DEV) for H, W in shapes]
    pos = [torch.randn(B, C, H, W, generator=gen).to(DEV) for H, W in shapes]
    flat = lambda ms: torch.cat([m.flatten(2).transpose(1, 2) for m in ms], 1)  # noqa: E731
    padded = (flat(feats), flat(pos), get_reference_points(shapes, packing.valid_ratios, DEV))
    x, p = pack_levels(feats, packing, pos)
    return packing, padded, (x, p, packed_reference_points(packing))


def _compare(model_fn, packing, padded, packed, rtol, atol):
    qp = padded[0].clone().requires_grad_(True)
    qk = packed[0].clone().requires_grad_(True)
    out_pad = model_fn(qp, padded[1], padded[2], None)
    out_pk = model_fn(qk, packed[1], packed[2], packing)
    valid = out_pad.reshape(-1, out_pad.shape[-1])[packing.value_index]
    torch.testing.assert_close(out_pk.float(), valid.float(), rtol=rtol, atol=atol)
    gy = torch.randn(out_pk.shape, generator=torch.Generator().manual_seed(3)).to(DEV)
    out_pk.float().backward(gy)
    out_pad.float().backward(unpack_tokens(gy, packing)[0])
    torch.testing.assert_close(qk.grad, qp.grad.reshape(-1, qp.shape[-1])[packing.value_index], rtol=rtol,
                               atol=atol * 10)


@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("layers", [1, 6])
def test_encoder_packed_matches_padded(layers, autocast):
    torch.manual_seed(0)
    shapes, mix_list = mixes(4)
    model = (DeformableEncoderLayer(256, 8, 1024, 0.0, 0.0) if layers == 1 else
             DeformableEncoder(256, 8, 1024, 0.0, 0.0, num_layers=6)).to(DEV)
    with torch.no_grad():
        for m in model.modules():
            if hasattr(m, "sampling_offsets"):
                m.sampling_offsets.weight.normal_(0, 0.02)
                m.attention_weights.weight.normal_(0, 0.02)
    packing, padded, packed = _batch(mix_list[0], shapes, 256, torch.Generator().manual_seed(layers))

    def fn(q, pos, ref, pk):
        kw = dict(query_pos=pos, reference_points=ref, spatial_shapes=packing.spatial_shapes,
                  level_start_index=packing.level_start_index, level_shapes=packing.level_shapes)
        if pk is None:
            kw["query_key_padding_mask"] = packing.padding_mask
        else:
            kw["packing"] = pk
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
            return model(q, **kw)

    tol = (5e-2, 1e-1) if autocast else (1e-4, 1e-4 * layers)
    _compare(fn, packing, padded, packed, *tol)


@pytest.mark.parametrize("autocast", [False, True])
def test_cross_attention_block_packed_matches_padded(autocast):
    torch.manual_seed(1)
    shapes, mix_list = mixes(4)
    block = DeformableCrossAttentionBlock(256, 8, 0.0).to(DEV)
    with torch.no_grad():
        block.attn.sampling_offsets.weight.normal_(0, 0.02)
    packing, padded, packed = _batch(mix_list[0], shapes, 256, torch.Generator().manual_seed(7))
    gen = torch.Generator().manual_seed(8)
    B, Q = packing.batch, 40
    query = torch.randn(B, Q, 256, generator=gen).to(DEV)
    qpos = torch.randn(B, Q, 256, generator=gen).to(DEV)
    boxes = torch.rand(B, Q, 4, generator=gen).to(DEV)
    mem_pad = padded[0].clone().requires_grad_(True)
    mem_pk = packed[0].clone().requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        out_pad = block(query, mem_pad, qpos, boxes, packing.valid_ratios, packing.spatial_shapes,
                        packing.level_start_index, key_padding_mask=packing.padding_mask)
        out_pk = block(query, mem_pk, qpos, boxes, packing.valid_ratios, packing.spatial_shapes,
                       packing.level_start_index, packing=packing)
    rtol, atol = (5e-2, 5e-2) if autocast else (1e-5, 1e-5)
    torch.testing.assert_close(out_pk.float(), out_pad.float(), rtol=rtol, atol=atol)
    gy = torch.randn(out_pk.shape, generator=gen).to(DEV)
    out_pk.float().backward(gy)
    out_pad.float().backward(gy)
    torch.testing.assert_close(mem_pk.grad, mem_pad.grad.reshape(-1, 256)[packing.value_index], rtol=rtol,
                               atol=atol * 10)


def test_cuda_graph_capture_of_packed_encoder():
    torch.manual_seed(2)
    shapes, mix_list = mixes(4)
    model = DeformableEncoder(256, 8, 1024, 0.0, 0.0, num_layers=2).to(DEV)
    packing, _, (x, pos, ref) = _batch(mix_list[0], shapes, 256, torch.Generator().manual_seed(9))
    static_x = x.clone().requires_grad_(True)

    def step():
        out = model(static_x, query_pos=pos, reference_points=ref, spatial_shapes=packing.spatial_shapes,
                    level_start_index=packing.level_start_index, packing=packing)
        out.square().sum().backward()
        return out

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    model.zero_grad(set_to_none=False)
    static_x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = step()
    graph.replay()
    torch.cuda.synchronize()
    got_out, got_grad = static_out.clone(), static_x.grad.clone()
    eager_x = x.clone().requires_grad_(True)
    eager = model(eager_x, query_pos=pos, reference_points=ref, spatial_shapes=packing.spatial_shapes,
                  level_start_index=packing.level_start_index, packing=packing)
    eager.square().sum().backward()
    assert torch.equal(got_out, eager)
    torch.testing.assert_close(got_grad, eager_x.grad, rtol=1e-4, atol=1e-4)

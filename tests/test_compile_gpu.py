"""torch.compile / torch.export of the module paths on the GPU: opcheck of every custom op, fullgraph compilation
(aot_eager) of the module, the encoder layer / 6-layer encoder, the cross-attention block and DCNv3 against eager,
inductor on the encoder layer, CUDA-graph replay (reduce-overhead), torch.export, and the deterministic switch."""

import pytest
import torch

from ir_ads_b200 import _lib, set_deterministic
from ir_ads_b200.dcnv3 import DCNv3
from ir_ads_b200.encoder import (DeformableCrossAttentionBlock, DeformableEncoder, DeformableEncoderLayer,
                                 get_reference_points)
from ir_ads_b200.module import MultiScaleDeformableAttention
from ir_ads_b200.packing import PackedLevels, pack_levels, packed_reference_points

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
OPS = torch.ops.ir_ads_b200
SHAPES = [(12, 17), (6, 9), (3, 5), (2, 3)]
EXTENTS = [SHAPES[:], [(1, 1)] * 4, [(8, 8), (4, 4), (2, 2), (1, 2)]]
AOT_ONLY = ("test_schema", "test_autograd_registration", "test_faketensor", "test_aot_dispatch_dynamic")
NO_AOT = ("test_schema", "test_autograd_registration", "test_faketensor")


def rand(*shape, dtype=torch.float32, gen, scale=1.0, grad=True):
    return (torch.randn(*shape, generator=gen) * scale).to(DEV, dtype).requires_grad_(grad)


@pytest.fixture(autouse=True)
def _fresh():
    torch._dynamo.reset()
    set_deterministic(False)
    yield
    set_deterministic(False)
    torch._dynamo.reset()


# ---- 1. opcheck ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("vdt,adt", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16)])
@pytest.mark.parametrize("masked,need_ref", [(True, False), (False, True)])
def test_opcheck_msda_fused(vdt, adt, masked, need_ref):
    gen = torch.Generator().manual_seed(1)
    L, H, D, P, B, Q = 4, 4, 32, 4, 2, 20
    S = sum(h * w for h, w in SHAPES)
    shapes = torch.tensor(SHAPES, dtype=torch.int64, device=DEV)
    lsi = torch.tensor([0, 204, 258, 273], dtype=torch.int64, device=DEV)
    mask = (torch.rand(B, S, generator=gen) < 0.2).to(DEV) if masked else None
    args = (rand(B, S, H, D, dtype=vdt, gen=gen), shapes, lsi, rand(B, Q, H, L, P, 2, dtype=adt, gen=gen),
            rand(B, Q, H, L * P, dtype=adt, gen=gen), torch.rand(B, Q, L, 4, generator=gen).to(DEV).requires_grad_(need_ref),
            mask)
    # float reds: the eager / AOT comparison could see another summation order; the deterministic route cannot
    torch.library.opcheck(OPS.msda_fused.default, args + (False,), test_utils=NO_AOT)
    torch.library.opcheck(OPS.msda_fused.default, args + (True,), test_utils=AOT_ONLY)


def _packed_args(packing, vdt, adt, gen, need_ref=False, H=4, D=32, P=4):
    T_v, T_q, L = packing.total_value, packing.total_query, packing.num_levels
    return (rand(T_v, H, D, dtype=vdt, gen=gen), rand(T_q, H, L, P, 2, dtype=adt, gen=gen),
            rand(T_q, H, L * P, dtype=adt, gen=gen), torch.rand(T_q, L, 2, generator=gen).to(DEV).requires_grad_(need_ref),
            packing.meta, packing.spatial_shapes, packing.level_start_index, packing.value_index, packing.query_index,
            packing.padding_mask, packing.max_value, packing.max_query, packing.query_pad)


@pytest.mark.parametrize("cross", [False, True])
def test_opcheck_msda_packed(cross):
    gen = torch.Generator().manual_seed(2)
    packing = PackedLevels(EXTENTS, SHAPES, DEV)
    packing = packing.cross(16) if cross else packing
    args = _packed_args(packing, torch.float32, torch.float32, gen, need_ref=cross)
    torch.library.opcheck(OPS.msda_packed.default, args + (False,), test_utils=NO_AOT)
    torch.library.opcheck(OPS.msda_packed.default, args + (True,), test_utils=AOT_ONLY)


@pytest.mark.parametrize("da,db", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16),
                                   (torch.bfloat16, torch.float32), (torch.float16, torch.float32)])
def test_opcheck_add_layer_norm(da, db):
    gen = torch.Generator().manual_seed(3)
    args = (rand(3, 5, 64, dtype=da, gen=gen), rand(3, 5, 64, dtype=db, gen=gen), rand(64, gen=gen),
            rand(64, gen=gen), 1e-5)
    torch.library.opcheck(OPS.add_layer_norm.default, args, test_utils=AOT_ONLY)


@pytest.mark.parametrize("vdt,adt", [(torch.float32, torch.float32), (torch.float16, torch.float16)])
def test_opcheck_dcnv3_fused(vdt, adt):
    gen = torch.Generator().manual_seed(4)
    N, H, W, G, gc, k = 2, 7, 9, 4, 16, 3
    args = (rand(N, H, W, G * gc, dtype=vdt, gen=gen), rand(N, H, W, G * k * k * 2, dtype=adt, gen=gen),
            rand(N, H, W, G * k * k, dtype=adt, gen=gen), k, k, 1, 1, 1, 1, 1, 1, G, gc, 1.0)
    torch.library.opcheck(OPS.dcnv3_fused.default, args + (False,), test_utils=NO_AOT)
    torch.library.opcheck(OPS.dcnv3_fused.default, args + (True,), test_utils=AOT_ONLY)


# ---- 2. fullgraph aot_eager against eager ---------------------------------------------------------------------------
def _perturb(model, seed):
    gen = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if "sampling_offsets.weight" in name or "attention_weights.weight" in name or name.endswith("offset.weight") \
                    or name.endswith("mask.weight"):
                p.copy_(torch.randn(p.shape, generator=gen) * 0.02)
    return model


def _run(fn, inputs, params, autocast):
    for t in list(inputs) + list(params):
        t.grad = None
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        out = fn(*inputs)
    out.float().square().sum().backward()
    return out.detach().clone(), [t.grad.clone() for t in list(inputs) + list(params) if t.requires_grad]


def _check(model, make_fn, inputs, autocast, deterministic):
    """forward bit for bit; every gradient bit for bit in deterministic mode, else within float-red order"""
    set_deterministic(deterministic)
    params = list(model.parameters())
    eager = _run(make_fn(model), inputs, params, autocast)
    compiled = torch.compile(make_fn(model), fullgraph=True, backend="aot_eager")
    got = _run(compiled, inputs, params, autocast)
    assert torch.equal(got[0], eager[0])
    for g, e in zip(got[1], eager[1]):
        if deterministic:
            assert torch.equal(g, e)
        else:
            torch.testing.assert_close(g.float(), e.float(), rtol=1e-4 if not autocast else 2e-2,
                                       atol=1e-5 * (1 + float(e.float().abs().max())) * (1 if not autocast else 100))


def _encoder_inputs(gen, C=256, B=2):
    S = sum(h * w for h, w in SHAPES)
    packing = PackedLevels([SHAPES[:], EXTENTS[2]], SHAPES, DEV)
    q = rand(B, S, C, gen=gen)
    pos = rand(B, S, C, gen=gen, grad=False)
    ref = get_reference_points(SHAPES, packing.valid_ratios, DEV)
    return packing, q, pos, ref


def _encoder_fn(packing):
    def make(model):
        def fn(q, pos, ref):
            return model(q, query_pos=pos, reference_points=ref, spatial_shapes=packing.spatial_shapes,
                         level_start_index=packing.level_start_index, level_shapes=packing.level_shapes,
                         query_key_padding_mask=packing.padding_mask)
        return fn
    return make


@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("which", ["module", "layer", "encoder6"])
def test_fullgraph_padded(which, autocast, deterministic):
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(5)
    packing, q, pos, ref = _encoder_inputs(gen)
    if which == "module":
        model = MultiScaleDeformableAttention(256, 8, 4, 4, dropout=0.0, batch_first=True).to(DEV)
        ref = ref.detach()

        def make(m):
            def fn(q, pos, ref):
                return m(q, query_pos=pos, key_padding_mask=packing.padding_mask, reference_points=ref,
                         spatial_shapes=packing.spatial_shapes, level_start_index=packing.level_start_index,
                         level_shapes=packing.level_shapes)
            return fn
    else:
        model = (DeformableEncoderLayer(256, 8, 1024, 0.0, 0.0) if which == "layer" else
                 DeformableEncoder(256, 8, 1024, 0.0, 0.0, num_layers=6)).to(DEV)
        make = _encoder_fn(packing)
    _check(_perturb(model, 1), make, (q, pos, ref), autocast, deterministic)


@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("which", ["module", "layer", "encoder6"])
def test_fullgraph_packed(which, autocast, deterministic):
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(6)
    packing = PackedLevels(EXTENTS, SHAPES, DEV)
    feats = [torch.randn(3, 256, h, w, generator=gen).to(DEV) for h, w in SHAPES]
    x, pos = pack_levels(feats, packing, feats)
    x = x.clone().requires_grad_(True)
    ref = packed_reference_points(packing)
    if which == "module":
        model = MultiScaleDeformableAttention(256, 8, 4, 4, dropout=0.0, batch_first=True).to(DEV)

        def make(m):
            return lambda q, p, r: m(q, query_pos=p, reference_points=r, packing=packing)
    else:
        model = (DeformableEncoderLayer(256, 8, 1024, 0.0, 0.0) if which == "layer" else
                 DeformableEncoder(256, 8, 1024, 0.0, 0.0, num_layers=6)).to(DEV)

        def make(m):
            return lambda q, p, r: m(q, query_pos=p, reference_points=r, packing=packing)
    _check(_perturb(model, 2), make, (x, pos, ref), autocast, deterministic)


@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("autocast", [False, True])
@pytest.mark.parametrize("packed", [False, True])
def test_fullgraph_cross_attention_block(packed, autocast, deterministic):
    torch.manual_seed(1)
    gen = torch.Generator().manual_seed(7)
    packing, mem, _, _ = _encoder_inputs(gen)
    block = _perturb(DeformableCrossAttentionBlock(256, 8, 0.0).to(DEV), 3)
    B, Q = 2, 40
    query, qpos, boxes = rand(B, Q, 256, gen=gen), rand(B, Q, 256, gen=gen, grad=False), rand(B, Q, 4, gen=gen,
                                                                                           grad=False).sigmoid()
    if packed:
        packing.cross(Q)                                       # the decoder form is built once, outside the graph
        mem = mem.detach().reshape(-1, 256)[packing.value_index].requires_grad_(True)

    def make(m):
        def fn(query, mem):
            return m(query, mem, qpos, boxes, packing.valid_ratios, packing.spatial_shapes, packing.level_start_index,
                     key_padding_mask=None if packed else packing.padding_mask, packing=packing if packed else None,
                     level_shapes=packing.level_shapes)
        return fn
    _check(block, make, (query, mem), autocast, deterministic)


@pytest.mark.parametrize("deterministic", [False, True])
@pytest.mark.parametrize("autocast", [False, True])
def test_fullgraph_dcnv3(autocast, deterministic):
    torch.manual_seed(2)
    gen = torch.Generator().manual_seed(8)
    model = _perturb(DCNv3(64, group=4).to(DEV), 4)
    x = rand(2, 14, 18, 64, gen=gen)
    _check(model, lambda m: (lambda x: m(x)), (x,), autocast, deterministic)


# ---- 3. inductor --------------------------------------------------------------------------------------------------
def test_inductor_encoder_layer():
    torch.manual_seed(3)
    gen = torch.Generator().manual_seed(9)
    packing, q, pos, ref = _encoder_inputs(gen)
    layer = _perturb(DeformableEncoderLayer(256, 8, 1024, 0.0, 0.0).to(DEV), 5)
    fn = _encoder_fn(packing)(layer)
    explain = torch._dynamo.explain(fn)(q, pos, ref)
    assert explain.graph_break_count == 0 and explain.graph_count == 1
    torch._dynamo.reset()
    params = list(layer.parameters())
    eager = _run(fn, (q, pos, ref), params, False)
    got = _run(torch.compile(fn, backend="inductor", fullgraph=True), (q, pos, ref), params, False)
    torch.testing.assert_close(got[0], eager[0], rtol=1e-4, atol=1e-4)
    for g, e in zip(got[1], eager[1]):
        torch.testing.assert_close(g, e, rtol=1e-4, atol=1e-4 * (1 + float(e.abs().max())))


# ---- 4. CUDA graphs ----------------------------------------------------------------------------------------------
def test_reduce_overhead_encoder_replays():
    torch.manual_seed(4)
    gen = torch.Generator().manual_seed(10)
    packing, q, pos, ref = _encoder_inputs(gen)
    enc = _perturb(DeformableEncoder(256, 8, 1024, 0.0, 0.0, num_layers=6).to(DEV), 6)
    fn = _encoder_fn(packing)(enc)
    compiled = torch.compile(fn, mode="reduce-overhead", fullgraph=True)
    for step in range(4):                                       # warm-up, record, then two replays on new inputs
        x = rand(*q.shape, gen=gen)
        torch.compiler.cudagraph_mark_step_begin()
        out = compiled(x, pos, ref)
        gy = torch.randn(out.shape, generator=gen).to(DEV)
        (gx,) = torch.autograd.grad(out, x, gy)
        out, gx = out.clone(), gx.clone()
        x_e = x.detach().clone().requires_grad_(True)
        out_e = fn(x_e, pos, ref)
        (gx_e,) = torch.autograd.grad(out_e, x_e, gy)
        torch.testing.assert_close(out, out_e, rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(gx, gx_e, rtol=1e-4, atol=1e-4 * (1 + float(gx_e.abs().max())))


# ---- 5. export ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("autocast", [False, True])
def test_export_encoder_layer(autocast):
    torch.manual_seed(5)
    gen = torch.Generator().manual_seed(11)
    packing, q, pos, ref = _encoder_inputs(gen)
    layer = _perturb(DeformableEncoderLayer(256, 8, 1024, 0.0, 0.0).to(DEV), 7).eval()
    q = q.detach()
    kw = dict(query_pos=pos, reference_points=ref, spatial_shapes=packing.spatial_shapes,
              level_start_index=packing.level_start_index, level_shapes=packing.level_shapes,
              query_key_padding_mask=packing.padding_mask)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        ep = torch.export.export(layer, (q,), kwargs=kw)
        targets = {str(n.target) for n in ep.graph.nodes}
        assert "ir_ads_b200.msda_fused.default" in targets and "ir_ads_b200.add_layer_norm.default" in targets
        got = ep.module()(q, **kw)
        want = layer(q, **kw)
    assert torch.equal(got, want)


# ---- 6. the deterministic switch -----------------------------------------------------------------------------------
def test_toggling_deterministic_recompiles():
    torch.manual_seed(6)
    gen = torch.Generator().manual_seed(12)
    packing, q, pos, ref = _encoder_inputs(gen)
    layer = _perturb(DeformableEncoderLayer(256, 8, 1024, 0.0, 0.0).to(DEV), 8)
    fn = _encoder_fn(packing)(layer)
    compiled = torch.compile(fn, fullgraph=True, backend="aot_eager")
    params = list(layer.parameters())

    def step(f):
        n0 = _lib.launch_count()
        res = _run(f, (q, pos, ref), params, False)
        torch.cuda.synchronize()
        return res, _lib.launch_count() - n0

    _, n_red_eager = step(fn)
    _, n_red = step(compiled)
    set_deterministic(True)
    (out1, g1), n_det = step(compiled)
    (out2, g2), _ = step(compiled)
    (out_e, g_e), n_det_eager = step(fn)
    assert n_red == n_red_eager and n_det == n_det_eager and n_det != n_red
    assert torch.equal(out1, out2) and torch.equal(out1, out_e)
    for a, b, c in zip(g1, g2, g_e):
        assert torch.equal(a, b) and torch.equal(a, c)

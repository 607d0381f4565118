"""The torch.library custom ops of ir_ads_b200/ops.py without a GPU: schemas, the library staying unloaded, and the
fake kernels (shapes / dtypes of outputs and gradients, through the registered autograd) on meta tensors."""
import os
import subprocess
import sys

import pytest
import torch
from torch._subclasses.fake_tensor import FakeTensorMode

import ir_ads_b200  # noqa: F401
from ir_ads_b200.packing import PackedLevels

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OPS = torch.ops.ir_ads_b200

SCHEMAS = {
    "msda_fused": "ir_ads_b200::msda_fused(Tensor value, Tensor spatial_shapes, Tensor level_start_index, "
                  "Tensor sampling_offsets, Tensor attn_logits, Tensor reference_points, Tensor? key_padding_mask, "
                  "bool deterministic) -> Tensor",
    "msda_fused_backward": "ir_ads_b200::msda_fused_backward(Tensor grad_output, Tensor value, Tensor spatial_shapes, "
                           "Tensor level_start_index, Tensor sampling_offsets, Tensor attn_logits, "
                           "Tensor reference_points, Tensor? key_padding_mask, bool deterministic, bool need_value, "
                           "bool need_ref) -> (Tensor?, Tensor, Tensor, Tensor?)",
    "msda_packed": "ir_ads_b200::msda_packed(Tensor value, Tensor sampling_offsets, Tensor attn_logits, "
                   "Tensor reference_points, Tensor meta, Tensor spatial_shapes, Tensor level_start_index, "
                   "Tensor value_index, Tensor query_index, Tensor padding_mask, SymInt max_value, SymInt max_query, "
                   "SymInt query_pad, bool deterministic) -> Tensor",
    "msda_packed_backward": "ir_ads_b200::msda_packed_backward(Tensor grad_output, Tensor value, "
                            "Tensor sampling_offsets, Tensor attn_logits, Tensor reference_points, Tensor meta, "
                            "Tensor spatial_shapes, Tensor level_start_index, Tensor value_index, Tensor query_index, "
                            "Tensor padding_mask, SymInt max_value, SymInt max_query, SymInt query_pad, "
                            "bool deterministic, bool need_value, bool need_ref) -> (Tensor?, Tensor, Tensor, Tensor?)",
    "add_layer_norm": "ir_ads_b200::add_layer_norm(Tensor a, Tensor b, Tensor weight, Tensor bias, float eps) "
                      "-> (Tensor, Tensor, Tensor)",
    "add_layer_norm_backward": "ir_ads_b200::add_layer_norm_backward(Tensor grad_y, Tensor a, Tensor b, "
                               "Tensor weight, Tensor mean, Tensor rstd) -> (Tensor, Tensor?, Tensor, Tensor)",
    "dcnv3_fused": "ir_ads_b200::dcnv3_fused(Tensor input, Tensor offset, Tensor mask_logits, SymInt kernel_h, "
                   "SymInt kernel_w, SymInt stride_h, SymInt stride_w, SymInt pad_h, SymInt pad_w, SymInt dilation_h, "
                   "SymInt dilation_w, SymInt group, SymInt group_channels, float offset_scale, bool deterministic) "
                   "-> Tensor",
    "dcnv3_fused_backward": "ir_ads_b200::dcnv3_fused_backward(Tensor grad_output, Tensor input, Tensor offset, "
                            "Tensor mask_logits, SymInt kernel_h, SymInt kernel_w, SymInt stride_h, SymInt stride_w, "
                            "SymInt pad_h, SymInt pad_w, SymInt dilation_h, SymInt dilation_w, SymInt group, "
                            "SymInt group_channels, float offset_scale, bool deterministic) -> (Tensor, Tensor, Tensor)",
}

VALUE_AUX = [(torch.float32, torch.float32), (torch.bfloat16, torch.float32), (torch.float16, torch.float32),
             (torch.bfloat16, torch.bfloat16), (torch.float16, torch.float16)]


@pytest.mark.parametrize("name", sorted(SCHEMAS))
def test_schema(name):
    assert str(getattr(OPS, name).default._schema) == SCHEMAS[name]
    assert not getattr(OPS, name).default._schema.is_mutable


def test_registering_the_ops_loads_no_library():
    code = ("import ir_ads_b200, ir_ads_b200.ops, torch; from ir_ads_b200 import _lib; "
            "assert hasattr(torch.ops.ir_ads_b200, 'msda_fused'); assert _lib._lib is None; "
            "assert 'libmsda_b200' not in open('/proc/self/maps').read()")
    subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT)


def _grads(out, inputs):
    """gradients through the registered autograd formula (the backward op's fake kernel)"""
    wanted = [t for t in inputs if t.requires_grad]
    got = iter(torch.autograd.grad(out, wanted, torch.ones_like(out)))
    return [next(got) if t.requires_grad else None for t in inputs]


def _assert_like(grad, t):
    assert grad.shape == t.shape and grad.dtype == t.dtype


@pytest.mark.parametrize("need_ref", [False, True])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("ref_dim", [2, 4])
@pytest.mark.parametrize("vdt,adt", VALUE_AUX)
def test_msda_fused_fake(vdt, adt, ref_dim, masked, need_ref):
    B, S, H, D, L, P, Q = 2, 85, 8, 32, 4, 4, 30
    with FakeTensorMode():
        value = torch.empty(B, S, H, D, dtype=vdt, device="meta", requires_grad=True)
        shapes = torch.empty(L, 2, dtype=torch.int64, device="meta")
        lsi = torch.empty(L, dtype=torch.int64, device="meta")
        off = torch.empty(B, Q, H, L, P, 2, dtype=adt, device="meta", requires_grad=True)
        logits = torch.empty(B, Q, H, L * P, dtype=adt, device="meta", requires_grad=True)
        ref = torch.empty(B, Q, L, ref_dim, device="meta", requires_grad=need_ref)
        mask = torch.empty(B, S, dtype=torch.bool, device="meta") if masked else None
        for det in (False, True):
            out = OPS.msda_fused(value, shapes, lsi, off, logits, ref, mask, det)
            assert out.shape == (B, Q, H * D) and out.dtype == vdt
            g = _grads(out, [value, off, logits, ref])
            for grad, t in zip(g, (value, off, logits, ref)):
                if t.requires_grad:
                    _assert_like(grad, t)
            if not need_ref:
                assert g[3] is None
    frozen = OPS.msda_fused_backward.default
    with FakeTensorMode():
        args = [torch.empty(s, dtype=d, device="meta") for s, d in (
            ((B, Q, H * D), vdt), ((B, S, H, D), vdt), ((L, 2), torch.int64), ((L,), torch.int64),
            ((B, Q, H, L, P, 2), adt), ((B, Q, H, L * P), adt), ((B, Q, L, ref_dim), torch.float32))]
        gv, go, gl, gr = frozen(*args, None, False, False, need_ref)
        assert gv is None and (gr is not None) == need_ref
        _assert_like(go, args[4]), _assert_like(gl, args[5])


@pytest.mark.parametrize("cross", [False, True])
@pytest.mark.parametrize("ref_dim", [2, 4])
@pytest.mark.parametrize("vdt,adt", VALUE_AUX)
def test_msda_packed_fake(vdt, adt, ref_dim, cross):
    shapes = [(12, 17), (6, 9), (3, 5), (2, 3)]
    packing = PackedLevels([shapes, [(1, 1)] * 4, [(8, 8), (4, 4), (2, 2), (1, 2)]], shapes, "cpu")
    if cross:
        packing = packing.cross(30)
    H, D, L, P = 8, 32, 4, 4
    T_v, T_q = packing.total_value, packing.total_query
    with FakeTensorMode(allow_non_fake_inputs=True) as mode:
        tables = [mode.from_tensor(t.to("meta")) for t in (packing.meta, packing.spatial_shapes,
                                                             packing.level_start_index, packing.value_index,
                                                             packing.query_index, packing.padding_mask)]
        value = torch.empty(T_v, H, D, dtype=vdt, device="meta", requires_grad=True)
        off = torch.empty(T_q, H, L, P, 2, dtype=adt, device="meta", requires_grad=True)
        logits = torch.empty(T_q, H, L * P, dtype=adt, device="meta", requires_grad=True)
        ref = torch.empty(T_q, L, ref_dim, device="meta", requires_grad=True)
        out = OPS.msda_packed(value, off, logits, ref, *tables, packing.max_value, packing.max_query,
                              packing.query_pad, False)
        assert out.shape == (T_q, H * D) and out.dtype == vdt
        for grad, t in zip(_grads(out, [value, off, logits, ref]), (value, off, logits, ref)):
            _assert_like(grad, t)


@pytest.mark.parametrize("dtypes", [(torch.float32, torch.float32), (torch.bfloat16, torch.bfloat16),
                                    (torch.float16, torch.float16), (torch.bfloat16, torch.float32),
                                    (torch.float16, torch.float32)])
def test_add_layer_norm_fake(dtypes):
    da, db = dtypes
    with FakeTensorMode():
        a = torch.empty(2, 7, 256, dtype=da, device="meta", requires_grad=True)
        b = torch.empty(2, 7, 256, dtype=db, device="meta", requires_grad=True)
        w = torch.empty(256, device="meta", requires_grad=True)
        bias = torch.empty(256, device="meta", requires_grad=True)
        y, mean, rstd = OPS.add_layer_norm(a, b, w, bias, 1e-5)
        assert y.shape == a.shape and y.dtype == db           # the mixed form's result is float32
        assert mean.shape == rstd.shape == (14,) and mean.dtype == rstd.dtype == torch.float32
        for grad, t in zip(_grads(y, [a, b, w, bias]), (a, b, w, bias)):
            _assert_like(grad, t)
        gb, ga, gw, gbias = OPS.add_layer_norm_backward(torch.empty_like(y), a, b, w, mean, rstd)
        assert (ga is None) == (da == db) and gb.dtype == db and gw.dtype == gbias.dtype == torch.float32


@pytest.mark.parametrize("vdt,adt", VALUE_AUX)
def test_dcnv3_fused_fake(vdt, adt):
    N, H, W, G, gc, k = 2, 9, 11, 4, 16, 3
    with FakeTensorMode():
        x = torch.empty(N, H, W, G * gc, dtype=vdt, device="meta", requires_grad=True)
        off = torch.empty(N, H, W, G * k * k * 2, dtype=adt, device="meta", requires_grad=True)
        logits = torch.empty(N, H, W, G * k * k, dtype=adt, device="meta", requires_grad=True)
        for det in (False, True):
            out = OPS.dcnv3_fused(x, off, logits, k, k, 1, 1, 1, 1, 1, 1, G, gc, 1.0, det)
            assert out.shape == (N, H, W, G * gc) and out.dtype == vdt
            for grad, t in zip(_grads(out, [x, off, logits]), (x, off, logits)):
                _assert_like(grad, t)


def test_fake_kernels_load_no_library():
    code = ("import torch, ir_ads_b200; from ir_ads_b200 import _lib; "
            "from torch._subclasses.fake_tensor import FakeTensorMode\n"
            "with FakeTensorMode():\n"
            "    a = torch.empty(4, 64, device='meta', requires_grad=True)\n"
            "    w = torch.empty(64, device='meta')\n"
            "    y = torch.ops.ir_ads_b200.add_layer_norm(a, a, w, w, 1e-5)[0]\n"
            "    y.sum().backward()\n"
            "assert _lib._lib is None and 'libmsda_b200' not in open('/proc/self/maps').read()")
    subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT)

"""CPU-side checks of deformable convolution (msda_dcnv2_im2col / msda_dcnv2_col2im, ir_ads_b200.dcnv2): exported and
declared, argument / alignment / dtype-tag errors and empty problems answered before any device work, the workspace
formula, a strict C99 program that links the entry points, the detectron2 module surface, CPU tensors refused, the
custom ops' fake kernels on meta tensors, and the library left unloaded by the import.  No GPU work."""
import ctypes
import os
import shutil
import subprocess
import sys

import pytest
import torch

from ir_ads_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NULL = ctypes.c_void_p(0)
INVALID, UNSUPPORTED, WORKSPACE = 1, 2, 3
P = ctypes.c_void_p(0x10000)   # a 16-byte aligned address that is never dereferenced: every call here fails first


def geom(B=2, C=64, H=9, W=11, k=3, s=1, p=1, d=1, groups=1, dg=1, Ho=None, Wo=None):
    size = (lambda n: (n + 2 * p - (max(d, 1) * (k - 1) + 1)) // max(s, 1) + 1)   # the C ABI rejects s, d < 1 first
    ho = size(H) if Ho is None else Ho
    wo = size(W) if Wo is None else Wo
    return [B, C, H, W, ho, wo, k, k, s, s, p, p, d, d, groups, dg]


def im2col(g, inp=P, off=P, mask=P, cols=P, dtype=_lib.MSDA_F32, flags=0):
    return _lib.lib().msda_dcnv2_im2col(NULL, inp, off, mask, *g, cols, dtype, flags)


def col2im(g, gcols=P, inp=P, off=P, mask=P, gi=P, goff=P, gm=P, ws=P, ws_bytes=1 << 40, dtype=_lib.MSDA_F32,
           flags=0):
    return _lib.lib().msda_dcnv2_col2im(NULL, gcols, inp, off, mask, *g, gi, goff, gm, ws, ws_bytes, dtype, flags)


def msg():
    return _lib.lib().msda_last_error_message()


def test_entry_points_are_exported_and_declared():
    h = _lib.lib()
    names = ("msda_dcnv2_im2col", "msda_dcnv2_col2im", "msda_dcnv2_col2im_workspace_bytes")
    assert all(hasattr(h, n) for n in names)
    header = open(os.path.join(ROOT, "include", "msda.h")).read()
    assert all(f"{n}(" in header for n in names)
    assert h.msda_abi_version() == 3 == _lib.ABI_VERSION   # additions only
    import ir_ads_b200
    for n in ("DeformConv", "ModulatedDeformConv", "deform_conv", "modulated_deform_conv"):
        assert n in ir_ads_b200.__all__ and hasattr(ir_ads_b200, n)


@pytest.mark.parametrize("call", [im2col, col2im])
def test_bad_geometry_and_tags(call):
    n0 = _lib.launch_count()
    for g in (geom(k=0), geom(s=0), geom(d=0), geom(p=-1), geom(B=-1), geom(C=-1), geom(groups=0), geom(dg=0),
              geom(H=0), geom(Ho=3), geom(Wo=99)):
        assert call(g) == INVALID, g
        assert b"dcnv2" in msg()
    assert call(geom(C=64, groups=3)) == INVALID and b"divisible" in msg()
    assert call(geom(C=64, dg=5)) == INVALID and b"divisible" in msg()
    assert call(geom(H=1, W=1, p=0)) == INVALID                          # the input is smaller than the kernel
    for tag in (-1, 6, 99):
        assert call(geom(), dtype=tag) == INVALID and b"dtype tag" in msg()
    assert _lib.launch_count() == n0


def test_null_and_misaligned_pointers():
    n0 = _lib.launch_count()
    odd = ctypes.c_void_p(0x10004)
    assert im2col(geom(), inp=NULL) == INVALID and b"null" in msg()
    assert im2col(geom(), cols=NULL) == INVALID
    for kw, name in (({"inp": odd}, b"input"), ({"off": odd}, b"offset"), ({"mask": odd}, b"mask"),
                     ({"cols": odd}, b"columns")):
        assert im2col(geom(), **kw) == INVALID and name in msg() and b"16-byte" in msg(), kw
    assert col2im(geom(), goff=NULL) == INVALID and b"grad_offset" in msg()
    assert col2im(geom(), gm=NULL) == INVALID                            # a mask needs its gradient
    assert col2im(geom(), gi=NULL) == INVALID and b"null" in msg()
    for kw, name in (({"gcols": odd}, b"grad_columns"), ({"gi": odd}, b"grad_input"), ({"goff": odd}, b"grad_offset"),
                     ({"gm": odd}, b"grad_mask"), ({"ws": odd}, b"workspace")):
        assert col2im(geom(), **kw) == INVALID and name in msg() and b"16-byte" in msg(), kw
    assert _lib.launch_count() == n0


def test_deterministic_backward_is_refused():
    """grad_input uses float reds: MSDA_FLAG_DETERMINISTIC is refused before any device work, empty problems too."""
    n0 = _lib.launch_count()
    assert col2im(geom(), flags=_lib.FLAG_DETERMINISTIC) == UNSUPPORTED and b"deterministic" in msg()
    assert col2im(geom(B=0), flags=_lib.FLAG_DETERMINISTIC) == UNSUPPORTED
    assert im2col(geom(B=0), flags=_lib.FLAG_DETERMINISTIC) == 0      # the forward ignores the flag
    assert _lib.launch_count() == n0


def test_workspace_is_required_for_16_bit_inputs():
    n0 = _lib.launch_count()
    assert col2im(geom(), dtype=_lib.MSDA_BF16, ws=NULL) == WORKSPACE
    assert col2im(geom(), dtype=_lib.MSDA_F16_AUX16, ws_bytes=100) == WORKSPACE
    assert b"workspace" in msg()
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("dtype", [_lib.MSDA_F32, _lib.MSDA_F64, _lib.MSDA_BF16, _lib.MSDA_F16, _lib.MSDA_BF16_AUX16,
                                   _lib.MSDA_F16_AUX16])
def test_empty_problems_do_nothing(dtype):
    n0 = _lib.launch_count()
    for flags in (0, _lib.FLAG_FORCE_GENERIC):
        assert im2col(geom(B=0), NULL, NULL, NULL, NULL, dtype=dtype, flags=flags) == 0
        assert im2col(geom(C=0), NULL, NULL, NULL, NULL, dtype=dtype, flags=flags) == 0
        assert col2im(geom(B=0), NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, 0, dtype=dtype, flags=flags) == 0
    assert _lib.launch_count() == n0


def test_workspace_formula():
    ws = _lib.lib().msda_dcnv2_col2im_workspace_bytes
    g = geom(B=3, C=48, H=13, W=17)
    for tag in (_lib.MSDA_BF16, _lib.MSDA_F16, _lib.MSDA_BF16_AUX16, _lib.MSDA_F16_AUX16):
        assert ws(*g, tag, 0) == 3 * 13 * 17 * 48 * 4
    assert ws(*g, _lib.MSDA_F32, 0) == 0 and ws(*g, _lib.MSDA_F64, 0) == 0
    assert ws(*geom(Ho=2), _lib.MSDA_BF16, 0) == 0                     # invalid geometry
    assert ws(*geom(B=0), _lib.MSDA_BF16, 0) == 0


def test_slim_builds_stub_the_dcnv2_entry_points():
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    src = os.path.join(ROOT, "ir_ads_b200", "csrc", "msda_dcnv2.cu")
    res = subprocess.run([nvcc, "-std=c++17", "-E", "-DMSDA_EXP_SLIM", "-x", "cu", src], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    for fn in ("dcnv2_im2col", "dcnv2_col2im"):
        body = res.stdout[res.stdout.rindex(f"int {fn}("):]
        body = body[:body.index("}")]
        assert "slim build: no DCNv2 kernels" in body and "<<<" not in body


def test_c_program_calls_the_dcnv2_entry_points(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "dcnv2.c"
    src.write_text(r'''
#include <stdio.h>
#include "msda.h"
int main(void) {
  /* batch 0: MSDA_OK, no device work */
  if (msda_dcnv2_im2col(NULL, NULL, NULL, NULL, 0, 64, 9, 11, 9, 11, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, NULL, MSDA_F32,
                        0u) != MSDA_OK) return 1;
  if (msda_dcnv2_col2im(NULL, NULL, NULL, NULL, NULL, 0, 64, 9, 11, 9, 11, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, NULL, NULL,
                        NULL, NULL, 0, MSDA_BF16_AUX16, 0u) != MSDA_OK) return 2;
  /* wrong output size, deterministic backward */
  if (msda_dcnv2_im2col(NULL, NULL, NULL, NULL, 2, 64, 9, 11, 8, 11, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, NULL, MSDA_F32,
                        0u) != MSDA_ERR_INVALID_ARGUMENT) return 3;
  if (msda_dcnv2_col2im(NULL, NULL, NULL, NULL, NULL, 2, 64, 9, 11, 9, 11, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, NULL, NULL,
                        NULL, NULL, 0, MSDA_F16, MSDA_FLAG_DETERMINISTIC) != MSDA_ERR_UNSUPPORTED) return 4;
  if (msda_dcnv2_col2im_workspace_bytes(2, 64, 9, 11, 9, 11, 3, 3, 1, 1, 1, 1, 1, 1, 1, 1, MSDA_F16, 0u) !=
      (size_t)2 * 9 * 11 * 64 * 4) return 5;
  printf("dcnv2 abi ok\n");
  return 0;
}
''')
    exe = tmp_path / "dcnv2"
    lib_dir = os.path.dirname(_lib.LIB_PATH)
    res = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I",
                          os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-L", lib_dir, "-l:libmsda_b200.so",
                          f"-Wl,-rpath,{lib_dir}"], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0 and "dcnv2 abi ok" in run.stdout, (run.returncode, run.stdout, run.stderr)


def test_module_surface_matches_detectron2():
    from ir_ads_b200 import DeformConv, ModulatedDeformConv
    torch.manual_seed(0)
    m = ModulatedDeformConv(64, 32, 3, stride=2, padding=1, dilation=1, groups=2, deformable_groups=4)
    assert [n for n, _ in m.named_parameters()] == ["weight", "bias"]
    assert tuple(m.weight.shape) == (32, 32, 3, 3) and tuple(m.bias.shape) == (32,)
    assert torch.count_nonzero(m.bias) == 0                              # constant 0
    bound = (6.0 / (32 * 9)) ** 0.5                                       # kaiming_uniform_, relu gain, fan_in
    assert m.weight.abs().max() <= bound and m.weight.abs().max() > 0.9 * bound
    assert (m.kernel_size, m.stride, m.padding, m.dilation) == ((3, 3), (2, 2), (1, 1), (1, 1))
    assert (m.groups, m.deformable_groups, m.with_bias) == (2, 4, True)
    assert ModulatedDeformConv(16, 16, (3, 1), bias=False).bias is None
    d = DeformConv(16, 8, 3, padding=1)
    assert [n for n, _ in d.named_parameters()] == ["weight"] and d.bias is None
    with pytest.raises(AssertionError):
        DeformConv(16, 8, 3, bias=True)
    with pytest.raises(AssertionError):
        ModulatedDeformConv(16, 8, 3, groups=3)
    norm = torch.nn.BatchNorm2d(8)
    assert DeformConv(16, 8, 3, norm=norm, activation=torch.relu).norm is norm
    sd = ModulatedDeformConv(64, 32, 3, groups=2, deformable_groups=4).state_dict()
    m.load_state_dict(sd)                                                 # detectron2 checkpoints load as they are


def test_cpu_tensors_raise():
    from ir_ads_b200 import deform_conv, modulated_deform_conv
    x, w = torch.zeros(1, 16, 5, 5), torch.zeros(8, 16, 3, 3)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        modulated_deform_conv(x, torch.zeros(1, 18, 5, 5), torch.zeros(1, 9, 5, 5), w, None, 1, 1)
    with pytest.raises(RuntimeError, match="Not implemented on the CPU"):
        deform_conv(x, torch.zeros(1, 18, 5, 5), w, 1, 1)


@pytest.mark.parametrize("channels_last", [False, True])
def test_fake_kernels_on_meta_tensors(channels_last):
    from ir_ads_b200 import ops
    fmt = torch.channels_last if channels_last else torch.contiguous_format
    x = torch.empty(2, 64, 20, 30, device="meta").contiguous(memory_format=fmt)
    w = torch.empty(32, 32, 3, 3, device="meta")
    off = torch.empty(2, 2 * 18, 10, 15, device="meta").contiguous(memory_format=fmt)
    mk = torch.empty(2, 2 * 9, 10, 15, device="meta").contiguous(memory_format=fmt)
    b = torch.empty(32, device="meta")
    y = ops.dcnv2(x, off, mk, w, b, 2, 2, 1, 1, 1, 1, 2, 2, 64)
    assert tuple(y.shape) == (2, 32, 10, 15) and y.is_contiguous(memory_format=fmt)
    gi, go, gm, gw, gb = ops.dcnv2_backward(y, x, off, mk, w, b, 2, 2, 1, 1, 1, 1, 2, 2, 64, True, True, True, True,
                                            True)
    assert gi.shape == x.shape and go.shape == off.shape and gm.shape == mk.shape
    assert gw.shape == w.shape and gb.shape == b.shape
    assert gi.is_contiguous(memory_format=fmt)
    none = ops.dcnv2_backward(y, x, off, None, w, None, 2, 2, 1, 1, 1, 1, 2, 2, 64, False, True, False, False, False)
    assert none[0] is None and none[2] is None and none[3] is None and none[4] is None


def test_import_loads_no_library():
    code = ("import sys; sys.path.insert(0, %r); import ir_ads_b200, ir_ads_b200.dcnv2; "
            "from ir_ads_b200 import _lib; assert _lib._lib is None; "
            "m = ir_ads_b200.ModulatedDeformConv(16, 16, 3, padding=1); assert _lib._lib is None; print('ok')" % ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert res.returncode == 0 and "ok" in res.stdout, res.stderr

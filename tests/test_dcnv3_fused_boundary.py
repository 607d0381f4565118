"""CPU-side checks of the fused DCNv3 entry points msda_dcnv3_fused_forward / msda_dcnv3_fused_backward (mask logits in,
the module's softmax inside the kernels): exported and declared, argument errors and empty problems answered before any
device work, and a plain C program that calls them.  No GPU work: every call here returns before it reaches the device."""
import ctypes
import os
import shutil
import subprocess

import pytest

from ir_ads_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NULL = ctypes.c_void_p(0)
UNSUPPORTED, INVALID = 2, 1


def _h():
    from ir_ads_b200.dcnv3 import _declare
    return _declare(_lib.lib())


def fwd(k=3, s=1, p=1, d=1, G=4, C=16, N=2, H=8, W=8, Ho=8, Wo=8, dtype=_lib.MSDA_F32, flags=0):
    """all tensor pointers null: only calls that return before touching them are made here"""
    return _h().msda_dcnv3_fused_forward(NULL, NULL, NULL, NULL, k, k, s, s, p, p, d, d, G, C, 1.0, N, H, W, Ho, Wo,
                                         NULL, dtype, flags)


def bwd(k=3, s=1, p=1, d=1, G=4, C=16, N=2, H=8, W=8, Ho=8, Wo=8, dtype=_lib.MSDA_F32, flags=0):
    return _h().msda_dcnv3_fused_backward(NULL, NULL, NULL, NULL, NULL, k, k, s, s, p, p, d, d, G, C, 1.0, N, H, W, Ho,
                                          Wo, NULL, NULL, NULL, NULL, 0, dtype, flags)


def test_entry_points_are_exported_and_declared():
    h = _lib.lib()
    assert hasattr(h, "msda_dcnv3_fused_forward") and hasattr(h, "msda_dcnv3_fused_backward")
    header = open(os.path.join(ROOT, "include", "msda.h")).read()
    assert "int msda_dcnv3_fused_forward(" in header and "int msda_dcnv3_fused_backward(" in header
    assert "const float* mask_logits" in header and "float* grad_mask_logits" in header
    # added to ABI 3 without a version bump
    assert h.msda_abi_version() == 3 == _lib.ABI_VERSION
    import ir_ads_b200
    assert "DCNv3FusedFunction" in ir_ads_b200.__all__


@pytest.mark.parametrize("call", [fwd, bwd])
def test_bad_geometry(call):
    for kw in ({"k": 0}, {"s": 0}, {"d": 0}, {"p": -1}, {"N": -1}, {"G": 0}, {"C": 0}, {"Ho": -1}):
        assert call(**kw) == INVALID, kw
        assert b"bad geometry" in _lib.lib().msda_last_error_message()


@pytest.mark.parametrize("call", [fwd, bwd])
def test_unsupported_shapes_and_dtypes(call):
    assert call(C=24) == UNSUPPORTED                      # group_channels outside {16, 32, 64, 128}
    assert b"group_channels" in _lib.lib().msda_last_error_message()
    assert call(k=9) == UNSUPPORTED                       # K = 81 > 64
    assert call(dtype=_lib.MSDA_F64) == UNSUPPORTED       # the generic composition serves float64, not these kernels
    assert b"float32 / bfloat16 / float16" in _lib.lib().msda_last_error_message()


@pytest.mark.parametrize("flags", [_lib.FLAG_DETERMINISTIC, _lib.FLAG_DETERMINISTIC | _lib.FLAG_DET_ATOMIC,
                                   _lib.FLAG_DETERMINISTIC | _lib.FLAG_DET_SEPARATE_FILL])
def test_deterministic_backward_is_refused(flags):
    """No fused deterministic form: refused before any device work, on real and on empty problems alike."""
    n0 = _lib.launch_count()
    assert bwd(flags=flags) == UNSUPPORTED
    assert b"deterministic" in _lib.lib().msda_last_error_message()
    assert bwd(N=0, flags=flags) == UNSUPPORTED
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("dtype", [_lib.MSDA_F32, _lib.MSDA_BF16, _lib.MSDA_F16])
def test_empty_problems_do_nothing(dtype):
    """Empty problems return MSDA_OK with null pointers and launch nothing; other flag bits are ignored."""
    n0 = _lib.launch_count()
    ignored = _lib.FLAG_FORCE_GENERIC | _lib.FLAG_NO_GRAD_VALUE | _lib.FLAG_ORDER_LINEAR
    for flags in (0, ignored):
        assert fwd(N=0, dtype=dtype, flags=flags) == 0
        assert fwd(Ho=0, dtype=dtype, flags=flags) == 0
        assert fwd(C=24, N=0, dtype=dtype) == 0           # nothing to compute: no shape check to fail
        assert bwd(N=0, dtype=dtype, flags=flags) == 0
        assert bwd(H=0, W=0, Ho=0, dtype=dtype, flags=flags) == 0
    assert fwd(dtype=dtype, flags=_lib.FLAG_DETERMINISTIC, N=0) == 0   # the forward ignores every flag
    assert _lib.launch_count() == n0


def test_null_output_is_an_argument_error():
    assert fwd() == INVALID
    assert b"output is null" in _lib.lib().msda_last_error_message()
    assert bwd() == INVALID
    assert b"gradient output pointer is null" in _lib.lib().msda_last_error_message()


def test_c_program_calls_the_fused_entry_points(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "dcn_fused.c"
    src.write_text(r'''
#include <stdio.h>
#include "msda.h"
int main(void) {
  /* empty problems: MSDA_OK, no device work */
  if (msda_dcnv3_fused_forward(NULL, NULL, NULL, NULL, 3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0f, 0, 8, 8, 8, 8, NULL,
                               MSDA_F32, 0u) != MSDA_OK) return 1;
  if (msda_dcnv3_fused_backward(NULL, NULL, NULL, NULL, NULL, 3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0f, 0, 8, 8, 8, 8, NULL,
                                NULL, NULL, NULL, 0, MSDA_F16, 0u) != MSDA_OK) return 2;
  /* group_channels 24 and the deterministic backward are refused */
  if (msda_dcnv3_fused_forward(NULL, NULL, NULL, NULL, 3, 3, 1, 1, 1, 1, 1, 1, 4, 24, 1.0f, 2, 8, 8, 8, 8, NULL,
                               MSDA_F32, 0u) != MSDA_ERR_UNSUPPORTED) return 3;
  if (msda_dcnv3_fused_backward(NULL, NULL, NULL, NULL, NULL, 3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0f, 2, 8, 8, 8, 8, NULL,
                                NULL, NULL, NULL, 0, MSDA_BF16, MSDA_FLAG_DETERMINISTIC) != MSDA_ERR_UNSUPPORTED)
    return 4;
  printf("dcnv3 fused abi ok\n");
  return 0;
}
''')
    exe = tmp_path / "dcn_fused"
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src),
           "-o", str(exe), "-L", libdir, "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + libdir,
           "-Wl,-rpath,/usr/local/cuda/lib64", "-Wl,--allow-shlib-undefined"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0 and "dcnv3 fused abi ok" in run.stdout, (run.returncode, run.stdout, run.stderr)

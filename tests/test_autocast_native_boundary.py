"""CPU-side checks of the autocast dtype tags MSDA_BF16_AUX16 / MSDA_F16_AUX16 (16-bit offsets / logits in the fused
module paths) and of the mixed add + LayerNorm entry points: the constants in the header and the loader, which entry
points accept or refuse the tags, the workspace answers, empty problems and a plain C program.  No GPU work: every call
here returns before it reaches the device."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from ir_ads_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NULL = ctypes.c_void_p(0)
INVALID, UNSUPPORTED = 1, 2
AUX16 = (_lib.MSDA_BF16_AUX16, _lib.MSDA_F16_AUX16)
VALUE_OF = {_lib.MSDA_BF16_AUX16: _lib.MSDA_BF16, _lib.MSDA_F16_AUX16: _lib.MSDA_F16}


def _h():
    from ir_ads_b200.dcnv3 import _declare
    return _declare(_lib.lib())


def test_tags_in_header_and_loader():
    header = open(os.path.join(ROOT, "include", "msda.h")).read()
    assert int(re.search(r"#define MSDA_BF16_AUX16 (\d+)", header).group(1)) == 4 == _lib.MSDA_BF16_AUX16
    assert int(re.search(r"#define MSDA_F16_AUX16 (\d+)", header).group(1)) == 5 == _lib.MSDA_F16_AUX16
    assert _lib.lib().msda_abi_version() == 3 == _lib.ABI_VERSION   # added without a version bump


def test_new_symbols_are_exported_and_declared():
    h = _lib.lib()
    header = open(os.path.join(ROOT, "include", "msda.h")).read()
    for name in ("msda_add_layernorm_mixed_forward", "msda_add_layernorm_mixed_backward"):
        assert hasattr(h, name) and f"int {name}(" in header
    # the offset / logit pointers of the four fused prototypes are untyped now
    assert "const void* sampling_offsets" in header and "void* grad_offsets" in header
    assert "const void* mask_logits" in header and "void* grad_mask_logits" in header


@pytest.mark.parametrize("tag", AUX16)
def test_operator_entry_points_refuse_the_tags(tag):
    """The plain operator, the plain DCNv3 pair and the same-dtype epilogue refuse the tags as an unknown tag, before
    any device work (an older library answers the fused entry points the same way)."""
    h = _h()
    n0 = _lib.launch_count()
    assert h.msda_forward(NULL, NULL, NULL, NULL, NULL, NULL, 1, 4, 2, 32, 1, 1, 1, NULL, tag, 0) == INVALID
    assert b"unknown dtype tag" in h.msda_last_error_message()
    assert h.msda_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 1, 4, 2, 32, 1, 1, 1, NULL, NULL, NULL, NULL, 0,
                           tag, 0) == INVALID
    assert b"unknown dtype tag" in h.msda_last_error_message()
    geo = [3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0, 2, 8, 8, 8, 8]
    assert h.msda_dcnv3_forward(NULL, NULL, NULL, NULL, *geo, NULL, tag, 0) == UNSUPPORTED
    assert h.msda_dcnv3_backward(NULL, NULL, NULL, NULL, NULL, *geo, NULL, NULL, NULL, NULL, 0, tag, 0) == UNSUPPORTED
    assert h.msda_add_layernorm_forward(NULL, NULL, NULL, NULL, NULL, 4, 64, 1e-5, NULL, NULL, NULL, tag) == UNSUPPORTED
    assert h.msda_add_layernorm_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 4, 64, NULL, NULL, NULL, NULL, 0,
                                         tag) == UNSUPPORTED
    # the mixed epilogue takes the 16-bit value tags of `a`, not the fused paths' tags, and not float32
    for bad in (tag, _lib.MSDA_F32, _lib.MSDA_F64):
        assert h.msda_add_layernorm_mixed_forward(NULL, NULL, NULL, NULL, NULL, 4, 64, 1e-5, NULL, NULL, NULL,
                                                  bad) == UNSUPPORTED
        assert h.msda_add_layernorm_mixed_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 4, 64, NULL, NULL, NULL,
                                                   NULL, NULL, 0, bad) == UNSUPPORTED
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("tag", AUX16)
def test_fused_supported_on_fast_shapes_only(tag):
    h = _lib.lib()
    assert h.msda_fused_supported(32, 4, 4, 22223, 8, tag, 0) == 1
    assert h.msda_fused_supported(128, 4, 8, 22223, 2, tag, 0) == 1
    assert h.msda_fused_supported(30, 4, 4, 22223, 8, tag, 0) == 0        # no fast kernel for D = 30
    assert h.msda_fused_supported(32, 17, 4, 22223, 8, tag, 0) == 0       # L > 16
    assert h.msda_fused_supported(32, 4, 4, 22223, 8, tag, _lib.FLAG_DETERMINISTIC) == 0
    assert h.msda_fused_supported(32, 4, 4, 22223, 8, tag, _lib.FLAG_FORCE_GENERIC) == 0
    assert h.msda_fused_supported(32, 4, 4, 22223, 8, 6, 0) == 0           # still no tag 6


@pytest.mark.parametrize("tag", AUX16)
def test_workspace_answers_equal_the_value_tag(tag):
    h = _h()
    vt = VALUE_OF[tag]
    det = _lib.FLAG_DETERMINISTIC
    for flags in (0, det, det | _lib.FLAG_DET_ATOMIC, det | _lib.FLAG_DET_SEPARATE_FILL):
        for dims in ((8, 22223, 8, 32, 4, 22223, 4), (2, 10, 2, 32, 1, 3, 2), (0, 10, 2, 32, 1, 3, 2)):
            assert h.msda_backward_workspace_bytes(*dims, tag, flags) == h.msda_backward_workspace_bytes(*dims, vt, flags)
        for geo in ((3, 3, 4, 16, 16, 200, 336, 200, 336), (5, 5, 8, 32, 2, 9, 7, 9, 7), (3, 3, 4, 16, 2, 8, 8, 0, 8)):
            assert (h.msda_dcnv3_backward_workspace_bytes(*geo, tag, flags)
                    == h.msda_dcnv3_backward_workspace_bytes(*geo, vt, flags))
    assert h.msda_backward_workspace_bytes(2, 10, 2, 32, 1, 3, 2, tag, 0) == 2 * 10 * 2 * 32 * 4


@pytest.mark.parametrize("tag", AUX16)
def test_fused_entry_points_accept_the_tags(tag):
    """Empty problems are no-ops; everything else answers what the value tag answers, before any device work."""
    h = _h()
    vt = VALUE_OF[tag]
    n0 = _lib.launch_count()

    def ffwd(dt, B=2, D=32, Q=5):
        return h.msda_fused_forward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 2, NULL, B, 10, 2, D, 1, Q, 2, NULL, dt, 0)

    def fbwd(dt, B=2, D=32, ref_dim=2, flags=0):
        return h.msda_fused_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, ref_dim, NULL, B, 10, 2, D, 1, 5,
                                     2, NULL, NULL, NULL, NULL, 0, dt, flags)

    assert ffwd(tag, B=0) == ffwd(tag, Q=0) == 0
    assert ffwd(tag) == ffwd(vt) == INVALID                     # null pointers, after the shape checks pass
    assert ffwd(tag, D=30) == ffwd(vt, D=30) == UNSUPPORTED
    assert fbwd(tag, B=0) == fbwd(vt, B=0) == UNSUPPORTED      # the fused backward needs a non-empty problem
    assert fbwd(tag, ref_dim=3) == fbwd(vt, ref_dim=3) == INVALID
    assert fbwd(tag, flags=_lib.FLAG_DETERMINISTIC) == UNSUPPORTED
    geo = [3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0]
    assert h.msda_dcnv3_fused_forward(NULL, NULL, NULL, NULL, *geo, 0, 8, 8, 8, 8, NULL, tag, 0) == 0
    assert h.msda_dcnv3_fused_backward(NULL, NULL, NULL, NULL, NULL, *geo, 0, 8, 8, 8, 8, NULL, NULL, NULL, NULL, 0,
                                       tag, 0) == 0
    assert h.msda_dcnv3_fused_backward(NULL, NULL, NULL, NULL, NULL, *geo, 2, 0, 0, 0, 8, NULL, NULL, NULL, NULL, 0,
                                       tag, 0) == 0
    assert h.msda_dcnv3_fused_forward(NULL, NULL, NULL, NULL, *geo, 2, 8, 8, 8, 8, NULL, tag, 0) == INVALID
    assert h.msda_dcnv3_fused_backward(NULL, NULL, NULL, NULL, NULL, *geo, 2, 8, 8, 8, 8, NULL, NULL, NULL, NULL, 0,
                                       tag, _lib.FLAG_DETERMINISTIC) == UNSUPPORTED
    geo24 = [3, 3, 1, 1, 1, 1, 1, 1, 4, 24, 1.0]
    assert h.msda_dcnv3_fused_forward(NULL, NULL, NULL, NULL, *geo24, 2, 8, 8, 8, 8, NULL, tag, 0) == UNSUPPORTED
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("a_dtype", [_lib.MSDA_BF16, _lib.MSDA_F16])
def test_epilogue_f16_and_mixed_empty_problems(a_dtype):
    h = _lib.lib()
    n0 = _lib.launch_count()
    # the same-dtype form takes float16 now
    assert h.msda_add_layernorm_forward(NULL, NULL, NULL, NULL, NULL, 0, 64, 1e-5, NULL, NULL, NULL, _lib.MSDA_F16) == 0
    assert h.msda_add_layernorm_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 4, 0, NULL, NULL, NULL, NULL, 0,
                                         _lib.MSDA_F16) == 0
    assert h.msda_add_layernorm_mixed_forward(NULL, NULL, NULL, NULL, NULL, 0, 64, 1e-5, NULL, NULL, NULL, a_dtype) == 0
    assert h.msda_add_layernorm_mixed_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 4, 0, NULL, NULL, NULL, NULL,
                                               NULL, 0, a_dtype) == 0
    assert h.msda_add_layernorm_mixed_forward(NULL, NULL, NULL, NULL, NULL, 4, 64, 1e-5, NULL, NULL, NULL,
                                              a_dtype) == INVALID
    assert h.msda_add_layernorm_mixed_forward(NULL, NULL, NULL, NULL, NULL, 4, 66, 1e-5, NULL, NULL, NULL,
                                              a_dtype) == UNSUPPORTED           # channels % 4 != 0
    assert h.msda_add_layernorm_mixed_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 4, 64, NULL, NULL, NULL, NULL,
                                               NULL, 0, a_dtype) == INVALID    # grad_gamma is null
    assert _lib.launch_count() == n0


def test_python_refuses_other_mixes():
    """Offsets / logits are float32, or in the value's 16-bit dtype; any other mix is refused (before any device
    work: the dtype checks run first)."""
    import torch
    from ir_ads_b200.functional import _aux_tag
    assert _aux_tag(torch.float32, torch.float32, "x") == _lib.MSDA_F32
    assert _aux_tag(torch.float16, torch.float32, "x") == _lib.MSDA_F16
    assert _aux_tag(torch.float16, torch.float16, "x") == _lib.MSDA_F16_AUX16
    assert _aux_tag(torch.bfloat16, torch.bfloat16, "x") == _lib.MSDA_BF16_AUX16
    for v, a in ((torch.float16, torch.bfloat16), (torch.bfloat16, torch.float16), (torch.float32, torch.float16),
                 (torch.float16, torch.float64)):
        with pytest.raises(RuntimeError, match="value's dtype"):
            _aux_tag(v, a, "sampling_offsets / attn_logits")


def test_c_program_calls_the_new_tags_and_the_mixed_epilogue(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "autocast.c"
    src.write_text(r'''
#include <stdio.h>
#include "msda.h"
int main(void) {
  const float* f32 = NULL; /* float pointers still convert to the widened `const void*` parameters */
  float* g32 = NULL;
  if (msda_fused_supported(32, 4, 4, 22223, 8, MSDA_BF16_AUX16, 0u) != 1) return 1;
  if (msda_fused_supported(32, 4, 4, 22223, 8, MSDA_F16_AUX16, 0u) != 1) return 2;
  if (msda_backward_workspace_bytes(2, 10, 2, 32, 1, 3, 2, MSDA_F16_AUX16, 0u) !=
      msda_backward_workspace_bytes(2, 10, 2, 32, 1, 3, 2, MSDA_F16, 0u)) return 3;
  if (msda_fused_forward(NULL, NULL, NULL, NULL, f32, f32, NULL, 2, NULL, 0, 10, 2, 32, 1, 5, 2, NULL,
                         MSDA_BF16_AUX16, 0u) != MSDA_OK) return 4;
  if (msda_fused_backward(NULL, NULL, NULL, NULL, NULL, f32, f32, NULL, 2, NULL, 2, 10, 2, 32, 1, 5, 2, NULL, g32, g32,
                          NULL, 0, MSDA_F32, MSDA_FLAG_DETERMINISTIC) != MSDA_ERR_UNSUPPORTED) return 5;
  if (msda_dcnv3_fused_forward(NULL, NULL, NULL, NULL, 3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0f, 0, 8, 8, 8, 8, NULL,
                               MSDA_F16_AUX16, 0u) != MSDA_OK) return 6;
  if (msda_dcnv3_fused_backward(NULL, NULL, NULL, NULL, NULL, 3, 3, 1, 1, 1, 1, 1, 1, 4, 16, 1.0f, 0, 8, 8, 8, 8, NULL,
                                NULL, NULL, NULL, 0, MSDA_BF16_AUX16, 0u) != MSDA_OK) return 7;
  if (msda_forward(NULL, NULL, NULL, NULL, NULL, NULL, 1, 4, 2, 32, 1, 1, 1, NULL, MSDA_F16_AUX16, 0u) !=
      MSDA_ERR_INVALID_ARGUMENT) return 8;
  if (msda_add_layernorm_forward(NULL, NULL, NULL, NULL, NULL, 4, 64, 1e-5f, NULL, NULL, NULL, MSDA_BF16_AUX16) !=
      MSDA_ERR_UNSUPPORTED) return 9;
  if (msda_add_layernorm_mixed_forward(NULL, NULL, NULL, NULL, NULL, 0, 64, 1e-5f, NULL, NULL, NULL, MSDA_F16) !=
      MSDA_OK) return 10;
  if (msda_add_layernorm_mixed_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 4, 64, NULL, NULL, NULL, NULL, NULL, 0,
                                        MSDA_F32) != MSDA_ERR_UNSUPPORTED) return 11;
  printf("autocast abi ok\n");
  return 0;
}
''')
    exe = tmp_path / "autocast"
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src),
           "-o", str(exe), "-L", libdir, "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + libdir,
           "-Wl,-rpath,/usr/local/cuda/lib64", "-Wl,--allow-shlib-undefined"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0 and "autocast abi ok" in run.stdout, (run.returncode, run.stdout, run.stderr)

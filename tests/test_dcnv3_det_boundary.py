"""CPU-side checks of the DCNv3 deterministic backward's C ABI: the workspace query msda_dcnv3_backward_workspace_bytes
(exported, today's rule without MSDA_FLAG_DETERMINISTIC, the documented formula with it) and a plain C program that
calls it.  No GPU work: every call here is host arithmetic or fails its argument checks before it reaches the device."""
import os
import shutil
import subprocess

import pytest

from ir_ads_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DET, ATOMIC, SEP = _lib.FLAG_DETERMINISTIC, _lib.FLAG_DET_ATOMIC, _lib.FLAG_DET_SEPARATE_FILL
SLOT = 256   # the one-level table at the front of the deterministic workspace (include/msda.h)


def _h():
    from ir_ads_b200.dcnv3 import _declare
    return _declare(_lib.lib())


def dcn_ws(k, G, C, N, H, W, Ho, Wo, dtype, flags):
    return _h().msda_dcnv3_backward_workspace_bytes(k, k, G, C, N, H, W, Ho, Wo, dtype, flags)


def plain_ws(N, S, G, C, Q, K, dtype, flags):
    return _lib.lib().msda_backward_workspace_bytes(N, S, G, C, 1, Q, K, dtype, flags)


def test_workspace_query_is_exported():
    assert hasattr(_lib.lib(), "msda_dcnv3_backward_workspace_bytes")
    header = open(os.path.join(ROOT, "include", "msda.h")).read()
    assert "size_t msda_dcnv3_backward_workspace_bytes(" in header
    # added to ABI 3 without a version bump, as MSDA_F16 was
    assert _lib.lib().msda_abi_version() == 3 == _lib.ABI_VERSION


@pytest.mark.parametrize("flags", [0, _lib.FLAG_FORCE_GENERIC | _lib.FLAG_NO_GRAD_VALUE, ATOMIC, SEP])
def test_default_rule_without_the_flag(flags):
    """Without MSDA_FLAG_DETERMINISTIC: 0 for float32, N*H_in*W_in*C floats for bfloat16 / float16; other bits (and
    the deterministic sub-flags on their own) do not matter."""
    N, H, W, G, C = 16, 200, 336, 4, 16
    n_value = N * H * W * G * C
    assert dcn_ws(3, G, C, N, H, W, H, W, _lib.MSDA_F32, flags) == 0
    assert dcn_ws(3, G, C, N, H, W, H, W, _lib.MSDA_BF16, flags) == n_value * 4
    assert dcn_ws(3, G, C, N, H, W, H, W, _lib.MSDA_F16, flags) == n_value * 4


@pytest.mark.parametrize("dtype", [_lib.MSDA_F32, _lib.MSDA_BF16, _lib.MSDA_F16])
@pytest.mark.parametrize("k,stride", [(3, 1), (3, 2), (1, 1), (5, 1)])
def test_deterministic_rule_is_the_one_level_layout(dtype, k, stride):
    """With the flag: the one-level table slot plus the deterministic layout of the equivalent one-level MSDeformAttn
    problem (value [N, H_in*W_in, G, C], Q = H_out*W_out, P = K); the same for every dtype."""
    N, H, W, G, C = 2, 56, 56, 4, 32
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    K = k * k
    for flags in (DET, DET | SEP, DET | _lib.FLAG_FORCE_GENERIC | _lib.FLAG_ORDER_LINEAR):
        want = SLOT + plain_ws(N, H * W, G, C, Ho * Wo, K, dtype, DET | (flags & SEP))
        assert dcn_ws(k, G, C, N, H, W, Ho, Wo, dtype, flags) == want
    # the sorted layout (no float workspace, whatever the dtype); dense problems carry the fixed-point accumulators
    n_value = N * H * W * G * C
    sorted_bytes = dcn_ws(k, G, C, N, H, W, Ho, Wo, dtype, DET)
    assert sorted_bytes == SLOT + plain_ws(N, H * W, G, C, Ho * Wo, K, _lib.MSDA_F32, DET)
    if Ho * Wo * K >= 4 * H * W:
        assert sorted_bytes > SLOT + n_value * 8
    else:
        assert sorted_bytes < SLOT + n_value * 8


@pytest.mark.parametrize("dtype", [_lib.MSDA_F32, _lib.MSDA_BF16, _lib.MSDA_F16])
def test_det_atomic_rule(dtype):
    """MSDA_FLAG_DET_ATOMIC: 64-bit fixed-point accumulators + {amax x2, scale}, after the slot."""
    N, H, W, G, C = 2, 40, 48, 8, 16
    n_value = N * H * W * G * C
    assert dcn_ws(3, G, C, N, H, W, H, W, dtype, DET | ATOMIC) == SLOT + n_value * 8 + 64
    assert dcn_ws(3, G, C, N, H, W, H, W, dtype, DET | ATOMIC | SEP) == SLOT + n_value * 8 + 64


@pytest.mark.parametrize("dtype", [_lib.MSDA_F32, _lib.MSDA_BF16])
def test_empty_problems_need_what_they_need_without_the_flag(dtype):
    for N, H, W, Ho, Wo in ((0, 8, 8, 8, 8), (2, 8, 8, 0, 8), (2, 8, 8, 8, 0), (2, 0, 8, 8, 8), (2, 8, 0, 8, 8)):
        assert dcn_ws(3, 2, 16, N, H, W, Ho, Wo, dtype, DET) == dcn_ws(3, 2, 16, N, H, W, Ho, Wo, dtype, 0)


def test_c_program_calls_the_workspace_query(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "dcn_ws.c"
    src.write_text(r'''
#include <stdio.h>
#include "msda.h"
int main(void) {
  const size_t n_value = (size_t)2 * 10 * 12 * 4 * 16;
  /* without the flag: today's rule */
  if (msda_dcnv3_backward_workspace_bytes(3, 3, 4, 16, 2, 10, 12, 10, 12, MSDA_F32, 0u) != 0) return 1;
  if (msda_dcnv3_backward_workspace_bytes(3, 3, 4, 16, 2, 10, 12, 10, 12, MSDA_BF16, 0u) != n_value * 4) return 2;
  if (msda_dcnv3_backward_workspace_bytes(3, 3, 4, 16, 2, 10, 12, 10, 12, MSDA_F16, 0u) != n_value * 4) return 3;
  /* with it: 256 + the one-level deterministic layout */
  if (msda_dcnv3_backward_workspace_bytes(3, 3, 4, 16, 2, 10, 12, 10, 12, MSDA_F16, MSDA_FLAG_DETERMINISTIC) !=
      256 + msda_backward_workspace_bytes(2, 120, 4, 16, 1, 120, 9, MSDA_F16, MSDA_FLAG_DETERMINISTIC)) return 4;
  if (msda_dcnv3_backward_workspace_bytes(3, 3, 4, 16, 2, 10, 12, 10, 12, MSDA_F32,
                                          MSDA_FLAG_DETERMINISTIC | MSDA_FLAG_DET_ATOMIC) != 256 + n_value * 8 + 64)
    return 5;
  printf("dcnv3 workspace abi ok\n");
  return 0;
}
''')
    exe = tmp_path / "dcn_ws"
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src),
           "-o", str(exe), "-L", libdir, "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + libdir,
           "-Wl,-rpath,/usr/local/cuda/lib64", "-Wl,--allow-shlib-undefined"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0 and "dcnv3 workspace abi ok" in run.stdout, (run.returncode, run.stdout, run.stderr)

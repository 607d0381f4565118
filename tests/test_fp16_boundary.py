"""CPU-side checks of the float16 value tag (MSDA_F16): the constant in the header and in the loader, dispatch names,
backward workspace sizes, the dtype checks of the Python wrappers, and a plain C program that uses the tag.  No GPU
work: every call here is host arithmetic or fails its argument checks before it reaches the device."""
import os
import re

import pytest
import torch

from ir_ads_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_f16_tag_in_header_and_loader():
    header = open(os.path.join(ROOT, "include", "msda.h")).read()
    m = re.search(r"#define MSDA_F16 (\d+)", header)
    assert m and int(m.group(1)) == 3 == _lib.MSDA_F16
    # the tag is additive: the ABI version stays
    assert re.search(r"#define MSDA_ABI_VERSION (\d+)", header).group(1) == "3" and _lib.ABI_VERSION == 3


def test_f16_dispatch_names():
    name = lambda D, flags=0, bwd=0, L=4, P=4: _lib.lib().msda_dispatch_name(D, L, P, 22223, 8, _lib.MSDA_F16, flags,
                                                                            bwd).decode()
    assert name(32) == "fwd_fast_d32_f16"
    assert name(16, bwd=1) == "bwd_fast_d16_f16"
    assert name(128) == "fwd_fast_d128_f16"
    assert name(30, bwd=1) == "bwd_generic_f16"
    assert name(32, _lib.FLAG_FORCE_GENERIC) == "fwd_generic_f16"
    assert name(32, _lib.FLAG_FORCE_GENERIC, bwd=1) == "bwd_generic_f16"
    assert name(32, L=17) == "fwd_generic_f16"


def test_f16_fused_supported():
    h = _lib.lib()
    assert h.msda_fused_supported(32, 4, 4, 22223, 8, _lib.MSDA_F16, 0) == 1
    assert h.msda_fused_supported(30, 4, 4, 22223, 8, _lib.MSDA_F16, 0) == 0
    assert h.msda_fused_supported(32, 4, 4, 22223, 8, _lib.MSDA_F16, _lib.FLAG_DETERMINISTIC) == 0


def test_f16_backward_workspace_sizes():
    """float16 follows the bfloat16 rule: float accumulators without the deterministic flag, and with it exactly
    what float32 needs (the fixed-point / sorted workspaces do not depend on the value type)."""
    h = _lib.lib()
    B, S, H, D, L, Q, P = 8, 22223, 8, 32, 4, 22223, 4
    n_value = B * S * H * D
    ws = lambda dt, flags, D=D, Q=Q: h.msda_backward_workspace_bytes(B, S, H, D, L, Q, P, dt, flags)
    det, atomic = _lib.FLAG_DETERMINISTIC, _lib.FLAG_DETERMINISTIC | _lib.FLAG_DET_ATOMIC
    assert ws(_lib.MSDA_F16, 0) == n_value * 4 == ws(_lib.MSDA_BF16, 0)
    assert ws(_lib.MSDA_F16, det) == ws(_lib.MSDA_F32, det) > n_value * 8               # sorted, dense
    assert ws(_lib.MSDA_F16, det, Q=300) == ws(_lib.MSDA_F32, det, Q=300) < n_value * 8  # sorted, sparse
    assert ws(_lib.MSDA_F16, atomic) == n_value * 8 + 64                                  # fixed-point reds
    assert ws(_lib.MSDA_F16, det, D=30) == B * S * H * 30 * 8 + 64                        # generic
    assert ws(_lib.MSDA_F16, _lib.FLAG_FORCE_GENERIC) == n_value * 4


def test_public_op_dtype_table_excludes_f16():
    """The reference-signature op keeps float / double (/ bf16); only the fused path and internal callers take f16."""
    from ir_ads_b200 import functional
    assert torch.float16 not in functional._DTYPE_TAG and functional._VALUE_TAG[torch.float16] == _lib.MSDA_F16


def test_c_program_uses_the_f16_tag(tmp_path):
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "f16.c"
    src.write_text(r'''
#include <stdio.h>
#include "msda.h"
int main(void) {
  /* negative dimension with the f16 tag: refused as an argument error, not as an unknown dtype */
  int s = msda_forward(NULL, NULL, NULL, NULL, NULL, NULL, -1, 4, 2, 32, 1, 1, 1, NULL, MSDA_F16, 0u);
  if (s != MSDA_ERR_INVALID_ARGUMENT) return 1;
  if (msda_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 2, -4, 2, 32, 1, 1, 1, NULL, NULL, NULL, NULL, 0,
                    MSDA_F16, 0u) != MSDA_ERR_INVALID_ARGUMENT) return 2;
  /* an empty problem is a no-op for f16 as for every other tag */
  if (msda_forward(NULL, NULL, NULL, NULL, NULL, NULL, 0, 4, 2, 32, 1, 1, 1, NULL, MSDA_F16, 0u) != MSDA_OK) return 3;
  if (msda_backward_workspace_bytes(2, 10, 2, 32, 1, 3, 2, MSDA_F16, 0u) != (size_t)2 * 10 * 2 * 32 * 4) return 4;
  if (!msda_fused_supported(32, 1, 2, 10, 2, MSDA_F16, 0u)) return 5;
  printf("f16 abi ok\n");
  return 0;
}
''')
    exe = tmp_path / "f16"
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src),
           "-o", str(exe), "-L", libdir, "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + libdir,
           "-Wl,-rpath,/usr/local/cuda/lib64", "-Wl,--allow-shlib-undefined"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0 and "f16 abi ok" in run.stdout, (run.returncode, run.stdout, run.stderr)

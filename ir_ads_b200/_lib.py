"""Loader for libmsda_b200.so (the C ABI of include/msda.h).

There is no fallback: if the library is missing or a call fails, the caller gets an exception.
The library is built in tree by ir_ads_b200/csrc/build.sh (``build()`` below runs it).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
# MSDA_B200_LIB overrides the library path (kernel-variant experiments); the default is the in-tree build
LIB_PATH = os.environ.get("MSDA_B200_LIB") or os.path.join(_PKG, "libmsda_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_PKG), "include", "msda.h")

# include/msda.h
MSDA_F32, MSDA_F64, MSDA_BF16, MSDA_F16 = 0, 1, 2, 3
# fused module paths under autocast: offsets / logits and their gradients in the value's 16-bit type as well
MSDA_BF16_AUX16, MSDA_F16_AUX16 = 4, 5
MSDA_OK = 0
FLAG_DETERMINISTIC = 1 << 0
FLAG_FORCE_GENERIC = 1 << 1
FLAG_ORDER_LINEAR = 1 << 2
FLAG_ORDER_STRIP = 1 << 4
FLAG_ORDER_TILE2D = 1 << 5
FLAG_DET_ATOMIC = 1 << 6
FLAG_NO_GRAD_VALUE = 1 << 11
FLAG_FOLD_ON = 1 << 12
FLAG_FOLD_OFF = 1 << 13
FLAG_DET_SEPARATE_FILL = 1 << 14
ABI_VERSION = 3

_lock = threading.Lock()
_lib = None


class MSDAError(RuntimeError):
    """A libmsda_b200 call returned a non-zero status (the reference raises RuntimeError from
    AT_ASSERTM / AT_ERROR at the same places: ms_deform_attn_cuda.cu:29-53)."""


def build(verbose: bool = False) -> str:
    """Compile the library for sm_100a (nvcc cross-compiles without a GPU)."""
    script = os.path.join(_PKG, "csrc", "build.sh")
    out = subprocess.run(["bash", script], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("building libmsda_b200.so failed:\n" + out.stdout + out.stderr)
    if verbose:
        print(out.stdout.strip())
    return LIB_PATH


def _declare(lib: ctypes.CDLL) -> None:
    vp, i, u, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint, ctypes.c_size_t
    lib.msda_abi_version.restype = i
    lib.msda_abi_version.argtypes = []
    lib.msda_build_config.restype = u
    lib.msda_build_config.argtypes = []
    lib.msda_forward.restype = i
    lib.msda_forward.argtypes = [vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, vp, i, u]
    lib.msda_backward_workspace_bytes.restype = sz
    lib.msda_backward_workspace_bytes.argtypes = [i, i, i, i, i, i, i, i, u]
    lib.msda_backward.restype = i
    lib.msda_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, vp, vp, vp, vp, sz, i, u]
    lib.msda_fused_supported.restype = i
    lib.msda_fused_supported.argtypes = [i, i, i, i, i, i, u]
    lib.msda_fused_forward.restype = i
    lib.msda_fused_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, vp, i, i, i, i, i, i, i, vp, i, u]
    lib.msda_fused_backward.restype = i
    lib.msda_fused_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i, vp, i, i, i, i, i, i, i, vp, vp, vp, vp,
                                        sz, i, u]
    lib.msda_packed_backward_workspace_bytes.restype = sz
    lib.msda_packed_backward_workspace_bytes.argtypes = [i, i, i, i, u]
    lib.msda_packed_forward.restype = i
    lib.msda_packed_forward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, i, i, i, vp, i, u]
    lib.msda_packed_backward.restype = i
    lib.msda_packed_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, i, i, i, vp, vp, vp,
                                         vp, sz, i, u]
    i64, f32 = ctypes.c_int64, ctypes.c_float
    lib.msda_add_layernorm_workspace_bytes.restype = sz
    lib.msda_add_layernorm_workspace_bytes.argtypes = [i64, i]
    lib.msda_add_layernorm_forward.restype = i
    lib.msda_add_layernorm_forward.argtypes = [vp, vp, vp, vp, vp, i64, i, f32, vp, vp, vp, i]
    lib.msda_add_layernorm_backward.restype = i
    lib.msda_add_layernorm_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, i, vp, vp, vp, vp, sz, i]
    lib.msda_add_layernorm_mixed_forward.restype = i
    lib.msda_add_layernorm_mixed_forward.argtypes = lib.msda_add_layernorm_forward.argtypes
    lib.msda_add_layernorm_mixed_backward.restype = i
    lib.msda_add_layernorm_mixed_backward.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, i, vp, vp, vp, vp, vp, sz, i]
    dcn2 = [i] * 16   # batch, channels, H_in, W_in, H_out, W_out, kernel, stride, pad, dilation (h, w), groups, dg
    lib.msda_dcnv2_col2im_workspace_bytes.restype = sz
    lib.msda_dcnv2_col2im_workspace_bytes.argtypes = dcn2 + [i, u]
    lib.msda_dcnv2_im2col.restype = i
    lib.msda_dcnv2_im2col.argtypes = [vp, vp, vp, vp] + dcn2 + [vp, i, u]
    lib.msda_dcnv2_col2im.restype = i
    lib.msda_dcnv2_col2im.argtypes = [vp, vp, vp, vp, vp] + dcn2 + [vp, vp, vp, vp, sz, i, u]
    lib.msda_debug_bookkeeping.restype = i
    lib.msda_debug_bookkeeping.argtypes = [vp, vp, vp, vp, i, i, i, i, i, i, i, vp, vp]
    lib.msda_debug_fastdiv.restype = u
    lib.msda_debug_fastdiv.argtypes = [u, u]
    lib.msda_status_string.restype = ctypes.c_char_p
    lib.msda_status_string.argtypes = [i]
    lib.msda_last_error_message.restype = ctypes.c_char_p
    lib.msda_last_error_message.argtypes = []
    lib.msda_kernel_launch_count.restype = ctypes.c_uint64
    lib.msda_kernel_launch_count.argtypes = []
    lib.msda_dispatch_name.restype = ctypes.c_char_p
    lib.msda_dispatch_name.argtypes = [i, i, i, i, i, i, u, i]


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise ImportError(
                        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "or ir_ads_b200/csrc/build.sh. There is no CPU or PyTorch fallback for this op.")
                handle = ctypes.CDLL(LIB_PATH)
                _declare(handle)
                got = handle.msda_abi_version()
                if got != ABI_VERSION:
                    raise ImportError(f"libmsda_b200.so ABI {got} != expected {ABI_VERSION}; rebuild it")
                _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    if status != MSDA_OK:
        handle = lib()
        name = handle.msda_status_string(status).decode()
        detail = handle.msda_last_error_message().decode()
        raise MSDAError(f"{what}: {name}: {detail}")


def has_experiments() -> bool:
    """True for a -DMSDA_EXPERIMENTS build (tools/build_variant.sh); the product library has none."""
    return bool(lib().msda_build_config() & 1)


def launch_count() -> int:
    return int(lib().msda_kernel_launch_count())

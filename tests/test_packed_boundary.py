"""CPU-side checks of the packed (padding-free) entry points msda_packed_forward / msda_packed_backward and of the host
side of ir_ads_b200/packing.py: exported and declared, argument / alignment / dtype errors, the deterministic flag
refused, empty problems answered before any device work, the slim-build stubs, a strict C99 caller, and valid_extents
against F.interpolate of CPU masks.  No GPU work: every library call here returns before it reaches the device."""
import ctypes
import os
import random
import shutil
import subprocess

import pytest
import torch
import torch.nn.functional as F

from ir_ads_b200 import _lib
from ir_ads_b200.packing import valid_extents

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NULL = ctypes.c_void_p(0)
INVALID, UNSUPPORTED, WORKSPACE = 1, 2, 3
FAKE = ctypes.c_void_p(0x10000)       # never dereferenced: every call below fails or returns before device work
ODD = ctypes.c_void_p(0x10008)


def fwd(B=2, Tv=100, H=8, D=32, L=4, Tq=100, P=4, mv=60, mq=60, ref_dim=2, dtype=_lib.MSDA_F32, flags=0, ptr=NULL,
        out=NULL, meta=NULL):
    return _lib.lib().msda_packed_forward(NULL, ptr, ptr, meta, ptr, ptr, ptr, ref_dim, B, Tv, H, D, L, Tq, P, mv, mq,
                                          out, dtype, flags)


def bwd(B=2, Tv=100, H=8, D=32, L=4, Tq=100, P=4, mv=60, mq=60, ref_dim=2, dtype=_lib.MSDA_F32, flags=0, ptr=NULL,
        grads=NULL, ws=NULL, ws_bytes=0, meta=NULL):
    return _lib.lib().msda_packed_backward(NULL, ptr, ptr, ptr, meta, ptr, ptr, ptr, ref_dim, B, Tv, H, D, L, Tq, P,
                                           mv, mq, ptr, grads, grads, ws, ws_bytes, dtype, flags)


def last_error():
    return _lib.lib().msda_last_error_message()


def test_entry_points_are_exported_and_declared():
    h = _lib.lib()
    for name in ("msda_packed_forward", "msda_packed_backward", "msda_packed_backward_workspace_bytes"):
        assert hasattr(h, name)
    header = open(os.path.join(ROOT, "include", "msda.h")).read()
    assert "int msda_packed_forward(" in header and "int msda_packed_backward(" in header
    assert "size_t msda_packed_backward_workspace_bytes(" in header
    assert "TRUSTED" in header                                   # the device metadata is not checked by the library
    assert h.msda_abi_version() == 3 == _lib.ABI_VERSION        # added to ABI 3 without a version bump
    import ir_ads_b200
    for name in ("MSDeformAttnPackedFunction", "PackedLevels", "valid_extents", "pack_levels",
                 "packed_reference_points", "unpack_tokens"):
        assert name in ir_ads_b200.__all__ and hasattr(ir_ads_b200, name)


@pytest.mark.parametrize("call", [fwd, bwd])
def test_argument_errors(call):
    n0 = _lib.launch_count()
    for kw in ({"B": -1}, {"Tv": -1}, {"Tq": -1}, {"H": -1}, {"ref_dim": 3}, {"dtype": 9}):
        assert call(**kw) == INVALID, kw
    assert call(mq=101) == INVALID and b"largest image" in last_error()     # more queries than the total
    assert call(mv=40) == INVALID and b"largest image" in last_error()      # 2 images x 40 < 100 values
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("call", [fwd, bwd])
def test_unsupported_shapes_and_dtypes(call):
    for kw in ({"D": 24}, {"L": 17}, {"P": 17}, {"dtype": _lib.MSDA_F64}, {"mv": 100, "Tv": 100, "D": 128, "H": 2 ** 17}):
        assert call(**kw) == UNSUPPORTED, kw
        assert b"packed path" in last_error()


def test_null_pointers_and_alignment():
    assert fwd() == INVALID and b"output is null" in last_error()
    assert fwd(out=FAKE) == INVALID and b"null tensor pointer" in last_error()
    assert fwd(out=FAKE, ptr=FAKE, meta=ODD) == INVALID and b"image_meta" in last_error()
    assert fwd(out=ODD, ptr=FAKE, meta=FAKE) == INVALID and b"16-byte" in last_error()
    assert bwd() == INVALID and b"gradient output pointer is null" in last_error()
    assert bwd(grads=FAKE) == INVALID and b"null tensor pointer" in last_error()
    assert bwd(grads=ODD, ptr=FAKE, meta=FAKE) == INVALID and b"16-byte" in last_error()
    # 16-bit values need a float workspace for grad_value
    assert bwd(grads=FAKE, ptr=FAKE, meta=FAKE, dtype=_lib.MSDA_BF16) == WORKSPACE


def test_workspace_bytes():
    h = _lib.lib()
    assert h.msda_packed_backward_workspace_bytes(100, 8, 32, _lib.MSDA_F32, 0) == 0
    for tag in (_lib.MSDA_BF16, _lib.MSDA_F16, _lib.MSDA_BF16_AUX16, _lib.MSDA_F16_AUX16):
        assert h.msda_packed_backward_workspace_bytes(100, 8, 32, tag, 0) == 100 * 8 * 32 * 4
    assert h.msda_packed_backward_workspace_bytes(0, 8, 32, _lib.MSDA_BF16, 0) == 0


def test_deterministic_backward_is_refused():
    """float reds only: refused before any device work, on real and on empty problems alike"""
    n0 = _lib.launch_count()
    for kw in ({}, {"B": 0}, {"Tq": 0}, {"grads": FAKE, "ptr": FAKE, "meta": FAKE}):
        assert bwd(flags=_lib.FLAG_DETERMINISTIC, **kw) == UNSUPPORTED, kw
        assert b"deterministic" in last_error()
    assert _lib.launch_count() == n0


@pytest.mark.parametrize("dtype", [_lib.MSDA_F32, _lib.MSDA_BF16, _lib.MSDA_F16, _lib.MSDA_BF16_AUX16,
                                   _lib.MSDA_F16_AUX16])
def test_empty_problems_do_nothing(dtype):
    n0 = _lib.launch_count()
    for kw in ({"B": 0}, {"Tq": 0, "mq": 0}, {"B": 0, "D": 24}, {"H": 0}):
        assert fwd(dtype=dtype, **kw) == 0, kw
        assert bwd(dtype=dtype, **kw) == 0, kw
    assert fwd(dtype=dtype, flags=_lib.FLAG_DETERMINISTIC, B=0) == 0    # the forward ignores the flag
    assert _lib.launch_count() == n0


def test_slim_builds_stub_the_packed_entry_points():
    """Slim variant builds (-DMSDA_EXP_SLIM) carry no packed kernels: the host functions behind the entry points
    return MSDA_ERR_UNSUPPORTED there (checked on the preprocessed sources)."""
    nvcc = "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("no nvcc")
    csrc = os.path.join(ROOT, "ir_ads_b200", "csrc")
    for unit, fn in (("msda_fwd.cu", "fwd_packed"), ("msda_bwd_aux.cu", "bwd_packed")):
        res = subprocess.run([nvcc, "-std=c++17", "-E", "-DMSDA_EXP_SLIM", "-x", "cu", os.path.join(csrc, unit)],
                             capture_output=True, text=True)
        assert res.returncode == 0, res.stderr[-2000:]
        body = res.stdout[res.stdout.rindex(f"int {fn}("):]
        body = body[:body.index("}")]
        assert "slim build: no packed kernels" in body and "launch_" not in body


def test_c_program_calls_the_packed_entry_points(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "packed.c"
    src.write_text(r'''
#include <stdio.h>
#include "msda.h"
int main(void) {
  /* empty problems: MSDA_OK, no device work */
  if (msda_packed_forward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 2, 0, 100, 8, 32, 4, 100, 4, 60, 60, NULL,
                          MSDA_F32, 0u) != MSDA_OK) return 1;
  if (msda_packed_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, 4, 2, 100, 8, 32, 4, 0, 4, 60, 0, NULL,
                           NULL, NULL, NULL, 0, MSDA_BF16_AUX16, 0u) != MSDA_OK) return 2;
  /* head dim 24 and the deterministic backward are refused */
  if (msda_packed_forward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 2, 2, 100, 8, 24, 4, 100, 4, 60, 60, NULL,
                          MSDA_F32, 0u) != MSDA_ERR_UNSUPPORTED) return 3;
  if (msda_packed_backward(NULL, NULL, NULL, NULL, NULL, NULL, NULL, NULL, 2, 2, 100, 8, 32, 4, 100, 4, 60, 60, NULL,
                           NULL, NULL, NULL, 0, MSDA_F16, MSDA_FLAG_DETERMINISTIC) != MSDA_ERR_UNSUPPORTED) return 4;
  if (msda_packed_backward_workspace_bytes(100, 8, 32, MSDA_F16, 0u) != (size_t)100 * 8 * 32 * 4) return 5;
  printf("packed abi ok\n");
  return 0;
}
''')
    exe = tmp_path / "packed"
    libdir = os.path.dirname(_lib.LIB_PATH)
    cmd = ["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src),
           "-o", str(exe), "-L", libdir, "-l:" + os.path.basename(_lib.LIB_PATH), "-Wl,-rpath," + libdir,
           "-Wl,-rpath,/usr/local/cuda/lib64", "-Wl,--allow-shlib-undefined"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0 and "packed abi ok" in run.stdout, (run.returncode, run.stdout, run.stderr)


def _interp_extents(h, w, Hp, Wp, shapes):
    mask = torch.ones(1, 1, Hp, Wp)
    mask[..., :h, :w] = 0
    out = []
    for H, W in shapes:
        m = F.interpolate(mask, size=(H, W), mode="nearest")[0, 0].bool()
        valid = ~m
        hv, wv = int(valid[:, 0].sum()), int(valid[0, :].sum())
        assert bool(valid[:hv, :wv].all()) and int(valid.sum()) == hv * wv     # a top-left rectangle
        out.append((hv, wv))
    return out


def test_valid_extents_match_interpolated_masks():
    """valid_extents against F.interpolate(mask, size, mode="nearest") of CPU masks: detrex-like size mixes (shorter
    side 480..800 step 32, longer side capped at 1333), levels at strides 8 / 16 / 32 / 64 of the padded size rounded
    up as a ResNet does, plus odd sizes, single-pixel images and unpadded images."""
    rng = random.Random(5)
    cases = []
    for _ in range(60):
        sizes = []
        for _ in range(rng.choice((1, 2, 3))):
            s = rng.randrange(480, 801, 32)
            l = min(1333, int(s * rng.choice((1.0, 1.33, 1.5, 1.78))))
            sizes.append((s, l) if rng.random() < 0.5 else (l, s))
        Hp, Wp = max(h for h, _ in sizes), max(w for _, w in sizes)
        Hp, Wp = -(-Hp // 32) * 32, -(-Wp // 32) * 32                     # size_divisibility 32
        cases.append((sizes, (Hp, Wp)))
    cases += [([(1, 1), (37, 53)], (37, 53)), ([(64, 64)], (64, 64)), ([(17, 300), (301, 5)], (301, 300))]
    for sizes, (Hp, Wp) in cases:
        shapes = []
        for s in (8, 16, 32, 64):
            shapes.append((-(-Hp // s), -(-Wp // s)))
        shapes += [(Hp, Wp), (2 * Hp, 2 * Wp), (max(1, Hp // 3), max(1, Wp // 7))]
        got = valid_extents(sizes, (Hp, Wp), shapes)
        for (h, w), ext in zip(sizes, got):
            assert ext == _interp_extents(h, w, Hp, Wp, shapes), (h, w, Hp, Wp)


def test_packing_tables_and_reference_points_on_cpu():
    """PackedLevels' host counts, metadata rows and padded-layout tables; pack_levels / unpack_tokens round trip;
    packed_reference_points = the valid rows of get_reference_points(get_valid_ratio(masks)) bit for bit."""
    from ir_ads_b200.encoder import flatten_levels, get_reference_points
    from ir_ads_b200.packing import PackedLevels, pack_levels, packed_reference_points, unpack_tokens
    sizes, padded = [(61, 90), (96, 64), (96, 90)], (96, 90)
    shapes = [(12, 12), (6, 6), (3, 3), (2, 2)]
    ext = valid_extents(sizes, padded, shapes)
    pk = PackedLevels(ext, shapes, "cpu")
    assert pk.batch == 3 and pk.padded_len == 144 + 36 + 9 + 4
    assert pk.value_counts == [sum(h * w for h, w in e) for e in ext] == pk.query_counts
    assert pk.meta.shape == (3, 4 + 3 * 4) and pk.meta[1, :4].tolist() == [pk.value_counts[0], pk.value_counts[1],
                                                                            pk.value_counts[0], pk.value_counts[1]]
    assert 0.0 < pk.padded_fraction() < 1.0 and pk.value_counts[2] == pk.padded_len
    masks, feats, pos = [], [], []
    g = torch.Generator().manual_seed(0)
    img_mask = torch.ones(3, *padded)
    for b, (h, w) in enumerate(sizes):
        img_mask[b, :h, :w] = 0
    for H, W in shapes:
        masks.append(F.interpolate(img_mask[None], size=(H, W)).bool()[0])
        feats.append(torch.randn(3, 8, H, W, generator=g))
        pos.append(torch.randn(3, 8, H, W, generator=g))
    lvl = torch.randn(4, 8, generator=g)
    feat, mask, pos_flat, _, _, level_shapes, ratios = flatten_levels(feats, masks, pos, lvl)
    assert torch.equal(mask, pk.padding_mask) and torch.equal(ratios, pk.valid_ratios)
    x, p = pack_levels(feats, pk, pos, lvl)
    assert torch.equal(x, feat[~mask]) and torch.equal(p, pos_flat[~mask])
    back, m = unpack_tokens(x, pk)
    assert torch.equal(back, feat.masked_fill(mask[..., None], 0)) and torch.equal(m, mask)
    ref = get_reference_points(level_shapes, ratios, "cpu")
    assert torch.equal(packed_reference_points(pk), ref[~mask])
    cross = pk.cross(7)
    assert cross is pk.cross(7) and cross.total_query == 21 and cross.meta[:, 2].tolist() == [0, 7, 14]

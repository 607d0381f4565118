"""The timing scripts under tools/ without a GPU: every one parses its command line, and the shared helpers in
tools/timing.py behave as the scripts rely on."""
import glob
import importlib.util
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOLS = os.path.join(ROOT, "tools")
SCRIPTS = sorted(glob.glob(os.path.join(TOOLS, "bench_*.py"))) + [os.path.join(TOOLS, "sweep.py")]
NO_DEVICE = dict(os.environ, CUDA_VISIBLE_DEVICES="")   # any CUDA call fails


def _timing():
    spec = importlib.util.spec_from_file_location("timing", os.path.join(TOOLS, "timing.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("script", SCRIPTS, ids=os.path.basename)
def test_help_runs_without_a_device(script):
    res = subprocess.run([sys.executable, script, "--help"], capture_output=True, text=True, env=NO_DEVICE, cwd=ROOT)
    assert res.returncode == 0, res.stderr
    assert res.stdout.startswith("usage:")


def test_card_raises_without_a_device():
    code = f"import sys; sys.path.insert(0, {TOOLS!r}); import timing; timing.card()"
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=NO_DEVICE, cwd=ROOT)
    assert res.returncode != 0
    assert "RuntimeError: no CUDA device" in res.stderr


# (set_bytes, lo, hi) -> sets, as the scripts computed them inline: the DCNv3 core and module stages
# (bench_dcnv3_fused, bench_autocast_native), DCNv2 at B = 2 and 8 (bench_dcnv2), the cfg2 encoder at B = 8
@pytest.mark.parametrize("set_bytes, lo, hi, sets", [
    (1014988800, 1, 8, 1), (507494400, 1, 8, 1), (253747200, 1, 8, 2), (126873600, 1, 8, 4), (391372800, 1, 8, 2),
    (550502400, 1, 4, 1), (275251200, 1, 4, 2), (137625600, 1, 4, 3), (68812800, 1, 4, 4),
    (136806400, 2, 8, 3), (34201600, 2, 8, 8), (17203200, 2, 8, 8), (8601600, 2, 8, 8),
    (547225600, 2, 8, 2), (68812800, 2, 8, 6), (34406400, 2, 8, 8),
    (364101632, 1, 3, 2),
])
def test_rotations(set_bytes, lo, hi, sets):
    assert _timing().rotations(set_bytes, lo, hi) == sets

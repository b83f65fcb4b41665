"""CPU: the schedule of the FK / Jacobian-only specialised kernels (kin_gen_skeleton.cuh, KSCHED: tiles claimed from a
counter, inputs prefetched into L2 one epoch at a time), checked without a GPU: which calls select it, and -- in the
NVRTC-compiled SoA headline kernel -- that the tile claim is one atomic, the prefetch is the bulk L2 prefetch, and no
grid-wide barrier (spin loop) is left; AoS calls keep the input batches behind a grid-wide barrier."""
import re
import shutil
import subprocess

import pytest

from kinematics_jl_b200 import lib as L
from test_const_fill_cpu import _dump


def _sass(cubin, func):
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    try:
        sass = subprocess.run([cuobjdump, "-sass", "-fun", func, str(cubin)], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.CalledProcessError):
        pytest.skip("cuobjdump not available")
    assert "Function : " + func in sass
    return sass


@pytest.mark.parametrize("tag, layout", [("soa", None), ("tiled", "tiled")])
def test_claimed_tiles_in_the_compiled_kernel(tmp_path, tag, layout):
    out = _dump(tmp_path, tag, 1 << 24, {None: None, "tiled": L.TILED32}[layout], compile_=1)
    cfg = (out / "kin_gen_config.h").read_text()
    assert "#define KSCHED 1" in cfg and "#define KPFD 1" in cfg
    sass = _sass(out / "kin_gen.cubin", "kin_gen_kernel")
    assert len(re.findall(r"\bATOMG\.", sass)) == 1                     # the tile claim, nothing else
    assert re.search(r"\bUBLKPF\b", sass)                               # cp.async.bulk.prefetch.L2
    assert "NANOSLEEP" not in sass and "TRAP" not in sass               # no barrier spin loop, no timeout trap
    assert not re.search(r"\bLDGSTS\b", sass)                           # no cp.async input batches


@pytest.mark.parametrize("tag, n, layout, precision, on", [
    ("soa_big", 1 << 20, None, None, 1),
    ("soa_f32", 1 << 20, None, "f32", 1),
    ("tiled", 1 << 20, "tiled", None, 1),
    ("aos", 1 << 20, "aos", None, 0),                # AoS keeps the input batches (measured faster there)
    ("soa_small", 1 << 16, None, None, 0),       # below kSchedMinBatch: static tiles
])
def test_schedule_selection(tmp_path, tag, n, layout, precision, on):
    lay = {None: None, "tiled": L.TILED32, "aos": L.AOS}[layout]
    out = _dump(tmp_path, tag, n, lay, L.F32 if precision == "f32" else None)
    cfg = (out / "kin_gen_config.h").read_text()
    assert ("#define KSCHED %d" % on) in cfg
    assert ("#define KQB 0" in cfg) == (layout != "aos" or n < (1 << 18))

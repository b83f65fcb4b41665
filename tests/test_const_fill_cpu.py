"""CPU: the table of configuration-independent output rows the code generator hands to the fill kernel of input-batched
SoA calls (GenOptions::const_fill, kin_gen_skeleton.cuh: kin_const_fill_kernel), checked without a GPU: its rows and values against the ORACLE
on random configurations, its selection (SoA input-batched FK / Jacobian calls only), and -- in the NVRTC-compiled
kernel -- that phase 1 then stores only the 173 varying rows of Fetch's FK-all + gripper Jacobian."""
import ctypes as C
import re
import shutil
import struct
import subprocess

import numpy as np
import pytest

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import make_desc
from oracle import ref_model as R
import scenes


def _dump(tmp_path, tag, n, layout=None, precision=None, compile_=0):
    import scene_fetch
    lib = L.lib()
    if not lib.kin_jit_status().startswith(b"ok"):
        pytest.skip("NVRTC not available: " + lib.kin_jit_status().decode())
    m, joints, _ = scene_fetch.product_fetch(False)
    d, keep = make_desc(m, [j.id for j in joints])
    fk = np.arange(1, 26, dtype=np.int32)
    jac = np.array([K.find_link(m, "gripper_link").id], dtype=np.int32)
    ip = C.POINTER(C.c_int32)
    c = L.KinCall()
    c.precision, c.layout, c.n, c.q = precision or L.F64, L.SOA if layout is None else layout, n, 1
    c.n_fk_links, c.fk_links, c.T_out = 25, fk.ctypes.data_as(ip), 1
    c.n_jac_links, c.jac_links, c.J_out, c.with_rot = 1, jac.ctypes.data_as(ip), 1, 1
    c.truncation_dist = float("inf")
    out = tmp_path / tag
    out.mkdir()
    L.check(lib.kin_codegen_dump(C.byref(d), C.byref(c), compile_, str(out).encode()))
    return out


def _hexval(lit):
    v = lit.strip()[len("real("):-1]
    return float.fromhex(v) if "x" in v else float(v)


def test_constant_row_table_holds_in_the_oracle(tmp_path):
    out = _dump(tmp_path, "big", 1 << 24, compile_=1)
    cfg = (out / "kin_gen_config.h").read_text()
    assert "#define KCFILL 1" in cfg
    nc = int(re.search(r"constexpr int KNCF = (\d+);", cfg).group(1))
    rows = [int(x) for x in re.search(r"KCF_ROW\[KNCF\] = \{([^}]*)\}", cfg).group(1).replace("\n", " ").split(",")]
    vals = [_hexval(x) for x in re.findall(r"real\([^)]*\)", re.search(r"KCF_VAL\[KNCF\] = \{([^}]*)\}", cfg, re.S).group(1))]
    assert nc == 175 and len(rows) == nc and len(vals) == nc
    # the table's values are the literals phase 1 stores for those rows, bit for bit (sign of zero included)
    src = (out / "kin_gen_phase1.inc").read_text()
    stores = {(a, int(k)): e.strip() for a, k, e in re.findall(r"KST_([TJ])\((\d+), ([^;]*)\);", src)}
    assert len(stores) == 348
    mo, jo, _ = scenes.oracle_fetch(False)
    q = scenes.random_configs(jo, 64, False, seed=11)
    T = R.batch_fk(mo, jo, q, mo.links[:25])[:, :, :3, :].transpose(0, 1, 3, 2).reshape(len(q), 300)
    J = R.batch_jacobian(mo, jo, q, [R.find_link(mo, "gripper_link")], True)[:, 0].transpose(0, 2, 1).reshape(len(q), 48)
    for row, v in zip(rows, vals):
        arr, k = ("T", row) if row >= 0 else ("J", -1 - row)
        lit = stores[(arr, k)]
        assert re.fullmatch(r"real\([^)]*\)", lit), (arr, k, lit)
        assert struct.pack("<d", _hexval(lit)) == struct.pack("<d", v), (arr, k)
        np.testing.assert_allclose((T if arr == "T" else J)[:, k], v, rtol=0, atol=1e-15, err_msg="%s row %d" % (arr, k))
    # every literal store of phase 1 is in the table: phase 1 keeps the 173 others
    assert sum(1 for e in stores.values() if re.fullmatch(r"real\([^)]*\)", e)) == nc
    # ... and the compiled kernel stores only those per thread (STG.E.EF.64: the streaming stores of KST_*)
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    try:
        sass = subprocess.run([cuobjdump, "-sass", str(out / "kin_gen.cubin")], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.CalledProcessError):
        pytest.skip("cuobjdump not available")
    assert len(re.findall(r"\bSTG\.E\.EF\.64\b", sass)) == 348 - nc
    assert re.search(r"\bSTG\.E\.ENL2\.256\b", sass) and "kin_const_fill_kernel" in sass     # the fill kernel's 32-byte stores


@pytest.mark.parametrize("tag, n, layout, precision, on", [
    ("soa_big", 1 << 20, None, None, 1),
    ("soa_f32", 1 << 20, None, "f32", 1),
    ("soa_small", 1 << 16, None, None, 0),           # below the input-batching threshold
    ("tiled", 1 << 20, "tiled", None, 0),            # a constant row is not contiguous in the tiled / AoS layouts
    ("aos", 1 << 20, "aos", None, 0),
])
def test_constant_fill_is_selected_for_input_batched_soa_calls_only(tmp_path, tag, n, layout, precision, on):
    lay = {None: None, "tiled": L.TILED32, "aos": L.AOS}[layout]
    out = _dump(tmp_path, tag, n, lay, L.F32 if precision == "f32" else None)
    cfg = (out / "kin_gen_config.h").read_text()
    assert ("#define KCFILL %d" % on) in cfg

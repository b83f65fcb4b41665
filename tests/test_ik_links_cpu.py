"""Multi-link pose targets of the batched IK (kin_ik_solve_links), host side: the C declaration and the ctypes binding of
the new entry point, the Julia method, the Python argument checks (made before anything touches a device), and the
generated one-launch IK kernel for two links of the dual-arm model, compiled for sm_100a without a GPU."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import make_desc
from conftest import ROOT
import scenes
import scenes_dual_arm as DA


def _read(*parts):
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def test_header_declares_kin_ik_solve_links_and_keeps_the_abi():
    h = _read("include", "kin_b200.h")
    decl = re.search(r"KIN_API int kin_ik_solve_links\(([^)]*)\);", h)
    assert decl, "kin_ik_solve_links is not declared"
    args = [" ".join(a.split()) for a in decl.group(1).split(",")]
    assert args == ["KinModel *model", "const KinIkCall *call", "int32_t n_links", "const int32_t *link_ids",
                    "const int32_t *with_rots", "int32_t self_collision", "double self_margin", "void *self_dmin_out"]
    assert re.search(r"#define KIN_IK_MAX_LINKS 4\b", h)
    assert re.search(r"#define KIN_B200_ABI_VERSION 4\b", h)
    body = h[h.index("typedef struct {\n    int64_t n;\n    int32_t link_id;"):h.index("} KinIkCall;")]
    assert body.rstrip().endswith("*/") and "void *dmin_out;" in body.splitlines()[-1]
    assert "(n_links - 1)(12 + rows n_dof)" in h


def test_ctypes_binding_exports_kin_ik_solve_links():
    assert "kin_ik_solve_links" in L.EXPORTS
    src = _read("kinematics.jl_b200", "lib.py")
    assert ("L.kin_ik_solve_links.argtypes = [C.c_void_p, C.POINTER(KinIkCall), C.c_int32, C.POINTER(C.c_int32), "
            "C.POINTER(C.c_int32),\n                                         C.c_int32, C.c_double, C.c_void_p]") in src


def test_julia_method_calls_kin_ik_solve_links():
    jl = _read("julia", "CUDABackend.jl")
    assert re.search(r"function inverse_kinematics_batch\(dm::DeviceMechanism, links::AbstractVector\{<:Link\}", jl)
    assert "ccall((:kin_ik_solve_links, libkin)" in jl


class _Link:
    def __init__(self, i):
        self.id = i


@pytest.mark.parametrize("call", ["ik_solve_device", "inverse_kinematics_batch"])
def test_malformed_link_lists_raise_before_any_device_call(call):
    fn = getattr(K, call)
    a, b = _Link(3), _Link(5)
    with pytest.raises(ValueError, match="1..4 links"):
        fn(None, [], [], None, None)
    with pytest.raises(ValueError, match="1..4 links"):
        fn(None, [_Link(i) for i in range(1, 6)], [], None, None)
    with pytest.raises(ValueError, match="distinct"):
        fn(None, [a, a], [], None, None)
    with pytest.raises(ValueError, match="with_rot"):
        fn(None, [a, b], [], None, None, with_rot=[True])


def test_single_problem_driver_checks_the_lists():
    a, b = _Link(3), _Link(5)
    with pytest.raises(ValueError, match="one target pose per link"):
        K.inverse_kinematics(None, [a, b], [], [np.zeros(6)])
    with pytest.raises(ValueError, match="with_rot"):
        K.inverse_kinematics(None, [a, b], [], [np.zeros(6)] * 2, with_rot=[True, False, True])


def test_batch_target_width_is_checked_before_the_solve():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("the targets are moved to the device first")
    m, joints, _ = scenes.product_fetch(False)
    links = [K.find_link(m, "gripper_link"), K.find_link(m, "elbow_flex_link")]
    with pytest.raises(ValueError, match="6 \\* number of links"):
        K.inverse_kinematics_batch(m, links, joints, np.zeros((4, 6)), np.zeros((4, 8)))


def _dump_two_tools(tmp_path, with_base, mask, tag):
    lib = L.lib()
    if not lib.kin_jit_status().startswith(b"ok"):
        pytest.skip("NVRTC not available: " + lib.kin_jit_status().decode())
    m, joints, _, _ = DA.product(with_base)
    d, keep = make_desc(m, [j.id for j in joints])
    ids = np.array([K.find_link(m, "l_tool").id, K.find_link(m, "r_tool").id], dtype=np.int32)
    ip = C.POINTER(C.c_int32)
    c = L.KinCall()
    c.precision, c.layout, c.n, c.q = L.F64, L.SOA, 1 << 18, 1
    c.n_fk_links, c.fk_links, c.T_out = 2, ids.ctypes.data_as(ip), 1
    c.n_jac_links, c.jac_links, c.J_out, c.with_rot, c.rpy_jac = 2, ids.ctypes.data_as(ip), 1, 1, 1
    c.truncation_dist = float("inf")
    out = tmp_path / tag
    out.mkdir()
    os.environ["KIN_DUMP_IK"] = mask
    try:
        L.check(lib.kin_codegen_dump(C.byref(d), C.byref(c), 1, str(out).encode()))
    finally:
        del os.environ["KIN_DUMP_IK"]
    return out


@pytest.mark.parametrize("with_base", [False, True])
def test_two_link_ik_kernel_compiles_for_sm_100a(tmp_path, with_base):
    out = _dump_two_tools(tmp_path, with_base, "3", "both")
    cfg = (out / "kin_gen_config.h").read_text()
    assert "#define KIK 1" in cfg and "#define KIKROT 0x3u" in cfg
    assert re.search(r"KND = %d, .*KNFK = 2, KNJAC = 2, KROWS = 6;" % (18 if with_base else 15), cfg)
    cubin = out / "kin_gen.cubin"
    assert cubin.stat().st_size > 0
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([tool, "-sass", str(cubin)], capture_output=True, text=True, check=True).stdout
    assert re.findall(r"Function : (\S+)", sass) == ["kin_ik_kernel"]
    res = subprocess.run([tool, "-res-usage", str(cubin)], capture_output=True, text=True, check=True).stdout
    regs = re.search(r"REG:(\d+) STACK:(\d+)", res)
    assert regs and 0 < int(regs.group(1)) <= 255
    print("2-link dual-arm IK kernel, %d columns: %s registers, %s B stack" % (18 if with_base else 15, regs.group(1), regs.group(2)))


def test_position_only_link_drops_its_rotation_rows(tmp_path):
    """Mask 0x1: the right tool is position-only; the generated config carries the mask."""
    out = _dump_two_tools(tmp_path, False, "0x1", "mixed")
    assert "#define KIKROT 0x1u" in (out / "kin_gen_config.h").read_text()

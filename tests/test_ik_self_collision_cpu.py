"""Self-collision as a hard constraint of the batched IK (kin_ik_solve_self), host side: the C declaration and the
ctypes binding of the new entry point, the Julia keyword, the Python argument handling (checked before anything
touches a device) and the pair tables the GPU tests and the benchmark use."""
import os
import re

import pytest

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from conftest import ROOT
import scenes
import scenes_dual_arm as DA

FETCH_IGNORE = [("wrist_flex_link", "elbow_flex_link")]


def _read(*parts):
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def test_header_declares_kin_ik_solve_self_and_keeps_the_abi():
    h = _read("include", "kin_b200.h")
    decl = re.search(r"KIN_API int kin_ik_solve_self\(([^)]*)\);", h)
    assert decl, "kin_ik_solve_self is not declared"
    args = [a.strip() for a in decl.group(1).split(",")]
    assert args == ["KinModel *model", "const KinIkCall *call", "double self_margin", "void *self_dmin_out"]
    assert re.search(r"#define KIN_B200_ABI_VERSION 4\b", h)
    # the call struct is unchanged: its last field is still dmin_out
    body = h[h.index("typedef struct {\n    int64_t n;\n    int32_t link_id;"):h.index("} KinIkCall;")]
    assert body.rstrip().endswith("*/") and "void *dmin_out;" in body.splitlines()[-1]


def test_ctypes_binding_exports_kin_ik_solve_self():
    assert "kin_ik_solve_self" in L.EXPORTS
    src = _read("kinematics.jl_b200", "lib.py")
    assert "L.kin_ik_solve_self.argtypes = [C.c_void_p, C.POINTER(KinIkCall), C.c_double, C.c_void_p]" in src


def test_julia_keyword_calls_kin_ik_solve_self():
    jl = _read("julia", "CUDABackend.jl")
    sig = jl[jl.index("function inverse_kinematics_batch("):]
    sig = sig[:sig.index(")\n")]
    assert "self_margin=nothing" in sig
    assert "ccall((:kin_ik_solve_self, libkin)" in jl


@pytest.mark.parametrize("call", ["ik_solve_device", "inverse_kinematics_batch"])
def test_self_margin_without_sscc_raises_before_any_device_call(call):
    # no mechanism, no targets, no CUDA: the check comes first
    with pytest.raises(ValueError, match="sscc"):
        getattr(K, call)(None, None, [], None, None, self_margin=0.02)


def test_single_problem_driver_self_margin_without_sscc_raises():
    with pytest.raises(ValueError, match="sscc"):
        K.inverse_kinematics(None, None, [], None, self_margin=0.02)


def test_non_finite_self_margin_raises_before_any_device_call():
    m, joints, sscc = scenes.product_fetch(False)
    for bad in (float("nan"), float("inf")):
        with pytest.raises(ValueError, match="finite"):
            K.ik_solve_device(m, None, joints, None, None, sscc=sscc, self_margin=bad)


def test_pair_tables_of_the_fixtures():
    """The dual-arm model keeps the default policy (145 pairs); on Fetch the constant pair that overlaps by 5.5 mm in
    every configuration is ignored, which leaves 64 pairs."""
    _, joints, sscc = scenes.product_fetch(False)
    assert len(K.self_collision_pairs(sscc, joints, ignore=FETCH_IGNORE)) == 64
    for with_base in (False, True):
        _, joints, sscc, _ = DA.product(with_base)
        assert len(K.self_collision_pairs(sscc, joints)) == 145

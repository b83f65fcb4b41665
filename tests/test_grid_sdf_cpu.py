"""Voxel-grid SDF rows (KIN_PRIM_GRID), host side: known answers of the restatement the GPU tests compare against
(tests/grid_sdf_ref.py), the C declarations, the ctypes and Julia bindings, and an sm_100a compile of a generated fused
kernel whose table carries general rows, without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import make_desc
from conftest import ROOT
from grid_sdf_ref import RefGrid
import scenes

A_FIELD, B_FIELD = np.array([1.0, -0.5, 2.0]), 0.125


def _read(*parts):
    with open(os.path.join(ROOT, *parts)) as f:
        return f.read()


def _affine_grid(pose=None):
    """(9, 7, 5) samples at s = 0.25 of a x + b: every sample is a dyadic rational, exact in float32."""
    g = RefGrid(np.zeros((9, 7, 5)), 0.25, pose)
    P = g.sample_points() if pose is None else RefGrid(np.zeros((9, 7, 5)), 0.25).sample_points()
    g.v = (P @ A_FIELD + B_FIELD).astype(np.float32)
    assert np.array_equal(g.v.astype(np.float64), P @ A_FIELD + B_FIELD)
    return g


def test_affine_field_is_reproduced_inside_with_its_gradient():
    rng = np.random.default_rng(1)
    for pose in (None, _pose(0.3, -0.2, 0.9, [0.1, -0.4, 0.7])):
        g = _affine_grid(pose)
        half = (g.n - 1) / 2.0 * g.s
        Rm = g.pose[:3, :3]
        for _ in range(200):
            l = rng.uniform(-half, half)
            p = Rm @ l + g.pose[:3, 3]
            d = g(p)
            assert abs(d - (A_FIELD @ g.local(p) + B_FIELD)) < 1e-12
            assert np.allclose(g.gradient(p, analytic=True), Rm @ A_FIELD, atol=1e-12, rtol=0)


def _pose(r, p, y, t):
    cr, sr, cp, sp, cy, sy = np.cos(r), np.sin(r), np.cos(p), np.sin(p), np.cos(y), np.sin(y)
    M = np.eye(4)
    M[:3, :3] = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]]) @ np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]]) @ \
        np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
    M[:3, 3] = t
    return M


def test_values_at_sample_points_are_the_stored_floats():
    rng = np.random.default_rng(2)
    g = RefGrid(rng.normal(size=(6, 5, 4)).astype(np.float32), 0.125)     # dyadic: the samples' coordinates are exact
    P = g.sample_points()
    for idx in np.ndindex(*g.v.shape):
        assert g(P[idx]) == float(g.v[idx])


def test_continuity_across_cell_faces_and_the_grid_box():
    rng = np.random.default_rng(3)
    g = RefGrid(rng.normal(size=(5, 6, 7)).astype(np.float32), 0.2)
    half = (g.n - 1) / 2.0 * g.s
    for _ in range(100):
        p = rng.uniform(-half, half)
        ax = rng.integers(3)
        p[ax] = (rng.integers(g.n[ax]) - (g.n[ax] - 1) / 2.0) * g.s       # on a cell face (or the box face)
        for dlt in (1e-9, -1e-9):
            q = p.copy()
            q[ax] += dlt
            assert abs(g(q) - g(p)) < 1e-7
    # across the grid box boundary: inside and outside the face agree in the limit
    for ax in range(3):
        p = np.zeros(3)
        p[ax] = half[ax]
        assert abs(g(p + 1e-9 * np.eye(3)[ax]) - g(p)) < 1e-8
        assert abs(g(p - 1e-9 * np.eye(3)[ax]) - g(p)) < 1e-7


def test_outside_value_adds_the_distance_to_the_grid_box():
    rng = np.random.default_rng(4)
    g = RefGrid(rng.normal(size=(4, 4, 4)).astype(np.float32), 0.5)
    half = (g.n - 1) / 2.0 * g.s
    for _ in range(100):
        p = rng.uniform(-4, 4, size=3)
        c = np.clip(p, -half, half)
        assert abs(g(p) - (g(c) + np.linalg.norm(p - c))) < 1e-12
    far = np.array([1e6, -2e6, 3e6])
    assert np.isfinite(g(far)) and abs(g(far) - np.linalg.norm(far - np.clip(far, -half, half))) < 10


def test_forward_difference_agrees_with_the_analytic_gradient_away_from_faces():
    rng = np.random.default_rng(5)
    g = RefGrid(rng.normal(size=(6, 6, 6)).astype(np.float32), 0.3, _pose(0.1, 0.5, -0.7, [0.2, 0.0, -0.1]))
    n_checked = 0
    for _ in range(400):
        p = rng.uniform(-2.5, 2.5, size=3)
        u = g.local(p) / g.s + (g.n - 1) / 2.0
        if np.min(np.abs(u - np.round(u))) < 1e-3:        # near a cell face: the FD may straddle it
            continue
        assert np.allclose(g.gradient(p), g.gradient(p, analytic=True), atol=1e-5, rtol=0)
        n_checked += 1
    assert n_checked > 300


def test_header_declares_the_grid_abi():
    h = _read("include", "kin_b200.h")
    assert re.search(r"KIN_PRIM_GRID = 3 \}", h)
    assert re.search(r"#define KIN_B200_ABI_VERSION 4\b", h)
    assert re.search(r"#define KIN_MAX_GRID_VALUES \(1 << 28\)", h)
    want = {
        "kin_grid_create": ["int32_t nx", "int32_t ny", "int32_t nz", "double spacing", "const float *values", "KinGrid **out"],
        "kin_grid_set_values": ["KinGrid *grid", "const float *values", "void *stream"],
        "kin_grid_destroy": ["KinGrid *grid"],
        "kin_model_set_scene": ["KinModel *model", "int32_t n", "const int32_t *kinds", "const double *pose",
                                "const double *size", "const KinGrid *const *grids"],
        "kin_sdf_points_scene": ["int32_t n", "const int32_t *kinds", "const double *pose", "const double *size",
                                 "const KinGrid *const *grids", "int32_t precision", "int32_t layout", "const void *pts",
                                 "int64_t n_pts", "int32_t grad_mode", "void *vals_out", "void *grads_out",
                                 "int32_t *argmin_out", "void *stream"],
    }
    for name, args in want.items():
        decl = re.search(r"KIN_API int %s\(([^)]*)\);" % name, h)
        assert decl, name
        assert [" ".join(a.split()) for a in decl.group(1).split(",")] == args, name
    # the lerp order the restatement follows is the one the header pins
    assert "a_jk = lerp(v_0jk, v_1jk, t_x),  b_k = lerp(a_0k, a_1k, t_y),  f = lerp(b_0, b_1, t_z)" in h


def test_bindings_export_the_grid_abi():
    names = {"kin_grid_create", "kin_grid_set_values", "kin_grid_destroy", "kin_model_set_scene", "kin_sdf_points_scene"}
    assert names <= set(L.EXPORTS)
    assert L.PRIM_GRID == 3 and L.MAX_GRID_VALUES == 1 << 28
    jl = _read("julia", "CUDABackend.jl")
    for n in ("kin_grid_create", "kin_grid_set_values", "kin_grid_destroy", "kin_model_set_scene"):
        assert "ccall((:%s, libkin)" % n in jl
    assert "finalizer(x -> ccall((:kin_grid_destroy, libkin)" in jl


def test_grid_sdf_checks_its_shape_before_any_device_call():
    with pytest.raises(ValueError, match="nx, ny, nz"):
        K.GridSDF(np.zeros((4, 4)), 0.1)


def test_generated_fused_kernel_with_general_rows_compiles_for_sm_100a(tmp_path):
    """A table with a grid row turns KPRIMS on exactly like a sphere row: the generated source is the one of any
    general table (KIN_JIT_FORCE_PRIMS on a box table), and its grid branch must compile under NVRTC for sm_100a."""
    lib = L.lib()
    if not lib.kin_jit_status().startswith(b"ok"):
        pytest.skip("NVRTC not available: " + lib.kin_jit_status().decode())
    m, joints, sscc = scenes.product_fetch(False)
    poses, widths = scenes.fridge_boxes_host()
    d, keep = make_desc(m, [j.id for j in joints], (sscc._parents, sscc._centers, sscc.sphere_radii), (poses, widths))
    c = L.KinCall()
    c.precision, c.layout, c.n, c.q = L.F64, L.SOA, 1 << 20, 1
    c.truncation_dist = float("inf")
    c.vals_out, c.grads_out = 1, 1
    c.grad_mode = L.GRAD_ANALYTIC
    os.environ["KIN_JIT_FORCE_PRIMS"] = "1"
    try:
        L.check(lib.kin_codegen_dump(C.byref(d), C.byref(c), 1, str(tmp_path).encode()))
    finally:
        del os.environ["KIN_JIT_FORCE_PRIMS"]
    assert "#define KPRIMS 1" in (tmp_path / "kin_gen_config.h").read_text()
    assert "grid_eval" in (tmp_path / "kin_device_math.cuh").read_text()
    assert (tmp_path / "kin_gen.cubin").stat().st_size > 0

"""CPU: the product's host half (URDF reader -> KinModelDesc -> compiled kinematic program) against
the oracle.  The program is executed by the numpy interpreter of tests/program_interp.py, which
mirrors the kernel.  What this pins without a GPU: link/joint id assignment, topological flattening,
constant folding of fixed chains, relevance masks, sphere pre-composition, box inversion, scratch
(stale column) ordering."""
import os
import re

import numpy as np
import pytest

import kinematics_jl_b200 as K
from oracle import ref_model as R
from conftest import DATA, GOLDEN
import scenes
from program_interp import dump_program, run_program


def test_library_exports_every_declared_symbol():
    import re
    hdr = open(os.path.join(os.path.dirname(DATA), "include", "kin_b200.h")).read()
    declared = set(re.findall(r"KIN_API [^;(]*?\b(kin_\w+)\s*\(", hdr))
    from kinematics_jl_b200 import lib as L
    assert declared == set(L.EXPORTS)
    for name in declared:
        assert hasattr(L.lib(), name), name
    assert L.lib().kin_abi_version() == 4
    assert L.lib().kin_build_id().decode() == L.source_id()        # the loaded binary is the one built from these sources


def test_no_device_is_a_loud_error():
    """Runs in a child process that sees no CUDA device, so that it also runs on a machine with a GPU."""
    import subprocess
    import sys
    root = os.path.dirname(DATA)
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import numpy as np, pytest, kinematics_jl_b200 as K, scenes\n"
            "m, joints, _ = scenes.product_fetch()\n"
            "K.set_joint_angles(m, joints, np.zeros(8))\n"
            "with pytest.raises(K.KinError, match='no CUDA device'):\n"
            "    K.get_transform(m, K.find_link(m, 'gripper_link'))\n") % (root, os.path.join(root, "tests"))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr


def test_mechanism_mirror_structure():
    """test_mechanism.jl:3-29, 54-67 through the product's parse_urdf."""
    m = K.parse_urdf(os.path.join(DATA, "fetch.urdf"))
    base = K.find_link(m, "base_link")
    assert {l.name for l in K.child_links(m, base)} == {"r_wheel_link", "l_wheel_link", "torso_lift_link",
                                                        "estop_link", "laser_link", "torso_fixed_link"}
    assert K.isroot(base) and base.pjoint_id == -1
    sh = K.find_link(m, "shoulder_pan_link")
    assert K.parent_joint(m, sh).name == "shoulder_pan_joint"
    assert K.parent_link(m, sh).name == "torso_lift_link"
    assert [l.name for l in K.child_links(m, sh)] == ["shoulder_lift_link"]
    assert [j.name for j in K.child_joints(m, sh)] == ["shoulder_lift_joint"]
    for name in ["r_wheel_link", "l_wheel_link", "r_gripper_finger_link", "l_gripper_finger_link", "bellows_link2",
                 "estop_link", "laser_link", "torso_fixed_link", "head_camera_rgb_optical_frame",
                 "head_camera_depth_optical_frame"]:
        assert K.isleaf(K.find_link(m, name)) and not K.find_link(m, name).cjoint_ids
    shoulder, wrist = K.find_joint(m, "shoulder_pan_joint"), K.find_link(m, "wrist_roll_link")
    assert K.is_relevant(m, K.find_joint(m, "torso_lift_joint"), K.find_link(m, "torso_lift_link"))
    assert K.is_relevant(m, shoulder, wrist) and not K.is_relevant(m, shoulder, base)
    new = K.add_new_link(m, K.Link("mylink", K.User), wrist, [0, 0, 0])
    assert K.is_relevant(m, K.find_joint(m, "torso_lift_joint"), new)
    # the mirror's ids and relevance table equal the oracle's
    mo = R.parse_urdf(os.path.join(DATA, "fetch.urdf"))
    R.add_new_link(mo, "mylink", R.find_link(mo, "wrist_roll_link"), [0, 0, 0])
    assert [l.name for l in m.links] == [l.name for l in mo.links]
    assert [j.name for j in m.joints] == [j.name for j in mo.joints]
    tab = m.rptable
    for j in mo.joints:
        for l in mo.links:
            assert tab[j.id - 1, l.id - 1] == R.is_relevant(mo, j, l)


@pytest.mark.parametrize("with_base", [False, True])
def test_program_fk_jacobian_vs_oracle(with_base):
    m, joints, _ = scenes.product_fetch(with_base)
    mo, jo, _ = scenes.oracle_fetch(with_base)
    q = scenes.random_configs(jo, 64, with_base, seed=1, zeros_every=16)
    link_ids = [l.id for l in m.links]
    h, ti, tr = dump_program(m, [j.id for j in joints], link_ids, link_ids)
    T_ref = R.batch_fk(mo, jo, q, mo.links)
    for rpy_jac in (False, True):
        out = run_program(h, ti, tr, q, with_rot=True, rpy_jac=rpy_jac)
        J_ref = R.batch_jacobian(mo, jo, q, mo.links, True, rpy_jac)
        np.testing.assert_allclose(out["T"], T_ref[:, :, :3, :], rtol=0, atol=2e-14)
        np.testing.assert_allclose(out["J"], J_ref, rtol=1e-12, atol=1e-12)
    out3 = run_program(h, ti, tr, q, with_rot=False)
    np.testing.assert_allclose(out3["J"], R.batch_jacobian(mo, jo, q, mo.links, False), rtol=1e-12, atol=1e-12)


def test_program_frozen_nonzero_joints_and_subset_requests():
    """Un-controlled joints frozen at non-zero angles (head, gripper fingers) fold into constants."""
    m, joints, _ = scenes.product_fetch(False)
    mo, jo, _ = scenes.oracle_fetch(False)
    extra = {"head_pan_joint": 0.4, "head_tilt_joint": -0.3, "l_gripper_finger_joint": 0.02, "bellows_joint": 0.0}
    for name, a in extra.items():
        if name in m.jointid_map:
            K.set_joint_angle(m, K.find_joint(m, name), a)
            R.set_joint_angles(mo, [R.find_joint(mo, name)], [a])
    ctrl = joints[1:6]                    # a strict subset, not starting at the torso
    ctrl_o = jo[1:6]
    K.set_joint_angle(m, joints[0], 0.2)
    R.set_joint_angles(mo, [jo[0]], [0.2])
    q = scenes.random_configs(ctrl_o, 32, False, seed=2)
    names = ["head_camera_rgb_optical_frame", "l_gripper_finger_link", "gripper_link", "base_link", "elbow_flex_link"]
    h, ti, tr = dump_program(m, [j.id for j in ctrl], [K.find_link(m, n).id for n in names],
                             [K.find_link(m, n).id for n in names])
    out = run_program(h, ti, tr, q, with_rot=True, rpy_jac=True)
    lo = [R.find_link(mo, n) for n in names]
    np.testing.assert_allclose(out["T"], R.batch_fk(mo, ctrl_o, q, lo)[:, :, :3, :], rtol=0, atol=2e-14)
    np.testing.assert_allclose(out["J"], R.batch_jacobian(mo, ctrl_o, q, lo, True, True), rtol=1e-12, atol=1e-12)


def test_program_pr2_mini_ground_truth():
    import json
    g = json.load(open(os.path.join(DATA, "ground_truth.json")))
    m = K.parse_urdf(os.path.join(GOLDEN, "pr2_right_arm_mini.urdf"))
    joints = [K.find_joint(m, n) for n in g["joint_names"]]
    links = [K.find_link(m, n) for n in g["link_names"]]
    h, ti, tr = dump_program(m, [j.id for j in joints], [l.id for l in links], [])
    T = run_program(h, ti, tr, np.array([g["angle_vector"]]))["T"][0]
    for Tl, pose in zip(T, g["pose_list"]):
        M = np.eye(4)
        M[:3] = Tl
        np.testing.assert_allclose(Tl[:, 3], pose[:3], rtol=0, atol=1e-14)
        np.testing.assert_allclose(K.rpy(K.Transform(M))[::-1], pose[3:], rtol=0, atol=1e-14)


@pytest.mark.parametrize("with_base", [False, True])
@pytest.mark.parametrize("truncation", [np.inf, 0.08])
def test_program_collision_vs_oracle(with_base, truncation):
    m, joints, sscc = scenes.product_fetch(with_base)
    mo, jo, so = scenes.oracle_fetch(with_base)
    sdf_o = scenes.oracle_fridge_sdf()
    boxes = scenes.fridge_boxes_host()
    q = scenes.random_configs(jo, 96, with_base, seed=3)
    spheres = (sscc._parents, sscc._centers, sscc.sphere_radii)
    h, ti, tr = dump_program(m, [j.id for j in joints], [], [], spheres, boxes)
    for scratch_ref, mode in ((True, R.SCRATCH_REFERENCE), (False, R.SCRATCH_CLEAN)):
        out = run_program(h, ti, tr, q, truncation=truncation, scratch_ref=scratch_ref)
        vals, grads, am = R.batch_collision(so, jo, sdf_o, q, truncation, R.GRAD_FD, mode)
        np.testing.assert_allclose(out["vals"], vals, rtol=1e-12, atol=1e-13)
        assert np.array_equal(out["argmin"], am)
        np.testing.assert_allclose(out["grads"], grads.transpose(0, 2, 1), rtol=0, atol=1e-7)
        if not scratch_ref:        # analytic oracle: the FD gradient is within FD error of it
            _, ga, _ = R.batch_collision(so, jo, sdf_o, q, truncation, R.GRAD_ANALYTIC, mode)
            assert np.abs(out["grads"] - ga.transpose(0, 2, 1)).max() < 1e-4


@pytest.mark.parametrize("with_base", [False, True])
@pytest.mark.parametrize("n_ctrl", [None, 4])
def test_program_synthetic_branching_tree(with_base, n_ctrl):
    """Branching tree, general axes, rpy origins, negative axes, frozen joints at non-zero angles, shuffled
    column order: exercises save slots, the Rodrigues path, general offsets and attachment folding."""
    import scenes_synthetic as SS
    m, joints, sscc, sdf = SS.product(with_base, n_ctrl)
    mo, jo, so, sdf_o = SS.oracle(with_base, n_ctrl)
    if n_ctrl is not None:          # the joints that are not controlled sit at non-zero angles
        for name, a in zip(SS.JOINTS[n_ctrl:], [0.3, -0.4, 0.5, 0.1, -0.2]):
            K.set_joint_angle(m, K.find_joint(m, name), a)
            R.set_joint_angles(mo, [R.find_joint(mo, name)], [a] + ([0, 0, 0] if with_base else []))
    q = SS.random_q(jo, 80, with_base, seed=5)
    ids = [l.id for l in m.links]
    h, ti, tr = dump_program(m, [j.id for j in joints], ids, ids, (sscc._parents, sscc._centers, sscc.sphere_radii),
                             (np.stack(SS.BOX_POSES), np.array(SS.BOX_WIDTHS)))
    if n_ctrl is None and not with_base:
        assert h["so_jf"] > h["so_save"]          # a branching tree needs at least one save slot
    T_ref = R.batch_fk(mo, jo, q, mo.links)
    out = run_program(h, ti, tr, q, with_rot=True, rpy_jac=True)
    np.testing.assert_allclose(out["T"], T_ref[:, :, :3, :], rtol=0, atol=5e-14)
    np.testing.assert_allclose(out["J"], R.batch_jacobian(mo, jo, q, mo.links, True, True), rtol=1e-11, atol=1e-11)
    for scratch_ref, mode in ((True, R.SCRATCH_REFERENCE), (False, R.SCRATCH_CLEAN)):
        o2 = run_program(h, ti, tr, q, truncation=0.3, scratch_ref=scratch_ref)
        vals, grads, am = R.batch_collision(so, jo, sdf_o, q, 0.3, R.GRAD_FD, mode)
        np.testing.assert_allclose(o2["vals"], vals, rtol=1e-12, atol=1e-13)
        assert np.array_equal(o2["argmin"], am)
        np.testing.assert_allclose(o2["grads"], grads.transpose(0, 2, 1), rtol=0, atol=1e-7)


def test_codegen_and_nvrtc_compile_without_a_gpu(tmp_path):
    """The model-specialised kernel source (csrc/kin_codegen.cpp) is generated and compiled with NVRTC for sm_100a
    on the CPU box: Fetch FK of all links + gripper Jacobian, and the fused call with the 16-sphere fixture."""
    import ctypes as C
    import scene_fetch
    from kinematics_jl_b200 import lib as L
    from kinematics_jl_b200.device import make_desc
    lib = L.lib()
    if not lib.kin_jit_status().startswith(b"ok"):
        pytest.skip("NVRTC not available: " + lib.kin_jit_status().decode())
    m, joints, sscc = scene_fetch.product_fetch(False)
    poses, widths = scenes.fridge_boxes_host()
    d, keep = make_desc(m, [j.id for j in joints], spheres=(sscc._parents, sscc._centers, sscc.sphere_radii), boxes=(poses, widths))
    fk = np.arange(1, 26, dtype=np.int32)
    jac = np.array([K.find_link(m, "gripper_link").id], dtype=np.int32)
    ip = C.POINTER(C.c_int32)
    for fused in (False, True):
        c = L.KinCall()
        c.precision, c.layout, c.n, c.q = L.F64, L.SOA, 1 << 20, 1
        c.n_fk_links, c.fk_links, c.T_out = 25, fk.ctypes.data_as(ip), 1
        c.n_jac_links, c.jac_links, c.J_out, c.with_rot = 1, jac.ctypes.data_as(ip), 1, 1
        c.truncation_dist = float("inf")
        if fused:
            c.vals_out, c.grads_out = 1, 1
        out = tmp_path / ("fused" if fused else "fkj")
        out.mkdir()
        L.check(lib.kin_codegen_dump(C.byref(d), C.byref(c), 1, str(out).encode()))
        p1 = (out / "kin_gen_phase1.inc").read_text()
        # constants are folded: the 25-link FK of Fetch needs fewer than 400 arithmetic statements (the
        # interpreting kernel executes ~1800 per configuration), and all 300 + 48 outputs are stored
        n_arith = sum(p1.count(op) for op in ("fma_(", "mul_(", "add_(", "sub_("))
        assert 100 < n_arith < 400
        assert p1.count("KST_T(") == 300 and p1.count("KST_J(") == 48
        assert (out / "kin_gen.cubin").stat().st_size > 10000
        # the measured launch shapes of the headline kernels (profiles/sweep_jit.py) are what the library picks for Fetch: the
        # fit-driven search of gen_options (models with a large per-thread scratch) must leave them alone
        cfg0 = (out / "kin_gen_config.h").read_text()
        shape = tuple(int(re.search(r"#define %s (\d+)" % k, cfg0).group(1)) for k in ("KBS", "KMINB"))
        assert shape == ((128, 2) if fused else (128, 1)), shape
        if fused:
            p2 = (out / "kin_gen_phase2.inc").read_text()
            assert p2.count("phase2b_group<") == 4 and p2.count("phase2a_group<") == 1   # four relevance masks, one shared box search
            cfg = (out / "kin_gen_config.h").read_text()
            assert "#define KPRIMS 0" in cfg                          # a table of boxes compiles the box-only code
    # the same fused kernel with the sphere / cylinder row test compiled in (extension, KPRIMS = 1), every layout + the
    # one-warp-per-configuration variant: must compile for sm_100a
    os.environ["KIN_JIT_FORCE_PRIMS"] = "1"
    try:
        for layout, n in ((L.SOA, 1 << 20), (L.AOS, 1 << 20), (L.TILED32, 1 << 20), (L.SOA, 64)):
            c = L.KinCall()
            c.precision, c.layout, c.n, c.q = L.F64, layout, n, 1
            c.n_fk_links, c.fk_links, c.T_out = 25, fk.ctypes.data_as(ip), 1
            c.truncation_dist = float("inf")
            c.vals_out, c.grads_out = 1, 1
            out = tmp_path / ("prims_%d_%d" % (layout, n))
            out.mkdir()
            L.check(lib.kin_codegen_dump(C.byref(d), C.byref(c), 1, str(out).encode()))
            assert "#define KPRIMS 1" in (out / "kin_gen_config.h").read_text()
            assert (out / "kin_gen.cubin").stat().st_size > 10000
    finally:
        del os.environ["KIN_JIT_FORCE_PRIMS"]


@pytest.mark.parametrize("with_base", [False, True])
def test_dual_arm_program_and_default_specialised_kernel_compile(with_base, tmp_path):
    """15 / 18 configuration columns (tests/scenes_dual_arm.py): the compiled program against the oracle through the
    numpy interpreter, and the specialised kernel of the fused call -- joint frames in registers, one phase-2b instance
    per relevance mask, CTA shrunk until the scratch fits -- compiled with NVRTC for sm_100a, every layout."""
    import ctypes as C
    import scenes_dual_arm as DA
    import scenes_synthetic as SS
    from kinematics_jl_b200 import lib as L
    from kinematics_jl_b200.device import make_desc
    m, joints, sscc, sdf = DA.product(with_base)
    mo, jo, so, sdf_o = DA.oracle(with_base)
    q = SS.random_q(jo, 60, with_base, seed=3)
    ids = [l.id for l in m.links]
    spheres = (sscc._parents, sscc._centers, sscc.sphere_radii)
    boxes = (np.stack(DA.BOX_POSES), np.array(DA.BOX_WIDTHS))
    h, ti, tr = dump_program(m, [j.id for j in joints], ids, ids, spheres, boxes)
    assert h["n_dof"] == (18 if with_base else 15)
    out = run_program(h, ti, tr, q, with_rot=True, rpy_jac=True)
    np.testing.assert_allclose(out["T"], R.batch_fk(mo, jo, q, mo.links)[:, :, :3, :], rtol=0, atol=5e-14)
    np.testing.assert_allclose(out["J"], R.batch_jacobian(mo, jo, q, mo.links, True, True), rtol=1e-11, atol=1e-11)
    for scratch_ref, mode in ((True, R.SCRATCH_REFERENCE), (False, R.SCRATCH_CLEAN)):
        o2 = run_program(h, ti, tr, q, truncation=0.3, scratch_ref=scratch_ref)
        vals, grads, am = R.batch_collision(so, jo, sdf_o, q, 0.3, R.GRAD_FD, mode)
        np.testing.assert_allclose(o2["vals"], vals, rtol=1e-12, atol=1e-13)
        assert np.array_equal(o2["argmin"], am)
        np.testing.assert_allclose(o2["grads"], grads.transpose(0, 2, 1), rtol=0, atol=1e-7)
    lib = L.lib()
    if not lib.kin_jit_status().startswith(b"ok"):
        pytest.skip("NVRTC not available: " + lib.kin_jit_status().decode())
    d, keep = make_desc(m, [j.id for j in joints], spheres=spheres, boxes=boxes)
    fk = np.array(ids, dtype=np.int32)
    import re
    # launch shape: the most threads per SM whose shared scratch fits (kin_b200.cu: gen_options); 15 columns keep the
    # default 128 x 2 (FP64) / 256 x 2 (FP32), 18 columns get one CTA of 224 (FP64) / 480 (FP32) threads
    expect = {(L.SOA, L.F64): (128, 2) if not with_base else (224, 1), (L.AOS, L.F64): None,
              (L.TILED32, L.F32): (256, 2) if not with_base else (480, 1), (L.TILED32, L.F64): (256, 1) if not with_base else (224, 1)}
    for (layout, prec), shape in expect.items():
        c = L.KinCall()
        c.precision, c.layout, c.n, c.q = prec, layout, 1 << 20, 1
        c.n_fk_links, c.fk_links, c.T_out = len(fk), fk.ctypes.data_as(C.POINTER(C.c_int32)), 1
        c.truncation_dist = float("inf")
        c.vals_out, c.grads_out = 1, 1
        out_dir = tmp_path / ("l%d_p%d" % (layout, prec))
        out_dir.mkdir()
        L.check(lib.kin_codegen_dump(C.byref(d), C.byref(c), 1, str(out_dir).encode()))
        cfg = (out_dir / "kin_gen_config.h").read_text()
        phase2 = (out_dir / "kin_gen_phase2.inc").read_text()
        assert "const JFrame<real> jfr[KND] = {" in phase2
        assert phase2.count("phase2b_group<") == 13          # one instance per distinct relevance mask
        kbs = int(re.search(r"#define KBS (\d+)", cfg).group(1))
        minb = int(re.search(r"#define KMINB (\d+)", cfg).group(1))
        assert kbs % 32 == 0 and 32 <= kbs <= 512
        if shape is not None:
            assert (kbs, minb) == shape, (layout, prec, kbs, minb)
        assert (out_dir / "kin_gen.cubin").stat().st_size > 10000


def test_constant_and_duplicate_rows_claimed_by_the_generator_hold_in_the_oracle(tmp_path):
    """kin_eval_host does not move over PCIe the output rows the code generator declares constant (stored as a literal)
    or equal to another row (stored from the same variable, possibly negated).  Both claims are checked here, without a
    GPU, against the ORACLE's outputs on random configurations: a literal row must hold that value for every
    configuration, two rows of one variable must be equal (or opposite) for every configuration."""
    import ctypes as C
    import re
    import scene_fetch
    from kinematics_jl_b200 import lib as L
    from kinematics_jl_b200.device import make_desc
    lib = L.lib()
    if not lib.kin_jit_status().startswith(b"ok"):
        pytest.skip("NVRTC not available: " + lib.kin_jit_status().decode())
    m, joints, sscc = scene_fetch.product_fetch(False)
    d, keep = make_desc(m, [j.id for j in joints])
    fk = np.arange(1, 26, dtype=np.int32)
    jac = np.array([K.find_link(m, "gripper_link").id], dtype=np.int32)
    ip = C.POINTER(C.c_int32)
    c = L.KinCall()
    c.precision, c.layout, c.n, c.q = L.F64, L.SOA, 1 << 20, 1
    c.n_fk_links, c.fk_links, c.T_out = 25, fk.ctypes.data_as(ip), 1
    c.n_jac_links, c.jac_links, c.J_out, c.with_rot = 1, jac.ctypes.data_as(ip), 1, 1
    c.truncation_dist = float("inf")
    L.check(lib.kin_codegen_dump(C.byref(d), C.byref(c), 0, str(tmp_path).encode()))
    src = (tmp_path / "kin_gen_phase1.inc").read_text()
    stores = re.findall(r"KST_([TJ])\((\d+), ([^;]*)\);", src)
    assert len(stores) == 348
    mo, jo, _ = scenes.oracle_fetch(False)
    q = scenes.random_configs(jo, 64, False, seed=5)
    T = R.batch_fk(mo, jo, q, mo.links[:25])[:, :, :3, :]                         # (N, 25, 3, 4)
    T = T.transpose(0, 1, 3, 2).reshape(len(q), 300)                               # 3x4 column-major per link
    J = R.batch_jacobian(mo, jo, q, [R.find_link(mo, "gripper_link")], True)[:, 0]  # (N, 6, 8)
    J = J.transpose(0, 2, 1).reshape(len(q), 48)                                   # column-major
    out = {"T": T, "J": J}
    first, n_const, n_dup = {}, 0, 0
    for arr, k, expr in stores:
        k, expr = int(k), expr.strip()
        col = out[arr][:, k]
        mlit = re.fullmatch(r"real\((-?[0-9a-fx.p+-]+)\)", expr)
        if mlit:
            n_const += 1
            np.testing.assert_allclose(col, float.fromhex(mlit.group(1)) if "x" in mlit.group(1) else float(mlit.group(1)),
                                       rtol=0, atol=1e-15, err_msg="%s row %d is not the constant %s" % (arr, k, expr))
            continue
        neg = expr.startswith("(-")
        canon = expr[2:-1] if neg else expr
        if canon in first:
            n_dup += 1
            np.testing.assert_allclose(col, -first[canon] if neg else first[canon], rtol=0, atol=1e-15,
                                       err_msg="%s row %d is not %s" % (arr, k, expr))
        elif not neg:
            first[canon] = col
    assert n_const == 175 and n_dup == 67          # the counts DESIGN.md / bench.py quote for Fetch with the 8 arm joints

"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C ABI of
libkin_b200.so (ctypes, via the host mirror), against the CPU oracle on the same seeded inputs.

Tolerances (SURVEY 8c): FP64 transforms / Jacobians / distances 1e-12 relative (1e-12 absolute near
zero); collision gradient 1e-12 vs the analytic oracle in analytic mode and 1e-7 absolute vs the
forward-difference oracle in FD mode (the reference's FD with eps 1e-7 amplifies 1-ulp differences of
sin/cos by 1e7); argmin box, truncation pattern and all index orders exact; FP32 mode 1e-5."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import device_model
from oracle import ref_model as R
from conftest import DATA, GOLDEN
import scenes

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-12, 1e-12


def dev(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")


def host(t):
    return t.double().cpu().numpy()


def soa(t):
    """(N, n_dof) tensor whose memory is (n_dof, N): consumed as KIN_LAYOUT_SOA."""
    return t.t().contiguous().t()


# ------------------------------------------------------------------------------------------------
# FK: data/ground_truth.json through the kernel (test_kinematics.jl:2-39)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_base", [False, True])
def test_fk_ground_truth_through_kernel(with_base):
    g = json.load(open(os.path.join(DATA, "ground_truth.json")))
    m = K.parse_urdf(os.path.join(GOLDEN, "pr2_right_arm_mini.urdf"), with_base=with_base)
    joints = [K.find_joint(m, n) for n in g["joint_names"]]
    links = [K.find_link(m, n) for n in g["link_names"]]
    angles = list(g["angle_vector"]) + ([0.3, 0.3, 0.3] if with_base else [])
    K.set_joint_angles(m, joints, angles)
    for _ in range(2):
        for link, pose in zip(links, g["pose_list"]):
            tf = K.get_transform(m, link)
            ypr = K.rpy(tf)[::-1]
            if with_base:
                from kinematics_jl_b200.transform import rotz
                np.testing.assert_allclose(K.translation(tf), rotz(0.3) @ pose[:3] + [0.3, 0.3, 0.0], rtol=0, atol=1e-13)
                np.testing.assert_allclose(ypr, np.array(pose[3:]) + [0.3, 0, 0], rtol=0, atol=1e-13)
            else:
                np.testing.assert_allclose(K.translation(tf), pose[:3], rtol=0, atol=1e-13)
                np.testing.assert_allclose(ypr, pose[3:], rtol=0, atol=1e-13)


# ------------------------------------------------------------------------------------------------
# FK + Jacobians, every Fetch link, random in-limit configurations, both layouts
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_base", [False, True])
@pytest.mark.parametrize("layout", ["aos", "soa"])
def test_fk_and_jacobian_all_links(with_base, layout):
    m, joints, _ = scenes.product_fetch(with_base)
    mo, jo, _ = scenes.oracle_fetch(with_base)
    q = scenes.random_configs(jo, 1000, with_base, seed=11, zeros_every=50)   # ragged: not a multiple of the CTA
    Q = dev(q)
    K.set_joint_angles(m, joints, soa(Q) if layout == "soa" else Q)
    T = host(K.get_transform(m, m.links))
    np.testing.assert_allclose(T, R.batch_fk(mo, jo, q, mo.links)[:, :, :3, :], rtol=RTOL, atol=ATOL)
    for with_rot, rpy_jac in ((True, False), (True, True), (False, False)):
        J = host(K.get_jacobian(m, m.links, joints, with_rot, rpy_jac=rpy_jac))
        Jr = R.batch_jacobian(mo, jo, q, mo.links, with_rot, rpy_jac)
        np.testing.assert_allclose(J, Jr, rtol=RTOL, atol=ATOL)


def test_fk_single_link_and_empty_batch():
    m, joints, _ = scenes.product_fetch(False)
    mo, jo, _ = scenes.oracle_fetch(False)
    q = scenes.random_configs(jo, 37, False, seed=5)
    K.set_joint_angles(m, joints, dev(q))
    g = K.find_link(m, "gripper_link")
    T = host(K.get_transform(m, g))
    assert T.shape == (37, 3, 4)
    np.testing.assert_allclose(T, R.batch_fk(mo, jo, q, [R.find_link(mo, "gripper_link")])[:, 0, :3, :], rtol=RTOL, atol=ATOL)
    K.set_joint_angles(m, joints, torch.zeros((0, 8), dtype=torch.float64, device="cuda"))
    assert K.get_transform(m, g).shape == (0, 3, 4)


def test_single_configuration_api_matches_reference_style():
    """The reference's own call pattern (test_kinematics.jl:45-72) on one configuration: Jacobian vs
    forward differences of get_transform, at the test angles and at zeros."""
    m, joints, _ = scenes.product_fetch(True)
    angles1 = np.array([0.2, 0.564, 0.35, -0.74, -0.7, -0.7, -0.17, -0.63, 0.3, 0.3, 0.3])
    eps = 1e-7
    for angles in (angles1, angles1 * 0):
        for link in [K.find_link(m, n) for n in ("gripper_link", "head_tilt_link", "elbow_flex_link", "base_link")]:
            K.set_joint_angles(m, joints, angles)
            Ja = K.get_jacobian(m, link, joints, True, rpy_jac=True)
            p0 = K.get_transform(m, link)
            Jn = np.zeros((6, 11))
            for i in range(11):
                a = angles.copy()
                a[i] += eps
                K.set_joint_angles(m, joints, a)
                p1 = K.get_transform(m, link)
                Jn[:3, i] = (K.translation(p1) - K.translation(p0)) / eps
                Jn[3:, i] = (K.rpy(p1) - K.rpy(p0)) / eps
            np.testing.assert_allclose(Jn[:3], Ja[:3], rtol=0, atol=1e-5)
            np.testing.assert_allclose(Jn[3:], Ja[3:], rtol=0, atol=1e-5)


def test_get_jacobian_inplace_keeps_irrelevant_columns():
    """get_jacobian! (algorithm.jl:91-96) writes only relevant columns."""
    m, joints, _ = scenes.product_fetch(False)
    mo, jo, _ = scenes.oracle_fetch(False)
    q = scenes.random_configs(jo, 8, False, seed=6)
    K.set_joint_angles(m, joints, dev(q))
    link = K.find_link(m, "head_pan_link")      # moved by the torso only
    store = torch.full((8, 8, 6), 7.0, dtype=torch.float64, device="cuda")   # AoS block (N, cols, rows)
    K.get_jacobian_(m, link, joints, True, store.permute(0, 2, 1))
    J = host(store.permute(0, 2, 1))
    for n in range(8):
        mat = np.full((6, 8), 7.0, order="F")
        R.set_joint_angles(mo, jo, q[n])
        R.get_jacobian_inplace(mo, R.find_link(mo, "head_pan_link"), jo, True, mat)
        np.testing.assert_allclose(J[n], mat, rtol=RTOL, atol=ATOL)
    assert np.all(J[:, :, 1:] == 7.0) and np.all(J[:, 3:, 0] == 7.0)   # prismatic: rows 4:6 untouched (:78-81)


def test_frozen_joints_and_subset_of_control_joints():
    m, joints, _ = scenes.product_fetch(False)
    mo, jo, _ = scenes.oracle_fetch(False)
    for name, a in {"head_pan_joint": 0.4, "head_tilt_joint": -0.3, "l_gripper_finger_joint": 0.02}.items():
        K.set_joint_angle(m, K.find_joint(m, name), a)
        R.set_joint_angles(mo, [R.find_joint(mo, name)], [a])
    K.set_joint_angle(m, joints[0], 0.2)
    R.set_joint_angles(mo, [jo[0]], [0.2])
    ctrl, ctrl_o = joints[1:6], jo[1:6]
    q = scenes.random_configs(ctrl_o, 64, False, seed=7)
    K.set_joint_angles(m, ctrl, dev(q))
    T = host(K.get_transform(m, m.links))
    np.testing.assert_allclose(T, R.batch_fk(mo, ctrl_o, q, mo.links)[:, :, :3, :], rtol=RTOL, atol=ATOL)


# ------------------------------------------------------------------------------------------------
# SDF at points (test_sdf.jl)
# ------------------------------------------------------------------------------------------------
def test_boxsdf_and_unionsdf_kats():
    from kinematics_jl_b200.transform import rotz
    pose = K.Transform(np.array([0.5, 0.5, 0.5]), rotz(0.3))
    box = K.BoxSDF(pose, [1, 1, 1])
    assert box(pose * [0.5, 0.5, 0.5]) == pytest.approx(0.0, abs=1e-12)      # test_sdf.jl:20-22
    assert box(pose * [0.0, 0.0, 0.0]) == pytest.approx(-0.5)
    assert box(pose * [0.0, 0.0, 1.0]) == pytest.approx(0.5)
    p1, p2 = K.Transform(np.array([0.5, 0.5, 0.0])), K.Transform(np.array([-0.5, -0.5, 0.0]))
    u = K.UnionSDF([K.BoxSDF(p1, [1, 1, 1]), K.BoxSDF(p2, [1, 1, 1])])
    assert u(p1 * [0.5, 0.5, 0.5]) == pytest.approx(0.0, abs=1e-12)           # test_sdf.jl:32-35
    assert u(p2 * [-0.5, -0.5, -0.5]) == pytest.approx(0.0, abs=1e-12)
    assert u(p1 * [0.5, 0.5, 1.5]) == pytest.approx(1.0)
    assert u(p1 * [-0.5, -0.5, -1.5]) == pytest.approx(1.0)
    assert u(np.array([0.0, 0.0, 2.0]), return_argmin=True)[1] == 1           # first minimum (sdf.jl:112)


def test_fridge_union_points_vs_oracle():
    fridge = K.parse_urdf(os.path.join(DATA, "fridge.urdf"), with_base=True)
    K.set_joint_angles(fridge, [K.find_joint(fridge, "door_joint")], scenes.FRIDGE_STATE)
    sdf = K.UnionSDF(fridge)
    so = scenes.oracle_fridge_sdf()
    poses, widths = sdf.world_boxes()
    assert len(poses) == 7
    np.testing.assert_allclose(poses, np.stack(so.poses), rtol=0, atol=1e-15)
    rng = np.random.default_rng(0)
    pts = np.array([1.2, 0, 0.75]) + (rng.random((5000, 3)) - 0.5) * 2.25       # the cloud of test_sdf.jl:43-45, shifted with the base
    vals, am = sdf(dev(pts), return_argmin=True)
    g_fd = sdf.gradient(dev(pts))
    g_an = sdf.gradient(dev(pts), grad_mode=K.GRAD_ANALYTIC)
    v_ref = np.array([so(p) for p in pts])
    am_ref = np.zeros(len(pts), dtype=np.int32)
    gf_ref, ga_ref = np.zeros_like(pts), np.zeros_like(pts)
    for i, p in enumerate(pts):
        so(p)
        am_ref[i] = so.argmin
        gf_ref[i], ga_ref[i] = so.gradient(p), so.gradient(p, analytic=True)
    np.testing.assert_allclose(host(vals), v_ref, rtol=RTOL, atol=1e-14)
    assert np.array_equal(am.cpu().numpy(), am_ref)
    np.testing.assert_allclose(host(g_an), ga_ref, rtol=RTOL, atol=1e-14)
    np.testing.assert_allclose(host(g_fd), gf_ref, rtol=0, atol=1e-7)


def _select_kernel(monkeypatch, specialised):
    """Run the following kin_eval calls on the model-specialised kernel (whatever the batch size) or on the
    interpreting kernel."""
    monkeypatch.delenv("KIN_DISABLE_JIT", raising=False)
    monkeypatch.delenv("KIN_FORCE_JIT", raising=False)
    monkeypatch.setenv("KIN_FORCE_JIT" if specialised else "KIN_DISABLE_JIT", "1")


@pytest.mark.parametrize("with_base", [False, True])
@pytest.mark.parametrize("layout", [L.SOA, L.TILED32])
@pytest.mark.parametrize("n", [1, 300, 70001])
def test_fused_kernels_are_bitwise_identical(layout, n, with_base, monkeypatch):
    """The fused call (FK of 25 links + two rpy Jacobians + collision) in FP64 SoA / tiled: the interpreting kernel
    and the model-specialised kernel run the same arithmetic in the same order, so every output must be bitwise
    identical (up to the sign of a zero) -- for ragged batches, with and without truncation, in both scratch modes
    and all gradient modes."""
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(with_base)
    q = scenes.random_configs(jo, n, with_base, seed=17, zeros_every=97)
    from kinematics_jl_b200.device import current_q, evaluate
    K.set_joint_angles(m, joints, dev(q))
    K.compute_coll_dists(sscc, joints, sdf)                         # uploads sphere / box tables
    dm = device_model(m)
    Q, ql, N = current_q(m)
    assert N == n and dm.n_dof == (11 if with_base else 8)
    fk = [l.id for l in m.links[:25]]
    jac = [K.find_link(m, "gripper_link").id, K.find_link(m, "wrist_flex_link").id]

    def run(**kw):
        out = evaluate(dm, Q, ql, N, layout=layout, fk_links=fk, jac_links=jac, with_rot=True, rpy_jac=True,
                       collision=True, want_argmin=True, launch_info=True, **kw)
        torch.cuda.synchronize()
        return {k: out[k].contiguous().clone() for k in ("T", "J", "vals", "grads", "argmin")}, out["launch"]["block"]

    cases = [dict(truncation_dist=np.inf, grad_mode=K.GRAD_FD, scratch_mode=K.SCRATCH_REFERENCE),
             dict(truncation_dist=0.08, grad_mode=K.GRAD_FD_DIRECT, scratch_mode=K.SCRATCH_REFERENCE, vals_offset=0.03),
             dict(truncation_dist=0.3, grad_mode=K.GRAD_ANALYTIC, scratch_mode=K.SCRATCH_CLEAN)]
    for kw in cases:
        _select_kernel(monkeypatch, specialised=False)
        n0 = L.lib().kin_launch_count()
        classic, block = run(**kw)
        assert L.lib().kin_launch_count() == n0 + 1 and block in (32, 64, 96, 128)
        _select_kernel(monkeypatch, specialised=True)
        spec, block = run(**kw)
        assert block < 0, L.lib().kin_jit_status()
        for k in classic:
            assert torch.equal(spec[k], classic[k]), (k, kw)
    # and against the oracle once
    v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q[:2000], np.inf, R.GRAD_FD, R.SCRATCH_REFERENCE)
    _select_kernel(monkeypatch, specialised=False)
    classic, block = run(**cases[0])
    assert block > 0
    np.testing.assert_allclose(host(classic["vals"])[:2000], v_ref, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(host(classic["grads"])[:2000], g_ref.transpose(0, 2, 1), rtol=0, atol=1e-7)


def test_fused_kernel_argument_combinations_and_streams(monkeypatch):
    """The fused call with outputs switched off one by one (collision only, distances only, no argmin,
    translation-only geometric Jacobian): the model-specialised kernel bitwise against the interpreting kernel; then,
    on the default kernel, launches in flight on two streams at once against the serial result."""
    from kinematics_jl_b200.device import current_q, evaluate
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    n = 40000
    q = scenes.random_configs(jo, n, False, seed=23)
    K.set_joint_angles(m, joints, dev(q))
    K.compute_coll_dists(sscc, joints, sdf)
    dm = device_model(m)
    Q, ql, N = current_q(m)
    fk = [K.find_link(m, "gripper_link").id, K.find_link(m, "head_camera_link").id]
    jac = [K.find_link(m, "elbow_flex_link").id]
    combos = [dict(collision=True),                                                        # collision only
              dict(collision=True, grad_mode=K.GRAD_ANALYTIC, scratch_mode=K.SCRATCH_CLEAN, want_argmin=True),
              dict(collision=True, truncation_dist=0.05, vals_offset=0.02),                # collision only, truncated
              dict(collision=True, with_grads=False, want_argmin=True),                    # distances + argmin
              dict(collision=True, fk_links=fk),                                           # no Jacobian
              dict(collision=True, jac_links=jac, with_rot=False),                         # 3 x n_dof Jacobian
              dict(collision=True, fk_links=fk, jac_links=jac, with_rot=True, rpy_jac=False, truncation_dist=0.1)]

    def run(kw, stream=None):
        out = evaluate(dm, Q, ql, N, layout=L.SOA, launch_info=True, stream=stream, **kw)
        return out

    for kw in combos:
        _select_kernel(monkeypatch, specialised=True)
        spec = run(kw)
        assert spec["launch"]["block"] < 0, L.lib().kin_jit_status()
        _select_kernel(monkeypatch, specialised=False)
        classic = run(kw)
        assert classic["launch"]["block"] > 0
        torch.cuda.synchronize()
        for k in spec:
            if k != "launch":
                assert torch.equal(spec[k].contiguous(), classic[k].contiguous()), (k, kw)
    # concurrent launches on two streams
    monkeypatch.delenv("KIN_DISABLE_JIT", raising=False)
    kw = combos[-1]
    serial = run(kw)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    outs = []
    for rep in range(4):
        for st in (s1, s2):
            with torch.cuda.stream(st):
                outs.append(run(kw, stream=st.cuda_stream))
    torch.cuda.synchronize()
    for o in outs:
        for k in ("T", "J", "vals", "grads"):
            assert torch.equal(o[k].contiguous(), serial[k].contiguous()), k


@pytest.mark.parametrize("with_base", [False, True])
def test_fused_kernel_on_a_second_model_vs_oracle(with_base, monkeypatch):
    """A different chain (the PR2 right arm of data/ground_truth.json: fixed joints between the controlled ones, so
    attachments carry non-trivial constant transforms), 10 spheres on 3 links in an order that is NOT the chain
    order, a union of 3 rotated boxes: the interpreting kernel against the oracle and bitwise against the
    model-specialised kernel."""
    from kinematics_jl_b200.device import current_q, evaluate
    from kinematics_jl_b200.transform import rotz
    g = json.load(open(os.path.join(DATA, "ground_truth.json")))
    path = os.path.join(GOLDEN, "pr2_right_arm_mini.urdf")
    m, mo = K.parse_urdf(path, with_base=with_base), R.parse_urdf(path, with_base=with_base)
    joints = [K.find_joint(m, n) for n in g["joint_names"]]
    jo = [R.find_joint(mo, n) for n in g["joint_names"]]
    sscc, so = K.SweptSphereCollisionChecker(m), R.SweptSphereCollisionChecker(mo)
    rng = np.random.default_rng(4)
    for name, k, rad in (("r_wrist_roll_link", 4, 0.05), ("r_shoulder_lift_link", 3, 0.09), ("r_forearm_link", 3, 0.06)):
        cents = [list(np.array([0.08 * i, 0.0, 0.0]) + rng.normal(0, 0.01, 3)) for i in range(k)]
        K.add_coll_links(sscc, K.find_link(m, name), cents, rad)
        R.add_coll_links(so, R.find_link(mo, name), cents, [rad] * k)
    poses, widths = [], []
    for c, yaw, w in (([0.7, -0.3, 0.9], 0.4, [0.3, 0.2, 0.5]), ([0.4, -0.9, 0.6], -0.8, [0.2, 0.6, 0.2]), ([0.9, 0.2, 1.3], 1.1, [0.4, 0.4, 0.1])):
        poses.append(K.Transform(np.array(c), rotz(yaw)))
        widths.append(w)
    sdf = K.UnionSDF([K.BoxSDF(p, w) for p, w in zip(poses, widths)])
    sdf_o = R.RefSDF([p.mat for p in poses], widths)
    n = 20000
    q = scenes.random_configs(jo, n, with_base, seed=9, zeros_every=211)
    K.set_joint_angles(m, joints, dev(q))
    K.compute_coll_dists(sscc, joints, sdf)
    dm = device_model(m)
    Q, ql, N = current_q(m)
    kw = dict(layout=L.SOA, fk_links=[l.id for l in m.links[:11]], jac_links=[K.find_link(m, "r_wrist_roll_link").id],
              with_rot=True, rpy_jac=True, collision=True, want_argmin=True, truncation_dist=0.4, launch_info=True)
    _select_kernel(monkeypatch, specialised=True)
    spec = evaluate(dm, Q, ql, N, **kw)
    assert spec["launch"]["block"] < 0, L.lib().kin_jit_status()
    _select_kernel(monkeypatch, specialised=False)
    classic = evaluate(dm, Q, ql, N, **kw)
    assert classic["launch"]["block"] > 0
    for k in ("T", "J", "vals", "grads", "argmin"):
        assert torch.equal(spec[k].contiguous(), classic[k].contiguous()), k
    v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q, 0.4, R.GRAD_FD, R.SCRATCH_REFERENCE)
    np.testing.assert_allclose(host(classic["vals"]), v_ref, rtol=RTOL, atol=ATOL)
    assert np.array_equal(classic["argmin"].cpu().numpy(), am_ref)
    np.testing.assert_allclose(host(classic["grads"]), g_ref.transpose(0, 2, 1), rtol=0, atol=1e-7)
    T_ref = R.batch_fk(mo, jo, q, mo.links[:11])[:, :, :3, :]
    np.testing.assert_allclose(host(classic["T"]), T_ref, rtol=RTOL, atol=ATOL)


def test_fd_series_matches_direct_fd_near_every_kink():
    """KIN_GRAD_FD evaluates the FD quotient of sdf.jl:34-41 from its closed form away from kinks and
    directly near them; KIN_GRAD_FD_DIRECT always perturbs the point as the reference does.  The two (and
    the oracle) must agree to the FD's own rounding noise everywhere, in particular for points placed a few
    eps from each kind of kink: faces (q_k = 0), the mid-planes (l_k = 0), edges/corners, the surface seen
    from outside, and the medial surfaces inside the box."""
    from kinematics_jl_b200.transform import rotz, rotation, translation
    cy, sy = np.cos(-0.5), np.sin(-0.5)
    pose = K.Transform(np.array([0.4, -0.2, 0.7]), rotz(0.3) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]]))
    half = np.array([0.3, 0.2, 0.5])
    box = K.BoxSDF(pose, 2 * half)
    rng = np.random.default_rng(5)
    eps = 1e-7
    offs = np.array([0.0, 0.3, 0.9, 1.1, 1.9, 2.1, 3.9, 4.1, 30.0, 1e4, 2e4]) * eps
    offs = np.concatenate([offs, -offs])
    local = [(rng.random((20000, 3)) - 0.5) * 2.4]                      # bulk: inside and outside
    for k in range(3):
        for o in offs:
            base = (rng.random((40, 3)) - 0.5) * 2.0 * half * 1.6
            a = base.copy(); a[:, k] = half[k] + o; local.append(a)      # near a face plane (inside the face or beyond its edges)
            a = base.copy(); a[:, k] = -half[k] - o; local.append(a)
            a = base.copy(); a[:, k] = o; local.append(a)                # near a mid-plane: sign(l_k) flips
            a = base.copy(); a[:, k] = half[k] + o; a[:, (k + 1) % 3] = half[(k + 1) % 3] + rng.choice(offs, 40)
            local.append(a)                                              # near an edge
    # inside, near the medial surfaces q_j == q_k
    m = (rng.random((400, 3)) - 0.5) * 2 * half
    for o in offs[:8]:
        a = m.copy(); a[:, 0] = half[0] - (half[1] - np.abs(a[:, 1])) + o; local.append(a)
    local = np.concatenate(local)
    pts = local @ rotation(pose).T + translation(pose)
    g_fd = host(box.gradient(dev(pts)))
    g_dir = host(box.gradient(dev(pts), grad_mode=K.GRAD_FD_DIRECT))
    so = R.BoxSDF(pose.mat, 2 * half)
    g_ref = np.zeros_like(pts)
    for i, p in enumerate(pts):
        so(p)                                   # the reference differences against the cached value (sdf.jl:116-119)
        g_ref[i] = so.gradient(p)
    # the direct path restates the reference's arithmetic: rounding-level agreement with the oracle
    np.testing.assert_allclose(g_dir, g_ref, rtol=0, atol=5e-8)
    # the series path agrees with both to the FD's rounding noise (~ulp(f)/eps)
    np.testing.assert_allclose(g_fd, g_dir, rtol=0, atol=5e-8)
    np.testing.assert_allclose(g_fd, g_ref, rtol=0, atol=5e-8)
    far = np.abs(g_fd - g_dir).max()
    assert far < 5e-8, far


def test_fd_series_matches_direct_fd_on_a_large_fused_batch():
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(True)
    K.set_joint_angles(m, joints, dev(scenes.random_configs(jo, 1 << 20, True, seed=11)))
    out = {}
    for mode in (K.GRAD_FD, K.GRAD_FD_DIRECT):
        v, g = K.compute_coll_dists_and_grads(sscc, joints, sdf, truncation_dist=0.25, grad_mode=mode)
        out[mode] = (host(v), host(g))
    assert np.array_equal(out[K.GRAD_FD][0], out[K.GRAD_FD_DIRECT][0])            # distances do not depend on the mode
    diff = np.abs(out[K.GRAD_FD][1] - out[K.GRAD_FD_DIRECT][1])
    assert diff.max() < 1e-7, diff.max()


# ------------------------------------------------------------------------------------------------
# collision (test_collision.jl + the 16-sphere / fridge scene)
# ------------------------------------------------------------------------------------------------
ANGLES_SOLVED = [0.026928521116837873, 0.2378996102914415, 0.6445784881862138, -0.24833437463054583,
                 -1.035118222590030, -0.170439396116480, -1.3891477169766988, -0.07058932825801573]


@pytest.mark.parametrize("with_base", [False, True])
def test_collision_reference_test_case(with_base):
    """test_collision.jl:1-47 on the product: grads vs forward differences of the distances."""
    m, joints, sscc = scenes.product_fetch(with_base, sphere_links=["wrist_flex_link"])
    box = K.BoxSDF(K.Transform(np.array([1.0, 0.0, 0.8])), [0.3, 0.3, 0.3])
    angles = np.array(ANGLES_SOLVED + ([0.0, 0, 0] if with_base else []))
    K.set_joint_angles(m, joints, angles)
    _, grads = K.compute_coll_dists_and_grads(sscc, joints, box)
    d0 = K.compute_coll_dists(sscc, joints, box)
    eps = 1e-7
    for i in range(len(joints)):
        av = angles.copy()
        av[i] += eps
        K.set_joint_angles(m, joints, av)
        d1 = K.compute_coll_dists(sscc, joints, box)
        np.testing.assert_allclose(grads[i, :], (d1 - d0) / eps, rtol=0, atol=1e-5)
    K.set_joint_angles(m, joints, angles)
    assert np.array_equal(K.compute_coll_dists(sscc, joints, box), K.compute_coll_dists_and_grads(sscc, joints, box)[0])


def _fridge_scene(with_base):
    m, joints, sscc = scenes.product_fetch(with_base)
    mo, jo, so = scenes.oracle_fetch(with_base)
    fridge = K.parse_urdf(os.path.join(DATA, "fridge.urdf"), with_base=True)
    K.set_joint_angles(fridge, [K.find_joint(fridge, "door_joint")], scenes.FRIDGE_STATE)
    return m, joints, sscc, K.UnionSDF(fridge), mo, jo, so, scenes.oracle_fridge_sdf()


@pytest.mark.parametrize("with_base", [False, True])
@pytest.mark.parametrize("layout", ["aos", "soa"])
@pytest.mark.parametrize("truncation", [np.inf, 0.08])
def test_collision_fridge_vs_oracle(with_base, layout, truncation):
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(with_base)
    q = scenes.random_configs(jo, 777, with_base, seed=21, zeros_every=100)
    Q = dev(q)
    K.set_joint_angles(m, joints, soa(Q) if layout == "soa" else Q)
    d_only, am0 = K.compute_coll_dists(sscc, joints, sdf, return_argmin=True)
    v_ref0, _, am_ref = R.batch_collision(so, jo, sdf_o, q, with_grads=False)
    np.testing.assert_allclose(host(d_only), v_ref0, rtol=RTOL, atol=ATOL)
    assert np.array_equal(am0.cpu().numpy(), am_ref)
    for scratch, scratch_o in ((K.SCRATCH_REFERENCE, R.SCRATCH_REFERENCE), (K.SCRATCH_CLEAN, R.SCRATCH_CLEAN)):
        for gm, gm_o, tol in ((K.GRAD_FD, R.GRAD_FD, 1e-7), (K.GRAD_ANALYTIC, R.GRAD_ANALYTIC, 1e-12)):
            vals, grads, am = K.compute_coll_dists_and_grads(sscc, joints, sdf, truncation_dist=truncation, grad_mode=gm,
                                                             scratch_mode=scratch, return_argmin=True)
            v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q, truncation, gm_o, scratch_o)
            np.testing.assert_allclose(host(vals), v_ref, rtol=RTOL, atol=ATOL)
            assert np.array_equal(am.cpu().numpy(), am_ref)
            assert np.array_equal(host(vals) == truncation, v_ref == truncation)          # truncation pattern exact
            np.testing.assert_allclose(host(grads), g_ref.transpose(0, 2, 1), rtol=tol if tol < 1e-9 else 0, atol=tol)


def test_stale_scratch_differs_from_clean_as_in_the_reference():
    m, joints, sscc, sdf, *_ = _fridge_scene(False)
    K.set_joint_angles(m, joints, np.array(ANGLES_SOLVED))
    _, g_ref = K.compute_coll_dists_and_grads(sscc, joints, sdf, scratch_mode=K.SCRATCH_REFERENCE)
    _, g_clean = K.compute_coll_dists_and_grads(sscc, joints, sdf, scratch_mode=K.SCRATCH_CLEAN)
    assert np.array_equal(g_ref[:, :4], g_clean[:, :4])
    assert np.all(g_clean[1:, 4:8] == 0.0) and np.any(g_ref[1:7, 4:8] != 0.0)


# ------------------------------------------------------------------------------------------------
# model-specialised (NVRTC) kernels: bit-identical to the interpreting kernels, and checked against the oracle
# ------------------------------------------------------------------------------------------------
def _eval_all(m, joints, sscc, sdf, Q, layout, jit, monkeypatch, warp_max=None, **kw):
    from kinematics_jl_b200.device import current_q, evaluate
    monkeypatch.delenv("KIN_DISABLE_JIT", raising=False)
    monkeypatch.delenv("KIN_FORCE_JIT", raising=False)
    monkeypatch.delenv("KIN_JIT_WARP_MAX", raising=False)
    monkeypatch.setenv("KIN_FORCE_JIT" if jit else "KIN_DISABLE_JIT", "1")
    if warp_max is not None:                  # batches up to this size: the one-warp-per-configuration kernel
        monkeypatch.setenv("KIN_JIT_WARP_MAX", str(warp_max))
    K.set_joint_angles(m, joints, Q)
    if sscc is not None:
        K.compute_coll_dists(sscc, joints, sdf)
    dm = device_model(m)
    Qc, ql, N = current_q(m)
    gl = K.find_link(m, "gripper_link").id
    out = evaluate(dm, Qc, ql, N, layout=layout, fk_links=list(range(1, 26)), jac_links=[gl, K.find_link(m, "elbow_flex_link").id],
                   collision=sscc is not None, want_argmin=sscc is not None, launch_info=True, **kw)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("with_base", [False, True])
@pytest.mark.parametrize("layout", [L.SOA, L.TILED32, L.AOS])
@pytest.mark.parametrize("n", [1, 77, 40013])
def test_specialised_kernel_is_bitwise_identical(layout, n, with_base, monkeypatch):
    """The NVRTC-compiled, model-specialised kernel (straight-line phase 1 with the model's constants folded in,
    phase 2 instantiated per relevance mask) against the interpreting ahead-of-time kernel on the same inputs: every
    output equal bit for bit (== treats the two zeros as equal: the sign of a zero is the one thing folding changes)."""
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(with_base)
    q = scenes.random_configs(jo, n, with_base, seed=23, zeros_every=50)
    Q = dev(q)
    lib = L.lib()
    combos = [dict(with_rot=True, rpy_jac=False, truncation_dist=np.inf, grad_mode=L.GRAD_FD, scratch_mode=L.SCRATCH_REFERENCE),
              dict(with_rot=True, rpy_jac=True, truncation_dist=0.08, grad_mode=L.GRAD_FD, scratch_mode=L.SCRATCH_CLEAN, vals_offset=0.03),
              dict(with_rot=False, keep_irrelevant=False, truncation_dist=np.inf, grad_mode=L.GRAD_ANALYTIC, scratch_mode=L.SCRATCH_REFERENCE)]
    for kw in combos:
        a = _eval_all(m, joints, sscc, sdf, Q, layout, False, monkeypatch, **kw)
        assert a["launch"]["block"] > 0
        b = _eval_all(m, joints, sscc, sdf, Q, layout, True, monkeypatch, **kw)
        assert b["launch"]["block"] < 0, lib.kin_jit_status()          # negative block size = specialised kernel
        for key in ("T", "J", "vals", "grads", "argmin"):
            assert torch.equal(a[key], b[key]), (key, kw)
        if n <= 2048:     # ... and the one-warp-per-configuration variant (not the default at any size, KIN_JIT_WARP_MAX)
            w = _eval_all(m, joints, sscc, sdf, Q, layout, True, monkeypatch, warp_max=2048, **kw)
            assert w["launch"]["block"] < 0 and w["launch"]["grid"] == (n + 3) // 4      # 4 warps = 4 configurations per CTA
            for key in ("T", "J", "vals", "grads", "argmin"):
                assert torch.equal(a[key], w[key]), (key, kw)
    # FK / Jacobian only (no collision): the straight-line kernel without any shared memory
    a = _eval_all(m, joints, None, None, Q, layout, False, monkeypatch, with_rot=True, rpy_jac=True)
    b = _eval_all(m, joints, None, None, Q, layout, True, monkeypatch, with_rot=True, rpy_jac=True)
    assert b["launch"]["block"] < 0
    assert torch.equal(a["T"], b["T"]) and torch.equal(a["J"], b["J"])
    # and against the oracle (the specialised results)
    sub = slice(0, min(n, 300))
    np.testing.assert_allclose(host(b["T"][sub]), R.batch_fk(mo, jo, q[sub], mo.links[:25])[:, :, :3, :], rtol=RTOL, atol=ATOL)
    Jo = R.batch_jacobian(mo, jo, q[sub], [R.find_link(mo, "gripper_link"), R.find_link(mo, "elbow_flex_link")], True, rpy_jac=True)
    np.testing.assert_allclose(host(b["J"][sub]), Jo, rtol=1e-11, atol=1e-11)
    compiles, hits, launches, failures = (C.c_int64() for _ in range(4))
    lib.kin_jit_stats(C.byref(compiles), C.byref(hits), C.byref(launches), C.byref(failures))
    assert failures.value == 0 and launches.value > 0


@pytest.mark.parametrize("warp_max", [None, 2048])
def test_small_batches_switch_to_the_warp_per_configuration_kernel(warp_max, monkeypatch):
    """A solver callback evaluates one configuration (IK) or n_wp of them (planning) over and over: after a few small
    calls of the same program the library builds a specialised kernel for it (one thread per configuration -- the faster
    one at every size, profiles/sweep_midsize.py -- or, with KIN_JIT_WARP_MAX, one warp per configuration); results stay
    bit-identical across the switch and match the oracle."""
    monkeypatch.delenv("KIN_DISABLE_JIT", raising=False)
    monkeypatch.delenv("KIN_FORCE_JIT", raising=False)
    monkeypatch.delenv("KIN_JIT_WARP_MAX", raising=False)
    if warp_max is not None:
        monkeypatch.setenv("KIN_JIT_WARP_MAX", str(warp_max))
    from kinematics_jl_b200.device import current_q, evaluate
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    q = scenes.random_configs(jo, 10, False, seed=37)
    K.set_joint_angles(m, joints, dev(q))
    K.compute_coll_dists(sscc, joints, sdf)
    dm = device_model(m)
    Qc, ql, N = current_q(m)
    outs, blocks = [], []
    for _ in range(8):
        o = evaluate(dm, Qc, ql, N, fk_links=list(range(1, 26)), jac_links=[K.find_link(m, "gripper_link").id], collision=True,
                     want_argmin=True, launch_info=True)
        torch.cuda.synchronize()
        outs.append({k: o[k].clone() for k in ("T", "J", "vals", "grads", "argmin")})
        blocks.append(o["launch"]["block"])
    assert blocks[0] > 0 and blocks[-1] < 0, blocks                   # interpreting kernel first, specialised kernel later
    for o in outs[1:]:
        for k in o:
            assert torch.equal(o[k], outs[0][k]), k
    v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q)
    np.testing.assert_allclose(host(outs[-1]["vals"]), v_ref, rtol=RTOL, atol=ATOL)
    assert np.array_equal(outs[-1]["argmin"].cpu().numpy(), am_ref)
    np.testing.assert_allclose(host(outs[-1]["grads"]), g_ref.transpose(0, 2, 1), rtol=0, atol=1e-7)
    np.testing.assert_allclose(host(outs[-1]["T"]), R.batch_fk(mo, jo, q, mo.links[:25])[:, :, :3, :], rtol=RTOL, atol=ATOL)


def test_specialised_kernel_fp32_and_general_models(monkeypatch):
    """FP32 instantiation of the specialised kernel (same folding in float) and models that exercise the general
    paths of the generator: a branching tree with general axes / rpy origins / frozen joints, and the PR2 chain."""
    import scenes_synthetic
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    q = scenes.random_configs(jo, 3000, False, seed=29)
    a = _eval_all(m, joints, sscc, sdf, dev(q, torch.float32), L.SOA, False, monkeypatch, grad_mode=L.GRAD_ANALYTIC, scratch_mode=L.SCRATCH_CLEAN)
    b = _eval_all(m, joints, sscc, sdf, dev(q, torch.float32), L.SOA, True, monkeypatch, grad_mode=L.GRAD_ANALYTIC, scratch_mode=L.SCRATCH_CLEAN)
    assert b["launch"]["block"] < 0 and b["T"].dtype == torch.float32
    for key in ("T", "J", "vals", "grads", "argmin"):
        assert torch.equal(a[key], b[key]), key
    # synthetic branching mechanism (tests/scenes_synthetic.py: general axes, rpy origins, frozen joints, save slots,
    # spheres on three branches, rotated boxes), all links, both kernels and the oracle
    for with_base in (False, True):
        mp_, jp, sp_, sdfp = scenes_synthetic.product(with_base)
        mo_, jo_, so_, sdfo_ = scenes_synthetic.oracle(with_base)
        qs = scenes_synthetic.random_q(jo_, 500, with_base, seed=30)
        outs = []
        for jit in (False, True):
            monkeypatch.delenv("KIN_DISABLE_JIT", raising=False)
            monkeypatch.delenv("KIN_FORCE_JIT", raising=False)
            monkeypatch.setenv("KIN_FORCE_JIT" if jit else "KIN_DISABLE_JIT", "1")
            K.set_joint_angles(mp_, jp, soa(dev(qs)))
            T = K.get_transform(mp_, mp_.links)
            J = K.get_jacobian(mp_, mp_.links, jp, True, rpy_jac=True)
            v, g, am = K.compute_coll_dists_and_grads(sp_, jp, sdfp, return_argmin=True)
            outs.append([x.clone() for x in (T, J, v, g, am)])
        for x, y in zip(*outs):
            assert torch.equal(x, y)
        np.testing.assert_allclose(host(outs[1][0]), R.batch_fk(mo_, jo_, qs, mo_.links)[:, :, :3, :], rtol=RTOL, atol=ATOL)
        v_ref, g_ref, am_ref = R.batch_collision(so_, jo_, sdfo_, qs)
        np.testing.assert_allclose(host(outs[1][2]), v_ref, rtol=RTOL, atol=ATOL)
        assert np.array_equal(outs[1][4].cpu().numpy(), am_ref)
        np.testing.assert_allclose(host(outs[1][3]), g_ref.transpose(0, 2, 1), rtol=0, atol=1e-7)
    compiles, hits, launches, failures = (C.c_int64() for _ in range(4))
    L.lib().kin_jit_stats(C.byref(compiles), C.byref(hits), C.byref(launches), C.byref(failures))
    assert failures.value == 0


@pytest.mark.parametrize("with_base", [False, True])
@pytest.mark.parametrize("layout", [L.SOA, L.AOS, L.TILED32])
def test_specialised_kernel_on_a_dual_arm_model(layout, with_base, monkeypatch):
    """15 / 18 configuration columns (tests/scenes_dual_arm.py: the PR2 size class of fridge_demo.jl): the per-thread
    shared scratch no longer fits the default launch shape, the specialised kernel keeps the joint frames of phase 2 in
    registers and shrinks the CTA until the scratch fits.  Bit-identical to the interpreting kernel, and both against
    the oracle; FP64 and FP32."""
    import scenes_dual_arm as DA
    import scenes_synthetic as SS
    from kinematics_jl_b200.device import current_q, evaluate
    m, joints, sscc, sdf = DA.product(with_base)
    mo, jo, so, sdf_o = DA.oracle(with_base)
    n = 5003
    q = SS.random_q(jo, n, with_base, seed=41)
    ids = [l.id for l in m.links]
    tools = [K.find_link(m, "l_tool").id, K.find_link(m, "r_tool").id]
    combos = (dict(truncation_dist=np.inf, grad_mode=L.GRAD_FD, scratch_mode=L.SCRATCH_REFERENCE),
              dict(truncation_dist=0.3, grad_mode=L.GRAD_FD, scratch_mode=L.SCRATCH_CLEAN, vals_offset=0.02),
              dict(truncation_dist=np.inf, grad_mode=L.GRAD_ANALYTIC, scratch_mode=L.SCRATCH_CLEAN))
    for dtype in (torch.float64, torch.float32):
        for kw in (combos if dtype == torch.float64 else combos[2:]):      # (every kernel is a 1-3 s NVRTC compile on a fresh box)
            outs = []
            for jit in (False, True):
                monkeypatch.delenv("KIN_DISABLE_JIT", raising=False)
                monkeypatch.delenv("KIN_FORCE_JIT", raising=False)
                monkeypatch.setenv("KIN_FORCE_JIT" if jit else "KIN_DISABLE_JIT", "1")
                K.set_joint_angles(m, joints, dev(q, dtype))
                K.compute_coll_dists(sscc, joints, sdf)
                dm = device_model(m)
                Qc, ql, N = current_q(m)
                o = evaluate(dm, Qc, ql, N, layout=layout, fk_links=ids, jac_links=tools, with_rot=True, rpy_jac=True,
                             collision=True, want_argmin=True, launch_info=True, **kw)
                torch.cuda.synchronize()
                assert (o["launch"]["block"] < 0) == jit, (jit, o["launch"], L.lib().kin_jit_status())
                outs.append(o)
            for key in ("T", "J", "vals", "grads", "argmin"):
                assert torch.equal(outs[0][key], outs[1][key]), (key, kw, dtype)
        if dtype == torch.float64:        # the last combination (analytic gradient is an extension: FD combination re-run for the oracle)
            sub = slice(0, 400)
            b = outs[1]
            np.testing.assert_allclose(host(b["T"][sub]), R.batch_fk(mo, jo, q[sub], mo.links)[:, :, :3, :], rtol=RTOL, atol=ATOL)
            Jo = R.batch_jacobian(mo, jo, q[sub], [R.find_link(mo, "l_tool"), R.find_link(mo, "r_tool")], True, rpy_jac=True)
            np.testing.assert_allclose(host(b["J"][sub]), Jo, rtol=1e-11, atol=1e-11)
            K.set_joint_angles(m, joints, dev(q[sub], dtype))
            for scratch, scratch_o in ((K.SCRATCH_REFERENCE, R.SCRATCH_REFERENCE), (K.SCRATCH_CLEAN, R.SCRATCH_CLEAN)):
                Qc, ql, N = current_q(m)
                o = evaluate(device_model(m), Qc, ql, N, layout=layout, collision=True, want_argmin=True, truncation_dist=0.3,
                             scratch_mode=scratch, launch_info=True)
                assert o["launch"]["block"] < 0
                v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q[sub], 0.3, R.GRAD_FD, scratch_o)
                np.testing.assert_allclose(host(o["vals"]), v_ref, rtol=RTOL, atol=ATOL)
                assert np.array_equal(o["argmin"].cpu().numpy(), am_ref)
                np.testing.assert_allclose(host(o["grads"]), g_ref.transpose(0, 2, 1), rtol=0, atol=1e-7)
    compiles, hits, launches, failures = (C.c_int64() for _ in range(4))
    L.lib().kin_jit_stats(C.byref(compiles), C.byref(hits), C.byref(launches), C.byref(failures))
    assert failures.value == 0


# ------------------------------------------------------------------------------------------------
# FP32 mode (1e-5)
# ------------------------------------------------------------------------------------------------
def test_fp32_mode():
    """north_star: "within a stated 1e-5 in the optional FP32 mode".  Transforms, Jacobians and distances are held
    to 1e-5 absolute.  The collision gradient is g = n' J with n the unit normal of the argmin box; n has a
    condition number of 1 / d (d = centre-to-box distance), so FP32 rounding of the sphere centre (~1e-6 after the
    9-joint chain) moves it by ~1e-6 / d, and a different argmin box or active-face set flips it altogether.
    Stated bound, asserted below: the argmin box agrees with the FP64 oracle on >= 99.5 % of the spheres; where it
    agrees and the sphere is at least 0.1 m from the surface the gradient is within 1e-5; closer in, within
    1e-5 + 2e-6 / d (on >= 99.9 % -- the rest sit within float rounding of a face / edge switch of the same box)."""
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    q = scenes.random_configs(jo, 4096, False, seed=31)
    K.set_joint_angles(m, joints, dev(q, torch.float32))
    T = K.get_transform(m, m.links)
    assert T.dtype == torch.float32
    np.testing.assert_allclose(host(T), R.batch_fk(mo, jo, q, mo.links[:25] + mo.links[25:])[:, :, :3, :], rtol=0, atol=1e-5)
    J = K.get_jacobian(m, K.find_link(m, "gripper_link"), joints, True)
    np.testing.assert_allclose(host(J), R.batch_jacobian(mo, jo, q, [R.find_link(mo, "gripper_link")], True)[:, 0], rtol=0, atol=1e-5)
    vals, grads, am = K.compute_coll_dists_and_grads(sscc, joints, sdf, grad_mode=K.GRAD_ANALYTIC, scratch_mode=K.SCRATCH_CLEAN,
                                                     return_argmin=True)
    assert vals.dtype == torch.float32 and grads.dtype == torch.float32
    v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q, np.inf, R.GRAD_ANALYTIC, R.SCRATCH_CLEAN)
    np.testing.assert_allclose(host(vals), v_ref, rtol=0, atol=1e-5)
    same = am.cpu().numpy() == am_ref                                   # (N, S)
    print("fp32: argmin box agrees on %.3f %% of %d spheres" % (100 * same.mean(), same.size))
    assert same.mean() >= 0.995
    radii = np.array(so.sphere_radii)
    d = np.abs(v_ref + radii[None, :])                                  # |sdf(centre)|: distance of the centre to the surface
    err = np.abs(host(grads) - g_ref.transpose(0, 2, 1)).max(axis=1)    # (N, S): worst column per sphere
    far = same & (d >= 0.1)
    print("fp32 gradient: max err %.2e on %d far spheres; near spheres: %.4f %% within 1e-5 + 2e-6/d"
          % (err[far].max(), far.sum(), 100 * (err[same & ~far] <= 1e-5 + 2e-6 / np.maximum(d[same & ~far], 1e-6)).mean()))
    assert err[far].max() <= 1e-5
    near = same & ~far
    assert (err[near] <= 1e-5 + 2e-6 / np.maximum(d[near], 1e-6)).mean() >= 0.999


# ------------------------------------------------------------------------------------------------
# the fused call + the host-buffer entry point, straight through the C ABI
# ------------------------------------------------------------------------------------------------
def _fused_call(dm, n, qptr, layout, fk, jac, T, J, V, G, A):
    c = L.KinCall()
    c.precision, c.layout, c.n, c.q = L.F64, layout, n, qptr
    c.n_fk_links, c.fk_links, c.T_out = len(fk), fk.ctypes.data_as(C.POINTER(C.c_int32)), T
    c.n_jac_links, c.jac_links, c.J_out = len(jac), jac.ctypes.data_as(C.POINTER(C.c_int32)), J
    c.with_rot = 1
    c.truncation_dist = float("inf")
    c.vals_out, c.grads_out, c.argmin_out = V, G, A
    return c


def test_host_entry_point_tiled_layout_ragged_sizes():
    """kin_eval_host with KIN_LAYOUT_TILED32 and N % 32 != 0, below and above one staging chunk: the staging carves
    are sized for whole tiles (host buffers hold roundup(N, 32) records)."""
    from kinematics_jl_b200.device import tile32, untile32
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    fk = np.arange(1, 26, dtype=np.int32)
    jac = np.array([K.find_link(m, "gripper_link").id], dtype=np.int32)
    nl, S, nd = 25, 16, 8
    for N in (1, 33, 1000, 131072 + 77):
        q = scenes.random_configs(jo, N, False, seed=43)
        K.set_joint_angles(m, joints, dev(q[:1]))
        K.compute_coll_dists(sscc, joints, sdf)
        dm = device_model(m)
        NT = (N + 31) // 32
        qt = tile32(torch.as_tensor(q)).numpy()                          # (NT, nd, 32), zero padded
        shapes = {"T": nl * 12, "J": 6 * nd, "V": S, "G": nd * S}
        guard = 4096                                                     # canary behind every host buffer
        bufs = {k: np.full(NT * c * 32 + guard, -7.0) for k, c in shapes.items()}
        amb = np.full(NT * S * 32 + guard, -7, dtype=np.int32)
        c = _fused_call(dm, N, qt.ctypes.data, L.TILED32, fk, jac, bufs["T"].ctypes.data, bufs["J"].ctypes.data,
                        bufs["V"].ctypes.data, bufs["G"].ctypes.data, amb.ctypes.data)
        L.check(L.lib().kin_eval_host(dm.h, C.byref(c)))
        for k, cnt in shapes.items():
            assert np.all(bufs[k][NT * cnt * 32:] == -7.0), k             # nothing written past the padded tiles
        assert np.all(amb[NT * S * 32:] == -7)
        un = lambda a, cnt: untile32(torch.as_tensor(a[:NT * cnt * 32].reshape(NT, cnt, 32)), N).numpy()
        sub = slice(max(0, N - 300), N)                                  # the ragged tail
        T = un(bufs["T"], nl * 12)[sub].reshape(-1, nl, 4, 3).transpose(0, 1, 3, 2)
        np.testing.assert_allclose(T, R.batch_fk(mo, jo, q[sub], mo.links[:25])[:, :, :3, :], rtol=RTOL, atol=ATOL)
        v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q[sub])
        np.testing.assert_allclose(un(bufs["V"], S)[sub], v_ref, rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(un(bufs["G"], nd * S)[sub].reshape(-1, S, nd), g_ref, rtol=0, atol=1e-7)
        assert np.array_equal(un(amb, S)[sub], am_ref)


def test_moving_obstacle_updates_boxes_in_place():
    """kin_model_set_boxes with an unchanged box count rewrites the box rows of the compiled programs in place
    (sdf.jl:14-32: the attached SDF follows its mechanism); results follow the obstacle and match the oracle."""
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    q = scenes.random_configs(jo, 500, False, seed=44)
    K.set_joint_angles(m, joints, dev(q))
    for k, xyz in enumerate(([1.0, 0.0, 0.8], [0.7, 0.2, 0.9], [0.5, -0.3, 0.6])):
        pose = target_pose(xyz, 0.3 * k)
        box, box_o = K.BoxSDF(K.Transform(pose), [0.3, 0.2, 0.4]), R.BoxSDF(pose, [0.3, 0.2, 0.4])
        vals, grads, am = K.compute_coll_dists_and_grads(sscc, joints, box, return_argmin=True)
        v_ref, g_ref, am_ref = R.batch_collision(so, jo, box_o, q)
        np.testing.assert_allclose(host(vals), v_ref, rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(host(grads), g_ref.transpose(0, 2, 1), rtol=0, atol=1e-7)


def target_pose(xyz, yaw):
    P = np.eye(4)
    P[:3, :3] = [[np.cos(yaw), -np.sin(yaw), 0], [np.sin(yaw), np.cos(yaw), 0], [0, 0, 1]]
    P[:3, 3] = xyz
    return P


def test_debug_build_bounds_checks_pass():
    """The -DKIN_DEBUG library (table / scratch indices range-checked inside the kernels, the analogue of the
    reference's @debugassert with debugging() = true, test/runtests.jl:8) runs the smoke scene without tripping."""
    import subprocess
    import sys
    if not os.path.exists(L.SO_PATH_DEBUG):
        pytest.skip("libkin_b200_debug.so not built")
    code = ("import sys; sys.path.insert(0, %r); import __graft_entry__ as g; "
            "from kinematics_jl_b200 import lib as L; assert L.lib().kin_debug_build() == 1; g.smoke()") % os.path.dirname(DATA)
    env = dict(os.environ, KIN_DEBUG="1")
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "smoke ok" in out.stdout and "KIN_DEBUG assertion failed" not in out.stdout + out.stderr


def _transfer_counters():
    vals = [C.c_int64() for _ in range(3)]
    L.check(L.lib().kin_host_transfer_bytes(*[C.byref(v) for v in vals]))
    return vals


@pytest.mark.parametrize("layout", [L.AOS, L.SOA])
def test_fused_device_and_host_entry_points(layout):
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    N = 140000                                  # > one staging chunk (131072) of kin_eval_host
    q = scenes.random_configs(jo, N, False, seed=41)
    K.set_joint_angles(m, joints, dev(q[:1]))
    K.compute_coll_dists(sscc, joints, sdf)     # uploads the sphere / box tables into the device model
    dm = device_model(m)
    fk = np.arange(1, 26, dtype=np.int32)
    jac = np.array([K.find_link(m, "gripper_link").id], dtype=np.int32)
    nl, S, nd = 25, 16, 8
    qh = np.ascontiguousarray(q if layout == L.AOS else q.T)
    shapes = {"T": nl * 12, "J": 6 * nd, "V": S, "G": nd * S}
    outs_h = {k: np.full((N, c) if layout == L.AOS else (c, N), -7.0) for k, c in shapes.items()}     # every element must be written
    am_h = np.zeros((N, S) if layout == L.AOS else (S, N), dtype=np.int32)
    c = _fused_call(dm, N, qh.ctypes.data, layout, fk, jac, outs_h["T"].ctypes.data, outs_h["J"].ctypes.data,
                    outs_h["V"].ctypes.data, outs_h["G"].ctypes.data, am_h.ctypes.data)
    cnt = lambda: tuple(x.value for x in _transfer_counters())
    b0 = cnt()
    L.check(L.lib().kin_eval_host(dm.h, C.byref(c)))
    h2d, d2h, filled = (a - b for a, b in zip(cnt(), b0))
    full = 8 * N * (nl * 12 + 6 * nd + S + nd * S) + 4 * N * S
    assert h2d == 8 * N * nd
    if layout == L.SOA:
        # the rows of T / J that do not depend on the configuration are filled by host threads, not copied over PCIe
        # ... nor are the rows that duplicate another row (same variable of the generated code, possibly negated):
        # 175 constant + 67 duplicate rows of the 348 for Fetch with the 8 arm joints
        assert filled >= 8 * N * 230 and d2h + filled == full
        outs_2 = {k: np.full_like(v, -7.0) for k, v in outs_h.items()}
        c2 = _fused_call(dm, N, qh.ctypes.data, layout, fk, jac, outs_2["T"].ctypes.data, outs_2["J"].ctypes.data,
                         outs_2["V"].ctypes.data, outs_2["G"].ctypes.data, am_h.ctypes.data)
        os.environ["KIN_HOST_NO_CONST_FILL"] = "1"
        try:
            L.check(L.lib().kin_eval_host(dm.h, C.byref(c2)))
        finally:
            del os.environ["KIN_HOST_NO_CONST_FILL"]
        for k in outs_h:
            assert np.array_equal(outs_h[k], outs_2[k]), k
    else:
        assert filled == 0 and d2h == full
    qd = dev(qh)
    outs_d = {k: torch.zeros(v.shape, dtype=torch.float64, device="cuda") for k, v in outs_h.items()}
    am_d = torch.zeros(am_h.shape, dtype=torch.int32, device="cuda")
    c = _fused_call(dm, N, qd.data_ptr(), layout, fk, jac, outs_d["T"].data_ptr(), outs_d["J"].data_ptr(),
                    outs_d["V"].data_ptr(), outs_d["G"].data_ptr(), am_d.data_ptr())
    c.stream = torch.cuda.current_stream().cuda_stream
    L.check(L.lib().kin_eval(dm.h, C.byref(c)))
    torch.cuda.synchronize()
    for k in outs_h:
        assert np.array_equal(outs_h[k], outs_d[k].cpu().numpy()), k      # same kernel, same bits
    assert np.array_equal(am_h, am_d.cpu().numpy())
    rec = (lambda a: a) if layout == L.AOS else (lambda a: a.T)
    sub = slice(0, 2000)
    T = rec(outs_h["T"])[sub].reshape(-1, nl, 4, 3).transpose(0, 1, 3, 2)
    np.testing.assert_allclose(T, R.batch_fk(mo, jo, q[sub], mo.links[:25])[:, :, :3, :], rtol=RTOL, atol=ATOL)
    J = rec(outs_h["J"])[sub].reshape(-1, nd, 6).transpose(0, 2, 1)
    np.testing.assert_allclose(J, R.batch_jacobian(mo, jo, q[sub], [R.find_link(mo, "gripper_link")], True)[:, 0], rtol=RTOL, atol=ATOL)
    v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q[sub])
    np.testing.assert_allclose(rec(outs_h["V"])[sub], v_ref, rtol=RTOL, atol=ATOL)
    np.testing.assert_allclose(rec(outs_h["G"])[sub].reshape(-1, S, nd), g_ref, rtol=0, atol=1e-7)
    assert np.array_equal(rec(am_h)[sub], am_ref)


# ------------------------------------------------------------------------------------------------
# BASELINE.json full size (2^24 configurations): size-independent properties
# ------------------------------------------------------------------------------------------------
def test_full_size_properties():
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    N = 1 << 24
    g = torch.Generator(device="cuda").manual_seed(0)
    lo = torch.tensor([j.lower_limit if np.isfinite(j.lower_limit) else -np.pi for j in joints], device="cuda", dtype=torch.float64)
    hi = torch.tensor([j.upper_limit if np.isfinite(j.upper_limit) else np.pi for j in joints], device="cuda", dtype=torch.float64)
    Qs = (lo[:, None] + (hi - lo)[:, None] * torch.rand((8, N), generator=g, device="cuda", dtype=torch.float64))
    K.set_joint_angles(m, joints, Qs.t())                       # SoA
    gl = K.find_link(m, "gripper_link")
    T = K.get_transform(m, m.links[:25])                        # (N, 25, 3, 4) view
    Rm = T[..., :3]
    # every link rotation is orthonormal with det +1
    err = (Rm.transpose(-1, -2) @ Rm - torch.eye(3, device="cuda", dtype=torch.float64)).abs().amax()
    assert float(err) < 1e-13
    assert float((torch.linalg.det(Rm[:, gl.id - 1]) - 1).abs().max()) < 1e-13
    # geometric Jacobian of the gripper: column of a revolute joint is orthogonal to its own angular part
    J = K.get_jacobian(m, gl, joints, True)                     # (N, 6, 8)
    dots = (J[:, :3, 1:] * J[:, 3:, 1:]).sum(1).abs().amax()
    assert float(dots) < 1e-13
    assert float((J[:, 3:, 1:].norm(dim=1) - 1).abs().max()) < 1e-13       # unit axes
    assert float(J[:, 3:, 0].abs().max()) == 0.0 and float((J[:, :3, 0].norm(dim=1) - 1).abs().max()) < 1e-13
    # reach bound: torso height (0.38 + 0.39) + arm length (~1.3 m) from the base origin
    assert float(T[:, gl.id - 1, :, 3].norm(dim=1).max()) < 2.3
    del T, Rm, J
    # collision: distances bounded by the workspace, argmin in range, first / last chunks equal the oracle
    vals, grads, am = K.compute_coll_dists_and_grads(sscc, joints, sdf, return_argmin=True)
    assert int(am.min()) >= 1 and int(am.max()) <= 7
    assert bool(torch.isfinite(vals).all()) and bool(torch.isfinite(grads).all())
    for sl in (slice(0, 512), slice(N - 512, N)):
        qs = Qs[:, sl].t().contiguous().cpu().numpy()
        v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, qs)
        np.testing.assert_allclose(host(vals[sl]), v_ref, rtol=RTOL, atol=ATOL)
        assert np.array_equal(am[sl].cpu().numpy(), am_ref)
        np.testing.assert_allclose(host(grads[sl]), g_ref.transpose(0, 2, 1), rtol=0, atol=1e-7)
    # checksum of checksums: AoS and SoA runs of the same kernel agree bit for bit
    sub = Qs[:, : 1 << 20]
    K.set_joint_angles(m, joints, sub.t())
    v_soa = K.compute_coll_dists(sscc, joints, sdf)
    K.set_joint_angles(m, joints, sub.t().contiguous())
    v_aos = K.compute_coll_dists(sscc, joints, sdf)
    assert torch.equal(v_soa, v_aos)


# ------------------------------------------------------------------------------------------------
# tiled (AoSoA-32) layout: same kernel, one contiguous block per warp
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_base", [False, True])
def test_tiled_layout_matches_soa_bitwise(with_base):
    from kinematics_jl_b200.device import current_q, evaluate
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(with_base)
    q = scenes.random_configs(jo, 1000, with_base, seed=81)         # ragged: 1000 = 31 tiles + 8
    K.set_joint_angles(m, joints, dev(q))
    K.compute_coll_dists(sscc, joints, sdf)                         # uploads sphere / box tables
    dm = device_model(m)
    Q, ql, N = current_q(m)
    kw = dict(fk_links=[l.id for l in m.links[:25]], jac_links=[K.find_link(m, "gripper_link").id], with_rot=True,
              collision=True, with_grads=True, want_argmin=True)
    a = evaluate(dm, Q, ql, N, layout=L.SOA, **kw)
    b = evaluate(dm, Q, ql, N, layout=L.TILED32, **kw)
    for k in ("T", "J", "vals", "grads", "argmin"):
        assert torch.equal(a[k].contiguous(), b[k].contiguous()), k
    np.testing.assert_allclose(host(b["T"]), R.batch_fk(mo, jo, q, mo.links[:25])[:, :, :3, :], rtol=RTOL, atol=ATOL)


# ------------------------------------------------------------------------------------------------
# generality: branching tree, general joint axes, rpy joint origins, frozen joints, shuffled columns
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_base", [False, True])
@pytest.mark.parametrize("n_ctrl", [None, 4])          # 9 columns: frames in shared scratch; 4: frames in registers
@pytest.mark.parametrize("layout", [L.SOA, L.AOS, L.TILED32])
def test_synthetic_branching_tree(with_base, n_ctrl, layout):
    import scenes_synthetic as SS
    from kinematics_jl_b200.device import current_q, evaluate
    m, joints, sscc, sdf = SS.product(with_base, n_ctrl)
    mo, jo, so, sdf_o = SS.oracle(with_base, n_ctrl)
    if n_ctrl is not None:
        for name, a in zip(SS.JOINTS[n_ctrl:], [0.3, -0.4, 0.5, 0.1, -0.2]):
            K.set_joint_angle(m, K.find_joint(m, name), a)
            R.set_joint_angles(mo, [R.find_joint(mo, name)], [a] + ([0, 0, 0] if with_base else []))
    q = SS.random_q(jo, 333, with_base, seed=7)
    K.set_joint_angles(m, joints, dev(q))
    K.compute_coll_dists(sscc, joints, sdf)
    dm = device_model(m)
    Q, ql, N = current_q(m)
    ids = [l.id for l in m.links]
    for rpy_jac in (False, True):
        for scratch, scratch_o in ((K.SCRATCH_REFERENCE, R.SCRATCH_REFERENCE), (K.SCRATCH_CLEAN, R.SCRATCH_CLEAN)):
            out = evaluate(dm, Q, ql, N, layout=layout, fk_links=ids, jac_links=ids, with_rot=True, rpy_jac=rpy_jac,
                           collision=True, with_grads=True, want_argmin=True, truncation_dist=0.3, scratch_mode=scratch)
            np.testing.assert_allclose(host(out["T"]), R.batch_fk(mo, jo, q, mo.links)[:, :, :3, :], rtol=RTOL, atol=ATOL)
            np.testing.assert_allclose(host(out["J"]), R.batch_jacobian(mo, jo, q, mo.links, True, rpy_jac), rtol=1e-11, atol=1e-11)
            v_ref, g_ref, am_ref = R.batch_collision(so, jo, sdf_o, q, 0.3, R.GRAD_FD, scratch_o)
            np.testing.assert_allclose(host(out["vals"]), v_ref, rtol=RTOL, atol=ATOL)
            assert np.array_equal(out["argmin"].cpu().numpy(), am_ref)
            np.testing.assert_allclose(host(out["grads"]), g_ref.transpose(0, 2, 1), rtol=0, atol=1e-7)


# ------------------------------------------------------------------------------------------------
# edge cases and error behaviour of the C ABI
# ------------------------------------------------------------------------------------------------
def test_edge_cases_and_errors():
    from kinematics_jl_b200.device import current_q, evaluate
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    # tiny and ragged batches in every layout
    for N in (1, 2, 31, 33, 129):
        q = scenes.random_configs(jo, N, False, seed=N)
        K.set_joint_angles(m, joints, dev(q))
        K.compute_coll_dists(sscc, joints, sdf)
        dm = device_model(m)
        Q, ql, n = current_q(m)
        ref_T = R.batch_fk(mo, jo, q, mo.links[:25])[:, :, :3, :]
        ref_v = R.batch_collision(so, jo, sdf_o, q, with_grads=False)[0]
        for layout in (L.SOA, L.AOS, L.TILED32):
            o = evaluate(dm, Q, ql, n, layout=layout, fk_links=[l.id for l in m.links[:25]], collision=True, with_grads=True)
            np.testing.assert_allclose(host(o["T"]), ref_T, rtol=RTOL, atol=ATOL)
            np.testing.assert_allclose(host(o["vals"]), ref_v, rtol=RTOL, atol=ATOL)
    # no control joints at all: every link is a constant; with a base: three columns only
    for with_base in (False, True):
        mm, _, _ = scenes.product_fetch(with_base)
        mmo, _, _ = scenes.oracle_fetch(with_base)
        K.set_joint_angle(mm, K.find_joint(mm, "head_pan_joint"), 0.3)
        R.set_joint_angles(mmo, [R.find_joint(mmo, "head_pan_joint")], [0.3] + ([0, 0, 0] if with_base else []))
        qb = np.array([[0.4, -0.2, 1.1], [0.0, 0.0, 0.0]]) if with_base else np.zeros((2, 0))
        K.set_joint_angles(mm, [], dev(qb) if with_base else torch.zeros((2, 0), dtype=torch.float64, device="cuda"))
        T = host(K.get_transform(mm, mm.links[:25]))
        np.testing.assert_allclose(T, R.batch_fk(mmo, [], qb, mmo.links[:25])[:, :, :3, :], rtol=RTOL, atol=ATOL)
    # errors are exceptions carrying kin_last_error(), never crashes
    K.set_joint_angles(m, joints, dev(scenes.random_configs(jo, 4, False, seed=1)))
    dm = device_model(m)
    Q, ql, n = current_q(m)
    with pytest.raises(K.KinError):
        evaluate(dm, Q, ql, n, fk_links=[0])                      # ids are 1-based
    with pytest.raises(K.KinError):
        evaluate(dm, Q, ql, n, fk_links=[len(m.links) + 1])
    m2, joints2, _ = scenes.product_fetch(False, sphere_links=[])
    K.set_joint_angles(m2, joints2, dev(scenes.random_configs(jo, 4, False, seed=1)))
    with pytest.raises(K.KinError):                               # collision without spheres / boxes
        evaluate(device_model(m2), *current_q(m2), collision=True)
    with pytest.raises(ValueError):                               # joints must be the ones of set_joint_angles
        K.get_jacobian(m, K.find_link(m, "gripper_link"), joints[:3], True)


# ------------------------------------------------------------------------------------------------
# per-configuration reductions of the sphere distances (kin_collision_summary, extension)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 777, (1 << 20) + 77])          # the last one spans two chunks of the temporary
def test_collision_summary_reductions(n, monkeypatch):
    from kinematics_jl_b200.device import tile32
    m, joints, sscc, sdf, mo, jo, so, sdf_o = _fridge_scene(False)
    q = scenes.random_configs(jo, n, False, seed=91, zeros_every=50)
    Q = dev(q)
    margin = 0.1
    K.set_joint_angles(m, joints, Q)                               # AoS: groups of lanes + warp shuffles
    d_all = K.compute_coll_dists(sscc, joints, sdf)
    dmin_a, amin_a, cost_a = K.compute_coll_summary(sscc, joints, sdf, margin=margin)
    K.set_joint_angles(m, joints, soa(Q))                          # SoA: one thread per configuration
    dmin_s, amin_s, cost_s = K.compute_coll_summary(sscc, joints, sdf, margin=margin)
    ref_min, ref_arg = d_all.min(dim=1)
    ref_cost = torch.clamp(margin - d_all, min=0).pow(2).sum(dim=1)
    for dmin, amin, cost in ((dmin_a, amin_a, cost_a), (dmin_s, amin_s, cost_s)):
        assert torch.equal(dmin, ref_min)                          # a minimum is exact whatever the order
        first = (d_all == ref_min[:, None]).int().argmax(dim=1)    # first minimum, as the serial walk
        assert torch.equal(amin.long(), first + 1)
        np.testing.assert_allclose(host(cost), host(ref_cost), rtol=1e-13, atol=1e-15)
    if n > 1:
        assert float(cost_a.max()) > 0 and bool((cost_a == 0).any())      # both branches of the hinge
    # tiled layout through the C ABI
    dm_ = device_model(m)
    Qt = tile32(Q)
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    am = torch.empty(n, dtype=torch.int32, device="cuda")
    co = torch.empty(n, dtype=torch.float64, device="cuda")
    L.check(L.lib().kin_collision_summary(dm_.h, L.F64, L.TILED32, Qt.data_ptr(), n, margin, out.data_ptr(), am.data_ptr(), co.data_ptr(),
                                          torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert torch.equal(out, ref_min) and torch.equal(am, amin_s) and torch.equal(co, cost_s)
    # against the oracle
    sub = slice(0, min(n, 400))
    v_ref, _, _ = R.batch_collision(so, jo, sdf_o, q[sub], with_grads=False)
    np.testing.assert_allclose(host(dmin_a[sub]), v_ref.min(axis=1), rtol=RTOL, atol=ATOL)
    assert np.array_equal(amin_a[sub].cpu().numpy(), v_ref.argmin(axis=1) + 1)
    np.testing.assert_allclose(host(cost_a[sub]), (np.clip(margin - v_ref, 0, None) ** 2).sum(axis=1), rtol=1e-11, atol=1e-13)


@pytest.mark.parametrize("precision", [L.F64, L.F32])
def test_host_entry_point_row_elision_with_padded_rows_and_fp32(precision):
    """kin_eval_host, SoA, host arrays whose rows are LONGER than the batch (batch_stride > n) and the FP32 mode: the rows
    that stay off PCIe (constants filled, duplicates copied by host threads) must land in the right place and hold the bits
    the device-resident call produces; the padding behind each row is not touched."""
    m, joints, _ = scenes.product_fetch(False)
    mo, jo, _ = scenes.oracle_fetch(False)
    N, ld = 140001, 140001 + 23                       # two staging chunks, ragged, padded rows
    q = scenes.random_configs(jo, N, False, seed=97)
    K.set_joint_angles(m, joints, dev(q[:1]))
    dm = device_model(m)
    fk = np.arange(1, 26, dtype=np.int32)
    jac = np.array([K.find_link(m, "gripper_link").id], dtype=np.int32)
    npdt = np.float64 if precision == L.F64 else np.float32
    tdt = torch.float64 if precision == L.F64 else torch.float32
    qh = np.zeros((8, ld), dtype=npdt)
    qh[:, :N] = q.T
    Th = np.full((300, ld), -7.0, dtype=npdt)
    Jh = np.full((48, ld), -7.0, dtype=npdt)

    def call(qp, tp, jp):
        c = L.KinCall()
        c.precision, c.layout, c.n, c.batch_stride, c.q = precision, L.SOA, N, ld, qp
        c.n_fk_links, c.fk_links, c.T_out = 25, fk.ctypes.data_as(C.POINTER(C.c_int32)), tp
        c.n_jac_links, c.jac_links, c.J_out, c.with_rot = 1, jac.ctypes.data_as(C.POINTER(C.c_int32)), jp, 1
        c.truncation_dist = float("inf")
        return c
    b0 = [x.value for x in _transfer_counters()]
    L.check(L.lib().kin_eval_host(dm.h, C.byref(call(qh.ctypes.data, Th.ctypes.data, Jh.ctypes.data))))
    h2d, d2h, filled = (a.value - b for a, b in zip(_transfer_counters(), b0))
    es = 8 if precision == L.F64 else 4
    assert d2h + filled == es * N * 348 and filled >= es * N * 230
    Qd = torch.as_tensor(qh, device="cuda")
    Td = torch.zeros((300, ld), dtype=tdt, device="cuda")
    Jd = torch.zeros((48, ld), dtype=tdt, device="cuda")
    c = call(Qd.data_ptr(), Td.data_ptr(), Jd.data_ptr())
    c.stream = torch.cuda.current_stream().cuda_stream
    L.check(L.lib().kin_eval(dm.h, C.byref(c)))
    torch.cuda.synchronize()
    assert np.array_equal(Th[:, :N], Td[:, :N].cpu().numpy()) and np.array_equal(Jh[:, :N], Jd[:, :N].cpu().numpy())
    assert np.all(Th[:, N:] == -7.0) and np.all(Jh[:, N:] == -7.0)
    if precision == L.F64:
        sub = slice(0, 500)
        T = Th[:, sub].T.reshape(-1, 25, 4, 3).transpose(0, 1, 3, 2)
        np.testing.assert_allclose(T, R.batch_fk(mo, jo, q[sub], mo.links[:25])[:, :, :3, :], rtol=RTOL, atol=ATOL)

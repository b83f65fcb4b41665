"""GPU tests of the self-collision extension (kin_self_collision; collision.jl has sphere-vs-environment only): the
product against the oracle of tests/self_collision_ref.py on Fetch and on the dual-arm model, the three layouts
against each other, the summary outputs against the values of the same call, gradients against central differences,
the C entry points' error paths, and the planner's self-collision constraint.
FP64 is held at rounding level (1e-12).  FP32: distances within 2e-5 and gradients within 2e-4 -- the sphere centres
carry FP32 rounding of ~1e-6 m after the chain, and the gradient's unit vector u = (c_i - c_j) / L amplifies it by 1 / L."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import device_model, tile32
from oracle import ref_model as R
from conftest import DATA, ROOT
import scenes
import scenes_dual_arm as DA
import self_collision_ref as SR
from test_gpu_parity import dev, host
from test_self_collision_cpu import ONE_JOINT_URDF

pytestmark = pytest.mark.gpu

N_RAGGED = 1000 + 7          # neither a multiple of 32 nor of any CTA size
LAYOUTS = (L.SOA, L.AOS, L.TILED32)


def _case(name, with_base):
    if name == "fetch":
        m, joints, sscc = scenes.product_fetch(with_base)
        mo, jo, so = scenes.oracle_fetch(with_base)
    else:
        m, joints, sscc, _ = DA.product(with_base)
        mo, jo, so, _ = DA.oracle(with_base)
    return m, joints, sscc, jo, so


def _run(m, joints, sscc, q, dtype, layout, pairs=None, trunc=np.inf, off=0.0):
    K.set_joint_angles(m, joints, dev(q, dtype))
    v, g = K.compute_self_coll_dists_and_grads(sscc, joints, pairs, truncation_dist=trunc, vals_offset=off, layout=layout)
    dmin, amin = K.compute_self_coll_summary(sscc, joints, pairs)
    return v, g, dmin, amin


@pytest.mark.parametrize("name,with_base", [("fetch", False), ("fetch", True), ("dual_arm", False), ("dual_arm", True)])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_vs_oracle_all_layouts(name, with_base, dtype):
    m, joints, sscc, jo, so = _case(name, with_base)
    pairs = K.self_collision_pairs(sscc, joints)
    assert len(pairs) == {"fetch": 80, "dual_arm": 145}[name]
    q = scenes.random_configs(jo, N_RAGGED, with_base, seed=3)
    vr, gr, raw = SR.batch(so, jo, q, pairs)
    assert (raw < 0).any() and (raw > 0).any()                        # pairs in contact and pairs apart
    if name == "dual_arm":
        assert (raw.min(1) < 0).any() and (raw.min(1) > 0).any()   # self-colliding and self-free configurations
    outs = [_run(m, joints, sscc, q, dtype, lay) for lay in LAYOUTS]
    v, g, dmin, amin = outs[0]
    assert v.shape == (N_RAGGED, len(pairs)) and g.shape == (N_RAGGED, len(jo) + (3 if with_base else 0), len(pairs))
    for o in outs[1:]:                                               # the layouts agree bit for bit
        assert torch.equal(o[0], v) and torch.equal(o[1], g) and torch.equal(o[2], dmin) and torch.equal(o[3], amin)
    # dmin / amin are the first-minimum reduction of the untruncated values of the same call
    assert torch.equal(dmin, v.min(dim=1).values) and torch.equal(amin.long(), v.argmin(dim=1) + 1)
    if dtype == torch.float64:
        np.testing.assert_allclose(host(v), vr, rtol=0, atol=1e-12)
        np.testing.assert_allclose(host(g), gr, rtol=0, atol=1e-12)
        np.testing.assert_allclose(host(dmin), raw.min(1), rtol=0, atol=1e-12)
        # the pair named by amin attains the oracle's minimum (pairs of mirror-image spheres can tie to rounding)
        a = amin.cpu().numpy()
        assert a.min() >= 1 and a.max() <= len(pairs)
        np.testing.assert_allclose(raw[np.arange(N_RAGGED), a - 1], raw.min(1), rtol=0, atol=1e-12)
        assert (a == raw.argmin(1) + 1).mean() > 0.99
    else:
        np.testing.assert_allclose(host(v), vr, rtol=0, atol=2e-5)
        np.testing.assert_allclose(host(g), gr, rtol=0, atol=2e-4)
        np.testing.assert_allclose(host(dmin), raw.min(1), rtol=0, atol=2e-5)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_truncation_and_offset(layout):
    m, joints, sscc, jo, so = _case("dual_arm", True)
    pairs = K.self_collision_pairs(sscc, joints)
    q = scenes.random_configs(jo, 333, True, seed=8)
    vr, gr, raw = SR.batch(so, jo, q, pairs, truncation_dist=0.07, offset=0.02)
    assert 0.1 < (raw > 0.07).mean() < 0.999
    v, g, dmin, _ = _run(m, joints, sscc, q, torch.float64, layout, trunc=0.07, off=0.02)
    np.testing.assert_allclose(host(v), vr, rtol=0, atol=1e-12)
    np.testing.assert_allclose(host(g), gr, rtol=0, atol=1e-12)
    assert np.all(host(g)[np.broadcast_to((raw > 0.07)[:, None, :], gr.shape)] == 0.0)
    np.testing.assert_allclose(host(dmin), raw.min(1), rtol=0, atol=1e-12)     # the summary ignores truncation


def test_gradient_is_the_central_difference_of_the_values():
    """Independent of the oracle's Jacobians: d vals / d q by central differences of the product's own values."""
    m, joints, sscc, jo, so = _case("dual_arm", True)
    q = scenes.random_configs(jo, 64, True, seed=12)
    v, g, _, _ = _run(m, joints, sscc, q, torch.float64, L.SOA)
    h = 1e-6
    for k in range(q.shape[1]):
        e = np.zeros(q.shape[1])
        e[k] = h
        vp = _run(m, joints, sscc, q + e, torch.float64, L.SOA)[0]
        vm = _run(m, joints, sscc, q - e, torch.float64, L.SOA)[0]
        np.testing.assert_allclose(host(g)[:, k, :], host(vp - vm) / (2 * h), rtol=0, atol=1e-7)


def test_coincident_centres_give_a_zero_gradient(tmp_path):
    p = tmp_path / "one.urdf"
    p.write_text(ONE_JOINT_URDF)
    m = K.parse_urdf(str(p))
    joints = [K.find_joint(m, "hinge")]
    sscc = K.SweptSphereCollisionChecker(m)
    a, b = 0.7, 0.4
    K.add_coll_links(sscc, K.find_link(m, "arm"), [[a, 0, 0], [0, 0, 0.1]], 0.05)
    K.add_coll_links(sscc, K.find_link(m, "base"), [[b, 0, 0], [0, 0, 0.1]], 0.08)
    pairs = [(1, 3), (2, 4)]                       # (2, 4): both centres on the axis, L == 0 at every angle
    t = np.linspace(-3, 3, 77)[:, None]
    for layout in LAYOUTS:
        K.set_joint_angles(m, joints, dev(t))
        v, g = K.compute_self_coll_dists_and_grads(sscc, joints, pairs, layout=layout)
        Lc = np.sqrt(a * a + b * b - 2 * a * b * np.cos(t[:, 0]))
        np.testing.assert_allclose(host(v)[:, 0], Lc - 0.13, rtol=0, atol=1e-14)
        np.testing.assert_allclose(host(g)[:, 0, 0], a * b * np.sin(t[:, 0]) / Lc, rtol=0, atol=1e-14)
        np.testing.assert_allclose(host(v)[:, 1], -0.13, rtol=0, atol=1e-15)
        assert np.all(host(g)[:, 0, 1] == 0.0)


def test_one_launch_per_call_and_summary_writes_nothing_else():
    m, joints, sscc, jo, so = _case("dual_arm", False)
    q = scenes.random_configs(jo, N_RAGGED, False, seed=4)
    K.set_joint_angles(m, joints, dev(q))
    v, _ = K.compute_self_coll_dists_and_grads(sscc, joints)            # sets up the model and the pair table
    dm = device_model(m)
    P, nd, N = dm.n_self_pairs, dm.n_dof, N_RAGGED
    Q = dev(q)
    lib = L.lib()
    stream = torch.cuda.current_stream().cuda_stream
    for layout in LAYOUTS:
        Qc = tile32(Q) if layout == L.TILED32 else (Q.t().contiguous() if layout == L.SOA else Q)
        # dmin / amin placed inside poisoned slabs: everything around them (and the vals / grads buffers that a
        # summary call does not get) must keep its bits
        slab = torch.full((3 * N,), float("nan"), dtype=torch.float64, device="cuda")
        islab = torch.full((3 * N,), -7, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        n0 = lib.kin_launch_count()
        L.check(lib.kin_self_collision(dm.h, L.F64, layout, Qc.data_ptr(), N, float("inf"), 0.0, None, None,
                                       slab[N:].data_ptr(), islab[N:].data_ptr(), stream))
        torch.cuda.synchronize()
        assert lib.kin_launch_count() - n0 == 1
        assert torch.isnan(slab[:N]).all() and torch.isnan(slab[2 * N:]).all()
        assert (islab[:N] == -7).all() and (islab[2 * N:] == -7).all()
        assert torch.equal(slab[N:2 * N], v.min(dim=1).values) and torch.equal(islab[N:2 * N].long(), v.argmin(dim=1) + 1)
        n0 = lib.kin_launch_count()
        K.compute_self_coll_dists_and_grads(sscc, joints, layout=layout)
        assert lib.kin_launch_count() - n0 == 1


def _pairs_rc(dm, pairs):
    a = np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))
    return L.lib().kin_model_set_self_pairs(dm.h, len(a), a.ctypes.data_as(C.POINTER(C.c_int32)))


def test_error_paths_and_a_model_without_boxes():
    m, joints, sscc = scenes.product_fetch()                     # spheres only: no SDF ever given to this model
    q = np.zeros((100, 8))
    K.set_joint_angles(m, joints, dev(q))
    d = K.compute_self_coll_dists(sscc, joints)
    dm = device_model(m)
    assert dm.n_boxes == 0 and L.lib().kin_model_n_boxes(dm.h) == 0 and d.shape == (100, 80)
    assert L.lib().kin_model_n_self_pairs(dm.h) == 80
    with pytest.raises(L.KinError):                               # environment collision still needs boxes
        L.check(L.lib().kin_collision_summary(dm.h, L.F64, L.AOS, dev(q).data_ptr(), 100, 0.0, dev(np.zeros(100)).data_ptr(),
                                              None, None, None))
    assert _pairs_rc(dm, [(1, 17)]) == -1 and _pairs_rc(dm, [(0, 2)]) == -1 and _pairs_rc(dm, [(3, 3)]) == -1
    assert "self-collision pair" in L.lib().kin_last_error().decode()
    assert _pairs_rc(dm, np.tile([1, 2], (4097, 1))) == -3
    assert _pairs_rc(dm, np.tile([1, 2], (4096, 1))) == 0 and L.lib().kin_model_n_self_pairs(dm.h) == 4096
    Q, out = dev(q), dev(np.zeros((100, 4096)))
    assert L.lib().kin_self_collision(dm.h, L.F64, L.AOS, Q.data_ptr(), 100, np.inf, 0.0, None, out.data_ptr(), None, None, None) == -1
    assert L.lib().kin_self_collision(dm.h, L.F64, L.AOS, Q.data_ptr(), 100, np.inf, 0.0, None, None, None, None, None) == -1
    assert L.lib().kin_self_collision(dm.h, L.F64, L.AOS, Q.data_ptr(), 100, np.inf, 0.0, out.data_ptr(), None, None, None, None) == 0
    torch.cuda.synchronize()
    assert np.allclose(host(out)[:, 0], host(out)[0, 0])
    assert _pairs_rc(dm, np.zeros((0, 2))) == 0 and L.lib().kin_model_n_self_pairs(dm.h) == 0
    rc = L.lib().kin_self_collision(dm.h, L.F64, L.AOS, Q.data_ptr(), 100, np.inf, 0.0, out.data_ptr(), None, None, None, None)
    assert rc == -1 and "no pair table" in L.lib().kin_last_error().decode()
    dm._pair_sig = None
    K.compute_self_coll_dists(sscc, joints)                       # the pair table again
    assert L.lib().kin_model_n_self_pairs(dm.h) == 80
    # a sphere table that actually changes drops the pair table in the library; the mirror re-applies it
    sscc.sphere_radii[0] += 0.01
    dm.set_spheres(sscc._parents, sscc._centers, sscc.sphere_radii)
    assert L.lib().kin_model_n_self_pairs(dm.h) == 0 and dm.n_self_pairs == 0
    d2 = K.compute_self_coll_dists(sscc, joints)
    assert device_model(m) is dm and L.lib().kin_model_n_self_pairs(dm.h) == 80
    np.testing.assert_allclose(host(d2[:, :16]), host(d[:, :16]) - (np.asarray(K.self_collision_pairs(sscc, joints))[:16, 0] == 1) * 0.01)


def test_pair_table_leaves_environment_collision_bit_identical():
    m, joints, sscc, sdf = DA.product(True)
    mo, jo, so, _ = DA.oracle(True)
    q = dev(scenes.random_configs(jo, 2048, True, seed=6))
    K.set_joint_angles(m, joints, q)
    before = K.compute_coll_dists_and_grads(sscc, joints, sdf, truncation_dist=0.07, layout=L.SOA)
    K.compute_self_coll_dists_and_grads(sscc, joints)
    K.set_joint_angles(m, joints, q)
    after = K.compute_coll_dists_and_grads(sscc, joints, sdf, truncation_dist=0.07, layout=L.SOA)
    assert torch.equal(before[0], after[0]) and torch.equal(before[1], after[1])


def test_debug_library_runs_a_self_collision_call_clean():
    if not os.path.exists(L.SO_PATH_DEBUG):
        pytest.skip("libkin_b200_debug.so not built")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import numpy as np, torch; "
            "import kinematics_jl_b200 as K; from kinematics_jl_b200 import lib as L; import scene_fetch as SF; "
            "assert L.lib().kin_debug_build() == 1; m, j, s, _ = SF.product_dual_arm(True); "
            "K.set_joint_angles(m, j, torch.rand(777, 18, dtype=torch.float64, device='cuda')); "
            "v, g = K.compute_self_coll_dists_and_grads(s, j, layout=L.AOS); d, a = K.compute_self_coll_summary(s, j); "
            "torch.cuda.synchronize(); print('self ok', v.shape, g.shape)") % (ROOT, os.path.join(ROOT, "tests"))
    out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, KIN_DEBUG="1"), capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "self ok" in out.stdout and "KIN_DEBUG assertion failed" not in out.stdout + out.stderr


def test_self_ineq_const_vs_oracle_at_planner_size():
    m, joints, sscc, jo, so = _case("dual_arm", False)
    P_, n_wp, margin = 64, 64, 0.02
    G = K.SelfIneqConst(sscc, joints, n_wp, margin)
    assert G.n_coll == 145 and G.n_cons == 145 * n_wp
    X = scenes.random_configs(jo, P_ * n_wp, False, seed=9).reshape(P_, n_wp, -1)
    vals, blocks = G(dev(X))
    assert vals.shape == (P_, n_wp, 145) and blocks.shape == (P_, n_wp, 15, 145)
    sel = np.random.default_rng(0).choice(P_ * n_wp, 300, replace=False)
    vr, gr, _ = SR.batch(so, jo, X.reshape(P_ * n_wp, -1)[sel], G.pairs, truncation_dist=margin + 0.05, offset=margin)
    np.testing.assert_allclose(host(vals).reshape(P_ * n_wp, -1)[sel], vr, rtol=0, atol=1e-12)
    np.testing.assert_allclose(host(blocks).reshape(P_ * n_wp, 15, -1)[sel], gr, rtol=0, atol=1e-12)
    v1, b1 = G(X[5].reshape(-1))                                  # the single-problem (flat xi) form
    np.testing.assert_array_equal(v1, host(vals[5]).reshape(-1))
    assert G.dense(b1).shape == (15 * n_wp, 145 * n_wp)


# Found with the oracle by a seeded search (one arm moves, the other stays): both ends are clear of the boxes and of
# self-collision by > 0.07, and the straight line between them drives the right arm through the left one.
Q_START = np.array([0.09, -0.617, -0.817, -0.328, -0.045, -0.09, 0.744, 1.291, -0.063, -0.359, 0.549, -0.177, -0.681, -1.083, -1.259])
Q_GOAL = np.array([0.09, -0.617, -0.817, -0.328, -0.045, -0.09, 0.744, 1.291, 0.276, -0.391, -0.942, -0.885, -0.065, -1.301, 0.753])


def test_plan_trajectory_with_self_margin_dual_arm():
    m, joints, sscc, sdf = DA.product(False)
    mo, jo, so, sdo = DA.oracle(False)
    pairs = K.self_collision_pairs(sscc, joints)
    n_wp = 10
    line = [Q_START + (Q_GOAL - Q_START) * k / (n_wp - 1) for k in range(n_wp)]
    assert SR.batch(so, jo, np.array(line), pairs)[2].min() < -0.03          # the straight line self-collides
    q_seq, ret = K.plan_trajectory(sscc, joints, sdf, Q_START, Q_GOAL, n_wp, self_margin=0.02)
    assert ret.success, ret.message
    np.testing.assert_allclose(q_seq[0], Q_START, atol=1e-6)
    np.testing.assert_allclose(q_seq[-1], Q_GOAL, atol=1e-6)
    raw = SR.batch(so, jo, q_seq, pairs)[2]
    assert raw.min() >= 0.02 - 1e-4, raw.min(1)
    for q in q_seq:                                                          # clear of the boxes as before
        R.set_joint_angles(mo, jo, q)
        assert R.compute_coll_dists(so, jo, sdo).min() >= 0.02 - 1e-4

"""Self-collision as a hard constraint of the device-resident batched IK (kin_ik_solve_self), on the B200: the dual-arm
model (run-time-sized step kernel, 15 / 18 columns, the default 145-pair table) and Fetch (unrolled step kernel, 8 columns,
the 64-pair table without the constant pair that overlaps in every configuration).  Returned distances and objectives
are held to the oracles (tests/self_collision_ref.py for the pairs, the C oracle for spheres vs boxes and the pose
objective); the solve without compaction is held to the default path bit for bit; the single-problem SLSQP driver is
held to the same scipy SLSQP driven by the oracles."""
import ctypes as C

import numpy as np
import pytest
import torch

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from oracle import ref_model as R
import scenes
import scenes_dual_arm as DA
import scenes_synthetic as SS
import scene_fetch
import self_collision_ref as SR
from test_gpu_callers import _dual_arm_target, _oracle_ik, _pose_err, _pose_targets, dev, target_T

pytestmark = pytest.mark.gpu

MARGIN = 0.02
FETCH_IGNORE = [("wrist_flex_link", "elbow_flex_link")]


def _limits(joints, nd):
    nb = nd - len(joints)
    return (np.array([j.lower_limit for j in joints] + [-np.inf] * nb), np.array([j.upper_limit for j in joints] + [np.inf] * nb))


def _self_dmin(m, joints, sscc, q, pairs=None):
    K.set_joint_angles(m, joints, q if isinstance(q, torch.Tensor) else dev(q))
    return K.compute_self_coll_summary(sscc, joints, pairs)[0].cpu().numpy()


def _dual_arm_problems(with_base, N, seed):
    """Tool targets of in-limit configurations whose pairs are all >= 0.05 apart; random in-limit seeds."""
    m, joints, sscc, sdf = DA.product(with_base)
    mo, jo, so, sdf_o = DA.oracle(with_base)
    qc = SS.random_q(jo, 4 * N, with_base, seed=seed)
    idx = np.nonzero(_self_dmin(m, joints, sscc, qc) >= 0.05)[0][:N]
    assert idx.size == N
    link = K.find_link(m, "l_tool")
    tg = _pose_targets(m, joints, link, qc[idx])
    q0 = SS.random_q(jo, N, with_base, seed=seed + 1)
    return m, joints, sscc, sdf, mo, jo, so, sdf_o, link, tg, q0


@pytest.mark.parametrize("with_base", [False, True])
def test_dual_arm_self_constrained_batch(with_base):
    N = 2048
    m, joints, sscc, sdf, mo, jo, so, sdf_o, link, tg, q0 = _dual_arm_problems(with_base, N, 21)
    link_o = R.find_link(mo, "l_tool")
    nd = q0.shape[1]
    pairs = K.self_collision_pairs(sscc, joints)
    assert len(pairs) == 145
    # pose only, from the random seeds: a visible share ends closer than the margin (the constraint is exercised)
    q_free, _ = K.inverse_kinematics_batch(m, link, joints, dev(tg), dev(q0), with_rot=True, iters=40)
    viol0 = (_self_dmin(m, joints, sscc, q_free) < MARGIN - 1e-5).mean()
    q, f, dmin, sd = K.inverse_kinematics_batch(m, link, joints, dev(tg), dev(q0), with_rot=True, iters=40, sscc=sscc,
                                                self_margin=MARGIN, restarts=2, return_dmin=True)
    assert dmin is None
    reached = (_pose_err(m, joints, link, q, tg) < 1e-3).cpu().numpy()
    clear = (sd >= MARGIN - 1e-3).cpu().numpy()
    print("dual-arm IK under self-collision (%d columns, %d pairs): pose-only violates the margin in %.1f %%; constrained "
          "with 2 restarts: reached %.1f %% / clear %.1f %% / both %.1f %%"
          % (nd, len(pairs), 100 * viol0, 100 * reached.mean(), 100 * clear.mean(), 100 * (reached & clear).mean()))
    assert viol0 > 0.03
    assert clear.mean() > 0.97
    # first B200 run: 93.4 % (fixed base) and 99.9 % (planar base) reached and clear.  With a fixed base only the torso
    # and the left arm move the tool and the pose-only solve itself reaches ~90 % with restarts
    # (test_device_resident_ik_solve_dual_arm); the floors sit a few points below the measured shares
    assert (reached & clear).mean() > (0.97 if with_base else 0.88)
    lo, hi = _limits(joints, nd)
    qn, fn, sdn = q.cpu().numpy(), f.cpu().numpy(), sd.cpu().numpy()
    assert np.all(qn >= lo - 1e-12) and np.all(qn <= hi + 1e-12)
    err = _pose_err(m, joints, link, q, tg).cpu().numpy()
    for n in range(0, N, 101):
        R.set_joint_angles(mo, jo, qn[n])
        _, _, raw = SR.self_coll_dists_and_grads(so, jo, pairs)
        np.testing.assert_allclose(sdn[n], raw.min(), rtol=1e-10, atol=1e-12)
        fo, _ = R.ik_objective(mo, link_o, jo, qn[n], target_T(tg[n, :3], tg[n, 3:]), True)
        if err[n] < 1e-1:                                    # no 2 pi wrap in play
            np.testing.assert_allclose(fn[n], fo, rtol=1e-9, atol=1e-18)


def test_dual_arm_boxes_and_pairs_together():
    N = 1024
    m, joints, sscc, sdf, mo, jo, so, sdf_o, link, tg, q0 = _dual_arm_problems(True, N, 31)
    pairs = K.self_collision_pairs(sscc, joints)
    q, f, dmin, sd = K.inverse_kinematics_batch(m, link, joints, dev(tg), dev(q0), with_rot=True, iters=40, sscc=sscc, sdf=sdf,
                                                margin=MARGIN, self_margin=MARGIN, restarts=2, return_dmin=True)
    clear_b = (dmin >= MARGIN - 1e-3).cpu().numpy()
    clear_s = (sd >= MARGIN - 1e-3).cpu().numpy()
    reached = (_pose_err(m, joints, link, q, tg) < 1e-3).cpu().numpy()
    print("dual-arm IK under boxes + pairs: reached %.1f %% / boxes clear %.1f %% / pairs clear %.1f %% / all %.1f %%"
          % (100 * reached.mean(), 100 * clear_b.mean(), 100 * clear_s.mean(), 100 * (reached & clear_b & clear_s).mean()))
    assert clear_b.mean() > 0.97 and clear_s.mean() > 0.97
    qn, dn, sdn = q.cpu().numpy(), dmin.cpu().numpy(), sd.cpu().numpy()
    for n in range(0, N, 101):
        R.set_joint_angles(mo, jo, qn[n])
        np.testing.assert_allclose(dn[n], R.compute_coll_dists(so, jo, sdf_o).min(), rtol=1e-10, atol=1e-12)
        _, _, raw = SR.self_coll_dists_and_grads(so, jo, pairs)
        np.testing.assert_allclose(sdn[n], raw.min(), rtol=1e-10, atol=1e-12)


def _fetch_problems(N, seed):
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    pairs = K.self_collision_pairs(sscc, joints, ignore=FETCH_IGNORE)
    qc = scenes.random_configs(jo, 4 * N, False, seed=seed)
    idx = np.nonzero(_self_dmin(m, joints, sscc, qc, pairs) >= 0.05)[0][:N]
    assert idx.size == N
    link = K.find_link(m, "gripper_link")
    tg = _pose_targets(m, joints, link, qc[idx])
    q0 = scenes.random_configs(jo, N, False, seed=seed + 1)
    return m, joints, sscc, mo, jo, so, pairs, link, tg, q0


def _solve(m, link, joints, tg, q0, **kw):
    out = K.ik_solve_device(m, link, joints, dev(tg), dev(q0), iters=40, self_margin=MARGIN, **kw)
    torch.cuda.synchronize()
    return out


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("with_rot", [True, False])
def test_one_solve_from_random_seeds(with_rot):
    """One solve under the pairs alone, from random in-limit seeds, with and without the rotation rows: the
    run-time-sized step kernel (dual arm, 18 columns, default table) and an unrolled one (Fetch, 8 columns, 64 pairs).
    Iterates inside the limits; the reported pair distance and objective are the oracles' at the returned q."""
    m, joints, sscc, _, mo, jo, so, _, link, tg, q0 = _dual_arm_problems(True, 512, 41)
    fm, fj, fs, fmo, fjo, fso, fpairs, flink, ftg, fq0 = _fetch_problems(512, 43)
    runs = (("dual arm", m, joints, sscc, mo, jo, so, link, "l_tool", tg, q0, None),
            ("Fetch", fm, fj, fs, fmo, fjo, fso, flink, "gripper_link", ftg, fq0, fpairs))
    for name, m, joints, sscc, mo, jo, so, link, link_name, tg, q0, pairs in runs:
        out = _solve(m, link, joints, tg, q0, with_rot=with_rot, sscc=sscc, self_pairs=pairs)
        assert len(out) == 4
        q, f, its, sd = out
        assert int(its.max()) > 1
        err = _pose_err(m, joints, link, q, tg, with_rot).cpu().numpy()
        clear = (sd >= MARGIN - 1e-3).cpu().numpy()
        print("%s IK under self-collision, one solve (with_rot=%s): reached %.1f %% / clear %.1f %% / both %.1f %%"
              % (name, with_rot, 100 * (err < 1e-3).mean(), 100 * clear.mean(), 100 * ((err < 1e-3) & clear).mean()))
        # first B200 run: 93.2 - 97.9 % reached and clear, 99.6 - 100 % clear
        assert clear.mean() > 0.97 and ((err < 1e-3) & clear).mean() > 0.88
        lo, hi = _limits(joints, q0.shape[1])
        qn, fn, sdn = q.cpu().numpy(), f.cpu().numpy(), sd.cpu().numpy()
        assert np.all(qn >= lo - 1e-12) and np.all(qn <= hi + 1e-12)
        pairs_o = K.self_collision_pairs(sscc, joints) if pairs is None else pairs
        link_o = R.find_link(mo, link_name)
        for n in range(0, len(qn), 37):
            R.set_joint_angles(mo, jo, qn[n])
            _, _, raw = SR.self_coll_dists_and_grads(so, jo, pairs_o)
            np.testing.assert_allclose(sdn[n], raw.min(), rtol=1e-10, atol=1e-12)
            fo, _ = R.ik_objective(mo, link_o, jo, qn[n], target_T(tg[n, :3], tg[n, 3:]), with_rot)
            if err[n] < 1e-1:                                # no 2 pi wrap in play
                np.testing.assert_allclose(fn[n], fo, rtol=1e-9, atol=1e-18)


def test_no_compaction_is_bitwise_the_active_list(monkeypatch):
    m, joints, sscc, sdf, _, _, _, _, link, tg, q0 = _dual_arm_problems(True, 4096, 51)
    ref = _solve(m, link, joints, tg, q0, sscc=sscc, with_rot=True)
    monkeypatch.setenv("KIN_IK_NO_COMPACT", "1")
    out = _solve(m, link, joints, tg, q0, sscc=sscc, with_rot=True)
    monkeypatch.delenv("KIN_IK_NO_COMPACT")
    _same(ref, out)
    # the same with the boxes too
    ref = _solve(m, link, joints, tg, q0, sscc=sscc, sdf=sdf, margin=MARGIN, with_rot=True)
    monkeypatch.setenv("KIN_IK_NO_COMPACT", "1")
    out = _solve(m, link, joints, tg, q0, sscc=sscc, sdf=sdf, margin=MARGIN, with_rot=True)
    monkeypatch.delenv("KIN_IK_NO_COMPACT")
    assert len(ref) == 5
    _same(ref, out)


def test_fetch_fridge_and_64_pairs():
    """Fetch with the 64-pair table and the fridge: kin_ik_solve_self with collision = 1 from the pose-only warm start
    keeps both margins; the reported distances are the oracles' at sampled problems."""
    N = 1024
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    sdf, sdf_o = scene_fetch.product_fridge_sdf(), scenes.oracle_fridge_sdf()
    pairs = K.self_collision_pairs(sscc, joints, ignore=FETCH_IGNORE)
    link = K.find_link(m, "gripper_link")
    qc = scenes.random_configs(jo, 40 * N, False, seed=61)
    K.set_joint_angles(m, joints, dev(qc))
    db = K.compute_coll_dists(sscc, joints, sdf).amin(dim=1).cpu().numpy()
    ds = _self_dmin(m, joints, sscc, qc, pairs)
    idx = np.nonzero((db >= 0.03) & (ds >= 0.03))[0][:N]
    assert idx.size == N
    tg = _pose_targets(m, joints, link, qc[idx])
    q0 = np.tile(np.array([0.2, 0, 0, 0, 0.5, 0, 0.5, 0]), (N, 1))
    q_free, _ = K.inverse_kinematics_batch(m, link, joints, dev(tg), dev(q0), with_rot=True, iters=40)
    q, f, its, dmin, sd = K.ik_solve_device(m, link, joints, dev(tg), q_free, with_rot=True, iters=60, sscc=sscc, sdf=sdf,
                                            margin=MARGIN, self_margin=MARGIN, self_pairs=pairs)
    reached = (_pose_err(m, joints, link, q, tg) < 1e-3).cpu().numpy()
    clear = ((dmin >= MARGIN - 1e-3) & (sd >= MARGIN - 1e-3)).cpu().numpy()
    print("Fetch + fridge + 64 pairs, one seed: reached %.1f %% / both margins kept %.1f %% / both %.1f %% (mean %.1f iterations)"
          % (100 * reached.mean(), 100 * clear.mean(), 100 * (reached & clear).mean(), float(its.double().mean())))
    assert clear.mean() > 0.97
    qn, dn, sdn = q.cpu().numpy(), dmin.cpu().numpy(), sd.cpu().numpy()
    for n in range(0, N, 97):
        R.set_joint_angles(mo, jo, qn[n])
        np.testing.assert_allclose(dn[n], R.compute_coll_dists(so, jo, sdf_o).min(), rtol=1e-10, atol=1e-12)
        _, _, raw = SR.self_coll_dists_and_grads(so, jo, pairs)
        np.testing.assert_allclose(sdn[n], raw.min(), rtol=1e-10, atol=1e-12)


def test_single_problem_slsqp_matches_the_oracle_driven_solver():
    """inverse_kinematics(..., self_margin=0.02) on the dual-arm model against the same scipy SLSQP driven by the oracle
    and tests/self_collision_ref.py (the pattern of test_inverse_kinematics_dual_arm_as_the_pr2_test)."""
    from scipy.optimize import minimize
    m, joints, sscc, _ = DA.product(False)
    mo, jo, so, sdf_o = DA.oracle(False)
    nd = len(joints)
    link, link_o = K.find_link(m, "l_tool"), R.find_link(mo, "l_tool")
    pairs = K.self_collision_pairs(sscc, joints)
    lo, hi = [j.lower for j in jo], [j.upper for j in jo]
    bounds = [(a if np.isfinite(a) else None, b if np.isfinite(b) else None) for a, b in zip(lo, hi)]

    def self_cons(x):
        R.set_joint_angles(mo, jo, x)
        v, g, _ = SR.self_coll_dists_and_grads(so, jo, pairs, truncation_dist=MARGIN + 0.05, offset=MARGIN)
        return v, g.T

    for trial in (0, 1):
        tgt = _dual_arm_target(mo, jo, so, sdf_o, False, trial)
        K.set_joint_angles(m, joints, np.zeros(nd))
        q, res = K.inverse_kinematics(m, link, joints, K.Transform(tgt), sscc=sscc, with_rot=True, self_margin=MARGIN, ftol=1e-8)
        d = np.asarray(K.compute_self_coll_dists(sscc, joints))
        assert res.success and d.min() >= MARGIN - 1e-5
        x0 = _oracle_ik(mo, jo, link_o, tgt, np.zeros(nd), True).x
        res_o = minimize(lambda x: R.ik_objective(mo, link_o, jo, x, tgt, True), x0, jac=True, method="SLSQP", bounds=bounds,
                         constraints=[{"type": "ineq", "fun": lambda x: self_cons(x)[0], "jac": lambda x: self_cons(x)[1]}],
                         options={"ftol": 1e-8, "maxiter": 200})
        assert res_o.success and res.nit == res_o.nit
        np.testing.assert_allclose(q, res_o.x, atol=1e-6)


def test_errors_launch_nothing():
    """No pair table, a NaN margin, collision = 1 without boxes: each returns its error code and launches nothing."""
    from kinematics_jl_b200.device import device_model
    m, joints, sscc = scenes.product_fetch(False)
    link = K.find_link(m, "gripper_link")
    N = 64
    q0 = torch.zeros((N, 8), dtype=torch.float64, device="cuda")
    K.set_joint_angles(m, joints, q0)
    dm = device_model(m)
    dm.set_spheres(sscc._parents, sscc._centers, sscc.sphere_radii)
    dm.set_boxes(np.zeros((0, 4, 4)), np.zeros((0, 3)))
    tg = torch.zeros((N, 6), dtype=torch.float64, device="cuda")
    q, f = torch.empty_like(q0), torch.empty(N, dtype=torch.float64, device="cuda")
    c = L.KinIkCall()
    c.n, c.link_id, c.with_rot, c.iters, c.ftol = N, link.id, 1, 10, 1e-10
    c.targets, c.q0, c.q_out, c.f_out = tg.data_ptr(), q0.data_ptr(), q.data_ptr(), f.data_ptr()
    lib = K.load_library()
    torch.cuda.synchronize()
    n0 = lib.kin_launch_count()
    dm.set_self_pairs(np.zeros((0, 2), dtype=np.int32))
    assert lib.kin_model_n_self_pairs(dm.h) == 0
    assert lib.kin_ik_solve_self(dm.h, C.byref(c), MARGIN, None) == -1                  # KIN_ERR_INVALID_ARGUMENT
    dm.set_self_pairs(K.self_collision_pairs(sscc, joints, ignore=FETCH_IGNORE))
    assert lib.kin_model_n_self_pairs(dm.h) == 64
    assert lib.kin_ik_solve_self(dm.h, C.byref(c), float("nan"), None) == -1
    c.collision, c.margin = 1, MARGIN
    assert lib.kin_model_n_boxes(dm.h) == 0
    assert lib.kin_ik_solve_self(dm.h, C.byref(c), MARGIN, None) == -1
    assert b"no boxes" in lib.kin_last_error()
    assert lib.kin_launch_count() == n0

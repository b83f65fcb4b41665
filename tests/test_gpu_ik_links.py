"""Multi-link pose targets in the device-resident batched IK (kin_ik_solve_links), on the B200: both tools of the dual-arm
model (generated one-launch kernel and the run-time-sized step kernel, 15 / 18 columns), a mixed rotation / position-only
pair of links on Fetch (unrolled 8-column step kernel).  One link through the new entry point is held to kin_ik_solve /
kin_ik_solve_self bit for bit; objectives and distances to the oracles; the solve without compaction and the staged
generated solve to the default paths bit for bit; the single-problem SLSQP driver to the same scipy SLSQP driven by the
oracle."""
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
from test_gpu_callers import _pose_err, _pose_targets, dev, target_T

pytestmark = pytest.mark.gpu

MARGIN = 0.02
FETCH_IGNORE = [("wrist_flex_link", "elbow_flex_link")]
TOOLS = ("l_tool", "r_tool")


def _limits(joints, nd):
    nb = nd - len(joints)
    return (np.array([j.lower_limit for j in joints] + [-np.inf] * nb), np.array([j.upper_limit for j in joints] + [np.inf] * nb))


def _self_dmin(m, joints, sscc, q, pairs=None):
    K.set_joint_angles(m, joints, q if isinstance(q, torch.Tensor) else dev(q))
    return K.compute_self_coll_summary(sscc, joints, pairs)[0].cpu().numpy()


def _two_tool_problems(with_base, N, seed):
    """Both tool targets from ONE in-limit configuration whose pairs are all >= 0.05 apart (jointly reachable);
    random in-limit seeds."""
    m, joints, sscc, sdf = DA.product(with_base)
    mo, jo, so, sdf_o = DA.oracle(with_base)
    qc = SS.random_q(jo, 4 * N, with_base, seed=seed)
    idx = np.nonzero(_self_dmin(m, joints, sscc, qc) >= 0.05)[0][:N]
    assert idx.size == N
    links = [K.find_link(m, n) for n in TOOLS]
    tg = np.concatenate([_pose_targets(m, joints, l, qc[idx]) for l in links], axis=1)
    q0 = SS.random_q(jo, N, with_base, seed=seed + 1)
    return m, joints, sscc, sdf, mo, jo, so, sdf_o, links, tg, q0


def _reached(m, joints, links, q, tg, with_rots=None):
    with_rots = with_rots or [True] * len(links)
    err = torch.stack([_pose_err(m, joints, l, q, tg[:, 6 * i:6 * i + 6], w)
                       for i, (l, w) in enumerate(zip(links, with_rots))], dim=1).amax(dim=1)
    return err.cpu().numpy()


def _oracle_f(mo, jo, names, q, tg, with_rots):
    f = 0.0
    for i, (nm, w) in enumerate(zip(names, with_rots)):
        fo, _ = R.ik_objective(mo, R.find_link(mo, nm), jo, q, target_T(tg[6 * i:6 * i + 3], tg[6 * i + 3:6 * i + 6]), w)
        f += fo
    return f


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def _fetch_problems(N, seed):
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    qc = scenes.random_configs(jo, N, False, seed=seed)
    links = [K.find_link(m, "gripper_link"), K.find_link(m, "elbow_flex_link")]
    tg = np.concatenate([_pose_targets(m, joints, l, qc) for l in links], axis=1)
    q0 = scenes.random_configs(jo, N, False, seed=seed + 1)
    return m, joints, sscc, mo, jo, so, links, tg, q0


@pytest.mark.parametrize("model", ["fetch", "dual_arm"])
def test_one_link_is_bitwise_the_single_link_calls(model, monkeypatch):
    """kin_ik_solve_links with n_links = 1 against kin_ik_solve (pose only: generated kernel and KIN_DISABLE_JIT;
    collision = 1) and kin_ik_solve_self: q, f, iterations, dmin and self_dmin identical."""
    N = 512
    if model == "fetch":
        m, joints, sscc, mo, jo, so, links, tg, q0 = _fetch_problems(N, 3)
        sdf = scene_fetch.product_fridge_sdf()
        pairs = K.self_collision_pairs(sscc, joints, ignore=FETCH_IGNORE)
        q0 = np.tile(np.array([0.2, 0, 0, 0, 0.5, 0, 0.5, 0]), (N, 1))
    else:
        m, joints, sscc, sdf, _, _, _, _, links, tg, q0 = _two_tool_problems(True, N, 5)
        pairs = None
    link, tg1 = links[0], tg[:, :6]
    for with_rot in (True, False):
        cases = [dict(), dict(jit=False), dict(sscc=sscc, sdf=sdf, margin=MARGIN),
                 dict(sscc=sscc, self_margin=MARGIN, self_pairs=pairs), dict(sscc=sscc, sdf=sdf, margin=MARGIN, self_margin=MARGIN, self_pairs=pairs)]
        for kw in cases:
            kw = dict(kw)
            if kw.pop("jit", True) is False:
                monkeypatch.setenv("KIN_DISABLE_JIT", "1")
            ref = K.ik_solve_device(m, link, joints, dev(tg1), dev(q0), with_rot=with_rot, iters=30, **kw)
            out = K.ik_solve_device(m, [link], joints, dev(tg1), dev(q0), with_rot=[with_rot], iters=30, **kw)
            torch.cuda.synchronize()
            monkeypatch.delenv("KIN_DISABLE_JIT", raising=False)
            assert int(ref[2].max()) > 1
            _same(ref, out)


@pytest.mark.parametrize("with_base", [False, True])
def test_dual_arm_both_tools(with_base):
    N = 2048
    m, joints, sscc, sdf, mo, jo, so, sdf_o, links, tg, q0 = _two_tool_problems(with_base, N, 21)
    nd = q0.shape[1]
    q, f, its = K.ik_solve_device(m, links, joints, dev(tg), dev(q0), with_rot=True, iters=40)
    err = _reached(m, joints, links, q, tg)
    q2, f2 = K.inverse_kinematics_batch(m, links, joints, dev(tg), dev(q0), with_rot=True, iters=40, restarts=2)
    err2 = _reached(m, joints, links, q2, tg)
    print("dual-arm IK, both tools (%d columns): %.1f %% reach both within 1e-3 after one solve, %.1f %% with two restarts, "
          "mean iterations %.1f" % (nd, 100 * (err < 1e-3).mean(), 100 * (err2 < 1e-3).mean(), float(its.double().mean())))
    # first B200 run: 43.6 % / 76.6 % (fixed base), 59.5 % / 91.1 % (planar base); the floors sit a few points below
    assert (err < 1e-3).mean() > (0.53 if with_base else 0.38)
    assert (err2 < 1e-3).mean() > (0.86 if with_base else 0.70)
    lo, hi = _limits(joints, nd)
    for qq in (q, q2):
        qn = qq.cpu().numpy()
        assert np.all(qn >= lo - 1e-12) and np.all(qn <= hi + 1e-12)
    qn, fn = q.cpu().numpy(), f.cpu().numpy()
    for n in range(0, N, 101):
        if err[n] < 1e-1:                                    # no 2 pi wrap in play
            np.testing.assert_allclose(fn[n], _oracle_f(mo, jo, TOOLS, qn[n], tg[n], (True, True)), rtol=1e-9, atol=1e-18)


@pytest.mark.parametrize("with_base", [False, True])
def test_dual_arm_both_tools_self_and_boxes(with_base):
    N = 2048
    m, joints, sscc, sdf, mo, jo, so, sdf_o, links, tg, q0 = _two_tool_problems(with_base, N, 31)
    pairs = K.self_collision_pairs(sscc, joints)
    nd = q0.shape[1]
    lo, hi = _limits(joints, nd)
    q, f, dmin, sd = K.inverse_kinematics_batch(m, links, joints, dev(tg), dev(q0), with_rot=True, iters=40, sscc=sscc,
                                                self_margin=MARGIN, restarts=2, return_dmin=True)
    reached = _reached(m, joints, links, q, tg) < 1e-3
    clear = (sd >= MARGIN - 1e-3).cpu().numpy()
    print("dual-arm IK, both tools + self (%d columns): reached %.1f %% / clear %.1f %% / both %.1f %%"
          % (nd, 100 * reached.mean(), 100 * clear.mean(), 100 * (reached & clear).mean()))
    # first B200 run: 79.9 % (fixed base) and 94.0 % (planar base) reached and clear
    assert clear.mean() > 0.97 and (reached & clear).mean() > (0.88 if with_base else 0.72)
    qn, fn, sdn = q.cpu().numpy(), f.cpu().numpy(), sd.cpu().numpy()
    assert np.all(qn >= lo - 1e-12) and np.all(qn <= hi + 1e-12)
    err = _reached(m, joints, links, q, tg)
    for n in range(0, N, 101):
        R.set_joint_angles(mo, jo, qn[n])
        _, _, raw = SR.self_coll_dists_and_grads(so, jo, pairs)
        np.testing.assert_allclose(sdn[n], raw.min(), rtol=1e-10, atol=1e-12)
        if err[n] < 1e-1:
            np.testing.assert_allclose(fn[n], _oracle_f(mo, jo, TOOLS, qn[n], tg[n], (True, True)), rtol=1e-9, atol=1e-18)
    # ... and the boxes too
    q, f, dmin, sd = K.inverse_kinematics_batch(m, links, joints, dev(tg), dev(q0), with_rot=True, iters=40, sscc=sscc, sdf=sdf,
                                                margin=MARGIN, self_margin=MARGIN, restarts=2, return_dmin=True)
    reached = _reached(m, joints, links, q, tg) < 1e-3
    clear = ((dmin >= MARGIN - 1e-3) & (sd >= MARGIN - 1e-3)).cpu().numpy()
    print("dual-arm IK, both tools + boxes + self (%d columns): reached %.1f %% / clear %.1f %% / both %.1f %%"
          % (nd, 100 * reached.mean(), 100 * clear.mean(), 100 * (reached & clear).mean()))
    # first B200 run: 54.9 % (fixed base) and 80.5 % (planar base) reached and clear
    assert clear.mean() > 0.96 and (reached & clear).mean() > (0.74 if with_base else 0.48)
    qn, dn, sdn = q.cpu().numpy(), dmin.cpu().numpy(), sd.cpu().numpy()
    assert np.all(qn >= lo - 1e-12) and np.all(qn <= hi + 1e-12)
    for n in range(0, N, 101):
        R.set_joint_angles(mo, jo, qn[n])
        np.testing.assert_allclose(dn[n], R.compute_coll_dists(so, jo, sdf_o).min(), rtol=1e-10, atol=1e-12)
        _, _, raw = SR.self_coll_dists_and_grads(so, jo, pairs)
        np.testing.assert_allclose(sdn[n], raw.min(), rtol=1e-10, atol=1e-12)


def test_fetch_gripper_pose_and_elbow_position(monkeypatch):
    """Mixed rotation on Fetch: the gripper with rotation, elbow_flex_link position-only (3 rows).  Generated kernel
    and the loop (KIN_DISABLE_JIT); the objective is the oracle's sum at q."""
    N = 2048
    m, joints, sscc, mo, jo, so, links, tg, q0 = _fetch_problems(N, 71)
    rots = [True, False]
    names = ("gripper_link", "elbow_flex_link")
    outs = [K.ik_solve_device(m, links, joints, dev(tg), dev(q0), with_rot=rots, iters=40)]
    monkeypatch.setenv("KIN_DISABLE_JIT", "1")
    outs.append(K.ik_solve_device(m, links, joints, dev(tg), dev(q0), with_rot=rots, iters=40))
    monkeypatch.delenv("KIN_DISABLE_JIT")
    for q, f, its in outs:
        err = _reached(m, joints, links, q, tg, rots)
        print("Fetch gripper pose + elbow position: %.1f %% within 1e-3, mean iterations %.1f" % (100 * (err < 1e-3).mean(), float(its.double().mean())))
        assert (err < 1e-3).mean() > 0.8                    # first B200 run: 86.2 %
        qn, fn = q.cpu().numpy(), f.cpu().numpy()
        for n in range(0, N, 97):
            if err[n] < 1e-1:
                np.testing.assert_allclose(fn[n], _oracle_f(mo, jo, names, qn[n], tg[n], rots), rtol=1e-9, atol=1e-18)


@pytest.mark.parametrize("with_rot", [True, False])
def test_one_constrained_solve_from_random_seeds(with_rot):
    """One solve from random in-limit seeds through the LINKS step kernels: run-time-sized (dual arm, 18 columns, both
    tools, under the pairs and under the boxes) and unrolled (Fetch, 8 columns, gripper with or without rotation and the
    elbow position-only, under the fridge).  Iterates inside the limits; the reported distances and objectives are the
    oracles' at the returned q."""
    N = 512
    m, joints, sscc, sdf, mo, jo, so, sdf_o, links, tg, q0 = _two_tool_problems(True, N, 41)
    fm, fj, fs, fmo, fjo, fso, flinks, ftg, fq0 = _fetch_problems(N, 43)
    fsdf, fsdf_o = scene_fetch.product_fridge_sdf(), scenes.oracle_fridge_sdf()
    pairs = K.self_collision_pairs(sscc, joints)
    runs = (("dual arm + pairs", m, links, joints, mo, jo, so, None, pairs, TOOLS, tg, q0, [with_rot] * 2,
             dict(sscc=sscc, self_margin=MARGIN)),
            ("dual arm + boxes", m, links, joints, mo, jo, so, sdf_o, None, TOOLS, tg, q0, [with_rot] * 2,
             dict(sscc=sscc, sdf=sdf, margin=MARGIN)),
            ("Fetch + fridge", fm, flinks, fj, fmo, fjo, fso, fsdf_o, None, ("gripper_link", "elbow_flex_link"), ftg, fq0,
             [with_rot, False], dict(sscc=fs, sdf=fsdf, margin=MARGIN)))
    for name, mm, ll, jj, mo_, jo_, so_, sdf_o_, pairs_, names, t, s0, rots, kw in runs:
        q, f, its, d = K.ik_solve_device(mm, ll, jj, dev(t), dev(s0), with_rot=rots, iters=40, **kw)
        torch.cuda.synchronize()
        assert int(its.max()) > 1
        err = _reached(mm, jj, ll, q, t, rots)
        clear = (d >= MARGIN - 1e-3).cpu().numpy()
        print("%s, one solve (with_rot=%s): reached %.1f %% / clear %.1f %% / both %.1f %%"
              % (name, rots, 100 * (err < 1e-3).mean(), 100 * clear.mean(), 100 * ((err < 1e-3) & clear).mean()))
        # first B200 run: 42.0 % (dual arm + boxes, both with rotation) to 86.3 % reached and clear, 92.6 - 99.4 % clear
        assert clear.mean() > 0.9 and ((err < 1e-3) & clear).mean() > 0.36
        lo, hi = _limits(jj, s0.shape[1])
        qn, fn, dn = q.cpu().numpy(), f.cpu().numpy(), d.cpu().numpy()
        assert np.all(qn >= lo - 1e-12) and np.all(qn <= hi + 1e-12)
        for n in range(0, N, 37):
            R.set_joint_angles(mo_, jo_, qn[n])
            if pairs_ is not None:
                _, _, raw = SR.self_coll_dists_and_grads(so_, jo_, pairs_)
                np.testing.assert_allclose(dn[n], raw.min(), rtol=1e-10, atol=1e-12)
            else:
                np.testing.assert_allclose(dn[n], R.compute_coll_dists(so_, jo_, sdf_o_).min(), rtol=1e-10, atol=1e-12)
            if err[n] < 1e-1:                                # no 2 pi wrap in play
                np.testing.assert_allclose(fn[n], _oracle_f(mo_, jo_, names, qn[n], t[n], rots), rtol=1e-9, atol=1e-18)


def test_no_compaction_is_bitwise_the_active_list(monkeypatch):
    m, joints, sscc, sdf, _, _, _, _, links, tg, q0 = _two_tool_problems(True, 4096, 51)
    for kw in (dict(jit=False), dict(sscc=sscc, self_margin=MARGIN), dict(sscc=sscc, sdf=sdf, margin=MARGIN, self_margin=MARGIN)):
        kw = dict(kw)
        if kw.pop("jit", True) is False:
            monkeypatch.setenv("KIN_DISABLE_JIT", "1")
        ref = K.ik_solve_device(m, links, joints, dev(tg), dev(q0), iters=40, **kw)
        monkeypatch.setenv("KIN_IK_NO_COMPACT", "1")
        out = K.ik_solve_device(m, links, joints, dev(tg), dev(q0), iters=40, **kw)
        monkeypatch.delenv("KIN_IK_NO_COMPACT")
        monkeypatch.delenv("KIN_DISABLE_JIT", raising=False)
        torch.cuda.synchronize()
        _same(ref, out)


def test_staged_generated_solve_is_bitwise_the_single_launch(monkeypatch):
    m, joints, _, _, _, _, _, _, links, tg, q0 = _two_tool_problems(True, 16384, 61)
    lib = K.load_library()
    monkeypatch.setenv("KIN_IK_STAGES", "0")
    n0 = lib.kin_launch_count()
    ref = K.ik_solve_device(m, links, joints, dev(tg), dev(q0), iters=40)
    torch.cuda.synchronize()
    assert lib.kin_launch_count() - n0 == 1
    monkeypatch.delenv("KIN_IK_STAGES")
    n0 = lib.kin_launch_count()
    out = K.ik_solve_device(m, links, joints, dev(tg), dev(q0), iters=40)
    torch.cuda.synchronize()
    assert lib.kin_launch_count() - n0 > 1
    _same(ref, out)


def test_single_problem_slsqp_two_tools_matches_the_oracle_driven_solver():
    from scipy.optimize import minimize
    m, joints, _, _ = DA.product(False)
    mo, jo, _, _ = DA.oracle(False)
    nd = len(joints)
    links = [K.find_link(m, n) for n in TOOLS]
    links_o = [R.find_link(mo, n) for n in TOOLS]
    lo, hi = [j.lower for j in jo], [j.upper for j in jo]
    bounds = [(a if np.isfinite(a) else None, b if np.isfinite(b) else None) for a, b in zip(lo, hi)]
    rng = np.random.default_rng(7)
    qt = np.array(lo) + (np.array(hi) - np.array(lo)) * (0.25 + 0.5 * rng.random(nd))
    R.set_joint_angles(mo, jo, qt)
    tgts = [R.get_transform(mo, l).copy() for l in links_o]

    def fo(x):
        f, g = 0.0, np.zeros(nd)
        for l, t in zip(links_o, tgts):
            fi, gi = R.ik_objective(mo, l, jo, x, t, True)
            f, g = f + fi, g + gi
        return f, g

    K.set_joint_angles(m, joints, np.zeros(nd))
    q, res = K.inverse_kinematics(m, links, joints, [K.Transform(t) for t in tgts], with_rot=True, ftol=1e-8)
    res_o = minimize(fo, np.zeros(nd), jac=True, method="SLSQP", bounds=bounds, options={"ftol": 1e-8, "maxiter": 200})
    assert res.success and res_o.success and res.nit == res_o.nit
    np.testing.assert_allclose(q, res_o.x, atol=1e-6)


def test_errors_launch_nothing():
    from kinematics_jl_b200.device import device_model
    m, joints, sscc = scenes.product_fetch(False)
    N = 64
    q0 = torch.zeros((N, 8), dtype=torch.float64, device="cuda")
    K.set_joint_angles(m, joints, q0)
    dm = device_model(m)
    dm.set_spheres(sscc._parents, sscc._centers, sscc.sphere_radii)
    dm.set_boxes(np.zeros((0, 4, 4)), np.zeros((0, 3)))
    tg = torch.zeros((N, 12), dtype=torch.float64, device="cuda")
    q, f = torch.empty_like(q0), torch.empty(N, dtype=torch.float64, device="cuda")
    c = L.KinIkCall()
    c.n, c.iters, c.ftol = N, 10, 1e-10
    c.targets, c.q0, c.q_out, c.f_out = tg.data_ptr(), q0.data_ptr(), q.data_ptr(), f.data_ptr()
    lib = K.load_library()
    ip = C.POINTER(C.c_int32)
    g, e = K.find_link(m, "gripper_link").id, K.find_link(m, "elbow_flex_link").id

    def call(ids, rots=None, n_links=None, self_collision=0, self_margin=MARGIN):
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        rots = np.ones(max(len(ids), 1), dtype=np.int32) if rots is None else rots
        return lib.kin_ik_solve_links(dm.h, C.byref(c), len(ids) if n_links is None else n_links,
                                      ids.ctypes.data_as(ip) if len(ids) else None, rots.ctypes.data_as(ip),
                                      self_collision, self_margin, None)

    torch.cuda.synchronize()
    n0 = lib.kin_launch_count()
    assert call([g, e], n_links=0) == -1
    assert call([g, e, 1, 2, 3]) == -1                                   # more than KIN_IK_MAX_LINKS
    assert call([]) == -1
    assert lib.kin_ik_solve_links(dm.h, C.byref(c), 2, np.array([g, e], dtype=np.int32).ctypes.data_as(ip), None, 0, 0.0, None) == -1
    assert call([g, 0]) == -1 and call([g, 10000]) == -1                 # out of range
    assert call([g, g]) == -1                                            # repeated
    assert call([g, e], self_collision=1, self_margin=float("nan")) == -1
    dm.set_self_pairs(np.zeros((0, 2), dtype=np.int32))
    assert call([g, e], self_collision=1) == -1                          # no pair table
    c.collision, c.margin = 1, MARGIN
    assert call([g, e]) == -1                                            # collision without boxes
    assert b"no boxes" in lib.kin_last_error()
    assert lib.kin_launch_count() == n0

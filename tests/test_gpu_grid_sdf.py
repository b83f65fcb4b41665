"""GPU tests of the voxel-grid SDF rows (KIN_PRIM_GRID, extension): point queries on a union of a grid, a box and a
sphere against the restatement of tests/grid_sdf_ref.py; Fetch's 16 spheres against the fridge rasterised with
GridSDF.from_sdf through compute_coll_dists_and_grads, in every layout and kernel; the grid against the boxes it was
sampled from; the collision-constrained batched IK into the rasterised fridge; in-place updates; the model's own
reference to a grid; and the error paths of the C ABI."""
import ctypes as C

import numpy as np
import pytest
import torch

import kinematics_jl_b200 as K
from kinematics_jl_b200 import lib as L
from kinematics_jl_b200.device import current_q, device_model, evaluate
from oracle import ref_model as R
from grid_sdf_ref import RefGrid, RefScene
from test_gpu_parity import dev, host
from test_primitives_cpu import _pose, _rot
import scene_fetch
import scenes

pytestmark = pytest.mark.gpu

S_FRIDGE = 0.02
GRID_POSE = _pose([0.6, 0.0, 0.9])
GRID_SHAPE = (121, 121, 121)          # 2.4 m cubed at 2 cm: Fetch's reach and the whole fridge


def _jit_compiles():
    v = [C.c_int64() for _ in range(4)]
    L.check(L.lib().kin_jit_stats(*[C.byref(x) for x in v]))
    return v[0].value + v[1].value


# ---------------------------------------------------------------------------------------------------------------------
# 1. points: a grid, a box and a sphere in one union
# ---------------------------------------------------------------------------------------------------------------------
def _union():
    rng = np.random.default_rng(11)
    gpose = _pose([0.5, 0.1, 0.4], _rot([1, -1, 2], 0.6))
    vals = (rng.normal(size=(9, 8, 7)) * 0.1 + 0.05).astype(np.float32)
    grid = K.GridSDF(vals, 0.1, K.Transform(gpose))
    bpose, bw = _pose([0.9, -0.2, 0.5], _rot([0, 1, 1], 0.3)), [0.3, 0.25, 0.4]
    spose, r = _pose([0.3, -0.3, 0.8]), 0.15
    sdf = K.UnionSDF([K.BoxSDF(K.Transform(bpose), bw), grid, K.SphereSDF(K.Transform(spose), r)])
    ref = RefScene([(bpose, bw, 0), RefGrid(vals, 0.1, gpose), (spose, [r, 0, 0], 1)])
    return sdf, ref, grid, RefGrid(vals, 0.1, gpose)


def _special_points(g):
    """On samples, on cell faces, on the grid box faces, far outside, deep inside the grid box."""
    pts = []
    Rm, t = g.pose[:3, :3], g.pose[:3, 3]
    half = (g.n - 1) / 2.0 * g.s
    P = g.sample_points()
    pts += [P[0, 0, 0], P[-1, -1, -1], P[3, 4, 2], P[8, 0, 6]]
    for ax in range(3):
        l = np.array([0.013, -0.027, 0.031])
        l[ax] = (2 - (g.n[ax] - 1) / 2.0) * g.s                         # a cell face
        pts.append(Rm @ l + t)
        l = np.array([0.013, -0.027, 0.031])
        l[ax] = half[ax]                                                # a face of the grid box
        pts.append(Rm @ l + t)
    pts += [Rm @ np.array([40.0, -25.0, 30.0]) + t, Rm @ np.array([0.02, 0.01, -0.03]) + t]
    return np.array(pts)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_grid_points_vs_reference(dtype):
    sdf, ref, grid, rg = _union()
    rng = np.random.default_rng(12)
    pts = np.array([0.55, 0.0, 0.5]) + (rng.random((3000, 3)) - 0.5) * 1.6
    pts = np.concatenate([pts, _special_points(rg)])
    P = dev(pts, dtype)
    vals, am = sdf(P, return_argmin=True)
    g_fd, g_an = sdf.gradient(P), sdf.gradient(P, grad_mode=K.GRAD_ANALYTIC)
    g_fdd = sdf.gradient(P, grad_mode=K.GRAD_FD_DIRECT)
    n = len(pts)
    v_ref, am_ref, gf_ref, ga_ref = np.zeros(n), np.zeros(n, dtype=np.int32), np.zeros((n, 3)), np.zeros((n, 3))
    for i, p in enumerate(pts):
        v_ref[i], am_ref[i], gf_ref[i] = ref.eval(p, 0)
        ga_ref[i] = ref.eval(p, 1)[2]
    assert set(am_ref) == {1, 2, 3} and (am_ref == 2).sum() > 500
    assert (v_ref[am_ref == 2] < 0).sum() > 50                           # the grid wins inside and outside
    if dtype == torch.float64:
        np.testing.assert_allclose(host(vals), v_ref, rtol=1e-12, atol=1e-14)
        assert np.array_equal(am.cpu().numpy(), am_ref)
        np.testing.assert_allclose(host(g_an), ga_ref, rtol=1e-11, atol=1e-11)
        np.testing.assert_allclose(host(g_fd), gf_ref, rtol=0, atol=1e-7)
        general = torch.as_tensor(am_ref != 1, device="cuda")            # a grid / sphere row has one FD; the box row
        assert torch.equal(g_fd[general], g_fdd[general])                # takes the closed-form quotient with GRAD_FD
    else:
        np.testing.assert_allclose(host(vals), v_ref, rtol=0, atol=1e-5)
        same = am.cpu().numpy() == am_ref
        assert same.mean() > 0.995
        u = np.array([rg.local(p) / rg.s + (rg.n - 1) / 2.0 for p in pts])
        away = np.min(np.abs(u - np.round(u)), axis=1) > 1e-3             # float rounding may pick the neighbouring cell
        on_grid = same & (am_ref == 2) & away
        np.testing.assert_allclose(host(g_an)[on_grid], ga_ref[on_grid], rtol=0, atol=2e-3)


# ---------------------------------------------------------------------------------------------------------------------
# 2.-4. Fetch against the rasterised fridge
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def fridge_grid():
    boxes = scene_fetch.product_fridge_sdf()
    grid = K.GridSDF.from_sdf(boxes, K.Transform(GRID_POSE), GRID_SHAPE, S_FRIDGE)
    # the same samples through numpy: what from_sdf stored, for the restatement and for a second handle
    ax = [(np.arange(n) - (n - 1) / 2.0) * S_FRIDGE for n in GRID_SHAPE]
    Lp = np.stack(np.meshgrid(*ax, indexing="ij"), axis=-1).reshape(-1, 3) + GRID_POSE[:3, 3]
    vals = host(boxes(dev(Lp))).reshape(GRID_SHAPE).astype(np.float32)
    return boxes, grid, vals


def _ref_collision(mo, jo, so, rg, q, truncation, grad_mode, scratch):
    """collision.jl:67-94 with the sphere centres / Jacobians of the oracle and the grid restatement."""
    S, nd = len(so.sphere_links), len(jo)
    vals, grads, am = np.zeros((len(q), S)), np.zeros((len(q), nd, S)), np.ones((len(q), S), dtype=np.int32)
    for n, qn in enumerate(q):
        R.set_joint_angles(mo, jo, qn)
        mat = np.zeros(3 * nd)
        for s, (link, r) in enumerate(zip(so.sphere_links, so.sphere_radii)):
            c = R.get_transform(mo, link)[:3, 3]
            d = rg(c)
            vals[n, s] = d - r
            if d - r > truncation:
                vals[n, s] = truncation
                continue
            if scratch == K.SCRATCH_CLEAN:
                mat[:] = 0.0
            R.get_jacobian_inplace(mo, link, jo, False, mat)
            J = mat.reshape(nd, 3).T
            grads[n, :, s] = J.T @ rg.gradient(c, analytic=grad_mode == K.GRAD_ANALYTIC, f=d)
    return vals, grads, am


def test_from_sdf_stores_the_samples_of_the_boxes(fridge_grid):
    boxes, grid, vals = fridge_grid
    twin = K.GridSDF(vals, S_FRIDGE, K.Transform(GRID_POSE))
    rng = np.random.default_rng(13)
    pts = dev(GRID_POSE[:3, 3] + (rng.random((20000, 3)) - 0.5) * 2.6)
    assert torch.equal(grid(pts), twin(pts))


@pytest.mark.parametrize("layout", ["aos", "soa"])
@pytest.mark.parametrize("truncation", [np.inf, 0.08])
def test_fetch_spheres_against_the_rasterised_fridge_vs_reference(fridge_grid, layout, truncation):
    boxes, grid, vals = fridge_grid
    rg = RefGrid(vals, S_FRIDGE, GRID_POSE)
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    q = scenes.random_configs(jo, 150, False, seed=44, zeros_every=50)
    Q = dev(q)
    K.set_joint_angles(m, joints, Q.t().contiguous().t() if layout == "soa" else Q)
    for scratch in (K.SCRATCH_REFERENCE, K.SCRATCH_CLEAN):
        for gm, tol in ((K.GRAD_FD, 1e-7), (K.GRAD_ANALYTIC, 1e-10)):
            v, g, am = K.compute_coll_dists_and_grads(sscc, joints, grid, truncation_dist=truncation, grad_mode=gm,
                                                      scratch_mode=scratch, return_argmin=True)
            v_ref, g_ref, am_ref = _ref_collision(mo, jo, so, rg, q, truncation, gm, scratch)
            np.testing.assert_allclose(host(v), v_ref, rtol=1e-12, atol=1e-13)
            assert np.array_equal(am.cpu().numpy(), am_ref)
            assert np.array_equal(host(v) == truncation, v_ref == truncation)
            np.testing.assert_allclose(host(g), g_ref, rtol=0, atol=tol)
    if np.isinf(truncation):
        assert (v_ref < 0.05).mean() > 0.01                        # the spheres do reach the fridge


@pytest.mark.parametrize("layout", [L.SOA, L.TILED32, L.AOS])
def test_every_kernel_agrees_bitwise_on_a_grid(fridge_grid, layout, monkeypatch):
    """Interpreting kernel, model-specialised kernel and one-warp-per-configuration kernel, a table of grid + boxes."""
    boxes, grid, vals = fridge_grid
    sdf = K.UnionSDF([grid, boxes])
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    gl = K.find_link(m, "gripper_link").id

    def run(n, mode, warp_max=None, **kw):
        for k in ("KIN_DISABLE_JIT", "KIN_FORCE_JIT", "KIN_JIT_WARP_MAX"):
            monkeypatch.delenv(k, raising=False)
        if mode:
            monkeypatch.setenv(mode, "1")
        if warp_max is not None:
            monkeypatch.setenv("KIN_JIT_WARP_MAX", str(warp_max))
        q = scenes.random_configs(jo, n, False, seed=45, zeros_every=50)
        K.set_joint_angles(m, joints, dev(q))
        K.compute_coll_dists(sscc, joints, sdf)
        Qc, ql, N = current_q(m)
        o = evaluate(device_model(m), Qc, ql, N, layout=layout, fk_links=[gl], jac_links=[gl], collision=True, want_argmin=True,
                     launch_info=True, **kw)
        torch.cuda.synchronize()
        return q, o

    for kw in (dict(truncation_dist=np.inf, grad_mode=L.GRAD_FD, scratch_mode=L.SCRATCH_REFERENCE),
               dict(truncation_dist=0.08, grad_mode=L.GRAD_ANALYTIC, scratch_mode=L.SCRATCH_CLEAN, vals_offset=0.03)):
        q, a = run(40013, "KIN_DISABLE_JIT", **kw)
        _, b = run(40013, None, **kw)
        assert a["launch"]["block"] > 0 and b["launch"]["block"] < 0, L.lib().kin_jit_status()
        for key in ("T", "J", "vals", "grads", "argmin"):
            assert torch.equal(a[key], b[key]), (key, kw)
        _, c = run(77, "KIN_DISABLE_JIT", **kw)
        _, d = run(77, "KIN_FORCE_JIT", **kw)
        _, e = run(77, "KIN_FORCE_JIT", warp_max=2048, **kw)
        for key in ("T", "J", "vals", "grads", "argmin"):
            assert torch.equal(c[key], d[key]) and torch.equal(c[key], e[key]), (key, kw)
    am = b["argmin"].cpu().numpy()
    assert (am == 1).any() and (am > 1).any()


def test_grid_is_within_sqrt3_s_of_the_boxes_it_samples(fridge_grid):
    """A union of box SDFs is 1-Lipschitz and every corner of a cell is within sqrt(3) s of a point in it."""
    boxes, grid, vals = fridge_grid
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    q = dev(scenes.random_configs(jo, 20000, False, seed=46))
    K.set_joint_angles(m, joints, q)
    dg = host(K.compute_coll_dists(sscc, joints, grid))
    db = host(K.compute_coll_dists(sscc, joints, boxes))
    assert np.max(np.abs(dg - db)) <= np.sqrt(3) * S_FRIDGE + 1e-6
    assert np.max(np.abs(dg - db)) > 0


def test_collision_constrained_ik_into_the_rasterised_fridge(fridge_grid):
    boxes, grid, vals = fridge_grid
    m, joints, sscc = scenes.product_fetch(False)
    link = K.find_link(m, "gripper_link")
    N, margin, ctol = 1024, 0.02, 1e-6
    rng = np.random.default_rng(7)
    tg = np.zeros((N, 6))
    tg[:, 0], tg[:, 1], tg[:, 2] = rng.uniform(0.75, 1.0, N), rng.uniform(-0.15, 0.15, N), rng.uniform(1.12, 1.35, N)
    q0 = np.tile(np.array([0.2, 0, 0, 0, 0.5, 0, 0.5, 0]), (N, 1))
    q, f, dmin = K.inverse_kinematics_batch(m, link, joints, dev(tg), dev(q0), with_rot=True, iters=40, sscc=sscc, sdf=grid,
                                            margin=margin, ctol=ctol, restarts=2, return_dmin=True)
    K.set_joint_angles(m, joints, q)
    p = K.compute_coll_dists(sscc, joints, boxes)
    solved = (host(f) < 1e-6) & (host(dmin) >= margin - ctol)
    print("IK into the rasterised fridge: %.1f %% solved" % (100 * solved.mean()))
    assert solved.sum() > 0
    assert np.all(host(dmin)[solved] >= margin - ctol)
    assert np.all(host(p).min(axis=1)[solved] >= margin - ctol - np.sqrt(3) * S_FRIDGE)
    np.testing.assert_allclose(host(K.compute_coll_dists(sscc, joints, grid)).min(axis=1), host(dmin), rtol=0, atol=1e-12)


# ---------------------------------------------------------------------------------------------------------------------
# 5.-7. updates, lifetime, errors
# ---------------------------------------------------------------------------------------------------------------------
def test_update_changes_results_without_a_compile():
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    rng = np.random.default_rng(8)
    v0 = (rng.normal(size=(20, 20, 20)) * 0.2 + 0.3).astype(np.float32)
    grid = K.GridSDF(v0, 0.1, K.Transform(_pose([0.6, 0.0, 0.9])))
    q = dev(scenes.random_configs(jo, 1 << 16, False, seed=47))
    K.set_joint_angles(m, joints, q)
    a = K.compute_coll_dists(sscc, joints, grid).clone()
    before = _jit_compiles()
    grid.update(v0 + np.float32(0.25))                                   # a constant shift: every inside value moves
    b = K.compute_coll_dists(sscc, joints, grid).clone()
    grid.update(dev(v0.astype(np.float64) - 0.5))                        # from a CUDA tensor
    c = K.compute_coll_dists(sscc, joints, grid)
    torch.cuda.synchronize()
    assert _jit_compiles() == before
    rg = RefGrid(v0 + np.float32(0.25), 0.1, _pose([0.6, 0.0, 0.9]))
    R.set_joint_angles(mo, jo, host(q[5]))
    for s, (link, r) in enumerate(zip(so.sphere_links, so.sphere_radii)):
        assert abs(float(b[5, s]) - (rg(R.get_transform(mo, link)[:3, 3]) - r)) < 1e-12
    assert not torch.equal(a, b) and not torch.equal(b, c)


def test_a_grid_the_caller_destroyed_still_evaluates_in_its_model():
    m, joints, sscc = scenes.product_fetch(False)
    mo, jo, so = scenes.oracle_fetch(False)
    rng = np.random.default_rng(9)
    v0 = (rng.normal(size=(16, 16, 16)) * 0.2).astype(np.float32)
    grid = K.GridSDF(v0, 0.12, K.Transform(_pose([0.5, 0.0, 0.8])))
    q = dev(scenes.random_configs(jo, 4096, False, seed=48))
    K.set_joint_angles(m, joints, q)
    a = K.compute_coll_dists(sscc, joints, grid).clone()
    dm = device_model(m)
    L.check(L.lib().kin_grid_destroy(grid.h))                            # the caller's reference goes ...
    grid.h = None
    junk = torch.full((1 << 22,), 7.0, device="cuda")                    # ... and the allocator gets busy meanwhile
    Qc, ql, N = current_q(m)
    b = evaluate(dm, Qc, ql, N, collision=True, with_grads=False)["vals"]
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    del junk


def test_error_paths_are_reported_before_anything_changes():
    lib = L.lib()
    h = C.c_void_p()
    v = np.zeros((4, 4, 4), dtype=np.float32)
    vp = v.ctypes.data
    assert lib.kin_grid_create(1, 4, 4, 0.1, vp, C.byref(h)) == -1
    assert lib.kin_grid_create(4, 4, 4, 0.0, vp, C.byref(h)) == -1
    assert lib.kin_grid_create(4, 4, 4, -0.1, vp, C.byref(h)) == -1
    assert lib.kin_grid_create(4, 4, 4, float("nan"), vp, C.byref(h)) == -1
    assert lib.kin_grid_create(4, 4, 4, float("inf"), vp, C.byref(h)) == -1
    assert lib.kin_grid_create(4, 4, 4, 0.1, None, C.byref(h)) == -1
    assert lib.kin_grid_create(1 << 10, 1 << 10, 1 << 9, 0.1, vp, C.byref(h)) == -3
    assert not h.value
    grid = K.GridSDF(v, 0.1)
    m, joints, sscc = scenes.product_fetch(False)
    box = K.BoxSDF(K.Transform(_pose([0.9, 0, 0.5])), [0.3, 0.3, 0.3])
    K.set_joint_angles(m, joints, dev(np.zeros((1, 8))))
    d0 = K.compute_coll_dists(sscc, joints, box)
    dm = device_model(m)
    pose = np.ascontiguousarray(np.eye(4).reshape(1, 16))
    size = np.zeros((1, 3))
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    for kind, handles in ((L.PRIM_GRID, [None]), (L.PRIM_BOX, [grid]), (L.PRIM_SPHERE, [grid])):
        kinds = np.array([kind], dtype=np.int32)
        arr = (C.c_void_p * 1)(*[g.h.value if g is not None else None for g in handles])
        assert lib.kin_model_set_scene(dm.h, 1, kinds.ctypes.data_as(ip), pose.ctypes.data_as(dp), size.ctypes.data_as(dp), arr) == -1
    kinds = np.array([L.PRIM_GRID], dtype=np.int32)
    assert lib.kin_model_set_primitives(dm.h, 1, kinds.ctypes.data_as(ip), pose.ctypes.data_as(dp), size.ctypes.data_as(dp)) == -1
    assert lib.kin_grid_set_values(None, vp, None) == -1 and lib.kin_grid_set_values(grid.h, None, None) == -1
    # the model kept its box: a failed call leaves it unchanged
    Qc, ql, N = current_q(m)
    after = host(evaluate(dm, Qc, ql, N, collision=True, with_grads=False)["vals"]).reshape(-1)
    assert np.array_equal(after, (host(d0) if torch.is_tensor(d0) else np.asarray(d0)).reshape(-1))
    if torch.cuda.device_count() > 1:                                    # a grid of another device
        with torch.cuda.device(1):
            other = K.GridSDF(v, 0.1)
        arr = (C.c_void_p * 1)(other.h.value)
        assert lib.kin_model_set_scene(dm.h, 1, kinds.ctypes.data_as(ip), pose.ctypes.data_as(dp), size.ctypes.data_as(dp), arr) == -1

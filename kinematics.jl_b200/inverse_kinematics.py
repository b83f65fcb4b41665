"""The per-iteration evaluations of the reference's IK driver (inverse_kinematics.jl:38-50) on the B200 backend,
batched over independent problems; the device-resident batched solvers built on them (pose only: one kernel launch, a few staged launches over the still-running problems for large batches;
collision constrained: one fused evaluation + one step kernel per iteration); and the reference's own single-problem
driver with SLSQP (scipy's, the reference's SCIPY back-end; NLopt is third party and not installed)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import lib as _lib
from .algorithm import _check_joints
from .device import current_q, device_model
from .mechanism import Mechanism, set_joint_angles
from .transform import Transform, rpy, translation


def _targets_tensor(targets, N, dtype, device):
    """targets: one entry per link -- a Transform (shared by the batch), a 6-vector, or an (N, 6) array / tensor of
    [x, y, z, roll, pitch, yaw].  -> (tensor (6 nl,) or (N, 6 nl), per_config flag)"""
    import torch
    cols, per = [], 0
    for target in targets:
        if isinstance(target, Transform):
            t = torch.tensor(np.concatenate([translation(target), rpy(target)]), dtype=dtype, device=device)
        else:
            t = target if isinstance(target, torch.Tensor) else torch.as_tensor(np.asarray(target, dtype=np.float64))
            t = t.to(device=device, dtype=dtype)
        if t.dim() == 2:
            assert t.shape == (N, 6), "targets must be (N, 6): x, y, z, roll, pitch, yaw"
            per = 1
        cols.append(t)
    if per:
        cols = [t if t.dim() == 2 else t[None, :].expand(N, 6) for t in cols]
        return torch.cat(cols, dim=1).contiguous(), 1
    return torch.cat(cols).contiguous(), 0


def _pose_residual(m: Mechanism, links, joints, targets, with_rots, mode):
    """All (link, target, with_rot) triples in ONE kin_pose_residual_multi call (two kernel launches)."""
    import torch
    _check_joints(m, joints)
    dm = device_model(m)
    Q, layout, N = current_q(m)
    nl, nd = len(links), dm.n_dof
    n_cons = sum(6 if w else 3 for w in with_rots)
    tg, per = _targets_tensor(targets, N, Q.dtype, Q.device)
    if per:   # bring the targets to the layout of q
        tg = tg.t().contiguous().t() if layout == _lib.SOA else tg.contiguous()
    soa = layout == _lib.SOA
    if mode == _lib.POSE_IK_OBJECTIVE:
        val = torch.empty(N, dtype=Q.dtype, device=Q.device)
        jac = torch.empty((nd, N) if soa else (N, nd), dtype=Q.dtype, device=Q.device)
        jac_view = jac.t() if soa else jac
    else:
        val = torch.empty((n_cons, N) if soa else (N, n_cons), dtype=Q.dtype, device=Q.device)
        jac = torch.empty((n_cons, nd, N) if soa else (N, n_cons, nd), dtype=Q.dtype, device=Q.device)
        jac_view = jac.permute(2, 1, 0) if soa else jac.permute(0, 2, 1)          # (N, n_dof, n_cons)
        val = val.t() if soa else val
    ids = np.ascontiguousarray([l.id for l in links], dtype=np.int32)
    rots = np.ascontiguousarray([1 if w else 0 for w in with_rots], dtype=np.int32)
    ip = C.POINTER(C.c_int32)
    _lib.check(_lib.lib().kin_pose_residual_multi(
        dm.h, _lib.F32 if Q.dtype == torch.float32 else _lib.F64, layout, Q.data_ptr(), N, nl, ids.ctypes.data_as(ip),
        rots.ctypes.data_as(ip), tg.data_ptr(), per, mode, val.data_ptr(), jac.data_ptr(),
        torch.cuda.current_stream(Q.device).cuda_stream))
    return val, jac_view


def ik_objective(m: Mechanism, link, joints, target_pose, with_rot=True):
    """``f_objective`` of inverse_kinematics.jl:38-50 at the configuration(s) of the last set_joint_angles:
    f = sum(pose_diff^2), grad = -2 J' pose_diff with the Euler-rate Jacobian.
    single -> (float, ndarray (n_dof,)); batch -> tensors (N,), (N, n_dof)."""
    f, g = _pose_residual(m, [link], joints, [target_pose], [with_rot], _lib.POSE_IK_OBJECTIVE)
    if m._single:
        return float(f[0]), g[0].double().cpu().numpy()
    return f, g


MAX_LINKS = 4      # KIN_IK_MAX_LINKS


def _link_list(link, with_rot, what):
    """``link``: one Link (-> None: the single-link calls) or a list of links (extension, ``kin_ik_solve_links``) with
    ``with_rot`` a bool or one bool per link -> (links, with_rots).  Checked before anything touches a device."""
    if not isinstance(link, (list, tuple)):
        return None
    links = list(link)
    if not 1 <= len(links) <= MAX_LINKS:
        raise ValueError("%s: 1..%d links, got %d" % (what, MAX_LINKS, len(links)))
    if len({id(l) for l in links}) != len(links) or len({getattr(l, "id", None) for l in links}) != len(links):
        raise ValueError("%s: the links must be distinct" % what)
    rots = list(with_rot) if isinstance(with_rot, (list, tuple)) else [with_rot] * len(links)
    if len(rots) != len(links):
        raise ValueError("%s: %d links but %d with_rot flags" % (what, len(links), len(rots)))
    return links, [bool(w) for w in rots]


def ik_solve_device(m: Mechanism, link, joints, targets, q0, with_rot=True, iters=100, ftol=1e-10, lambda0=1e-2,
                    sscc=None, sdf=None, margin=0.02, coll_weight=100.0, ctol=1e-6, self_margin=None, self_pairs=None):
    """The device-resident batched solve (``kin_ik_solve``).  ``targets`` (N, 6), ``q0`` (N, n_dof) CUDA tensors.

    Without ``sscc`` / ``sdf``: the whole pose-only Levenberg-Marquardt solve in ONE kernel launch around the generated
    FK + Euler-rate Jacobian of ``link`` -> (q (N, n_dof), f (N,), iterations (N,) int32); without the run-time
    compiler the same method runs as one ``kin_eval`` + one step kernel per iteration.

    With ``sscc`` and ``sdf``: the reference's constrained problem (inverse_kinematics.jl:14-19: the same objective
    subject to ``dists - margin >= 0``) from the warm start ``q0``, by an augmented-Lagrangian Levenberg-Marquardt
    iteration that issues one fused ``kin_eval`` and one step kernel per iteration over the still-running problems (active list)
    (csrc/kin_ik_coll.cuh) -> (q, f, iterations, dmin) with dmin (N,) the smallest signed sphere distance at q.

    With ``self_margin`` (extension; ``kin_ik_solve_self``): also ``d_p - self_margin >= 0`` for every self-collision
    pair of the table ``self_pairs`` ((P, 2) 1-based sphere ids, default ``self_collision_pairs(sscc, joints)``), in
    the same loop with one more launch per iteration.  ``sscc`` is required, ``sdf`` optional (without it only the pairs
    constrain the solve).  Returns (q, f, iterations[, dmin], self_dmin), self_dmin (N,) the smallest pair distance at
    q.  On the Fetch sphere fixture the default policy keeps a pair of constant distance that overlaps by 5.5 mm in
    every configuration, which no solver can satisfy: pass ``self_collision_pairs(sscc, joints,
    ignore=[("wrist_flex_link", "elbow_flex_link")])`` (64 pairs) there.

    Several links (extension; ``kin_ik_solve_links``): ``link`` a list of up to 4 distinct links, ``with_rot`` a bool
    or one bool per link, ``targets`` (N, 6 L) with the 6 values of each link in link order; the objective is the sum
    of the links' |e_l|^2 and everything else works as above.  A single Link keeps the single-link calls."""
    import torch
    multi = _link_list(link, with_rot, "ik_solve_device")
    if self_margin is not None:
        if sscc is None:
            raise ValueError("ik_solve_device: self_margin needs the collision checker sscc (its spheres form the pairs)")
        if not np.isfinite(float(self_margin)):
            raise ValueError("ik_solve_device: self_margin must be finite")
    collide = sscc is not None and sdf is not None
    q0 = torch.as_tensor(q0, dtype=torch.float64, device="cuda").contiguous()
    set_joint_angles(m, joints, q0)            # defines the configuration columns (and the device model) as every caller does
    if collide:
        from .collision import _prepare
        _, dm = _prepare(sscc, joints, sdf)
    else:
        dm = device_model(m)
    if self_margin is not None:
        from .collision import _prepare_self
        _, dm = _prepare_self(sscc, joints, self_pairs)
    nb = 3 if m.with_base else 0
    lo = np.ascontiguousarray([j.lower_limit for j in joints] + [-np.inf] * nb, dtype=np.float64)
    hi = np.ascontiguousarray([j.upper_limit for j in joints] + [np.inf] * nb, dtype=np.float64)
    tg = torch.as_tensor(targets, dtype=torch.float64, device="cuda").contiguous()
    N, nd = q0.shape
    assert tg.shape == (N, 6 * (len(multi[0]) if multi else 1)) and nd == dm.n_dof
    q = torch.empty_like(q0)
    f = torch.empty(N, dtype=torch.float64, device="cuda")
    its = torch.empty(N, dtype=torch.int32, device="cuda")
    c = _lib.KinIkCall()
    c.n, c.iters, c.ftol, c.lambda0 = N, int(iters), float(ftol), float(lambda0)
    if not multi:
        c.link_id, c.with_rot = link.id, int(with_rot)
    c.targets, c.q0 = tg.data_ptr(), q0.data_ptr()
    c.lower, c.upper = lo.ctypes.data_as(C.POINTER(C.c_double)), hi.ctypes.data_as(C.POINTER(C.c_double))
    c.q_out, c.f_out, c.iters_out = q.data_ptr(), f.data_ptr(), its.data_ptr()
    c.stream = torch.cuda.current_stream().cuda_stream
    if collide:
        dmin = torch.empty(N, dtype=torch.float64, device="cuda")
        c.collision, c.margin, c.coll_weight, c.ctol, c.dmin_out = 1, float(margin), float(coll_weight), float(ctol), dmin.data_ptr()
    if self_margin is not None:
        c.coll_weight, c.ctol = float(coll_weight), float(ctol)
        self_dmin = torch.empty(N, dtype=torch.float64, device="cuda")
    if multi:
        ids = np.ascontiguousarray([l.id for l in multi[0]], dtype=np.int32)
        rots = np.ascontiguousarray(multi[1], dtype=np.int32)
        ip = C.POINTER(C.c_int32)
        _lib.check(_lib.lib().kin_ik_solve_links(dm.h, C.byref(c), len(ids), ids.ctypes.data_as(ip), rots.ctypes.data_as(ip),
                                                 int(self_margin is not None), float(self_margin or 0.0),
                                                 self_dmin.data_ptr() if self_margin is not None else None))
    elif self_margin is None:
        _lib.check(_lib.lib().kin_ik_solve(dm.h, C.byref(c)))
    else:
        _lib.check(_lib.lib().kin_ik_solve_self(dm.h, C.byref(c), float(self_margin), self_dmin.data_ptr()))
    if self_margin is None:
        return (q, f, its, dmin) if collide else (q, f, its)
    return (q, f, its, dmin, self_dmin) if collide else (q, f, its, self_dmin)


def _seed_limits(m, joints):
    import torch
    nb = 3 if m.with_base else 0
    lo = torch.tensor([j.lower_limit if np.isfinite(j.lower_limit) else -np.pi for j in joints] + [-1.0, -1.0, -np.pi][:nb],
                      device="cuda", dtype=torch.float64)
    hi = torch.tensor([j.upper_limit if np.isfinite(j.upper_limit) else np.pi for j in joints] + [1.0, 1.0, np.pi][:nb],
                      device="cuda", dtype=torch.float64)
    return lo, hi


def inverse_kinematics_batch(m: Mechanism, link, joints, targets, q0, with_rot=True, iters=100, ftol=1e-10,
                             sscc=None, sdf=None, margin=0.02, coll_weight=100.0, use_bistage=True, restarts=0, tol=1e-3, seed=0,
                             coll_iters=60, ctol=1e-6, return_dmin=False, self_margin=None, self_pairs=None):
    """Batched IK for N independent pose targets (config 4 of BASELINE.json) on the reference's objective
    f = |[p - p_t; rpy - rpy_t]|^2 (inverse_kinematics.jl:38-50), iterates clamped to the joint limits (:52-63).

    Without ``sscc`` / ``sdf`` the whole solve is one kernel launch (``ik_solve_device``; large batches: a few stages over
    the still-running problems, same iterates); ``restarts`` > 0 re-solves
    the problems that did not reach ``tol`` (max |pose error|, as test/test_inverse_kinematics.jl:22-23 measures it)
    from random in-limit seeds, that many times -- a local method started from one seed leaves a few per cent of the
    reachable targets in a local minimum at a joint limit.

    With ``sscc`` and ``sdf`` the reference's two-stage driver (inverse_kinematics.jl:1-21) runs on the device for the
    whole batch: the collision-free warm start (``use_bistage``, :8-13) and then the solve under the HARD constraint
    ``dists - margin >= 0`` (IneqConst with margin 0.02, :14-19), an augmented-Lagrangian Levenberg-Marquardt loop of
    at most ``coll_iters`` (fused evaluation, step kernel) launch pairs over the still-running problems (the active list is re-compacted about ten times per solve).  ``restarts``
    re-seeds the problems that end with pose error > ``tol`` or a distance below ``margin - ctol`` (a local method can
    end pressed against the obstacle on the wrong side of it).
    ``self_margin`` (extension, ``kin_ik_solve_self``; needs ``sscc``, ``sdf`` optional): the solve also keeps every
    self-collision pair of ``self_pairs`` (default ``self_collision_pairs(sscc, joints)``) at least ``self_margin``
    apart; the warm start stays pose-only, a problem counts as solved only with its smallest pair distance
    >= ``self_margin - 10 ctol``, and restarts re-seed the others too.  On the Fetch sphere fixture pass
    ``self_collision_pairs(sscc, joints, ignore=[("wrist_flex_link", "elbow_flex_link")])``: the default table keeps a
    pair that overlaps by 5.5 mm in every configuration.
    ``targets`` (N, 6) [x y z roll pitch yaw], ``q0`` (N, n_dof).  Returns (q, f) with f the pose objective
    (and the smallest signed sphere distance per problem with ``return_dmin``; with ``self_margin`` and ``return_dmin``:
    (q, f, dmin or None, self_dmin)).
    Several links (extension, ``kin_ik_solve_links``): ``link`` a list, ``with_rot`` a bool or a per-link list,
    ``targets`` (N, 6 L); f is the sum over the links, and a problem is solved when f <= tol^2 (every residual of
    every link within tol) and the constraints hold."""
    import torch
    multi = _link_list(link, with_rot, "inverse_kinematics_batch")
    selfc = self_margin is not None
    if selfc and sscc is None:
        raise ValueError("inverse_kinematics_batch: self_margin needs the collision checker sscc")
    collide = sscc is not None and sdf is not None
    targets = torch.as_tensor(targets, dtype=torch.float64, device="cuda")
    q0 = torch.as_tensor(q0, dtype=torch.float64, device="cuda")
    if targets.dim() != 2 or targets.shape != (q0.shape[0], 6 * (len(multi[0]) if multi else 1)):
        raise ValueError("inverse_kinematics_batch: targets must be (N, 6 * number of links), got %s" % (tuple(targets.shape),))

    def pose_only(tg, qs):
        return ik_solve_device(m, link, joints, tg, qs, with_rot=with_rot, iters=iters, ftol=ftol)[:2]

    def solve(tg, qs):
        """-> q, f, dmin, self_dmin, good (N,) bool"""
        if not collide and not selfc:
            q, f = pose_only(tg, qs)
            return q, f, None, None, f <= tol * tol
        if use_bistage:
            qs, _ = pose_only(tg, qs)
        out = ik_solve_device(m, link, joints, tg, qs, with_rot=with_rot, iters=coll_iters, ftol=ftol, sscc=sscc,
                              sdf=sdf if collide else None, margin=margin, coll_weight=coll_weight, ctol=ctol,
                              self_margin=self_margin, self_pairs=self_pairs)
        q, f = out[0], out[1]
        dmin = out[3] if collide else None
        sdmin = out[-1] if selfc else None
        # f = sum of squared residuals: max |e| <= tol is implied by f <= tol^2
        good = f <= tol * tol
        if collide:
            good = good & (dmin >= margin - 10 * ctol)
        if selfc:
            good = good & (sdmin >= self_margin - 10 * ctol)
        return q, f, dmin, sdmin, good

    q, f, dmin, sdmin, good = solve(targets, q0)
    if restarts > 0:
        lo, hi = _seed_limits(m, joints)
        gen = torch.Generator(device="cuda").manual_seed(seed)
        for _ in range(restarts):
            bad = torch.nonzero(~good, as_tuple=False).squeeze(1)
            if bad.numel() == 0:
                break
            qs = lo + (hi - lo) * torch.rand((bad.numel(), q.shape[1]), generator=gen, device="cuda", dtype=torch.float64)
            q2, f2, d2, s2, g2 = solve(targets[bad], qs)
            # a restart replaces a failed problem when it succeeds, or (pose only) when it is closer
            better = g2 if (collide or selfc) else (f2 < f[bad])
            q[bad[better]] = q2[better]
            f[bad[better]] = f2[better]
            if collide:
                dmin[bad[better]] = d2[better]
            if selfc:
                sdmin[bad[better]] = s2[better]
            good[bad[better]] = g2[better]
    set_joint_angles(m, joints, q)
    if selfc and return_dmin:
        return q, f, dmin, sdmin
    if collide and return_dmin:
        return q, f, dmin
    return q, f


def inverse_kinematics(m: Mechanism, link, joints, target_pose, sscc=None, sdf=None, use_bistage=True, ftol=1e-5,
                       with_rot=True, margin=0.02, self_margin=None, self_pairs=None):
    """``inverse_kinematics!`` (inverse_kinematics.jl:1-30) for ONE target, driven by SLSQP as in the reference.
    The reference calls NLopt's LD_SLSQP; NLopt is not installed here, scipy's SLSQP (the same Kraft routine, which
    the reference itself uses as its SCIPY back-end in planning.jl:388-394) drives the same callbacks: the objective
    ``f_objective`` (:38-50, ``ik_objective``), the joint-limit bounds (:52-63) and, with ``sscc`` / ``sdf``, the HARD
    inequality constraint ``dists - margin >= 0`` of ``IneqConst(sscc, joints, sdf, 1, 0.02)`` (:14-19) after the
    collision-free warm start (:8-13).  ``self_margin`` (extension): also the self-collision constraint
    ``SelfIneqConst(sscc, joints, 1, self_margin, self_pairs)`` as a second inequality, as ``plan_trajectory`` adds it;
    the warm start stays unconstrained.  Every evaluation runs on the GPU (N = 1).  Returns (q, scipy result); the
    mechanism is left at the solution like the reference leaves it.
    Several links (extension): ``link`` a list of links, ``target_pose`` a list of as many poses (Transform or
    6-vector), ``with_rot`` a bool or one per link; the objective is the sum of the links' f_objective, the stacked
    ``_pose_residual`` of ``kin_pose_residual_multi``."""
    from scipy.optimize import minimize
    from .planning import IneqConst, SelfIneqConst, scipynize
    multi = _link_list(link, with_rot, "inverse_kinematics")
    if multi and (not isinstance(target_pose, (list, tuple)) or len(target_pose) != len(multi[0])):
        raise ValueError("inverse_kinematics: one target pose per link")
    if self_margin is not None and sscc is None:
        raise ValueError("inverse_kinematics: self_margin needs the collision checker sscc")
    nb = 3 if m.with_base else 0
    lo = [j.lower_limit for j in joints] + [-np.inf] * nb
    hi = [j.upper_limit for j in joints] + [np.inf] * nb
    bounds = [(a if np.isfinite(a) else None, b if np.isfinite(b) else None) for a, b in zip(lo, hi)]

    def fun(x):
        set_joint_angles(m, joints, np.asarray(x, dtype=np.float64))
        if multi:
            f, g = _pose_residual(m, multi[0], joints, list(target_pose), multi[1], _lib.POSE_IK_OBJECTIVE)
            return float(f[0]), g[0].double().cpu().numpy()
        return ik_objective(m, link, joints, target_pose, with_rot)

    def solve(x0, constraints):
        return minimize(fun, x0, jac=True, method="SLSQP", bounds=bounds, constraints=constraints,
                        options={"ftol": ftol, "maxiter": 200})

    x0 = np.array([m.angles[j.id - 1] for j in joints] + (list(m.base_pose) if m.with_base else []))
    cons = []
    if sscc is not None and sdf is not None:
        g, dg = scipynize(IneqConst(sscc, joints, sdf, 1, margin))
        cons.append({"type": "ineq", "fun": g, "jac": dg})
    if self_margin is not None:
        gs, dgs = scipynize(SelfIneqConst(sscc, joints, 1, self_margin, self_pairs))
        cons.append({"type": "ineq", "fun": gs, "jac": dgs})
    if not cons:
        res = solve(x0, ())
    else:
        if use_bistage:
            x0 = solve(x0, ()).x
        res = solve(x0, cons)
    set_joint_angles(m, joints, res.x)
    return res.x, res

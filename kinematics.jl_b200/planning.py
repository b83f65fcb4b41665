"""Per-waypoint constraint evaluations of the reference's trajectory planner (planning.jl) on the B200
backend.  Waypoints are independent on this path (planning.jl:59-67), so (problem, waypoint) pairs are
flattened into the batch axis and the block-diagonal constraint Jacobian is stored as its blocks only
(the reference materialises a dense (n_dof n_wp) x (n_coll n_wp) matrix, planning.jl:50,64-65).
The solvers (NLopt SLSQP / Ipopt / scipy, planning.jl:332-401) are third-party and out of scope."""
from __future__ import annotations

import numpy as np

from . import lib as _lib
from .collision import compute_coll_dists_and_grads, compute_self_coll_dists_and_grads, self_collision_pairs
from .mechanism import set_joint_angles


def create_straight_trajectory(q_start, q_goal, n_wp):
    """planning.jl:304-308.  Vectors -> the flat xi (n_dof * n_wp,) of the reference;
    (P, n_dof) tensors -> (P, n_wp, n_dof) on the device of the inputs."""
    import torch
    if isinstance(q_start, torch.Tensor) and q_start.dim() == 2:
        interval = (q_goal - q_start) / (n_wp - 1)
        steps = torch.arange(n_wp, dtype=q_start.dtype, device=q_start.device)
        return q_start[:, None, :] + interval[:, None, :] * steps[None, :, None]
    q_start, q_goal = np.asarray(q_start, dtype=np.float64), np.asarray(q_goal, dtype=np.float64)
    interval = (q_goal - q_start) / (n_wp - 1)
    return np.concatenate([q_start + interval * i for i in range(n_wp)])


class IneqConst:
    """planning.jl:32-68: per-waypoint collision stack, ``val = dists - margin`` with
    ``truncation_dist = margin + 0.05``."""

    def __init__(self, sscc, joints, sdf, n_wp, margin):
        self.sscc, self.joints, self.sdf = sscc, list(joints), sdf
        self.n_wp, self.margin = int(n_wp), float(margin)
        self.n_dof = len(joints) + (3 if sscc.mech.with_base else 0)
        self.n_coll = len(sscc.sphere_links)
        self.n_cons = self.n_coll * self.n_wp

    def __call__(self, xi, grad_mode=_lib.GRAD_FD, scratch_mode=_lib.SCRATCH_REFERENCE):
        """xi: the reference's flat vector (n_dof * n_wp,) -> (val_vec (n_cons,), blocks (n_wp, n_dof, n_coll)) as
        numpy; or a CUDA tensor (P, n_wp, n_dof) of P problems -> tensors (P, n_wp, n_coll), (P, n_wp, n_dof, n_coll)."""
        import torch
        single = not (isinstance(xi, torch.Tensor) and xi.dim() == 3)
        if single:
            X = torch.as_tensor(np.asarray(xi, dtype=np.float64).reshape(1, self.n_wp, self.n_dof), device="cuda")
        else:
            X = xi
        P = X.shape[0]
        set_joint_angles(self.sscc.mech, self.joints, X.reshape(P * self.n_wp, self.n_dof))
        # evaluated in the SoA layout (coalesced stores); the batch-first views below hide the storage order
        vals, grads = compute_coll_dists_and_grads(self.sscc, self.joints, self.sdf, truncation_dist=self.margin + 0.05,
                                                   grad_mode=grad_mode, scratch_mode=scratch_mode, vals_offset=self.margin,
                                                   layout=_lib.SOA)
        vals = vals.reshape(P, self.n_wp, self.n_coll)
        grads = grads.reshape(P, self.n_wp, self.n_dof, self.n_coll)
        if single:
            return vals[0].reshape(-1).cpu().numpy(), grads[0].cpu().numpy()
        return vals, grads

    def evaluate_packed(self, X, slab=None, grad_mode=_lib.GRAD_FD, scratch_mode=_lib.SCRATCH_REFERENCE):
        """X (P, n_wp, n_dof) CUDA tensor -> (slab, vals view (P, n_wp, n_coll), grads view (P, n_wp, n_dof, n_coll)).
        The kernel writes values and Jacobian blocks straight into ONE SoA slab (n_coll + n_coll n_dof, P n_wp)
        [vals rows | grads rows], which ``gather_packed`` hands to a single all-gather."""
        import torch
        from .device import current_q, device_model, evaluate
        from .collision import _prepare
        P, S, nd = X.shape[0], self.n_coll, self.n_dof
        N = P * self.n_wp
        set_joint_angles(self.sscc.mech, self.joints, X.reshape(N, nd))
        m, dm = _prepare(self.sscc, self.joints, self.sdf)
        Q, ql, _ = current_q(m)
        if slab is None:
            slab = torch.empty((S + S * nd, N), dtype=Q.dtype, device=Q.device)
        out = evaluate(dm, Q, ql, N, layout=_lib.SOA, collision=True, with_grads=True, truncation_dist=self.margin + 0.05,
                       grad_mode=grad_mode, scratch_mode=scratch_mode, vals_offset=self.margin,
                       vals_into=slab[:S], grads_into=slab[S:].view(S, nd, N))
        return slab, out["vals"].reshape(P, self.n_wp, S), out["grads"].reshape(P, self.n_wp, nd, S)

    def dense(self, blocks):
        """The reference's dense jac_mat (n_dof n_wp, n_coll n_wp) from the diagonal blocks of one problem."""
        J = np.zeros((self.n_dof * self.n_wp, self.n_cons))
        for i in range(self.n_wp):
            J[i * self.n_dof:(i + 1) * self.n_dof, i * self.n_coll:(i + 1) * self.n_coll] = blocks[i]
        return J


class SelfIneqConst:
    """The self-collision counterpart of ``IneqConst`` (extension): per waypoint ``val = self dists - margin`` over a
    pair table (default ``self_collision_pairs(sscc, joints)``), truncated at ``margin + 0.05`` like ``IneqConst``, with
    the same ``(vals, blocks)`` contract; ``n_coll`` is the number of pairs."""

    def __init__(self, sscc, joints, n_wp, margin, pairs=None):
        self.sscc, self.joints = sscc, list(joints)
        self.pairs = self_collision_pairs(sscc, joints) if pairs is None else np.asarray(pairs, dtype=np.int32).reshape(-1, 2)
        self.n_wp, self.margin = int(n_wp), float(margin)
        self.n_dof = len(joints) + (3 if sscc.mech.with_base else 0)
        self.n_coll = len(self.pairs)
        self.n_cons = self.n_coll * self.n_wp

    def __call__(self, xi):
        """xi: flat (n_dof * n_wp,) -> numpy (val_vec (n_cons,), blocks (n_wp, n_dof, n_coll)); CUDA tensor
        (P, n_wp, n_dof) -> tensors (P, n_wp, n_coll), (P, n_wp, n_dof, n_coll)."""
        import torch
        single = not (isinstance(xi, torch.Tensor) and xi.dim() == 3)
        X = torch.as_tensor(np.asarray(xi, dtype=np.float64).reshape(1, self.n_wp, self.n_dof), device="cuda") if single else xi
        P = X.shape[0]
        set_joint_angles(self.sscc.mech, self.joints, X.reshape(P * self.n_wp, self.n_dof))
        vals, grads = compute_self_coll_dists_and_grads(self.sscc, self.joints, self.pairs, truncation_dist=self.margin + 0.05,
                                                        vals_offset=self.margin, layout=_lib.SOA)
        vals = vals.reshape(P, self.n_wp, self.n_coll)
        grads = grads.reshape(P, self.n_wp, self.n_dof, self.n_coll)
        if single:
            return vals[0].reshape(-1).cpu().numpy(), grads[0].cpu().numpy()
        return vals, grads

    dense = IneqConst.dense


def nloptize(cons):
    """planning.jl:178-185: NLopt's sign convention (constraint <= 0)."""
    def inner(xi):
        val, jac = cons(xi)
        return -val, -jac
    return inner


def pose_constraint(m, link, joints, target, with_rot=True):
    """The (link, target, with_rot) loop of ``PoseConstraint`` (planning.jl:124-137) at the configuration(s) of the
    last set_joint_angles, in one library call: val = stacked [p - p_t; rpy - rpy_t] (n_cons = sum of 3 | 6),
    jac_T (n_dof, n_cons) = transpose of the Euler-rate Jacobians.  ``link`` / ``target`` / ``with_rot`` may be lists.
    single -> ndarrays (n_cons,), (n_dof, n_cons); batch -> tensors (N, n_cons), (N, n_dof, n_cons)."""
    from .inverse_kinematics import _pose_residual
    if not isinstance(link, (list, tuple)):
        link, target, with_rot = [link], [target], [with_rot]
    val, jt = _pose_residual(m, list(link), joints, list(target), list(with_rot), _lib.POSE_CONSTRAINT)
    if m._single:
        return val[0].double().cpu().numpy(), jt[0].double().cpu().numpy()
    return val, jt


class PoseConstraint:
    """planning.jl:90-138."""

    def __init__(self, idx_wp, n_dof, move_links, target_poses, with_rots, mech, joints):
        if not isinstance(move_links, (list, tuple)):
            move_links, target_poses, with_rots = [move_links], [target_poses], [with_rots]
        self.idx_wp, self.n_dof = idx_wp, n_dof
        self.move_links, self.target_poses, self.with_rots = list(move_links), list(target_poses), list(with_rots)
        self.mech, self.joints = mech, list(joints)
        self.n_cons = sum(6 if w else 3 for w in self.with_rots)

    def __call__(self, q):
        """q: (n_dof,) -> (val (n_cons,), jac_rows (n_dof, n_cons)) -- the rows j_start:j_end of the reference's
        jac_mat; q (P, n_dof) CUDA tensor -> tensors (P, n_cons), (P, n_dof, n_cons).  One library call for all links."""
        import torch
        if isinstance(q, torch.Tensor):
            set_joint_angles(self.mech, self.joints, q)
        else:
            set_joint_angles(self.mech, self.joints, np.asarray(q, dtype=np.float64))
        return pose_constraint(self.mech, self.move_links, self.joints, self.target_poses, self.with_rots)


class ConfigurationConstraint:
    """planning.jl:72-88 (trivial; host side or torch)."""

    def __init__(self, idx_wp, n_dof, q_const):
        self.idx_wp, self.n_dof, self.n_cons = idx_wp, n_dof, n_dof
        self.q_const = q_const if _is_tensor(q_const) else np.asarray(q_const, dtype=np.float64)

    def __call__(self, q):
        if _is_tensor(q):
            import torch
            eye = -torch.eye(self.n_dof, dtype=q.dtype, device=q.device)
            return torch.as_tensor(self.q_const, dtype=q.dtype, device=q.device) - q, eye.expand(q.shape[0], -1, -1)
        return self.q_const - np.asarray(q), -np.eye(self.n_dof)


def _is_tensor(x):
    import torch
    return isinstance(x, torch.Tensor)


class EqConst:
    """planning.jl:140-176: stacks the partial constraints (``ConfigurationConstraint`` / ``PoseConstraint``), each
    acting on one waypoint, into ``val_vec`` (n_cons,) and the (n_dof n_wp, n_cons) ``jac_mat`` -- constraint k
    occupies columns i_start:i_end and the rows of its waypoint (1-based ``idx_wp``, as in the reference).
    Batched form: xi (P, n_wp, n_dof) CUDA tensor -> val (P, n_cons) and the NON-ZERO row blocks only,
    blocks (P, n_dof, n_cons) (block k sits in rows idx_wp of constraint k: ``dense_batch`` expands it)."""

    def __init__(self, n_wp, cons_arr):
        assert len(cons_arr) > 0 and all(c.n_dof == cons_arr[0].n_dof for c in cons_arr)
        self.n_dof, self.n_wp, self.cons_arr = cons_arr[0].n_dof, int(n_wp), list(cons_arr)
        self.n_cons = sum(c.n_cons for c in cons_arr)

    def __call__(self, xi):
        if _is_tensor(xi) and xi.dim() == 3:
            import torch
            vals, blocks = [], []
            for cons in self.cons_arr:
                v, j = cons(xi[:, cons.idx_wp - 1, :])
                vals.append(v)
                blocks.append(j)
            return torch.cat(vals, dim=1), torch.cat(blocks, dim=2)
        n_dof, n_wp = self.n_dof, self.n_wp
        X = np.asarray(xi, dtype=np.float64).reshape(n_wp, n_dof)       # column-major (n_dof, n_wp) of the reference
        val_vec, jac_mat = np.zeros(self.n_cons), np.zeros((n_dof * n_wp, self.n_cons))
        i_end = 0
        for cons in self.cons_arr:
            i_start, i_end = i_end, i_end + cons.n_cons
            v, j = cons(X[cons.idx_wp - 1])
            val_vec[i_start:i_end] = v
            j0 = (cons.idx_wp - 1) * n_dof
            jac_mat[j0:j0 + n_dof, i_start:i_end] = j
        return val_vec, jac_mat

    def dense_batch(self, blocks):
        """(P, n_dof, n_cons) row blocks -> the dense (P, n_dof n_wp, n_cons) matrices."""
        import torch
        P = blocks.shape[0]
        out = torch.zeros((P, self.n_dof * self.n_wp, self.n_cons), dtype=blocks.dtype, device=blocks.device)
        i_end = 0
        for cons in self.cons_arr:
            i_start, i_end = i_end, i_end + cons.n_cons
            j0 = (cons.idx_wp - 1) * self.n_dof
            out[:, j0:j0 + self.n_dof, i_start:i_end] = blocks[:, :, i_start:i_end]
        return out


class Objective:
    """planning.jl:1-28: xi' A xi with A = kron(acceleration stencil, diag(weights^2)); callable as in the
    reference (``val = F(xi, grad)`` fills ``grad`` in place when it is non-empty)."""

    def __init__(self, n_wp, weights):
        acc_block = np.array([[1.0, -2.0, 1.0], [-2.0, 4.0, -2.0], [1.0, -2.0, 1.0]])
        A_sub = np.zeros((n_wp, n_wp))
        for i in range(1, n_wp - 1):
            A_sub[i - 1:i + 2, i - 1:i + 2] += acc_block
        self.A = np.kron(A_sub, np.diag(np.asarray(weights, dtype=np.float64) ** 2))
        self.n_dim = self.A.shape[1]

    def __call__(self, xi, grad=None):
        tmp = self.A @ np.asarray(xi, dtype=np.float64)
        if grad is not None and len(grad) > 0:
            grad[:] = 2.0 * tmp
        return float(np.dot(xi, tmp))


def scipynize(obj):
    """planning.jl:187-205: (value, derivative) closure pairs in scipy's convention.  For a constraint the
    derivative is ``transpose(jac_mat)`` (n_cons, n_dof n_wp); an ``IneqConst`` is expanded to its dense matrix."""
    if isinstance(obj, Objective):
        grad = np.zeros(obj.n_dim)

        def inner_val(xi):
            return obj(xi, grad)
        return inner_val, (lambda xi: grad)       # returns the cached gradient, like the reference
    cache = {}

    def evaluate(xi):
        key = np.asarray(xi, dtype=np.float64).tobytes()
        if cache.get("key") != key:
            val, jac = obj(xi)
            if isinstance(obj, (IneqConst, SelfIneqConst)):
                jac = obj.dense(jac)
            cache.update(key=key, val=val, jac=jac)
        return cache["val"], cache["jac"]
    return (lambda xi: evaluate(xi)[0]), (lambda xi: evaluate(xi)[1].T)


def construct_problem(sscc, joints, sdf, q_start, q_goal, n_wp, n_dof, margin, partial_consts=()):
    """planning.jl:310-330 -> (F, G, H, n_whole)."""
    eq = [ConfigurationConstraint(1, n_dof, q_start), ConfigurationConstraint(n_wp, n_dof, q_goal)] + list(partial_consts)
    return Objective(n_wp, np.ones(n_dof)), IneqConst(sscc, joints, sdf, n_wp, margin), EqConst(n_wp, eq), n_dof * n_wp


def plan_trajectory(sscc, joints, sdf, q_start, q_goal, n_wp, margin=2e-2, partial_consts=(), ftol_abs=1e-3,
                    solver="SCIPY", self_margin=None):
    """planning.jl:332-401.  The three back-ends of the reference are third-party solvers; of them only scipy is
    installed here, and it is the reference's own ``solver=:SCIPY`` path (:388-394) that is reproduced: SLSQP with
    the scipynize'd objective, inequality (collision) and equality (start / goal / pose) constraints.  Every
    constraint evaluation -- n_wp waypoints per SLSQP iteration -- is one batched GPU call.  (NLopt's LD_SLSQP, the
    default of the reference, is the same algorithm; its joint-limit bounds are passed to scipy as well.)
    ``self_margin`` (extension): also keep every default self-collision pair (``self_collision_pairs``) at least this far
    apart -- a ``SelfIneqConst`` as a second inequality constraint; start / goal must then be free of self-collision too.
    Returns (q_seq (n_wp, n_dof), scipy result)."""
    from .collision import compute_coll_dists, compute_self_coll_dists
    m = sscc.mech
    n_dof = len(joints) + (3 if m.with_base else 0)
    q_start, q_goal = np.asarray(q_start, dtype=np.float64), np.asarray(q_goal, dtype=np.float64)
    assert len(q_start) == n_dof and len(q_goal) == n_dof
    for q in (q_start, q_goal):                                        # planning.jl:349-353
        set_joint_angles(m, joints, q)
        assert np.all(compute_coll_dists(sscc, joints, sdf) > 0.0), "start / goal configuration is in collision"
        if self_margin is not None:
            assert np.all(compute_self_coll_dists(sscc, joints) > 0.0), "start / goal configuration is in self-collision"
    xi_init = create_straight_trajectory(q_start, q_goal, n_wp)
    F, G, H, n_whole = construct_problem(sscc, joints, sdf, q_start, q_goal, n_wp, n_dof, margin, partial_consts)
    if solver != "SCIPY":
        raise _lib.KinError("plan_trajectory: solver %r is not available here (NLopt / Ipopt are third-party and not "
                            "installed); use solver='SCIPY', the reference's scipy SLSQP back-end" % (solver,))
    from scipy.optimize import minimize
    lo = [j.lower_limit for j in joints] + [-np.inf] * (3 if m.with_base else 0)
    hi = [j.upper_limit for j in joints] + [np.inf] * (3 if m.with_base else 0)
    bounds = [(a if np.isfinite(a) else None, b if np.isfinite(b) else None) for a, b in zip(lo, hi)] * n_wp
    f, df = scipynize(F)
    g, dg = scipynize(G)
    h, dh = scipynize(H)
    constraints = [{"type": "ineq", "fun": g, "jac": dg}, {"type": "eq", "fun": h, "jac": dh}]
    if self_margin is not None:
        gs, dgs = scipynize(SelfIneqConst(sscc, joints, n_wp, self_margin))
        constraints.insert(1, {"type": "ineq", "fun": gs, "jac": dgs})
    ret = minimize(f, xi_init, jac=df, method="SLSQP", bounds=bounds, options={"ftol": ftol_abs, "maxiter": 200},
                   constraints=constraints)
    return ret.x.reshape(n_wp, n_dof), ret


def smoothness_objective(xi, n_wp, weights):
    """``Objective`` of planning.jl:1-28: xi' A xi with A = kron(acceleration stencil, diag(w^2)); off the hot
    path (cheap), batched with torch.  xi (P, n_wp, n_dof) -> (val (P,), grad (P, n_wp, n_dof))."""
    import torch
    w2 = torch.as_tensor(np.asarray(weights, dtype=np.float64) ** 2, device=xi.device, dtype=xi.dtype)
    acc = xi[:, :-2] - 2 * xi[:, 1:-1] + xi[:, 2:]                 # (P, n_wp-2, n_dof)
    val = (acc * acc * w2).sum(dim=(1, 2))
    grad = torch.zeros_like(xi)
    g = 2 * acc * w2
    grad[:, :-2] += g
    grad[:, 1:-1] -= 2 * g
    grad[:, 2:] += g
    return val, grad


def gather_stacked(vals, grads, group=None):
    """Config 5 (SURVEY 8e): all-gather the per-rank slabs of stacked constraint values / Jacobian blocks so
    that every rank holds all problems.  vals (P_local, n_wp, n_coll), grads (P_local, n_wp, n_dof, n_coll);
    NCCL on GPUs (gloo in the CPU tests).  Returns the concatenation over ranks along the problem axis.
    Generic form (two collectives on copies); ``IneqConst.evaluate_packed`` + ``gather_packed`` is the fast path."""
    import torch
    import torch.distributed as dist
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return vals, grads
    W = dist.get_world_size(group)
    # equal shard sizes (P divisible by the world size) are required, as in config 5 (4096 problems)
    v_all = torch.empty((W * vals.shape[0],) + tuple(vals.shape[1:]), dtype=vals.dtype, device=vals.device)
    g_all = torch.empty((W * grads.shape[0],) + tuple(grads.shape[1:]), dtype=grads.dtype, device=grads.device)
    dist.all_gather_into_tensor(v_all, vals.contiguous(), group=group)
    dist.all_gather_into_tensor(g_all, grads.contiguous(), group=group)
    return v_all, g_all


def gather_packed(slab, n_wp, n_dof, n_coll, out=None, group=None):
    """ONE collective for the stacked outputs of config 5: ``slab`` is the (n_coll + n_coll n_dof, P_local n_wp)
    SoA storage the kernel wrote [vals rows | grads rows] (``IneqConst.evaluate_packed``); it is all-gathered as it
    is into ``out`` (W, n_coll + n_coll n_dof, P_local n_wp) -- no packing copy, no per-array collective.  Returns
    VIEWS of ``out``: vals (W, P_local, n_wp, n_coll), grads (W, P_local, n_wp, n_dof, n_coll); the problem axis
    of the stacked system is (rank, local problem), i.e. problem p of rank r is global problem r P_local + p.

    Bound (DESIGN.md 5): every rank must RECEIVE (W - 1) / W of the stacked outputs, 1152 B per waypoint at
    S = 16, D = 8 -> 264 MB at 4096 x 64 waypoints on 8 GPUs, >= 0.34 ms at the measured 770 GB/s of NVLink
    inbound, against 0.19 ms for evaluating all waypoints on ONE GPU: sharding + gathering this evaluation can
    not beat a single GPU at any size (1.3 ns per waypoint to receive vs 0.7 ns to compute); shard it only when
    the consumers of the outputs are sharded too (independent problems per rank, no gather)."""
    import torch
    import torch.distributed as dist
    C_, Nl = slab.shape
    S = n_coll
    assert C_ == S + S * n_dof and Nl % n_wp == 0
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        W, out = 1, slab[None]
    else:
        W = dist.get_world_size(group)
        if out is None:
            out = torch.empty((W, C_, Nl), dtype=slab.dtype, device=slab.device)
        dist.all_gather_into_tensor(out.view(W * C_, Nl), slab, group=group)      # concatenation along dim 0
    Pl = Nl // n_wp
    vals = out[:, :S, :].reshape(W, S, Pl, n_wp).permute(0, 2, 3, 1)
    grads = out[:, S:, :].reshape(W, S, n_dof, Pl, n_wp).permute(0, 3, 4, 2, 1)
    return vals, grads


def shard_range(n_total, rank, world):
    """Contiguous batch shard of SURVEY 8e: rank r gets [r N / G, (r + 1) N / G)."""
    return (n_total * rank) // world, (n_total * (rank + 1)) // world

"""SweptSphereCollisionChecker and compute_coll_dists[_and_grads] (collision.jl:1-103) on the B200
backend."""
from __future__ import annotations

import uuid

import numpy as np

from . import lib as _lib
from .algorithm import _check_joints
from .device import current_q, device_model, evaluate, evaluate_self
from .mechanism import Link, Mechanism, SphereMetaData, add_new_link
from .transform import Transform


class SweptSphereCollisionChecker:         # collision.jl:32-37
    def __init__(self, mech: Mechanism):
        self.mech = mech
        self.sphere_links, self.sphere_radii = [], []
        self._parents, self._centers = [], []


def add_coll_links(sscc: SweptSphereCollisionChecker, coll_link: Link, centers=None, radii=None, vertices=None, mesh_dirs=(),
                   n_sphere=None, tol=0.1):
    """collision.jl:39-49.  The reference obtains (centers, radius) from scikit-robot's swept-sphere fit of the
    link's collision mesh (collision.jl:16-30).  Here, in order of precedence:
      * ``centers`` (k, 3) in the link frame + ``radii`` (scalar or (k,)): an explicit sphere table;
      * ``vertices`` (n, 3): the fit of swept_sphere.compute_swept_sphere (mesh-free restatement of the algorithm);
      * otherwise the link's own collision geometry: a box / cylinder / sphere primitive is sampled, a mesh is read
        from an STL under ``mesh_dirs``; a link without usable geometry adds no spheres, as in the reference
        (collision.jl:18) -- except that a mesh that cannot be found raises (the meshes of data/fetch.urdf do not
        ship with the reference)."""
    if centers is None:
        from . import swept_sphere as SS
        from .mechanism import MeshMetaData
        if vertices is None:
            vertices = SS.link_vertices(coll_link, mesh_dirs)
            if vertices is None:
                if isinstance(coll_link.geometric_meta_data, MeshMetaData):
                    raise _lib.KinError("add_coll_links: collision mesh %r of link %r not found (searched %r); pass centers= / radii= "
                                        "or vertices=" % (coll_link.geometric_meta_data.file_path, coll_link.name, list(mesh_dirs)))
                return
        centers, radii = SS.compute_swept_sphere(vertices, n_sphere=n_sphere, tol=tol)
    centers = np.asarray(centers, dtype=np.float64).reshape(-1, 3)
    radii = np.broadcast_to(np.asarray(radii, dtype=np.float64), (len(centers),))
    for c, r in zip(centers, radii):
        new_link = Link("sphere_" + str(uuid.uuid1()), link_type="CollSphere",
                        geometric_meta_data=SphereMetaData(r, Transform()))
        add_new_link(sscc.mech, new_link, coll_link, c)
        sscc.sphere_links.append(new_link)
        sscc.sphere_radii.append(float(r))
        sscc._parents.append(coll_link.id)
        sscc._centers.append(c.copy())


def _prepare(sscc, joints, sdf):
    m = sscc.mech
    _check_joints(m, joints)
    dm = device_model(m)
    dm.set_spheres(sscc._parents, sscc._centers, sscc.sphere_radii)
    dm.set_boxes(*sdf.world_scene())
    return m, dm


def compute_coll_dists(sscc, joints, sdf, layout=None, dtype=None, return_argmin=False):
    """collision.jl:51-65: ``vals[i] = sdf(centre_i) - r_i``.  single -> ndarray (S,); batch -> tensor (N, S)."""
    m, dm = _prepare(sscc, joints, sdf)
    Q, ql, N = current_q(m, dtype)
    out = evaluate(dm, Q, ql, N, layout=layout, collision=True, with_grads=False, want_argmin=return_argmin)
    vals = out["vals"][0].double().cpu().numpy() if m._single else out["vals"]
    if return_argmin:
        return vals, (out["argmin"][0].cpu().numpy() if m._single else out["argmin"])
    return vals


def compute_coll_dists_and_grads(sscc, joints, sdf, truncation_dist=np.inf, grad_mode=_lib.GRAD_FD,
                                 scratch_mode=_lib.SCRATCH_REFERENCE, layout=None, dtype=None, return_argmin=False,
                                 vals_offset=0.0):
    """collision.jl:67-103.  single -> (vals (S,), grads (n_dof, S)); batch -> (N, S), (N, n_dof, S).
    ``scratch_mode`` defaults to the reference's behaviour (one Jacobian scratch shared by all spheres,
    collision.jl:76,90); ``SCRATCH_CLEAN`` gives the gradient with the untouched columns zeroed."""
    m, dm = _prepare(sscc, joints, sdf)
    Q, ql, N = current_q(m, dtype)
    out = evaluate(dm, Q, ql, N, layout=layout, collision=True, with_grads=True, truncation_dist=truncation_dist,
                   grad_mode=grad_mode, scratch_mode=scratch_mode, want_argmin=return_argmin, vals_offset=vals_offset)
    if m._single:
        res = (out["vals"][0].double().cpu().numpy(), out["grads"][0].double().cpu().numpy())
        return res + (out["argmin"][0].cpu().numpy(),) if return_argmin else res
    res = (out["vals"], out["grads"])
    return res + (out["argmin"],) if return_argmin else res


def compute_coll_summary(sscc, joints, sdf, margin=0.0, dtype=None):
    """Reductions of ``compute_coll_dists`` per configuration (extension; ``kin_collision_summary``): the smallest sphere
    distance, the sphere that attains it (1-based, first minimum) and the hinge cost ``sum_s max(0, margin - d_s)^2``.
    single -> (float, int, float); batch -> tensors (N,), (N,) int32, (N,)."""
    import torch
    m, dm = _prepare(sscc, joints, sdf)
    Q, ql, N = current_q(m, dtype)
    dmin = torch.empty(N, dtype=Q.dtype, device=Q.device)
    cost = torch.empty(N, dtype=Q.dtype, device=Q.device)
    amin = torch.empty(N, dtype=torch.int32, device=Q.device)
    _lib.check(_lib.lib().kin_collision_summary(dm.h, _lib.F32 if Q.dtype == torch.float32 else _lib.F64, ql, Q.data_ptr(), N,
                                                float(margin), dmin.data_ptr(), amin.data_ptr(), cost.data_ptr(),
                                                torch.cuda.current_stream(Q.device).cuda_stream))
    if m._single:
        return float(dmin[0]), int(amin[0]), float(cost[0])
    return dmin, amin, cost


# ---- self-collision between the checker's spheres (an extension: collision.jl is sphere-vs-environment only) ----
def self_collision_pairs(sscc, joints, ignore=(), skip_adjacent=True):
    """The default self-collision pair table of ``sscc`` under the control joints ``joints``: (P, 2) int32 1-based
    sphere ids (i < j, in sphere order).  A pair of spheres is dropped when
      * both sit on the same link;
      * their links move rigidly together: they have the same nearest ancestor whose parent joint is in ``joints``
        (or none), so their distance is constant -- leaving a joint out of ``joints`` merges the links around it;
      * ``skip_adjacent``: one link is the parent of the other through a single joint (SRDF "Adjacent");
      * the (unordered) pair of their link names is in ``ignore``."""
    m = sscc.mech
    ctrl = {j.id for j in joints}

    def group(lid):                       # nearest controlled ancestor (the root when there is none)
        l = m.links[lid - 1]
        while l.plink_id != -1 and l.pjoint_id not in ctrl:
            l = m.links[l.plink_id - 1]
        return l.id

    ignored = {frozenset(p) for p in ignore}
    parents = list(sscc._parents)
    groups = [group(l) for l in parents]
    pairs = []
    for i in range(len(parents)):
        for j in range(i + 1, len(parents)):
            li, lj = m.links[parents[i] - 1], m.links[parents[j] - 1]
            if li.id == lj.id or groups[i] == groups[j]:
                continue
            if skip_adjacent and (li.plink_id == lj.id or lj.plink_id == li.id):
                continue
            if frozenset((li.name, lj.name)) in ignored:
                continue
            pairs.append((i + 1, j + 1))
    return np.asarray(pairs, dtype=np.int32).reshape(-1, 2)


def _prepare_self(sscc, joints, pairs):
    m = sscc.mech
    _check_joints(m, joints)
    dm = device_model(m)
    dm.set_spheres(sscc._parents, sscc._centers, sscc.sphere_radii)
    dm.set_self_pairs(self_collision_pairs(sscc, joints) if pairs is None else pairs)
    return m, dm


def compute_self_coll_dists(sscc, joints, pairs=None, layout=None, dtype=None):
    """Self-collision distances ``d_p = |c_i - c_j| - r_i - r_j`` of the sphere pairs (extension; ``kin_self_collision``;
    ``pairs`` (P, 2) 1-based, default ``self_collision_pairs(sscc, joints)``).  single -> ndarray (P,); batch -> (N, P)."""
    m, dm = _prepare_self(sscc, joints, pairs)
    Q, ql, N = current_q(m, dtype)
    vals = evaluate_self(dm, Q, ql, N, layout=layout)["vals"]
    return vals[0].double().cpu().numpy() if m._single else vals


def compute_self_coll_dists_and_grads(sscc, joints, pairs=None, truncation_dist=np.inf, vals_offset=0.0, layout=None,
                                      dtype=None):
    """... and their gradients ``u . (J_i - J_j)`` in q (0 where the centres coincide); ``d > truncation_dist`` gives
    ``truncation_dist`` and a zero gradient (collision.jl:84-86), then ``vals_offset`` is subtracted.
    single -> (vals (P,), grads (n_dof, P)); batch -> (N, P), (N, n_dof, P)."""
    m, dm = _prepare_self(sscc, joints, pairs)
    Q, ql, N = current_q(m, dtype)
    out = evaluate_self(dm, Q, ql, N, layout=layout, with_grads=True, truncation_dist=truncation_dist,
                        vals_offset=vals_offset)
    if m._single:
        return out["vals"][0].double().cpu().numpy(), out["grads"][0].double().cpu().numpy()
    return out["vals"], out["grads"]


def compute_self_coll_summary(sscc, joints, pairs=None, dtype=None):
    """Per configuration the smallest self-collision distance and the pair attaining it (1-based, first minimum), without
    materialising the P distances.  single -> (float, int); batch -> tensors (N,), (N,) int32."""
    m, dm = _prepare_self(sscc, joints, pairs)
    Q, ql, N = current_q(m, dtype)
    out = evaluate_self(dm, Q, ql, N, with_vals=False, want_summary=True)
    if m._single:
        return float(out["dmin"][0]), int(out["amin"][0])
    return out["dmin"], out["amin"]

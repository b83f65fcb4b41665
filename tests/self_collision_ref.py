"""Oracle of the self-collision extension (kin_self_collision; the reference has sphere-vs-environment collision only),
built from nothing but the oracle's own get_transform / get_jacobian(..., with_rot=False) of the sphere links that
add_coll_links adds.  It shares no code with the product."""
import numpy as np

from oracle import ref_model as R


def self_coll_dists_and_grads(sscc, joints, pairs, truncation_dist=np.inf, offset=0.0):
    """At the mechanism's current angles, per pair p = (i, j) (1-based sphere ids): d = |c_i - c_j| - r_i - r_j and
    grad = u' (J_i - J_j), u = (c_i - c_j) / |c_i - c_j| (0 when the centres coincide).  d > truncation_dist gives
    truncation_dist and a zero gradient (collision.jl:84-86); offset is subtracted from every value.
    -> (vals (P,), grads (n_dof, P), untruncated d (P,))."""
    m = sscc.mech
    n_dof = len(joints) + m.n_dof_extra
    cent = [R.get_transform(m, l)[:3, 3] for l in sscc.sphere_links]
    jac = [R.get_jacobian(m, l, joints, with_rot=False) for l in sscc.sphere_links]
    P = len(pairs)
    vals, grads, raw = np.zeros(P), np.zeros((n_dof, P)), np.zeros(P)
    for p, (i, j) in enumerate(pairs):
        v = cent[i - 1] - cent[j - 1]
        L = np.linalg.norm(v)
        raw[p] = d = L - sscc.sphere_radii[i - 1] - sscc.sphere_radii[j - 1]
        if d > truncation_dist:
            vals[p] = truncation_dist - offset
            continue
        vals[p] = d - offset
        if L > 0:
            grads[:, p] = (v / L) @ (jac[i - 1] - jac[j - 1])
    return vals, grads, raw


def batch(sscc, joints, q, pairs, truncation_dist=np.inf, offset=0.0):
    """The same over a batch q (N, n_dof) -> vals (N, P), grads (N, n_dof, P), untruncated d (N, P)."""
    out = []
    for qn in q:
        R.set_joint_angles(sscc.mech, joints, qn)
        out.append(self_coll_dists_and_grads(sscc, joints, pairs, truncation_dist, offset))
    return tuple(np.stack(x) for x in zip(*out))

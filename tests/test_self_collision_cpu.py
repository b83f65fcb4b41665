"""Self-collision between collision spheres (an extension: collision.jl has sphere-vs-environment only), host side:
the oracle of tests/self_collision_ref.py against a closed form and against central differences of itself, the
default pair policy (collision.self_collision_pairs), and the C declarations of the new entry points."""
import os
import re

import numpy as np
import pytest

import kinematics_jl_b200 as K
from oracle import ref_model as R
from conftest import ROOT
import scenes
import scenes_dual_arm as DA
import self_collision_ref as SR

ONE_JOINT_URDF = """<robot name="one">
  <link name="base"/>
  <link name="arm"/>
  <joint name="hinge" type="revolute">
    <parent link="base"/><child link="arm"/><origin xyz="0 0 0" rpy="0 0 0"/><axis xyz="0 0 1"/>
    <limit lower="-3.2" upper="3.2"/>
  </joint>
</robot>"""


def test_oracle_one_revolute_joint_closed_form(tmp_path):
    """One sphere at radius a from the axis, one fixed at distance b: d = sqrt(a^2 + b^2 - 2ab cos t) - r1 - r2 and
    dd/dt = ab sin t / L; truncation and offset as collision.jl:84-86 / planning.jl:66; coincident centres: gradient 0."""
    p = tmp_path / "one.urdf"
    p.write_text(ONE_JOINT_URDF)
    m = R.parse_urdf(str(p))
    joints = [R.find_joint(m, "hinge")]
    a, b, r1, r2 = 0.7, 0.4, 0.05, 0.08
    sscc = R.SweptSphereCollisionChecker(m)
    R.add_coll_links(sscc, R.find_link(m, "arm"), [[a, 0, 0]], [r1])
    R.add_coll_links(sscc, R.find_link(m, "base"), [[b, 0, 0]], [r2])
    for t in np.linspace(-3.0, 3.0, 13):
        R.set_joint_angles(m, joints, [t])
        vals, grads, raw = SR.self_coll_dists_and_grads(sscc, joints, [(1, 2)])
        L = np.sqrt(a * a + b * b - 2 * a * b * np.cos(t))
        np.testing.assert_allclose(vals[0], L - r1 - r2, rtol=0, atol=1e-14)
        np.testing.assert_allclose(grads[0, 0], a * b * np.sin(t) / L, rtol=0, atol=1e-14)
        # the pair in the other order: same distance, same gradient (u and J_i - J_j both flip)
        v2, g2, _ = SR.self_coll_dists_and_grads(sscc, joints, [(2, 1)])
        np.testing.assert_allclose(v2, vals, atol=1e-15)
        np.testing.assert_allclose(g2, grads, atol=1e-15)
        tr = L - r1 - r2 - 0.1
        v3, g3, raw3 = SR.self_coll_dists_and_grads(sscc, joints, [(1, 2)], truncation_dist=tr, offset=0.02)
        assert v3[0] == tr - 0.02 and g3[0, 0] == 0.0 and raw3[0] == raw[0]
    sscc2 = R.SweptSphereCollisionChecker(m)                 # both centres on the axis: L == 0 at every angle
    R.add_coll_links(sscc2, R.find_link(m, "arm"), [[0, 0, 0.1]], [r1])
    R.add_coll_links(sscc2, R.find_link(m, "base"), [[0, 0, 0.1]], [r2])
    R.set_joint_angles(m, joints, [0.3])
    vals, grads, _ = SR.self_coll_dists_and_grads(sscc2, joints, [(1, 2)])
    assert vals[0] == -r1 - r2 and grads[0, 0] == 0.0


def _fixtures():
    for with_base in (False, True):
        m, joints, sscc = scenes.product_fetch(with_base)
        mo, jo, so = scenes.oracle_fetch(with_base)
        yield "fetch", with_base, K.self_collision_pairs(sscc, joints), jo, so
        m, joints, sscc, _ = DA.product(with_base)
        mo, jo, so, _ = DA.oracle(with_base)
        yield "dual_arm", with_base, K.self_collision_pairs(sscc, joints), jo, so


@pytest.mark.parametrize("case", range(4))
def test_oracle_gradient_is_the_central_difference_of_its_distance(case):
    name, with_base, pairs, jo, so = list(_fixtures())[case]
    q = scenes.random_configs(jo, 6, with_base, seed=21 + case)
    h = 1e-6
    for qn in q:
        R.set_joint_angles(so.mech, jo, qn)
        _, g, _ = SR.self_coll_dists_and_grads(so, jo, pairs)
        fd = np.zeros_like(g)
        for k in range(len(qn)):
            e = np.zeros_like(qn)
            e[k] = h
            R.set_joint_angles(so.mech, jo, qn + e)
            dp = SR.self_coll_dists_and_grads(so, jo, pairs)[2]
            R.set_joint_angles(so.mech, jo, qn - e)
            dm = SR.self_coll_dists_and_grads(so, jo, pairs)[2]
            fd[k] = (dp - dm) / (2 * h)
        np.testing.assert_allclose(g, fd, rtol=0, atol=1e-7, err_msg=name)
        assert np.abs(g).max() > 0.1


def test_default_pair_policy_counts():
    """Fetch, 8 arm joints: 5 link pairs x 16 sphere pairs = 80 (upperarm_roll_link / elbow_flex_link are adjacent);
    dual-arm: C(19, 2) = 171 minus 6 same-link minus 20 adjacent = 145, with or without the planar base."""
    m, joints, sscc = scenes.product_fetch()
    pairs = K.self_collision_pairs(sscc, joints)
    assert pairs.shape == (80, 2) and pairs.dtype == np.int32
    assert np.all(pairs[:, 0] < pairs[:, 1]) and pairs.min() >= 1 and pairs.max() <= 16
    names = {frozenset((m.links[sscc._parents[i - 1] - 1].name, m.links[sscc._parents[j - 1] - 1].name)) for i, j in pairs}
    assert len(names) == 5 and frozenset(("upperarm_roll_link", "elbow_flex_link")) not in names
    for with_base in (False, True):
        m, joints, sscc, _ = DA.product(with_base)
        assert len(K.self_collision_pairs(sscc, joints)) == 145
        assert len(K.self_collision_pairs(sscc, joints, skip_adjacent=False)) == 165


def test_pair_policy_ignore_and_frozen_joints():
    m, joints, sscc = scenes.product_fetch()
    full = K.self_collision_pairs(sscc, joints)
    ign = K.self_collision_pairs(sscc, joints, ignore=[("wrist_flex_link", "torso_lift_link")])
    assert len(ign) == 64
    assert {tuple(p) for p in ign} < {tuple(p) for p in full}
    # leaving forearm_roll_joint and wrist_flex_joint out makes wrist_flex_link rigid with elbow_flex_link
    frozen = [j for j in joints if j.name not in ("forearm_roll_joint", "wrist_flex_joint")]
    fr = K.self_collision_pairs(sscc, frozen)
    assert len(fr) == 64
    par = lambda s: m.links[sscc._parents[s - 1] - 1].name
    assert not any({par(i), par(j)} == {"elbow_flex_link", "wrist_flex_link"} for i, j in fr)
    # leaving torso_lift_joint out merges the torso with the root: nothing else changes
    assert len(K.self_collision_pairs(sscc, joints[1:])) == 80


def test_header_declares_the_self_collision_entry_points():
    h = open(os.path.join(ROOT, "include", "kin_b200.h")).read()
    assert re.search(r"#define KIN_MAX_SELF_PAIRS \d+", h)
    for name in ("kin_model_set_self_pairs", "kin_model_n_self_pairs", "kin_self_collision"):
        assert re.search(r"KIN_API int %s\(" % name, h), name
    from kinematics_jl_b200 import lib as L
    assert {"kin_model_set_self_pairs", "kin_model_n_self_pairs", "kin_self_collision"} <= set(L.EXPORTS)
    assert "#define KIN_B200_ABI_VERSION 4" in h

"""Public surface of the B200 backend: the export list of the reference (Kinematics.jl:45-70) for the
hot path, same names and argument meaning, evaluated by libkin_b200 (no CPU fallback)."""
from .lib import (AOS, F32, F64, GRAD_ANALYTIC, GRAD_FD, GRAD_FD_DIRECT, SCRATCH_CLEAN, SCRATCH_REFERENCE, SOA, TILED32, KinError, build)
from .lib import lib as load_library
from .transform import Transform, rotation, rpy, translation
from .mechanism import (FIXED, PRISMATIC, REVOLUTE, BoxMetaData, CylinderMetaData, Joint, Link, Mechanism, MeshMetaData, SphereMetaData,
                        User, add_new_link, child_joints, child_link, child_links, find_joint, find_link,
                        get_joint_angles, is_relevant, isleaf, isroot, joint_angle, lower_limit, parent_joint,
                        parent_link, set_base_pose, set_joint_angle, set_joint_angles, upper_limit)
from .load_urdf import parse_urdf
from .algorithm import get_jacobian, get_jacobian_, get_transform
from .sdf import BoxSDF, CylinderSDF, GridSDF, SphereSDF, UnionSDF
from .collision import (SweptSphereCollisionChecker, add_coll_links, compute_coll_dists,
                        compute_coll_dists_and_grads, compute_coll_summary, compute_self_coll_dists,
                        compute_self_coll_dists_and_grads, compute_self_coll_summary, self_collision_pairs)

from .inverse_kinematics import ik_objective, ik_solve_device, inverse_kinematics, inverse_kinematics_batch
from .planning import (ConfigurationConstraint, EqConst, IneqConst, Objective, PoseConstraint, SelfIneqConst, construct_problem,
                       create_straight_trajectory, gather_packed, gather_stacked, nloptize, plan_trajectory, pose_constraint, scipynize,
                       shard_range, smoothness_objective)
from .lib import POSE_CONSTRAINT, POSE_IK_OBJECTIVE
from .swept_sphere import compute_swept_sphere, load_stl_vertices, primitive_vertices

__all__ = [n for n in dir() if not n.startswith("_")]

# CUDABackend.jl -- the Julia side of the drop-in: a module to `include` from Kinematics.jl
# (after planning.jl) that binds libkin_b200.so with `ccall` and adds batched methods to the
# reference's own exported functions (export list Kinematics.jl:45-70).  The reference's
# single-configuration API is untouched.
#
# NOT EXECUTED in the build image (Julia is not installed there).  What IS checked there:
#   * tests/test_julia_binding.py parses the two struct declarations below and compares field order, types, sizes
#     and offsets with the C structs of include/kin_b200.h (as laid out by gcc: tests/abi_layout.c), and checks that
#     every `ccall` names an exported symbol with the right number of arguments;
#   * the Python host mirror kinematics.jl_b200/ (device.py, algorithm.py, collision.py, sdf.py, planning.py,
#     inverse_kinematics.py) makes the same calls, in the same order, and is tested on B200 against the oracle.
#
# Layout note.  The library is fastest with batch-index-fastest arrays: a Julia CuMatrix of size (N, n_dof) IS
# KIN_LAYOUT_SOA.  The reference-native layout -- one configuration per COLUMN, (n_dof, N), e.g. `xi` reshaped to
# (n_dof, n_wp) in planning.jl:58 -- is KIN_LAYOUT_AOS; every method below accepts it with `layout=:aos`
# (large batches stage each warp's records through shared memory and write them in whole sectors: FK / Jacobian calls
# run at 0.97 of the HBM peak in this layout -- faster than SoA --, the fused FK + Jacobian + collision call at 0.8x SoA).
#
#   dm = CUDABackend.DeviceMechanism(mech, joints; sscc=sscc, sdf=sdf)
#   Q  = CUDA.rand(Float64, N, n_dof)                                   # SoA
#   T  = get_transform(dm, links, Q)                                    # (N, 12, length(links))
#   J  = get_jacobian(dm, link, Q, true; rpy_jac=false)                 # (N, rows, n_dof)
#   get_jacobian!(dm, link, Q, true, J)                                 # writes only the relevant columns
#   v, g = compute_coll_dists_and_grads(dm, Q; truncation_dist=Inf)     # (N, S), (N, n_dof, S)
#   f, df = f_objective(dm, link, Q, target; with_rot=true)             # inverse_kinematics.jl:38-50, batched
#   v, jt = pose_constraint(dm, links, Q, targets, with_rots)           # planning.jl:114-138, all links in one call
#   v, blocks = ineq_const(dm, Xi, margin)                              # planning.jl:55-68 for (n_dof, n_wp * P) columns
#   d = sdf_points(sdf, P); g = sdf_gradient(sdf, P)                    # sdf.jl:34-41,67-74,108-119 for (N, 3) points
#   q, f, its, dmin = inverse_kinematics_batch(dm, link, targets, q0, joints; collision=true, margin=0.02)
#                                                                       # inverse_kinematics.jl:1-30 for N targets at once
#   set_self_pairs!(dm, pairs); v, g = compute_self_coll_dists_and_grads(dm, Q)   # self-collision (extension), (N, P)
module CUDABackend

using CUDA
using ..Kinematics
using ..Kinematics: Mechanism, Link, Joint, Fixed, Revolute, Prismatic, Transform, SweptSphereCollisionChecker,
                    AbstractSDF, BoxSDF, UnionSDF, parent_joint, isroot, inv_pose, translation, rpy, lower_limit, upper_limit
import ..Kinematics: get_transform, get_jacobian, get_jacobian!, compute_coll_dists, compute_coll_dists_and_grads

const libkin = get(ENV, "KIN_B200_LIB", "libkin_b200.so")

const KIN_F64, KIN_F32 = Cint(0), Cint(1)
const KIN_LAYOUT_SOA, KIN_LAYOUT_AOS, KIN_LAYOUT_TILED32 = Cint(0), Cint(1), Cint(2)
const KIN_GRAD_FD, KIN_GRAD_ANALYTIC, KIN_GRAD_FD_DIRECT = Cint(0), Cint(1), Cint(2)
const KIN_SCRATCH_REFERENCE, KIN_SCRATCH_CLEAN = Cint(0), Cint(1)
const KIN_POSE_IK_OBJECTIVE, KIN_POSE_CONSTRAINT = Cint(0), Cint(1)

# include/kin_b200.h: KinModelDesc
struct KinModelDesc
    n_links::Cint
    parent_link::Ptr{Cint}
    joint_type::Ptr{Cint}
    joint_pose::Ptr{Cdouble}
    joint_axis::Ptr{Cdouble}
    q_index::Ptr{Cint}
    default_angle::Ptr{Cdouble}
    n_joints::Cint
    with_base::Cint
    n_spheres::Cint
    sphere_link::Ptr{Cint}
    sphere_center::Ptr{Cdouble}
    sphere_radius::Ptr{Cdouble}
    n_boxes::Cint
    box_pose::Ptr{Cdouble}
    box_width::Ptr{Cdouble}
end

# include/kin_b200.h: KinCall
struct KinCall
    precision::Cint
    layout::Cint
    n::Int64
    batch_stride::Int64
    q::CuPtr{Cvoid}
    n_fk_links::Cint
    fk_links::Ptr{Cint}
    T_out::CuPtr{Cvoid}
    n_jac_links::Cint
    jac_links::Ptr{Cint}
    with_rot::Cint
    rpy_jac::Cint
    keep_irrelevant::Cint
    J_out::CuPtr{Cvoid}
    truncation_dist::Cdouble
    grad_mode::Cint
    scratch_mode::Cint
    vals_out::CuPtr{Cvoid}
    grads_out::CuPtr{Cvoid}
    argmin_out::CuPtr{Cint}
    vals_offset::Cdouble
    stream::Ptr{Cvoid}
end

# include/kin_b200.h: KinIkCall
struct KinIkCall
    n::Int64
    link_id::Cint
    with_rot::Cint
    iters::Cint
    ftol::Cdouble
    lambda0::Cdouble
    targets::CuPtr{Cvoid}
    q0::CuPtr{Cvoid}
    lower::Ptr{Cdouble}
    upper::Ptr{Cdouble}
    q_out::CuPtr{Cvoid}
    f_out::CuPtr{Cvoid}
    iters_out::CuPtr{Cint}
    stream::Ptr{Cvoid}
    collision::Cint
    reserved_::Cint
    margin::Cdouble
    coll_weight::Cdouble
    ctol::Cdouble
    dmin_out::CuPtr{Cvoid}
end

check(rc) = rc == 0 || error("libkin_b200: " * unsafe_string(ccall((:kin_last_error, libkin), Cstring, ())))
layout_code(l::Symbol) = l === :soa ? KIN_LAYOUT_SOA : l === :aos ? KIN_LAYOUT_AOS : error("layout must be :soa or :aos")
cuda_stream() = Base.unsafe_convert(Ptr{Cvoid}, CUDA.stream().handle)
# batch size of a configuration matrix in the given layout
nbatch(Q, layout) = layout === :soa ? size(Q, 1) : size(Q, 2)
# allocate an output with `dims` per configuration: SoA (N, dims...), AoS (dims..., N)
out_array(N, layout, dims...) = layout === :soa ? CuArray{Float64}(undef, N, dims...) : CuArray{Float64}(undef, dims..., N)

joint_type_code(::Joint{Fixed}) = Cint(0)
joint_type_code(::Joint{Revolute}) = Cint(1)
joint_type_code(::Joint{Prismatic}) = Cint(2)
joint_axis(j::Joint{Fixed}) = (0.0, 0.0, 0.0)
joint_axis(j::Joint) = Tuple(j.jt.axis)

# world box table of an SDF: column-major 4x4 poses + widths (sdf.jl:48-65, 82-97)
function box_tables(sdf::AbstractSDF)
    boxes = sdf isa UnionSDF ? sdf.sdfs : [sdf]
    B = length(boxes)
    bpose = zeros(Cdouble, 16, B); bwidth = zeros(Cdouble, 3, B)
    for (i, b) in enumerate(boxes)
        inv_pose(b)                                    # refreshes b.pose for attached boxes (sdf.jl:24-32)
        bpose[:, i] = vec(b.pose.mat); bwidth[:, i] .= b.width
    end
    return B, bpose, bwidth
end

mutable struct DeviceMechanism
    handle::Ptr{Cvoid}
    n_dof::Int
    n_spheres::Int
    function DeviceMechanism(m::Mechanism, joints::Vector{<:Joint};
                             sscc::Union{SweptSphereCollisionChecker, Nothing}=nothing,
                             sdf::Union{AbstractSDF, Nothing}=nothing)
        L = length(m.links)
        parent = fill(Cint(-1), L); jtype = zeros(Cint, L); qidx = fill(Cint(-1), L)
        pose = zeros(Cdouble, 16, L); axis = zeros(Cdouble, 3, L); defang = zeros(Cdouble, L)
        col = Dict(j.id => Cint(c - 1) for (c, j) in enumerate(joints))
        for l in m.links
            isroot(l) && continue
            j = parent_joint(m, l)
            parent[l.id] = l.plink_id
            jtype[l.id] = joint_type_code(j)
            pose[:, l.id] = vec(j.pose.mat)            # Transform.mat is already column-major 4x4
            axis[:, l.id] .= joint_axis(j)
            qidx[l.id] = get(col, j.id, Cint(-1))
            defang[l.id] = m.angles[j.id]
        end
        # spheres: sscc.sphere_links are children of the collision link through a pure translation
        S = sscc === nothing ? 0 : length(sscc.sphere_links)
        slink = Cint[sscc.sphere_links[i].plink_id for i in 1:S]
        scen = zeros(Cdouble, 3, S)
        for i in 1:S
            scen[:, i] = m.joints[sscc.sphere_links[i].pjoint_id].pose.mat[1:3, 4]
        end
        srad = S == 0 ? Cdouble[] : Vector{Cdouble}(sscc.sphere_radii)
        B, bpose, bwidth = sdf === nothing ? (0, zeros(Cdouble, 16, 0), zeros(Cdouble, 3, 0)) : box_tables(sdf)
        handle = Ref{Ptr{Cvoid}}(C_NULL)
        GC.@preserve parent jtype pose axis qidx defang slink scen srad bpose bwidth begin
            desc = KinModelDesc(L, pointer(parent), pointer(jtype), pointer(pose), pointer(axis), pointer(qidx),
                                pointer(defang), length(joints), m.with_base, S, pointer(slink), pointer(scen),
                                pointer(srad), B, pointer(bpose), pointer(bwidth))
            check(ccall((:kin_model_create, libkin), Cint, (Ref{KinModelDesc}, Ref{Ptr{Cvoid}}), desc, handle))
        end
        dm = new(handle[], length(joints) + (m.with_base ? 3 : 0), S)
        finalizer(x -> ccall((:kin_model_destroy, libkin), Cint, (Ptr{Cvoid},), x.handle), dm)
        return dm
    end
end

# the obstacle moved (sdf.jl:14-32): same number of boxes => the box rows are rewritten in place, nothing recompiles
function set_boxes!(dm::DeviceMechanism, sdf::AbstractSDF)
    B, bpose, bwidth = box_tables(sdf)
    GC.@preserve bpose bwidth check(ccall((:kin_model_set_boxes, libkin), Cint, (Ptr{Cvoid}, Cint, Ptr{Cdouble}, Ptr{Cdouble}),
                                          dm.handle, B, pointer(bpose), pointer(bwidth)))
end

# Extension (no reference counterpart: the reference's SDFs are boxes, sdf.jl:92-94): a table of mixed primitives.
# kinds[i] = 0 box (size = widths) | 1 sphere (radius, -, -) | 2 cylinder along local z (radius, length, -);
# pose (16, n) column-major world poses, size (3, n).
function set_primitives!(dm::DeviceMechanism, kinds::Vector{Cint}, pose::Matrix{Cdouble}, size_::Matrix{Cdouble})
    @assert size(pose) == (16, length(kinds)) && size(size_) == (3, length(kinds))
    GC.@preserve kinds pose size_ check(ccall((:kin_model_set_primitives, libkin), Cint,
        (Ptr{Cvoid}, Cint, Ptr{Cint}, Ptr{Cdouble}, Ptr{Cdouble}), dm.handle, length(kinds), pointer(kinds), pointer(pose), pointer(size_)))
end

function make_call(dm, Q, layout, fk_links, T, jac_links, J, with_rot, rpy_jac, keep_irrelevant, vals, grads, argmin,
                   truncation_dist, grad_mode, scratch_mode, vals_offset, qptr, dptr, stream)
    N = nbatch(Q, layout)
    @assert (layout === :soa ? size(Q, 2) : size(Q, 1)) == dm.n_dof
    KinCall(KIN_F64, layout_code(layout), N, 0, qptr(Q), length(fk_links), pointer(fk_links), dptr(T),
            length(jac_links), pointer(jac_links), with_rot, rpy_jac, keep_irrelevant, dptr(J), truncation_dist, grad_mode,
            scratch_mode, dptr(vals), dptr(grads), argmin === nothing ? CuPtr{Cint}(0) : reinterpret(CuPtr{Cint}, dptr(argmin)),
            vals_offset, stream)
end

# One fused kin_eval on device arrays.
function eval!(dm::DeviceMechanism, Q::CuMatrix{Float64}; layout::Symbol=:soa, fk_links=Cint[], T=nothing, jac_links=Cint[],
               J=nothing, with_rot=true, rpy_jac=false, keep_irrelevant=false, vals=nothing, grads=nothing, argmin=nothing,
               truncation_dist=Inf, grad_mode=KIN_GRAD_FD, scratch_mode=KIN_SCRATCH_REFERENCE, vals_offset=0.0)
    dptr(x) = x === nothing ? CuPtr{Cvoid}(0) : reinterpret(CuPtr{Cvoid}, pointer(x))
    GC.@preserve fk_links jac_links begin
        call = make_call(dm, Q, layout, fk_links, T, jac_links, J, with_rot, rpy_jac, keep_irrelevant, vals, grads, argmin,
                         truncation_dist, grad_mode, scratch_mode, vals_offset, dptr, dptr, cuda_stream())
        check(ccall((:kin_eval, libkin), Cint, (Ptr{Cvoid}, Ref{KinCall}), dm.handle, call))
    end
end

# The same call on HOST arrays (pageable or pinned `Array`s): the library stages chunks through the device on its own
# streams and returns when every output is in host memory (kin_eval_host).  The pointer fields of KinCall are plain
# addresses, so host pointers are passed in the same slots.
function eval_host!(dm::DeviceMechanism, Q::Matrix{Float64}; layout::Symbol=:soa, fk_links=Cint[], T=nothing, jac_links=Cint[],
                    J=nothing, with_rot=true, rpy_jac=false, keep_irrelevant=false, vals=nothing, grads=nothing, argmin=nothing,
                    truncation_dist=Inf, grad_mode=KIN_GRAD_FD, scratch_mode=KIN_SCRATCH_REFERENCE, vals_offset=0.0)
    hptr(x) = x === nothing ? CuPtr{Cvoid}(0) : CuPtr{Cvoid}(UInt(pointer(x)))
    GC.@preserve Q T J vals grads argmin fk_links jac_links begin
        call = make_call(dm, Q, layout, fk_links, T, jac_links, J, with_rot, rpy_jac, keep_irrelevant, vals, grads, argmin,
                         truncation_dist, grad_mode, scratch_mode, vals_offset, hptr, hptr, C_NULL)
        check(ccall((:kin_eval_host, libkin), Cint, (Ptr{Cvoid}, Ref{KinCall}), dm.handle, call))
    end
end

# get_transform(m, link) for a batch: (N, 12, n_links) [SoA] / (12, n_links, N) [AoS], 3x4 column-major (algorithm.jl:1)
function get_transform(dm::DeviceMechanism, links::Vector{<:Link}, Q::CuMatrix{Float64}; layout::Symbol=:soa)
    ids = Cint[l.id for l in links]
    T = out_array(nbatch(Q, layout), layout, 12, length(links))
    eval!(dm, Q; layout=layout, fk_links=ids, T=T)
    return T
end

# get_jacobian(m, link, joints, with_rot; rpy_jac) for a batch: (N, rows, n_dof) / (rows, n_dof, N) (algorithm.jl:108)
function get_jacobian(dm::DeviceMechanism, link::Link, Q::CuMatrix{Float64}, with_rot::Bool; rpy_jac=false, layout::Symbol=:soa)
    J = out_array(nbatch(Q, layout), layout, with_rot ? 6 : 3, dm.n_dof)
    eval!(dm, Q; layout=layout, jac_links=Cint[link.id], J=J, with_rot=with_rot, rpy_jac=rpy_jac)
    return J
end

# get_jacobian!(m, link, joints, with_rot, mat_out; rpy_jac) (algorithm.jl:83-106): ONLY the columns of joints that move
# `link` (plus the base block) are written, the rest of the caller's array keeps its contents (keep_irrelevant = 1)
function get_jacobian!(dm::DeviceMechanism, link::Link, Q::CuMatrix{Float64}, with_rot::Bool, mat_out::CuArray{Float64, 3};
                       rpy_jac=false, layout::Symbol=:soa)
    rows = with_rot ? 6 : 3
    @assert size(mat_out) == (layout === :soa ? (nbatch(Q, layout), rows, dm.n_dof) : (rows, dm.n_dof, nbatch(Q, layout)))
    eval!(dm, Q; layout=layout, jac_links=Cint[link.id], J=mat_out, with_rot=with_rot, rpy_jac=rpy_jac, keep_irrelevant=true)
    return mat_out
end

# compute_coll_dists (collision.jl:51-65): (N, S) / (S, N)
function compute_coll_dists(dm::DeviceMechanism, Q::CuMatrix{Float64}; layout::Symbol=:soa)
    vals = out_array(nbatch(Q, layout), layout, dm.n_spheres)
    eval!(dm, Q; layout=layout, vals=vals)
    return vals
end

# compute_coll_dists_and_grads (collision.jl:67-103): (N, S), (N, n_dof, S) / (S, N), (n_dof, S, N)
function compute_coll_dists_and_grads(dm::DeviceMechanism, Q::CuMatrix{Float64}; truncation_dist=Inf, grad_mode=KIN_GRAD_FD,
                                      scratch_mode=KIN_SCRATCH_REFERENCE, margin=0.0, layout::Symbol=:soa)
    N = nbatch(Q, layout)
    vals = out_array(N, layout, dm.n_spheres)
    grads = out_array(N, layout, dm.n_dof, dm.n_spheres)
    eval!(dm, Q; layout=layout, vals=vals, grads=grads, truncation_dist=truncation_dist, grad_mode=grad_mode,
          scratch_mode=scratch_mode, vals_offset=margin)
    return vals, grads
end

# IneqConst.(xi, val, jac) (planning.jl:55-68) for every waypoint column of Xi (n_dof, n_wp * P), the reference-native
# layout of `reshape(xi, (n_dof, n_wp))`: val = dists - margin (S, n_wp * P), and the (n_dof, S) diagonal blocks of the
# dense jac_mat, stacked along the last axis (n_dof, S, n_wp * P).  truncation_dist = margin + 0.05 as in planning.jl:56.
function ineq_const(dm::DeviceMechanism, Xi::CuMatrix{Float64}, margin::Float64; grad_mode=KIN_GRAD_FD,
                    scratch_mode=KIN_SCRATCH_REFERENCE)
    return compute_coll_dists_and_grads(dm, Xi; truncation_dist=margin + 0.05, grad_mode=grad_mode, scratch_mode=scratch_mode,
                                        margin=margin, layout=:aos)
end

# nloptize (planning.jl:178-185): NLopt's sign convention
nloptize_values(val, jac) = (-val, -jac)

pose_target(t::Transform) = vcat(Vector(translation(t)), Vector(rpy(t)))      # [x y z roll pitch yaw]

function pose_residual(dm::DeviceMechanism, links::Vector{<:Link}, Q::CuMatrix{Float64}, targets::Vector{Transform},
                       with_rots::Vector{Bool}, mode::Cint; layout::Symbol=:soa)
    N = nbatch(Q, layout)
    ids = Cint[l.id for l in links]
    rots = Cint[w ? 1 : 0 for w in with_rots]
    n_cons = sum(w ? 6 : 3 for w in with_rots)
    tg = CuArray(reduce(vcat, pose_target.(targets)))                         # 6 values per link, shared by the batch
    val = mode == KIN_POSE_IK_OBJECTIVE ? CuArray{Float64}(undef, N) : out_array(N, layout, n_cons)
    jac = mode == KIN_POSE_IK_OBJECTIVE ? out_array(N, layout, dm.n_dof) : out_array(N, layout, dm.n_dof, n_cons)
    GC.@preserve ids rots check(ccall((:kin_pose_residual_multi, libkin), Cint,
        (Ptr{Cvoid}, Cint, Cint, CuPtr{Cvoid}, Int64, Cint, Ptr{Cint}, Ptr{Cint}, CuPtr{Cvoid}, Cint, Cint, CuPtr{Cvoid}, CuPtr{Cvoid}, Ptr{Cvoid}),
        dm.handle, KIN_F64, layout_code(layout), pointer(Q), N, length(ids), pointer(ids), pointer(rots), pointer(tg), 0, mode,
        pointer(val), pointer(jac), cuda_stream()))
    return val, jac
end

# f_objective of inverse_kinematics.jl:38-50 for a batch: f = sum(pose_diff.^2) (N,), grad = -2 J' pose_diff (N, n_dof)
f_objective(dm::DeviceMechanism, link::Link, Q::CuMatrix{Float64}, target::Transform; with_rot=true, layout::Symbol=:soa) =
    pose_residual(dm, [link], Q, [target], [with_rot], KIN_POSE_IK_OBJECTIVE; layout=layout)

# PoseConstraint.(q, val, jac) of planning.jl:114-138: all (link, target, with_rot) triples in ONE library call;
# val (N, n_cons), jac_T (N, n_dof, n_cons) = the rows j_start:j_end of the reference's jac_mat
pose_constraint(dm::DeviceMechanism, links::Vector{<:Link}, Q::CuMatrix{Float64}, targets::Vector{Transform},
                with_rots::Vector{Bool}; layout::Symbol=:soa) =
    pose_residual(dm, links, Q, targets, with_rots, KIN_POSE_CONSTRAINT; layout=layout)

# inverse_kinematics! (inverse_kinematics.jl:1-30) for N independent targets at once (kin_ik_solve).  `targets` (6, N):
# [x y z roll pitch yaw] per column, `q0` (n_dof, N) seeds -- the reference-native column-per-problem layout.
# collision=false: the pose objective f_objective (:38-50) under the joint-limit bounds (:52-63), the whole
# Levenberg-Marquardt solve in one kernel launch.  collision=true: the constrained stage (:14-19), dists - margin >= 0
# for the spheres / boxes the DeviceMechanism was created with, from the warm start q0 (pass the result of a
# collision=false solve for the reference's two-stage scheme, :8-13).  Returns (q (n_dof, N), f (N,), iterations (N,),
# dmin (N,) -- the smallest signed sphere distance at q; all zeros without collision).
# self_margin (extension, kin_ik_solve_self): also keep every pair of the self-collision table (set_self_pairs!) at least
# self_margin apart, with or without collision; then a fifth result, self_dmin (N,), the smallest pair distance at q.
function inverse_kinematics_batch(dm::DeviceMechanism, link::Link, targets::CuMatrix{Float64}, q0::CuMatrix{Float64},
                                  joints::Vector{<:Joint}; with_rot=true, iters=100, ftol=1e-10, collision=false, margin=0.02,
                                  coll_weight=100.0, ctol=1e-6, with_base=false, self_margin=nothing)
    N = size(q0, 2)
    @assert size(targets) == (6, N) && size(q0, 1) == dm.n_dof
    lo = Cdouble[lower_limit(j) for j in joints]; hi = Cdouble[upper_limit(j) for j in joints]     # inverse_kinematics.jl:54-55
    with_base && (append!(lo, fill(-Inf, 3)); append!(hi, fill(Inf, 3)))
    q = similar(q0); f = CuArray{Float64}(undef, N); its = CuArray{Cint}(undef, N); dmin = CUDA.zeros(Float64, N)
    self_dmin = self_margin === nothing ? nothing : CuArray{Float64}(undef, N)
    vp(x) = reinterpret(CuPtr{Cvoid}, pointer(x))
    GC.@preserve lo hi begin
        call = KinIkCall(N, link.id, with_rot, iters, ftol, 1e-2, vp(targets), vp(q0), pointer(lo), pointer(hi), vp(q), vp(f),
                         pointer(its), cuda_stream(), collision, 0, margin, coll_weight, ctol, vp(dmin))
        if self_margin === nothing
            check(ccall((:kin_ik_solve, libkin), Cint, (Ptr{Cvoid}, Ref{KinIkCall}), dm.handle, call))
        else
            check(ccall((:kin_ik_solve_self, libkin), Cint, (Ptr{Cvoid}, Ref{KinIkCall}, Cdouble, CuPtr{Cvoid}),
                        dm.handle, call, Float64(self_margin), pointer(self_dmin)))
        end
    end
    return self_margin === nothing ? (q, f, its, dmin) : (q, f, its, dmin, self_dmin)
end

# Several links per problem (extension, kin_ik_solve_links; the reference's inverse_kinematics! places one link):
# `targets` (6 L, N), the 6 values of each link in link order; the objective is the sum of the links' f_objective, a link
# whose with_rots entry is false contributing its 3 position rows.  Everything else and the results as above.
function inverse_kinematics_batch(dm::DeviceMechanism, links::AbstractVector{<:Link}, targets::CuMatrix{Float64},
                                  q0::CuMatrix{Float64}, joints::Vector{<:Joint}; with_rots=fill(true, length(links)),
                                  iters=100, ftol=1e-10, collision=false, margin=0.02, coll_weight=100.0, ctol=1e-6,
                                  with_base=false, self_margin=nothing)
    N = size(q0, 2); L = length(links)
    @assert 1 <= L <= 4 && length(with_rots) == L && size(targets) == (6L, N) && size(q0, 1) == dm.n_dof
    lo = Cdouble[lower_limit(j) for j in joints]; hi = Cdouble[upper_limit(j) for j in joints]
    with_base && (append!(lo, fill(-Inf, 3)); append!(hi, fill(Inf, 3)))
    ids = Cint[l.id for l in links]; rots = Cint[w ? 1 : 0 for w in with_rots]
    q = similar(q0); f = CuArray{Float64}(undef, N); its = CuArray{Cint}(undef, N); dmin = CUDA.zeros(Float64, N)
    self_dmin = self_margin === nothing ? CUDA.zeros(Float64, 1) : CuArray{Float64}(undef, N)
    vp(x) = reinterpret(CuPtr{Cvoid}, pointer(x))
    GC.@preserve lo hi ids rots begin
        call = KinIkCall(N, 0, 0, iters, ftol, 1e-2, vp(targets), vp(q0), pointer(lo), pointer(hi), vp(q), vp(f),
                         pointer(its), cuda_stream(), collision, 0, margin, coll_weight, ctol, vp(dmin))
        check(ccall((:kin_ik_solve_links, libkin), Cint,
                    (Ptr{Cvoid}, Ref{KinIkCall}, Cint, Ptr{Cint}, Ptr{Cint}, Cint, Cdouble, CuPtr{Cvoid}),
                    dm.handle, call, Cint(L), ids, rots, Cint(self_margin === nothing ? 0 : 1),
                    Float64(self_margin === nothing ? 0.0 : self_margin),
                    self_margin === nothing ? CuPtr{Cvoid}(0) : pointer(self_dmin)))
    end
    return self_margin === nothing ? (q, f, its, dmin) : (q, f, its, dmin, self_dmin)
end

# Reductions of compute_coll_dists per configuration (extension): smallest sphere distance, the sphere attaining it
# (1-based, first minimum), hinge cost sum_s max(0, margin - d_s)^2
function collision_summary(dm::DeviceMechanism, Q::CuMatrix{Float64}; layout::Symbol=:soa, margin::Float64=0.0)
    N = nbatch(Q, layout)
    dmin = CuArray{Float64}(undef, N); amin = CuArray{Cint}(undef, N); cost = CuArray{Float64}(undef, N)
    check(ccall((:kin_collision_summary, libkin), Cint,
        (Ptr{Cvoid}, Cint, Cint, CuPtr{Cvoid}, Int64, Cdouble, CuPtr{Cvoid}, CuPtr{Cint}, CuPtr{Cvoid}, Ptr{Cvoid}),
        dm.handle, KIN_F64, layout_code(layout), pointer(Q), N, margin, pointer(dmin), pointer(amin), pointer(cost), cuda_stream()))
    return dmin, amin, cost
end

# Self-collision between the collision spheres (extension: collision.jl is sphere-vs-environment only).  The pair table
# is explicit here: pairs (2, P), column p = 1-based sphere ids (i, j), i != j (the default policy -- no same-link, rigid
# or adjacent pairs -- lives in the Python mirror's self_collision_pairs).  Replacing the sphere table drops it.
function set_self_pairs!(dm::DeviceMechanism, pairs::Matrix{Cint})
    @assert size(pairs, 1) == 2
    GC.@preserve pairs check(ccall((:kin_model_set_self_pairs, libkin), Cint, (Ptr{Cvoid}, Cint, Ptr{Cint}),
                                   dm.handle, size(pairs, 2), pointer(pairs)))
end

n_self_pairs(dm::DeviceMechanism) = Int(ccall((:kin_model_n_self_pairs, libkin), Cint, (Ptr{Cvoid},), dm.handle))

function self_collision!(dm::DeviceMechanism, Q::CuMatrix{Float64}, layout::Symbol, truncation_dist, margin, vals, grads,
                         dmin, amin)
    vp(x) = x === nothing ? CuPtr{Cvoid}(0) : reinterpret(CuPtr{Cvoid}, pointer(x))
    check(ccall((:kin_self_collision, libkin), Cint,
        (Ptr{Cvoid}, Cint, Cint, CuPtr{Cvoid}, Int64, Cdouble, Cdouble, CuPtr{Cvoid}, CuPtr{Cvoid}, CuPtr{Cvoid}, CuPtr{Cint}, Ptr{Cvoid}),
        dm.handle, KIN_F64, layout_code(layout), pointer(Q), nbatch(Q, layout), truncation_dist, margin, vp(vals), vp(grads),
        vp(dmin), amin === nothing ? CuPtr{Cint}(0) : pointer(amin), cuda_stream()))
end

# d_p = |c_i - c_j| - r_i - r_j per pair: (N, P) / (P, N)
function compute_self_coll_dists(dm::DeviceMechanism, Q::CuMatrix{Float64}; layout::Symbol=:soa)
    vals = out_array(nbatch(Q, layout), layout, n_self_pairs(dm))
    self_collision!(dm, Q, layout, Inf, 0.0, vals, nothing, nothing, nothing)
    return vals
end

# ... and d d_p / d q = u' (J_i - J_j), u = (c_i - c_j) / |c_i - c_j| (0 when the centres coincide); d_p > truncation_dist
# gives truncation_dist and a zero gradient, then margin is subtracted: (N, P), (N, n_dof, P) / (P, N), (n_dof, P, N)
function compute_self_coll_dists_and_grads(dm::DeviceMechanism, Q::CuMatrix{Float64}; truncation_dist=Inf, margin=0.0,
                                           layout::Symbol=:soa)
    N, P = nbatch(Q, layout), n_self_pairs(dm)
    vals = out_array(N, layout, P)
    grads = out_array(N, layout, dm.n_dof, P)
    self_collision!(dm, Q, layout, truncation_dist, margin, vals, grads, nothing, nothing)
    return vals, grads
end

# the smallest untruncated d_p per configuration and the first pair attaining it (1-based): 12 bytes written per configuration
function self_collision_summary(dm::DeviceMechanism, Q::CuMatrix{Float64}; layout::Symbol=:soa)
    N = nbatch(Q, layout)
    dmin = CuArray{Float64}(undef, N); amin = CuArray{Cint}(undef, N)
    self_collision!(dm, Q, layout, Inf, 0.0, nothing, nothing, dmin, amin)
    return dmin, amin
end

# sdf(p) and gradient!(sdf, p, out) (sdf.jl:34-41, 67-74, 108-119) for a batch of points P (N, 3) [SoA] / (3, N) [AoS]
function sdf_points(sdf::AbstractSDF, P::CuMatrix{Float64}; layout::Symbol=:soa, with_grad=false, grad_mode=KIN_GRAD_FD)
    N = nbatch(P, layout)
    B, bpose, bwidth = box_tables(sdf)
    vals = CuArray{Float64}(undef, N)
    grads = with_grad ? out_array(N, layout, 3) : nothing
    argmin = CuArray{Cint}(undef, N)
    GC.@preserve bpose bwidth check(ccall((:kin_sdf_points, libkin), Cint,
        (Cint, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Cint, CuPtr{Cvoid}, Int64, Cint, CuPtr{Cvoid}, CuPtr{Cvoid}, CuPtr{Cint}, Ptr{Cvoid}),
        B, pointer(bpose), pointer(bwidth), KIN_F64, layout_code(layout), pointer(P), N, grad_mode, pointer(vals),
        grads === nothing ? CuPtr{Cvoid}(0) : pointer(grads), pointer(argmin), cuda_stream()))
    return with_grad ? (vals, grads, argmin) : vals
end
sdf_gradient(sdf::AbstractSDF, P::CuMatrix{Float64}; layout::Symbol=:soa, grad_mode=KIN_GRAD_FD) =
    sdf_points(sdf, P; layout=layout, with_grad=true, grad_mode=grad_mode)[2]

end # module

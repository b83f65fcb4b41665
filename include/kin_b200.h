/*
 * kin_b200.h -- C ABI of libkin_b200.so, the B200 (sm_100a) backend for the data-parallel hot
 * path of HiroIshida/Kinematics.jl: batched forward kinematics, geometric / Euler-rate Jacobians
 * and the sphere-vs-box-SDF collision cost + gradient.
 *
 * The reference has NO FFI on this path (it is plain Julia, SURVEY 8b); the functions below are
 * what a `CUDABackend` Julia module binds with `ccall` (julia/CUDABackend.jl, INTEGRATION.md) and
 * what the Python host mirror binds with ctypes.  Each entry point names the reference function
 * it replaces (paths relative to the reference's src/).
 *
 * Conventions
 *   - every function returns 0 on success, a negative KinStatus otherwise; the text of the last
 *     error on the calling thread is kin_last_error().  Nothing throws, nothing calls exit().
 *   - ids are 1-BASED exactly as the reference assigns them: links / joints in URDF document
 *     order (load_urdf.jl:22-32), appended links after them (mechanism.jl:239-243); boxes in
 *     UnionSDF.sdfs order (sdf.jl:84-95); spheres in sscc.sphere_links order (collision.jl:41-48).
 *   - 4x4 matrices are COLUMN-MAJOR, i.e. the memory of the reference's `Transform.mat`
 *     (transform.jl:3-5), so Julia passes `pose.mat` by reference unchanged.
 *   - a "configuration" is the reference's `angles` vector of set_joint_angles
 *     (mechanism.jl:223-231): the n_joints control-joint values in the caller's `joints` order,
 *     followed by (x, y, theta) of the planar base when the model was created with_base.
 *   - batched arrays come in two layouts (KinLayout).  With n_dof = n_joints (+3), for batch N:
 *       KIN_LAYOUT_SOA  batch index fastest:   q[c*ld + n],  T[(l*12+k)*ld + n], ...
 *                       = Julia Array of size (N, n_dof), (N, 12, L), (N, rows, cols, n_req), (N, n_dof, S)
 *       KIN_LAYOUT_AOS  one contiguous record per configuration: q[n*n_dof + c], T[(n*L + l)*12 + k], ...
 *                       = Julia Array of size (n_dof, N), (3, 4, L, N), (rows, cols, n_req, N), (n_dof, S, N)
 *                         i.e. the per-configuration arrays of the reference stacked along a last axis
 *                         (xi of planning.jl:58 is exactly (n_dof, n_wp)).
 *       KIN_LAYOUT_TILED32  AoSoA with 32 configurations per tile: x[((n / 32) * rec + comp) * 32 + n % 32]
 *                       = Julia Array of size (32, rec, cld(N, 32)); every buffer holds whole tiles (N rounded up
 *                         to a multiple of 32).  One warp reads / writes one contiguous block: the fastest layout.
 *     `ld` (batch_stride) is the SoA distance between consecutive components, >= N; 0 means N.
 *   - a transform is written as 3x4 column-major (k = col*3 + row: R columns then t); the constant
 *     bottom row of the reference's 4x4 is not materialised.
 *   - a Jacobian block is (rows, cols) column-major with rows = 3 or 6 and cols = n_dof, columns
 *     in the caller's `joints` order then the 3 base columns (algorithm.jl:83-106).
 *   - collision gradients are (n_dof, n_spheres) column-major per configuration (collision.jl:91).
 *   - all device pointers are caller-owned; calls are asynchronous and ordered on `stream`
 *     (a cudaStream_t passed as void*; NULL = legacy default stream).
 *   - a KinModel is immutable after creation except through kin_model_set_boxes /
 *     kin_model_set_spheres (which must not race with launches that use the model); concurrent
 *     kin_eval calls on different streams are allowed.  One model per device.
 *   - which kernel runs is the library's business and never changes a result bit: batches of >= 32768 configurations
 *     (and small batches that keep coming) run kernels generated for the model and compiled with NVRTC on first use
 *     (see kin_jit_status below); everything else, and every call when NVRTC is unavailable, runs the interpreting
 *     kernel.
 *   - KIN_LAYOUT_TILED32 buffers hold WHOLE tiles: the kernels may write the padding slots of the last tile.
 */
#ifndef KIN_B200_H
#define KIN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KIN_B200_ABI_VERSION 4

#if defined(__GNUC__)
#define KIN_API __attribute__((visibility("default")))
#else
#define KIN_API
#endif

typedef enum {
    KIN_OK = 0,
    KIN_ERR_INVALID_ARGUMENT = -1,
    KIN_ERR_CUDA = -2,
    KIN_ERR_LIMIT = -3,       /* model exceeds a compiled-in limit (KIN_MAX_*) */
    KIN_ERR_NO_DEVICE = -4,
    KIN_ERR_ALLOC = -5,
    KIN_ERR_UNAVAILABLE = -6  /* the operation needs the run-time compiler (NVRTC) and it is not available */
} KinStatus;

typedef enum { KIN_F64 = 0, KIN_F32 = 1 } KinPrecision;
typedef enum { KIN_LAYOUT_SOA = 0, KIN_LAYOUT_AOS = 1, KIN_LAYOUT_TILED32 = 2 } KinLayout;
typedef enum { KIN_JOINT_FIXED = 0, KIN_JOINT_REVOLUTE = 1, KIN_JOINT_PRISMATIC = 2 } KinJointType;
/* sdf.jl:34-41,116-119 is a forward difference (eps 1e-7) on the argmin box.
 *   KIN_GRAD_FD         the reference's FD quotient.  Away from the kinks of the box SDF it is computed from the
 *                       closed form of the quotient (series in eps / f, truncation < 1e-12); within 2 eps of a
 *                       kink or 1e-3 of the surface the three perturbed points are evaluated directly.
 *   KIN_GRAD_FD_DIRECT  always evaluates the three perturbed points (what the reference literally does;
 *                       ~10 % slower, agrees with KIN_GRAD_FD to the rounding noise of the FD, ~1e-9).
 *   KIN_GRAD_ANALYTIC   the closed-form gradient of the same box (an extension, off by default). */
typedef enum { KIN_GRAD_FD = 0, KIN_GRAD_ANALYTIC = 1, KIN_GRAD_FD_DIRECT = 2 } KinGradMode;
/* collision.jl:76,90 reuses ONE 3 x n_dof Jacobian scratch across the spheres of a call and
 * get_jacobian! (algorithm.jl:91-96) only overwrites relevant columns, so a sphere inherits the
 * columns of joints that do not move it from the previous non-truncated sphere.
 * KIN_SCRATCH_REFERENCE reproduces that bit for bit in sphere order; KIN_SCRATCH_CLEAN zeroes
 * them (the mathematically correct gradient). */
typedef enum { KIN_SCRATCH_REFERENCE = 0, KIN_SCRATCH_CLEAN = 1 } KinScratchMode;

/* SDF primitives.  The reference has boxes only (load_urdf.jl:10-15 prints "primitive type other than box is not
 * supported yet", sdf.jl:92-94 warns); spheres and cylinders are an EXTENSION (SURVEY 8 f4) that plugs into the same
 * contract: value at a point, the generic forward-difference gradient! of sdf.jl:34-41 (or the closed form with
 * KIN_GRAD_ANALYTIC), first-minimum argmin inside a UnionSDF.  A table row of any kind has a pose (the primitive's
 * frame in the world) and a size triple:
 *   KIN_PRIM_BOX       size = full extents (BoxSDF.width)
 *   KIN_PRIM_SPHERE    size = (radius, -, -)
 *   KIN_PRIM_CYLINDER  size = (radius, length, -), axis = local z, centred on the pose (URDF <cylinder>)
 *   KIN_PRIM_GRID      size ignored; a sampled signed-distance grid (KinGrid below), centred on the pose */
typedef enum { KIN_PRIM_BOX = 0, KIN_PRIM_SPHERE = 1, KIN_PRIM_CYLINDER = 2, KIN_PRIM_GRID = 3 } KinPrimKind;

/* Voxel-grid signed distance fields (EXTENSION: what a depth camera, a mesh or a mapping stack delivers).
 * A grid has nx, ny, nz >= 2 float32 samples at spacing s > 0, x fastest: v[(k*ny + j)*nx + i] (a Julia
 * Array{Float32}(nx, ny, nz), numpy (nz, ny, nx) in C order).  Centred on its row's pose: sample (i, j, k) sits at the
 * local point ((i - (nx-1)/2) s, (j - (ny-1)/2) s, (k - (nz-1)/2) s).  At a world point p, per axis:
 *   l = inv_pose * p,  u = fma(l, 1/s, (n-1)/2),  c = clamp(u, 0, n-1),  i0 = min(floor(c), n-2),  t = c - i0
 *   f = trilinear interpolation of the 8 corners of cell i0, each widened exactly to the call's precision, in the
 *       order  a_jk = lerp(v_0jk, v_1jk, t_x),  b_k = lerp(a_0k, a_1k, t_y),  f = lerp(b_0, b_1, t_z)
 *       with lerp(a, b, t) = fma(t, b - a, a)
 *   d = fma(s, |u - c|, f): outside the grid box the distance to the box is added, so d is continuous everywhere
 *       and finite far away; inside, d = f.
 * A grid row competes in the union's first-minimum argmin like every other kind.  Gradients: KIN_GRAD_FD /
 * KIN_GRAD_FD_DIRECT take the generic forward difference (eps 1e-7, against the cached value); KIN_GRAD_ANALYTIC the
 * gradient of d in the chosen cell: (1/s) df/dt on the axes where u lies in [0, n-1], (u - c) / |u - c| on the others,
 * rotated to the world (R * g_local).  FP64 calls interpolate in double and FP32 calls in float; the samples are float32
 * in both.  The kernels read the corners through L1 / L2 (never shared memory): a 1-2 cm grid of a room is MBs to tens
 * of MBs and stays resident in the B200's 126 MB L2. */
typedef struct KinGrid KinGrid;
#define KIN_MAX_GRID_VALUES (1 << 28)   /* nx * ny * nz: 1 GB of samples */

#define KIN_MAX_LINKS 512
#define KIN_MAX_JOINTS 32          /* control joints (bitmask width), base columns excluded */
#define KIN_MAX_SPHERES 512
#define KIN_MAX_BOXES 128
/* Self-collision pairs per model (kin_model_set_self_pairs).  The kernel does not stage the table: every lane of a warp
 * loads the same 8-byte entry at the same time (one broadcast load through L1), so the table costs no shared memory and
 * no occupancy.  4096 pairs are 32 KB, a table that stays resident in L1 beside the collision kernels' shared scratch,
 * and hold every pair of 91 spheres -- several times the pair counts of the default policy on the models here. */
#define KIN_MAX_SELF_PAIRS 4096

typedef struct KinModel KinModel;

/*
 * Flattened mechanism: what load_urdf.jl:20-80 + mechanism.jl:147-181 hold as Link / Joint
 * objects, as tables indexed by link (0-based position i <-> reference link id i+1).
 * All pointers are HOST memory and are copied; they may be freed after kin_model_create.
 */
typedef struct {
    int32_t n_links;
    const int32_t *parent_link;   /* [n_links] 1-based id of the parent link, -1 for the root (Link.plink_id) */
    const int32_t *joint_type;    /* [n_links] KinJointType of the link's parent joint (root: fixed) */
    const double *joint_pose;     /* [n_links][16] column-major Joint.pose (mechanism.jl:79), root: ignored */
    const double *joint_axis;     /* [n_links][3]  unit axis in the joint frame (fixed: ignored) */
    const int32_t *q_index;       /* [n_links] 0-based column of the configuration that drives the parent
                                     joint (position in the caller's `joints` vector), or -1: the joint is
                                     not controlled and sits at default_angle (Mechanism.angles) */
    const double *default_angle;  /* [n_links] */
    int32_t n_joints;             /* number of control joints D (length of `joints`) */
    int32_t with_base;            /* Mechanism.with_base: 3 extra columns (x, y, theta), transform.jl:33-37 */

    /* swept-sphere table: SweptSphereCollisionChecker (collision.jl:32-49). A sphere is a link
     * attached to sphere_link through a fixed joint of pure translation sphere_center. */
    int32_t n_spheres;
    const int32_t *sphere_link;   /* [n_spheres] 1-based link id of the parent link */
    const double *sphere_center;  /* [n_spheres][3] in the parent link frame */
    const double *sphere_radius;  /* [n_spheres] */

    /* UnionSDF of boxes (sdf.jl:48-114): world pose and full widths; a single BoxSDF is n_boxes = 1 */
    int32_t n_boxes;
    const double *box_pose;       /* [n_boxes][16] column-major world pose (BoxSDF.pose) */
    const double *box_width;      /* [n_boxes][3] full extents (BoxSDF.width) */
} KinModelDesc;

/*
 * One batched evaluation.  Any output pointer may be NULL, then that part is skipped.
 * What is computed per configuration:
 *   T_out     get_transform(m, link) for each fk_links[i]          (algorithm.jl:1-37)
 *   J_out     get_jacobian(m, link, joints, with_rot; rpy_jac)     (algorithm.jl:83-114) for each jac_links[i]
 *   vals_out  compute_coll_dists[_and_grads]!                      (collision.jl:51-58, 67-94)
 *   grads_out                                                      (collision.jl:67-94)
 *   argmin_out  UnionSDF.min_idx_cache per sphere, 1-based         (sdf.jl:112)
 */
typedef struct {
    int32_t precision;         /* KinPrecision: element type of q and of every floating output */
    int32_t layout;            /* KinLayout of q and of every output */
    int64_t n;                 /* batch size N */
    int64_t batch_stride;      /* SoA only: ld (>= n), 0 => n */
    const void *q;             /* DEVICE: configurations, n_dof = n_joints (+3) per configuration */

    int32_t n_fk_links;        /* 0 => no FK output */
    const int32_t *fk_links;   /* HOST [n_fk_links] 1-based link ids, output order */
    void *T_out;               /* DEVICE 12 * n_fk_links per configuration */

    int32_t n_jac_links;
    const int32_t *jac_links;  /* HOST [n_jac_links] 1-based link ids */
    int32_t with_rot;          /* rows = with_rot ? 6 : 3 */
    int32_t rpy_jac;           /* rows 4:6 = Euler-rate map (algorithm.jl:56-63) instead of the axis */
    int32_t keep_irrelevant;   /* 1 => get_jacobian! semantics: columns of joints that do not move the
                                  link are NOT written (caller's buffer keeps its values); 0 => zeros */
    void *J_out;               /* DEVICE rows * n_dof * n_jac_links per configuration */

    double truncation_dist;    /* collision.jl:68; +inf => never truncate */
    int32_t grad_mode;         /* KinGradMode */
    int32_t scratch_mode;      /* KinScratchMode */
    void *vals_out;            /* DEVICE n_spheres per configuration */
    void *grads_out;           /* DEVICE n_dof * n_spheres per configuration; NULL => dists only */
    int32_t *argmin_out;       /* DEVICE n_spheres int32 per configuration, or NULL */
    double vals_offset;        /* subtracted from every value written to vals_out: planning.jl:66
                                  (`dists .- margin`); 0 for the plain collision call */

    void *stream;              /* cudaStream_t */
} KinCall;

KIN_API const char *kin_last_error(void);
KIN_API int kin_abi_version(void);
/* Hex digest of the sources the library was compiled from (csrc/ and this header, baked in with -DKIN_BUILD_ID by
 * kinematics.jl_b200/lib.py: build).  The Python host refuses a library whose id differs from the sources beside
 * it, so a stale prebuilt binary cannot be loaded silently. */
KIN_API const char *kin_build_id(void);
/* 1 when the library was compiled with -DKIN_DEBUG (bounds checks on every table / scratch index inside the
 * kernels -- the analogue of the reference's @debugassert, Kinematics.jl:25-30; a violation traps). */
KIN_API int kin_debug_build(void);

/* load_urdf.jl:20-80 / mechanism.jl:147-181 -> device tables on the CURRENT cuda device */
KIN_API int kin_model_create(const KinModelDesc *desc, KinModel **out);
KIN_API int kin_model_destroy(KinModel *model);
/* add_coll_links (collision.jl:39-49): replaces the whole sphere table */
KIN_API int kin_model_set_spheres(KinModel *model, int32_t n_spheres, const int32_t *sphere_link,
                          const double *sphere_center, const double *sphere_radius);
/* UnionSDF / BoxSDF poses after the obstacle moved (sdf.jl:14-32): replaces the whole box table */
KIN_API int kin_model_set_boxes(KinModel *model, int32_t n_boxes, const double *box_pose, const double *box_width);
/* The same table with mixed primitive kinds (kinds[n]: KinPrimKind; NULL = all boxes; size[n][3] as described at
 * KinPrimKind).  A table with a sphere / cylinder row makes the specialised kernels carry one warp-uniform test per
 * row; box-only tables compile exactly the code they always did. */
KIN_API int kin_model_set_primitives(KinModel *model, int32_t n, const int32_t *kinds, const double *pose, const double *size);
/* kin_model_set_primitives with voxel-grid rows: grids[n] is non-null exactly on the KIN_PRIM_GRID rows (whose size is
 * not read); grids == NULL is kin_model_set_primitives.  The model keeps its own reference to every grid it names, so
 * the caller may kin_grid_destroy its handle at once.  Errors before anything changes (KIN_ERR_INVALID_ARGUMENT): a grid
 * row without a grid, a grid on another row, a grid created on another device than the model. */
KIN_API int kin_model_set_scene(KinModel *model, int32_t n, const int32_t *kinds, const double *pose, const double *size,
                                const KinGrid *const *grids);
/* Creates a grid on the CURRENT device from nx*ny*nz float32 samples (host or device memory; copied with
 * cudaMemcpyAsync on the legacy default stream, then synchronised).  Errors: a dimension < 2, a spacing that is not
 * positive and finite, null values (KIN_ERR_INVALID_ARGUMENT); nx*ny*nz > KIN_MAX_GRID_VALUES (KIN_ERR_LIMIT). */
KIN_API int kin_grid_create(int32_t nx, int32_t ny, int32_t nz, double spacing, const float *values, KinGrid **out);
/* Rewrites the samples in place (host or device memory, ordered on `stream`), e.g. a perception refresh.  Must not race
 * with launches that read the grid, the rule of kin_model_set_boxes; nothing is recompiled. */
KIN_API int kin_grid_set_values(KinGrid *grid, const float *values, void *stream);
/* Releases the caller's reference; the storage goes with the last reference (the models whose table names it). */
KIN_API int kin_grid_destroy(KinGrid *grid);
KIN_API int kin_model_n_dof(const KinModel *model);      /* n_joints (+3) */
KIN_API int kin_model_n_spheres(const KinModel *model);
KIN_API int kin_model_n_boxes(const KinModel *model);

/* The fused entry point: FK + Jacobians + collision in one pass over the batch. */
KIN_API int kin_eval(KinModel *model, const KinCall *call);

/* Same call with HOST q / outputs (pageable or pinned): the library stages chunks through its own
 * device and pinned buffers on internal streams (H2D, kernel and D2H of consecutive chunks overlap)
 * and returns when every output is in host memory.  `stream` is ignored. */
KIN_API int kin_eval_host(KinModel *model, const KinCall *call);

/* SoA calls: the rows of T_out / J_out that do not depend on the configuration (links no control joint moves, zero /
 * unit rotation entries, Jacobian columns of joints that do not move the link -- known to the code generator) are not
 * copied back over PCIe, which is what bounds this call: up to 4 host threads (KIN_HOST_FILL_THREADS) write them into
 * the caller's arrays while the device produces the rest.  The values are the ones the kernels write (up to the sign of
 * a zero).  keep_irrelevant = 1 and KIN_HOST_NO_CONST_FILL=1 opt out.
 * Likewise the rows that hold the same variable of the generated code as an earlier row, possibly negated (rotation
 * blocks of links joined by fixed pure-translation joints, geometric Jacobian rows 4:6 that are a column of a link
 * rotation, ...): the first occurrence crosses PCIe, up to 6 host threads (KIN_HOST_DUP_THREADS) copy / negate it into
 * the other rows behind each staging chunk; bit-identical by construction.  KIN_HOST_NO_DUP_COPY=1 opts out.
 * Under torchrun (LOCAL_WORLD_SIZE ranks on one host) the thread counts are scaled to this rank's share of the cores.
 * kin_host_transfer_bytes: bytes kin_eval_host moved host -> device, device -> host, and filled on the host, since load. */
KIN_API int kin_host_transfer_bytes(int64_t *h2d, int64_t *d2h, int64_t *host_filled);

/* Convenience wrappers with the names of SURVEY 8b; each fills a KinCall and calls kin_eval. */
/* get_transform, algorithm.jl:1 */
KIN_API int kin_fk_links(KinModel *model, int32_t precision, int32_t layout, const void *q, int64_t n,
                 const int32_t *link_ids, int32_t n_req, void *T_out, void *stream);
/* get_transform + get_jacobian, algorithm.jl:1,108 */
KIN_API int kin_fk_jacobian(KinModel *model, int32_t precision, int32_t layout, const void *q, int64_t n,
                    const int32_t *link_ids, int32_t n_req, int32_t with_rot, int32_t rpy_jac,
                    void *T_out, void *J_out, void *stream);
/* compute_coll_dists! / compute_coll_dists_and_grads!, collision.jl:51,67 */
KIN_API int kin_collision(KinModel *model, int32_t precision, int32_t layout, const void *q, int64_t n,
                  double truncation_dist, int32_t grad_mode, int32_t scratch_mode,
                  void *vals_out, void *grads_out, int32_t *argmin_out, void *stream);

/* Per-configuration reductions of compute_coll_dists! (collision.jl:51-58; an extension -- what a sampling-based planner
 * or a penalty method consumes instead of the S individual distances), untruncated distances d_s = sdf(c_s) - r_s:
 *   dmin_out[N]  min_s d_s                       amin_out[N]  the sphere attaining it, 1-based, first minimum (nullable)
 *   cost_out[N]  sum_s max(0, margin - d_s)^2    (nullable)
 * q in `layout`; the outputs are plain [N] arrays of the call's precision (amin: int32).  The distances go through a
 * stream-ordered temporary in chunks of 2^20 configurations and are reduced by coll_summary_kernel (AoS: one group of
 * lanes per configuration, warp-shuffle min / argmin / sum; SoA, tiled: one thread per configuration). */
KIN_API int kin_collision_summary(KinModel *model, int32_t precision, int32_t layout, const void *q, int64_t n, double margin,
                                  void *dmin_out, int32_t *amin_out, void *cost_out, void *stream);

/* Self-collision between the model's collision spheres (an EXTENSION: collision.jl has sphere-vs-environment only).
 * The model holds a table of P sphere pairs (i, j).  Per configuration and pair p, with world centres c_i, c_j and radii
 * r_i, r_j:
 *   L = |c_i - c_j|,  d_p = L - r_i - r_j
 *   grad_p[k] = u . (J_i[:,k] - J_j[:,k]),  u = (c_i - c_j) / L,  J_s = 3 x n_dof positional Jacobian of sphere s's centre
 *               (zero in the columns that do not move s).  When L == 0 the gradient is 0.
 *   truncation as collision.jl:84-86: d_p > truncation_dist -> value truncation_dist, gradient 0; then vals_offset is
 *   subtracted from every written value (IneqConst's d - margin directly).
 *   dmin[n] = min_p d_p (untruncated, no offset), amin[n] = 1-based index of the first pair attaining it, in table order.
 * No box table is needed.  One kernel launch per call: phase 1 of kin_eval (FK, joint frames, sphere centres) followed by
 * the pair loop, for every batch size, precision and layout. */
/* replaces the model's self-collision pair table; pairs[n_pairs][2] = 1-based sphere ids, i != j, both <= n_spheres.
 * n_pairs = 0 removes it.  kin_model_set_spheres removes it too (its ids would be stale); set_boxes / set_primitives keep it. */
KIN_API int kin_model_set_self_pairs(KinModel *model, int32_t n_pairs, const int32_t *pairs);
KIN_API int kin_model_n_self_pairs(const KinModel *model);
/* vals_out: P per configuration; grads_out: (n_dof, P) column-major per configuration; dmin_out [N]; amin_out [N].
 * Every output is nullable, but at least one of vals_out / dmin_out must be given.  Layout and precision as kin_collision
 * (vals / grads in `layout`, dmin / amin plain [N] arrays; amin int32).  A call with dmin / amin only writes those. */
KIN_API int kin_self_collision(KinModel *model, int32_t precision, int32_t layout, const void *q, int64_t n,
                               double truncation_dist, double vals_offset, void *vals_out, void *grads_out,
                               void *dmin_out, int32_t *amin_out, void *stream);

/* BoxSDF / UnionSDF call and gradient! at arbitrary points (sdf.jl:34-41, 67-74, 108-119): for a
 * union of n_boxes boxes (HOST tables, same format as KinModelDesc), pts (DEVICE, N points x 3
 * components in `layout`) -> vals_out[N], grads_out (3 per point in `layout`, nullable),
 * argmin_out[N] (1-based box index, nullable). */
KIN_API int kin_sdf_points(int32_t n_boxes, const double *box_pose, const double *box_width, int32_t precision,
                   int32_t layout, const void *pts, int64_t n, int32_t grad_mode, void *vals_out,
                   void *grads_out, int32_t *argmin_out, void *stream);

/* ... for a union of mixed primitives (kinds / size as in kin_model_set_primitives) */
KIN_API int kin_sdf_points_prims(int32_t n, const int32_t *kinds, const double *pose, const double *size, int32_t precision,
                                 int32_t layout, const void *pts, int64_t n_pts, int32_t grad_mode, void *vals_out,
                                 void *grads_out, int32_t *argmin_out, void *stream);
/* ... with voxel-grid rows (grids as in kin_model_set_scene; every grid on the current device) */
KIN_API int kin_sdf_points_scene(int32_t n, const int32_t *kinds, const double *pose, const double *size,
                                 const KinGrid *const *grids, int32_t precision, int32_t layout, const void *pts, int64_t n_pts,
                                 int32_t grad_mode, void *vals_out, void *grads_out, int32_t *argmin_out, void *stream);

/* Pose residuals of one link against target poses -- the per-iteration evaluations of the IK and
 * planning callers:
 *   KIN_POSE_IK_OBJECTIVE  inverse_kinematics.jl:38-50: e = [p_t - p; rpy_t - rpy] (3 or 6 rows),
 *                          val_out[N] = sum(e.^2), jac_out (n_dof per configuration) = -2 J' e
 *   KIN_POSE_CONSTRAINT    planning.jl:114-138: val_out (dim = 3|6 per configuration) = [p - p_t; rpy - rpy_t],
 *                          jac_out ((n_dof, dim) column-major per configuration) = transpose of the Jacobian
 * J is the Euler-rate Jacobian (rpy_jac = true), rpy = [roll, pitch, yaw] of RotZYX (transform.jl:45-48).
 * target: DEVICE, [x, y, z, roll, pitch, yaw] per configuration in `layout` (6 components), or ONE
 * target shared by the batch when target_per_config == 0 (6 contiguous values). */
typedef enum { KIN_POSE_IK_OBJECTIVE = 0, KIN_POSE_CONSTRAINT = 1 } KinPoseMode;
KIN_API int kin_pose_residual(KinModel *model, int32_t precision, int32_t layout, const void *q, int64_t n,
                              int32_t link_id, const void *target, int32_t target_per_config, int32_t with_rot,
                              int32_t mode, void *val_out, void *jac_out, void *stream);
/* The whole (link, target, with_rot) loop of one PoseConstraint (planning.jl:124-137) in one call: n_links
 * links (HOST ids / flags), target = 6 values per link, per configuration (6 * n_links components in `layout`) or
 * shared (6 * n_links contiguous values).  With n_cons = sum(with_rots[l] ? 6 : 3):
 *   KIN_POSE_CONSTRAINT    val_out (n_cons per configuration) = the stacked pose differences, jac_out ((n_dof, n_cons)
 *                          column-major per configuration) = the rows j_start:j_end of the reference's jac_mat
 *   KIN_POSE_IK_OBJECTIVE  val_out[N] = sum over links of sum(e.^2), jac_out (n_dof) = its gradient
 * Two kernel launches in total (kin_eval for the n_links transforms + Euler-rate Jacobians, then the residuals). */
KIN_API int kin_pose_residual_multi(KinModel *model, int32_t precision, int32_t layout, const void *q, int64_t n,
                                    int32_t n_links, const int32_t *link_ids, const int32_t *with_rots, const void *target,
                                    int32_t target_per_config, int32_t mode, void *val_out, void *jac_out, void *stream);

/* The whole batched IK solve of config 4 in ONE kernel launch (device-resident loop; no host round trip per
 * iteration) -- for n >= 16384 in a few launches ("stages" of 3, 4, 6, 9 and the remaining iterations; KIN_IK_STAGES)
 * over the still-running problems, whose index list is compacted between stages (its length, 8 bytes, is read back:
 * the call then synchronises `stream` once per stage); the iterates are the ones of the single launch, bit for bit.  One thread per problem runs up to `iters` Levenberg-Marquardt iterations on the reference's objective
 * f = |[p - p_t; rpy - rpy_t]|^2 (inverse_kinematics.jl:38-50; angle residuals wrapped to (-pi, pi]) with the joint
 * limits as bounds (inverse_kinematics.jl:52-63: active set + clamping) and stops on its own when f < ftol.  The
 * kernel is generated for this model / link (straight-line FK + Euler-rate Jacobian, csrc/kin_codegen.cpp) and
 * compiled with NVRTC on first use; without NVRTC the same method runs as one kin_eval + one step kernel per
 * iteration (the loop of the collision-constrained solve below, without spheres).  FP64, per-problem contiguous
 * arrays (AoS), DEVICE pointers:
 * targets[n][6] = x y z roll pitch yaw, q0 / q_out [n][n_dof], f_out[n], iters_out[n] (nullable); lower / upper are
 * HOST [n_dof] (+-inf allowed, NULL = unbounded).  n_dof <= 20 (up to 12 columns the normal
 * equations of a problem live in registers; above, in local memory). */
typedef struct {
    int64_t n;
    int32_t link_id;           /* 1-based id of the link to place */
    int32_t with_rot;          /* 6 residual rows (position + rpy) or 3 */
    int32_t iters;             /* maximum number of iterations */
    double ftol;               /* a problem stops when f < ftol */
    double lambda0;            /* initial damping (<= 0: 1e-2) */
    const void *targets;
    const void *q0;
    const double *lower;
    const double *upper;
    void *q_out;
    void *f_out;
    int32_t *iters_out;
    void *stream;
    /* ---- collision-constrained solve (ABI version 3) ----
     * collision != 0: the reference's two-stage problem (inverse_kinematics.jl:8-19): the pose objective subject to
     * dists(q) - margin >= 0 for every sphere of the model's sphere table against the model's boxes (IneqConst with
     * margin 0.02 in the reference), q0 being the warm start (normally the result of a collision == 0 solve).  The
     * constraint is enforced by an augmented-Lagrangian Levenberg-Marquardt iteration (csrc/kin_ik_coll.cuh): per
     * iteration ONE kin_eval over the batch (link transform + Euler-rate Jacobian + sphere distances and gradients,
     * truncated at margin + 0.05 as planning.jl:56, forward-difference SDF gradient, clean Jacobian scratch) and ONE
     * step kernel (accept / multiplier update / normal equations / Cholesky), `iters` iterations at most.  For
     * n >= 4096 the still-running problems are compacted into an active list at iterations 1, 2, 3, 4, 6, 8, 12, 16,
     * 24, ... and the list length (8 bytes) is read back, so that later iterations cover only them: the call then
     * synchronises `stream` about ten times (KIN_IK_NO_COMPACT=1: fully asynchronous, every iteration over the whole batch).  A problem stops when f < ftol and every dist >= margin - ctol.  Works without NVRTC (the
     * interpreting kernels evaluate).  ~ (30 + 21 n_dof + 2 S + S n_dof) * 8 bytes of stream-ordered scratch per problem. */
    int32_t collision;
    int32_t reserved_;
    double margin;             /* the reference uses 0.02 */
    double coll_weight;        /* penalty parameter mu of the augmented Lagrangian (<= 0: 100) */
    double ctol;               /* constraint tolerance (<= 0: 1e-6) */
    void *dmin_out;            /* DEVICE [n], nullable: min over spheres of the UNtruncated signed distance at q_out */
} KinIkCall;
KIN_API int kin_ik_solve(KinModel *model, const KinIkCall *call);
/* kin_ik_solve with the extra hard constraint d_p(q) - self_margin >= 0 for every pair p of the model's self-collision
 * table (kin_model_set_self_pairs; d_p as kin_self_collision).  Everything else as kin_ik_solve with the AL loop:
 * with call->collision != 0 the sphere-vs-box constraint applies too; with call->collision == 0 only the pairs do,
 * and the model needs spheres + a pair table but no boxes.  self_dmin_out: DEVICE [n], nullable: min over pairs of
 * the untruncated d_p at q_out.
 * Per iteration: kin_eval (pose, + spheres with collision), ONE kin_self_collision launch over the same active list
 * (pair values and gradients, truncated at self_margin + 0.05), the step kernel; the pairs share the penalty parameter
 * coll_weight with the spheres, and a problem stops when f < ftol and every sphere and pair holds to ctol.  The
 * constraint-free pose-only solve is never used here.  Errors, before anything is launched: no pair table or a NaN
 * self_margin (KIN_ERR_INVALID_ARGUMENT), collision != 0 without spheres / boxes (as kin_ik_solve), n_dof > 20
 * (KIN_ERR_LIMIT).  Workspace: on top of kin_ik_solve's, P (n_dof + 2) * 8 bytes of stream-ordered scratch per problem
 * (pair values, gradients and multipliers) -- 23.2 KB on a model of 18 columns and 145 pairs, i.e. 6.1 GB at 2^18
 * problems and 24.3 GB at 2^20; a pool allocation that fails is returned as KIN_ERR_CUDA. */
KIN_API int kin_ik_solve_self(KinModel *model, const KinIkCall *call, double self_margin, void *self_dmin_out);
/* Several links per problem (extension: the reference's inverse_kinematics! places one link).  The objective is
 * f = sum_l |e_l|^2 with e_l = [p_l - p_t,l ; rpy_l - rpy_t,l] (angles wrapped to (-pi, pi]); a link with
 * with_rots[l] == 0 contributes its 3 position rows only -- the stacked pose constraint of kin_pose_residual_multi.
 * link_ids / with_rots: HOST [n_links], 1-based distinct ids.  call->link_id and call->with_rot are not read;
 * call->targets is DEVICE [n][6 n_links], the 6 values of each link in link order (the angles of a position-only link
 * are not read).  Everything else as kin_ik_solve (self_collision == 0: the pose-only solve, or the AL loop with
 * call->collision) or kin_ik_solve_self (self_collision != 0; self_dmin_out nullable); f_out is the sum over the
 * links.  n_links == 1 is bit for bit the call of kin_ik_solve / kin_ik_solve_self.  Errors, before anything is
 * launched: n_links outside 1..KIN_IK_MAX_LINKS, a null array, an id out of range or repeated, a NaN self_margin
 * (KIN_ERR_INVALID_ARGUMENT); self_collision without a pair table, collision without spheres / boxes
 * (KIN_ERR_INVALID_ARGUMENT, as the two single-link calls); n_dof > 20 (KIN_ERR_LIMIT).  Workspace of the AL loop: on
 * top of the single-link solve's, (n_links - 1)(12 + rows n_dof) * 8 bytes of stream-ordered scratch per problem
 * (rows = 6 when any link has rotation, else 3): the links' transforms and Jacobians. */
#define KIN_IK_MAX_LINKS 4
KIN_API int kin_ik_solve_links(KinModel *model, const KinIkCall *call, int32_t n_links, const int32_t *link_ids,
                               const int32_t *with_rots, int32_t self_collision, double self_margin, void *self_dmin_out);

/* Diagnostics for bench.py / tests: kernel launches issued by this library since load, and the
 * static resources of the kernel a call would use (registers / thread, dynamic shared memory bytes /
 * CTA, threads / CTA, CTAs in the grid).  */
KIN_API int64_t kin_launch_count(void);
KIN_API int kin_query_launch(KinModel *model, const KinCall *call, int32_t *regs, int32_t *smem_bytes,
                     int32_t *block, int32_t *grid);

/* Model-specialised kernels.  For batches of >= 32768 configurations (KIN_JIT_MIN_BATCH) in the SoA / tiled layouts
 * the library generates the source of a kernel for this model and these requested outputs (csrc/kin_codegen.cpp: the
 * chain walk becomes straight-line code with the model's constants folded in; results are bit-identical to the
 * interpreting kernels up to the sign of a zero) and compiles it with NVRTC for sm_100a on first use (1-3 s, then
 * cached in the model and on disk under KIN_JIT_CACHE_DIR, default /tmp/kin_b200_jit-<uid>).  libnvrtc is loaded with
 * dlopen (KIN_NVRTC_PATH overrides the search); without it, or with KIN_DISABLE_JIT set, every call runs the
 * ahead-of-time interpreting kernels -- as do AoS calls with keep_irrelevant on batches above 2048 (KIN_MAX_JOINTS = 32
 * columns is the limit of every kernel; on models whose per-thread shared scratch is large -- many columns / spheres --
 * the specialised collision kernels take the launch shape with the most threads per SM that fits).  kin_query_launch reports a NEGATIVE block size for a specialised kernel.
 *   kin_jit_status   "ok: <library> (<version>)" or the reason NVRTC is unavailable
 *   kin_jit_stats    kernels compiled / taken from the disk cache / launched / failed since load
 *   kin_codegen_dump host-only: writes the generated source of the kernel `call` would run (its pointers are only
 *                    tested for NULL) into out_dir; with compile != 0 also the NVRTC cubin + log.  No device needed. */
KIN_API const char *kin_jit_status(void);
KIN_API int kin_jit_stats(int64_t *compiles, int64_t *cache_hits, int64_t *launches, int64_t *failures);
KIN_API int kin_codegen_dump(const KinModelDesc *desc, const KinCall *call, int32_t compile, const char *out_dir);

/* FP64 peak of the current device, measured: 8 independent DFMA chains per thread, 8 x 256 threads per SM.  Returns
 * TFLOP/s (2 flops per DFMA), DFMA per clock per SM at the device's nominal maximum SM clock, and that clock.  This is
 * the denominator of the "FP64 pipe" fractions in DESIGN.md / profiles (SURVEY 6 asks for it). */
KIN_API int kin_probe_fp64(double *tflops_out, double *dfma_per_clk_per_sm_out, double *sm_mhz_out);

/* Host-only (no device needed): compile the kinematic program a call with these requests would run
 * and copy its tables out; the CPU test-suite interprets them against the oracle.  header_out
 * receives the ProgHeader of csrc/kin_program.h as int32 words. */
KIN_API int kin_program_dump(const KinModelDesc *desc, const int32_t *fk_links, int32_t n_fk,
                             const int32_t *jac_links, int32_t n_jac, int32_t want_coll, int32_t want_stale,
                             int32_t *header_out, int32_t header_cap, int32_t *ints_out, int32_t ints_cap,
                             double *reals_out, int32_t reals_cap);

#ifdef __cplusplus
}
#endif
#endif /* KIN_B200_H */

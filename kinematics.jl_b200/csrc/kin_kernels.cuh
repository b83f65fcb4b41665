// kin_kernels.cuh -- the sm_100a kernel of libkin_b200: one pass per configuration over the
// compiled kinematic program (kin_program.h) doing
//   phase 1  forward kinematics of the dynamic nodes (algorithm.jl:1-37, mechanism.jl:90-103),
//            world joint frames (algorithm.jl:42-54), requested link transforms, requested
//            Jacobians (algorithm.jl:56-114) and collision-sphere centres (collision.jl:39-49);
//   phase 2  per sphere, in sscc.sphere_links order: union-of-boxes SDF with first-minimum argmin
//            (sdf.jl:67-74,108-114), truncation, forward-difference or analytic gradient
//            (sdf.jl:34-41,116-119) chain-ruled through the sphere's 3 x n_dof Jacobian
//            (collision.jl:67-94), with the reference's shared-scratch behaviour reproducible.
//
// Mapping: one thread = one configuration.  Everything indexed by a run-time table index lives in
// shared memory as [slot][thread] (bank-conflict free, no local memory); the running transform
// stays in registers.  Program tables are staged once per CTA into shared memory and read with
// warp-uniform (broadcast) loads.  CTAs are persistent over tiles of blockDim configurations.
// SoA outputs are written as full 256-B (f64) / 128-B (f32) warp rows.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>

#include "kin_program.h"
#include "kin_device_math.cuh"

// Debug build (-DKIN_DEBUG, kinematics.jl_b200/lib.py: build(debug=True) -> libkin_b200_debug.so): every table
// index and scratch-slot index the kernels derive from the program tables is range-checked; a violation prints
// the condition and traps.  This is the analogue of the reference's @debugassert (Kinematics.jl:25-30, cache.jl:24,35,
// stack.jl:15,21, algorithm.jl:9-10,43).  compiles to nothing in the release build.
#ifdef KIN_DEBUG
#include <cstdio>
#define KIN_DASSERT(cond)                                                                                   \
    do {                                                                                                    \
        if (!(cond)) {                                                                                      \
            printf("KIN_DEBUG assertion failed: %s (%s:%d, block %d thread %d)\n", #cond, __FILE__, __LINE__, \
                   (int)blockIdx.x, (int)threadIdx.x);                                                      \
            __trap();                                                                                       \
        }                                                                                                   \
    } while (0)
#else
#define KIN_DASSERT(cond) ((void)0)
#endif

namespace kin {

struct KernelArgs {
    ProgHeader h;
    const int32_t *tab_i;       // device: int section
    const void *tab_r;          // device: real section (element type = real)
    const void *q;
    void *T_out, *J_out, *vals_out, *grads_out;
    int32_t *argmin_out;
    long long n, ld;
    int with_rot, rpy_jac, keep_irrelevant;
    int grad_mode, scratch_ref;  // scratch_ref = 1: reproduce the reference's shared Jacobian scratch
    double truncation_dist, vals_offset;
    void *ws_ring;               // kin_eval_ws_kernel only: global hand-over ring (kin_kernels_ws.cuh)
    // self-collision instances only (SELF = true); appended so that the fields above keep their offsets
    const int2 *self_pairs;      // [n_self_pairs] 0-based sphere ids (i, j), read with warp-uniform loads through L1
    void *dmin_out;              // [n] min over pairs of the untruncated distance, nullable
    int32_t *amin_out;           // [n] 1-based pair index of the first minimum, nullable
    int n_self_pairs;
};

// AoS layout only.  A thread owns one record, so a plain store of component k by 32 lanes hits 32
// different sectors.  Instead the warp stages R values per lane in a warp-private shared buffer
// ([k][33] padded) and writes the 32 x R block with the lanes running ALONG the records: consecutive
// lanes write consecutive addresses, every sector is written whole.  `rec0` = address of the block's
// first component in the record of the warp's first configuration, `rec` = record stride (elements),
// `n_valid` = number of lanes whose record exists (lanes past the end re-write the last one).
constexpr int AOS_STAGE_ROWS = 12;
constexpr int AOS_STAGE_REALS = AOS_STAGE_ROWS * 33;
template <typename real, int RMAX>
__device__ __forceinline__ void warp_store_records(real *stage, real *rec0, size_t rec, const real (&v)[RMAX], int R, int lane, int n_valid) {
    #pragma unroll
    for (int k = 0; k < RMAX; ++k)
        if (k < R) stage[k * 33 + lane] = v[k];
    __syncwarp();
    int c = lane / R, k = lane - c * R;          // element e = i * 32 + lane of the block: record e / R, component e % R
    const int dc = 32 / R, dk = 32 - dc * R;
    for (int i = 0; i < R; ++i) {
        const int cc = min(c, n_valid - 1);
        rec0[(size_t)cc * rec + k] = stage[k * 33 + cc];
        c += dc; k += dk;
        if (k >= R) { k -= R; ++c; }
    }
    __syncwarp();
}

// JR = 0: joint frames live in the shared scratch (any number of columns, rolled loops);
// JR > 0: the model has at most JR columns and the frames live in registers (static indexing through
//         fully unrolled loops), which frees 6 * n_dof scratch slots per thread and lets a third CTA fit.
// Register budget: registers are allocated per SM sub-partition (16 K each), so 8 resident warps (4 CTAs
// of 64 threads, 2 warps per sub-partition) may use up to 255 registers per thread, while a 9th warp
// would cap every thread at 168 and spill.  With the frames in registers the collision kernel is
// therefore built for 4 x 64 threads per SM.
// SELF (with COLL; kin_self_collision, an extension): phase 1 as for a collision call (sphere centres, joint frames),
// then the self-collision phase over the model's pair table instead of phase 2.
template <typename real, int LAY, int BS, bool COLL, int JR, bool SELF = false>
__global__ void __launch_bounds__(BS, (JR > 0 && COLL) ? (BS == 64 ? 4 : BS == 128 ? 2 : BS == 32 ? 8 : 2) : 1)
kin_eval_kernel(const __grid_constant__ KernelArgs A) {
    // LAY: 0 = SoA (x[comp * ld + n]), 1 = AoS (x[n * rec + comp]), 2 = tiled (AoSoA-32:
    // x[((n / 32) * rec + comp) * 32 + n % 32], one contiguous block per warp, immediate offsets)
    constexpr bool AOS = LAY == 1, TILED = LAY == 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const ProgHeader &h = A.h;
    int32_t *ti = reinterpret_cast<int32_t *>(smem_raw);
    real *tr = reinterpret_cast<real *>(smem_raw + sizeof(int32_t) * (size_t)h.n_int);
    const int tid = threadIdx.x;
    real *scr = tr + h.n_real + tid;                   // [slot][thread]: SCR(slot) = scr[slot * BS]
    #define SCR(slot) scr[(slot) * BS]
    // AoS: warp-private staging buffer behind the scratch
    const int lane = tid & 31;
    real *stage = tr + h.n_real + (size_t)h.n_slots * BS + (tid >> 5) * AOS_STAGE_REALS;

    // ---- stage the program tables once per CTA ----
    {
        const int4 *src = reinterpret_cast<const int4 *>(A.tab_i);
        int4 *dst = reinterpret_cast<int4 *>(ti);
        for (int i = tid; i < h.n_int / 4; i += BS) dst[i] = src[i];
        const real *rs = reinterpret_cast<const real *>(A.tab_r);
        for (int i = tid; i < h.n_real; i += BS) tr[i] = rs[i];
    }
    __syncthreads();

    // The planar base is compiled into three ordinary nodes (prismatic x, y; revolute z), so every one of
    // the ND columns is an ordinary joint column here; DC = columns that are control joints.
    const int DC = h.n_joints, ND = h.n_dof;
    // header fields used in loops, as locals (kernel parameters are otherwise re-read from the constant bank)
    const int n_nodes = h.n_nodes, n_box = h.n_box, S = h.n_sph, n_fk = h.n_fk;
    const int io_node = h.io_node, io_att = h.io_att, io_sph_order = h.io_sph_order, io_sph_mask = h.io_sph_mask;
    const int ro_node = h.ro_node, ro_att = h.ro_att, ro_sph = h.ro_sph, ro_box = h.ro_box;
    const int so_save = h.so_save, so_cent = h.so_cent;
    unsigned rev_mask = 0;              // bit j: column j is a revolute joint
    for (int j = 0; j < ND; ++j) rev_mask |= (ti[h.io_col_type + j] == 1 ? 1u : 0u) << j;
    real *jf0 = &SCR(h.so_jf);          // JR == 0 only
    real *stale0 = &SCR(h.so_stale);
    const int rows = A.with_rot ? 6 : 3;
    // distance between consecutive components of one configuration's record
    const size_t es = AOS ? size_t(1) : TILED ? size_t(32) : (size_t)A.ld;
    // offset of component 0 of configuration n_ in an array with `rec` components per configuration
    auto rec_base = [&](long long n_, long long rec) -> long long {
        return AOS ? n_ * rec : TILED ? (n_ >> 5) * (rec * 32) + (n_ & 31) : n_;
    };

    // frame of column j: registers (j is a compile-time constant after unrolling) or scratch
    JFrame<real> jfr[JR > 0 ? JR : 1];
    #define JF_LOAD(f, j, ptr)                                                              \
        JFrame<real> f;                                                                     \
        if (JR > 0) f = jfr[j];                                                             \
        else { f.o[0] = (ptr)[0]; f.o[1] = (ptr)[BS]; f.o[2] = (ptr)[2 * BS];               \
               f.a[0] = (ptr)[3 * BS]; f.a[1] = (ptr)[4 * BS]; f.a[2] = (ptr)[5 * BS]; }
    // for (j = 0; j < ND; ++j): unrolled to JR iterations with an early exit, or rolled
    #define FOR_COLUMNS(j) _Pragma("unroll") for (int j = 0; j < (JR > 0 ? JR : ND); ++j) if (JR > 0 && j >= ND) break; else

    // configuration -> scratch with cp.async, double-buffered across tiles (buffers so_q / so_q2)
    const int q_stride = h.so_q2 - h.so_q;
    auto prefetch_q = [&](long long tile_, int buf) {
        const long long n_ = min(tile_ * BS + tid, (long long)A.n - 1);
        {
            const real *qn = reinterpret_cast<const real *>(A.q) + rec_base(n_, ND);
            real *dst = &SCR(h.so_q + buf * q_stride);
            for (int c = 0; c < ND; ++c) cp_async_elem(dst + c * BS, qn + c * es);
        }
        cp_async_commit();
    };
    const long long n_tiles = (A.n + BS - 1) / BS;
    if ((long long)blockIdx.x < n_tiles) prefetch_q(blockIdx.x, 0);
    int buf = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, buf ^= 1) {
        // threads past the end of the batch redo the last configuration (identical values, benign duplicate
        // stores) so that the whole CTA can meet at the phase barriers below
        const long long n = min(tile * BS + tid, (long long)A.n - 1);
        if (tile + gridDim.x < n_tiles) { prefetch_q(tile + gridDim.x, buf ^ 1); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        const int so_q = h.so_q + buf * q_stride;
        // AoS staging: first configuration of this warp and how many of its 32 records exist
        const long long n_w0 = min(tile * BS + (tid & ~31), (long long)A.n - 1);
        const int n_valid = (int)min((long long)32, A.n - n_w0);
        __syncthreads();             // the CTA's warps walk each phase together: one instruction fetch serves all
        real *Tn = reinterpret_cast<real *>(A.T_out) + rec_base(n, 12 * n_fk);
        real *Jn = reinterpret_cast<real *>(A.J_out) + rec_base(n, rows * ND * h.n_jac);

        Tf<real> T;                   // running world transform of the current node

        // =========================== phase 1 ===========================
        for (int node = 0; node < n_nodes; ++node) {
            const int32_t *ni = ti + io_node + node * NODE_INTS;
            const real *nr = tr + ro_node + node * NODE_REALS;
            const int jtype = ni[1];
            if (jtype == NODE_ROOT) {
                #pragma unroll
                for (int i = 0; i < 9; ++i) T.r[i] = (i % 4 == 0) ? real(1) : real(0);
                T.p[0] = T.p[1] = T.p[2] = real(0);
            } else {
                const int psrc = ni[0], flags = ni[2], qcol = ni[3];
                KIN_DASSERT(qcol >= 0 && qcol < ND);
                KIN_DASSERT(psrc < 0 || so_save + 12 * (psrc + 1) <= h.so_jf);
                if (psrc >= 0) {
                    const real *sv = &SCR(so_save + 12 * psrc);
                    #pragma unroll
                    for (int i = 0; i < 9; ++i) T.r[i] = sv[i * BS];
                    #pragma unroll
                    for (int i = 0; i < 3; ++i) T.p[i] = sv[(9 + i) * BS];
                }
                // A = T_parent * joint.pose : the joint frame (algorithm.jl:47-48)
                Tf<real> Aj;
                tf_mul_const(T, nr, flags & NF_OFF_R_IDENTITY, Aj);
                const int code = (flags >> NF_AXIS_SHIFT) & NF_AXIS_MASK;
                JFrame<real> f;           // world joint origin and axis (algorithm.jl:49-50)
                f.o[0] = Aj.p[0]; f.o[1] = Aj.p[1]; f.o[2] = Aj.p[2];
                const real sgn = code >= 4 ? real(-1) : real(1);
                switch (code) {
                    case 1: case 4: f.a[0] = sgn * Aj.r[0]; f.a[1] = sgn * Aj.r[3]; f.a[2] = sgn * Aj.r[6]; break;
                    case 2: case 5: f.a[0] = sgn * Aj.r[1]; f.a[1] = sgn * Aj.r[4]; f.a[2] = sgn * Aj.r[7]; break;
                    case 3: case 6: f.a[0] = sgn * Aj.r[2]; f.a[1] = sgn * Aj.r[5]; f.a[2] = sgn * Aj.r[8]; break;
                    default:
                        f.a[0] = fma_(Aj.r[0], nr[12], fma_(Aj.r[1], nr[13], Aj.r[2] * nr[14]));
                        f.a[1] = fma_(Aj.r[3], nr[12], fma_(Aj.r[4], nr[13], Aj.r[5] * nr[14]));
                        f.a[2] = fma_(Aj.r[6], nr[12], fma_(Aj.r[7], nr[13], Aj.r[8] * nr[14]));
                }
                if (JR > 0) {
                    switch (qcol) {       // uniform branch: one register copy, static indices
                        #define KIN_CASE(k) case k: if (k < JR) { asm volatile(""); jfr[k < JR ? k : 0] = f; } break;
                        KIN_CASE(0) KIN_CASE(1) KIN_CASE(2) KIN_CASE(3) KIN_CASE(4) KIN_CASE(5) KIN_CASE(6) KIN_CASE(7)
                        #undef KIN_CASE
                        default: break;
                    }
                } else {
                    real *jf = jf0 + 6 * BS * qcol;
                    jf[0] = f.o[0]; jf[BS] = f.o[1]; jf[2 * BS] = f.o[2];
                    jf[3 * BS] = f.a[0]; jf[4 * BS] = f.a[1]; jf[5 * BS] = f.a[2];
                }
                const real qa = SCR(so_q + qcol);
                T = Aj;
                if (jtype == 2) {          // prismatic: pose * Trans(axis * a), mechanism.jl:100-103
                    T.p[0] = fma_(f.a[0], qa, Aj.p[0]); T.p[1] = fma_(f.a[1], qa, Aj.p[1]); T.p[2] = fma_(f.a[2], qa, Aj.p[2]);
                } else {                   // revolute: pose * R(axis, a), mechanism.jl:94-98
                    real s, c;
                    sincos_(code >= 4 ? -qa : qa, &s, &c);
                    // rotation about a coordinate axis mixes the two other columns
                    #define GIVENS(u, v)                                                      \
                        _Pragma("unroll") for (int i = 0; i < 3; ++i) {                       \
                            real cu = Aj.r[i * 3 + u], cv = Aj.r[i * 3 + v];                  \
                            T.r[i * 3 + u] = fma_(c, cu, s * cv);                             \
                            T.r[i * 3 + v] = fma_(c, cv, -(s * cu));                          \
                        }
                    switch (code) {
                        case 1: case 4: GIVENS(1, 2) break;
                        case 2: case 5: GIVENS(2, 0) break;
                        case 3: case 6: GIVENS(0, 1) break;
                        default: {
                            // Rodrigues form of the reference's quaternion rotation:
                            // Rot = c I + s [a]x + (1-c) a a'
                            const real x = nr[12], y = nr[13], z = nr[14], t = real(1) - c;
                            real m[9];
                            m[0] = fma_(t * x, x, c);      m[1] = fma_(t * x, y, -(s * z)); m[2] = fma_(t * x, z, s * y);
                            m[3] = fma_(t * x, y, s * z);  m[4] = fma_(t * y, y, c);        m[5] = fma_(t * y, z, -(s * x));
                            m[6] = fma_(t * x, z, -(s * y)); m[7] = fma_(t * y, z, s * x);  m[8] = fma_(t * z, z, c);
                            #pragma unroll
                            for (int i = 0; i < 3; ++i)
                                #pragma unroll
                                for (int j = 0; j < 3; ++j)
                                    T.r[i * 3 + j] = fma_(Aj.r[i * 3 + 0], m[j], fma_(Aj.r[i * 3 + 1], m[3 + j], Aj.r[i * 3 + 2] * m[6 + j]));
                        }
                    }
                    #undef GIVENS
                }
            }
            if (ni[4] >= 0) {
                KIN_DASSERT(so_save + 12 * (ni[4] + 1) <= h.so_jf);
                real *sv = &SCR(so_save + 12 * ni[4]);
                #pragma unroll
                for (int i = 0; i < 9; ++i) sv[i * BS] = T.r[i];
                #pragma unroll
                for (int i = 0; i < 3; ++i) sv[(9 + i) * BS] = T.p[i];
            }

            // ---- requested links hanging from this node ----
            for (int a = ni[5]; a < ni[6]; ++a) {
                const int32_t *ai = ti + io_att + a * ATT_INTS;
                const real *ar = tr + ro_att + a * ATT_REALS;
                KIN_DASSERT(a >= 0 && a < h.n_att && ai[0] < n_fk && ai[2] < h.n_jac);
                Tf<real> Tl;
                tf_mul_const(T, ar, ai[1] & AF_R_IDENTITY, Tl);
                if (ai[0] >= 0 && A.T_out) {       // get_transform, as 3x4 column-major
                    if (AOS) {                     // staged: lanes run along the records
                        real v[12];
                        #pragma unroll
                        for (int c = 0; c < 3; ++c)
                            #pragma unroll
                            for (int r = 0; r < 3; ++r) v[c * 3 + r] = Tl.r[r * 3 + c];
                        #pragma unroll
                        for (int r = 0; r < 3; ++r) v[9 + r] = Tl.p[r];
                        const size_t rec = (size_t)12 * n_fk;
                        warp_store_records<real, 12>(stage, reinterpret_cast<real *>(A.T_out) + n_w0 * rec + 12 * ai[0], rec, v, 12, lane, n_valid);
                    } else {
                        real *o = Tn + (size_t)(12 * ai[0]) * es;
                        #pragma unroll
                        for (int c = 0; c < 3; ++c)
                            #pragma unroll
                            for (int r = 0; r < 3; ++r) o[(c * 3 + r) * es] = Tl.r[r * 3 + c];
                        #pragma unroll
                        for (int r = 0; r < 3; ++r) o[(9 + r) * es] = Tl.p[r];
                    }
                }
                if (ai[2] >= 0 && A.J_out) {       // get_jacobian, algorithm.jl:83-114
                    real *o = Jn + (size_t)(ai[2] * rows * ND) * es;
                    const unsigned mask = (unsigned)ai[3];
                    real k[6] = {0, 0, 0, 0, 0, 0};
                    if (A.with_rot && A.rpy_jac) rpy_rate_coeffs(Tl, k);
                    const real *jf = jf0;
                    #pragma unroll 1
                    for (int j = 0; j < ND; ++j) {      // rolled: executed once per requested link only
                        if ((mask >> j) & 1u) {
                            JFrame<real> f;
                            if (JR > 0) {
                                switch (j) {
                                    #define KIN_CASE(k) case k: f = jfr[k < JR ? k : 0]; break;
                                    KIN_CASE(0) KIN_CASE(1) KIN_CASE(2) KIN_CASE(3) KIN_CASE(4) KIN_CASE(5) KIN_CASE(6) KIN_CASE(7)
                                    #undef KIN_CASE
                                    default: f = jfr[0]; break;
                                }
                            } else {
                                f.o[0] = jf[0]; f.o[1] = jf[BS]; f.o[2] = jf[2 * BS];
                                f.a[0] = jf[3 * BS]; f.a[1] = jf[4 * BS]; f.a[2] = jf[5 * BS];
                            }
                            real cx, cy, cz;
                            const bool rev = (rev_mask >> j) & 1u;
                            jac_col(f, rev, Tl.p[0], Tl.p[1], Tl.p[2], cx, cy, cz);
                            o[0] = cx; o[es] = cy; o[2 * es] = cz;
                            if (A.with_rot) {
                                if (rev) {
                                    if (A.rpy_jac) {
                                        real o3, o4, o5;
                                        rpy_rows(k, f.a[0], f.a[1], f.a[2], o3, o4, o5);
                                        o[3 * es] = o3; o[4 * es] = o4; o[5 * es] = o5;
                                    } else {
                                        o[3 * es] = f.a[0]; o[4 * es] = f.a[1]; o[5 * es] = f.a[2];
                                    }
                                } else if (!A.keep_irrelevant || j >= DC) {
                                    // prismatic: rows 4:6 untouched by the reference (algorithm.jl:78-81), except in
                                    // the base block, which it always writes (algorithm.jl:102-104)
                                    o[3 * es] = real(0); o[4 * es] = real(0); o[5 * es] = real(0);
                                }
                            }
                        } else if (!A.keep_irrelevant) {
                            for (int r = 0; r < rows; ++r) o[r * es] = real(0);
                        }
                        o += rows * es;
                        jf += 6 * BS;
                    }
                }
            }

            // ---- collision-sphere centres on this node (collision.jl:54 / :80) ----
            if (COLL) {
                for (int k = ni[7]; k < ni[8]; ++k) {
                    const int s = ti[io_sph_order + k];
                    KIN_DASSERT(k >= 0 && k < S && s >= 0 && s < S);
                    const real *sr = tr + ro_sph + s * SPH_REALS;
                    const real c0 = sr[0], c1 = sr[1], c2 = sr[2];
                    real *cs = &SCR(so_cent + 3 * s);
                    #pragma unroll
                    for (int i = 0; i < 3; ++i)
                        cs[i * BS] = fma_(T.r[i * 3 + 0], c0, fma_(T.r[i * 3 + 1], c1, fma_(T.r[i * 3 + 2], c2, T.p[i])));
                }
            }
        }

        // =========================== phase 2 ===========================
        if (COLL && !SELF) {
            __syncthreads();
            const bool want_grads = A.grads_out != nullptr;
            const bool stale = want_grads && A.scratch_ref;
            const real trunc = (real)A.truncation_dist, voff = (real)A.vals_offset;
            if (stale)
                for (int i = 0; i < 3 * ND; ++i) stale0[i * BS] = real(0);   // jac = zeros(3, n_dof), collision.jl:76
            real *Vp = reinterpret_cast<real *>(A.vals_out) + rec_base(n, S);
            real *Gp = reinterpret_cast<real *>(A.grads_out) + rec_base(n, (long long)ND * S);
            int32_t *Ap = A.argmin_out ? A.argmin_out + rec_base(n, S) : nullptr;
            real *hand = &SCR(so_q);      // q is dead: (dmin, argmin) of the current sphere group

            for (int s0 = 0; s0 < S; s0 += SPH_GROUP) {
                // ---- 2a: distances of SPH_GROUP spheres; one box-table row feeds all of them ----
                {
                    real px[SPH_GROUP], py[SPH_GROUP], pz[SPH_GROUP], kmin[SPH_GROUP];
                    int kidx[SPH_GROUP];
                    #pragma unroll
                    for (int g = 0; g < SPH_GROUP; ++g) {
                        const real *cs = &SCR(so_cent + 3 * min(s0 + g, S - 1));
                        px[g] = cs[0]; py[g] = cs[BS]; pz[g] = cs[2 * BS];
                        kmin[g] = CUDART_INF; kidx[g] = 0;
                    }
                    // UnionSDF: all boxes, first minimum wins (sdf.jl:108-114)
                    for (int b = 0; b < n_box; ++b) {
                        BoxRow<real> row;
                        load_box(tr + ro_box + b * BOX_REALS, row);
                        real key[SPH_GROUP], qx[SPH_GROUP], qy[SPH_GROUP], qz[SPH_GROUP];
                        if (KPRIMS && row.kind != real(0)) {     // a sphere / cylinder row (extension): warp-uniform, out of line
                            #pragma unroll 1
                            for (int g = 0; g < SPH_GROUP; ++g)
                                key[g] = dist_to_key(prim_dist_general(tr + ro_box + b * BOX_REALS, px[g], py[g], pz[g]));
                        } else {
                        bool any_inside = false;
                        #pragma unroll
                        for (int g = 0; g < SPH_GROUP; ++g) {
                            key[g] = box_key_outside(row, px[g], py[g], pz[g], qx[g], qy[g], qz[g]);
                            any_inside |= !(key[g] > real(0));
                        }
                        if (any_inside) {       // rare: some centre is inside (or on) this box -- one branch per row
                            #pragma unroll
                            for (int g = 0; g < SPH_GROUP; ++g)
                                if (!(key[g] > real(0))) key[g] = box_inside_key(qx[g], qy[g], qz[g]);
                        }
                        }
                        #pragma unroll
                        for (int g = 0; g < SPH_GROUP; ++g)
                            if (key[g] < kmin[g]) { kmin[g] = key[g]; kidx[g] = b; }
                    }
                    #pragma unroll
                    for (int g = 0; g < SPH_GROUP; ++g) {
                        hand[g * BS] = key_to_dist(kmin[g]);     // four independent sqrt chains interleave here
                        reinterpret_cast<int *>(&hand[(SPH_GROUP + g) * BS])[0] = kidx[g];
                    }
                }
                // ---- 2b: per sphere, IN sphere order (the shared scratch of collision.jl:76,90 makes the
                //      order observable): value, truncation, gradient, chain rule ----
                #pragma unroll 1
                for (int g = 0; g < SPH_GROUP && s0 + g < S; ++g) {
                    const int s = s0 + g;
                    const real dmin = hand[g * BS];
                    const int kmin = reinterpret_cast<const int *>(&hand[(SPH_GROUP + g) * BS])[0];
                    KIN_DASSERT(kmin >= 0 && kmin < n_box);
                    const real dist0 = dmin - tr[ro_sph + s * SPH_REALS + 3];
                    const bool truncated = dist0 > trunc;
                    *Vp = (truncated ? trunc : dist0) - voff;
                    Vp += es;
                    if (Ap) { *Ap = kmin + 1; Ap += es; }
                    if (!want_grads) continue;
                    if (AOS && JR > 0) {
                        // AoS: the n_dof gradients of this sphere are collected in registers and written by the
                        // whole warp (truncated lanes contribute zeros: collision.jl:84-86), so control flow
                        // stays convergent up to the staged store
                        real gv[JR > 0 ? JR : 1];
                        #pragma unroll
                        for (int j = 0; j < (JR > 0 ? JR : 1); ++j) gv[j] = real(0);
                        if (!truncated) {
                            const real *cs = &SCR(so_cent + 3 * s);
                            const real px = cs[0], py = cs[BS], pz = cs[2 * BS];
                            real grad[3];
                            {
                                BoxRow<real> row;
                                load_box(tr + ro_box + kmin * BOX_REALS, row);
                                sdf_row_gradient(tr + ro_box + kmin * BOX_REALS, row, A.grad_mode, px, py, pz, dmin, grad);
                            }
                            const unsigned mask = (unsigned)ti[io_sph_mask + s];
                            real *st = stale0;
                            FOR_COLUMNS(j) {
                                real cx, cy, cz;
                                if ((mask >> j) & 1u) {
                                    jac_col(jfr[j], (rev_mask >> j) & 1u, px, py, pz, cx, cy, cz);
                                    if (stale) { st[0] = cx; st[BS] = cy; st[2 * BS] = cz; }
                                } else if (stale) { cx = st[0]; cy = st[BS]; cz = st[2 * BS]; }
                                else { cx = cy = cz = real(0); }
                                gv[j] = fma_(grad[0], cx, fma_(grad[1], cy, grad[2] * cz));
                                st += 3 * BS;
                            }
                        }
                        const size_t rec = (size_t)ND * S;
                        warp_store_records<real, (JR > 0 ? JR : 1)>(stage, reinterpret_cast<real *>(A.grads_out) + n_w0 * rec + (size_t)s * ND,
                                                                    rec, gv, ND, lane, n_valid);
                        continue;
                    }
                    if (!want_grads) continue;
                    if (truncated) {            // collision.jl:84-86
                        for (int j = 0; j < ND; ++j) Gp[(size_t)j * es] = real(0);
                        Gp += (size_t)ND * es;
                        continue;
                    }
                    const real *cs = &SCR(so_cent + 3 * s);
                    const real px = cs[0], py = cs[BS], pz = cs[2 * BS];
                    real grad[3];
                    {
                        BoxRow<real> row;
                        load_box(tr + ro_box + kmin * BOX_REALS, row);
                        sdf_row_gradient(tr + ro_box + kmin * BOX_REALS, row, A.grad_mode, px, py, pz, dmin, grad);
                    }
                    const unsigned mask = (unsigned)ti[io_sph_mask + s];
                    const real *jf = jf0;
                    real *st = stale0;
                    FOR_COLUMNS(j) {
                        real cx, cy, cz;
                        if ((mask >> j) & 1u) {   // joint_jacobian!, algorithm.jl:65-81
                            JF_LOAD(f, j, jf)
                            jac_col(f, (rev_mask >> j) & 1u, px, py, pz, cx, cy, cz);
                            if (stale) { st[0] = cx; st[BS] = cy; st[2 * BS] = cz; }
                        } else if (stale) {     // column left over from an earlier sphere (collision.jl:76,90)
                            cx = st[0]; cy = st[BS]; cz = st[2 * BS];
                        } else { cx = cy = cz = real(0); }
                        Gp[(size_t)j * es] = fma_(grad[0], cx, fma_(grad[1], cy, grad[2] * cz));   // transpose(grad) * jac
                        jf += 6 * BS; st += 3 * BS;
                    }
                    Gp += (size_t)ND * es;      // (a pointer bumped inside the loop is live across its early exit: two extra moves per column)
                }
            }
        }

        // ===================== self-collision phase (extension) =====================
        // Pair p = (i, j) of the model's table: L = |c_i - c_j|, d = L - r_i - r_j; gradient column k =
        // u . (J_i[:,k] - J_j[:,k]) with u = (c_i - c_j) / L (0 when L == 0).  A column that moves both spheres moves
        // them rigidly together, so its two terms cancel exactly: only the columns of mask_i XOR mask_j are evaluated,
        // the others are written as 0.  Truncation and offset as phase 2; (dmin, amin) over the untruncated d.
        if constexpr (SELF) {
            const int P = A.n_self_pairs;
            const real trunc = (real)A.truncation_dist, voff = (real)A.vals_offset;
            real *Vp = A.vals_out ? reinterpret_cast<real *>(A.vals_out) + rec_base(n, P) : nullptr;
            real *Gp = A.grads_out ? reinterpret_cast<real *>(A.grads_out) + rec_base(n, (long long)ND * P) : nullptr;
            real best = CUDART_INF;
            int bi = 0;
            #pragma unroll 1
            for (int p = 0; p < P; ++p) {
                const int2 pr = __ldg(A.self_pairs + p);          // the same address in every lane: one broadcast load
                KIN_DASSERT(pr.x >= 0 && pr.x < S && pr.y >= 0 && pr.y < S && pr.x != pr.y);
                const real *ci = &SCR(so_cent + 3 * pr.x), *cj = &SCR(so_cent + 3 * pr.y);
                const real xi = ci[0], yi = ci[BS], zi = ci[2 * BS], xj = cj[0], yj = cj[BS], zj = cj[2 * BS];
                const real dx = xi - xj, dy = yi - yj, dz = zi - zj;
                const real L = sqrt_(fma_(dx, dx, fma_(dy, dy, dz * dz)));
                const real d = L - tr[ro_sph + pr.x * SPH_REALS + 3] - tr[ro_sph + pr.y * SPH_REALS + 3];
                if (d < best) { best = d; bi = p; }
                if (!Vp) continue;
                const bool truncated = d > trunc;
                *Vp = (truncated ? trunc : d) - voff;
                Vp += es;
                if (!Gp) continue;
                const unsigned mi = (unsigned)ti[io_sph_mask + pr.x], mj = (unsigned)ti[io_sph_mask + pr.y];
                const unsigned mx = (truncated || !(L > real(0))) ? 0u : (mi ^ mj);
                const real inv = mx ? real(1) / L : real(0);
                const real ux = dx * inv, uy = dy * inv, uz = dz * inv;
                // column j of this pair's gradient; the frame of j comes from registers (jfr, j static) or scratch
                auto column = [&](const JFrame<real> &f, int j) -> real {
                    const bool on_i = (mi >> j) & 1u;
                    real cx, cy, cz;
                    jac_col(f, (rev_mask >> j) & 1u, on_i ? xi : xj, on_i ? yi : yj, on_i ? zi : zj, cx, cy, cz);
                    const real g = fma_(ux, cx, fma_(uy, cy, uz * cz));
                    return on_i ? g : -g;
                };
                if (AOS) {
                    // the ND values of this pair are contiguous in the configuration's record: staged in chunks of
                    // AOS_STAGE_ROWS columns and written by the whole warp (control flow is warp-uniform up to here)
                    const size_t rec = (size_t)ND * P;
                    for (int k0 = 0; k0 < (JR > 0 ? 1 : ND); k0 += AOS_STAGE_ROWS) {
                        real gv[AOS_STAGE_ROWS];
                        #pragma unroll
                        for (int kk = 0; kk < AOS_STAGE_ROWS; ++kk) {
                            const int j = JR > 0 ? kk : k0 + kk;
                            gv[kk] = real(0);
                            if (j < ND && ((mx >> j) & 1u)) {
                                JFrame<real> f;
                                if (JR > 0) f = jfr[kk < (JR > 0 ? JR : 1) ? kk : 0];
                                else {
                                    const real *jf = jf0 + 6 * BS * j;
                                    f.o[0] = jf[0]; f.o[1] = jf[BS]; f.o[2] = jf[2 * BS];
                                    f.a[0] = jf[3 * BS]; f.a[1] = jf[4 * BS]; f.a[2] = jf[5 * BS];
                                }
                                gv[kk] = column(f, j);
                            }
                        }
                        warp_store_records<real, AOS_STAGE_ROWS>(stage, reinterpret_cast<real *>(A.grads_out) + n_w0 * rec + (size_t)p * ND + k0,
                                                                 rec, gv, min(AOS_STAGE_ROWS, ND - k0), lane, n_valid);
                    }
                    continue;
                }
                const real *jf = jf0;
                FOR_COLUMNS(j) {
                    real g = real(0);
                    if ((mx >> j) & 1u) {
                        JF_LOAD(f, j, jf)
                        g = column(f, j);
                    }
                    Gp[(size_t)j * es] = g;
                    jf += 6 * BS;
                }
                Gp += (size_t)ND * es;
            }
            if (A.dmin_out) reinterpret_cast<real *>(A.dmin_out)[n] = best;
            if (A.amin_out) A.amin_out[n] = bi + 1;
        }
    }
    #undef SCR
    #undef JF_LOAD
    #undef FOR_COLUMNS
}

// sdf(p) and gradient!(sdf, p, out) for a batch of points (sdf.jl:34-41, 67-74, 108-119).
template <typename real, bool AOS>
__global__ void __launch_bounds__(256)
sdf_points_kernel(const real *__restrict__ boxes, int n_box, const real *__restrict__ pts, long long n_pts,
                  int grad_mode, real *__restrict__ vals, real *__restrict__ grads, int32_t *__restrict__ argmin) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    real *tb = reinterpret_cast<real *>(smem_raw);
    for (int i = threadIdx.x; i < n_box * BOX_REALS; i += blockDim.x) tb[i] = boxes[i];
    __syncthreads();
    for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < n_pts; n += (long long)gridDim.x * blockDim.x) {
        const real px = AOS ? pts[3 * n] : pts[n], py = AOS ? pts[3 * n + 1] : pts[n_pts + n],
                   pz = AOS ? pts[3 * n + 2] : pts[2 * n_pts + n];
        real kmin = CUDART_INF;
        int kidx = 0;
        BoxRow<real> row;
        for (int b = 0; b < n_box; ++b) {
            load_box(tb + b * BOX_REALS, row);
            const real key = sdf_row_key(tb + b * BOX_REALS, row, px, py, pz);
            if (key < kmin) { kmin = key; kidx = b; }
        }
        const real dmin = key_to_dist(kmin);
        vals[n] = dmin;
        if (argmin) argmin[n] = kidx + 1;
        if (grads) {
            real g[3];
            load_box(tb + kidx * BOX_REALS, row);
            sdf_row_gradient(tb + kidx * BOX_REALS, row, grad_mode, px, py, pz, dmin, g);
            #pragma unroll
            for (int i = 0; i < 3; ++i) grads[AOS ? 3 * n + i : (long long)i * n_pts + n] = g[i];
        }
    }
}

// Per-configuration reductions over the S sphere distances of a collision call (kin_collision_summary): the minimum
// distance, the sphere that attains it (first minimum, 1-based) and the hinge cost sum_s max(0, margin - d_s)^2.
//   SoA / tiled: one thread per configuration walks its S values (coalesced across the threads);
//   AoS: the S values of a configuration are contiguous, so a group of G = 2^k >= min(S, 32) lanes takes one
//        configuration (lane = sphere) and the group reduces with warp shuffles: min / argmin by a butterfly on
//        (value, index) pairs, the cost by a butterfly sum.
template <typename real, int LAY>
__global__ void __launch_bounds__(256)
coll_summary_kernel(const real *__restrict__ vals, long long n, long long ld, int S, real margin, real *__restrict__ dmin,
                    int32_t *__restrict__ amin, real *__restrict__ cost) {
    if (LAY != 1) {
        for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (long long)gridDim.x * blockDim.x) {
            const real *v = vals + (LAY == 2 ? (c >> 5) * ((long long)S * 32) + (c & 31) : c);
            const long long es = LAY == 2 ? 32 : ld;
            real best = CUDART_INF, sum = real(0);
            int bi = 0;
            for (int s = 0; s < S; ++s) {
                const real d = v[s * es];
                if (d < best) { best = d; bi = s; }
                const real h = margin - d;
                if (h > real(0)) sum = fma_(h, h, sum);
            }
            dmin[c] = best;
            if (amin) amin[c] = bi + 1;
            if (cost) cost[c] = sum;
        }
        return;
    }
    int G = 1;
    while (G < S && G < 32) G <<= 1;
    const int lane = threadIdx.x & 31, lg = lane & (G - 1), per_warp = 32 / G;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long c0 = warp * per_warp; c0 < n; c0 += n_warps * per_warp) {     // warp-uniform trip count
        const long long c = c0 + lane / G;
        real best = CUDART_INF, sum = real(0);
        int bi = 0x7fffffff;
        if (c < n)
            for (int s = lg; s < S; s += G) {
                const real d = vals[c * S + s];
                if (d < best) { best = d; bi = s; }
                const real h = margin - d;
                if (h > real(0)) sum = fma_(h, h, sum);
            }
        for (int off = G >> 1; off > 0; off >>= 1) {
            const real ob = __shfl_xor_sync(0xffffffffu, best, off);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
            const real os = __shfl_xor_sync(0xffffffffu, sum, off);
            if (ob < best || (ob == best && oi < bi)) { best = ob; bi = oi; }   // first minimum wins, as in the serial walk
            sum += os;
        }
        if (c < n && lg == 0) {
            dmin[c] = best;
            if (amin) amin[c] = bi + 1;
            if (cost) cost[c] = sum;
        }
    }
}

// Pose residuals / IK objective from the link transforms T (12 per link per configuration) and their Euler-rate
// Jacobians J (rows_j x n_dof per link), both produced by kin_eval_kernel in the same layout, for ALL the
// (link, target, with_rot) triples of a constraint in one launch (the loop of planning.jl:124-137).
//   mode 0  inverse_kinematics.jl:38-50   f = sum(e^2), grad = -2 J' e,   e = [p_t - p; rpy_t - rpy]  (summed over links)
//   mode 1  planning.jl:114-138           val = [p - p_t; rpy - rpy_t] per link, stacked;  jac_T(n_dof, n_cons) = J'
// rot_mask bit l: link l constrains the rotation too (dim 6, else 3); rows_j = 6 when any bit is set, else 3.
// target: 6 values per link ([x y z roll pitch yaw]), per configuration or shared.
template <typename real, bool AOS>
__global__ void __launch_bounds__(256)
pose_residual_kernel(const real *__restrict__ T, const real *__restrict__ J, const real *__restrict__ target,
                     int target_per_config, long long n_cfg, int nd, int nl, unsigned rot_mask, int mode,
                     real *__restrict__ val_out, real *__restrict__ jac_out) {
    const int rows_j = rot_mask ? 6 : 3;
    int n_cons = 0;
    for (int l = 0; l < nl; ++l) n_cons += ((rot_mask >> l) & 1u) ? 6 : 3;
    for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < n_cfg; n += (long long)gridDim.x * blockDim.x) {
        const size_t es = AOS ? size_t(1) : (size_t)n_cfg;
        const size_t ts = target_per_config ? es : size_t(1);
        real f = 0;
        real *g = jac_out + (AOS ? n * nd : n);                       // mode 0: gradient (n_dof)
        real *v = val_out + (AOS ? n * n_cons : n);                   // mode 1: values (n_cons)
        real *jt = jac_out + (AOS ? n * (long long)(n_cons * nd) : n);   // mode 1: (n_dof, n_cons) column-major
        if (mode == 0)
            for (int j = 0; j < nd; ++j) g[j * es] = real(0);
        int c0 = 0;
        for (int l = 0; l < nl; ++l) {
            const bool with_rot = (rot_mask >> l) & 1u;
            const int rows = with_rot ? 6 : 3;
            const real *Tn = T + (AOS ? n * (long long)(12 * nl) : n) + (size_t)(12 * l) * es;
            const real *Jn = J + (AOS ? n * (long long)(rows_j * nd * nl) : n) + (size_t)(l * rows_j * nd) * es;
            const real *tg = target + (target_per_config ? (AOS ? n * (long long)(6 * nl) : n) : 0) + (size_t)(6 * l) * ts;
            real e[6];
            #pragma unroll
            for (int i = 0; i < 3; ++i) e[i] = Tn[(9 + i) * es] - tg[i * ts];          // p - p_t
            if (with_rot) {   // rpy(T), transform.jl:45-48 (RotZYX): R[r][c] = T[c*3 + r]
                const real r00 = Tn[0], r10 = Tn[es], r20 = Tn[2 * es], r01 = Tn[3 * es], r11 = Tn[4 * es],
                           r21 = Tn[5 * es], r02 = Tn[6 * es], r12 = Tn[7 * es], r22 = Tn[8 * es];
                const real yaw = atan2_(r10, r00);
                real s1, c1;
                sincos_(yaw, &s1, &c1);
                const real pitch = atan2_(-r20, sqrt_(fma_(r21, r21, r22 * r22)));
                const real roll = atan2_(fma_(r02, s1, -(r12 * c1)), fma_(r11, c1, -(r01 * s1)));
                e[3] = roll - tg[3 * ts]; e[4] = pitch - tg[4 * ts]; e[5] = yaw - tg[5 * ts];
            }
            if (mode == 0) {
                for (int r = 0; r < rows; ++r) { e[r] = -e[r]; f = fma_(e[r], e[r], f); }   // e = target - now
                for (int j = 0; j < nd; ++j) {
                    real acc = 0;
                    for (int r = 0; r < rows; ++r) acc = fma_(Jn[(size_t)(j * rows_j + r) * es], e[r], acc);
                    g[j * es] = fma_(real(-2), acc, g[j * es]);
                }
            } else {
                for (int r = 0; r < rows; ++r) v[(size_t)(c0 + r) * es] = e[r];
                for (int r = 0; r < rows; ++r)
                    for (int j = 0; j < nd; ++j) jt[(size_t)((c0 + r) * nd + j) * es] = Jn[(size_t)(j * rows_j + r) * es];
            }
            c0 += rows;
        }
        if (mode == 0) val_out[n] = f;
    }
}


}  // namespace kin

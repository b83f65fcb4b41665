// kin_gen_skeleton.cuh -- the fixed part of the model-specialised kernels (compiled by NVRTC at run time together with
// the text kin_codegen.cpp generates; this file is embedded in the library).  Compilation unit:
//     #include "kin_gen_config.h"      generated: KREAL, KND, KS, KREV, KSTALE, ..., KRADIUS[]
//     #include "kin_device_math.cuh"   the shared arithmetic (same functions as the interpreting kernels)
//     #include "kin_gen_skeleton.cuh"  this file; it includes
//         "kin_gen_phase1.inc"         generated straight-line phase 1 (uses KQ, KST_T, KST_J, KCEN_SET, KJF_OUT)
//         "kin_gen_phase2.inc"         generated: joint frames + one phase2_run<MASK> call per run of spheres
// One thread = one configuration, persistent CTAs, SoA or tiled layout (kin_b200.h).  No table is interpreted: the
// only run-time tables left are the boxes (kin_model_set_boxes moves them without recompiling) and the radii.
#pragma once

namespace kin {

typedef KREAL real;

// ---- phase 2, as in kin_eval_kernel but split so that the code that does not depend on the relevance mask exists
//      once: 2a (union SDF of a group of up to SPH_GROUP spheres; sdf.jl:108-114) is shared, 2b (value, truncation,
//      gradient, chain rule: collision.jl:78-93) is instantiated per mask, with the mask, the column count / types and
//      the scratch / gradient / argmin switches as compile-time constants ----
template <typename real_>
__device__ __forceinline__ void phase2a_group(const int s0, const int ge, const real_ *__restrict__ tb, const int n_box,
                                              const real_ *cent0, real_ *hand) {
    typedef real_ real;
    constexpr int BS = KBS;
    real px[SPH_GROUP], py[SPH_GROUP], pz[SPH_GROUP], kmin[SPH_GROUP];
    int kidx[SPH_GROUP];
    #pragma unroll
    for (int g = 0; g < SPH_GROUP; ++g) {
        const real *cs = cent0 + 3 * min(s0 + g, ge - 1) * BS;
        px[g] = cs[0]; py[g] = cs[BS]; pz[g] = cs[2 * BS];
        kmin[g] = CUDART_INF; kidx[g] = 0;
    }
    #pragma unroll 1
    for (int b = 0; b < n_box; ++b) {         // UnionSDF: all boxes, first minimum wins (sdf.jl:108-114)
        BoxRow<real> row;
        load_box(tb + b * BOX_REALS, row);
        real key[SPH_GROUP], qx[SPH_GROUP], qy[SPH_GROUP], qz[SPH_GROUP];
        if (KPRIMS && row.kind != real(0)) {     // a sphere / cylinder row (extension): warp-uniform, out of line
            #pragma unroll 1
            for (int g = 0; g < SPH_GROUP; ++g) key[g] = dist_to_key(prim_dist_general(tb + b * BOX_REALS, px[g], py[g], pz[g]));
        } else {
        bool any_inside = false;
        #pragma unroll
        for (int g = 0; g < SPH_GROUP; ++g) {
            key[g] = box_key_outside(row, px[g], py[g], pz[g], qx[g], qy[g], qz[g]);
            any_inside |= !(key[g] > real(0));
        }
        if (any_inside) {
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
        hand[g * BS] = key_to_dist(kmin[g]);
        reinterpret_cast<int *>(&hand[(SPH_GROUP + g) * BS])[0] = kidx[g];
    }
}

#if KAOS && !KWARP && !KIK
// ---- AoS outputs of the one-thread-per-configuration kernel.  A thread owns a record, so a plain store would scatter
//      8 bytes per lane over 32 records.  Instead every lane PUTs its values into rows of a warp-private stage in
//      shared memory (row = component, 33 reals per row: conflict free) and the warp writes the 32 records of the
//      chunk with the lanes running ALONG the records: CNT lanes per record, 32 / CNT records per store instruction,
//      whole sectors.  REC (values per record) and CNT are compile-time, so lane -> (record, component) is computed
//      once and every load / store of the loop has an immediate offset. ----
// A chunk of CNT values per record is written by LPR = the next power of two >= CNT lanes per record (the first CNT of
// them active), 32 / LPR records per store instruction.  The row pitch of the stage depends on LPR so that the 16 lanes
// of a half-warp (one shared-memory wavefront of 8-byte words) hit 16 different banks on the transposed read:
// pitch mod 16 = 16 / (records per half-warp); the PUTs (lanes along a row) are conflict free with any pitch.
// (The FK / Jacobian-only kernels are bound by the DRAM write path, not by shared memory: there CNT lanes per record,
// packed, with pitch 33 measured 5 % faster -- 0.97 against 0.92 of the HBM peak -- and is kept.)
__host__ __device__ constexpr int aos_lpr(int cnt) { return !KCOLL ? cnt : cnt > 16 ? 32 : cnt > 8 ? 16 : cnt > 4 ? 8 : cnt > 2 ? 4 : cnt > 1 ? 2 : 1; }
__host__ __device__ constexpr int aos_ld(int cnt) {
    return !KCOLL ? 33 : 32 + (aos_lpr(cnt) == 16 ? 1 : aos_lpr(cnt) == 8 ? 2 : aos_lpr(cnt) == 4 ? 4 : aos_lpr(cnt) == 2 ? 8 : 1);
}
constexpr int AOS_STAGE_G = (KND > 12 ? KND : 12) * 34;                    // reals for link transform / Jacobian chunks / gradients
constexpr int AOS_STAGE_V = SPH_GROUP * 36;                                // distances (and argmins) of one sphere group
constexpr int AOS_STAGE_REALS = AOS_STAGE_G + (KCOLL ? 2 * AOS_STAGE_V : 0);

template <typename T, int CNT, int REC, typename real_>
__device__ __forceinline__ void aos_flush(const real_ *area, T *dst, const int nvalid, const int lane) {
    constexpr int LPR = aos_lpr(CNT), RPI = 32 / LPR, ITERS = (32 + RPI - 1) / RPI, LD = aos_ld(CNT);
    const int rl = lane / LPR, c = lane % LPR;
    const real_ *src = area + c * LD + rl;
    T *d = dst + (long long)rl * REC + c;
    __syncwarp();
    if (c < CNT && rl < RPI) {
        #pragma unroll
        for (int i = 0; i < ITERS; ++i)
            if (i * RPI + rl < nvalid) __stcs(d + (long long)i * RPI * REC, *reinterpret_cast<const T *>(src + i * RPI));
    }
    __syncwarp();
}
// a sphere group holds 1 .. SPH_GROUP spheres: always the 4-lanes-per-record pattern, cnt lanes of each 4 active
template <typename T, int REC, typename real_>
__device__ __forceinline__ void aos_flush_group(const real_ *area, T *dst, const int cnt, const int nvalid, const int lane) {
    constexpr int LPR = 4, RPI = 8, LD = aos_ld(4);
    const int rl = lane / LPR, c = lane % LPR;
    const real_ *src = area + c * LD + rl;
    T *d = dst + (long long)rl * REC + c;
    __syncwarp();
    if (c < cnt) {
        #pragma unroll
        for (int i = 0; i < 32 / RPI; ++i)
            if (i * RPI + rl < nvalid) __stcs(d + (long long)i * RPI * REC, *reinterpret_cast<const T *>(src + i * RPI));
    }
    __syncwarp();
}
static_assert(SPH_GROUP <= 4, "aos_flush_group covers groups of up to 4 spheres");
#endif

// per sphere, IN sphere order (the shared scratch of collision.jl:76,90 makes the order observable)
// AoS: Vp0 / Gp0 / Ap0 point at the FIRST record of the warp, es = lane, stw = the warp's stage, nvalid = records of the
// warp inside the batch; the control flow below is warp-uniform except for the truncation branch, which re-converges
// before each flush.
template <typename real_, int ND, unsigned MASK>
__device__ __forceinline__ void phase2b_group(const int s0, const int ge, const real_ *__restrict__ tb,
                                              const real_ *__restrict__ rad, const real_ *cent0, real_ *stale0, const real_ *hand,
                                              const JFrame<real_> (&jfr)[ND > 0 ? ND : 1], const int grad_mode, const real_ trunc,
                                              const real_ voff, real_ *Vp0, real_ *Gp0, int32_t *Ap0, const size_t es
#if KAOS && !KWARP && !KIK
                                              , real_ *stw, const int nvalid
#endif
                                              , const real_ *jfs     // KJFSMEM: this thread's joint frames in the shared scratch, [6 j + i][thread]
                                              , const unsigned rmask // KP2RTMASK: the relevance mask of this run of spheres at run time
                                              ) {
    typedef real_ real;
    constexpr int BS = KBS;
    // One instance per distinct relevance mask (MASK: the column loop below keeps only what that mask needs) -- or (opt-in,
    // KIN_JIT_RTMASK: for models with many distinct masks, e.g. 13 instances of an 18-column loop on a dual-arm mechanism)
    // ONE instance that tests the mask of the run at run time: warp-uniform branches, 2.4 x less code, measured within
    // +-8 % of the per-mask instances (kin_b200.cu: gen_options)
    const unsigned mask_ = KP2RTMASK ? rmask : MASK;
#if KAOS && !KWARP && !KIK
    const int lane = (int)es;
    real *stg = stw + lane;
    #define KP2_V(s_, g_, v_) stg[AOS_STAGE_G + (g_) * aos_ld(4)] = (v_)
    #define KP2_A(s_, g_, v_) reinterpret_cast<int *>(&stg[AOS_STAGE_G + AOS_STAGE_V + (g_) * aos_ld(4)])[0] = (v_)
    #define KP2_G(j_, v_) stg[(j_) * aos_ld(ND)] = (v_)
#else
    #define KP2_V(s_, g_, v_) __stcs(Vp0 + (size_t)(s_) * es, (v_))
    #define KP2_A(s_, g_, v_) __stcs(Ap0 + (size_t)(s_) * es, (v_))
    #define KP2_G(j_, v_) __stcs(&Gp[(size_t)(j_) * es], (v_))
#endif
    #pragma unroll 1
    for (int s = s0; s < ge; ++s) {
        const int g = s - s0;
        const real dmin = hand[g * BS];
        const int kmin = reinterpret_cast<const int *>(&hand[(SPH_GROUP + g) * BS])[0];
        const real dist0 = dmin - rad[s];
        const bool truncated = dist0 > trunc;
        KP2_V(s, g, (truncated ? trunc : dist0) - voff);
        if (KARGMIN) KP2_A(s, g, kmin + 1);
        if (!KGRADS) continue;
#if !(KAOS && !KWARP && !KIK)
        real *Gp = Gp0 + (size_t)s * ND * es;
#endif
        if (truncated) {            // collision.jl:84-86
            #pragma unroll
            for (int j = 0; j < ND; ++j) KP2_G(j, real(0));
        } else {
            const real *cs = cent0 + 3 * s * BS;
            const real px = cs[0], py = cs[BS], pz = cs[2 * BS];
            real grad[3];
            {
                BoxRow<real> row;
                load_box(tb + kmin * BOX_REALS, row);
                sdf_row_gradient(tb + kmin * BOX_REALS, row, KGRADMODE >= 0 ? KGRADMODE : grad_mode, px, py, pz, dmin, grad);
            }
            #pragma unroll
            for (int j = 0; j < ND; ++j) {
                real *st = stale0 + 3 * j * BS;
                if ((mask_ >> j) & 1u) {      // joint_jacobian!, algorithm.jl:65-81
                    real cx, cy, cz;
#if KJFSMEM
                    // more than 12 columns: the frames do not fit in registers; six shared loads with immediate offsets
                    JFrame<real> fj;
                    fj.o[0] = jfs[(6 * j + 0) * BS]; fj.o[1] = jfs[(6 * j + 1) * BS]; fj.o[2] = jfs[(6 * j + 2) * BS];
                    fj.a[0] = jfs[(6 * j + 3) * BS]; fj.a[1] = jfs[(6 * j + 4) * BS]; fj.a[2] = jfs[(6 * j + 5) * BS];
                    jac_col(fj, ((KREV >> j) & 1u) != 0, px, py, pz, cx, cy, cz);
#else
                    jac_col(jfr[j], ((KREV >> j) & 1u) != 0, px, py, pz, cx, cy, cz);
#endif
                    if (KSTALE) { st[0] = cx; st[BS] = cy; st[2 * BS] = cz; }
                    KP2_G(j, fma_(grad[0], cx, fma_(grad[1], cy, grad[2] * cz)));   // transpose(grad) * jac
                } else if (KSTALE) {          // column left over from an earlier sphere (collision.jl:76,90)
                    const real cx = st[0], cy = st[BS], cz = st[2 * BS];
                    KP2_G(j, fma_(grad[0], cx, fma_(grad[1], cy, grad[2] * cz)));
                } else {
                    KP2_G(j, real(0));      // a zero column (clean scratch): transpose(grad) * 0
                }
            }
        }
#if KAOS && !KWARP && !KIK
        aos_flush<real, ND, ND * KS>(stw, Gp0 + (size_t)s * ND, nvalid, lane);
#endif
    }
#if KAOS && !KWARP && !KIK
    aos_flush_group<real, KS>(stw + AOS_STAGE_G, Vp0 + s0, ge - s0, nvalid, lane);
    if (KARGMIN) aos_flush_group<int32_t, KS>(stw + AOS_STAGE_G + AOS_STAGE_V, Ap0 + s0, ge - s0, nvalid, lane);
#endif
    #undef KP2_V
    #undef KP2_A
    #undef KP2_G
}

}  // namespace kin

// =====================================================================================================================
// Monolithic kernel: phase 1 and phase 2 in the same thread.
// Dynamic shared memory: [box table n_box * BOX_REALS][radii KS] then the per-thread scratch [slot][thread]:
//   3 KS sphere-centre coordinates, 3 KND stale-Jacobian columns (KSTALE), 2 SPH_GROUP hand-over slots.
//
// KSCHED: CLAIMED TILES, INPUTS STAGED THROUGH L2 IN ONE BURST PER EPOCH (the FK / Jacobian-only kernels).  They are bound
// by the DRAM write path (2784 B of results per configuration against 64 B of input), and on HBM3e a trickle of small
// reads in the middle of a saturated write stream is disproportionately expensive (a store-only probe with this output
// pattern sustains 6.05 TB/s, the same probe reading its 8 inputs per thread 5.22 TB/s; profiles/probe_store.cu): every
// read interrupts the write drain of the channels it touches.  So the reads are clustered in time without lock-stepping
// the grid: the tiles are taken in ascending order (CTA b starts with the tiles b and b + grid, then claims 2 grid,
// 2 grid + 1, ... from the counter A.tile_next), in epochs of KEPOCH tiles; whoever takes tile t with t mod KEPOCH < P
// (P = min(grid, KEPOCH)) issues piece t mod KEPOCH of epoch t / KEPOCH + KPFD -- one cp.async.bulk.prefetch.L2 of that
// piece's tiles per input row (SoA) or of its one contiguous block (tiled, AoS), evict_last -- so the q of a whole
// epoch enters L2 in one burst, KPFD epochs ahead, and the per-thread loads hit L2.  No grid-wide barrier, no
// cooperative launch: an SM whose writes drain faster takes more tiles (DESIGN 4.4).
//
// KQB > 0 (AoS, where the claimed tiles measured slower): INPUT BATCHING.  The configurations of KQB tiles per CTA are
// fetched at once with cp.async into shared memory ([2][KQB][KND][BS] after the output stages), one batch ahead, and ALL
// CTAs issue the fetch of a batch at the same moment, behind a grid-wide barrier: one read burst per batch.  The grid
// is launched cooperatively (all CTAs resident), the barrier words live in A.sync.
// =====================================================================================================================
#if KIK
// =====================================================================================================================
// Batched inverse kinematics (config 4 of BASELINE.json): ONE kernel launch runs the whole damped least-squares solve,
// one thread per problem.  Per iteration the generated straight-line phase 1 gives the link transform and its
// Euler-rate Jacobian (the evaluations of f_objective, inverse_kinematics.jl:38-50: e = [p - p_t; rpy - rpy_t],
// rpy of RotZYX, transform.jl:45-48); the rest is the Levenberg-Marquardt update (the same one ik_coll_step_kernel of
// kin_ik_coll.cuh performs as a separate launch): normal equations H = J'J, g = J'e in registers, joints that sit on
// a limit and are pushed outward frozen, Cholesky of H + lambda (I + diag H), trial point clamped to the limits
// (inverse_kinematics.jl:52-63), accept / reject with the damping scaled by 0.3 / 4.  Angle residuals are wrapped to
// (-pi, pi].  A problem stops on its own when f < ftol.  The reference drives the same evaluations with NLopt SLSQP
// (third party); this replaces the per-iteration host round trips of a solver callback by a device-resident loop.
// =====================================================================================================================
extern "C" __global__ void __launch_bounds__(KBS, KMINB) kin_ik_kernel(const __grid_constant__ kin::IkArgs A) {
    using namespace kin;
    constexpr int BS = KBS, ND = KND, ROWS = KROWS;
    const long long li = (long long)blockIdx.x * BS + threadIdx.x;      // position in the active list
    if (li >= A.n) return;
    const long long n = A.idx ? A.idx[li] : li;                         // problem
    const real PI = real(3.14159265358979323846);
    real q[ND], qt[ND], g[ND], tg[6], H[ND][ND];
    {
        const real *q0 = reinterpret_cast<const real *>(A.q0) + n * ND;
        const real *tp = reinterpret_cast<const real *>(A.targets) + n * 6;
        #pragma unroll
        for (int c = 0; c < ND; ++c) { q[c] = q0[c]; qt[c] = q0[c]; g[c] = real(0); }
        #pragma unroll
        for (int i = 0; i < 6; ++i) tg[i] = tp[i];
        #pragma unroll
        for (int a = 0; a < ND; ++a)
            #pragma unroll
            for (int b = 0; b <= a; ++b) H[a][b] = real(0);
    }
    real f = CUDART_INF, lam = (A.lam_io && A.it0 > 0) ? (real)A.lam_io[n] : (real)A.lambda0;
    int it = 0;
    #pragma unroll 1
    for (;; ++it) {
        // ---- evaluate at qt: link transform Tl (3x4 column-major) and Euler-rate Jacobian Jm[j * ROWS + r] ----
        real Tl[12], Jm[ROWS * ND];
        #pragma unroll
        for (int k = 0; k < ROWS * ND; ++k) Jm[k] = real(0);
        {
            #define KQ(c) qt[c]
            #define KST_T(k, v) Tl[k] = (v)
            #define KST_J(k, v) Jm[k] = (v)
            #define KCEN_SET(s, i, v)
            #define KJF_OUT(j, i, v)
            #define KSYNC()
#include "kin_gen_phase1.inc"
        }
        real e[ROWS];
        #pragma unroll
        for (int i = 0; i < 3; ++i) e[i] = Tl[9 + i] - tg[i];
        if (ROWS == 6) {   // rpy(T), transform.jl:45-48 (RotZYX): R[r][c] = Tl[c*3 + r]
            const real yaw = atan2_(Tl[1], Tl[0]);
            real s1, c1;
            sincos_(yaw, &s1, &c1);
            const real pitch = atan2_(-Tl[2], sqrt_(fma_(Tl[5], Tl[5], Tl[8] * Tl[8])));
            const real roll = atan2_(fma_(Tl[6], s1, -(Tl[7] * c1)), fma_(Tl[4], c1, -(Tl[3] * s1)));
            const real ang[3] = {roll - tg[3], pitch - tg[4], yaw - tg[5]};
            #pragma unroll
            for (int i = 0; i < 3; ++i) {            // wrap to (-pi, pi]
                real a = ang[i];
                a = a - real(2) * PI * floor((a + PI) / (real(2) * PI));
                e[3 + i] = a;
            }
        }
        real ft = real(0);
        #pragma unroll
        for (int r = 0; r < ROWS; ++r) ft = fma_(e[r], e[r], ft);
        const bool ok = ft < f;
        if (it > 0) {
            lam *= ok ? real(0.3) : real(4.0);
            lam = lam < real(1e-9) ? real(1e-9) : (lam > real(1e4) ? real(1e4) : lam);
        }
        if (ok) {
            f = ft;
            #pragma unroll
            for (int a = 0; a < ND; ++a) {
                q[a] = qt[a];
                real ga = real(0);
                #pragma unroll
                for (int r = 0; r < ROWS; ++r) ga = fma_(Jm[a * ROWS + r], e[r], ga);
                g[a] = ga;
                #pragma unroll
                for (int b = 0; b <= a; ++b) {
                    real hab = real(0);
                    #pragma unroll
                    for (int r = 0; r < ROWS; ++r) hab = fma_(Jm[a * ROWS + r], Jm[b * ROWS + r], hab);
                    H[a][b] = hab;
                }
            }
        }
        if (f < (real)A.ftol || it >= A.iters) break;
        // ---- step: active set on the limits, Cholesky of H + lam (I + diag H), qt = clamp(q - x) ----
        bool fr[ND];
        real L[ND][ND], x[ND];
        #pragma unroll
        for (int a = 0; a < ND; ++a) {
            const real lo = (real)A.lo[a], hi = (real)A.hi[a];
            fr[a] = !(((q[a] <= lo + real(1e-12)) && (g[a] > real(0))) || ((q[a] >= hi - real(1e-12)) && (g[a] < real(0))));
        }
        #pragma unroll
        for (int a = 0; a < ND; ++a) {
            #pragma unroll
            for (int b = 0; b < a; ++b) L[a][b] = (fr[a] && fr[b]) ? H[a][b] : real(0);
            L[a][a] = fr[a] ? fma_(lam, real(1) + H[a][a], H[a][a]) : real(1);
            x[a] = fr[a] ? g[a] : real(0);
        }
        #pragma unroll
        for (int a = 0; a < ND; ++a) {
            #pragma unroll
            for (int b = 0; b <= a; ++b) {
                real sum = L[a][b];
                #pragma unroll
                for (int k = 0; k < b; ++k) sum = fma_(-L[a][k], L[b][k], sum);
                if (a == b) L[a][a] = sqrt_(sum > real(1e-300) ? sum : real(1e-300));
                else L[a][b] = sum / L[b][b];
            }
        }
        #pragma unroll
        for (int a = 0; a < ND; ++a) {
            real sum = x[a];
            #pragma unroll
            for (int k = 0; k < a; ++k) sum = fma_(-L[a][k], x[k], sum);
            x[a] = sum / L[a][a];
        }
        #pragma unroll
        for (int a = ND - 1; a >= 0; --a) {
            real sum = x[a];
            #pragma unroll
            for (int k = a + 1; k < ND; ++k) sum = fma_(-L[k][a], x[k], sum);
            x[a] = sum / L[a][a];
        }
        #pragma unroll
        for (int a = 0; a < ND; ++a) {
            const real lo = (real)A.lo[a], hi = (real)A.hi[a];
            real v = q[a] - x[a];
            v = v < lo ? lo : (v > hi ? hi : v);
            qt[a] = v;
        }
    }
    real *qo = reinterpret_cast<real *>(A.q_out) + n * ND;
    #pragma unroll
    for (int c = 0; c < ND; ++c) qo[c] = q[c];
    reinterpret_cast<real *>(A.f_out)[n] = f;
    if (A.iters_out) A.iters_out[n] = A.it0 + it;
    if (A.lam_io) A.lam_io[n] = (double)lam;
}
#endif

#if KWARP
// =====================================================================================================================
// Small-batch kernel: one WARP per configuration.  The reference's real callers evaluate ONE configuration per solver
// iteration (IK, inverse_kinematics.jl:38-50) or n_wp = 10 .. 64 per iteration (planning.jl:59-67); with one thread per
// configuration such a call is a single thread walking ~19k dependent instructions (37 us).  Here every lane of the
// warp walks the chain (phase 1 is straight-line, a few microseconds; its stores are spread over the lanes), and in
// phase 2 lane s owns sphere s: its union-SDF search, truncation, gradient and chain rule run side by side.  The one
// thing that couples the spheres -- the shared Jacobian scratch of collision.jl:76,90, through which a sphere inherits
// the columns of joints that do not move it from the last non-truncated sphere before it -- becomes a warp ballot
// ("which earlier lanes wrote column j") and a shuffle from the last of them.  Same helpers, same operation order per
// sphere: results are bit-identical to the other kernels.  KS <= 32.
// =====================================================================================================================
extern "C" __global__ void __launch_bounds__(KBS, 1) kin_gen_kernel(const __grid_constant__ kin::GenArgs A) {
    using namespace kin;
    const int lane = threadIdx.x & 31;
    const long long n = (long long)blockIdx.x * (KBS / 32) + (threadIdx.x >> 5);       // this warp's configuration
    if (n >= A.n) return;
    // all three layouts: SoA, tiled, and AoS (one contiguous record per configuration -- the reference-native layout,
    // which is what a solver callback hands over)
    const size_t es = KAOS ? size_t(1) : KTILED ? size_t(32) : (size_t)A.ld;
    #define KREC_BASE(rec) (KAOS ? n * (long long)(rec) : KTILED ? (n >> 5) * ((long long)(rec) * 32) + (n & 31) : n)
    const real *qn = reinterpret_cast<const real *>(A.q) + KREC_BASE(KND);
    #define KQ(c) __ldg(qn + (size_t)(c) * es)
    // output component k is stored by lane k mod 32 (every lane holds every value)
#if KWANT_T
    real *Tn = reinterpret_cast<real *>(A.T_out) + KREC_BASE(12 * KNFK);
    #define KST_T(k, v) do { if (lane == ((k) & 31)) Tn[(size_t)(k) * es] = (v); } while (0)
#else
    #define KST_T(k, v)
#endif
#if KWANT_J
    real *Jn = reinterpret_cast<real *>(A.J_out) + KREC_BASE(KROWS * KND * KNJAC);
    #define KST_J(k, v) do { if (lane == ((k) & 31)) Jn[(size_t)(k) * es] = (v); } while (0)
#else
    #define KST_J(k, v)
#endif
#if KCOLL
    real px = real(0), py = real(0), pz = real(0);            // the centre of THIS lane's sphere
    #define KCEN_SET(s, i, v) do { if (lane == (s)) { if ((i) == 0) px = (v); else if ((i) == 1) py = (v); else pz = (v); } } while (0)
#else
    #define KCEN_SET(s, i, v)
#endif
    #define KJF_OUT(j, i, v)
    #define KSYNC()
    {
#include "kin_gen_phase1.inc"
#if KCOLL
#include "kin_gen_phase2.inc"
        const bool has = lane < KS;
        const int s = has ? lane : KS - 1;
        const real *tb = reinterpret_cast<const real *>(A.boxes);
        const int n_box = A.n_box;
        const real trunc = (real)A.truncation_dist, voff = (real)A.vals_offset;
        // ---- 2a: union SDF of this lane's sphere (sdf.jl:108-114) ----
        real kmin = CUDART_INF;
        int kidx = 0;
        #pragma unroll 1
        for (int b = 0; b < n_box; ++b) {
            BoxRow<real> row;
            #pragma unroll
            for (int i = 0; i < 9; ++i) row.r[i] = __ldg(tb + b * BOX_REALS + i);
            #pragma unroll
            for (int i = 0; i < 3; ++i) { row.t[i] = __ldg(tb + b * BOX_REALS + 9 + i); row.h[i] = __ldg(tb + b * BOX_REALS + 12 + i); }
            row.kind = KPRIMS ? __ldg(tb + b * BOX_REALS + 15) : real(0);
            const real key = sdf_row_key(tb + b * BOX_REALS, row, px, py, pz);
            if (key < kmin) { kmin = key; kidx = b; }
        }
        const real dmin = key_to_dist(kmin);
        const real dist0 = dmin - KRADIUS[s];
        const bool truncated = dist0 > trunc;
        if (has) {
            reinterpret_cast<real *>(A.vals_out)[KREC_BASE(KS) + (size_t)s * es] = (truncated ? trunc : dist0) - voff;
            if (KARGMIN) A.argmin_out[KREC_BASE(KS) + (size_t)s * es] = kidx + 1;
        }
        if (KGRADS) {
            // ---- 2b: gradient of the argmin box, chain rule through the sphere's Jacobian (collision.jl:78-93) ----
            real grad[3] = {real(0), real(0), real(0)};
            if (has && !truncated) {
                BoxRow<real> row;
                #pragma unroll
                for (int i = 0; i < 9; ++i) row.r[i] = __ldg(tb + kidx * BOX_REALS + i);
                #pragma unroll
                for (int i = 0; i < 3; ++i) { row.t[i] = __ldg(tb + kidx * BOX_REALS + 9 + i); row.h[i] = __ldg(tb + kidx * BOX_REALS + 12 + i); }
                row.kind = KPRIMS ? __ldg(tb + kidx * BOX_REALS + 15) : real(0);
                sdf_row_gradient(tb + kidx * BOX_REALS, row, KGRADMODE >= 0 ? KGRADMODE : A.grad_mode, px, py, pz, dmin, grad);
            }
            const unsigned mask = KSPHMASK[s];
            real *Gp = reinterpret_cast<real *>(A.grads_out) + KREC_BASE((long long)KND * KS) + (size_t)s * KND * es;
            const unsigned below = (1u << lane) - 1u;
            #pragma unroll
            for (int j = 0; j < KND; ++j) {
                const bool mine = has && !truncated && ((mask >> j) & 1u);
                real cx = real(0), cy = real(0), cz = real(0);
                if (mine) jac_col(jfr[j], ((KREV >> j) & 1u) != 0, px, py, pz, cx, cy, cz);
                if (KSTALE) {
                    // the scratch column j as sphere s sees it: written by the last non-truncated sphere before it
                    // that is moved by joint j (collision.jl:76,90), zero if there is none
                    const unsigned writers = __ballot_sync(0xffffffffu, mine);
                    const unsigned prev = writers & below;
                    const int src = prev ? 31 - __clz(prev) : lane;
                    const real sx = __shfl_sync(0xffffffffu, cx, src), sy = __shfl_sync(0xffffffffu, cy, src),
                               sz = __shfl_sync(0xffffffffu, cz, src);
                    if (!mine && prev) { cx = sx; cy = sy; cz = sz; }
                }
                if (has) {
                    real gj = real(0);
                    if (!truncated && (mine || KSTALE)) gj = fma_(grad[0], cx, fma_(grad[1], cy, grad[2] * cz));
                    Gp[(size_t)j * es] = gj;
                }
            }
        }
#endif
    }
}
#endif

#if !KWS && !KIK && !KWARP
#if KQB > 0
__device__ __forceinline__ void kin_grid_barrier(unsigned *sync, unsigned n_cta) {
    __syncthreads();
    if (threadIdx.x == 0) {
        volatile unsigned *gen_p = sync + 1;
        const unsigned gen = *gen_p;
        __threadfence();
        if (atomicAdd(sync, 1u) == n_cta - 1) {
            *sync = 0;
            __threadfence();
            *gen_p = gen + 1;
        } else {
            unsigned polls = 0;
            while (*gen_p == gen) {
                __nanosleep(64);
                if (++polls > (1u << 28)) __trap();     // a barrier that never completes must not hang the GPU
            }
        }
        __threadfence();
    }
    __syncthreads();
}
#endif
#if KSCHED
// bytes [lo, hi) of q into L2, evict_last; the 16-byte-aligned part only (the size of a bulk copy is a multiple of 16 and
// nothing outside q is touched), the few bytes at the ends are left to the loads
__device__ __forceinline__ void l2_prefetch(const void *lo, const void *hi, const unsigned long long pol) {
    const unsigned long long a = ((unsigned long long)lo + 15) & ~15ull, b = (unsigned long long)hi & ~15ull;
    if (b > a) asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(a), "r"((unsigned)(b - a)), "l"(pol) : "memory");
}
// piece p of epoch e: tiles [e E + p E / P, e E + (p + 1) E / P), configurations below n only
__device__ __forceinline__ void prefetch_piece(const kin::GenArgs &A, const long long n_tiles, const long long e, const int p, const int P) {
    using namespace kin;
    const long long t0 = e * KEPOCH + (long long)p * KEPOCH / P, t1 = min(n_tiles, e * KEPOCH + (long long)(p + 1) * KEPOCH / P);
    if (t0 >= t1) return;
    const long long c0 = t0 * KBS, c1 = min(t1 * KBS, A.n);
    const real *q = reinterpret_cast<const real *>(A.q);
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    if (KAOS) {
        l2_prefetch(q + c0 * KND, q + c1 * KND, pol);
    } else if (KTILED) {
        l2_prefetch(q + (c0 >> 5) * (KND * 32), q + ((c1 - 1) >> 5) * (KND * 32) + (KND - 1) * 32 + ((c1 - 1) & 31) + 1, pol);
    } else {
        #pragma unroll 1
        for (int c = 0; c < KND; ++c) l2_prefetch(q + c * A.ld + c0, q + c * A.ld + c1, pol);
    }
}
#endif

#if KBULK
// ---- tiled layout, FK / Jacobian-only kernels: outputs leave through the TMA engine.  In the tiled layout the
//      components of one tile are contiguous (256 B per component for doubles), so a chunk of cnt <= 12 components of a
//      warp's 32 configurations is ONE contiguous cnt x 256 B block: every lane PUTs its values into a [12][32] stage of
//      its warp and lane 0 hands the block to cp.async.bulk (SASS: UBLKCP) -- 29 bulk stores per tile instead of 348
//      STG per thread.  Two stage buffers per warp: a buffer is refilled only after the bulk group issued from it one
//      flush earlier has been read (wait_group.read 1). ----
__device__ __forceinline__ void bulk_store(void *gdst, const void *ssrc, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"((unsigned)__cvta_generic_to_shared(ssrc)), "r"(bytes) : "memory");
}
template <typename real_>
__device__ __forceinline__ void bulk_flush(real_ *gdst, real_ *&b0, real_ *&b1, const int cnt, const bool active, const int lane) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // this lane's stage writes -> visible to the async proxy
    __syncwarp();
    if (lane == 0) {                                                  // (lane 0's column pointer is the buffer's base)
        if (active) bulk_store(gdst, b0, (unsigned)(cnt * 32 * sizeof(real_)));
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");      // an empty group when inactive keeps the count uniform
        asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");  // the OTHER buffer's group has been read
    }
    real_ *t = b0; b0 = b1; b1 = t;
    __syncwarp();
}
#endif

#if KCFILL
// =====================================================================================================================
// The SoA outputs that do not depend on the configuration (GenOptions::const_fill; for Fetch with the 8 arm joints 175
// of the 348 rows of FK-all + gripper Jacobian).  Phase 1 does not store them (KST_* drops the components kcf_T / kcf_J
// list at compile time); this kernel, launched right after kin_gen_kernel on the same stream, writes those KNCF rows,
// columns [0, n), one 32-byte vector (STG.E.ENL2.256) per thread, one short-lived CTA per 256 vectors of a row
// (blockIdx.y = row).  That shape fills at ~7.6 TB/s on B200; a fill inside the persistent kernel -- static split,
// claimed pieces or slices between the tiles -- measured slower than storing the rows per thread (DESIGN 4.4).  CTA 0 of
// a row also writes its scalar head / tail where the row does not start / end on a 32-byte boundary (batch_stride % 4
// != 0, offset pointers, ragged n); padding columns (ld > n) are never touched.
// =====================================================================================================================
__device__ __forceinline__ void st_fill32(double *p, const double v) {
    asm volatile("st.global.v4.f64 [%0], {%1, %1, %1, %1};" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void st_fill32(float *p, const float v) {
    asm volatile("st.global.v8.f32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"l"(p), "f"(v) : "memory");
}
extern "C" __global__ void __launch_bounds__(256) kin_const_fill_kernel(const __grid_constant__ kin::GenArgs A) {
    using namespace kin;
    constexpr int E = 32 / (int)sizeof(real);
    const int row = KCF_ROW[blockIdx.y];
    const real v = KCF_VAL[blockIdx.y];
    real *p = row >= 0 ? reinterpret_cast<real *>(A.T_out) + row * A.ld : reinterpret_cast<real *>(A.J_out) + (-1 - row) * A.ld;
    const long long n = A.n;
    const long long head = min(n, (long long)((32 - ((unsigned long long)p & 31)) & 31) / (long long)sizeof(real));
    const long long body = (n - head) / E, tail = head + body * E;
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < body) st_fill32(p + head + j * E, v);
    if (blockIdx.x == 0) {
        if (threadIdx.x < head) p[threadIdx.x] = v;
        if (tail + threadIdx.x < n) p[tail + threadIdx.x] = v;
    }
}
#endif

extern "C" __global__ void __launch_bounds__(KBS, KMINB) kin_gen_kernel(const __grid_constant__ kin::GenArgs A) {
    using namespace kin;
    constexpr int BS = KBS;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int tid = threadIdx.x;
    real *smem_next = reinterpret_cast<real *>(smem_raw);
#if KCOLL
    real *tb = smem_next;
    const int n_box = A.n_box;
    const int tab_reals = (n_box * BOX_REALS + KS + 1) & ~1;
    real *rad = tb + n_box * BOX_REALS;
    real *scr = tb + tab_reals + tid;                         // scr[slot * BS]
    real *cent0 = scr;
    real *stale0 = scr + 3 * KS * BS;
    real *hand = stale0 + (KSTALE ? 3 * KND : 0) * BS;
    real *jfs = hand + 2 * SPH_GROUP * BS;                    // KJFSMEM: joint frames [6 j + i][thread]
    smem_next = tb + tab_reals + (3 * KS + (KSTALE ? 3 * KND : 0) + 2 * SPH_GROUP + (KJFSMEM ? 6 * KND : 0)) * BS;
    {
        const real *src = reinterpret_cast<const real *>(A.boxes);
        for (int i = tid; i < n_box * BOX_REALS; i += BS) tb[i] = src[i];
        for (int i = tid; i < KS; i += BS) rad[i] = KRADIUS[i];
    }
    __syncthreads();
    const real trunc = (real)A.truncation_dist, voff = (real)A.vals_offset;
#endif
    const size_t es = KAOS ? size_t(1) : KTILED ? size_t(32) : (size_t)A.ld;
#if KAOS
    const int lane = tid & 31;
    real *stw = smem_next + (tid >> 5) * AOS_STAGE_REALS;   // this warp's output stage
    real *stg = stw + lane;
    smem_next += (BS / 32) * AOS_STAGE_REALS;
#endif
#if KBULK
    const int lane = tid & 31;
    real *bst0 = smem_next + (tid >> 5) * (2 * 12 * 32) + lane, *bst1 = bst0 + 12 * 32;     // this lane's column of the warp's two stages
    smem_next += (BS / 32) * (2 * 12 * 32);
#endif
#if KES32 && !KTILED && !KAOS
    // the component stride as a 32-bit value: address = base + es32 * (8 k) is ONE 32 x 32 -> 64-bit multiply-add per
    // store (IMAD.WIDE.U32 with the immediate 8 k) instead of a 64-bit multiply
    const unsigned es32 = (unsigned)A.ld;
    #define KOFF(k) ((unsigned long long)es32 * (unsigned)(k))
#else
    #define KOFF(k) ((size_t)(k) * es)
#endif
#if KSYNC_ON
    #define KSYNC() __syncthreads()
#else
    #define KSYNC()
#endif
    const long long n_tiles = (A.n + BS - 1) / BS;
    auto q_ptr = [&](long long tile_) {
        const long long n_ = min(tile_ * BS + tid, (long long)A.n - 1);
        return reinterpret_cast<const real *>(A.q) + (KAOS ? n_ * KND : KTILED ? (n_ >> 5) * ((long long)KND * 32) + (n_ & 31) : n_);
    };
#if KSCHED
    // claimed tiles (see above): tile is computed, the inputs of tile_nxt are loaded meanwhile, and thread 0 claims the
    // one after (claim_s[i & 1], read by every thread after the barrier that ends tile i)
    __shared__ long long claim_s[2];
    const int pf_pieces = min((int)gridDim.x, KEPOCH);
    long long tile = blockIdx.x, tile_nxt = tile + gridDim.x;
    auto took = [&](const long long t) {
        if (KPFD > 0 && t < n_tiles && t % KEPOCH < pf_pieces) prefetch_piece(A, n_tiles, t / KEPOCH + KPFD, (int)(t % KEPOCH), pf_pieces);
    };
    if (tid == 0) {
        if (KPFD > 0 && (int)blockIdx.x < pf_pieces) {
            #pragma unroll 1
            for (int e = 0; e < KPFD; ++e) prefetch_piece(A, n_tiles, e, blockIdx.x, pf_pieces);
        }
        took(tile);
        took(tile_nxt);
    }
    real qcur[KND > 0 ? KND : 1];
    if (tile < n_tiles) {
        const real *qp = q_ptr(tile);
        #pragma unroll
        for (int c = 0; c < KND; ++c) qcur[c] = KAOS ? __ldg(qp + c) : __ldcs(qp + (size_t)c * es);
    }
    {
        #pragma unroll 1
        for (int claim_i = 0; tile < n_tiles; ++claim_i) {
            if (tid == 0) {
                const long long t = 2ll * gridDim.x + atomicAdd(A.tile_next, 1u);
                claim_s[claim_i & 1] = t;
                took(t);
            }
            real qnxt[KND > 0 ? KND : 1];
            {
                const real *qp = q_ptr(tile_nxt < n_tiles ? tile_nxt : tile);
                #pragma unroll
                for (int c = 0; c < KND; ++c) qnxt[c] = KAOS ? __ldg(qp + c) : __ldcs(qp + (size_t)c * es);
            }
            #define KQ(c) qcur[c]
#elif KQB > 0
    real *sq = smem_next;                                     // [2][KQB][KND][BS]
    const long long my_tiles = (long long)blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const long long max_tiles = (n_tiles + gridDim.x - 1) / gridDim.x, max_batches = (max_tiles + KQB - 1) / KQB;
    auto issue = [&](long long b, int buf) {
        #pragma unroll 1
        for (int r = 0; r < KQB; ++r) {
            const long long k = b * KQB + r;
            if (k < my_tiles) {
                const real *qp = q_ptr(blockIdx.x + k * gridDim.x);
                real *dst = sq + ((size_t)(buf * KQB + r) * KND) * BS + tid;
                #pragma unroll
                for (int c = 0; c < KND; ++c) cp_async_elem(dst + c * BS, qp + (size_t)c * es);
            }
        }
        cp_async_commit();
    };
    kin_grid_barrier(A.sync, gridDim.x);
    issue(0, 0);
    for (long long b = 0; b < max_batches; ++b) {
        const int buf = (int)(b & 1);
        kin_grid_barrier(A.sync, gridDim.x);                  // every SM fetches its next batch NOW
        issue(b + 1, buf ^ 1);
        cp_async_wait<1>();
        __syncthreads();
        #pragma unroll 1
        for (int r = 0; r < KQB; ++r) {
            const long long k = b * KQB + r;
            if (k >= my_tiles) break;
            const long long tile = blockIdx.x + k * gridDim.x;
            const real *sqt = sq + ((size_t)(buf * KQB + r) * KND) * BS + tid;
            #define KQ(c) sqt[(c) * BS]
#else
    // no batching: the configuration of the NEXT tile is loaded into registers while the current one is computed
    real qcur[KND > 0 ? KND : 1];
    if ((long long)blockIdx.x < n_tiles) {
        const real *qp = q_ptr(blockIdx.x);
        #pragma unroll
        for (int c = 0; c < KND; ++c) qcur[c] = KAOS ? __ldg(qp + c) : __ldcs(qp + (size_t)c * es);
    }
    {
        for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            real qnxt[KND > 0 ? KND : 1];
            {
                const long long tn = tile + gridDim.x < n_tiles ? tile + gridDim.x : tile;
                const real *qp = q_ptr(tn);
                #pragma unroll
                for (int c = 0; c < KND; ++c) qnxt[c] = KAOS ? __ldg(qp + c) : __ldcs(qp + (size_t)c * es);
            }
            #define KQ(c) qcur[c]
#endif
            // ---------------- one tile: threads past the end of the batch redo the last configuration (identical
            //                  values, benign duplicate stores) ----------------
            const long long n = min(tile * BS + tid, (long long)A.n - 1);
#if KAOS
            // AoS: the warp's 32 records are written together from the stage (aos_flush); n_w0 = its first record
            const long long n_w0 = tile * BS + (tid & ~31);
            const int nvalid = (int)max(0ll, min(32ll, (long long)A.n - n_w0));
            #define KREC_BASE(rec) (n_w0 * (long long)(rec))
            #define KPUT(cnt, i, v) stg[(i) * aos_ld(cnt)] = (v)
#if KWANT_T
            real *Tw = reinterpret_cast<real *>(A.T_out) + KREC_BASE(12 * KNFK);
            #define KFLUSH_T(off, cnt) aos_flush<real, cnt, 12 * KNFK>(stw, Tw + (off), nvalid, lane)
#endif
#if KWANT_J
            real *Jw = reinterpret_cast<real *>(A.J_out) + KREC_BASE(KROWS * KND * KNJAC);
            #define KFLUSH_J(off, cnt) aos_flush<real, cnt, KROWS * KND * KNJAC>(stw, Jw + (off), nvalid, lane)
#endif
#elif KBULK
            // tiled + bulk stores: the warp's tile is written chunk by chunk from the stage (bulk_flush)
            const long long n_w0 = tile * BS + (tid & ~31);
            const bool w_active = n_w0 < (long long)A.n;
            #define KREC_BASE(rec) ((n_w0 >> 5) * ((long long)(rec) * 32))
            #define KPUT(cnt, i, v) bst0[(i) * 32] = (v)
#if KWANT_T
            real *Tw = reinterpret_cast<real *>(A.T_out) + KREC_BASE(12 * KNFK);
            #define KFLUSH_T(off, cnt) bulk_flush<real>(Tw + (off) * 32, bst0, bst1, cnt, w_active, lane)
#endif
#if KWANT_J
            real *Jw = reinterpret_cast<real *>(A.J_out) + KREC_BASE(KROWS * KND * KNJAC);
            #define KFLUSH_J(off, cnt) bulk_flush<real>(Jw + (off) * 32, bst0, bst1, cnt, w_active, lane)
#endif
#else
            #define KREC_BASE(rec) (KTILED ? (n >> 5) * ((long long)(rec) * 32) + (n & 31) : n)
#if KWANT_T
            real *Tn = reinterpret_cast<real *>(A.T_out) + KREC_BASE(12 * KNFK);
            #define KST_T(k, v) do { if (!kcf_T(k)) __stcs(Tn + KOFF(k), (v)); } while (0)
#else
            #define KST_T(k, v)
#endif
#if KWANT_J
            real *Jn = reinterpret_cast<real *>(A.J_out) + KREC_BASE(KROWS * KND * KNJAC);
            #define KST_J(k, v) do { if (!kcf_J(k)) __stcs(Jn + KOFF(k), (v)); } while (0)
#else
            #define KST_J(k, v)
#endif
#endif
#if KCOLL
            #define KCEN_SET(s, i, v) cent0[(3 * (s) + (i)) * BS] = (v)
#else
            #define KCEN_SET(s, i, v)
#endif
#if KJFSMEM
            #define KJF_OUT(j, i, v) jfs[(6 * (j) + (i)) * BS] = (v)
#else
            #define KJF_OUT(j, i, v)
#endif
            {
#include "kin_gen_phase1.inc"
#if KCOLL
                if (KSTALE && KGRADS) {
                    #pragma unroll
                    for (int i = 0; i < 3 * KND; ++i) stale0[i * BS] = real(0);   // jac = zeros(3, n_dof), collision.jl:76
                }
                real *Vp0 = reinterpret_cast<real *>(A.vals_out) + KREC_BASE(KS);
                real *Gp0 = reinterpret_cast<real *>(A.grads_out) + KREC_BASE((long long)KND * KS);
                int32_t *Ap0 = KARGMIN ? A.argmin_out + KREC_BASE(KS) : nullptr;
                #define KP2AARGS tb, n_box, cent0, hand
#if KJFSMEM
                #define KJFR_DEFINED
                JFrame<real> jfr[KND];                        // unused: the frames were parked in the scratch by KJF_OUT
#endif
#if KAOS
                #define KP2BARGS tb, rad, cent0, stale0, hand, jfr, A.grad_mode, trunc, voff, Vp0, Gp0, Ap0, (size_t)lane, stw, nvalid, jfs, mk
#else
                #define KP2BARGS tb, rad, cent0, stale0, hand, jfr, A.grad_mode, trunc, voff, Vp0, Gp0, Ap0, es, jfs, mk
#endif
#include "kin_gen_phase2.inc"
#endif
            }
#if KSCHED
            __syncthreads();
            tile = tile_nxt;
            tile_nxt = claim_s[claim_i & 1];
            #pragma unroll
            for (int c = 0; c < KND; ++c) qcur[c] = qnxt[c];
        }
    }
#elif KQB > 0
        }
        __syncthreads();                                      // the batch buffer is refilled two iterations later
    }
#else
            #pragma unroll
            for (int c = 0; c < KND; ++c) qcur[c] = qnxt[c];
        }
    }
#endif
#if KBULK
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");     // every bulk store of this warp has completed
#endif
}
#endif

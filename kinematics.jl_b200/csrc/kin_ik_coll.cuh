// kin_ik_coll.cuh -- the collision-CONSTRAINED batched IK of config 4 (BASELINE.json: "1M independent gripper pose
// targets solved in parallel, Jacobian + SDF per iteration"), device resident.
//
// The reference solves   min |[p - p_t; rpy - rpy_t]|^2   s.t.  dists(q) - margin >= 0,  lo <= q <= hi
// (inverse_kinematics.jl:1-30: f_objective :38-50, IneqConst(sscc, joints, sdf, 1, 0.02) with tolerance 1e-8 :14-19,
// bounds :52-63) one problem at a time with NLopt SLSQP (third party).  Here every problem of the batch runs an
// augmented-Lagrangian Levenberg-Marquardt iteration on the same functions:
//     merit  phi(q) = |e(q)|^2 + mu * sum_s psi_s^2,   psi_s = max(0, margin - d_s(q) + lambda_s / mu)
// Per iteration the host issues TWO launches on the caller's stream, with no host synchronisation in between:
//   1. kin_eval (the fused hot-path kernel) at the trial points: link transform, Euler-rate Jacobian, sphere distances
//      and their gradients (truncated at margin + 0.05 like planning.jl:56), SoA;
//   2. ik_coll_step_kernel (this file), one thread per problem: residuals, accept / reject against the merit, first-order
//      multiplier update lambda_s <- mu * psi_s at every accepted point, Gauss-Newton normal equations
//      H = J'J + mu * sum_{psi_s > 0} g_s g_s',  g = J'e - mu * sum psi_s g_s  in registers, joints on a limit that are
//      pushed outward frozen, Cholesky of H + damping (I + diag H), next trial point clamped to the limits.
// A problem stops when |e|^2 < ftol and every constraint holds to ctol.  All state is SoA in a stream-ordered workspace.
// ACTIVE LIST: most problems stop after 2-3 iterations, a few need dozens.  At a handful of iterations (1, 2, 3, 4, 6, 8,
// 12, 16, 24, ...) the still-running problems are compacted into an index list (ik_coll_compact_kernel), the host reads
// its length (8 bytes, one stream synchronisation) and the following launches cover only that many problems: the trial
// points / kin_eval outputs are then indexed by list position i, the solver state by problem act[i].  Between two
// compactions a problem that stops stays in the list (its evaluation is repeated, results ignored).
// SELF-COLLISION (kin_ik_solve_self): a kin_self_collision launch between 1. and 2. evaluates the model's sphere pairs at
// the same trial points, and the SELF instances of the step kernels add the pairs as a second constraint block.
// SEVERAL LINKS (kin_ik_solve_links): kin_eval returns every link's transform and Euler-rate Jacobian, and the LINKS
// instances of the step kernels sum the links' residual blocks into the objective and the normal equations.
#pragma once

#include <cstdint>
#include <type_traits>

namespace kin {

constexpr int IKC_MAX_DOF = 20;         // configuration columns kin_ik_solve accepts (a dual-arm mechanism with the planar base: 17-18)
constexpr int IKC_MAX_DOF_STATIC = 12;  // up to here the step kernel is instantiated per column count (everything in registers)

struct IkCollArgs {
    long long n, ld;                 // problems, SoA stride of every array below
    long long n_act;                 // launch width: length of the active list (== n before the first compaction)
    const int32_t *act;              // list position -> problem (null: identity)
    int n_sph, it, nd;               // nd: configuration columns (read by the run-time-sized instance of the step kernel)
    double margin, mu, ftol, ctol, lambda0, trunc;
    const double *targets;           // [n][6] AoS (caller's)
    const double *T, *J, *V, *G;     // kin_eval outputs at the trial points (SoA)
    double *q_try;                   // [ND][ld]  trial points = input of the next kin_eval (indexed by list position)
    double *q, *H, *g;               // current point, its normal equations (lower triangle, row-major packed) and gradient
    double *phi, *fpose, *damp, *viol, *mult;      // merit, |e|^2, LM damping, max_s (margin - d_s), multipliers [S][ld]
    int32_t *status;                 // 0 running, 1 stopped (converged)
    int32_t *its;                    // iterations used
    double lo[IKC_MAX_DOF], hi[IKC_MAX_DOF];
};

// The self-collision block of kin_ik_solve_self (SELF instances of the step kernels): the hard constraint
// d_p(q) - self_margin >= 0 for every pair p of the model's table, from the kin_self_collision launch of the same
// iteration.  A derived struct, so that the fields of IkCollArgs keep their offsets and the init / compact / finish
// kernels, which take further parameters behind an IkCollArgs, keep theirs.
struct IkCollSelfArgs : IkCollArgs {
    int n_pairs;
    double self_margin, self_trunc;
    const double *VP, *GP;           // pair values [P][ld] and gradients [P][ND][ld] at the trial points (list position)
    double *multP;                   // pair multipliers [P][ld] (problem)
};
// The multi-link pose block of kin_ik_solve_links (LINKS instances of the step kernels): the objective is
// f = sum_l |e_l|^2 over n_links links.  T holds 12 rows per link and J ROWS n_dof rows per link (ROWS = 6 when any link
// has rotation, as kin_eval writes them); a link whose bit of rot_mask is clear contributes its 3 position rows only.
// The targets are [n][6 n_links].  Derived from IkCollSelfArgs so that one struct carries both blocks.
constexpr int IKC_MAX_LINKS = 4;        // KIN_IK_MAX_LINKS
struct IkCollLinksArgs : IkCollSelfArgs {
    int n_links;
    unsigned rot_mask;
};
template <bool SELF, bool LINKS = false>
using IkcArgsT = typename std::conditional<LINKS, IkCollLinksArgs,
                                           typename std::conditional<SELF, IkCollSelfArgs, IkCollArgs>::type>::type;

// e_l = [p - p_t; rpy - rpy_t] of one link (planning.jl:114-138 sign), angles wrapped; Tn points at the link's 12 rows
// of stride ld, tg at its 6 target values.  The same operations as the residual block of the single-link kernels.
__device__ __forceinline__ void ikc_link_residual(const double *Tn, long long ld, const double *tg, bool rot, double e[6]) {
    const double PI = 3.14159265358979323846;
    #pragma unroll
    for (int k = 0; k < 3; ++k) e[k] = Tn[(9 + k) * ld] - tg[k];
    if (rot) {
        const double r00 = Tn[0], r10 = Tn[ld], r20 = Tn[2 * ld], r01 = Tn[3 * ld], r11 = Tn[4 * ld], r21 = Tn[5 * ld],
                     r02 = Tn[6 * ld], r12 = Tn[7 * ld], r22 = Tn[8 * ld];
        const double yaw = atan2(r10, r00);
        double s1, c1;
        sincos(yaw, &s1, &c1);
        const double pitch = atan2(-r20, sqrt(fma(r21, r21, r22 * r22)));
        const double roll = atan2(fma(r02, s1, -(r12 * c1)), fma(r11, c1, -(r01 * s1)));
        const double ang[3] = {roll - tg[3], pitch - tg[4], yaw - tg[5]};
        #pragma unroll
        for (int k = 0; k < 3; ++k) e[3 + k] = ang[k] - 2.0 * PI * floor((ang[k] + PI) / (2.0 * PI));
    } else {
        e[3] = e[4] = e[5] = 0.0;
    }
}

// q0 (AoS, caller's) -> q_try and q (SoA); merit +inf so that the first evaluation is accepted
__global__ void __launch_bounds__(256) ik_coll_init_kernel(const IkCollArgs A, const double *__restrict__ q0, int nd) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= A.n) return;
    for (int a = 0; a < nd; ++a) {
        const double v = fmin(fmax(q0[n * nd + a], A.lo[a]), A.hi[a]);
        A.q_try[a * A.ld + n] = v;
        A.q[a * A.ld + n] = v;
        A.g[a * A.ld + n] = 0.0;
    }
    for (int k = 0; k < nd * (nd + 1) / 2; ++k) A.H[k * A.ld + n] = 0.0;
    for (int s = 0; s < A.n_sph; ++s) A.mult[s * A.ld + n] = 0.0;
    A.phi[n] = CUDART_INF;
    A.fpose[n] = CUDART_INF;
    A.viol[n] = CUDART_INF;
    A.damp[n] = A.lambda0;
    A.status[n] = 0;
    A.its[n] = 0;
}

// Where a problem's normal equations live while a thread works on them.
//   NDT > 0: the column count is a template constant (1 .. IKC_MAX_DOF_STATIC): plain arrays, every loop unrolled,
//            everything in registers.
//   NDT == 0: the column count is read from A.nd at run time (up to IKC_MAX_DOF columns; 17 columns would need 2 x 153
//            doubles of triangle in registers).  The packed lower triangle and the three work vectors sit in SHARED memory,
//            [slot][thread] (conflict free, immediate latency ~30 cycles); the host sizes the CTA so that
//            (nd (nd + 1) / 2 + 3 nd) doubles per thread fit.  (First version: local memory -- ~5000 dependent L2 round
//            trips per thread in the Cholesky loops, 1.5 ms per launch on 42 k problems; ncu launch list in profiles/.)
template <int NDT>
struct IkcStore {
    double H_[NDT][NDT], g_[NDT], x_[NDT], v_[NDT];
    __device__ __forceinline__ IkcStore(double *, int, int, int) {}
    __device__ __forceinline__ double &H(int a, int b) { return H_[a][b]; }
    __device__ __forceinline__ double &g(int a) { return g_[a]; }
    __device__ __forceinline__ double &x(int a) { return x_[a]; }
    __device__ __forceinline__ double &v(int a) { return v_[a]; }
};
template <>
struct IkcStore<0> {
    double *base;
    int bs, tri, nd;
    __device__ __forceinline__ IkcStore(double *smem, int tid, int bs_, int nd_) : base(smem + tid), bs(bs_), tri(nd_ * (nd_ + 1) / 2), nd(nd_) {}
    __device__ __forceinline__ double &H(int a, int b) { return base[(a * (a + 1) / 2 + b) * bs]; }
    __device__ __forceinline__ double &g(int a) { return base[(tri + a) * bs]; }
    __device__ __forceinline__ double &x(int a) { return base[(tri + nd + a) * bs]; }
    __device__ __forceinline__ double &v(int a) { return base[(tri + 2 * nd + a) * bs]; }
};
__host__ __device__ inline size_t ikc_dyn_smem_per_thread(int nd) { return sizeof(double) * (size_t)(nd * (nd + 1) / 2 + 3 * nd); }

// SELF (kin_ik_solve_self): a second constraint block over the self-collision pairs, the same operations per entry as
// the sphere block (merit term mu psi_p^2, multiplier update, rank-one update of H and g where psi_p > 0, viol) and the
// same weight mu, after it.  Written with `if constexpr`: the instances without it are the code they were before.
// LINKS (kin_ik_solve_links, n_links >= 2): the residual and the J'J / J'e accumulation run over the links, link by
// link and row by row.
template <int NDT, bool ROT, bool SELF = false, bool LINKS = false>
__global__ void __launch_bounds__(128) ik_coll_step_kernel(const IkcArgsT<SELF, LINKS> A) {
    extern __shared__ double ikc_smem[];
    constexpr int NDA = NDT > 0 ? NDT : IKC_MAX_DOF;
    const int ND = NDT > 0 ? NDT : A.nd;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // position in the active list
    if (i >= A.n_act) return;
    const long long n = A.act ? A.act[i] : i;                                  // problem
    if (A.status[n]) return;
    constexpr int ROWS = ROT ? 6 : 3;
    const long long ld = A.ld;
    const double PI = 3.14159265358979323846;
    const double mu = A.mu, margin = A.margin;
    const int S = A.n_sph;
    IkcStore<NDT> W(ikc_smem, (int)threadIdx.x, (int)blockDim.x, ND);

    // ---- residual at the trial point: e = [p - p_t; rpy - rpy_t] (planning.jl:114-138 sign), angles wrapped ----
    double e[LINKS ? 6 * IKC_MAX_LINKS : ROWS];
    if constexpr (LINKS) {
        #pragma unroll
        for (int l = 0; l < IKC_MAX_LINKS; ++l)
            if (l < A.n_links) ikc_link_residual(A.T + 12 * l * ld + i, ld, A.targets + n * 6 * A.n_links + 6 * l, (A.rot_mask >> l) & 1u, e + 6 * l);
    } else {
        const double *Tn = A.T + i, *tg = A.targets + n * 6;
        #pragma unroll
        for (int i = 0; i < 3; ++i) e[i] = Tn[(9 + i) * ld] - tg[i];
        if (ROT) {        // rpy(T), transform.jl:45-48 (RotZYX): R[r][c] = T[c*3 + r]
            const double r00 = Tn[0], r10 = Tn[ld], r20 = Tn[2 * ld], r01 = Tn[3 * ld], r11 = Tn[4 * ld], r21 = Tn[5 * ld],
                         r02 = Tn[6 * ld], r12 = Tn[7 * ld], r22 = Tn[8 * ld];
            const double yaw = atan2(r10, r00);
            double s1, c1;
            sincos(yaw, &s1, &c1);
            const double pitch = atan2(-r20, sqrt(fma(r21, r21, r22 * r22)));
            const double roll = atan2(fma(r02, s1, -(r12 * c1)), fma(r11, c1, -(r01 * s1)));
            const double ang[3] = {roll - tg[3], pitch - tg[4], yaw - tg[5]};
            #pragma unroll
            for (int i = 0; i < 3; ++i) e[3 + i] = ang[i] - 2.0 * PI * floor((ang[i] + PI) / (2.0 * PI));
        }
    }
    double ft = 0.0;
    if constexpr (LINKS) {
        #pragma unroll
        for (int l = 0; l < IKC_MAX_LINKS; ++l)
            if (l < A.n_links) {
                const int rl = ((A.rot_mask >> l) & 1u) ? 6 : 3;
                #pragma unroll
                for (int r = 0; r < 6; ++r)
                    if (r < rl) ft = fma(e[6 * l + r], e[6 * l + r], ft);
            }
    } else {
        #pragma unroll
        for (int r = 0; r < ROWS; ++r) ft = fma(e[r], e[r], ft);
    }

    // ---- merit under the CURRENT multipliers ----
    double phi_t = ft;
    for (int s = 0; s < S; ++s) {
        const double d = A.V[s * ld + i];
        const double psi = d >= A.trunc ? 0.0 : fmax(0.0, margin - d + A.mult[s * ld + n] / mu);
        phi_t = fma(mu * psi, psi, phi_t);
    }
    if constexpr (SELF) {
        #pragma unroll 1
        for (int p = 0; p < A.n_pairs; ++p) {
            const double d = A.VP[p * ld + i];
            const double psi = d >= A.self_trunc ? 0.0 : fmax(0.0, A.self_margin - d + A.multP[p * ld + n] / mu);
            phi_t = fma(mu * psi, psi, phi_t);
        }
    }
    const bool ok = phi_t < A.phi[n];
    double damp = A.damp[n];
    if (A.it > 0) {
        damp *= ok ? 0.3 : 4.0;
        damp = fmin(fmax(damp, 1e-9), 1e4);
        A.damp[n] = damp;
    }

    double q[NDA];
    if (ok) {
        // ---- accepted: multipliers, merit and normal equations at this point ----
        #pragma unroll
        for (int a = 0; a < ND; ++a) {
            q[a] = A.q_try[a * ld + i];
            W.g(a) = 0.0;
            #pragma unroll
            for (int b = 0; b <= a; ++b) W.H(a, b) = 0.0;
        }
        if constexpr (LINKS) {
            #pragma unroll
            for (int l = 0; l < IKC_MAX_LINKS; ++l) {
                if (l >= A.n_links) break;
                const int rl = ((A.rot_mask >> l) & 1u) ? 6 : 3;
                const double *Jl = A.J + (long long)l * ROWS * ND * ld;
                double el[6];
                #pragma unroll
                for (int r = 0; r < 6; ++r) el[r] = e[6 * l + r];
                #pragma unroll 1
                for (int r = 0; r < rl; ++r) {
                    #pragma unroll
                    for (int a = 0; a < ND; ++a) W.v(a) = Jl[(long long)(a * ROWS + r) * ld + i];
                    double er = el[0];
                    #pragma unroll
                    for (int k = 1; k < 6; ++k)
                        if (r == k) er = el[k];
                    #pragma unroll
                    for (int a = 0; a < ND; ++a) {
                        const double ja = W.v(a);
                        W.g(a) = fma(ja, er, W.g(a));
                        #pragma unroll
                        for (int b = 0; b <= a; ++b) W.H(a, b) = fma(ja, W.v(b), W.H(a, b));
                    }
                }
            }
        } else {
            #pragma unroll
            for (int r = 0; r < ROWS; ++r) {
                #pragma unroll
                for (int a = 0; a < ND; ++a) W.v(a) = A.J[(long long)(a * ROWS + r) * ld + i];
                #pragma unroll
                for (int a = 0; a < ND; ++a) {
                    const double ja = W.v(a);
                    W.g(a) = fma(ja, e[r], W.g(a));
                    #pragma unroll
                    for (int b = 0; b <= a; ++b) W.H(a, b) = fma(ja, W.v(b), W.H(a, b));
                }
            }
        }
        double phi_n = ft, viol = -CUDART_INF;
        #pragma unroll 1
        for (int s = 0; s < S; ++s) {
            const double d = A.V[s * ld + i];
            double lam = 0.0, psi = 0.0;
            if (d < A.trunc) {
                viol = fmax(viol, margin - d);
                lam = mu * fmax(0.0, margin - d + A.mult[s * ld + n] / mu);    // first-order multiplier update
                psi = fmax(0.0, margin - d + lam / mu);
            }
            A.mult[s * ld + n] = lam;
            if (psi > 0.0) {
                #pragma unroll
                for (int a = 0; a < ND; ++a) W.v(a) = A.G[(long long)(s * ND + a) * ld + i];
                const double w = mu * psi;
                #pragma unroll
                for (int a = 0; a < ND; ++a) {
                    const double ga = W.v(a);
                    W.g(a) = fma(-w, ga, W.g(a));
                    const double ma = mu * ga;
                    #pragma unroll
                    for (int b = 0; b <= a; ++b) W.H(a, b) = fma(ma, W.v(b), W.H(a, b));
                }
                phi_n = fma(w, psi, phi_n);
            }
        }
        if constexpr (SELF) {
            const double sm = A.self_margin;
            #pragma unroll 1
            for (int p = 0; p < A.n_pairs; ++p) {
                const double d = A.VP[p * ld + i];
                double lam = 0.0, psi = 0.0;
                if (d < A.self_trunc) {
                    viol = fmax(viol, sm - d);
                    lam = mu * fmax(0.0, sm - d + A.multP[p * ld + n] / mu);
                    psi = fmax(0.0, sm - d + lam / mu);
                }
                A.multP[p * ld + n] = lam;
                if (psi > 0.0) {                     // only active pairs load their gradient row
                    #pragma unroll
                    for (int a = 0; a < ND; ++a) W.v(a) = A.GP[(long long)(p * ND + a) * ld + i];
                    const double w = mu * psi;
                    #pragma unroll
                    for (int a = 0; a < ND; ++a) {
                        const double ga = W.v(a);
                        W.g(a) = fma(-w, ga, W.g(a));
                        const double ma = mu * ga;
                        #pragma unroll
                        for (int b = 0; b <= a; ++b) W.H(a, b) = fma(ma, W.v(b), W.H(a, b));
                    }
                    phi_n = fma(w, psi, phi_n);
                }
            }
        }
        #pragma unroll
        for (int a = 0; a < ND; ++a) {
            A.q[a * ld + n] = q[a];
            A.g[a * ld + n] = W.g(a);
            #pragma unroll
            for (int b = 0; b <= a; ++b) A.H[(long long)(a * (a + 1) / 2 + b) * ld + n] = W.H(a, b);
        }
        A.phi[n] = phi_n;
        A.fpose[n] = ft;
        A.viol[n] = viol;
        A.its[n] = A.it;
        if (ft < A.ftol && viol <= A.ctol) {       // q_try == q already
            A.status[n] = 1;
            return;
        }
    } else {
        #pragma unroll
        for (int a = 0; a < ND; ++a) {
            q[a] = A.q[a * ld + n];
            W.g(a) = A.g[a * ld + n];
            #pragma unroll
            for (int b = 0; b <= a; ++b) W.H(a, b) = A.H[(long long)(a * (a + 1) / 2 + b) * ld + n];
        }
    }

    // ---- step: active set on the limits, Cholesky of H + damp (I + diag H), q_try = clamp(q - x) ----
    bool fr[NDA];
    #pragma unroll
    for (int a = 0; a < ND; ++a) {
        const double ga = W.g(a);
        fr[a] = !(((q[a] <= A.lo[a] + 1e-12) && (ga > 0.0)) || ((q[a] >= A.hi[a] - 1e-12) && (ga < 0.0)));
    }
    #pragma unroll
    for (int a = 0; a < ND; ++a) {
        #pragma unroll
        for (int b = 0; b < a; ++b) W.H(a, b) = (fr[a] && fr[b]) ? W.H(a, b) : 0.0;
        W.H(a, a) = fr[a] ? fma(damp, 1.0 + W.H(a, a), W.H(a, a)) : 1.0;
        W.x(a) = fr[a] ? W.g(a) : 0.0;
    }
    #pragma unroll
    for (int a = 0; a < ND; ++a) {
        #pragma unroll
        for (int b = 0; b <= a; ++b) {
            double sum = W.H(a, b);
            #pragma unroll
            for (int k = 0; k < b; ++k) sum = fma(-W.H(a, k), W.H(b, k), sum);
            if (a == b) W.H(a, a) = sqrt(sum > 1e-300 ? sum : 1e-300);
            else W.H(a, b) = sum / W.H(b, b);
        }
    }
    #pragma unroll
    for (int a = 0; a < ND; ++a) {
        double sum = W.x(a);
        #pragma unroll
        for (int k = 0; k < a; ++k) sum = fma(-W.H(a, k), W.x(k), sum);
        W.x(a) = sum / W.H(a, a);
    }
    #pragma unroll
    for (int a = ND - 1; a >= 0; --a) {
        double sum = W.x(a);
        #pragma unroll
        for (int k = a + 1; k < ND; ++k) sum = fma(-W.H(k, a), W.x(k), sum);
        W.x(a) = sum / W.H(a, a);
    }
    #pragma unroll
    for (int a = 0; a < ND; ++a) A.q_try[a * ld + i] = fmin(fmax(q[a] - W.x(a), A.lo[a]), A.hi[a]);
}

// Compaction of the active list: every still-running problem of the current list (act_in, or the identity when null)
// appends itself to act_out and takes its trial point along (q_try_in[., i] -> q_try_out[., j]).  The order of the new
// list depends on the scheduling of the atomics; nothing else does (problems are independent, every kernel evaluates a
// configuration the same way wherever it sits).  count[0] must be zero on entry.
__global__ void __launch_bounds__(256) ik_coll_compact_kernel(const IkCollArgs A, int nd, const double *__restrict__ q_try_in,
                                                              int32_t *__restrict__ act_out, double *__restrict__ q_try_out,
                                                              unsigned long long *__restrict__ count) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < A.n_act && !A.status[A.act ? A.act[i] : i];
    // one atomic per warp
    const unsigned ballot = __ballot_sync(0xffffffffu, live);
    if (!ballot) return;
    const int lane = threadIdx.x & 31, leader = __ffs(ballot) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(count, (unsigned long long)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (!live) return;
    const long long j = (long long)base + __popc(ballot & ((1u << lane) - 1u));
    act_out[j] = (int32_t)(A.act ? A.act[i] : i);
    for (int a = 0; a < nd; ++a) q_try_out[a * A.ld + j] = q_try_in[a * A.ld + i];
}

// The same for the staged pose-only solve (kin_gen_skeleton.cuh: kin_ik_kernel, IkArgs::idx): a problem is still running
// while its objective f is >= ftol.  Only the index list is built, the kernel reads the caller's arrays through it.
__global__ void __launch_bounds__(256) ik_compact_kernel(long long n_act, const int32_t *__restrict__ act_in, const double *__restrict__ f,
                                                         double ftol, int32_t *__restrict__ act_out, unsigned long long *__restrict__ count) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n = i < n_act ? (act_in ? act_in[i] : i) : 0;
    const bool live = i < n_act && !(f[n] < ftol);
    const unsigned ballot = __ballot_sync(0xffffffffu, live);
    if (!ballot) return;
    const int lane = threadIdx.x & 31, leader = __ffs(ballot) - 1;
    unsigned long long base = 0;
    if (lane == leader) base = atomicAdd(count, (unsigned long long)__popc(ballot));
    base = __shfl_sync(0xffffffffu, base, leader);
    if (live) act_out[(long long)base + __popc(ballot & ((1u << lane) - 1u))] = (int32_t)n;
}

// q (SoA) -> q_out (AoS, caller's), |e|^2, iterations, and the smallest signed distance of the final configuration
// (from a final UNtruncated distance evaluation Vfin at q)
__global__ void __launch_bounds__(256) ik_coll_finish_kernel(const IkCollArgs A, const double *__restrict__ Vfin, int nd,
                                                             double *__restrict__ q_out, double *__restrict__ f_out,
                                                             int32_t *__restrict__ iters_out, double *__restrict__ dmin_out) {
    const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= A.n) return;
    for (int a = 0; a < nd; ++a) q_out[n * nd + a] = A.q[a * A.ld + n];
    f_out[n] = A.fpose[n];
    if (iters_out) iters_out[n] = A.its[n];
    if (dmin_out) {
        double dm = CUDART_INF;
        for (int s = 0; s < A.n_sph; ++s) dm = fmin(dm, Vfin[s * A.ld + n]);
        dmin_out[n] = dm;
    }
}

}  // namespace kin

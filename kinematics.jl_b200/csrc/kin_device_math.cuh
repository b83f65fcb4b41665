// kin_device_math.cuh -- the per-configuration arithmetic of libkin_b200 as plain device functions: rigid
// transforms (transform.jl), the box SDF in key form and its gradients (sdf.jl:34-41,67-74,108-119), Euler-rate
// coefficients (algorithm.jl:56-63), Jacobian columns (algorithm.jl:65-81).  Shared by the ahead-of-time kernels
// (kin_kernels.cuh) and by the model-specialised kernels that kin_codegen.cpp generates and NVRTC
// compiles at run time (this file is embedded in the library as text for that purpose), so it must compile under
// NVRTC without any host header.
#pragma once
#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#else
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
typedef unsigned long size_t;
#define CUDART_INF __longlong_as_double(0x7ff0000000000000LL)
#endif

namespace kin {

template <typename real> struct Tf { real r[9]; real p[3]; };   // rotation row-major

__device__ __forceinline__ void sincos_(double x, double *s, double *c) { sincos(x, s, c); }
__device__ __forceinline__ void sincos_(float x, float *s, float *c) { sincosf(x, s, c); }
__device__ __forceinline__ double fma_(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float fma_(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double sqrt_(double x) { return sqrt(x); }
__device__ __forceinline__ float sqrt_(float x) { return sqrtf(x); }
__device__ __forceinline__ double atan2_(double y, double x) { return atan2(y, x); }
__device__ __forceinline__ float atan2_(float y, float x) { return atan2f(y, x); }
__device__ __forceinline__ double abs_(double x) { return fabs(x); }
__device__ __forceinline__ float abs_(float x) { return fabsf(x); }
// max(x, 0) without the NaN plumbing of fmax(): clear every bit when the sign bit is set.
// (fmax/fmin on doubles expand to ~8 instructions each on sm_100a; this is 3 integer ops.)
__device__ __forceinline__ double relu_(double x) {
    const int hi = __double2hiint(x), lo = __double2loint(x), m = ~(hi >> 31);
    return __hiloint2double(hi & m, lo & m);
}
__device__ __forceinline__ float relu_(float x) { return fmaxf(x, 0.0f); }

// out = a * b  (a: running transform, b: constant from the table at `c`, R row-major then t)
template <typename real>
__device__ __forceinline__ void tf_mul_const(const Tf<real> &a, const real *__restrict__ c, bool r_identity, Tf<real> &o) {
    // the table row goes to registers first: the compiler cannot prove that scratch stores in between do
    // not alias the table and would otherwise re-load every operand
    const real t0 = c[9], t1 = c[10], t2 = c[11];
    #pragma unroll
    for (int i = 0; i < 3; ++i)
        o.p[i] = fma_(a.r[i * 3 + 0], t0, fma_(a.r[i * 3 + 1], t1, fma_(a.r[i * 3 + 2], t2, a.p[i])));
    if (r_identity) {
        #pragma unroll
        for (int i = 0; i < 9; ++i) o.r[i] = a.r[i];
    } else {
        real m[9];
        #pragma unroll
        for (int i = 0; i < 9; ++i) m[i] = c[i];
        #pragma unroll
        for (int i = 0; i < 3; ++i)
            #pragma unroll
            for (int j = 0; j < 3; ++j)
                o.r[i * 3 + j] = fma_(a.r[i * 3 + 0], m[j], fma_(a.r[i * 3 + 1], m[3 + j], a.r[i * 3 + 2] * m[6 + j]));
    }
}

// KPRIMS: 1 = the SDF table may hold primitives other than boxes (sphere / cylinder rows, an extension beyond the
// reference, which has boxes only: load_urdf.jl:10-15, sdf.jl:92-94); every row loop then tests the row's kind (a
// warp-uniform branch) and leaves the box code path untouched.  The generated kernels define it per model (0 for a
// box-only table: the test compiles out); the ahead-of-time kernels always carry the test.
#ifndef KPRIMS
#define KPRIMS 1
#endif

// One row of the SDF table in registers: inv_R[9] row-major, inv_t[3], half extents[3], kind (slot 15: 0 = box,
// 1 = rounded box -- a sphere is a rounded box with zero half extents --, 2 = cylinder along the local z axis with
// h[0] = radius, h[2] = half length, 3 = voxel grid, see GridHeader); slot 16 holds the rounding radius (read only on
// the general path).
template <typename real> struct BoxRow { real r[9], t[3], h[3], kind; };
__device__ __forceinline__ void load_box(const float *__restrict__ b, BoxRow<float> &o) {
    #pragma unroll
    for (int i = 0; i < 9; ++i) o.r[i] = b[i];
    #pragma unroll
    for (int i = 0; i < 3; ++i) { o.t[i] = b[9 + i]; o.h[i] = b[12 + i]; }
    o.kind = KPRIMS ? b[15] : 0.0f;
}
// FP64 rows are 16-byte aligned (even BOX_REALS, even ro_box, 16-byte aligned table): 8 x 128-bit loads
__device__ __forceinline__ void load_box(const double *__restrict__ b, BoxRow<double> &o) {
    const double2 *b2 = reinterpret_cast<const double2 *>(b);
    double v[16];
    #pragma unroll
    for (int i = 0; i < 8; ++i) { const double2 x = b2[i]; v[2 * i] = x.x; v[2 * i + 1] = x.y; }
    #pragma unroll
    for (int i = 0; i < 9; ++i) o.r[i] = v[i];
    #pragma unroll
    for (int i = 0; i < 3; ++i) { o.t[i] = v[9 + i]; o.h[i] = v[12 + i]; }
    o.kind = v[15];              // the eighth 128-bit load brings it along for free
}

// BoxSDF call (sdf.jl:67-74) in "key" form.  With q = |inv_pose * p| - w/2 and s = |max(q,0)|^2 the
// reference value is d = sqrt(s) + min(max(q), 0); exactly one of the two terms is non-zero, so
//     key = 4 s          if s > 0   (outside: d = sqrt(s) = sqrt(key) / 2 > 0)
//         = min(max q,0) if s == 0  (inside / on the surface: d = key <= 0)
// is a monotone function of d.  The union's argmin (sdf.jl:108-114) is taken on the key with the same
// first-minimum rule, which needs ONE sqrt per sphere instead of one per box; it can differ from the
// reference only when two boxes' distances tie within 1 ulp.
// 2 max(q, 0) = q + |q| exactly, and scaling by 2 / 4 commutes with rounding, so sqrt(key) / 2 is
// bit-identical to sqrt(s): the clamp costs one DADD per axis instead of a compare-and-select.
template <typename real>
__device__ __noinline__ real box_inside_key(real qx, real qy, real qz) {   // rare: centre inside the box
    real t = qx > qy ? qx : qy;
    t = t > qz ? t : qz;
    return t < real(0) ? t : real(0);
}
// outside part of the key and the q vector (needed only if the key turns out to be zero)
template <typename real>
__device__ __forceinline__ real box_key_outside(const BoxRow<real> &b, real px, real py, real pz, real &qx, real &qy, real &qz) {
    const real lx = fma_(b.r[0], px, fma_(b.r[1], py, fma_(b.r[2], pz, b.t[0])));
    const real ly = fma_(b.r[3], px, fma_(b.r[4], py, fma_(b.r[5], pz, b.t[1])));
    const real lz = fma_(b.r[6], px, fma_(b.r[7], py, fma_(b.r[8], pz, b.t[2])));
    qx = abs_(lx) - b.h[0]; qy = abs_(ly) - b.h[1]; qz = abs_(lz) - b.h[2];
    const real mx = qx + abs_(qx), my = qy + abs_(qy), mz = qz + abs_(qz);
    return fma_(mx, mx, fma_(my, my, mz * mz));
}
template <typename real>
__device__ __forceinline__ real box_key(const BoxRow<real> &b, real px, real py, real pz) {
    real qx, qy, qz;
    real key = box_key_outside(b, px, py, pz, qx, qy, qz);
    if (!(key > real(0))) key = box_inside_key(qx, qy, qz);
    return key;
}
template <typename real>
__device__ __forceinline__ real key_to_dist(real key) { return key > real(0) ? real(0.5) * sqrt_(key) : key; }

// 1 / (2 f) for f > 0: a single-precision MUFU.RCP seed refined by Newton steps (two steps: 2^-23 -> 2^-92, i.e. to the
// last bits of a double; one step for a float) -- a full IEEE division costs ~4x more and the kernels are issue bound
__device__ __forceinline__ double half_recip_(double f) {
    float seed;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(seed) : "f"((float)f));
    double r = (double)seed;
    r = fma(r, fma(-f, r, 1.0), r);
    r = fma(r, fma(-f, r, 1.0), r);
    return 0.5 * r;
}
__device__ __forceinline__ float half_recip_(float f) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(f));
    r = fmaf(r, fmaf(-f, r, 1.0f), r);
    return 0.5f * r;
}
__device__ __forceinline__ double copysign_(double x, double s) { return copysign(x, s); }
__device__ __forceinline__ float copysign_(float x, float s) { return copysignf(x, s); }

// closed-form gradient of one box, world frame (extension; KIN_GRAD_ANALYTIC).  f = the box distance at p (already
// known from the union search: |max(q, 0)| outside, max q inside).  Outside: grad = R' (m sigma) / f -- the leading
// term of the forward-difference series below, with one reciprocal and no square root; inside / on the surface: the
// signed axis of the arg-max face.
template <typename real>
__device__ __forceinline__ void box_grad_analytic(const BoxRow<real> &b, real px, real py, real pz, real f, real g[3]) {
    real l[3], q[3];
    l[0] = fma_(b.r[0], px, fma_(b.r[1], py, fma_(b.r[2], pz, b.t[0])));
    l[1] = fma_(b.r[3], px, fma_(b.r[4], py, fma_(b.r[5], pz, b.t[1])));
    l[2] = fma_(b.r[6], px, fma_(b.r[7], py, fma_(b.r[8], pz, b.t[2])));
    #pragma unroll
    for (int i = 0; i < 3; ++i) q[i] = abs_(l[i]) - b.h[i];
    if (f > real(0)) {
        const real hf = half_recip_(f);
        real n2[3];
        #pragma unroll
        for (int i = 0; i < 3; ++i) n2[i] = copysign_(q[i] + abs_(q[i]), l[i]);      // 2 m_k sigma_k (exact clamp)
        // world = R * g_local, and the table holds inv_R = R' row-major => R[r][c] = b.r[c*3 + r]
        #pragma unroll
        for (int r = 0; r < 3; ++r) g[r] = fma_(b.r[0 + r], n2[0], fma_(b.r[3 + r], n2[1], b.r[6 + r] * n2[2])) * hf;
    } else {
        int k = 0;
        if (q[1] > q[k]) k = 1;
        if (q[2] > (k == 1 ? q[1] : q[0])) k = 2;
        const real lk = k == 0 ? l[0] : (k == 1 ? l[1] : l[2]);
        const real sg = lk < real(0) ? real(-1) : real(1);
        #pragma unroll
        for (int r = 0; r < 3; ++r) g[r] = sg * (k == 0 ? b.r[r] : (k == 1 ? b.r[3 + r] : b.r[6 + r]));
    }
}

// The reference's forward difference  g_i = (f(p + eps e_i) - f(p)) / eps,  eps = 1e-7  (sdf.jl:34-41), evaluated
// directly: three more box evaluations and three square roots.
template <typename real>
__device__ __forceinline__ void box_gradient_fd_direct(const BoxRow<real> &b, real px, real py, real pz, real dmin, real g[3]) {
    // the division is done as a multiplication by 1e7 (differs from x / 1e-7 by at most 1 ulp of the quotient).
    // The three evaluations share ONE rare "inside the box" branch so that their dependency chains interleave.
    const real eps = real(1e-7), ieps = real(1e7);
    real k[3], qx[3], qy[3], qz[3];
    k[0] = box_key_outside(b, px + eps, py, pz, qx[0], qy[0], qz[0]);
    k[1] = box_key_outside(b, px, py + eps, pz, qx[1], qy[1], qz[1]);
    k[2] = box_key_outside(b, px, py, pz + eps, qx[2], qy[2], qz[2]);
    if (!(k[0] > real(0)) || !(k[1] > real(0)) || !(k[2] > real(0))) {
        #pragma unroll
        for (int i = 0; i < 3; ++i)
            if (!(k[i] > real(0))) k[i] = box_inside_key(qx[i], qy[i], qz[i]);
    }
    #pragma unroll
    for (int i = 0; i < 3; ++i) g[i] = (key_to_dist(k[i]) - dmin) * ieps;
}

// The same forward-difference QUOTIENT from the closed form of the box distance (FP64 only).
// With l = inv_pose * p, q_k = |l_k| - h_k, sigma_k = sign(l_k) and away from every kink of the SDF (no l_k
// changes sign, no q_k crosses zero, the arg-max of q does not change within eps):
//   outside (f = |max(q,0)| > 0):  f(p + eps e_i)^2 = f^2 + 2 a eps + v eps^2  with  a = sum_k m_k sigma_k R_ki,
//     v = sum_{k: q_k > 0} R_ki^2, hence with u = a / f, w = eps / (2 f):
//         (f(p + eps e_i) - f) / eps = u + (v - u^2) w (1 - 2 u w) + O((eps / f)^3)
//     (first term = the analytic gradient, the rest = exactly the truncation error the reference's FD carries);
//   inside  (f = max_k q_k = q_j < 0):  the quotient is sigma_j R_ji exactly.
// For f > 1e-3 the neglected term is < 1e-12, far below the rounding noise of the direct evaluation itself
// (~2 ulp(f) / eps ~ 1e-9).  Returns false when the point is within 2 eps of a kink, within 1e-3 of the surface
// from outside, or the inside arg-max is not separated by 4 eps: the caller then evaluates the FD directly.
__device__ __forceinline__ bool box_gradient_fd_series(const BoxRow<double> &b, double px, double py, double pz, double f, double g[3]) {
    const double eps = 1e-7;
    double l[3], q[3];
    l[0] = fma(b.r[0], px, fma(b.r[1], py, fma(b.r[2], pz, b.t[0])));
    l[1] = fma(b.r[3], px, fma(b.r[4], py, fma(b.r[5], pz, b.t[1])));
    l[2] = fma(b.r[6], px, fma(b.r[7], py, fma(b.r[8], pz, b.t[2])));
    const double two_eps = 2 * eps;
    #pragma unroll
    for (int k = 0; k < 3; ++k) q[k] = fabs(l[k]) - b.h[k];
    // six DSETPs chained on one predicate (no short-circuit: '&', not '&&')
    const bool clear = (fabs(l[0]) > two_eps) & (fabs(l[1]) > two_eps) & (fabs(l[2]) > two_eps) &
                       (fabs(q[0]) > two_eps) & (fabs(q[1]) > two_eps) & (fabs(q[2]) > two_eps);
    if (!clear) return false;
    if (f > 0.0) {
        if (!(f > 1e-3)) return false;
        // 1 / f to ~1e-14 relative (single-precision seed + one Newton step; f > 1e-3 is well inside the float range):
        // the quotient only has to match the reference's FD to its rounding noise, a full IEEE division costs 4x more
        float seed;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(seed) : "f"((float)f));      // one MUFU.RCP
        const double r0 = (double)seed;
        const double hf = 0.5 * fma(r0, fma(-f, r0, 1.0), r0), w = eps * hf;
        double n2[3], act[3];
        #pragma unroll
        for (int k = 0; k < 3; ++k) {
            n2[k] = copysign(q[k] + fabs(q[k]), l[k]);            // 2 m_k sigma_k (the exact clamp of box_key_outside)
            act[k] = q[k] > 0.0 ? 1.0 : 0.0;
        }
        #pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double r0 = b.r[i], r1 = b.r[3 + i], r2 = b.r[6 + i];               // column i of inv_R
            const double u = fma(n2[0], r0, fma(n2[1], r1, n2[2] * r2)) * hf;         // a / f
            const double v = fma(act[0] * r0, r0, fma(act[1] * r1, r1, act[2] * r2 * r2));
            const double c = fma(-u, u, v);
            g[i] = fma(c * w, fma(-2.0 * u, w, 1.0), u);
        }
        return true;
    }
    // inside: f = max_k q_k; the arg-max must be stable under the perturbation
    int j = 0;
    if (q[1] > q[j]) j = 1;
    if (q[2] > (j == 1 ? q[1] : q[0])) j = 2;
    const double qj = j == 0 ? q[0] : (j == 1 ? q[1] : q[2]);
    double second = -1e300;
    #pragma unroll
    for (int k = 0; k < 3; ++k) if (k != j && q[k] > second) second = q[k];
    if (!(qj - second > 4 * eps)) return false;
    const double lj = j == 0 ? l[0] : (j == 1 ? l[1] : l[2]);
    const double sg = lj < 0.0 ? -1.0 : 1.0;
    #pragma unroll
    for (int i = 0; i < 3; ++i) g[i] = sg * (j == 0 ? b.r[i] : (j == 1 ? b.r[3 + i] : b.r[6 + i]));
    return true;
}
__device__ __forceinline__ bool box_gradient_fd_series(const BoxRow<float> &, float, float, float, float, float[3]) { return false; }

// ---- voxel-grid SDF rows (kind 3, extension; include/kin_b200.h: KinGrid) ----
// A grid row holds the inverse pose (slots 0-11) and kind 3 (slot 15); the device address of its grid storage sits as
// raw bits in the row's last 8 bytes (FP64: slot 17, FP32: slots 16-17, low word first), written explicitly into both
// copies of the table because a conversion of the doubles would destroy it.  The storage starts with this header; the
// float32 samples follow at GRID_VALUES_OFFSET, x fastest.
struct GridHeader {
    int32_t n[3], pad;
    double s, inv_s;            // spacing and 1 / spacing in both precisions
    float s_f, inv_s_f, pad_f[2];
};
constexpr int GRID_VALUES_OFFSET = 64;
static_assert(sizeof(GridHeader) <= GRID_VALUES_OFFSET, "grid header overlaps the values");

__device__ __forceinline__ const GridHeader *grid_of(const double *rowp) {
    return reinterpret_cast<const GridHeader *>(__double_as_longlong(rowp[17]));
}
__device__ __forceinline__ const GridHeader *grid_of(const float *rowp) {
    const unsigned long long lo = __float_as_uint(rowp[16]), hi = __float_as_uint(rowp[17]);
    return reinterpret_cast<const GridHeader *>(lo | (hi << 32));
}
__device__ __forceinline__ void grid_scale(const GridHeader *G, double &s, double &is) { s = __ldg(&G->s); is = __ldg(&G->inv_s); }
__device__ __forceinline__ void grid_scale(const GridHeader *G, float &s, float &is) { s = __ldg(&G->s_f); is = __ldg(&G->inv_s_f); }
template <typename real> __device__ __forceinline__ real lerp_(real a, real b, real t) { return fma_(t, b - a, a); }

// d = f(c) + s |u - c| at the local point l (include/kin_b200.h states the formula and the interpolation order).  With
// GRAD, gl receives its gradient in the grid frame: (1/s) df/dc on the axes where u lies in [0, n-1], (u - c) / |u - c|
// on the others.  The 8 corners are read through the read-only cache (__ldg): a scene-sized grid lives in L2.
template <typename real, bool GRAD>
__device__ __forceinline__ real grid_eval(const GridHeader *G, real lx, real ly, real lz, real gl[3]) {
    real s, is;
    grid_scale(G, s, is);
    const real l[3] = {lx, ly, lz};
    int n[3], i0[3];
    real t[3], e[3];
    #pragma unroll
    for (int k = 0; k < 3; ++k) {
        n[k] = __ldg(&G->n[k]);
        const real top = real(n[k] - 1);
        const real u = fma_(l[k], is, real(0.5) * top);
        const real c = fmin(fmax(u, real(0)), top);         // a NaN coordinate lands on 0: no read outside the grid
        i0[k] = min((int)floor(c), n[k] - 2);
        t[k] = c - real(i0[k]);
        e[k] = u - c;
    }
    const long long nx = n[0], nxy = (long long)n[0] * n[1];
    const float *v = reinterpret_cast<const float *>(reinterpret_cast<const char *>(G) + GRID_VALUES_OFFSET) +
                     ((long long)i0[2] * nxy + (long long)i0[1] * nx + i0[0]);
    const real v000 = __ldg(v), v100 = __ldg(v + 1), v010 = __ldg(v + nx), v110 = __ldg(v + nx + 1);
    const real v001 = __ldg(v + nxy), v101 = __ldg(v + nxy + 1), v011 = __ldg(v + nxy + nx), v111 = __ldg(v + nxy + nx + 1);
    const real a00 = lerp_(v000, v100, t[0]), a10 = lerp_(v010, v110, t[0]);
    const real a01 = lerp_(v001, v101, t[0]), a11 = lerp_(v011, v111, t[0]);
    const real b0 = lerp_(a00, a10, t[1]), b1 = lerp_(a01, a11, t[1]);
    const real f = lerp_(b0, b1, t[2]);
    const real o = sqrt_(fma_(e[0], e[0], fma_(e[1], e[1], e[2] * e[2])));
    if (GRAD) {
        real df[3];
        df[0] = lerp_(lerp_(v100 - v000, v110 - v010, t[1]), lerp_(v101 - v001, v111 - v011, t[1]), t[2]);
        df[1] = lerp_(a10 - a00, a11 - a01, t[2]);
        df[2] = b1 - b0;
        #pragma unroll
        for (int k = 0; k < 3; ++k) gl[k] = e[k] != real(0) ? e[k] / o : df[k] * is;
    }
    return fma_(s, o, f);
}

// ---- primitives other than boxes (extension; KPRIMS) ----
// Signed distance of one general row at p.  Out of line and rare by construction (a scene of boxes never gets here):
// it reads the row through the pointer so that the call carries four arguments.
//   kind 1  rounded box:  d = |max(q, 0)| + min(max q, 0) - rho,  q = |inv_pose p| - h   (sphere: h = 0, rho = radius)
//   kind 2  cylinder:     the same formula on q = (hypot(l_x, l_y) - radius, |l_z| - half length)
//   kind 3  voxel grid:   grid_eval above
template <typename real>
__device__ __noinline__ real prim_dist_general(const real *rowp, real px, real py, real pz) {
    const real lx = fma_(rowp[0], px, fma_(rowp[1], py, fma_(rowp[2], pz, rowp[9])));
    const real ly = fma_(rowp[3], px, fma_(rowp[4], py, fma_(rowp[5], pz, rowp[10])));
    const real lz = fma_(rowp[6], px, fma_(rowp[7], py, fma_(rowp[8], pz, rowp[11])));
    if (rowp[15] == real(3)) return grid_eval<real, false>(grid_of(rowp), lx, ly, lz, nullptr);
    if (rowp[15] == real(2)) {
        const real q0 = sqrt_(fma_(lx, lx, ly * ly)) - rowp[12], q1 = abs_(lz) - rowp[14];
        const real m0 = relu_(q0), m1 = relu_(q1), mx = q0 > q1 ? q0 : q1;
        return sqrt_(fma_(m0, m0, m1 * m1)) + (mx < real(0) ? mx : real(0));
    }
    const real q0 = abs_(lx) - rowp[12], q1 = abs_(ly) - rowp[13], q2 = abs_(lz) - rowp[14];
    const real m0 = relu_(q0), m1 = relu_(q1), m2 = relu_(q2);
    real mx = q0 > q1 ? q0 : q1;
    mx = mx > q2 ? mx : q2;
    return sqrt_(fma_(m0, m0, fma_(m1, m1, m2 * m2))) + (mx < real(0) ? mx : real(0)) - rowp[16];
}
// distance -> the monotone key of the union search (key_to_dist inverts it exactly: sqrt((2 d)^2) = 2 |d| in binary
// floating point)
template <typename real>
__device__ __forceinline__ real dist_to_key(real d) { return d > real(0) ? real(4) * d * d : d; }

// gradient!(sdf, p, out) of a general row: the reference's generic forward difference (sdf.jl:34-41; eps 1e-7, against
// the cached value f), or the closed form with KIN_GRAD_ANALYTIC.
template <typename real>
__device__ __noinline__ void prim_gradient_general(const real *rowp, int grad_mode, real px, real py, real pz, real f, real g[3]) {
    if (grad_mode != 1) {
        const real eps = real(1e-7), ieps = real(1e7);
        g[0] = (prim_dist_general(rowp, px + eps, py, pz) - f) * ieps;
        g[1] = (prim_dist_general(rowp, px, py + eps, pz) - f) * ieps;
        g[2] = (prim_dist_general(rowp, px, py, pz + eps) - f) * ieps;
        return;
    }
    real l[3], gl[3] = {real(0), real(0), real(0)};
    l[0] = fma_(rowp[0], px, fma_(rowp[1], py, fma_(rowp[2], pz, rowp[9])));
    l[1] = fma_(rowp[3], px, fma_(rowp[4], py, fma_(rowp[5], pz, rowp[10])));
    l[2] = fma_(rowp[6], px, fma_(rowp[7], py, fma_(rowp[8], pz, rowp[11])));
    if (rowp[15] == real(3)) {
        grid_eval<real, true>(grid_of(rowp), l[0], l[1], l[2], gl);
    } else if (rowp[15] == real(2)) {
        const real rxy = sqrt_(fma_(l[0], l[0], l[1] * l[1]));
        const real q0 = rxy - rowp[12], q1 = abs_(l[2]) - rowp[14];
        const real m0 = relu_(q0), m1 = relu_(q1), nrm = sqrt_(fma_(m0, m0, m1 * m1));
        const real ux = rxy > real(0) ? l[0] / rxy : real(0), uy = rxy > real(0) ? l[1] / rxy : real(0);
        const real sz = l[2] < real(0) ? real(-1) : real(1);
        if (nrm > real(0)) { gl[0] = m0 / nrm * ux; gl[1] = m0 / nrm * uy; gl[2] = m1 / nrm * sz; }
        else if (q0 > q1) { gl[0] = ux; gl[1] = uy; }
        else gl[2] = sz;
    } else {
        real q[3], m[3];
        #pragma unroll
        for (int i = 0; i < 3; ++i) { q[i] = abs_(l[i]) - rowp[12 + i]; m[i] = relu_(q[i]); }
        const real nrm = sqrt_(fma_(m[0], m[0], fma_(m[1], m[1], m[2] * m[2])));
        if (nrm > real(0)) {
            #pragma unroll
            for (int i = 0; i < 3; ++i) gl[i] = (m[i] / nrm) * (l[i] < real(0) ? real(-1) : real(1));
        } else {
            int k = 0;
            if (q[1] > q[k]) k = 1;
            if (q[2] > (k == 1 ? q[1] : q[0])) k = 2;
            #pragma unroll
            for (int i = 0; i < 3; ++i) if (i == k) gl[i] = l[i] < real(0) ? real(-1) : real(1);
        }
    }
    #pragma unroll
    for (int r = 0; r < 3; ++r) g[r] = fma_(rowp[0 + r], gl[0], fma_(rowp[3 + r], gl[1], rowp[6 + r] * gl[2]));   // R * g_local
}

// key of one table row at p: the box fast path, or the general primitive
template <typename real>
__device__ __forceinline__ real sdf_row_key(const real *rowp, const BoxRow<real> &row, real px, real py, real pz) {
    if (KPRIMS && row.kind != real(0)) return dist_to_key(prim_dist_general(rowp, px, py, pz));
    return box_key(row, px, py, pz);
}

// gradient!(sdf, p, out) on the argmin box (sdf.jl:34-41, 116-119).
// grad_mode 0 = forward difference (series where valid, else direct), 1 = analytic, 2 = forward difference, always direct
template <typename real>
__device__ __forceinline__ void box_gradient(const BoxRow<real> &b, int grad_mode, real px, real py, real pz, real dmin, real g[3]) {
    if (grad_mode == 1) { box_grad_analytic(b, px, py, pz, dmin, g); return; }
    if (grad_mode == 0) {
        if (box_gradient_fd_series(b, px, py, pz, dmin, g)) return;
        box_gradient_fd_direct(b, px, py, pz, dmin, g);
        return;
    }
    box_gradient_fd_direct(b, px, py, pz, dmin, g);
}
// ... on the argmin ROW, whatever its kind
template <typename real>
__device__ __forceinline__ void sdf_row_gradient(const real *rowp, const BoxRow<real> &row, int grad_mode, real px, real py, real pz, real dmin, real g[3]) {
    if (KPRIMS && row.kind != real(0)) { prim_gradient_general(rowp, grad_mode, px, py, pz, dmin, g); return; }
    box_gradient(row, grad_mode, px, py, pz, dmin, g);
}

// Euler-rate coefficients of rpy_derivative! (algorithm.jl:56-63) for the link rotation R (row-major):
// rows 4:6 of a revolute column are (k[0] x - k[1] y, k[2] x + k[3] y, k[4] x + k[5] y + z).
// The reference takes sin/cos of -pitch and -yaw after extracting them with atan2 (transform.jl:45-48);
// sin/cos of an atan2 are ratios of the same matrix entries, so no inverse trigonometry is needed:
//   yaw   = atan2(R21, R11)                  -> cos = R11 / hypot(R11, R21),  sin = R21 / hypot(R11, R21)
//   pitch = atan2(-R31, hypot(R32, R33))     -> cos = hypot(R32, R33) / |row 3| ,  sin = -R31 / |row 3|
template <typename real>
__device__ __forceinline__ void rpy_rate_coeffs(const Tf<real> &T, real k[6]) {
    const real hy = sqrt_(fma_(T.r[0], T.r[0], T.r[3] * T.r[3]));
    const real ihy = real(1) / hy;
    const real cy = hy > real(0) ? T.r[0] * ihy : real(1);      // atan2(0, 0) = 0
    const real sy = hy > real(0) ? T.r[3] * ihy : real(0);
    const real hp = sqrt_(fma_(T.r[7], T.r[7], T.r[8] * T.r[8]));
    const real in = real(1) / sqrt_(fma_(T.r[6], T.r[6], hp * hp));
    const real cp = hp * in, sp = -T.r[6] * in;
    // a2 = -pitch, a3 = -yaw: c2 = cp, s2 = -sp, c3 = cy, s3 = -sy
    const real ic2 = real(1) / cp;
    k[0] = cy * ic2; k[1] = -sy * ic2; k[2] = -sy; k[3] = cy; k[4] = cy * sp * ic2; k[5] = sy * sp * ic2;
}

constexpr int SPH_GROUP = 4;   // spheres evaluated together against each box row (register blocking)
constexpr int JF_REGS = 8;     // joint frames kept in registers when the model has at most this many columns
static_assert(JF_REGS == 8, "the switch statements in kin_eval_kernel enumerate 8 cases");

// World joint frame (origin, axis) of one configuration column: FloatingAxis, mechanism.jl:105-108.
template <typename real> struct JFrame { real o[3], a[3]; };

// One Jacobian column of a point p w.r.t. column j (joint_jacobian!, algorithm.jl:65-81)
template <typename real>
__device__ __forceinline__ void jac_col(const JFrame<real> &f, bool revolute, real px, real py, real pz, real &cx, real &cy, real &cz) {
    if (revolute) {
        const real dx = px - f.o[0], dy = py - f.o[1], dz = pz - f.o[2];
        cx = fma_(f.a[1], dz, -(f.a[2] * dy)); cy = fma_(f.a[2], dx, -(f.a[0] * dz)); cz = fma_(f.a[0], dy, -(f.a[1] * dx));
    } else { cx = f.a[0]; cy = f.a[1]; cz = f.a[2]; }
}


// rows 4:6 of a revolute column under rpy_jac (rpy_derivative!, algorithm.jl:56-63) from the coefficients above;
// every operation explicit so that all kernels (hand-written and generated) round identically
template <typename real>
__device__ __forceinline__ void rpy_rows(const real k[6], real ax, real ay, real az, real &o3, real &o4, real &o5);

// cp.async of one element global -> shared (LDGSTS): the next tile's configuration lands in the scratch
// while the current tile is being computed
__device__ __forceinline__ void cp_async_elem(double *smem_dst, const double *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_elem(float *smem_dst, const float *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Kernel parameter of the model-specialised kernels (kin_gen_skeleton.cuh); shared with the host (kin_b200.cu).
struct GenArgs {
    const void *q;
    void *T_out, *J_out, *vals_out, *grads_out;
    int32_t *argmin_out;
    const void *boxes;           // device: n_box rows of BOX_REALS reals (rewritten in place by kin_model_set_boxes)
    unsigned *tile_next;         // claimed tiles (KSCHED): the tile counter, zeroed before every launch
    unsigned *sync;              // input batching (KQB > 0): two zero-initialised words of the grid-wide barrier
    long long n, ld;
    int n_box, grad_mode;
    double truncation_dist, vals_offset;
};

// Kernel parameter of the generated batched-IK kernel (kin_gen_skeleton.cuh: kin_ik_kernel).
struct IkArgs {
    const void *targets;         // [n][6]: x y z roll pitch yaw
    const void *q0;              // [n][n_dof]
    void *q_out;                 // [n][n_dof]
    void *f_out;                 // [n] pose objective at q_out
    int32_t *iters_out;          // [n] iterations used, or null
    long long n;                 // launch width (length of idx when it is set)
    int iters;
    double ftol, lambda0;
    double lo[32], hi[32];       // joint limits per column (+-inf allowed)
    // staged solve (kin_ik_solve splits a long solve into a few launches over the still-running problems):
    const int32_t *idx;          // list position -> problem (null: identity); every array above is indexed by problem
    double *lam_io;              // [n problems] damping carried from stage to stage (null: lambda0, nothing stored)
    int it0;                     // iterations done by earlier stages (0: first stage, the damping starts at lambda0)
};


// Explicitly rounded single operations (never contracted into an FMA by the compiler): the generated kernels emit
// every multiplication / addition through these, so that their results are bit-for-bit the ones of the hand-written
// kernels, where the same operations appear as arguments of fma() (which are never contracted either).
__device__ __forceinline__ double mul_(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double add_(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double sub_(double a, double b) { return __dadd_rn(a, -b); }
__device__ __forceinline__ float sub_(float a, float b) { return __fadd_rn(a, -b); }

template <typename real>
__device__ __forceinline__ void rpy_rows(const real k[6], real ax, real ay, real az, real &o3, real &o4, real &o5) {
    o3 = fma_(k[0], ax, -mul_(k[1], ay));
    o4 = fma_(k[2], ax, mul_(k[3], ay));
    o5 = add_(fma_(k[4], ax, mul_(k[5], ay)), az);
}

}  // namespace kin

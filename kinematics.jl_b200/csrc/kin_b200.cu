// kin_b200.cu -- C ABI of libkin_b200.so (include/kin_b200.h): model handles, program cache,
// launch configuration and the host-staged variant.  The kernel itself is kin_kernels.cuh.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/kin_b200.h"
#include "kin_kernels.cuh"
#include "kin_ik_coll.cuh"
#include "kin_model.hpp"
#include "kin_codegen.hpp"
#include "kin_jit.hpp"

#include <chrono>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <fstream>

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0}, g_jit_compiles{0}, g_jit_cache_hits{0}, g_jit_launches{0}, g_jit_failures{0};
std::atomic<long long> g_h2d_bytes{0}, g_d2h_bytes{0}, g_host_fill_bytes{0};     // kin_eval_host traffic since load

int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
int fail_cuda(cudaError_t e, const char *what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return KIN_ERR_CUDA;
}
#define CUDA_TRY(expr)                                          \
    do {                                                        \
        cudaError_t e__ = (expr);                               \
        if (e__ != cudaSuccess) return fail_cuda(e__, #expr);   \
    } while (0)

// One NVRTC-compiled, model-specialised kernel (kin_codegen.hpp) of a program, per option set.
struct JitKernel {
    cudaLibrary_t lib = nullptr;
    cudaKernel_t kern = nullptr;
    bool ok = false, from_cache = false;
    int regs = 0, block = 0, occ = 0, slots = 0, smem_limit = 0;
    bool sched = false;             // claimed tiles: a zeroed tile counter per launch
    bool cooperative = false;       // AoS input batching: a grid-wide barrier inside, launched cooperatively
    cudaKernel_t fill = nullptr;    // const_fill: the kernel writing the configuration-independent rows (KNCF of them)
    int fill_rows = 0;
    double compile_ms = 0;
    std::string log;
    ~JitKernel() { if (lib) cudaLibraryUnload(lib); }
};

using KernelFn = void (*)(const kin::KernelArgs);

// What an ahead-of-time kernel instance computes: FK / Jacobian only, with collision, or the self-collision phase
// over the model's pair table instead of phase 2 (kin_self_collision: kin_eval_kernel<..., SELF = true>).
enum Kind { KIND_FKJ = 0, KIND_COLL = 1, KIND_SELF = 2 };

// The ahead-of-time kernel a program runs for one (precision, layout, kind) and its launch shape (configure).
struct LaunchShape {
    KernelFn kernel = nullptr;
    int block = 0, occ = 0, regs = 0;     // block == 0: not configured yet
    size_t smem = 0;
};

struct DeviceProgram {
    kin::Program prog;
    std::mutex jit_mu;
    std::map<std::string, std::shared_ptr<JitKernel>> jit;
    std::atomic<int> small_calls{0};     // small-batch launches of this program so far (see jit_wanted)
    int32_t *d_int = nullptr;
    double *d_r64 = nullptr;
    float *d_r32 = nullptr;
    ~DeviceProgram() { cudaFree(d_int); cudaFree(d_r64); cudaFree(d_r32); }
    LaunchShape shape[2][3][3];          // [precision][layout][kind], configured on first use
};

// A model's self-collision pair table on its device (kin_model_set_self_pairs): 0-based sphere ids.  Reference-counted
// like the programs, so that a launch keeps the table it was given alive while the table is replaced.
struct DevicePairs {
    int2 *d = nullptr;
    int n = 0;
    ~DevicePairs() { cudaFree(d); }
};

// What kin::compile_program builds a program from, and the key of a model's program cache: 0-based ids of the links
// whose transforms and Jacobians it computes, the collision phase and whether that keeps the reference's stale scratch.
struct ProgramRequest {
    std::vector<int> fk, jac;
    bool coll, stale;
    ProgramRequest(const int32_t *fk_links, int n_fk, const int32_t *jac_links, int n_jac, bool coll_, bool stale_)
        : coll(coll_), stale(stale_) {
        for (int i = 0; i < n_fk; ++i) fk.push_back(fk_links[i] - 1);
        for (int i = 0; i < n_jac; ++i) jac.push_back(jac_links[i] - 1);
    }
    // a kin_eval call's: the links of the outputs it asks for; only the presence of the output pointers counts
    explicit ProgramRequest(const KinCall *c)
        : ProgramRequest(c->fk_links, c->T_out ? c->n_fk_links : 0, c->jac_links, c->J_out ? c->n_jac_links : 0, c->vals_out != nullptr,
                         c->vals_out && c->grads_out && c->scratch_mode == KIN_SCRATCH_REFERENCE) {}
    bool operator<(const ProgramRequest &o) const { return std::tie(coll, stale, fk, jac) < std::tie(o.coll, o.stale, o.fk, o.jac); }
    bool compile(const kin::HostModel &hm, kin::Program &p, std::string &err) const {
        return kin::compile_program(hm, fk, jac, coll, stale, kin::JF_REGS, p, err);
    }
};

struct HostStage {          // resources of kin_eval_host, created on first use
    static constexpr int kStreams = 3;
    cudaStream_t stream[kStreams] = {nullptr, nullptr, nullptr};
    void *buf[kStreams] = {nullptr, nullptr, nullptr};
    size_t bytes = 0;
};

}  // namespace

// Device storage of a voxel-grid SDF (kin_grid_create): a kin::GridHeader, then the float32 samples at
// kin::GRID_VALUES_OFFSET.  Shared by the caller's KinGrid handle and every model whose table names the grid.
struct GridStore {
    int device = 0;
    int32_t n[3] = {0, 0, 0};
    void *d = nullptr;
    size_t values() const { return (size_t)n[0] * n[1] * n[2]; }
    ~GridStore();
};
struct KinGrid { std::shared_ptr<GridStore> st; };

struct KinModel {
    kin::HostModel hm;
    std::vector<std::shared_ptr<GridStore>> grids;   // the grids the SDF table names (their rows hold the addresses)
    int device = 0, n_sm = 0, dev_smem = 0;
    cudaMemPool_t pool = nullptr;   // stream-ordered workspace pool that keeps its memory between calls
    std::mutex mu;            // guards hm and the program cache (held only while a program is looked up / compiled)
    std::mutex stage_mu;      // one host-staged call at a time per model (kin_eval_host)
    // programs are reference-counted: a launch keeps its program alive even if kin_model_set_spheres /
    // kin_model_set_boxes on another thread drops the cache entry meanwhile
    std::map<ProgramRequest, std::shared_ptr<DeviceProgram>> cache;
    std::shared_ptr<DevicePairs> self_pairs;   // null: no pair table
    HostStage stage;
};

namespace {

void clear_cache(KinModel *m) { m->cache.clear(); }

// Every entry point that touches the device runs on the model's device, whatever the caller's current device is
// (the pool, the function attributes and the program tables belong to it), and restores the caller's device.
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) switched = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

}  // namespace

GridStore::~GridStore() {
    DeviceGuard guard(device);
    cudaFree(d);
}

namespace {

int load_spheres(kin::HostModel &hm, int32_t n, const int32_t *link, const double *center, const double *radius) {
    if (n < 0 || n > KIN_MAX_SPHERES) return fail(KIN_ERR_LIMIT, "n_spheres exceeds KIN_MAX_SPHERES");
    if (n > 0 && (!link || !center || !radius)) return fail(KIN_ERR_INVALID_ARGUMENT, "null sphere table");
    for (int s = 0; s < n; ++s)          // validate before touching the model: a failed call leaves it unchanged
        if (link[s] < 1 || link[s] > hm.n_links) return fail(KIN_ERR_INVALID_ARGUMENT, "sphere_link id out of range");
    hm.n_sph = n;
    hm.sph_link.assign(n, 0); hm.sph_c.assign(3 * (size_t)n, 0.0); hm.sph_r.assign(n, 0.0);
    for (int s = 0; s < n; ++s) {
        hm.sph_link[s] = link[s] - 1;
        for (int k = 0; k < 3; ++k) hm.sph_c[3 * s + k] = center[3 * s + k];
        hm.sph_r[s] = radius[s];
    }
    return KIN_OK;
}

// The SDF table: boxes (BoxSDF, sdf.jl:48-74) and, as an extension, spheres / cylinders / voxel grids.  kinds == null:
// all boxes.  size: box = full widths; sphere = (radius, -, -); cylinder = (radius, length, -), axis = local z (URDF
// convention); grid: ignored, grids[b] names the grid (grids == null: no grid rows).  device >= 0: every grid must live
// on that device.
int load_prims(kin::HostModel &hm, int32_t n, const int32_t *kinds, const double *pose, const double *size,
               const KinGrid *const *grids = nullptr, int device = -1) {
    if (n < 0 || n > KIN_MAX_BOXES) return fail(KIN_ERR_LIMIT, "n_boxes exceeds KIN_MAX_BOXES");
    if (n > 0 && (!pose || (!size && !grids))) return fail(KIN_ERR_INVALID_ARGUMENT, "null box table");
    for (int b = 0; b < n; ++b) {            // validate before mutating
        const int k = kinds ? kinds[b] : KIN_PRIM_BOX;
        const KinGrid *g = grids ? grids[b] : nullptr;
        if (k != KIN_PRIM_BOX && k != KIN_PRIM_SPHERE && k != KIN_PRIM_CYLINDER && k != KIN_PRIM_GRID)
            return fail(KIN_ERR_INVALID_ARGUMENT, "unknown primitive kind");
        if (k == KIN_PRIM_GRID && !g) return fail(KIN_ERR_INVALID_ARGUMENT, "a KIN_PRIM_GRID row without a grid");
        if (k != KIN_PRIM_GRID && g) return fail(KIN_ERR_INVALID_ARGUMENT, "a grid on a row that is not KIN_PRIM_GRID");
        if (k != KIN_PRIM_GRID && !size) return fail(KIN_ERR_INVALID_ARGUMENT, "null size table");
        if (k != KIN_PRIM_BOX && k != KIN_PRIM_GRID && !(size[3 * b] >= 0.0)) return fail(KIN_ERR_INVALID_ARGUMENT, "negative radius");
        if (g && device >= 0 && g->st->device != device) return fail(KIN_ERR_INVALID_ARGUMENT, "the grid lives on another device");
    }
    hm.n_box = n;
    hm.box_inv.resize(n); hm.box_half.assign(3 * (size_t)n, 0.0);
    hm.box_kind.assign(n, 0); hm.box_round.assign(n, 0.0); hm.box_grid.assign(n, 0ull);
    for (int b = 0; b < n; ++b) {
        kin::Xf P = kin::Xf::from_colmajor16(pose + 16 * b), inv;
        // inv(tf) = (-R' t, R')  (transform.jl:62-65)
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) inv.r[r * 3 + c] = P.r[c * 3 + r];
        for (int r = 0; r < 3; ++r)
            inv.p[r] = (-inv.r[r * 3 + 0]) * P.p[0] + (-inv.r[r * 3 + 1]) * P.p[1] + (-inv.r[r * 3 + 2]) * P.p[2];
        hm.box_inv[b] = inv;
        const int k = kinds ? kinds[b] : KIN_PRIM_BOX;
        if (k == KIN_PRIM_SPHERE) {            // a rounded box with zero half extents
            hm.box_kind[b] = 1; hm.box_round[b] = size[3 * b];
        } else if (k == KIN_PRIM_GRID) {
            hm.box_kind[b] = 3; hm.box_grid[b] = (unsigned long long)(uintptr_t)grids[b]->st->d;
        } else if (k == KIN_PRIM_CYLINDER) {
            hm.box_kind[b] = 2;
            hm.box_half[3 * b] = hm.box_half[3 * b + 1] = size[3 * b];
            hm.box_half[3 * b + 2] = 0.5 * size[3 * b + 1];
        } else {
            for (int i = 0; i < 3; ++i) hm.box_half[3 * b + i] = 0.5 * size[3 * b + i];   // sdf.jl:68
        }
    }
    return KIN_OK;
}
int load_boxes(kin::HostModel &hm, int32_t n, const double *pose, const double *width) { return load_prims(hm, n, nullptr, pose, width); }

int host_model_from_desc(const KinModelDesc *d, kin::HostModel &hm) {
    if (d->n_links <= 0 || d->n_links > KIN_MAX_LINKS) return fail(KIN_ERR_LIMIT, "n_links out of range (KIN_MAX_LINKS)");
    if (d->n_joints < 0 || d->n_joints > KIN_MAX_JOINTS) return fail(KIN_ERR_LIMIT, "n_joints out of range (KIN_MAX_JOINTS)");
    if (!d->parent_link || !d->joint_type || !d->joint_pose || !d->joint_axis || !d->q_index || !d->default_angle)
        return fail(KIN_ERR_INVALID_ARGUMENT, "null mechanism table");
    const int L = d->n_links;
    hm.n_links = L; hm.n_joints = d->n_joints; hm.with_base = d->with_base ? 1 : 0;
    hm.parent.resize(L); hm.jtype.resize(L); hm.qidx.resize(L); hm.pose.resize(L);
    hm.axis.assign(3 * (size_t)L, 0.0); hm.defang.resize(L);
    for (int l = 0; l < L; ++l) {
        const int p = d->parent_link[l];
        if (p == 0 || p < -1 || p > L) return fail(KIN_ERR_INVALID_ARGUMENT, "parent_link must be a 1-based id or -1");
        hm.parent[l] = p < 0 ? -1 : p - 1;
        hm.jtype[l] = d->joint_type[l];
        hm.qidx[l] = d->q_index[l];
        hm.pose[l] = p < 0 ? kin::Xf::identity() : kin::Xf::from_colmajor16(d->joint_pose + 16 * (size_t)l);
        for (int k = 0; k < 3; ++k) hm.axis[3 * l + k] = d->joint_axis[3 * l + k];
        hm.defang[l] = d->default_angle[l];
    }
    std::string err;
    if (!hm.finalize(err)) return fail(KIN_ERR_INVALID_ARGUMENT, err);
    int rc = load_spheres(hm, d->n_spheres, d->sphere_link, d->sphere_center, d->sphere_radius);
    if (rc == KIN_OK) rc = load_boxes(hm, d->n_boxes, d->box_pose, d->box_width);
    return rc;
}

constexpr int kNumBS = 4;
const int kBS[kNumBS] = {128, 96, 64, 32};

// [precision][layout][block size][kind][joint frames in registers]
#define KIN_K(real, lay, bs, coll, self) \
    {kin::kin_eval_kernel<real, lay, bs, coll, 0, self>, kin::kin_eval_kernel<real, lay, bs, coll, kin::JF_REGS, self>}
#define KIN_KINDS(real, lay, bs) {KIN_K(real, lay, bs, false, false), KIN_K(real, lay, bs, true, false), KIN_K(real, lay, bs, true, true)}
#define KIN_BS_ROW(real, lay) {KIN_KINDS(real, lay, 128), KIN_KINDS(real, lay, 96), KIN_KINDS(real, lay, 64), KIN_KINDS(real, lay, 32)}
const KernelFn kKernels[2][3][kNumBS][3][2] = {{KIN_BS_ROW(double, 0), KIN_BS_ROW(double, 1), KIN_BS_ROW(double, 2)},
                                               {KIN_BS_ROW(float, 0), KIN_BS_ROW(float, 1), KIN_BS_ROW(float, 2)}};

// does the program's SDF table hold rows other than boxes (slot 15 of a row = kind)?
bool prog_has_prims(const kin::Program &p) {
    for (int b = 0; b < p.h.n_box; ++b)
        if (p.reals[(size_t)p.h.ro_box + (size_t)b * kin::BOX_REALS + 15] != 0.0) return true;
    return false;
}

// Persistent CTAs: as many as are resident on the device at once, but no more than there are tiles of `block`
// configurations.
long long persistent_grid(const KinModel *m, int occ, int block, long long n) {
    return std::min<long long>((long long)occ * m->n_sm, (n + block - 1) / block);
}

// The CTA size of the program's ahead-of-time kernel of `kind` with the most resident threads.  Called with m->mu held.
int configure(KinModel *m, DeviceProgram *dp, int pi, int li, int kind) {
    const kin::ProgHeader &h = dp->prog.h;
    const int jr = (kind != KIND_FKJ && h.n_dof <= kin::JF_REGS) ? 1 : 0;
    const size_t rs = pi ? sizeof(float) : sizeof(double);
    const size_t tab = sizeof(int32_t) * (size_t)h.n_int + rs * (size_t)h.n_real;
    int dev_smem = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, m->device));
    int best = -1, best_threads = 0, best_occ = 0;
    size_t best_smem = 0;
    for (int bi = 0; bi < kNumBS; ++bi) {
        const int b = kBS[bi];
        size_t smem = tab + rs * (size_t)h.n_slots * b;
        if (li == KIN_LAYOUT_AOS) smem += rs * (size_t)kin::AOS_STAGE_REALS * (b / 32);   // warp-private staging
        if (smem > (size_t)dev_smem) continue;
        KernelFn k = kKernels[pi][li][bi][kind][jr];
        CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, dev_smem));
        int occ = 0;
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, b, smem));
        if (occ * b > best_threads) { best = bi; best_threads = occ * b; best_occ = occ; best_smem = smem; }
    }
    if (best < 0) return fail(KIN_ERR_LIMIT, "model does not fit the shared-memory scratch of one CTA");
    const KernelFn k = kKernels[pi][li][best][kind][jr];
    cudaFuncAttributes fa;
    CUDA_TRY(cudaFuncGetAttributes(&fa, k));
    dp->shape[pi][li][kind] = {k, kBS[best], best_occ, fa.numRegs, best_smem};
    return KIN_OK;
}

int eval_kind(const KinCall *c) { return c->vals_out ? KIND_COLL : KIND_FKJ; }

// The call's program (compiled and uploaded on first use), with the shape of its ahead-of-time kernel of `kind`.
int get_program(KinModel *m, const KinCall *c, int kind, std::shared_ptr<DeviceProgram> &out) {
    const ProgramRequest r(c);
    std::lock_guard<std::mutex> lock(m->mu);
    auto it = m->cache.find(r);
    if (it == m->cache.end()) {
        std::shared_ptr<DeviceProgram> dp = std::make_shared<DeviceProgram>();
        std::string err;
        if (!r.compile(m->hm, dp->prog, err)) return fail(KIN_ERR_INVALID_ARGUMENT, err);
        const kin::Program &p = dp->prog;
        std::vector<float> r32(p.reals.begin(), p.reals.end());
        kin::fix_grid_rows_f32(p.reals.data() + p.h.ro_box, r32.data() + p.h.ro_box, p.h.n_box);
        cudaError_t e;
        if ((e = cudaMalloc(&dp->d_int, sizeof(int32_t) * p.ints.size())) != cudaSuccess ||
            (e = cudaMalloc(&dp->d_r64, sizeof(double) * p.reals.size())) != cudaSuccess ||
            (e = cudaMalloc(&dp->d_r32, sizeof(float) * r32.size())) != cudaSuccess ||
            (e = cudaMemcpy(dp->d_int, p.ints.data(), sizeof(int32_t) * p.ints.size(), cudaMemcpyHostToDevice)) != cudaSuccess ||
            (e = cudaMemcpy(dp->d_r64, p.reals.data(), sizeof(double) * p.reals.size(), cudaMemcpyHostToDevice)) != cudaSuccess ||
            (e = cudaMemcpy(dp->d_r32, r32.data(), sizeof(float) * r32.size(), cudaMemcpyHostToDevice)) != cudaSuccess) {
            return fail_cuda(e, "uploading the kinematic program");
        }
        it = m->cache.emplace(r, dp).first;
    }
    std::shared_ptr<DeviceProgram> dp = it->second;
    const int pi = c->precision == KIN_F32 ? 1 : 0, li = c->layout;
    if (dp->shape[pi][li][kind].block == 0) {
        int rc = configure(m, dp.get(), pi, li, kind);
        if (rc != KIN_OK) return rc;
    }
    out = dp;
    return KIN_OK;
}

// Fails unless a device is present (the entry points that create device state have no CPU fallback).
int require_device() {
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
        cudaGetLastError();
        return fail(KIN_ERR_NO_DEVICE, "no CUDA device: libkin_b200 has no CPU fallback");
    }
    return KIN_OK;
}

constexpr unsigned kAnyLayout = 1u << KIN_LAYOUT_SOA | 1u << KIN_LAYOUT_AOS | 1u << KIN_LAYOUT_TILED32;
constexpr unsigned kSoaAos = 1u << KIN_LAYOUT_SOA | 1u << KIN_LAYOUT_AOS;

// The batch of an entry point: precision, layout (one of the mask `layouts` of 1 << KIN_LAYOUT_*), size and input.
int check_batch(int32_t precision, int32_t layout, long long n, const void *q, unsigned layouts) {
    if (precision != KIN_F64 && precision != KIN_F32) return fail(KIN_ERR_INVALID_ARGUMENT, "unknown precision");
    if (layout != KIN_LAYOUT_SOA && layout != KIN_LAYOUT_AOS && layout != KIN_LAYOUT_TILED32) return fail(KIN_ERR_INVALID_ARGUMENT, "unknown layout");
    if (!(layouts >> layout & 1u)) return fail(KIN_ERR_INVALID_ARGUMENT, "this call supports the SoA and AoS layouts only");
    if (n < 0) return fail(KIN_ERR_INVALID_ARGUMENT, "negative batch size");
    if (n > 0 && !q) return fail(KIN_ERR_INVALID_ARGUMENT, "q is null");
    return KIN_OK;
}

int validate_call(const KinModel *m, const KinCall *c) {
    if (!m || !c) return fail(KIN_ERR_INVALID_ARGUMENT, "null model or call");
    if (int rc = check_batch(c->precision, c->layout, c->n, c->q, kAnyLayout)) return rc;
    if (c->batch_stride != 0 && c->batch_stride < c->n) return fail(KIN_ERR_INVALID_ARGUMENT, "batch_stride < n");
    if (c->T_out && (c->n_fk_links <= 0 || !c->fk_links)) return fail(KIN_ERR_INVALID_ARGUMENT, "T_out without fk_links");
    if (c->J_out && (c->n_jac_links <= 0 || !c->jac_links)) return fail(KIN_ERR_INVALID_ARGUMENT, "J_out without jac_links");
    if (c->n_fk_links > KIN_MAX_LINKS || c->n_jac_links > KIN_MAX_LINKS) return fail(KIN_ERR_LIMIT, "too many requested links");
    if ((c->grads_out || c->argmin_out) && !c->vals_out) return fail(KIN_ERR_INVALID_ARGUMENT, "grads_out/argmin_out need vals_out");
    if (c->vals_out && m->hm.n_sph == 0) return fail(KIN_ERR_INVALID_ARGUMENT, "collision requested but the model has no spheres");
    if (c->vals_out && m->hm.n_box == 0) return fail(KIN_ERR_INVALID_ARGUMENT, "collision requested but the model has no boxes");
    if (c->grad_mode != KIN_GRAD_FD && c->grad_mode != KIN_GRAD_ANALYTIC && c->grad_mode != KIN_GRAD_FD_DIRECT) return fail(KIN_ERR_INVALID_ARGUMENT, "unknown grad_mode");
    if (c->scratch_mode != KIN_SCRATCH_REFERENCE && c->scratch_mode != KIN_SCRATCH_CLEAN) return fail(KIN_ERR_INVALID_ARGUMENT, "unknown scratch_mode");
    if (std::isnan(c->truncation_dist)) return fail(KIN_ERR_INVALID_ARGUMENT, "truncation_dist is NaN");
    return KIN_OK;
}

// ---- model-specialised kernels (kin_codegen.hpp / kin_jit.hpp) ----
constexpr long long kJitMinBatch = 32 * 1024;      // below this the compile is not worth it: interpreting kernels ...
constexpr long long kWarpMaxBatch = 2048;          // ... except for smaller batches that keep coming (a solver loop): after
constexpr int kSmallCallsBeforeJit = 4;            // this many calls of the same program its specialised kernel is built
constexpr long long kSchedMinBatch = 1 << 18;      // claimed tiles + L2 epochs + constant-row fill: from this batch size on

long long env_ll(const char *name, long long dflt) {
    const char *e = std::getenv(name);
    return e && *e ? std::atoll(e) : dflt;
}

int jit_slots(const kin::GenOptions &o, const kin::ProgHeader &h);
size_t jit_smem(const kin::GenOptions &o, const kin::ProgHeader &h, const JitKernel &k);

// Which specialised kernel serves a batch below the large-batch threshold?  Measured (profiles/sweep_midsize.py, fused call,
// device time per launch): one THREAD per configuration 18.7 us at n = 1, 22.7 us at n = 1024 .. 4096, 24.8 us at 16384 --
// one WARP per configuration 31.0 / 32.9 / 96 us -- interpreting kernel 37 / 39 / 40 us.  So the thread-per-configuration
// kernel is the default at every size; the warp-per-configuration kernel is kept for what the other cannot do
// (get_jacobian! semantics -- columns left untouched -- in the AoS layout) and behind KIN_JIT_WARP_MAX.
bool use_warp_kernel(const KinCall *c, const kin::ProgHeader &h) {
    if (c->vals_out && h.n_sph > 32) return false;
    const long long wm = env_ll("KIN_JIT_WARP_MAX", -1);
    if (wm >= 0) return c->n <= wm;
    return c->n <= kWarpMaxBatch && c->layout == KIN_LAYOUT_AOS && c->J_out && c->keep_irrelevant;
}

kin::GenOptions gen_options(const KinModel *m, const KinCall *c, const DeviceProgram *dp) {
    const kin::ProgHeader &h = dp->prog.h;
    kin::GenOptions o;
    // (KIN_JIT_FORCE_PRIMS: compile the row-kind test into a box-only kernel -- build check / cost measurement)
    o.prims = (c->vals_out != nullptr && h.n_sph > 0 && (prog_has_prims(dp->prog) || std::getenv("KIN_JIT_FORCE_PRIMS"))) ? 1 : 0;
    o.precision = c->precision == KIN_F32 ? 1 : 0;
    o.layout = c->layout;
    o.want_T = c->T_out != nullptr && h.n_fk > 0;
    o.want_J = c->J_out != nullptr && h.n_jac > 0;
    o.coll = c->vals_out != nullptr && h.n_sph > 0;
    o.with_rot = c->with_rot ? 1 : 0;
    o.rpy_jac = (o.want_J && c->with_rot && c->rpy_jac) ? 1 : 0;
    o.keep_irrelevant = (o.want_J && c->keep_irrelevant) ? 1 : 0;
    o.want_grads = o.coll && c->grads_out != nullptr;
    o.want_argmin = o.coll && c->argmin_out != nullptr;
    o.stale = o.want_grads && c->scratch_mode == KIN_SCRATCH_REFERENCE;
    // Launch shape and code-shape switches, from the sweeps in profiles/ (sweep_jit.py; ms per 2^22 fused configurations):
    //   collision, SoA:   128 threads x 2 CTAs/SM with a CTA-wide barrier after every node of the straight-line phase 1
    //                     (the warps of a CTA then share instruction fetches: the fused kernel is 90 KB of code, far
    //                     beyond the instruction cache) and 32-bit component strides: 3.68 -> 3.13
    //   collision, tiled: 256 threads x 1 CTA/SM, no barriers: 3.11
    //   FK / Jacobian only: 128 threads, as many CTAs/SM as the registers allow (2), claimed tiles (below)
    const bool tiled = c->layout == KIN_LAYOUT_TILED32;
    // small batches: one warp per configuration (kin_gen_skeleton.cuh, KWARP)
    o.warp = use_warp_kernel(c, h) ? 1 : 0;
    if (o.warp) {
        o.block = 128; o.min_blocks = 1; o.ksync = 0; o.es32 = 0;
        o.grad_mode = o.want_grads ? c->grad_mode : -1;
        return o;
    }
    //   collision, FP32:  an FP32 thread holds half the state, so twice the warps fit if the register allocation is
    //                     bounded accordingly: 256 threads x 2 CTAs/SM (<= 128 registers, 16 warps/SM) instead of 8 warps
    //                     at 254 registers: SoA 1.85 -> 1.61, tiled 1.48 -> 1.46 (profiles/sweep_jit_f32.py)
    const bool f32c = o.coll && o.precision == 1;
    o.block = (int)env_ll("KIN_JIT_BLOCK", ((o.coll && tiled) || f32c) ? 256 : 128);
    o.min_blocks = (int)env_ll("KIN_JIT_MINB", o.coll ? ((tiled && !f32c) ? 1 : 2) : 1);
    o.grad_mode = o.want_grads ? c->grad_mode : -1;
    o.ksync = (int)env_ll("KIN_JIT_KSYNC", (o.coll && !tiled) ? 1 : 0);
    o.es32 = (o.layout == KIN_LAYOUT_SOA && (c->batch_stride ? c->batch_stride : c->n) < (1ll << 32)) ? (int)env_ll("KIN_JIT_ES32", 1) : 0;
    // Models with many columns / spheres (a dual-arm mechanism with the planar base: 18 columns, 19 spheres = 952 B of
    // per-thread shared scratch in FP64): the default shape no longer fits the SM's shared memory.  Measured
    // (profiles/sweep_dual_arm.py, 18 columns, 2^21 configurations, collision-only, ms): what counts is the number of
    // threads per SM -- 96 x 2: 3.27, 128 x 1: 4.87, 160 x 1: 3.88, 192 x 1: 3.28, 224 x 1: 2.84 (interpreting kernel: 6.91);
    // FP32 256 x 1: 2.41, 192 x 2: 1.61, 224 x 2: 1.84, 384 x 1: 1.59, 448 x 1: 1.47 -- so the shape with the most threads
    // that fits is taken (up to what the register file holds: 256 threads at 255 registers, 512 at 128 in FP32).
    // The joint frames of phase 2 stay in registers at any column count: parking them in the shared scratch costs
    // threads and measured slower (DESIGN 7, round 2d).
    if (o.coll && !std::getenv("KIN_JIT_BLOCK")) {
        const size_t cta_max = (size_t)(m ? m->dev_smem : 227 * 1024), sm_total = cta_max + 1024;   // 228 KB per SM, 1 KB reserved per CTA
        auto fits = [&](int block, int minb) {
            JitKernel probe;
            probe.block = block; probe.slots = jit_slots(o, h);
            const size_t need = jit_smem(o, h, probe);
            return need <= cta_max && (size_t)minb * (need + 1024) <= sm_total;
        };
        if (!fits(o.block, o.min_blocks)) {
            const int cap = o.precision == 1 ? 512 : 256;
            int best_b = 32, best_m = 1;
            for (int minb = 1; minb <= 2; ++minb)
                for (int b = 32; b * minb <= cap; b += 32)
                    if (fits(b, minb) && b * minb > best_b * best_m) { best_b = b; best_m = minb; }
            o.block = best_b; o.min_blocks = best_m;
        }
    }
    if (o.layout == KIN_LAYOUT_AOS) o.keep_irrelevant = 0;     // (calls with keep_irrelevant never get here: jit_wanted)
    // tiled FK / Jacobian-only kernels: outputs staged per warp and written by the TMA engine (cp.async.bulk; kin_gen_skeleton.cuh)
    // 2^24 configurations, FK-all + Jacobian: 7.67 -> 7.61 ms (0.950 -> 0.959 of the HBM peak), 8.36 -> 8.05 without the input
    // batching (profiles/sweep_bulk.py): the write path, not the store instructions, bounds the kernel -- a small gain
    o.bulk = (tiled && !o.coll && !o.keep_irrelevant && (o.want_T || o.want_J)) ? (int)env_ll("KIN_JIT_BULK", 1) : 0;
    // FK / Jacobian-only kernels, bound by the DRAM write path: tiles claimed from a counter, the inputs of an epoch of
    // tiles prefetched into L2 in one burst (kin_gen_skeleton.cuh, KSCHED; measurements: DESIGN 4.4, profiles/ab_sched.py).
    // A call that writes little per configuration (the gripper transform + its Jacobian: 480 B) is not write-bound:
    // plain loads, static tiles, 3 CTAs/SM (sweep_jit.py fkg).  Below kSchedMinBatch the static tiles are kept as well,
    // without the constant-row fill and its second launch (profiles/ab_sched.py --sizes).
    // KIN_JIT_EPOCH_MB / KIN_JIT_PF_DIST / KIN_JIT_SCHED_MIN_N: sweep knobs.
    if (h.n_dof > 0 && !o.coll && c->n >= env_ll("KIN_JIT_SCHED_MIN_N", kSchedMinBatch)) {
        const size_t rs = o.precision ? sizeof(float) : sizeof(double);
        const size_t out_bytes = rs * ((o.want_T ? (size_t)12 * h.n_fk : 0) + (o.want_J ? (size_t)(o.with_rot ? 6 : 3) * h.n_dof * h.n_jac : 0));
        // AoS: the claimed tiles measured slower than the input batches (2^22 configurations: 2.44 against 1.89 ms,
        // DESIGN 4.4), so that layout keeps them: the configurations of as many tiles as fit twice in ~176 KB fetched
        // per batch with cp.async, behind a grid-wide barrier (one CTA per SM, cooperative launch)
        const long long qb = std::min<long long>(16, (long long)((std::min<size_t>((size_t)(m ? m->dev_smem : 227 * 1024), 200 * 1024) - 24 * 1024) /
                                                                 (2 * (size_t)h.n_dof * o.block * rs)));
        if (out_bytes >= 1024 && o.layout == KIN_LAYOUT_AOS && qb >= 2) {
            o.qbatch = (int)qb;
            o.min_blocks = 1;
        } else if (out_bytes >= 1024) {
            o.sched = 1;
            o.epoch = (int)std::max<long long>(1, (env_ll("KIN_JIT_EPOCH_MB", 8) << 20) / ((long long)o.block * h.n_dof * rs));
            o.pf_dist = (int)env_ll("KIN_JIT_PF_DIST", 1);
        }
    }
    // ... whose rows that do not depend on the configuration (175 of the 348 of FK-all + gripper Jacobian for Fetch) are
    // then written by a second, fill-shaped kernel instead of one store per configuration (kin_gen_skeleton.cuh:
    // kin_const_fill_kernel; DESIGN 4.4).  SoA only: a constant row is one contiguous run there, not in the tiled / AoS
    // layouts.  (KIN_JIT_CONST_FILL=0 stores every row per thread, for A/B measurements.)
    if (o.layout == KIN_LAYOUT_SOA && o.sched && (o.want_T || o.want_J))
        o.const_fill = (int)env_ll("KIN_JIT_CONST_FILL", 1) ? 1 : 0;
    return o;
}

// The links a solve places (kin_ik_solve / kin_ik_solve_self: the call's one link; kin_ik_solve_links: up to
// KIN_IK_MAX_LINKS), in the order of the targets.  rows: residual rows per link in the kin_eval Jacobian (6 when any
// link has rotation).
static_assert(kin::IKC_MAX_LINKS == KIN_IK_MAX_LINKS, "the step kernels hold KIN_IK_MAX_LINKS residual blocks");
struct IkLinks {
    int n = 1;
    int32_t ids[KIN_IK_MAX_LINKS] = {};
    unsigned rot_mask = 0;
    int rows() const { return rot_mask ? 6 : 3; }
};
IkLinks ik_one_link(const KinIkCall *c) {
    IkLinks lk;
    lk.ids[0] = c->link_id;
    lk.rot_mask = c->with_rot ? 1u : 0u;
    return lk;
}

// The generated one-launch IK kernel (kin_gen_skeleton.cuh: kin_ik_kernel) around the links' FK + Euler-rate Jacobians
// (FP64 SoA, 128 threads: the defaults of GenOptions).
kin::GenOptions ik_gen_options(const IkLinks &lk) {
    kin::GenOptions o;
    o.want_T = o.want_J = true; o.with_rot = lk.rot_mask ? 1 : 0; o.rpy_jac = 1;
    o.ik = 1; o.ik_rot = lk.n > 1 ? lk.rot_mask : 0u;
    return o;
}

bool jit_wanted(const KinModel *m, const KinCall *c, const DeviceProgram *dp, bool count) {
    (void)m;
    if (std::getenv("KIN_DISABLE_JIT")) return false;
    const bool small = use_warp_kernel(c, dp->prog.h);
    // large AoS batches: outputs staged through shared memory (kin_gen_skeleton.cuh: aos_flush); get_jacobian!
    // semantics (columns left untouched) cannot be staged and stay with the interpreting kernel
    if (c->layout == KIN_LAYOUT_AOS && !small && c->J_out && c->keep_irrelevant) return false;
    if (dp->prog.h.n_dof > 32) return false;                   // relevance masks of the generated phase 2 are 32 bits wide
    if (c->n < env_ll("KIN_JIT_MIN_BATCH", kJitMinBatch) && !std::getenv("KIN_FORCE_JIT")) {
        // a batch too small to be worth a compile on its own: specialise once the same program keeps being called, as a
        // solver callback (one configuration, n_wp waypoints, the active list of the batched IK) does
        if (std::getenv("KIN_JIT_NO_SMALL")) return false;
        std::atomic<int> &calls = const_cast<DeviceProgram *>(dp)->small_calls;
        return (count ? calls.fetch_add(1) + 1 : calls.load()) >= kSmallCallsBeforeJit;
    }
    return true;
}

std::string jit_main_source() {
    return "#include \"kin_gen_config.h\"\n#include \"kin_device_math.cuh\"\n#include \"kin_gen_skeleton.cuh\"\n";
}

kin::JitHeaders jit_headers(const kin::GenSource &g) {
    kin::JitHeaders hs;
    std::string cfg = g.config;
    cfg += "namespace kin { constexpr int BOX_REALS = " + std::to_string(kin::BOX_REALS) + "; }\n";
    hs.emplace_back("kin_gen_config.h", cfg);
    hs.emplace_back("kin_device_math.cuh", kin::embedded_device_math());
    hs.emplace_back("kin_gen_skeleton.cuh", kin::embedded_gen_skeleton());
    hs.emplace_back("kin_gen_phase1.inc", g.phase1);
    hs.emplace_back("kin_gen_phase2.inc", g.phase2);
    return hs;
}

// per-thread scratch slots of the generated kernel (kin_gen_skeleton.cuh)
int jit_slots(const kin::GenOptions &o, const kin::ProgHeader &h) {
    if (!o.coll) return 0;
    return 3 * h.n_sph + (o.stale ? 3 * h.n_dof : 0) + 2 * kin::SPH_GROUP;
}

size_t jit_smem(const kin::GenOptions &o, const kin::ProgHeader &h, const JitKernel &k) {
    const size_t rs = o.precision ? sizeof(float) : sizeof(double);
    size_t reals = 0;
    if (o.warp) return 0;                  // the one-warp-per-configuration kernel keeps everything in registers
    if (o.coll) reals += (((size_t)h.n_box * kin::BOX_REALS + h.n_sph + 1) & ~size_t(1)) + (size_t)k.slots * k.block;
    if (o.layout == KIN_LAYOUT_AOS)      // the warps' output stages (AOS_STAGE_ROWS x 33 per warp)
        reals += (size_t)(k.block / 32) * (34 * std::max(12, (int)h.n_dof) + (o.coll ? 2 * 36 * kin::SPH_GROUP : 0));   // AOS_STAGE_REALS
    if (o.bulk && o.layout == KIN_LAYOUT_TILED32) reals += (size_t)k.block * 24;     // (block / 32) warps x 2 stages x 12 x 32
    if (o.qbatch > 0) reals += (size_t)2 * o.qbatch * h.n_dof * k.block;
    return rs * reals;
}

// Returns the compiled kernel for this option set (compiling it on first use), or null when specialisation is
// unavailable for it (NVRTC missing, compile error, does not fit): the caller then uses the interpreting kernels.
std::shared_ptr<JitKernel> get_jit_with(KinModel *m, DeviceProgram *dp, const kin::GenOptions &o, const char *kernel_name) {
    const std::string key = o.key();
    std::lock_guard<std::mutex> lock(dp->jit_mu);
    auto it = dp->jit.find(key);
    if (it != dp->jit.end()) return it->second->ok ? it->second : nullptr;
    auto k = std::make_shared<JitKernel>();
    dp->jit[key] = k;
    const auto t0 = std::chrono::steady_clock::now();
    kin::GenSource g;
    std::string err;
    if (!kin::generate_source(dp->prog, o, g, err)) { k->log = "codegen: " + err; g_jit_failures.fetch_add(1); return nullptr; }
    std::vector<char> cubin;
    bool cached = false;
    if (!kin::jit_compile(jit_main_source(), jit_headers(g), "sm_100a", cubin, k->log, &cached)) {
        g_jit_failures.fetch_add(1);
        if (std::getenv("KIN_JIT_VERBOSE")) std::fprintf(stderr, "[libkin_b200] specialisation failed, using the interpreting kernel: %s\n", k->log.c_str());
        return nullptr;
    }
    k->from_cache = cached;
    (cached ? g_jit_cache_hits : g_jit_compiles).fetch_add(1);
    cudaError_t e = cudaLibraryLoadData(&k->lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e == cudaSuccess) e = cudaLibraryGetKernel(&k->kern, k->lib, kernel_name);
    cudaFuncAttributes fa;
    if (e == cudaSuccess) e = cudaFuncGetAttributes(&fa, (const void *)k->kern);
    if (e != cudaSuccess) {
        k->log = std::string("loading the compiled kernel: ") + cudaGetErrorString(e);
        cudaGetLastError();
        g_jit_failures.fetch_add(1);
        return nullptr;
    }
    k->regs = fa.numRegs;
    k->block = o.block;
    k->slots = jit_slots(o, dp->prog.h);
    const size_t smem = jit_smem(o, dp->prog.h, *k);
    if (smem > (size_t)m->dev_smem) { k->log = "scratch does not fit in shared memory"; g_jit_failures.fetch_add(1); return nullptr; }
    if (smem > 48 * 1024) {
        e = cudaFuncSetAttribute((const void *)k->kern, cudaFuncAttributeMaxDynamicSharedMemorySize, m->dev_smem);
        if (e != cudaSuccess) { k->log = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e); cudaGetLastError(); g_jit_failures.fetch_add(1); return nullptr; }
    }
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&k->occ, (const void *)k->kern, k->block, smem);
    if (e != cudaSuccess || k->occ < 1) { k->log = "occupancy query failed"; cudaGetLastError(); g_jit_failures.fetch_add(1); return nullptr; }
    k->sched = o.sched != 0;
    k->cooperative = o.qbatch > 0;
    k->fill_rows = g.config.find("#define KCFILL 1") != std::string::npos ? (int)(g.const_T.size() + g.const_J.size()) : 0;
    if (k->fill_rows > 0 && cudaLibraryGetKernel(&k->fill, k->lib, "kin_const_fill_kernel") != cudaSuccess) {
        k->log = "loading the constant-row fill kernel";
        cudaGetLastError();
        g_jit_failures.fetch_add(1);
        return nullptr;
    }
    k->compile_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (std::getenv("KIN_JIT_VERBOSE"))
        std::fprintf(stderr, "[libkin_b200] specialised kernel %s: %d registers, %zu B shared, %d CTAs/SM, %.0f ms%s\n", key.c_str(), k->regs, smem,
                     k->occ, k->compile_ms, cached ? " (disk cache)" : "");
    k->ok = true;
    return k;
}

// Which kernel a kin_eval call runs and with what launch shape: launch() launches it, kin_query_launch() reports it.
struct LaunchPlan {
    std::shared_ptr<JitKernel> jit;     // the model-specialised kernel, or null: `kernel`, an interpreting one
    kin::GenOptions opt;                // the option set of `jit`
    KernelFn kernel = nullptr;
    int block = 0, regs = 0;
    long long grid = 0;
    size_t smem = 0;
};

// The ahead-of-time kernel of `kind` with the shape get_program configured for it.
LaunchPlan plan_ahead_of_time(const KinModel *m, const KinCall *c, const DeviceProgram *dp, int kind) {
    const LaunchShape &s = dp->shape[c->precision == KIN_F32 ? 1 : 0][c->layout][kind];
    LaunchPlan p;
    p.kernel = s.kernel;
    p.block = s.block; p.regs = s.regs; p.smem = s.smem;
    p.grid = persistent_grid(m, s.occ, s.block, c->n);
    return p;
}

// count_small_calls: whether this call counts towards specialising a program that keeps being called with small
// batches (jit_wanted).
LaunchPlan plan_launch(KinModel *m, const KinCall *c, DeviceProgram *dp, bool count_small_calls) {
    if (jit_wanted(m, c, dp, count_small_calls)) {
        LaunchPlan p;
        p.opt = gen_options(m, c, dp);
        p.jit = get_jit_with(m, dp, p.opt, "kin_gen_kernel");
        if (p.jit) {
            const JitKernel &k = *p.jit;
            p.block = k.block; p.regs = k.regs;
            p.smem = jit_smem(p.opt, dp->prog.h, k);
            p.grid = p.opt.warp ? (c->n + k.block / 32 - 1) / (k.block / 32)      // one warp per configuration, not persistent
                                : persistent_grid(m, k.occ, k.block, c->n);
            return p;
        }
    }
    return plan_ahead_of_time(m, c, dp, eval_kind(c));
}

int launch_jit(KinModel *m, const KinCall *c, DeviceProgram *dp, const LaunchPlan &p, cudaStream_t stream) {
    const kin::GenOptions &o = p.opt;
    const JitKernel &k = *p.jit;
    const kin::ProgHeader &h = dp->prog.h;
    kin::GenArgs a;
    std::memset(&a, 0, sizeof a);
    a.q = c->q;
    a.T_out = c->T_out; a.J_out = c->J_out; a.vals_out = c->vals_out; a.grads_out = c->grads_out; a.argmin_out = c->argmin_out;
    a.boxes = o.precision ? (const void *)(dp->d_r32 + h.ro_box) : (const void *)(dp->d_r64 + h.ro_box);
    a.n = c->n; a.ld = c->batch_stride ? c->batch_stride : c->n;
    a.n_box = h.n_box; a.grad_mode = c->grad_mode;
    a.truncation_dist = c->truncation_dist; a.vals_offset = c->vals_offset;
    void *args[] = {&a};
    if (k.sched) {
        // a zero-initialised tile counter per launch (stream-ordered, so concurrent launches have their own)
        unsigned *next = nullptr;
        CUDA_TRY(cudaMallocFromPoolAsync((void **)&next, sizeof(unsigned), m->pool, stream));
        a.tile_next = next;
        cudaError_t e = cudaMemsetAsync(next, 0, sizeof(unsigned), stream);
        if (e == cudaSuccess) e = cudaLaunchKernel((const void *)k.kern, dim3((unsigned)p.grid), dim3((unsigned)k.block), args, p.smem, stream);
        cudaFreeAsync(next, stream);
        if (e != cudaSuccess) return fail_cuda(e, "launching the specialised kernel");
    } else if (k.cooperative) {
        // two zero-initialised barrier words per launch (stream-ordered, so concurrent launches have their own)
        unsigned *sync = nullptr;
        CUDA_TRY(cudaMallocFromPoolAsync((void **)&sync, 2 * sizeof(unsigned), m->pool, stream));
        cudaError_t e = cudaMemsetAsync(sync, 0, 2 * sizeof(unsigned), stream);
        a.sync = sync;
        cudaLaunchConfig_t cfg;
        std::memset(&cfg, 0, sizeof cfg);
        cfg.gridDim = dim3((unsigned)p.grid); cfg.blockDim = dim3((unsigned)k.block);
        cfg.dynamicSmemBytes = p.smem; cfg.stream = stream;
        cudaLaunchAttribute attr;
        attr.id = cudaLaunchAttributeCooperative;
        attr.val.cooperative = 1;
        cfg.attrs = &attr; cfg.numAttrs = 1;
        if (e == cudaSuccess) e = cudaLaunchKernelExC(&cfg, (const void *)k.kern, args);
        cudaFreeAsync(sync, stream);
        if (e != cudaSuccess) return fail_cuda(e, "launching the specialised kernel (cooperative)");
    } else {
        CUDA_TRY(cudaLaunchKernel((const void *)k.kern, dim3((unsigned)p.grid), dim3((unsigned)k.block), args, p.smem, stream));
    }
    g_launches.fetch_add(1);
    g_jit_launches.fetch_add(1);
    if (k.fill_rows > 0) {
        // one 32-byte vector per thread, 256 threads per CTA, blockIdx.y = constant row
        const long long vec = 32 / (o.precision ? sizeof(float) : sizeof(double));
        const long long gx = (c->n / vec + 1 + 255) / 256;
        CUDA_TRY(cudaLaunchKernel((const void *)k.fill, dim3((unsigned)gx, (unsigned)k.fill_rows), dim3(256), args, 0, stream));
        g_launches.fetch_add(1);
        g_jit_launches.fetch_add(1);
    }
    return KIN_OK;
}

// The arguments of an ahead-of-time kernel for a call (the self-collision fields stay zero).
kin::KernelArgs kernel_args(const KinCall *c, const DeviceProgram *dp) {
    kin::KernelArgs a;
    std::memset(&a, 0, sizeof a);
    a.h = dp->prog.h;
    a.tab_i = dp->d_int;
    a.tab_r = c->precision == KIN_F32 ? (const void *)dp->d_r32 : (const void *)dp->d_r64;
    a.q = c->q;
    a.T_out = c->T_out; a.J_out = c->J_out; a.vals_out = c->vals_out; a.grads_out = c->grads_out;
    a.argmin_out = c->argmin_out;
    a.n = c->n; a.ld = c->batch_stride ? c->batch_stride : c->n;
    a.with_rot = c->with_rot ? 1 : 0; a.rpy_jac = c->rpy_jac ? 1 : 0; a.keep_irrelevant = c->keep_irrelevant ? 1 : 0;
    a.grad_mode = c->grad_mode; a.scratch_ref = c->scratch_mode == KIN_SCRATCH_REFERENCE;
    a.truncation_dist = c->truncation_dist; a.vals_offset = c->vals_offset;
    return a;
}

int launch_ahead_of_time(const LaunchPlan &p, const kin::KernelArgs &a, cudaStream_t stream) {
    p.kernel<<<(unsigned)p.grid, p.block, p.smem, stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    g_launches.fetch_add(1);
    return KIN_OK;
}

int launch(KinModel *m, const KinCall *c, DeviceProgram *dp, cudaStream_t stream) {
    const LaunchPlan p = plan_launch(m, c, dp, /*count_small_calls=*/true);
    if (p.grid < 1) return KIN_OK;
    if (p.jit) return launch_jit(m, c, dp, p, stream);
    return launch_ahead_of_time(p, kernel_args(c, dp), stream);
}

}  // namespace

extern "C" {

const char *kin_last_error(void) { return g_err.c_str(); }
int kin_abi_version(void) { return KIN_B200_ABI_VERSION; }
#ifndef KIN_BUILD_ID
#define KIN_BUILD_ID "unknown"
#endif
// the id sits behind a marker so that lib.py can read it from the file without loading the library
extern "C" __attribute__((visibility("default"), used)) const char kin_build_id_marker[] = "KIN_BUILD_ID=" KIN_BUILD_ID;
const char *kin_build_id(void) { return kin_build_id_marker + 13; }
int kin_debug_build(void) {
#ifdef KIN_DEBUG
    return 1;
#else
    return 0;
#endif
}
int64_t kin_launch_count(void) { return g_launches.load(); }

const char *kin_jit_status(void) {
    static thread_local std::string s;
    s = kin::jit_status();
    return s.c_str();
}

int kin_jit_stats(int64_t *compiles, int64_t *cache_hits, int64_t *launches, int64_t *failures) {
    if (compiles) *compiles = g_jit_compiles.load();
    if (cache_hits) *cache_hits = g_jit_cache_hits.load();
    if (launches) *launches = g_jit_launches.load();
    if (failures) *failures = g_jit_failures.load();
    return KIN_OK;
}

// Host-only: generate the specialised source a call would run (pointers of `call` are only tested for NULL) into
// out_dir, and with compile != 0 also compile it with NVRTC (kin_gen.cubin, kin_gen.log).  No device needed.
int kin_codegen_dump(const KinModelDesc *d, const KinCall *c, int32_t compile, const char *out_dir) {
    if (!d || !c || !out_dir) return fail(KIN_ERR_INVALID_ARGUMENT, "null argument");
    kin::HostModel hm;
    int rc = host_model_from_desc(d, hm);
    if (rc != KIN_OK) return rc;
    DeviceProgram dp;
    std::string err;
    if (!ProgramRequest(c).compile(hm, dp.prog, err)) return fail(KIN_ERR_INVALID_ARGUMENT, err);
    kin::GenOptions o = gen_options(nullptr, c, &dp);
    if (const char *ik = std::getenv("KIN_DUMP_IK")) {   // development aid: the batched-IK kernel of the call's links instead
        IkLinks lk;
        lk.n = dp.prog.h.n_fk;
        // several links (kin_ik_solve_links): the value is the rotation mask (bit l: link l has rotation rows)
        lk.rot_mask = lk.n > 1 ? (unsigned)std::strtoul(ik, nullptr, 0) : (c->with_rot ? 1u : 0u);
        o = ik_gen_options(lk);
    }
    kin::GenSource g;
    if (!kin::generate_source(dp.prog, o, g, err)) return fail(KIN_ERR_INVALID_ARGUMENT, "codegen: " + err);
    const std::string dir(out_dir);
    const kin::JitHeaders hs = jit_headers(g);
    auto put = [&](const std::string &name, const std::string &text) { std::ofstream f(dir + "/" + name, std::ios::binary); f << text; };
    put("kin_gen.cu", jit_main_source());
    for (const auto &hd : hs) put(hd.first, hd.second);
    if (compile) {
        std::vector<char> cubin;
        std::string log;
        bool cached = false;
        const bool ok = kin::jit_compile(jit_main_source(), hs, "sm_100a", cubin, log, &cached);
        put("kin_gen.log", log);
        if (!ok) return fail(KIN_ERR_CUDA, "NVRTC: " + log);
        std::ofstream f(dir + "/kin_gen.cubin", std::ios::binary);
        f.write(cubin.data(), (std::streamsize)cubin.size());
    }
    return KIN_OK;
}

int kin_model_create(const KinModelDesc *d, KinModel **out) {
    if (!d || !out) return fail(KIN_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    if (int rc = require_device()) return rc;
    KinModel *m = new KinModel();
    int rc = host_model_from_desc(d, m->hm);
    if (rc != KIN_OK) { delete m; return rc; }
    cudaError_t e = cudaGetDevice(&m->device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&m->n_sm, cudaDevAttrMultiProcessorCount, m->device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&m->dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, m->device);
    if (e == cudaSuccess) {
        // workspaces (kin_pose_residual, kin_sdf_points) come from a private pool whose release threshold is
        // "never": the default pool hands memory back at every synchronisation and re-mapping hundreds of MB
        // per call costs milliseconds
        cudaMemPoolProps props;
        std::memset(&props, 0, sizeof props);
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = m->device;
        e = cudaMemPoolCreate(&m->pool, &props);
        if (e == cudaSuccess) {
            unsigned long long keep = ~0ull;
            e = cudaMemPoolSetAttribute(m->pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    if (e != cudaSuccess) { delete m; return fail_cuda(e, "querying the device"); }
    *out = m;
    return KIN_OK;
}

// Host-only: compile the program a call would run and hand the tables back (no device needed).
// Used by the CPU test-suite to check the flattener against the oracle.
int kin_program_dump(const KinModelDesc *d, const int32_t *fk_links, int32_t n_fk, const int32_t *jac_links,
                     int32_t n_jac, int32_t want_coll, int32_t want_stale, int32_t *header_out, int32_t header_cap,
                     int32_t *ints_out, int32_t ints_cap, double *reals_out, int32_t reals_cap) {
    if (!d) return fail(KIN_ERR_INVALID_ARGUMENT, "null argument");
    kin::HostModel hm;
    int rc = host_model_from_desc(d, hm);
    if (rc != KIN_OK) return rc;
    kin::Program p;
    std::string err;
    if (!ProgramRequest(fk_links, n_fk, jac_links, n_jac, want_coll != 0, want_stale != 0).compile(hm, p, err))
        return fail(KIN_ERR_INVALID_ARGUMENT, err);
    const int hn = (int)(sizeof(kin::ProgHeader) / sizeof(int32_t));
    if (header_cap < hn || ints_cap < (int)p.ints.size() || reals_cap < (int)p.reals.size())
        return fail(KIN_ERR_LIMIT, "kin_program_dump: output buffers too small");
    std::memcpy(header_out, &p.h, sizeof(kin::ProgHeader));
    std::memcpy(ints_out, p.ints.data(), sizeof(int32_t) * p.ints.size());
    std::memcpy(reals_out, p.reals.data(), sizeof(double) * p.reals.size());
    return KIN_OK;
}

int kin_model_destroy(KinModel *m) {
    if (!m) return KIN_OK;
    DeviceGuard guard(m->device);
    clear_cache(m);
    for (int i = 0; i < HostStage::kStreams; ++i) {
        if (m->stage.stream[i]) cudaStreamDestroy(m->stage.stream[i]);
        if (m->stage.buf[i]) cudaFree(m->stage.buf[i]);
    }
    if (m->pool) cudaMemPoolDestroy(m->pool);
    delete m;
    return KIN_OK;
}

int kin_model_set_spheres(KinModel *m, int32_t n, const int32_t *link, const double *center, const double *radius) {
    if (!m) return fail(KIN_ERR_INVALID_ARGUMENT, "null model");
    DeviceGuard guard(m->device);
    std::lock_guard<std::mutex> lock(m->mu);
    int rc = load_spheres(m->hm, n, link, center, radius);
    if (rc == KIN_OK) { clear_cache(m); m->self_pairs.reset(); }     // the pair table's sphere ids would be stale
    return rc;
}

int kin_model_set_boxes(KinModel *m, int32_t n, const double *pose, const double *width) {
    return kin_model_set_primitives(m, n, nullptr, pose, width);
}

int kin_model_set_primitives(KinModel *m, int32_t n, const int32_t *kinds, const double *pose, const double *width) {
    return kin_model_set_scene(m, n, kinds, pose, width, nullptr);
}

int kin_model_set_scene(KinModel *m, int32_t n, const int32_t *kinds, const double *pose, const double *width,
                        const KinGrid *const *grids) {
    if (!m) return fail(KIN_ERR_INVALID_ARGUMENT, "null model");
    DeviceGuard guard(m->device);
    std::lock_guard<std::mutex> lock(m->mu);
    const int old_n = m->hm.n_box;
    int rc = load_prims(m->hm, n, kinds, pose, width, grids, m->device);
    if (rc != KIN_OK) return rc;
    m->grids.clear();                            // the model's own references: the caller may destroy its handles
    for (int b = 0; grids && b < n; ++b)
        if (grids[b]) m->grids.push_back(grids[b]->st);
    if (n != old_n) { clear_cache(m); return KIN_OK; }
    // Same number of boxes (the obstacle moved, sdf.jl:14-32): the compiled programs stay valid, only the box rows
    // of their real sections are rewritten in place -- no recompilation, no cudaMalloc / cudaFree.
    for (auto &kv : m->cache) {
        DeviceProgram *dp = kv.second.get();
        const kin::ProgHeader &h = dp->prog.h;
        if (h.n_box != n || n == 0) continue;
        double *rows = &dp->prog.reals[h.ro_box];
        kin::emit_box_rows(m->hm, rows);
        std::vector<float> r32(rows, rows + (size_t)n * kin::BOX_REALS);
        kin::fix_grid_rows_f32(rows, r32.data(), n);
        CUDA_TRY(cudaMemcpy(dp->d_r64 + h.ro_box, rows, sizeof(double) * r32.size(), cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(dp->d_r32 + h.ro_box, r32.data(), sizeof(float) * r32.size(), cudaMemcpyHostToDevice));
    }
    return KIN_OK;
}

int kin_grid_create(int32_t nx, int32_t ny, int32_t nz, double spacing, const float *values, KinGrid **out) {
    if (!out) return fail(KIN_ERR_INVALID_ARGUMENT, "null argument");
    *out = nullptr;
    if (!values) return fail(KIN_ERR_INVALID_ARGUMENT, "null grid values");
    if (nx < 2 || ny < 2 || nz < 2) return fail(KIN_ERR_INVALID_ARGUMENT, "a grid needs at least 2 samples per axis");
    if ((double)nx * ny * nz > (double)KIN_MAX_GRID_VALUES) return fail(KIN_ERR_LIMIT, "grid exceeds KIN_MAX_GRID_VALUES");
    if (!(spacing > 0.0) || std::isinf(spacing)) return fail(KIN_ERR_INVALID_ARGUMENT, "grid spacing must be positive and finite");
    if (int rc = require_device()) return rc;
    auto st = std::make_shared<GridStore>();
    CUDA_TRY(cudaGetDevice(&st->device));
    st->n[0] = nx; st->n[1] = ny; st->n[2] = nz;
    kin::GridHeader hd;
    std::memset(&hd, 0, sizeof hd);
    for (int k = 0; k < 3; ++k) hd.n[k] = st->n[k];
    hd.s = spacing; hd.inv_s = 1.0 / spacing;
    hd.s_f = (float)spacing; hd.inv_s_f = 1.0f / (float)spacing;
    const size_t bytes = sizeof(float) * st->values();
    CUDA_TRY(cudaMalloc(&st->d, kin::GRID_VALUES_OFFSET + bytes));
    CUDA_TRY(cudaMemcpyAsync(st->d, &hd, sizeof hd, cudaMemcpyHostToDevice, 0));
    CUDA_TRY(cudaMemcpyAsync((char *)st->d + kin::GRID_VALUES_OFFSET, values, bytes, cudaMemcpyDefault, 0));
    CUDA_TRY(cudaStreamSynchronize(0));
    *out = new KinGrid{st};
    return KIN_OK;
}

int kin_grid_set_values(KinGrid *grid, const float *values, void *stream) {
    if (!grid || !values) return fail(KIN_ERR_INVALID_ARGUMENT, "null argument");
    DeviceGuard guard(grid->st->device);
    CUDA_TRY(cudaMemcpyAsync((char *)grid->st->d + kin::GRID_VALUES_OFFSET, values, sizeof(float) * grid->st->values(),
                             cudaMemcpyDefault, (cudaStream_t)stream));
    return KIN_OK;
}

int kin_grid_destroy(KinGrid *grid) {
    delete grid;
    return KIN_OK;
}

int kin_model_set_self_pairs(KinModel *m, int32_t n_pairs, const int32_t *pairs) {
    if (!m) return fail(KIN_ERR_INVALID_ARGUMENT, "null model");
    if (n_pairs < 0) return fail(KIN_ERR_INVALID_ARGUMENT, "negative n_pairs");
    if (n_pairs > KIN_MAX_SELF_PAIRS) return fail(KIN_ERR_LIMIT, "n_pairs exceeds KIN_MAX_SELF_PAIRS");
    if (n_pairs > 0 && !pairs) return fail(KIN_ERR_INVALID_ARGUMENT, "null pair table");
    DeviceGuard guard(m->device);
    std::lock_guard<std::mutex> lock(m->mu);
    const int S = m->hm.n_sph;
    std::vector<int2> host(n_pairs);
    for (int p = 0; p < n_pairs; ++p) {      // validate before touching the model: a failed call leaves it unchanged
        const int i = pairs[2 * p], j = pairs[2 * p + 1];
        if (i < 1 || i > S || j < 1 || j > S) return fail(KIN_ERR_INVALID_ARGUMENT, "self-collision pair: sphere id out of range");
        if (i == j) return fail(KIN_ERR_INVALID_ARGUMENT, "self-collision pair: a sphere paired with itself");
        host[p] = make_int2(i - 1, j - 1);
    }
    if (n_pairs == 0) { m->self_pairs.reset(); return KIN_OK; }
    auto dp = std::make_shared<DevicePairs>();
    CUDA_TRY(cudaMalloc(&dp->d, sizeof(int2) * host.size()));
    CUDA_TRY(cudaMemcpy(dp->d, host.data(), sizeof(int2) * host.size(), cudaMemcpyHostToDevice));
    dp->n = n_pairs;
    m->self_pairs = dp;
    return KIN_OK;
}

int kin_model_n_self_pairs(const KinModel *m) { return m && m->self_pairs ? m->self_pairs->n : 0; }

int kin_model_n_dof(const KinModel *m) { return m ? m->hm.n_dof() : 0; }
int kin_model_n_spheres(const KinModel *m) { return m ? m->hm.n_sph : 0; }
int kin_model_n_boxes(const KinModel *m) { return m ? m->hm.n_box : 0; }

int kin_eval(KinModel *m, const KinCall *c) {
    int rc = validate_call(m, c);
    if (rc != KIN_OK) return rc;
    if (c->n == 0) return KIN_OK;
    if (!c->T_out && !c->J_out && !c->vals_out) return KIN_OK;
    DeviceGuard guard(m->device);
    std::shared_ptr<DeviceProgram> dp;
    rc = get_program(m, c, eval_kind(c), dp);
    if (rc != KIN_OK) return rc;
    return launch(m, c, dp.get(), (cudaStream_t)c->stream);
}

int kin_query_launch(KinModel *m, const KinCall *c, int32_t *regs, int32_t *smem_bytes, int32_t *block, int32_t *grid) {
    int rc = validate_call(m, c);
    if (rc != KIN_OK) return rc;
    DeviceGuard guard(m->device);
    std::shared_ptr<DeviceProgram> dp;
    rc = get_program(m, c, eval_kind(c), dp);
    if (rc != KIN_OK) return rc;
    const LaunchPlan p = plan_launch(m, c, dp.get(), /*count_small_calls=*/false);
    if (regs) *regs = p.regs;
    if (smem_bytes) *smem_bytes = (int32_t)p.smem;
    if (block) *block = p.jit ? -p.block : p.block;      // negative block size: the model-specialised (NVRTC) kernel
    if (grid) *grid = (int32_t)p.grid;
    return KIN_OK;
}

// Host-buffer variant: chunks of the batch are staged through kStreams device buffers; within a
// stream the order is H2D(q) -> kernel -> D2H(outputs), and the streams overlap each other.
}  // extern "C"
namespace {

// ---- constant output rows of a host-staged SoA call: filled by host threads instead of crossing PCIe ----
void fill_row(void *dst, size_t n, double v, bool f32) {
    if (f32) {
        float *p = (float *)dst;
        const float x = (float)v;
        size_t i = 0;
#if defined(__SSE2__)
        for (; i < n && ((uintptr_t)(p + i) & 15); ++i) p[i] = x;
        const __m128 xv = _mm_set1_ps(x);
        for (; i + 4 <= n; i += 4) _mm_stream_ps(p + i, xv);      // non-temporal: no read-for-ownership of the output
        _mm_sfence();
#endif
        for (; i < n; ++i) p[i] = x;
    } else {
        double *p = (double *)dst;
        size_t i = 0;
#if defined(__SSE2__)
        for (; i < n && ((uintptr_t)(p + i) & 15); ++i) p[i] = v;
        const __m128d xv = _mm_set1_pd(v);
        for (; i + 2 <= n; i += 2) _mm_stream_pd(p + i, xv);
        _mm_sfence();
#endif
        for (; i < n; ++i) p[i] = v;
    }
}

struct RowPlan {                         // of one output array with `comps` component rows
    std::vector<std::pair<int, int>> runs;                 // [begin, end) runs of rows that depend on the configuration
    std::vector<std::pair<int, double>> consts;            // (row, value) of the others
    void build(size_t comps, const std::vector<std::pair<int, double>> &cs, const std::vector<int> &dup_rows = {}) {
        std::vector<char> is_const(comps, 0);
        for (const auto &kv : cs)
            if (kv.first >= 0 && (size_t)kv.first < comps && !is_const[kv.first]) { is_const[kv.first] = 1; consts.push_back(kv); }
        for (int r : dup_rows)             // rows the host copies from another row that did cross PCIe
            if (r >= 0 && (size_t)r < comps) is_const[r] = 1;
        for (size_t r = 0; r < comps;) {
            if (is_const[r]) { ++r; continue; }
            size_t e = r;
            while (e < comps && !is_const[e]) ++e;
            runs.emplace_back((int)r, (int)e);
            r = e;
        }
    }
};

// dst[i] = +-src[i] with non-temporal stores (the duplicate rows of a host-staged call)
void copy_row(void *dst, const void *src, size_t n, bool negate, bool f32) {
    if (f32) {
        float *d = (float *)dst;
        const float *p = (const float *)src;
        for (size_t i = 0; i < n; ++i) d[i] = negate ? -p[i] : p[i];
        return;
    }
    double *d = (double *)dst;
    const double *p = (const double *)src;
    size_t i = 0;
#if defined(__SSE2__)
    for (; i < n && ((uintptr_t)(d + i) & 15); ++i) d[i] = negate ? -p[i] : p[i];
    const __m128d sign = _mm_set1_pd(negate ? -0.0 : 0.0);
    for (; i + 2 <= n; i += 2) _mm_stream_pd(d + i, _mm_xor_pd(_mm_loadu_pd(p + i), sign));
    _mm_sfence();
#endif
    for (; i < n; ++i) d[i] = negate ? -p[i] : p[i];
}

struct DupRow { unsigned char *dst; const unsigned char *src; bool negate; };

// Progress of the chunk loop, for the threads that complete the duplicate rows behind it: chunk i may be read once
// `issued` > i (its event has been recorded) and the event has completed.
struct ChunkFeed {
    std::mutex mu;
    std::condition_variable cv;
    long long issued = 0;
    bool done = false;                   // no further chunk will be issued (normal end or error exit)
    std::vector<cudaEvent_t> ev;
    std::vector<std::pair<long long, long long>> span;     // (n0, count) of chunk i
    void publish(long long n0, long long cnt) {
        { std::lock_guard<std::mutex> l(mu); span.emplace_back(n0, cnt); ++issued; }
        cv.notify_all();
    }
    void finish() {
        { std::lock_guard<std::mutex> l(mu); done = true; }
        cv.notify_all();
    }
    ~ChunkFeed() { for (auto e : ev) cudaEventDestroy(e); }
};

struct FillJobs {                        // joins its threads on every exit path
    std::vector<std::thread> threads;
    ~FillJobs() { for (auto &t : threads) if (t.joinable()) t.join(); }
};

}  // namespace
extern "C" {

int kin_host_transfer_bytes(int64_t *h2d, int64_t *d2h, int64_t *host_filled) {
    if (h2d) *h2d = g_h2d_bytes.load();
    if (d2h) *d2h = g_d2h_bytes.load();
    if (host_filled) *host_filled = g_host_fill_bytes.load();
    return KIN_OK;
}

int kin_eval_host(KinModel *m, const KinCall *c) {
    int rc = validate_call(m, c);
    if (rc != KIN_OK) return rc;
    if (c->n == 0) return KIN_OK;
    if (!c->T_out && !c->J_out && !c->vals_out) return KIN_OK;
    DeviceGuard guard(m->device);
    std::shared_ptr<DeviceProgram> dp_;
    rc = get_program(m, c, eval_kind(c), dp_);
    if (rc != KIN_OK) return rc;
    DeviceProgram *dp = dp_.get();
    const size_t es = c->precision == KIN_F32 ? 4 : 8;
    const int ND = m->hm.n_dof(), S = m->hm.n_sph;
    const int rows = c->with_rot ? 6 : 3;
    // per-configuration element counts of each array
    const size_t cq = ND, cT = c->T_out ? 12 * (size_t)c->n_fk_links : 0,
                 cJ = c->J_out ? (size_t)rows * ND * c->n_jac_links : 0, cV = c->vals_out ? S : 0,
                 cG = c->grads_out ? (size_t)ND * S : 0, cA = c->argmin_out ? S : 0;
    const size_t per_cfg = es * (cq + cT + cJ + cV + cG) + 4 * cA;
    long long chunk = env_ll("KIN_HOST_CHUNK", 1 << 17);       // measured (profiles/sweep_e2e_host.sh): 2^15 .. 2^18 within 3 %
    if (chunk < 32) chunk = 32;
    if (chunk > c->n) chunk = c->n;
    // tiled storage holds whole tiles of 32 configurations: size the staging carves for the padded chunk (the
    // kernel addresses, and the copies move, roundup(count, 32) records; host buffers are padded likewise)
    if (c->layout == KIN_LAYOUT_TILED32) chunk = (chunk + 31) / 32 * 32;
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t need = align(es * cq * chunk) + align(es * cT * chunk) + align(es * cJ * chunk) +
                        align(es * cV * chunk) + align(es * cG * chunk) + align(4 * cA * chunk);
    (void)per_cfg;
    std::lock_guard<std::mutex> lock(m->stage_mu);   // one host-staged call at a time per model (m->mu stays free)
    HostStage &st = m->stage;
    if (st.bytes < need) {
        for (int i = 0; i < HostStage::kStreams; ++i) {
            if (st.buf[i]) { cudaFree(st.buf[i]); st.buf[i] = nullptr; }
            CUDA_TRY(cudaMalloc(&st.buf[i], need));
        }
        st.bytes = need;
    }
    for (int i = 0; i < HostStage::kStreams; ++i)
        if (!st.stream[i]) CUDA_TRY(cudaStreamCreateWithFlags(&st.stream[i], cudaStreamNonBlocking));

    const long long N = c->n, ldh = c->batch_stride ? c->batch_stride : N;
    const bool aos = c->layout != KIN_LAYOUT_SOA;          // AoS and tiled: one contiguous block per chunk
    const bool tiled = c->layout == KIN_LAYOUT_TILED32;
    // SoA: the rows of T / J that do not depend on the configuration (for Fetch with the 8 arm joints: 175 of the 348:
    // links no control joint moves, zero / unit rotation entries, Jacobian columns of joints that do not move the
    // link -- the code generator knows them, kin_codegen.hpp) are NOT copied back over PCIe, which is what bounds this
    // call: host threads fill them while the device works on the rest.  Same values as the kernels write (up to the
    // sign of a zero).  get_jacobian! semantics (rows the kernel leaves untouched) and KIN_HOST_NO_CONST_FILL opt out.
    RowPlan planT, planJ;
    auto dups = std::make_shared<std::vector<DupRow>>();
    bool elide = !aos && (cT || cJ) && !(c->J_out && c->keep_irrelevant) && !std::getenv("KIN_HOST_NO_CONST_FILL");
    if (elide) {
        kin::GenSource g;
        std::string err;
        elide = kin::generate_source(dp->prog, gen_options(m, c, dp), g, err);
        if (elide) {
            // outputs that hold the same variable of the generated code (possibly negated): the first one crosses
            // PCIe, the host copies the others from it (KIN_HOST_NO_DUP_COPY opts out)
            std::vector<int> dupT, dupJ;
            if (!std::getenv("KIN_HOST_NO_DUP_COPY")) {
                std::map<std::string, const unsigned char *> first;
                auto scan = [&](const std::vector<std::pair<int, std::string>> &ex, void *base_, size_t comps, std::vector<int> &dup) {
                    for (const auto &kv : ex) {
                        if (kv.first < 0 || (size_t)kv.first >= comps) continue;
                        const bool neg = kv.second.size() > 3 && kv.second[0] == '(' && kv.second[1] == '-';
                        const std::string canon = neg ? kv.second.substr(2, kv.second.size() - 3) : kv.second;
                        unsigned char *row = (unsigned char *)base_ + es * (size_t)kv.first * ldh;
                        auto it = first.find(canon);
                        // the primary must hold +x: a negated first occurrence stays an ordinary row
                        if (it == first.end()) { if (!neg) first.emplace(canon, row); continue; }
                        dups->push_back({row, it->second, neg});
                        dup.push_back(kv.first);
                    }
                };
                if (cT) scan(g.expr_T, c->T_out, cT, dupT);
                if (cJ) scan(g.expr_J, c->J_out, cJ, dupJ);
            }
            planT.build(cT, g.const_T, dupT);
            planJ.build(cJ, g.const_J, dupJ);
        }
        if (planT.consts.empty() && planJ.consts.empty() && dups->empty()) elide = false;
    }
    ChunkFeed feed;
    FillJobs fill;
    if (elide) {
        struct Job { unsigned char *row; double v; };
        auto jobs = std::make_shared<std::vector<Job>>();
        for (const auto &kv : planT.consts) jobs->push_back({(unsigned char *)c->T_out + es * (size_t)kv.first * ldh, kv.second});
        for (const auto &kv : planJ.consts) jobs->push_back({(unsigned char *)c->J_out + es * (size_t)kv.first * ldh, kv.second});
        // host threads of this process's share of the machine (one process per GPU under torchrun: LOCAL_WORLD_SIZE)
        const unsigned hw = std::max<unsigned>(2u, std::thread::hardware_concurrency() / (unsigned)std::max<long long>(1, env_ll("LOCAL_WORLD_SIZE", 1)));
        // 2 .. 4 threads keep up with the PCIe stream; more only compete with the DMA writes for host memory bandwidth
        long long nt = env_ll("KIN_HOST_FILL_THREADS", std::min<long long>(4, std::max<long long>(1, hw / 2)));
        nt = std::max<long long>(1, std::min<long long>(nt, (long long)jobs->size()));
        const bool f32 = c->precision == KIN_F32;
        const size_t n_fill = (size_t)N;
        for (long long t = 0; t < nt; ++t)
            fill.threads.emplace_back([jobs, t, nt, n_fill, f32] {
                for (size_t j = (size_t)t; j < jobs->size(); j += (size_t)nt) fill_row((*jobs)[j].row, n_fill, (*jobs)[j].v, f32);
            });
        g_host_fill_bytes.fetch_add((long long)(es * (jobs->size() + dups->size()) * (size_t)N));
        if (!dups->empty()) {
            // the duplicate rows of chunk i are copied once its device -> host copies have landed
            long long nd = env_ll("KIN_HOST_DUP_THREADS", std::min<long long>(6, std::max<long long>(1, hw / 2)));
            nd = std::max<long long>(1, std::min<long long>(nd, (long long)dups->size()));
            ChunkFeed *fd = &feed;
            for (long long t = 0; t < nd; ++t)
                fill.threads.emplace_back([dups, fd, t, nd, f32, es] {
                    for (long long i = 0;; ++i) {
                        cudaEvent_t ev;
                        std::pair<long long, long long> sp;
                        {
                            std::unique_lock<std::mutex> l(fd->mu);
                            fd->cv.wait(l, [&] { return fd->issued > i || fd->done; });
                            if (fd->issued <= i) return;
                            ev = fd->ev[(size_t)i]; sp = fd->span[(size_t)i];
                        }
                        if (cudaEventSynchronize(ev) != cudaSuccess) return;
                        for (size_t j = (size_t)t; j < dups->size(); j += (size_t)nd) {
                            const DupRow &d = (*dups)[j];
                            copy_row(d.dst + es * (size_t)sp.first, d.src + es * (size_t)sp.first, (size_t)sp.second, d.negate, f32);
                        }
                    }
                });
        }
    }
    struct FeedCloser { ChunkFeed &f; ~FeedCloser() { f.finish(); } } feed_closer{feed};     // declared after `fill`: runs first
    int k = 0;
    for (long long n0 = 0; n0 < N; n0 += chunk, k = (k + 1) % HostStage::kStreams) {
        const long long mcount = (N - n0 < chunk) ? N - n0 : chunk;
        cudaStream_t s = st.stream[k];
        unsigned char *base = (unsigned char *)st.buf[k];
        size_t off = 0;
        auto carve = [&](size_t bytes) { void *p = base + off; off += align(bytes); return p; };
        void *dq = carve(es * cq * chunk), *dT = carve(es * cT * chunk), *dJ = carve(es * cJ * chunk),
             *dV = carve(es * cV * chunk), *dG = carve(es * cG * chunk), *dA = carve(4 * cA * chunk);
        // host <-> device copy of one array with `comps` components per configuration
        auto copy = [&](void *dev, const void *host_c, void *host_m, size_t comps, size_t esz, bool to_dev) -> cudaError_t {
            if (comps == 0) return cudaSuccess;
            if (aos) {
                const size_t cnt = tiled ? (size_t)((mcount + 31) / 32 * 32) : (size_t)mcount;   // chunk starts are multiples of 32
                const size_t bytes = esz * comps * cnt, hoff = esz * comps * n0;
                return to_dev ? cudaMemcpyAsync(dev, (const unsigned char *)host_c + hoff, bytes, cudaMemcpyHostToDevice, s)
                              : cudaMemcpyAsync((unsigned char *)host_m + hoff, dev, bytes, cudaMemcpyDeviceToHost, s);
            }
            const size_t hoff = esz * n0, width = esz * mcount;
            return to_dev ? cudaMemcpy2DAsync(dev, esz * mcount, (const unsigned char *)host_c + hoff, esz * ldh, width, comps, cudaMemcpyHostToDevice, s)
                          : cudaMemcpy2DAsync((unsigned char *)host_m + hoff, esz * ldh, dev, esz * mcount, width, comps, cudaMemcpyDeviceToHost, s);
        };
        // device -> host copy of the configuration-dependent rows only (SoA, see above)
        auto copy_runs = [&](void *dev, void *host_m, const RowPlan &plan) -> cudaError_t {
            for (const auto &run : plan.runs) {
                const size_t r0 = (size_t)run.first, nr = (size_t)(run.second - run.first);
                cudaError_t e = cudaMemcpy2DAsync((unsigned char *)host_m + es * (r0 * ldh + n0), es * ldh,
                                                  (unsigned char *)dev + es * r0 * mcount, es * mcount, es * mcount, nr,
                                                  cudaMemcpyDeviceToHost, s);
                if (e != cudaSuccess) return e;
                g_d2h_bytes.fetch_add((long long)(es * mcount * nr));
            }
            return cudaSuccess;
        };
        CUDA_TRY(copy(dq, c->q, nullptr, cq, es, true));
        g_h2d_bytes.fetch_add((long long)(es * cq * mcount));
        KinCall cc = *c;
        cc.n = mcount; cc.batch_stride = 0; cc.q = dq;
        cc.T_out = cT ? dT : nullptr; cc.J_out = cJ ? dJ : nullptr; cc.vals_out = cV ? dV : nullptr;
        cc.grads_out = cG ? dG : nullptr; cc.argmin_out = cA ? (int32_t *)dA : nullptr;
        rc = launch(m, &cc, dp, s);
        if (rc != KIN_OK) return rc;
        if (elide) {
            if (cT) CUDA_TRY(copy_runs(dT, c->T_out, planT));
            if (cJ) CUDA_TRY(copy_runs(dJ, c->J_out, planJ));
        } else {
            CUDA_TRY(copy(dT, nullptr, c->T_out, cT, es, false));
            CUDA_TRY(copy(dJ, nullptr, c->J_out, cJ, es, false));
            g_d2h_bytes.fetch_add((long long)(es * (cT + cJ) * mcount));
        }
        g_d2h_bytes.fetch_add((long long)((es * (cV + cG) + 4 * cA) * mcount));
        CUDA_TRY(copy(dV, nullptr, c->vals_out, cV, es, false));
        CUDA_TRY(copy(dG, nullptr, c->grads_out, cG, es, false));
        CUDA_TRY(copy(dA, nullptr, c->argmin_out, cA, 4, false));
        if (!dups->empty()) {
            cudaEvent_t ev;
            CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming | cudaEventBlockingSync));
            { std::lock_guard<std::mutex> l(feed.mu); feed.ev.push_back(ev); }
            CUDA_TRY(cudaEventRecord(ev, s));
            feed.publish(n0, mcount);
        }
    }
    feed.finish();
    for (int i = 0; i < HostStage::kStreams; ++i) CUDA_TRY(cudaStreamSynchronize(st.stream[i]));
    for (auto &t : fill.threads) t.join();
    return KIN_OK;
}

int kin_sdf_points(int32_t n_boxes, const double *box_pose, const double *box_width, int32_t precision, int32_t layout,
                   const void *pts, int64_t n, int32_t grad_mode, void *vals_out, void *grads_out, int32_t *argmin_out,
                   void *stream_) {
    return kin_sdf_points_prims(n_boxes, nullptr, box_pose, box_width, precision, layout, pts, n, grad_mode, vals_out, grads_out,
                                argmin_out, stream_);
}

int kin_sdf_points_prims(int32_t n_boxes, const int32_t *kinds, const double *box_pose, const double *box_width, int32_t precision,
                         int32_t layout, const void *pts, int64_t n, int32_t grad_mode, void *vals_out, void *grads_out,
                         int32_t *argmin_out, void *stream_) {
    return kin_sdf_points_scene(n_boxes, kinds, box_pose, box_width, nullptr, precision, layout, pts, n, grad_mode, vals_out,
                                grads_out, argmin_out, stream_);
}

int kin_sdf_points_scene(int32_t n_boxes, const int32_t *kinds, const double *box_pose, const double *box_width,
                         const KinGrid *const *grids, int32_t precision, int32_t layout, const void *pts, int64_t n,
                         int32_t grad_mode, void *vals_out, void *grads_out, int32_t *argmin_out, void *stream_) {
    if (n < 0 || (n > 0 && (!pts || !vals_out))) return fail(KIN_ERR_INVALID_ARGUMENT, "null points or vals_out");
    if (n_boxes <= 0) return fail(KIN_ERR_INVALID_ARGUMENT, "kin_sdf_points needs at least one box");
    int rc = check_batch(precision, layout, n, pts, kSoaAos);
    if (rc != KIN_OK) return rc;
    if (grad_mode != KIN_GRAD_FD && grad_mode != KIN_GRAD_ANALYTIC && grad_mode != KIN_GRAD_FD_DIRECT) return fail(KIN_ERR_INVALID_ARGUMENT, "unknown grad_mode");
    if ((rc = require_device()) != KIN_OK) return rc;
    int cur = 0;
    CUDA_TRY(cudaGetDevice(&cur));
    kin::HostModel hm;
    rc = load_prims(hm, n_boxes, kinds, box_pose, box_width, grids, cur);
    if (rc != KIN_OK) return rc;
    if (n == 0) return KIN_OK;
    std::vector<double> t64((size_t)n_boxes * kin::BOX_REALS, 0.0);
    kin::emit_box_rows(hm, t64.data());
    std::vector<float> t32(t64.begin(), t64.end());
    kin::fix_grid_rows_f32(t64.data(), t32.data(), n_boxes);
    const size_t es = precision == KIN_F32 ? 4 : 8, bytes = es * t64.size();
    cudaStream_t stream = (cudaStream_t)stream_;
    void *d_tab = nullptr;
    CUDA_TRY(cudaMallocAsync(&d_tab, bytes, stream));
    // pageable source: the copy is staged before the call returns, so the vectors may go out of scope
    CUDA_TRY(cudaMemcpyAsync(d_tab, precision == KIN_F32 ? (const void *)t32.data() : (const void *)t64.data(), bytes,
                             cudaMemcpyHostToDevice, stream));
    const int block = 256;
    long long grid = (n + block - 1) / block;
    {
        int dev = 0, n_sm = 0;
        CUDA_TRY(cudaGetDevice(&dev));
        CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
        if (grid > (long long)n_sm * 8) grid = (long long)n_sm * 8;
    }
    const bool aos = layout == KIN_LAYOUT_AOS;
    if (precision == KIN_F64) {
        if (aos) kin::sdf_points_kernel<double, true><<<(unsigned)grid, block, bytes, stream>>>((const double *)d_tab, n_boxes, (const double *)pts, n, grad_mode, (double *)vals_out, (double *)grads_out, argmin_out);
        else kin::sdf_points_kernel<double, false><<<(unsigned)grid, block, bytes, stream>>>((const double *)d_tab, n_boxes, (const double *)pts, n, grad_mode, (double *)vals_out, (double *)grads_out, argmin_out);
    } else {
        if (aos) kin::sdf_points_kernel<float, true><<<(unsigned)grid, block, bytes, stream>>>((const float *)d_tab, n_boxes, (const float *)pts, n, grad_mode, (float *)vals_out, (float *)grads_out, argmin_out);
        else kin::sdf_points_kernel<float, false><<<(unsigned)grid, block, bytes, stream>>>((const float *)d_tab, n_boxes, (const float *)pts, n, grad_mode, (float *)vals_out, (float *)grads_out, argmin_out);
    }
    CUDA_TRY(cudaGetLastError());
    g_launches.fetch_add(1);
    CUDA_TRY(cudaFreeAsync(d_tab, stream));
    return KIN_OK;
}

int kin_pose_residual_multi(KinModel *m, int32_t precision, int32_t layout, const void *q, int64_t n, int32_t n_links,
                            const int32_t *link_ids, const int32_t *with_rots, const void *target, int32_t target_per_config,
                            int32_t mode, void *val_out, void *jac_out, void *stream_) {
    if (!m) return fail(KIN_ERR_INVALID_ARGUMENT, "null model");
    if (int rc = check_batch(precision, layout, n, q, kSoaAos)) return rc;
    if (n > 0 && (!target || !val_out || !jac_out)) return fail(KIN_ERR_INVALID_ARGUMENT, "null argument");
    if (n_links < 1 || n_links > 32 || !link_ids || !with_rots) return fail(KIN_ERR_INVALID_ARGUMENT, "kin_pose_residual: 1..32 links");
    if (mode != KIN_POSE_IK_OBJECTIVE && mode != KIN_POSE_CONSTRAINT) return fail(KIN_ERR_INVALID_ARGUMENT, "unknown pose mode");
    if (n == 0) return KIN_OK;
    DeviceGuard guard(m->device);
    cudaStream_t stream = (cudaStream_t)stream_;
    const size_t es = precision == KIN_F32 ? 4 : 8;
    unsigned rot_mask = 0;
    for (int l = 0; l < n_links; ++l) rot_mask |= (with_rots[l] ? 1u : 0u) << l;
    const int nd = m->hm.n_dof(), rows = rot_mask ? 6 : 3;
    void *ws = nullptr;
    const size_t tb = es * 12 * (size_t)n_links * (size_t)n, jb = es * (size_t)rows * nd * (size_t)n_links * (size_t)n;
    CUDA_TRY(cudaMallocFromPoolAsync(&ws, tb + jb, m->pool, stream));
    KinCall c;
    std::memset(&c, 0, sizeof c);
    c.precision = precision; c.layout = layout; c.n = n; c.q = q;
    c.n_fk_links = n_links; c.fk_links = link_ids; c.T_out = ws;
    c.n_jac_links = n_links; c.jac_links = link_ids; c.with_rot = rot_mask ? 1 : 0; c.rpy_jac = 1; c.J_out = (unsigned char *)ws + tb;
    c.truncation_dist = INFINITY; c.stream = stream_;
    int rc = kin_eval(m, &c);
    if (rc != KIN_OK) { cudaFreeAsync(ws, stream); return rc; }
    const int block = 256;
    long long grid = (n + block - 1) / block;
    if (grid > (long long)m->n_sm * 16) grid = (long long)m->n_sm * 16;
    const bool aos = layout == KIN_LAYOUT_AOS;
    if (precision == KIN_F64) {
        auto T = (const double *)ws, J = (const double *)((unsigned char *)ws + tb);
        if (aos) kin::pose_residual_kernel<double, true><<<(unsigned)grid, block, 0, stream>>>(T, J, (const double *)target, target_per_config, n, nd, n_links, rot_mask, mode, (double *)val_out, (double *)jac_out);
        else kin::pose_residual_kernel<double, false><<<(unsigned)grid, block, 0, stream>>>(T, J, (const double *)target, target_per_config, n, nd, n_links, rot_mask, mode, (double *)val_out, (double *)jac_out);
    } else {
        auto T = (const float *)ws, J = (const float *)((unsigned char *)ws + tb);
        if (aos) kin::pose_residual_kernel<float, true><<<(unsigned)grid, block, 0, stream>>>(T, J, (const float *)target, target_per_config, n, nd, n_links, rot_mask, mode, (float *)val_out, (float *)jac_out);
        else kin::pose_residual_kernel<float, false><<<(unsigned)grid, block, 0, stream>>>(T, J, (const float *)target, target_per_config, n, nd, n_links, rot_mask, mode, (float *)val_out, (float *)jac_out);
    }
    {
        cudaError_t le = cudaGetLastError();
        if (le != cudaSuccess) { cudaFreeAsync(ws, stream); return fail_cuda(le, "launching pose_residual_kernel"); }
    }
    g_launches.fetch_add(1);
    CUDA_TRY(cudaFreeAsync(ws, stream));
    return KIN_OK;
}

int kin_pose_residual(KinModel *m, int32_t precision, int32_t layout, const void *q, int64_t n, int32_t link_id,
                      const void *target, int32_t target_per_config, int32_t with_rot, int32_t mode, void *val_out,
                      void *jac_out, void *stream_) {
    return kin_pose_residual_multi(m, precision, layout, q, n, 1, &link_id, &with_rot, target, target_per_config, mode,
                                   val_out, jac_out, stream_);
}

}  // extern "C"
namespace {

// One launch of the self-collision kernel (kin_eval_kernel<..., SELF = true>) over `pairs`: n configurations, SoA rows
// of stride ld (the other layouts ignore it).  kin_self_collision calls it with ld = n; kin_ik_solve_self with the
// stride of its workspace over the active list.
int self_collision_launch(KinModel *m, const DevicePairs &pairs, int32_t precision, int32_t layout, const void *q, long long n,
                          long long ld, double truncation_dist, double vals_offset, void *vals_out, void *grads_out,
                          void *dmin_out, int32_t *amin_out, cudaStream_t stream) {
    // phase 1 of a collision call computes the sphere centres and joint frames: the self-collision kernels run the
    // program of a plain collision call (no links requested, clean scratch); only the pointer's presence matters.
    // Always the ahead-of-time kernel, and never counted in small_calls: kin_collision calls in KIN_SCRATCH_CLEAN share
    // that program, and when they get specialised must not depend on self-collision calls.
    KinCall c;
    std::memset(&c, 0, sizeof c);
    c.precision = precision; c.layout = layout; c.n = n; c.batch_stride = ld; c.q = q;
    c.vals_out = vals_out ? vals_out : dmin_out; c.grads_out = grads_out; c.scratch_mode = KIN_SCRATCH_CLEAN;
    c.truncation_dist = truncation_dist; c.vals_offset = vals_offset;
    std::shared_ptr<DeviceProgram> dp;
    int rc = get_program(m, &c, KIND_SELF, dp);
    if (rc != KIN_OK) return rc;
    kin::KernelArgs a = kernel_args(&c, dp.get());
    a.vals_out = vals_out;                  // (c.vals_out holds dmin_out when only the summary is asked for)
    a.self_pairs = pairs.d; a.n_self_pairs = pairs.n;
    a.dmin_out = dmin_out; a.amin_out = amin_out;
    return launch_ahead_of_time(plan_ahead_of_time(m, &c, dp.get(), KIND_SELF), a, stream);
}

// The pair block of kin_ik_solve_self: the table (kept alive for the whole solve) and the margin.
struct IkSelfBlock {
    std::shared_ptr<DevicePairs> pairs;
    double margin = 0.0;
    void *dmin_out = nullptr;
};

template <int ND, bool SELF, bool LINKS>
void launch_ik_coll_step(const kin::IkcArgsT<SELF, LINKS> &a, bool rot, cudaStream_t stream, int dev_smem) {
    int block = 128;
    size_t smem = 0;
    auto kern = rot ? kin::ik_coll_step_kernel<ND, true, SELF, LINKS> : kin::ik_coll_step_kernel<ND, false, SELF, LINKS>;
    if (ND == 0) {
        // run-time-sized instance (13 .. IKC_MAX_DOF columns): the normal equations of a problem live in shared memory,
        // [slot][thread]; the largest CTA whose slots fit (18 columns: 1800 B per thread, 128 threads = 225 KB; 20 columns: 96 threads)
        const size_t per = kin::ikc_dyn_smem_per_thread(a.nd);
        while (block > 32 && per * (size_t)block > (size_t)dev_smem) block -= 32;
        smem = per * (size_t)block;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    }
    const unsigned grid = (unsigned)((a.n_act + block - 1) / block);
    kern<<<grid, block, smem, stream>>>(a);
}

template <bool SELF, bool LINKS>
void launch_ik_coll_step_any(const kin::IkcArgsT<SELF, LINKS> &a, int nd, int rows, cudaStream_t stream, int dev_smem) {
    switch (nd) {
#define KIN_IKC_CASE(N_) case N_: launch_ik_coll_step<N_, SELF, LINKS>(a, rows == 6, stream, dev_smem); break;
        KIN_IKC_CASE(1) KIN_IKC_CASE(2) KIN_IKC_CASE(3) KIN_IKC_CASE(4) KIN_IKC_CASE(5) KIN_IKC_CASE(6)
        KIN_IKC_CASE(7) KIN_IKC_CASE(8) KIN_IKC_CASE(9) KIN_IKC_CASE(10) KIN_IKC_CASE(11) KIN_IKC_CASE(12)
#undef KIN_IKC_CASE
        default: launch_ik_coll_step<0, SELF, LINKS>(a, rows == 6, stream, dev_smem); break;       // 13 .. IKC_MAX_DOF columns: run-time-sized instance
    }
}

// The collision-constrained solve of kin_ik_solve (csrc/kin_ik_coll.cuh): a loop of (kin_eval, step kernel) pairs on the
// caller's stream over a stream-ordered workspace.  At iterations 1, 2, 3, 4, 6, 8, 12, 16, 24, ... the still-running
// problems are compacted into an active list and its length (8 bytes) is read back -- the only host synchronisations --
// so that the following pairs cover only those problems (KIN_IK_NO_COMPACT=1: every pair covers the whole batch and
// nothing is read back).
// With c->collision == 0 (the pose-only problem when the run-time compiler is unavailable) no sphere is evaluated.
// With sb (kin_ik_solve_self) every iteration also evaluates the self-collision pairs at the trial points (one
// kin_self_collision launch over the same active list, between kin_eval and the step) and the step kernels run their
// SELF instances; pair values and gradients are indexed by list position like V and G, the pair multipliers by problem
// like mult, so the compaction carries nothing new.
// With several links (kin_ik_solve_links) kin_eval returns every link's transform and Euler-rate Jacobian, T and J
// grow by (n_links - 1)(12 + rows n_dof) doubles per problem, and the step kernels run their LINKS instances.
int ik_solve_coll(KinModel *m, const KinIkCall *c, const IkLinks &lk, const IkSelfBlock *sb = nullptr) {
    const int nd = m->hm.n_dof(), S = c->collision ? m->hm.n_sph : 0, rows = lk.rows(), NL = lk.n;
    const int P = sb ? sb->pairs->n : 0;
    DeviceGuard guard(m->device);
    cudaStream_t stream = (cudaStream_t)c->stream;
    const long long n = c->n, ld = (n + 31) / 32 * 32;
    // workspace (doubles per problem): q_try, T, J, V, G | q, H, g, phi, fpose, damp, viol, mult | Vfin | q_try_b
    // | VP, GP, multP (pairs only) ; then int32 status, its, two lists
    const long long nh = (long long)nd * (nd + 1) / 2;
    const long long per = nd + 12LL * NL + (long long)NL * rows * nd + S + (long long)S * nd + nd + nh + nd + 4 + S + S + nd + (long long)P * (nd + 2);
    double *ws = nullptr;
    CUDA_TRY(cudaMallocFromPoolAsync((void **)&ws, sizeof(double) * (size_t)(per * ld + 2) + 4 * sizeof(int32_t) * (size_t)ld, m->pool, stream));
    kin::IkCollLinksArgs a;
    std::memset(&a, 0, sizeof a);
    double *p = ws;
    auto take = [&](long long k) { double *r = p; p += k * ld; return r; };
    a.n = n; a.ld = ld; a.n_sph = S;
    a.q_try = take(nd);
    double *T = take(12LL * NL), *J = take((long long)NL * rows * nd), *V = take(S), *G = take((long long)S * nd);
    a.T = T; a.J = J; a.V = V; a.G = G;
    a.q = take(nd); a.H = take(nh); a.g = take(nd);
    a.phi = take(1); a.fpose = take(1); a.damp = take(1); a.viol = take(1); a.mult = take(S);
    double *Vfin = take(S);
    double *q_try_b = take(nd);                                  // second trial-point buffer (compaction ping-pong)
    double *VP = take(P), *GP = take((long long)P * nd);
    a.VP = VP; a.GP = GP; a.multP = take(P);
    unsigned long long *d_count = (unsigned long long *)p;
    p += 2;
    a.status = (int32_t *)p; a.its = a.status + ld;
    int32_t *act_buf[2] = {a.its + ld, a.its + 2 * ld};
    a.n_act = n; a.act = nullptr;
    a.margin = c->margin; a.mu = c->coll_weight > 0 ? c->coll_weight : 100.0; a.ftol = c->ftol;
    a.ctol = c->ctol > 0 ? c->ctol : 1e-6; a.lambda0 = c->lambda0 > 0 ? c->lambda0 : 1e-2;
    a.trunc = c->margin + 0.05;                                  // planning.jl:56
    a.targets = (const double *)c->targets;
    a.nd = nd;
    for (int j = 0; j < nd; ++j) {
        a.lo[j] = c->lower ? c->lower[j] : -INFINITY;
        a.hi[j] = c->upper ? c->upper[j] : INFINITY;
    }
    a.n_pairs = P;
    a.n_links = NL; a.rot_mask = lk.rot_mask;
    if (sb) { a.self_margin = sb->margin; a.self_trunc = sb->margin + 0.05; }      // as the sphere block (planning.jl:56)
    int rc = KIN_OK;
    kin::ik_coll_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(a, (const double *)c->q0, nd);
    g_launches.fetch_add(1);
    if (sb) {
        cudaError_t le = cudaMemsetAsync(a.multP, 0, sizeof(double) * (size_t)P * (size_t)ld, stream);      // multipliers 0
        if (le != cudaSuccess) { cudaFreeAsync(ws, stream); return fail_cuda(le, "clearing the pair multipliers of kin_ik_solve_self"); }
    }
    KinCall ec;
    std::memset(&ec, 0, sizeof ec);
    ec.precision = KIN_F64; ec.layout = KIN_LAYOUT_SOA; ec.n = n; ec.batch_stride = ld; ec.q = a.q_try;
    ec.n_fk_links = NL; ec.fk_links = lk.ids; ec.T_out = T;
    ec.n_jac_links = NL; ec.jac_links = lk.ids; ec.with_rot = lk.rot_mask ? 1 : 0; ec.rpy_jac = 1; ec.J_out = J;
    ec.truncation_dist = a.trunc; ec.grad_mode = KIN_GRAD_FD; ec.scratch_mode = KIN_SCRATCH_CLEAN;
    if (S > 0) { ec.vals_out = V; ec.grads_out = G; }
    ec.stream = c->stream;
    const bool compact = !std::getenv("KIN_IK_NO_COMPACT") && n >= 4096;
    int next_compact = 1, compact_step = 1, act_i = 0;
    for (int it = 0; it <= c->iters && rc == KIN_OK; ++it) {
        if (compact && it == next_compact) {
            // iterations 1, 2, 3, 4, 6, 8, 12, 16, 24, 32, 48, ...
            if (it >= 4 && (it & (it - 1)) == 0) compact_step = it / 2;
            next_compact = it + compact_step;
            cudaError_t le = cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), stream);
            double *q_in = a.q_try, *q_out_ = (a.q_try == q_try_b) ? ws : q_try_b;       // ws = the first buffer (take order)
            kin::ik_coll_compact_kernel<<<(unsigned)((a.n_act + 255) / 256), 256, 0, stream>>>(a, nd, q_in, act_buf[act_i], q_out_, d_count);
            if (le == cudaSuccess) le = cudaGetLastError();
            g_launches.fetch_add(1);
            unsigned long long cnt = 0;
            if (le == cudaSuccess) le = cudaMemcpyAsync(&cnt, d_count, sizeof cnt, cudaMemcpyDeviceToHost, stream);
            if (le == cudaSuccess) le = cudaStreamSynchronize(stream);
            if (le != cudaSuccess) { rc = fail_cuda(le, "compacting the active list of kin_ik_solve"); break; }
            a.act = act_buf[act_i]; a.n_act = (long long)cnt; a.q_try = q_out_;
            act_i ^= 1;
            ec.q = a.q_try; ec.n = a.n_act;
            if (cnt == 0) break;                                 // every problem has stopped
        }
        rc = kin_eval(m, &ec);
        if (rc != KIN_OK) break;
        if (sb) {           // the pairs at the same trial points, SoA FP64 of stride ld, truncated like the spheres
            rc = self_collision_launch(m, *sb->pairs, KIN_F64, KIN_LAYOUT_SOA, a.q_try, a.n_act, ld, a.self_trunc, 0.0, VP, GP,
                                       nullptr, nullptr, stream);
            if (rc != KIN_OK) break;
        }
        a.it = it;
        if (NL > 1 && sb) launch_ik_coll_step_any<true, true>(a, nd, rows, stream, m->dev_smem);
        else if (NL > 1) launch_ik_coll_step_any<false, true>(a, nd, rows, stream, m->dev_smem);
        else if (sb) launch_ik_coll_step_any<true, false>(a, nd, rows, stream, m->dev_smem);
        else launch_ik_coll_step_any<false, false>(a, nd, rows, stream, m->dev_smem);
        cudaError_t le = cudaGetLastError();
        if (le != cudaSuccess) { rc = fail_cuda(le, "launching ik_coll_step_kernel"); break; }
        g_launches.fetch_add(1);
    }
    if (rc == KIN_OK) {
        // the UNtruncated distances of the final configurations (for dmin_out)
        if (c->dmin_out && S > 0) {
            KinCall fc;
            std::memset(&fc, 0, sizeof fc);
            fc.precision = KIN_F64; fc.layout = KIN_LAYOUT_SOA; fc.n = n; fc.batch_stride = ld; fc.q = a.q;
            fc.truncation_dist = INFINITY; fc.vals_out = Vfin; fc.stream = c->stream;
            rc = kin_eval(m, &fc);
        }
        // ... and the smallest untruncated pair distance (a dmin-only self-collision launch at q)
        if (rc == KIN_OK && sb && sb->dmin_out)
            rc = self_collision_launch(m, *sb->pairs, KIN_F64, KIN_LAYOUT_SOA, a.q, n, ld, INFINITY, 0.0, nullptr, nullptr,
                                       sb->dmin_out, nullptr, stream);
        if (rc == KIN_OK) {
            kin::ik_coll_finish_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(a, Vfin, nd, (double *)c->q_out, (double *)c->f_out,
                                                                                     c->iters_out, S > 0 ? (double *)c->dmin_out : nullptr);
            cudaError_t le = cudaGetLastError();
            if (le != cudaSuccess) rc = fail_cuda(le, "launching ik_coll_finish_kernel");
            g_launches.fetch_add(1);
        }
    }
    cudaFreeAsync(ws, stream);
    return rc;
}

// The pose-only solve: the generated one-launch kernel (kin_gen_skeleton.cuh: kin_ik_kernel) around the links'
// straight-line FK + Euler-rate Jacobians, staged over the still-running problems for large batches.  Without the
// run-time compiler: the loop of ik_solve_coll without spheres.
int ik_solve_pose(KinModel *m, const KinIkCall *c, const IkLinks &lk) {
    const int nd = m->hm.n_dof();
    if (std::getenv("KIN_DISABLE_JIT")) return ik_solve_coll(m, c, lk);      // no run-time compiler: (kin_eval, step kernel) pairs
    DeviceGuard guard(m->device);
    // the program of (the links' transforms + their Euler-rate Jacobians)
    KinCall pc;
    std::memset(&pc, 0, sizeof pc);
    pc.precision = KIN_F64; pc.layout = KIN_LAYOUT_SOA; pc.n = c->n; pc.q = c->q0;
    pc.n_fk_links = lk.n; pc.fk_links = lk.ids; pc.T_out = (void *)c->q_out;
    pc.n_jac_links = lk.n; pc.jac_links = lk.ids; pc.J_out = (void *)c->q_out; pc.with_rot = lk.rot_mask ? 1 : 0; pc.rpy_jac = 1;
    pc.truncation_dist = INFINITY;
    std::shared_ptr<DeviceProgram> dp;
    int rc = get_program(m, &pc, KIND_FKJ, dp);
    if (rc != KIN_OK) return rc;
    std::shared_ptr<JitKernel> k = get_jit_with(m, dp.get(), ik_gen_options(lk), "kin_ik_kernel");
    if (!k) return ik_solve_coll(m, c, lk);
    kin::IkArgs a;
    std::memset(&a, 0, sizeof a);
    a.targets = c->targets; a.q0 = c->q0; a.q_out = c->q_out; a.f_out = c->f_out; a.iters_out = c->iters_out;
    a.n = c->n; a.iters = c->iters; a.ftol = c->ftol; a.lambda0 = c->lambda0 > 0 ? c->lambda0 : 1e-2;
    for (int j = 0; j < nd; ++j) {
        a.lo[j] = c->lower ? c->lower[j] : -INFINITY;
        a.hi[j] = c->upper ? c->upper[j] : INFINITY;
    }
    cudaStream_t stream = (cudaStream_t)c->stream;
    auto launch_stage = [&](kin::IkArgs &st) -> cudaError_t {
        void *args[] = {&st};
        const long long grid = (st.n + k->block - 1) / k->block;
        g_launches.fetch_add(1);
        g_jit_launches.fetch_add(1);
        return cudaLaunchKernel((const void *)k->kern, dim3((unsigned)grid), dim3((unsigned)k->block), args, 0, stream);
    };
    // STAGES.  One thread per problem leaves a warp busy until its slowest problem stops: most problems need 5-10
    // iterations, a few per cent all of them, so nearly every warp runs the whole budget.  A long solve over a large
    // batch is therefore split into a few launches (default: 3, 4, 6, 9 and the remaining iterations; 2^20 Fetch targets x 40
    // iterations: 17.9 -> 6.1 ms, profiles/sweep_ik_stages.sh); between two of them
    // the still-running problems (f >= ftol) are compacted into an index list whose length (8 bytes) is the only thing
    // read back.  A later stage restarts from the best point and the damping of the one before, re-evaluates there
    // (one extra evaluation per stage) and takes exactly the steps the single launch would have taken: same results.
    // KIN_IK_STAGES="a,b,..." overrides the schedule, KIN_IK_STAGES=0 disables it.
    std::vector<int> stages;
    {
        const char *e = std::getenv("KIN_IK_STAGES");
        std::string spec = e ? e : "3,4,6,9";
        if (c->n >= 16384 && spec != "0") {
            int left = c->iters;
            size_t pos = 0;
            while (pos < spec.size() && left > 0) {
                const int v = std::atoi(spec.c_str() + pos);
                if (v <= 0 || v >= left) break;
                stages.push_back(v);
                left -= v;
                pos = spec.find(',', pos);
                if (pos == std::string::npos) break;
                ++pos;
            }
            if (!stages.empty()) stages.push_back(left);
        }
    }
    if (stages.empty()) {
        CUDA_TRY(launch_stage(a));
        return KIN_OK;
    }
    // workspace: damping per problem, two index lists, the counter
    const long long n = c->n;
    unsigned char *ws = nullptr;
    CUDA_TRY(cudaMallocFromPoolAsync((void **)&ws, sizeof(double) * (size_t)(n + 2) + 2 * sizeof(int32_t) * (size_t)n, m->pool, stream));
    double *lam = (double *)ws;
    unsigned long long *d_count = (unsigned long long *)(lam + n);
    int32_t *lists[2] = {(int32_t *)(lam + n + 2), (int32_t *)(lam + n + 2) + n};
    a.lam_io = lam;
    cudaError_t le = cudaSuccess;
    long long n_act = n;
    const int32_t *act = nullptr;
    int done = 0;
    for (size_t si = 0; si < stages.size() && le == cudaSuccess && n_act > 0; ++si) {
        kin::IkArgs st = a;
        st.n = n_act; st.idx = act; st.iters = stages[si]; st.it0 = done;
        if (si > 0) st.q0 = c->q_out;                      // restart from the best point of the previous stage
        le = launch_stage(st);
        done += stages[si];
        if (le != cudaSuccess || si + 1 == stages.size()) break;
        int32_t *next = lists[si & 1];
        le = cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), stream);
        if (le == cudaSuccess) {
            kin::ik_compact_kernel<<<(unsigned)((n_act + 255) / 256), 256, 0, stream>>>(n_act, act, (const double *)c->f_out, c->ftol, next, d_count);
            le = cudaGetLastError();
            g_launches.fetch_add(1);
        }
        unsigned long long cnt = 0;
        if (le == cudaSuccess) le = cudaMemcpyAsync(&cnt, d_count, sizeof cnt, cudaMemcpyDeviceToHost, stream);
        if (le == cudaSuccess) le = cudaStreamSynchronize(stream);
        act = next; n_act = (long long)cnt;
    }
    cudaFreeAsync(ws, stream);
    if (le != cudaSuccess) return fail_cuda(le, "staged kin_ik_solve");
    return KIN_OK;
}

// The checks every solve makes before anything is launched (collision and pair table: ik_solve_checked).
int ik_check_call(KinModel *m, const KinIkCall *c, const char *what) {
    if (!m || !c) return fail(KIN_ERR_INVALID_ARGUMENT, "null model or call");
    if (c->n < 0 || (c->n > 0 && (!c->targets || !c->q0 || !c->q_out || !c->f_out))) return fail(KIN_ERR_INVALID_ARGUMENT, "null argument");
    if (c->iters < 0) return fail(KIN_ERR_INVALID_ARGUMENT, "negative iteration count");
    const int nd = m->hm.n_dof();
    if (nd < 1 || nd > kin::IKC_MAX_DOF) return fail(KIN_ERR_LIMIT, std::string(what) + ": 1..20 configuration columns");
    return KIN_OK;
}

// Every solve: the pair table (self_collision != 0) and the sphere / box tables (collision != 0) are checked before
// anything is launched, then the common path.
int ik_solve_checked(KinModel *m, const KinIkCall *c, const IkLinks &lk, bool self_collision, double self_margin,
                     void *self_dmin_out, const char *what) {
    if (self_collision && std::isnan(self_margin)) return fail(KIN_ERR_INVALID_ARGUMENT, std::string(what) + ": self_margin is NaN");
    IkSelfBlock sb;
    if (self_collision) {
        {
            std::lock_guard<std::mutex> lock(m->mu);
            sb.pairs = m->self_pairs;
        }
        if (!sb.pairs) return fail(KIN_ERR_INVALID_ARGUMENT, std::string(what) + ": the model has no pair table (kin_model_set_self_pairs)");
    }
    if (c->collision && (m->hm.n_sph < 1 || m->hm.n_box < 1))
        return fail(KIN_ERR_INVALID_ARGUMENT, "kin_ik_solve: collision requested but the model has no spheres / no boxes");
    if (c->collision && std::isnan(c->margin)) return fail(KIN_ERR_INVALID_ARGUMENT, "kin_ik_solve: margin is NaN");
    if (c->n == 0) return KIN_OK;
    if (!self_collision) return c->collision ? ik_solve_coll(m, c, lk) : ik_solve_pose(m, c, lk);
    sb.margin = self_margin;
    sb.dmin_out = self_dmin_out;
    return ik_solve_coll(m, c, lk, &sb);
}

}  // namespace
extern "C" {

int kin_ik_solve(KinModel *m, const KinIkCall *c) {
    int rc = ik_check_call(m, c, "kin_ik_solve");
    if (rc != KIN_OK) return rc;
    if (c->link_id < 1 || c->link_id > m->hm.n_links) return fail(KIN_ERR_INVALID_ARGUMENT, "link id out of range");
    return ik_solve_checked(m, c, ik_one_link(c), false, 0.0, nullptr, "kin_ik_solve");
}

// kin_ik_solve plus the self-collision pairs as a hard constraint: always the augmented-Lagrangian loop of ik_solve_coll.
// Every argument is checked before anything is launched.
int kin_ik_solve_self(KinModel *m, const KinIkCall *c, double self_margin, void *self_dmin_out) {
    int rc = ik_check_call(m, c, "kin_ik_solve_self");
    if (rc != KIN_OK) return rc;
    if (c->link_id < 1 || c->link_id > m->hm.n_links) return fail(KIN_ERR_INVALID_ARGUMENT, "link id out of range");
    return ik_solve_checked(m, c, ik_one_link(c), true, self_margin, self_dmin_out, "kin_ik_solve_self");
}

// Several links at once (extension): kin_ik_solve / kin_ik_solve_self on f = sum_l |e_l|^2.  One link is exactly the
// call of those two.  Every argument is checked before anything is launched.
int kin_ik_solve_links(KinModel *m, const KinIkCall *c, int32_t n_links, const int32_t *link_ids, const int32_t *with_rots,
                       int32_t self_collision, double self_margin, void *self_dmin_out) {
    int rc = ik_check_call(m, c, "kin_ik_solve_links");
    if (rc != KIN_OK) return rc;
    if (n_links < 1 || n_links > KIN_IK_MAX_LINKS) return fail(KIN_ERR_INVALID_ARGUMENT, "kin_ik_solve_links: 1..KIN_IK_MAX_LINKS links");
    if (!link_ids || !with_rots) return fail(KIN_ERR_INVALID_ARGUMENT, "kin_ik_solve_links: null link_ids / with_rots");
    IkLinks lk;
    lk.n = n_links;
    for (int l = 0; l < n_links; ++l) {
        if (link_ids[l] < 1 || link_ids[l] > m->hm.n_links) return fail(KIN_ERR_INVALID_ARGUMENT, "link id out of range");
        for (int k = 0; k < l; ++k)
            if (link_ids[k] == link_ids[l]) return fail(KIN_ERR_INVALID_ARGUMENT, "kin_ik_solve_links: repeated link id");
        lk.ids[l] = link_ids[l];
        if (with_rots[l]) lk.rot_mask |= 1u << l;
    }
    return ik_solve_checked(m, c, lk, self_collision != 0, self_margin, self_dmin_out, "kin_ik_solve_links");
}

// FP64 peak probe (the denominator of the "FP64 pipe" column of the rooflines): every thread runs 8 independent
// DFMA chains, 8 CTAs of 256 threads per SM.
int kin_collision_summary(KinModel *m, int32_t precision, int32_t layout, const void *q, int64_t n, double margin,
                          void *dmin_out, int32_t *amin_out, void *cost_out, void *stream_) {
    if (!m) return fail(KIN_ERR_INVALID_ARGUMENT, "null model");
    if (int rc = check_batch(precision, layout, n, q, kAnyLayout)) return rc;
    if (n > 0 && !dmin_out) return fail(KIN_ERR_INVALID_ARGUMENT, "null dmin_out");
    if (n == 0) return KIN_OK;
    DeviceGuard guard(m->device);
    const int S = m->hm.n_sph, nd = m->hm.n_dof();
    if (S < 1 || m->hm.n_box < 1) return fail(KIN_ERR_INVALID_ARGUMENT, "collision summary: the model has no spheres / no boxes");
    cudaStream_t stream = (cudaStream_t)stream_;
    const size_t es = precision == KIN_F32 ? 4 : 8;
    // the distances of a chunk go through a stream-ordered temporary (S values per configuration), then the reduction
    long long chunk = std::max<long long>(32, env_ll("KIN_SUMMARY_CHUNK", 1 << 20)) / 32 * 32;      // a multiple of 32 (tiled: whole tiles)
    if (chunk > n) chunk = n;
    void *tmp = nullptr;
    CUDA_TRY(cudaMallocFromPoolAsync(&tmp, es * (size_t)S * (size_t)((chunk + 31) / 32 * 32), m->pool, stream));
    int rc = KIN_OK;
    for (long long n0 = 0; n0 < n && rc == KIN_OK; n0 += chunk) {
        const long long cnt = std::min<long long>(chunk, n - n0);
        KinCall c;
        std::memset(&c, 0, sizeof c);
        c.precision = precision; c.layout = layout; c.n = cnt; c.stream = stream_;
        c.truncation_dist = INFINITY; c.vals_out = tmp;
        // AoS / tiled: a chunk is a contiguous part of q (chunk starts are multiples of 32).  SoA: q and the outputs of
        // one call share one row stride, so a chunk of a longer batch gets its q rows gathered into a [n_dof][cnt] block
        c.q = (const unsigned char *)q + es * (size_t)n0 * nd;
        void *qtmp = nullptr;
        if (layout == KIN_LAYOUT_SOA) {
            c.q = q;
            if (cnt != n) {
                cudaError_t e = cudaMallocFromPoolAsync(&qtmp, es * (size_t)nd * (size_t)cnt, m->pool, stream);
                if (e == cudaSuccess)
                    e = cudaMemcpy2DAsync(qtmp, es * cnt, (const unsigned char *)q + es * (size_t)n0, es * (size_t)n, es * cnt, nd,
                                          cudaMemcpyDeviceToDevice, stream);
                if (e != cudaSuccess) { if (qtmp) cudaFreeAsync(qtmp, stream); rc = fail_cuda(e, "staging a SoA chunk"); break; }
                c.q = qtmp;
            }
        }
        rc = kin_eval(m, &c);
        if (qtmp) cudaFreeAsync(qtmp, stream);
        if (rc != KIN_OK) break;
        const long long ld = cnt;                                  // row stride of the temporary (SoA)
        const bool aos = layout == KIN_LAYOUT_AOS;
        long long grid = aos ? (cnt * 32 + 255) / 256 : (cnt + 255) / 256;
        grid = std::max<long long>(1, std::min<long long>(grid, (long long)m->n_sm * 16));
        unsigned char *dm = (unsigned char *)dmin_out + es * (size_t)n0, *co = cost_out ? (unsigned char *)cost_out + es * (size_t)n0 : nullptr;
        int32_t *am = amin_out ? amin_out + n0 : nullptr;
#define KIN_SUMMARY(real, lay) kin::coll_summary_kernel<real, lay><<<(unsigned)grid, 256, 0, stream>>>((const real *)tmp, cnt, ld, S, (real)margin, (real *)dm, am, (real *)co)
        if (precision == KIN_F64) { if (layout == KIN_LAYOUT_SOA) KIN_SUMMARY(double, 0); else if (aos) KIN_SUMMARY(double, 1); else KIN_SUMMARY(double, 2); }
        else { if (layout == KIN_LAYOUT_SOA) KIN_SUMMARY(float, 0); else if (aos) KIN_SUMMARY(float, 1); else KIN_SUMMARY(float, 2); }
#undef KIN_SUMMARY
        cudaError_t le = cudaGetLastError();
        if (le != cudaSuccess) { rc = fail_cuda(le, "launching coll_summary_kernel"); break; }
        g_launches.fetch_add(1);
    }
    cudaFreeAsync(tmp, stream);
    return rc;
}

}  // extern "C"
namespace {
__global__ void __launch_bounds__(256) probe_dfma_kernel(double *out, int iters) {
    double a[8];
    #pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = 1e-9 * (threadIdx.x + k);
    const double b = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        #pragma unroll
        for (int k = 0; k < 8; ++k) a[k] = fma(a[k], b, c);
    }
    double s = 0;
    #pragma unroll
    for (int k = 0; k < 8; ++k) s += a[k];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}
}  // namespace
extern "C" {

int kin_probe_fp64(double *tflops_out, double *dfma_per_clk_per_sm_out, double *sm_mhz_out) {
    int dev = 0, n_sm = 0, khz = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    CUDA_TRY(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, dev));
    const int grid = n_sm * 8, block = 256, iters = 1 << 16;
    double *buf = nullptr;
    CUDA_TRY(cudaMalloc(&buf, sizeof(double) * (size_t)grid * block));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {          // first repetition = warm-up
        CUDA_TRY(cudaEventRecord(e0, 0));
        probe_dfma_kernel<<<grid, block>>>(buf, iters);
        CUDA_TRY(cudaEventRecord(e1, 0));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    g_launches.fetch_add(4);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf);
    const double dfma = 8.0 * iters * (double)grid * block;
    if (tflops_out) *tflops_out = 2.0 * dfma / (best * 1e-3) / 1e12;
    // per clock at the NOMINAL maximum SM clock (the achieved clock is sampled by the caller with nvidia-smi)
    if (dfma_per_clk_per_sm_out) *dfma_per_clk_per_sm_out = dfma / (best * 1e-3) / ((double)khz * 1e3) / n_sm;
    if (sm_mhz_out) *sm_mhz_out = khz / 1e3;
    return KIN_OK;
}

int kin_fk_links(KinModel *m, int32_t precision, int32_t layout, const void *q, int64_t n, const int32_t *link_ids,
                 int32_t n_req, void *T_out, void *stream) {
    KinCall c;
    std::memset(&c, 0, sizeof c);
    c.precision = precision; c.layout = layout; c.n = n; c.q = q;
    c.n_fk_links = n_req; c.fk_links = link_ids; c.T_out = T_out; c.stream = stream;
    c.truncation_dist = INFINITY;
    return kin_eval(m, &c);
}

int kin_fk_jacobian(KinModel *m, int32_t precision, int32_t layout, const void *q, int64_t n, const int32_t *link_ids,
                    int32_t n_req, int32_t with_rot, int32_t rpy_jac, void *T_out, void *J_out, void *stream) {
    KinCall c;
    std::memset(&c, 0, sizeof c);
    c.precision = precision; c.layout = layout; c.n = n; c.q = q;
    c.n_fk_links = n_req; c.fk_links = link_ids; c.T_out = T_out;
    c.n_jac_links = n_req; c.jac_links = link_ids; c.with_rot = with_rot; c.rpy_jac = rpy_jac; c.J_out = J_out;
    c.stream = stream; c.truncation_dist = INFINITY;
    return kin_eval(m, &c);
}

int kin_collision(KinModel *m, int32_t precision, int32_t layout, const void *q, int64_t n, double truncation_dist,
                  int32_t grad_mode, int32_t scratch_mode, void *vals_out, void *grads_out, int32_t *argmin_out,
                  void *stream) {
    KinCall c;
    std::memset(&c, 0, sizeof c);
    c.precision = precision; c.layout = layout; c.n = n; c.q = q;
    c.truncation_dist = truncation_dist; c.grad_mode = grad_mode; c.scratch_mode = scratch_mode;
    c.vals_out = vals_out; c.grads_out = grads_out; c.argmin_out = argmin_out; c.stream = stream;
    return kin_eval(m, &c);
}

int kin_self_collision(KinModel *m, int32_t precision, int32_t layout, const void *q, int64_t n, double truncation_dist,
                       double vals_offset, void *vals_out, void *grads_out, void *dmin_out, int32_t *amin_out, void *stream) {
    if (!m) return fail(KIN_ERR_INVALID_ARGUMENT, "null model");
    if (int rc = check_batch(precision, layout, n, q, kAnyLayout)) return rc;
    if (!vals_out && !dmin_out) return fail(KIN_ERR_INVALID_ARGUMENT, "self collision: neither vals_out nor dmin_out given");
    if (grads_out && !vals_out) return fail(KIN_ERR_INVALID_ARGUMENT, "self collision: grads_out needs vals_out");
    if (std::isnan(truncation_dist)) return fail(KIN_ERR_INVALID_ARGUMENT, "truncation_dist is NaN");
    DeviceGuard guard(m->device);
    std::shared_ptr<DevicePairs> pairs;
    {
        std::lock_guard<std::mutex> lock(m->mu);
        pairs = m->self_pairs;
    }
    if (!pairs) return fail(KIN_ERR_INVALID_ARGUMENT, "self collision: the model has no pair table (kin_model_set_self_pairs)");
    if (n == 0) return KIN_OK;
    return self_collision_launch(m, *pairs, precision, layout, q, n, n, truncation_dist, vals_offset, vals_out, grads_out,
                                 dmin_out, amin_out, (cudaStream_t)stream);
}

}  // extern "C"

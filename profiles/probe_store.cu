// probe_store.cu -- what write bandwidth does B200 HBM3e sustain for the OUTPUT PATTERNS of the FK kernel, with no
// arithmetic at all?  348 doubles per configuration (25 links x 12 + 6 x 8 Jacobian), N configurations.
//   fill      contiguous grid-stride stores (the roof)
//   soa       x[comp * N + n]: a CTA tile of 128 configurations writes 1 KB to each of 348 rows (plain / st.cs)
//   tiled     x[((n / 32) * 348 + comp) * 32 + n % 32]: each warp writes one contiguous 89 KB block
//   soa_bulk  as soa, staged per warp through shared memory, 256-B cp.async.bulk per component row
//   tiled_bulk as tiled, staged per warp: 12 components x 32 lanes = 3 KB per cp.async.bulk
//   soa_cta_bulk  CTA-wide staging [12][128], one 1-KB cp.async.bulk per component row
// `probe_store fill [rounds]` instead runs the write-ceiling section (DESIGN 4.4, profiles/probe_fill.py): a contiguous
// 8 GiB fill with each store form, and the headline's output mix at 2^22 configurations with its 175 configuration-
// independent rows written as contiguous fills; every variant once per round, rounds repeated, median / min / max.
// Build: nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o profiles/_bin/probe_store profiles/probe_store.cu
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <functional>
#include <vector>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1); } } while (0)
constexpr int REC = 348, BS = 128;

__global__ void k_fill(double *x, long long total) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) x[i] = 1.0;
}
template <bool CS, bool TILED>
__global__ void __launch_bounds__(BS) k_pattern(double *x, long long N) {
    const long long n_tiles = N / BS;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long n = tile * BS + threadIdx.x;
        double *p = TILED ? x + (n >> 5) * (long long)(REC * 32) + (n & 31) : x + n;
        const size_t es = TILED ? 32 : (size_t)N;
        const double v = (double)n;
        #pragma unroll 12
        for (int c = 0; c < REC; ++c) {
            if (CS) __stcs(p + c * es, v + c); else p[c * es] = v + c;
        }
    }
}
// the same pattern with the things the real kernel has and the plain probe lacks, one at a time:
//   READQ    8 coalesced loads per configuration before the stores (mixed read / write traffic)
//   DELAY    a dependent DFMA chain of that length in front of every group of 12 stores (the stores of a warp are
//            spread over the computation instead of being issued back to back)
//   PERMUTE  the 29 groups of 12 components are visited in a scattered order (DFS order != output order)
template <bool TILED, bool READQ, int DELAY, bool PERMUTE>
__global__ void __launch_bounds__(BS) k_real(double *x, const double *q, long long N) {
    const long long n_tiles = N / BS;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long n = tile * BS + threadIdx.x;
        double *p = TILED ? x + (n >> 5) * (long long)(REC * 32) + (n & 31) : x + n;
        const size_t es = TILED ? 32 : (size_t)N;
        double v = (double)n;
        if (READQ) {
            const double *qp = TILED ? q + (n >> 5) * (long long)(8 * 32) + (n & 31) : q + n;
            #pragma unroll
            for (int c = 0; c < 8; ++c) v += qp[c * es];
        }
        #pragma unroll 1
        for (int g0 = 0; g0 < 29; ++g0) {
            const int g = PERMUTE ? (g0 * 11 + 7) % 29 : g0;
            #pragma unroll
            for (int d = 0; d < DELAY; ++d) v = fma(v, 1.0000001, 1e-9);
            #pragma unroll
            for (int c = 0; c < 12; ++c) p[(g * 12 + c) * es] = v + c;
        }
    }
}

// READQ with the reads clustered in time: every PF-th tile each CTA prefetches the configurations of its tiles
// k + PF .. k + 2 PF - 1 into L2 (evict_last); the CTAs run in near lock-step, so the DRAM sees the reads of a whole
// period as one burst instead of a trickle that keeps interrupting the write drain.
template <bool TILED, int PF>
__global__ void __launch_bounds__(BS) k_real_pf(double *x, const double *q, long long N) {
    const long long n_tiles = N / BS;
    long long k = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++k) {
        if (k % PF == 0) {
            // lines of 128 B: per tile 8 rows x 8 lines (SoA) or one contiguous 8 KB block (tiled: 64 lines)
            for (int i = threadIdx.x; i < PF * 64; i += BS) {
                const long long t2 = tile + (long long)(PF + i / 64) * gridDim.x;
                if (t2 < n_tiles) {
                    const int l = i % 64;
                    const double *a = TILED ? q + t2 * (long long)(BS * 8) + l * 16 : q + (long long)(l / 8) * N + t2 * BS + (l % 8) * 16;
                    asm volatile("prefetch.global.L2::evict_last [%0];" ::"l"(a));
                }
            }
        }
        const long long n = tile * BS + threadIdx.x;
        double *p = TILED ? x + (n >> 5) * (long long)(REC * 32) + (n & 31) : x + n;
        const size_t es = TILED ? 32 : (size_t)N;
        double v = (double)n;
        const double *qp = TILED ? q + (n >> 5) * (long long)(8 * 32) + (n & 31) : q + n;
        #pragma unroll
        for (int c = 0; c < 8; ++c) v += qp[c * es];
        #pragma unroll 1
        for (int g = 0; g < 29; ++g) {
            #pragma unroll
            for (int c = 0; c < 12; ++c) p[(g * 12 + c) * es] = v + c;
        }
    }
}

// More ways of getting the 8 input doubles per configuration in (SoA outputs throughout):
//   MODE 0  per-thread loads with a cache operator (CACHE: 0 plain, 1 .cg, 2 .cs, 3 .nc)
//   MODE 1  warp 0 loads the whole tile (8 rows x 1 KB) with 16-byte loads into shared memory, then a barrier
//   MODE 2  every RT-th tile the CTA loads the inputs of RT tiles into shared memory (8 rows x RT KB)
//   MODE 3  the inputs are stored tiled (one contiguous 8 KB block per tile of 128), outputs stay SoA
template <int MODE, int CACHE, int RT>
__global__ void __launch_bounds__(BS) k_real2(double *x, const double *q, long long N) {
    __shared__ __align__(16) double sq[(MODE == 2 ? RT : 1) * 8 * BS];
    const long long n_tiles = N / BS;
    long long k = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++k) {
        const long long n = tile * BS + threadIdx.x;
        double v = (double)n;
        if (MODE == 0) {
            #pragma unroll
            for (int c = 0; c < 8; ++c) {
                const double *a = q + (long long)c * N + n;
                double t;
                if (CACHE == 1) asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(t) : "l"(a));
                else if (CACHE == 2) asm volatile("ld.global.cs.f64 %0, [%1];" : "=d"(t) : "l"(a));
                else if (CACHE == 3) asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(t) : "l"(a));
                else t = *a;
                v += t;
            }
        } else if (MODE == 1) {
            __syncthreads();
            if (threadIdx.x < 32)
                #pragma unroll
                for (int i = 0; i < 16; ++i) {        // 8 rows x 64 double2 = 512 double2, 32 lanes x 16
                    const int e = i * 32 + threadIdx.x, row = e / 64, col = e % 64;
                    reinterpret_cast<double2 *>(sq)[row * 64 + col] = reinterpret_cast<const double2 *>(q + (long long)row * N + tile * BS)[col];
                }
            __syncthreads();
            #pragma unroll
            for (int c = 0; c < 8; ++c) v += sq[c * BS + threadIdx.x];
        } else if (MODE == 2) {
            if (k % RT == 0) {
                __syncthreads();
                for (int r = 0; r < RT; ++r) {
                    const long long t2 = tile + (long long)r * gridDim.x;
                    if (t2 < n_tiles)
                        #pragma unroll
                        for (int c = 0; c < 8; ++c) sq[(r * 8 + c) * BS + threadIdx.x] = q[(long long)c * N + t2 * BS + threadIdx.x];
                }
                __syncthreads();
            }
            #pragma unroll
            for (int c = 0; c < 8; ++c) v += sq[((k % RT) * 8 + c) * BS + threadIdx.x];
        } else {
            const double *qp = q + tile * (long long)(BS * 8) + threadIdx.x;
            #pragma unroll
            for (int c = 0; c < 8; ++c) v += qp[c * BS];
        }
        double *p = x + n;
        #pragma unroll 1
        for (int g = 0; g < 29; ++g) {
            #pragma unroll
            for (int c = 0; c < 12; ++c) p[(size_t)(g * 12 + c) * N] = v + c;
        }
    }
}

// Inputs of RT tiles per batch, double-buffered in DYNAMIC shared memory with cp.async (the next batch is in flight
// while the current one is processed); optionally every CTA waits at a grid-wide barrier before issuing the loads of
// a batch, so that all SMs read at the same moment (one read burst per batch for the whole GPU).
__device__ unsigned g_bar_count = 0;
__device__ volatile unsigned g_bar_gen = 0;
__device__ __forceinline__ void grid_barrier(unsigned n_cta) {
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned gen = g_bar_gen;
        __threadfence();
        if (atomicAdd(&g_bar_count, 1) == n_cta - 1) { g_bar_count = 0; __threadfence(); g_bar_gen = gen + 1; }
        else while (g_bar_gen == gen) __nanosleep(100);
    }
    __syncthreads();
}
template <bool GRIDSYNC>
__global__ void __launch_bounds__(BS) k_batched(double *x, const double *q, long long N, int RT) {
    extern __shared__ __align__(16) double sqd[];          // [2][RT][8][BS]
    const long long n_tiles = N / BS;
    const long long my_tiles = (long long)blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const long long n_batches = (my_tiles + RT - 1) / RT;
    const long long max_tiles = (n_tiles + gridDim.x - 1) / gridDim.x, max_batches = (max_tiles + RT - 1) / RT;
    auto issue = [&](long long b, int buf) {
        for (int r = 0; r < RT; ++r) {
            const long long k = b * RT + r;
            if (k < my_tiles) {
                const long long t2 = blockIdx.x + k * gridDim.x;
                #pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const double *src = q + (long long)c * N + t2 * BS + threadIdx.x;
                    double *dst = sqd + ((size_t)(buf * RT + r) * 8 + c) * BS + threadIdx.x;
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src));
                }
            }
        }
        asm volatile("cp.async.commit_group;");
    };
    if (GRIDSYNC) grid_barrier(gridDim.x);
    issue(0, 0);
    for (long long b = 0; b < max_batches; ++b) {
        const int buf = (int)(b & 1);
        if (GRIDSYNC) grid_barrier(gridDim.x);
        issue(b + 1, buf ^ 1);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();
        if (b < n_batches)
            for (int r = 0; r < RT; ++r) {
                const long long k = b * RT + r;
                if (k >= my_tiles) break;
                const long long n = (blockIdx.x + k * gridDim.x) * BS + threadIdx.x;
                double v = (double)n;
                #pragma unroll
                for (int c = 0; c < 8; ++c) v += sqd[((size_t)(buf * RT + r) * 8 + c) * BS + threadIdx.x];
                double *p = x + n;
                #pragma unroll 1
                for (int g = 0; g < 29; ++g) {
                    #pragma unroll
                    for (int c = 0; c < 12; ++c) p[(size_t)(g * 12 + c) * N] = v + c;
                }
            }
        __syncthreads();
    }
}

__device__ __forceinline__ void bulk_store(void *gdst, const void *ssrc, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"((unsigned)__cvta_generic_to_shared(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N_> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N_) : "memory"); }
__device__ __forceinline__ void fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// per-warp staging: CH components x 32 lanes, double buffered
template <bool TILED, int CH>
__global__ void __launch_bounds__(BS) k_warp_bulk(double *x, long long N) {
    __shared__ __align__(128) double stage[BS / 32][2][CH][32];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long n_tiles = N / BS;
    int buf = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long n0 = tile * BS + w * 32;          // first configuration of this warp
        const double v = (double)(n0 + lane);
        for (int c0 = 0; c0 < REC; c0 += CH) {
            if (lane == 0) bulk_wait_read<1>();            // the buffer we are about to overwrite has been read
            __syncwarp();
            const int ch = min(CH, REC - c0);
            #pragma unroll
            for (int c = 0; c < CH; ++c) if (c < ch) stage[w][buf][c][lane] = v + c0 + c;
            fence_async();
            __syncwarp();
            if (lane == 0) {
                if (TILED) bulk_store(x + (n0 >> 5) * (long long)(REC * 32) + (long long)c0 * 32, &stage[w][buf][0][0], ch * 32 * 8);
                else
                    for (int c = 0; c < ch; ++c) bulk_store(x + (long long)(c0 + c) * N + n0, &stage[w][buf][c][0], 32 * 8);
                bulk_commit();
            }
            buf ^= 1;
        }
    }
    if (lane == 0) bulk_wait_read<0>();
}
// CTA-wide staging [CH][128]: one 1-KB bulk store per component row, issued by warp 0's lanes
template <int CH>
__global__ void __launch_bounds__(BS) k_cta_bulk(double *x, long long N) {
    __shared__ __align__(128) double stage[2][CH][BS];
    const long long n_tiles = N / BS;
    int buf = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long n0 = tile * BS;
        const double v = (double)(n0 + threadIdx.x);
        for (int c0 = 0; c0 < REC; c0 += CH) {
            if (threadIdx.x < CH) bulk_wait_read<1>();
            __syncthreads();
            #pragma unroll
            for (int c = 0; c < CH; ++c) stage[buf][c][threadIdx.x] = v + c0 + c;
            fence_async();
            __syncthreads();
            if (threadIdx.x < CH) {
                bulk_store(x + (long long)(c0 + threadIdx.x) * N + n0, &stage[buf][threadIdx.x][0], BS * 8);
                bulk_commit();
            }
            buf ^= 1;
        }
    }
    if (threadIdx.x < CH) bulk_wait_read<0>();
}

// ---- write-ceiling section ----
// one store of VB bytes of the value v at p (VB = 8: STG.E.64, 16: STG.E.128, 32: STG.E.ENL2.256), optionally .cs
template <int VB, bool CS> __device__ __forceinline__ void st_vec(double *p, double v) {
    if (VB == 8) { if (CS) __stcs(p, v); else *p = v; }
    else if (VB == 16) { if (CS) asm volatile("st.global.cs.v2.f64 [%0], {%1, %1};" ::"l"(p), "d"(v) : "memory");
                         else asm volatile("st.global.v2.f64 [%0], {%1, %1};" ::"l"(p), "d"(v) : "memory"); }
    else { if (CS) asm volatile("st.global.cs.v4.f64 [%0], {%1, %1, %1, %1};" ::"l"(p), "d"(v) : "memory");
           else asm volatile("st.global.v4.f64 [%0], {%1, %1, %1, %1};" ::"l"(p), "d"(v) : "memory"); }
}
// contiguous fill, grid-stride over VB-byte vectors
template <int VB, bool CS> __global__ void k_fill_vec(double *x, long long total) {
    constexpr int E = VB / 8;
    const long long nv = total / E;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) st_vec<VB, CS>(x + i * E, 1.0);
}
// contiguous fill, one vector per thread, one short-lived CTA per 256 vectors (the shape of torch's fill_ kernel)
template <int VB> __global__ void k_fill_np(double *x) {
    st_vec<VB, false>(x + ((long long)blockIdx.x * blockDim.x + threadIdx.x) * (VB / 8), 1.0);
}
// ... the same with the CTAs' addresses scattered (CTA b writes block (b * 7919) mod gridDim.x): same bytes, same
// shape, no single advancing write front
template <int VB> __global__ void k_fill_np_scatter(double *x) {
    const long long b = ((long long)blockIdx.x * 7919) % gridDim.x;
    st_vec<VB, false>(x + (b * blockDim.x + threadIdx.x) * (VB / 8), 1.0);
}
// persistent grid-stride fill, 1 CTA of 128 per SM, with a grid-wide barrier every SYNC iterations (the CTAs kept
// within SYNC x 4.7 MB of each other)
template <int VB, int SYNC> __global__ void __launch_bounds__(BS) k_fill_sync(double *x, long long total) {
    constexpr int E = VB / 8;
    const long long nv = total / E, stride = (long long)gridDim.x * blockDim.x;
    int k = 0;
    for (long long i0 = 0; i0 < nv; i0 += stride) {
        const long long i = i0 + (long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (i < nv) st_vec<VB, false>(x + i * E, 1.0);
        if (++k == SYNC) { k = 0; grid_barrier(gridDim.x); }
    }
}
// contiguous fill, every CTA one contiguous range of total / gridDim.x (the split of the in-kernel fill of the mix below)
template <int VB> __global__ void k_fill_chunk(double *x, long long total) {
    constexpr int E = VB / 8;
    const long long per = total / gridDim.x / E;
    double *p = x + (long long)blockIdx.x * per * E;
    #pragma unroll 4
    for (long long j = threadIdx.x; j < per; j += blockDim.x) st_vec<VB, false>(p + j * E, 1.0);
}
// persistent fill, 1 CTA of 128 per SM, with DYNAMIC work distribution: a CTA claims the next CHUNK bytes from a global
// counter (zeroed before every launch), so an SM whose writes drain faster takes more of the work
__device__ unsigned long long g_fill_next = 0;
template <int VB, int CHUNK> __global__ void __launch_bounds__(BS) k_fill_dyn(double *x, long long total) {
    __shared__ long long s_c;
    constexpr int E = VB / 8;
    constexpr long long CE = CHUNK / 8;
    for (;;) {
        if (threadIdx.x == 0) s_c = (long long)atomicAdd(&g_fill_next, 1ull);
        __syncthreads();
        const long long c = s_c;
        __syncthreads();
        if (c >= total / CE) break;
        double *p = x + c * CE;
        #pragma unroll 4
        for (int j = threadIdx.x; j < CE / E; j += BS) st_vec<VB, false>(p + j * E, 1.0);
    }
}
// contiguous fill by the TMA engine: one lane per warp sends PIECE-byte copies of a shared buffer holding the value
template <int PIECE> __global__ void __launch_bounds__(BS) k_fill_bulk(double *x, long long total) {
    __shared__ __align__(128) double buf[PIECE / 8];
    for (int i = threadIdx.x; i < PIECE / 8; i += BS) buf[i] = 1.0;
    fence_async();
    __syncthreads();
    if ((threadIdx.x & 31) == 0) {
        const long long np = total / (PIECE / 8), w = (long long)blockIdx.x * (BS / 32) + (threadIdx.x >> 5), nw = (long long)gridDim.x * (BS / 32);
        for (long long i = w; i < np; i += nw) { bulk_store(x + i * (PIECE / 8), buf, PIECE); bulk_commit(); }
        asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
}
// the headline's output mix: of the 348 rows, 175 (spread over the record like the real constant rows) hold one value
// for every configuration.  OLD: all 348 rows stored per thread (the kernel as it stands: input batches of RT tiles
// behind a grid-wide barrier, 1 CTA / SM).  Otherwise the 173 varying rows are stored per thread and the 175 constant
// rows are filled contiguously (each CTA one contiguous range of the flattened (row, column) space, VB-byte stores):
// all of it before the first batch (MODE 1) or one slice of it after every batch (MODE 2).
__host__ __device__ constexpr bool mix_const(int c) { return (c * 175) / REC != ((c + 1) * 175) / REC; }
__constant__ int c_const_rows[175];                        // the rows c with mix_const(c), in order
template <int VB, bool CS>
__device__ __forceinline__ void fill_range(double *x, long long N, long long i0, long long i1) {
    constexpr int E = VB / 8;
    while (i0 < i1) {
        const long long r = i0 / N, c0 = i0 - r * N, len = (i1 - i0 < N - c0) ? i1 - i0 : N - c0;
        const int row = c_const_rows[r];
        double *p = x + (long long)row * N + c0;
        const double v = 2.0 + row;
        long long head = (long long)((((unsigned long long)-(long long)p) & (VB - 1)) / 8);
        if (head > len) head = len;
        const long long body = (len - head) / E, tail0 = head + body * E;
        if (threadIdx.x < head) p[threadIdx.x] = v;
        #pragma unroll 4
        for (long long j = threadIdx.x; j < body; j += BS) st_vec<VB, CS>(p + head + j * E, v);
        if (tail0 + threadIdx.x < len) p[tail0 + threadIdx.x] = v;
        i0 += len;
    }
}
// the 175 constant rows of the mix by short-lived CTAs (the torch fill_ shape), one VB-byte vector per thread: a second
// launch, for comparison with the fill inside the persistent kernel
template <int VB> __global__ void k_fill_rows_np(double *x, long long N) {
    const long long per_row = N / (VB / 8) / blockDim.x;
    const int row = c_const_rows[blockIdx.x / per_row];
    st_vec<VB, false>(x + (long long)row * N + ((blockIdx.x % per_row) * blockDim.x + threadIdx.x) * (VB / 8), 2.0 + row);
}
template <int MODE, int VB, bool CS>      // MODE 0 old, 1 fill first, 2 fill per batch, 3 the 173 varying rows only,
                                          // 4 fill first in dynamically claimed pieces
__global__ void __launch_bounds__(BS) k_mix(double *x, const double *q, long long N, int RT) {
    constexpr bool OLD = MODE == 0, SLICED = MODE == 2;
    extern __shared__ __align__(16) double sqd[];          // [2][RT][8][BS]
    const long long n_tiles = N / BS;
    const long long my_tiles = (long long)blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const long long max_tiles = (n_tiles + gridDim.x - 1) / gridDim.x, max_batches = (max_tiles + RT - 1) / RT;
    const long long fill_total = 175 * N, per_cta = (fill_total + gridDim.x - 1) / gridDim.x;
    const long long f0 = min(fill_total, (long long)blockIdx.x * per_cta), f1 = min(fill_total, f0 + per_cta);
    const long long per_batch = (f1 - f0 + max_batches - 1) / max_batches;
    auto issue = [&](long long b, int buf) {
        for (int r = 0; r < RT; ++r) {
            const long long k = b * RT + r;
            if (k < my_tiles) {
                const long long t2 = blockIdx.x + k * gridDim.x;
                #pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const double *src = q + (long long)c * N + t2 * BS + threadIdx.x;
                    double *dst = sqd + ((size_t)(buf * RT + r) * 8 + c) * BS + threadIdx.x;
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src));
                }
            }
        }
        asm volatile("cp.async.commit_group;");
    };
    if (MODE == 1) fill_range<VB, CS>(x, N, f0, f1);
    if (MODE == 4 || MODE == 5) {                       // fill first, 256-KB pieces claimed dynamically (k_fill_dyn),
        __shared__ long long s_c;                       // the next piece claimed while the current one is written
        constexpr long long CH = 32768;
        if (threadIdx.x == 0) s_c = (long long)atomicAdd(&g_fill_next, 1ull);
        __syncthreads();
        long long c = s_c;
        __syncthreads();
        while (c * CH < fill_total) {
            if (threadIdx.x == 0) s_c = (long long)atomicAdd(&g_fill_next, 1ull);
            fill_range<VB, CS>(x, N, c * CH, min(fill_total, (c + 1) * CH));
            __syncthreads();
            c = s_c;
            __syncthreads();
        }
    }
    if (MODE == 5) return;                              // the fill alone
    grid_barrier(gridDim.x);
    issue(0, 0);
    for (long long b = 0; b < max_batches; ++b) {
        const int buf = (int)(b & 1);
        grid_barrier(gridDim.x);
        issue(b + 1, buf ^ 1);
        asm volatile("cp.async.wait_group 1;" ::: "memory");
        __syncthreads();
        for (int r = 0; r < RT; ++r) {
            const long long k = b * RT + r;
            if (k >= my_tiles) break;
            const long long n = (blockIdx.x + k * gridDim.x) * BS + threadIdx.x;
            double v = (double)n;
            #pragma unroll
            for (int c = 0; c < 8; ++c) v += sqd[((size_t)(buf * RT + r) * 8 + c) * BS + threadIdx.x];
            double *p = x + n;
            #pragma unroll
            for (int c = 0; c < REC; ++c)
                if (OLD || !mix_const(c)) p[(size_t)c * N] = v + c;
        }
        if (SLICED) fill_range<VB, CS>(x, N, min(f1, f0 + b * per_batch), min(f1, f0 + (b + 1) * per_batch));
        __syncthreads();
    }
}

template <typename F> float timeit(F launch, int reps) {
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    launch(); launch();
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(a));
    for (int i = 0; i < reps; ++i) launch();
    CK(cudaEventRecord(b));
    CK(cudaEventSynchronize(b));
    float ms; CK(cudaEventElapsedTime(&ms, a, b));
    return ms / reps;
}

int fill_main(int rounds) {
    int n_sm; CK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, 0));
    const long long total = 1ll << 30;                       // 8 GiB of doubles
    const long long N = 1ll << 22, RT = 12;
    double *x, *q;
    CK(cudaMalloc(&x, (size_t)total * 8 > (size_t)4 * N * REC * 8 ? (size_t)total * 8 : (size_t)4 * N * REC * 8));   // up to 2^24 configurations
    CK(cudaMalloc(&q, N * 8 * 8));
    CK(cudaMemset(q, 0, N * 8 * 8));
    struct V { const char *name; double gb; std::function<void()> run; std::vector<float> ms; };
    std::vector<V> vs;
    const double fill_gb = total * 8 / 1e9, mix_gb = (N * REC * 8 + N * 64) / 1e9;
    const int g4 = n_sm * 4;
    vs.push_back({"fill  8 B STG", fill_gb, [&] { k_fill_vec<8, false><<<g4, 256>>>(x, total); }, {}});
    vs.push_back({"fill  8 B STG .cs", fill_gb, [&] { k_fill_vec<8, true><<<g4, 256>>>(x, total); }, {}});
    vs.push_back({"fill 16 B STG", fill_gb, [&] { k_fill_vec<16, false><<<g4, 256>>>(x, total); }, {}});
    vs.push_back({"fill 16 B STG .cs", fill_gb, [&] { k_fill_vec<16, true><<<g4, 256>>>(x, total); }, {}});
    vs.push_back({"fill 32 B STG", fill_gb, [&] { k_fill_vec<32, false><<<g4, 256>>>(x, total); }, {}});
    vs.push_back({"fill 32 B STG .cs", fill_gb, [&] { k_fill_vec<32, true><<<g4, 256>>>(x, total); }, {}});
    vs.push_back({"fill 32 B STG, 128 threads/SM", fill_gb, [&] { k_fill_vec<32, false><<<n_sm, 128>>>(x, total); }, {}});
    vs.push_back({"fill 32 B STG, 2048 threads/SM", fill_gb, [&] { k_fill_vec<32, false><<<n_sm * 8, 256>>>(x, total); }, {}});
    vs.push_back({"fill 16 B STG, 2048 threads/SM", fill_gb, [&] { k_fill_vec<16, false><<<n_sm * 8, 256>>>(x, total); }, {}});
    vs.push_back({"fill 16 B, one vector / thread, 2^21 CTAs", fill_gb, [&] { k_fill_np<16><<<(unsigned)(total / 2 / 256), 256>>>(x); }, {}});
    vs.push_back({"fill 32 B, one vector / thread, 2^20 CTAs", fill_gb, [&] { k_fill_np<32><<<(unsigned)(total / 4 / 256), 256>>>(x); }, {}});
    vs.push_back({"fill 32 B, one vector / thread, CTAs scattered", fill_gb, [&] { k_fill_np_scatter<32><<<(unsigned)(total / 4 / 256), 256>>>(x); }, {}});
    vs.push_back({"fill 32 B, 1 x 128 / SM, grid barrier / 64 it", fill_gb, [&] { k_fill_sync<32, 64><<<n_sm, BS>>>(x, total); }, {}});
    vs.push_back({"fill 32 B, 1 x 128 / SM, grid barrier / 8 it", fill_gb, [&] { k_fill_sync<32, 8><<<n_sm, BS>>>(x, total); }, {}});
    vs.push_back({"fill 32 B, range per CTA, 1 x 128 / SM", fill_gb, [&] { k_fill_chunk<32><<<n_sm, 128>>>(x, total); }, {}});
    vs.push_back({"fill 32 B, range per CTA, 8 x 256 / SM", fill_gb, [&] { k_fill_chunk<32><<<n_sm * 8, 256>>>(x, total); }, {}});
    unsigned long long *d_next;
    CK(cudaGetSymbolAddress((void **)&d_next, g_fill_next));
    vs.push_back({"fill 32 B, 1 x 128 / SM, dynamic 16 KB pieces", fill_gb, [&] { cudaMemsetAsync(d_next, 0, 8); k_fill_dyn<32, 16384><<<n_sm, BS>>>(x, total); }, {}});
    vs.push_back({"fill 32 B, 1 x 128 / SM, dynamic 1 MB pieces", fill_gb, [&] { cudaMemsetAsync(d_next, 0, 8); k_fill_dyn<32, 1 << 20><<<n_sm, BS>>>(x, total); }, {}});
    vs.push_back({"fill 32 B, 1 x 128 / SM, dynamic 64 KB pieces", fill_gb, [&] { cudaMemsetAsync(d_next, 0, 8); k_fill_dyn<32, 65536><<<n_sm, BS>>>(x, total); }, {}});
    vs.push_back({"fill 32 B, 1 x 128 / SM, dynamic 256 KB pieces", fill_gb, [&] { cudaMemsetAsync(d_next, 0, 8); k_fill_dyn<32, 262144><<<n_sm, BS>>>(x, total); }, {}});
    vs.push_back({"fill 32 B, 4 x 128 / SM, dynamic 64 KB pieces", fill_gb, [&] { cudaMemsetAsync(d_next, 0, 8); k_fill_dyn<32, 65536><<<n_sm * 4, BS>>>(x, total); }, {}});
    vs.push_back({"fill cp.async.bulk 16 KB, 4 CTAs / SM", fill_gb, [&] { k_fill_bulk<16384><<<n_sm * 4, BS>>>(x, total); }, {}});
    vs.push_back({"fill cp.async.bulk 1 KB", fill_gb, [&] { k_fill_bulk<1024><<<n_sm, BS>>>(x, total); }, {}});
    vs.push_back({"fill cp.async.bulk 4 KB", fill_gb, [&] { k_fill_bulk<4096><<<n_sm, BS>>>(x, total); }, {}});
    vs.push_back({"fill cp.async.bulk 16 KB", fill_gb, [&] { k_fill_bulk<16384><<<n_sm, BS>>>(x, total); }, {}});
    {
        int rows[175];
        for (int c = 0, k = 0; c < REC; ++c) if (mix_const(c)) rows[k++] = c;
        CK(cudaMemcpyToSymbol(c_const_rows, rows, sizeof rows));
    }
    const size_t smem = (size_t)2 * RT * 8 * BS * 8;
#define MIX(NAME, MODE, VB, CS)                                                                                           \
    CK(cudaFuncSetAttribute(k_mix<MODE, VB, CS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));              \
    vs.push_back({NAME, mix_gb, [&] { k_mix<MODE, VB, CS><<<n_sm, BS, smem>>>(x, q, N, (int)RT); }, {}});
    MIX("mix 2^22: old, 348 rows per thread", 0, 8, false)
    MIX("mix 2^22: 173 rows + fill first, 8 B", 1, 8, false)
    MIX("mix 2^22: 173 rows + fill first, 16 B", 1, 16, false)
    MIX("mix 2^22: 173 rows + fill first, 32 B", 1, 32, false)
    MIX("mix 2^22: 173 rows + fill first, 32 B .cs", 1, 32, true)
    MIX("mix 2^22: 173 rows + fill per batch, 16 B", 2, 16, false)
    MIX("mix 2^22: 173 rows + fill per batch, 32 B", 2, 32, false)
    MIX("mix 2^22: 173 rows + fill per batch, 32 B .cs", 2, 32, true)
    MIX("mix 2^22: 173 rows only (GB/s of all 348)", 3, 8, false)
    CK(cudaFuncSetAttribute(k_mix<5, 32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    vs.push_back({"mix 2^22: the claimed fill alone (GB/s of 175 rows)", 175 * N * 8 / 1e9, [&] { cudaMemsetAsync(d_next, 0, 8); k_mix<5, 32, false><<<n_sm, BS, smem>>>(x, q, N, (int)RT); }, {}});
    vs.push_back({"mix 2^24: the claimed fill alone (GB/s of 175 rows)", 175 * (4 * N) * 8 / 1e9, [&] { cudaMemsetAsync(d_next, 0, 8); k_mix<5, 32, false><<<n_sm, BS, smem>>>(x, q, 4 * N, (int)RT); }, {}});
    CK(cudaFuncSetAttribute(k_mix<4, 32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    vs.push_back({"mix 2^22: 173 rows + fill first, dynamic, 32 B", mix_gb, [&] { cudaMemsetAsync(d_next, 0, 8); k_mix<4, 32, false><<<n_sm, BS, smem>>>(x, q, N, (int)RT); }, {}});
    vs.push_back({"mix 2^22: memset + old (launch cost of the above)", mix_gb, [&] { cudaMemsetAsync(d_next, 0, 8); k_mix<0, 8, false><<<n_sm, BS, smem>>>(x, q, N, (int)RT); }, {}});
#undef MIX
    vs.push_back({"mix 2^22: 173 rows, then fill kernel (2 launches)", mix_gb, [&] {
        k_mix<3, 8, false><<<n_sm, BS, smem>>>(x, q, N, (int)RT);
        k_fill_rows_np<32><<<(unsigned)(175 * (N / 4 / 256)), 256>>>(x, N);
    }, {}});
    for (int r = 0; r < rounds; ++r)
        for (auto &v : vs) v.ms.push_back(timeit(v.run, 5));
    printf("%-48s %9s %9s %9s %9s   (%d rounds of 5 launches each, variants alternating)\n", "variant", "med ms", "min ms", "max ms", "med GB/s", rounds);
    for (auto &v : vs) {
        std::vector<float> s = v.ms;
        std::sort(s.begin(), s.end());
        const float med = s[s.size() / 2];
        printf("%-48s %9.4f %9.4f %9.4f %9.1f\n", v.name, med, s.front(), s.back(), v.gb / (med * 1e-3));
    }
    CK(cudaFree(x)); CK(cudaFree(q));
    return 0;
}

int main(int argc, char **argv) {
    if (argc > 1 && !strcmp(argv[1], "fill")) return fill_main(argc > 2 ? atoi(argv[2]) : 7);
    const long long N = argc > 1 ? atoll(argv[1]) : (1ll << 22);
    const long long total = N * REC;
    double *x;
    CK(cudaMalloc(&x, total * 8));
    int n_sm; CK(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, 0));
    const double gb = total * 8 / 1e9;
    auto rep = [&](const char *name, float ms) { printf("%-34s %8.3f ms  %8.1f GB/s\n", name, ms, gb / (ms * 1e-3)); };
    rep("fill (contiguous)", timeit([&] { k_fill<<<n_sm * 16, 256>>>(x, total); }, 5));
    for (int occ : {3, 4, 8, 16}) {
        char nm[64];
        snprintf(nm, sizeof nm, "soa plain        grid %d/SM", occ); rep(nm, timeit([&] { k_pattern<false, false><<<n_sm * occ, BS>>>(x, N); }, 5));
        snprintf(nm, sizeof nm, "soa st.cs        grid %d/SM", occ); rep(nm, timeit([&] { k_pattern<true, false><<<n_sm * occ, BS>>>(x, N); }, 5));
        snprintf(nm, sizeof nm, "tiled plain      grid %d/SM", occ); rep(nm, timeit([&] { k_pattern<false, true><<<n_sm * occ, BS>>>(x, N); }, 5));
        snprintf(nm, sizeof nm, "tiled st.cs      grid %d/SM", occ); rep(nm, timeit([&] { k_pattern<true, true><<<n_sm * occ, BS>>>(x, N); }, 5));
    }
    {
        double *q;
        CK(cudaMalloc(&q, N * 8 * 8));
        CK(cudaMemset(q, 0, N * 8 * 8));
        const int g3 = n_sm * 3;
        rep("soa   real: base (3/SM)", timeit([&] { k_real<false, false, 0, false><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: +read q", timeit([&] { k_real<false, true, 0, false><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: +delay 16", timeit([&] { k_real<false, false, 16, false><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: +delay 64", timeit([&] { k_real<false, false, 64, false><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: +permute", timeit([&] { k_real<false, false, 0, true><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: all (delay 16)", timeit([&] { k_real<false, true, 16, true><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real2: ld.cg", timeit([&] { k_real2<0, 1, 1><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real2: ld.cs", timeit([&] { k_real2<0, 2, 1><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real2: ld.nc no_allocate", timeit([&] { k_real2<0, 3, 1><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real2: warp 0 loads tile -> smem", timeit([&] { k_real2<1, 0, 1><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real2: 4 tiles at a time -> smem", timeit([&] { k_real2<2, 0, 4><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real2: 5 tiles at a time -> smem", timeit([&] { k_real2<2, 0, 5><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real2: tiled q, soa out", timeit([&] { k_real2<3, 0, 1><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real2: plain, 1 CTA/SM", timeit([&] { k_real2<0, 0, 1><<<n_sm, BS>>>(x, q, N); }, 5));
        rep("soa   real2: plain, 2 CTA/SM", timeit([&] { k_real2<0, 0, 1><<<n_sm * 2, BS>>>(x, q, N); }, 5));
        rep("soa   real2: plain, 6 CTA/SM", timeit([&] { k_real2<0, 0, 1><<<n_sm * 6, BS>>>(x, q, N); }, 5));
        for (int occ : {1, 2}) for (int RT : {2, 4, 6, 12}) {
            const size_t smem = (size_t)2 * RT * 8 * BS * 8;
            if (smem * occ > 220 * 1024) continue;
            CK(cudaFuncSetAttribute(k_batched<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CK(cudaFuncSetAttribute(k_batched<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            char nm[80];
            snprintf(nm, sizeof nm, "soa batched cp.async RT=%d, %d CTA/SM", RT, occ);
            rep(nm, timeit([&] { k_batched<false><<<n_sm * occ, BS, smem>>>(x, q, N, RT); }, 5));
            snprintf(nm, sizeof nm, "soa batched+gridsync RT=%d, %d CTA/SM", RT, occ);
            rep(nm, timeit([&] { k_batched<true><<<n_sm * occ, BS, smem>>>(x, q, N, RT); }, 5));
        }
        rep("soa   real: +read q, L2 prefetch P=2", timeit([&] { k_real_pf<false, 2><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: +read q, L2 prefetch P=4", timeit([&] { k_real_pf<false, 4><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: +read q, L2 prefetch P=8", timeit([&] { k_real_pf<false, 8><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: +read q, L2 prefetch P=16", timeit([&] { k_real_pf<false, 16><<<g3, BS>>>(x, q, N); }, 5));
        rep("soa   real: +read q, L2 prefetch P=32", timeit([&] { k_real_pf<false, 32><<<g3, BS>>>(x, q, N); }, 5));
        rep("tiled real: +read q, L2 prefetch P=4", timeit([&] { k_real_pf<true, 4><<<g3, BS>>>(x, q, N); }, 5));
        rep("tiled real: +read q, L2 prefetch P=16", timeit([&] { k_real_pf<true, 16><<<g3, BS>>>(x, q, N); }, 5));
        rep("tiled real: base (3/SM)", timeit([&] { k_real<true, false, 0, false><<<g3, BS>>>(x, q, N); }, 5));
        rep("tiled real: +read q", timeit([&] { k_real<true, true, 0, false><<<g3, BS>>>(x, q, N); }, 5));
        rep("tiled real: +delay 16", timeit([&] { k_real<true, false, 16, false><<<g3, BS>>>(x, q, N); }, 5));
        rep("tiled real: +delay 64", timeit([&] { k_real<true, false, 64, false><<<g3, BS>>>(x, q, N); }, 5));
        rep("tiled real: +permute", timeit([&] { k_real<true, false, 0, true><<<g3, BS>>>(x, q, N); }, 5));
        rep("tiled real: all (delay 16)", timeit([&] { k_real<true, true, 16, true><<<g3, BS>>>(x, q, N); }, 5));
        CK(cudaFree(q));
    }
    for (int occ : {3, 8}) {
        char nm[64];
        snprintf(nm, sizeof nm, "soa warp-bulk 256B  grid %d/SM", occ); rep(nm, timeit([&] { k_warp_bulk<false, 12><<<n_sm * occ, BS>>>(x, N); }, 5));
        snprintf(nm, sizeof nm, "tiled warp-bulk 3KB grid %d/SM", occ); rep(nm, timeit([&] { k_warp_bulk<true, 12><<<n_sm * occ, BS>>>(x, N); }, 5));
        snprintf(nm, sizeof nm, "tiled warp-bulk 6KB grid %d/SM", occ); rep(nm, timeit([&] { k_warp_bulk<true, 24><<<n_sm * occ, BS>>>(x, N); }, 5));
        snprintf(nm, sizeof nm, "soa cta-bulk 1KB    grid %d/SM", occ); rep(nm, timeit([&] { k_cta_bulk<12><<<n_sm * occ, BS>>>(x, N); }, 5));
    }
    CK(cudaFree(x));
    return 0;
}

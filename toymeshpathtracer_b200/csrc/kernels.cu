// kernels.cu -- CUDA kernels (sm_100a) and the compute half of the C ABI (include/tmpt.h).
//
//   K1  BVH build      k_prim_bounds, k_prim_boxes, k_sah_build (binned SAH, all levels in one cooperative launch; default) or
//                      k_morton, k_radix_sort, k_leaf_boxes, k_karras, k_refit (LBVH); then k_collapse_all to 4-wide nodes
//                      (replaces Scene::BuildOctree, scene.cpp:75-160)
//   K2  closest hit    k_hit_scene<CLOSEST>   (Scene::HitScene, scene.cpp:86-97, batched)
//   K3  any hit        k_hit_scene<ANY>       (the shadow query of Scatter, main.cpp:59)
//       brute force    k_hit_scene<BRUTE>     (upstream's all-triangle scan; cross-check only)
//   K4  path tracing   k_render, k_resolve    (TraceImageBody / Trace / Scatter, main.cpp:44-119, 192-238)
//   K5  share gather   k_unpack_stripes       (rank 0 after the multi-GPU gather; the default multi-GPU path has no gather:
//                                              every rank's k_render stores its pixels into rank 0's frame over NVLink)
//   K6  refit          k_refit_pending, k_refit_wide  (tmpt_scene_refit: moved vertices, same topology)
//   K9  denoise        k_denoise_prep, k_denoise_atrous, k_denoise_copy  (tmpt_denoise: a-trous filter over the radiance and AOVs)
//
// There is no CPU fallback in this file: every entry point needs a CUDA device.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "build_logic.cuh"
#include "common.h"
#include "denoise.cuh"
#include "integrator.cuh"
// The render kernel with per-lane ray regeneration (k_render_regen: measured in rounds 1 and 2, 31 % slower, DESIGN.md 5) is
// compiled only with -DTMPT_EXPERIMENTS=1; the shipped library does not contain it.  (Round 1's three experimental HitScene
// kernels -- warp queue, deferred triangle tests, cooperative leaf phase -- were removed in round 2: git history, profiles/r1_*.)
#ifndef TMPT_EXPERIMENTS
#define TMPT_EXPERIMENTS 0
#endif

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
namespace tmpt {
static thread_local std::string g_err;
static std::atomic<uint64_t> g_launches{0};
int fail(int status, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return status;
}
void count_launch(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
}  // namespace tmpt

extern "C" const char* tmpt_last_error(void) { return tmpt::g_err.c_str(); }
extern "C" uint64_t tmpt_launch_count(void) { return tmpt::g_launches.load(); }
extern "C" int tmpt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

#define CU_TRY(expr)                                                                                       \
    do {                                                                                                   \
        cudaError_t e_ = (expr);                                                                           \
        if (e_ != cudaSuccess) return tmpt::fail(e_ == cudaErrorMemoryAllocation ? TMPT_ERR_OOM : TMPT_ERR_CUDA, \
                                                 "%s:%d %s: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e_)); \
    } while (0)
#define TRY(expr)                                \
    do {                                         \
        const int rc_ = (expr);                  \
        if (rc_ != TMPT_OK) return rc_;          \
    } while (0)
#define LAUNCH(kernel, grid, block, smem, stream, ...)      \
    do {                                                    \
        kernel<<<(grid), (block), (smem), (stream)>>>(__VA_ARGS__); \
        tmpt::count_launch();                               \
    } while (0)

static inline int div_up(long long a, long long b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------
// owned memory: every device and pinned host allocation of a scene or a call
// ------------------------------------------------------------------------------------------
namespace {
struct DeviceMem {
    static cudaError_t alloc(void** p, size_t bytes) { return cudaMalloc(p, bytes); }
    static void free(void* p) { cudaFree(p); }
};
struct PinnedMem {  // page-locked host memory: asynchronous copies to and from it
    static cudaError_t alloc(void** p, size_t bytes) { return cudaHostAlloc(p, bytes, cudaHostAllocDefault); }
    static void free(void* p) { cudaFreeHost(p); }
};
// n elements of T: freed by the destructor, grown (not shrunk) on demand and reused, contents not preserved.
template <class T, class Mem = DeviceMem>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;  // elements
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { reset(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
        return *this;
    }
    ~DevBuf() { reset(); }
    void reset() { if (p) Mem::free(p); p = nullptr; cap = 0; }
    // Room for at least n elements (at least 1).  Growing first waits for `st`, where work may still use the old memory, and
    // allocates max(n, allocN) elements.  A failed allocation leaves the buffer empty, so the next call tries again.
    cudaError_t grow(size_t n, cudaStream_t st, size_t allocN = 0) {
        n = std::max<size_t>(n, 1);
        if (cap >= n) return cudaSuccess;
        if (p) {
            const cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) return e;
        }
        reset();
        n = std::max(n, allocN);
        const cudaError_t e = Mem::alloc((void**)&p, n * sizeof(T));
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = n;
        return cudaSuccess;
    }
};
template <class T>
using PinnedBuf = DevBuf<T, PinnedMem>;
}  // namespace

// ------------------------------------------------------------------------------------------
// the scene object behind tmpt_scene*
// ------------------------------------------------------------------------------------------
struct tmpt_scene {
    int device = 0;
    int triCount = 0;
    int smCount = 148;
    cudaStream_t stream = nullptr;
    DevBuf<float> d_tris9;         // caller's triangles, original order
    DevBuf<float4> d_nodes;        // wide nodes, 7 x float4 each: what the walk reads; then the views below
    DevBuf<uint4> d_qnodes;        // wide nodes, quantised: only in a -DTMPT_QNODES=1 build (an experiment, not the default)
    float4* d_tris = nullptr;      // leaf-ordered MT slots
    float4* d_hitdata = nullptr;   // per original triangle: vertices + precomputed normal
    uint32_t* d_parent = nullptr;  // per wide node: parent index (refit)
    uint32_t* d_pending = nullptr; // per wide node: inner children not yet refitted (refit scratch)
    uint32_t* d_bounds = nullptr;  // scene bounds as ordered uints (refit scratch)
    DevBuf<uint32_t> d_status;     // [0] status bits
    // render scratch
    DevBuf<uint32_t> d_tileCounter;
    DevBuf<unsigned long long> d_rayCount;
    DevBuf<unsigned long long> d_fetchCounter;  // ray queue head of the persistent HitScene kernel
    // rgba, radiance, normal, depth, triangle staged on the device (indexed like Staging::user): tmpt_render_outputs(TMPT_HOST)
    // and tmpt_denoise(TMPT_HOST); [0] is also the frame of a call that asks for none, and tmpt_render_multi's frame
    DevBuf<char> staged[5];
    DevBuf<float4> d_accum;        // chunk sums of the band being rendered
    DevBuf<float4> d_sum;          // progressive render: running per-pixel sums
    int progW = 0, progH = 0, progChunks = -1;  // -1: no progressive render begun
    int progAdaptive = -1;         // the session's kind, fixed by its first pass: -1 none yet, 0 uniform, 1 adaptive
    // adaptive passes (tmpt_progressive_pass_adaptive), allocated by a session's first adaptive pass: per pixel (tile-padded
    // frame) the chunk count and (mean, M2) of the chunk-mean luminance; the select flags, their exclusive scan and scan totals;
    // the active list
    DevBuf<uint32_t> d_adN;
    DevBuf<float2> d_adStat;
    DevBuf<uint32_t> d_adFlags, d_adOffs, d_adTotals;  // d_adTotals: scan totals, then the grand total
    DevBuf<uint2> d_adList;
    DevBuf<unsigned int> d_adActive;  // [0] pixels left active by the pass, [1] the session's largest chunk count n
    DevBuf<int32_t> d_samples;     // tmpt_progressive_pass_adaptive(TMPT_HOST): samples staged on the device
    DevBuf<float4> d_denoise;      // tmpt_denoise: [4][pixels] float4: two state buffers (ping-pong), guideA, guideB (denoise.cuh)
    // staging of tmpt_hit_scene(TMPT_HOST): one device and one pinned host buffer per scene, grown on demand and reused (the
    // entry point is called in a loop by batched-query users: five cudaMalloc / cudaFree pairs and pageable copies per call
    // cost more than the kernel for batches under a million rays)
    DevBuf<char> d_stage;
    PinnedBuf<char> h_stage;
    // serialises the entry points that use or reallocate per-scene scratch (staging, frame, accum, progressive sums, sun grid,
    // counters) or the timing events ev0 / ev1
    std::mutex hostCallMutex;
    DevBuf<uint32_t> d_sunStart, d_sunCount;  // sun grid (sungrid.cuh): cell offsets; counts / fill cursors + scan scratch
    DevBuf<uint2> d_sunEntries;
    uint32_t sunEntries = 0;
    uint64_t sunBytes = 0;
    // render-kernel choice (k_render vs k_render_paths), cached per camera / frame size: see k_probe_paths
    tmpt_camera probeCam{};
    int probeW = 0, probeH = 0, probeUsePaths = -1;  // -1: no decision yet
    int lastUsedPaths = -1;                           // what the last frame ran (tmpt_render_kernel_choice)
    bool probePending = false;                        // a probe is in flight: h_probe is valid once probeDone has passed
    float probeEscape = 0.0f;
    DevBuf<unsigned int> d_probe;  // device counters
    PinnedBuf<unsigned int> h_probe;  // their pinned copy
    cudaEvent_t probeDone = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bvh::SceneView view{};
    tmpt_scene_info info{};
};

// ------------------------------------------------------------------------------------------
// K1: BVH build
// ------------------------------------------------------------------------------------------
// bounds[0..2] = min, [3..5] = max as order-preserving uints
__global__ void k_prim_bounds(const float* __restrict__ tris9, int n, uint32_t* __restrict__ bounds) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    bld::Box b{3.0e38f, 3.0e38f, 3.0e38f, -3.0e38f, -3.0e38f, -3.0e38f};
    if (i < n) b = bld::tri_box(tris9 + (size_t)i * 9);
    // warp reduce, then one atomic per warp
    for (int o = 16; o > 0; o >>= 1) {
        b.lox = fminf(b.lox, __shfl_xor_sync(0xffffffffu, b.lox, o));
        b.loy = fminf(b.loy, __shfl_xor_sync(0xffffffffu, b.loy, o));
        b.loz = fminf(b.loz, __shfl_xor_sync(0xffffffffu, b.loz, o));
        b.hix = fmaxf(b.hix, __shfl_xor_sync(0xffffffffu, b.hix, o));
        b.hiy = fmaxf(b.hiy, __shfl_xor_sync(0xffffffffu, b.hiy, o));
        b.hiz = fmaxf(b.hiz, __shfl_xor_sync(0xffffffffu, b.hiz, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(&bounds[0], bld::float_to_ordered(b.lox));
        atomicMin(&bounds[1], bld::float_to_ordered(b.loy));
        atomicMin(&bounds[2], bld::float_to_ordered(b.loz));
        atomicMax(&bounds[3], bld::float_to_ordered(b.hix));
        atomicMax(&bounds[4], bld::float_to_ordered(b.hiy));
        atomicMax(&bounds[5], bld::float_to_ordered(b.hiz));
    }
}

__device__ __forceinline__ bld::Box load_scene_box(const uint32_t* bounds) {
    return bld::Box{bld::ordered_to_float(bounds[0]), bld::ordered_to_float(bounds[1]), bld::ordered_to_float(bounds[2]),
                    bld::ordered_to_float(bounds[3]), bld::ordered_to_float(bounds[4]), bld::ordered_to_float(bounds[5])};
}

__global__ void k_morton(const float* __restrict__ tris9, int n, const uint32_t* __restrict__ bounds,
                         uint64_t* __restrict__ keys, uint32_t* __restrict__ prim) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bld::Box scene = load_scene_box(bounds);
    const bld::Box b = bld::tri_box(tris9 + (size_t)i * 9);
    keys[i] = bld::morton63(0.5f * (b.lox + b.hix), 0.5f * (b.loy + b.hiy), 0.5f * (b.loz + b.hiz), scene);
    prim[i] = (uint32_t)i;
}

// Stable LSD radix sort of (key, value) pairs by ONE cooperative CTA, 4 bits per pass.
// Thread t owns the contiguous chunk [t*per, (t+1)*per): it counts its 16 digits, the CTA
// scans the (digit-major, thread-minor) table in shared memory, and the thread scatters its
// chunk in order -- stable because chunk order is thread order.  The build is a one-off of
// <= a few 100k primitives (untimed by the reference, main.cpp:312), so one SM is enough.
constexpr int SORT_THREADS = 1024;
__global__ void __launch_bounds__(SORT_THREADS) k_radix_sort(uint64_t* keysA, uint32_t* valsA, uint64_t* keysB, uint32_t* valsB, int n,
                                                            int passes) {
    extern __shared__ uint32_t table[];  // 16 * SORT_THREADS entries = 64 KB (dynamic: above the static limit)
    __shared__ uint32_t warpTotals[32];
    const int t = threadIdx.x;
    const int per = (n + SORT_THREADS - 1) / SORT_THREADS;
    const int b = min(t * per, n), e = min(b + per, n);
    uint64_t* kin = keysA; uint32_t* vin = valsA; uint64_t* kout = keysB; uint32_t* vout = valsB;
    for (int pass = 0; pass < passes; ++pass) {
        const int shift = pass * 4;
        uint32_t cnt[16];
#pragma unroll
        for (int d = 0; d < 16; ++d) cnt[d] = 0;
        for (int i = b; i < e; ++i) {
            const int dgt = (int)((kin[i] >> shift) & 15);
#pragma unroll
            for (int d = 0; d < 16; ++d) cnt[d] += (d == dgt);
        }
#pragma unroll
        for (int d = 0; d < 16; ++d) table[d * SORT_THREADS + t] = cnt[d];
        __syncthreads();
        // exclusive scan of the 16*1024 table: each thread scans 16 consecutive entries
        uint32_t local[16];
        uint32_t sum = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k) { local[k] = sum; sum += table[t * 16 + k]; }
        uint32_t incl = sum;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
            if ((t & 31) >= o) incl += y;
        }
        if ((t & 31) == 31) warpTotals[t >> 5] = incl;
        __syncthreads();
        if (t < 32) {
            uint32_t w = warpTotals[t];
            uint32_t wi = w;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, wi, o);
                if (t >= o) wi += y;
            }
            warpTotals[t] = wi - w;
        }
        __syncthreads();
        const uint32_t base = warpTotals[t >> 5] + incl - sum;
#pragma unroll
        for (int k = 0; k < 16; ++k) table[t * 16 + k] = base + local[k];
        __syncthreads();
        uint32_t off[16];
#pragma unroll
        for (int d = 0; d < 16; ++d) off[d] = table[d * SORT_THREADS + t];
        for (int i = b; i < e; ++i) {
            const uint64_t k = kin[i];
            const int dgt = (int)((k >> shift) & 15);
            uint32_t dst = 0;
#pragma unroll
            for (int d = 0; d < 16; ++d) {
                if (d == dgt) { dst = off[d]; off[d] = dst + 1; }
            }
            kout[dst] = k;
            vout[dst] = vin[i];
        }
        __syncthreads();
        uint64_t* tk = kin; kin = kout; kout = tk;
        uint32_t* tv = vin; vin = vout; vout = tv;
    }
}

// leaf j of the binary tree = sorted position j: padded box, cost of a 1-triangle leaf, count 1
__global__ void k_leaf_boxes(const float* __restrict__ tris9, const uint32_t* __restrict__ prim, int n,
                             const uint32_t* __restrict__ bounds, float cTri, float4* __restrict__ lo, float4* __restrict__ hi,
                             int* __restrict__ first) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const bld::Box scene = load_scene_box(bounds);
    const float maxAbs = fmaxf(fmaxf(fmaxf(fabsf(scene.lox), fabsf(scene.hix)), fmaxf(fabsf(scene.loy), fabsf(scene.hiy))),
                               fmaxf(fabsf(scene.loz), fabsf(scene.hiz)));
    bld::Box b = bld::tri_box(tris9 + (size_t)prim[j] * 9);
    const float dx = b.hix - b.lox, dy = b.hiy - b.loy, dz = b.hiz - b.loz;
    const float pad = bld::pad_for(sqrtf(dx * dx + dy * dy + dz * dz), maxAbs);
    b.lox -= pad; b.loy -= pad; b.loz -= pad; b.hix += pad; b.hiy += pad; b.hiz += pad;
    lo[n - 1 + j] = make_float4(b.lox, b.loy, b.loz, cTri * bld::box_half_area(b));
    hi[n - 1 + j] = make_float4(b.hix, b.hiy, b.hiz, ex::u2f((uint32_t)-1));  // one triangle, a leaf
    first[n - 1 + j] = j;
}

__global__ void k_karras(bld::BinTree t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < t.n - 1) bld::karras_node(t, i);
}

// bottom-up: the second child to arrive at a node combines both (Karras 2012, section 4)
__global__ void k_refit(bld::BinTree t, bld::SahParams sp) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= t.n) return;
    int node = t.parent[t.n - 1 + j];
    while (node >= 0) {
        __threadfence();
        if (atomicAdd(&t.visits[node], 1u) == 0u) return;
        __threadfence();
        bld::refit_node(t, node, sp);
        node = t.parent[node];
    }
}

// per original triangle: (v0, n.x) (v1, n.y) (v2, n.z), n = normalize(e1 x e2) exactly as maths.cpp:375 computes it per hit
__global__ void k_hitdata(const float* __restrict__ tris9, int n, float4* __restrict__ hitdata) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = tris9 + (size_t)i * 9;
    const ex::V3 v0 = ex::v3(p[0], p[1], p[2]), v1 = ex::v3(p[3], p[4], p[5]), v2 = ex::v3(p[6], p[7], p[8]);
    const ex::V3 nrm = bvh::tri_normal(v0, v1, v2);
    hitdata[(size_t)i * 3 + 0] = make_float4(v0.x, v0.y, v0.z, nrm.x);
    hitdata[(size_t)i * 3 + 1] = make_float4(v1.x, v1.y, v1.z, nrm.y);
    hitdata[(size_t)i * 3 + 2] = make_float4(v2.x, v2.y, v2.z, nrm.z);
}

// ---- binned-SAH top-down builder (the default): one CTA per (node, range) task per level ----
__global__ void k_prim_boxes(const float* __restrict__ tris9, int n, const uint32_t* __restrict__ bounds, float4* __restrict__ pLo,
                             float4* __restrict__ pHi, uint32_t* __restrict__ idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bld::Box scene = load_scene_box(bounds);
    const float maxAbs = fmaxf(fmaxf(fmaxf(fabsf(scene.lox), fabsf(scene.hix)), fmaxf(fabsf(scene.loy), fabsf(scene.hiy))),
                               fmaxf(fabsf(scene.loz), fabsf(scene.hiz)));
    bld::Box b = bld::tri_box(tris9 + (size_t)i * 9);
    const float dx = b.hix - b.lox, dy = b.hiy - b.loy, dz = b.hiz - b.loz;
    const float pad = bld::pad_for(sqrtf(dx * dx + dy * dy + dz * dz), maxAbs);
    pLo[i] = make_float4(b.lox - pad, b.loy - pad, b.loz - pad, 0.0f);
    pHi[i] = make_float4(b.hix + pad, b.hiy + pad, b.hiz + pad, 0.0f);
    idx[i] = (uint32_t)i;
}

struct SahTask {
    int node, first, count, depth;
};
constexpr int SAH_THREADS = 256;

__device__ __forceinline__ void smem_box_grow(uint32_t* b6, float lox, float loy, float loz, float hix, float hiy, float hiz) {
    atomicMin(&b6[0], bld::float_to_ordered(lox)); atomicMin(&b6[1], bld::float_to_ordered(loy)); atomicMin(&b6[2], bld::float_to_ordered(loz));
    atomicMax(&b6[3], bld::float_to_ordered(hix)); atomicMax(&b6[4], bld::float_to_ordered(hiy)); atomicMax(&b6[5], bld::float_to_ordered(hiz));
}
__device__ __forceinline__ bld::Box smem_box_load(const uint32_t* b6) {
    return bld::Box{bld::ordered_to_float(b6[0]), bld::ordered_to_float(b6[1]), bld::ordered_to_float(b6[2]),
                    bld::ordered_to_float(b6[3]), bld::ordered_to_float(b6[4]), bld::ordered_to_float(b6[5])};
}

// One (node, range) task, by one CTA: node box, binning, plane choice, partition into the other index buffer.
__device__ __forceinline__ void sah_task(const SahTask tk, const bld::BinTree& t, const float4* __restrict__ pLo, const float4* __restrict__ pHi,
                                         const uint32_t* __restrict__ idxIn, uint32_t* __restrict__ idxOut, uint32_t* __restrict__ primFinal,
                                         SahTask* __restrict__ outQ, uint32_t* __restrict__ outCount, uint32_t* __restrict__ nodeCounter,
                                         const bld::SahParams& sp) {
    __shared__ uint32_t sNode[6], sCen[6];
    __shared__ uint32_t sBinBox[3][bld::SAH_BINS][6];
    __shared__ int sBinCnt[3][bld::SAH_BINS];
    __shared__ float sCost[3 * (bld::SAH_BINS - 1)];
    __shared__ int sLeft[3 * (bld::SAH_BINS - 1)];
    __shared__ bld::SahDecision sDec;
    __shared__ int sNl, sNr;
    const int tid = threadIdx.x;
    if (tid < 6) { sNode[tid] = tid < 3 ? 0xFFFFFFFFu : 0u; sCen[tid] = tid < 3 ? 0xFFFFFFFFu : 0u; }
    for (int k = tid; k < 3 * bld::SAH_BINS; k += SAH_THREADS) {
        uint32_t* b = &sBinBox[0][0][0] + k * 6;
        b[0] = b[1] = b[2] = 0xFFFFFFFFu; b[3] = b[4] = b[5] = 0u;
        (&sBinCnt[0][0])[k] = 0;
    }
    if (tid == 0) { sNl = 0; sNr = 0; }
    __syncthreads();
    // 1. node box and centroid box: per-thread, then per-warp, then one shared atomic per warp
    {
        bld::Box nb = bld::empty_box(), cb = bld::empty_box();
        for (int i = tid; i < tk.count; i += SAH_THREADS) {
            const uint32_t id = __ldcg(&idxIn[tk.first + i]);
            const float4 lo = pLo[id], hi = pHi[id];
            nb = bld::box_union(nb, bld::Box{lo.x, lo.y, lo.z, hi.x, hi.y, hi.z});
            const float cx = 0.5f * (lo.x + hi.x), cy = 0.5f * (lo.y + hi.y), cz = 0.5f * (lo.z + hi.z);
            cb = bld::box_union(cb, bld::Box{cx, cy, cz, cx, cy, cz});
        }
        for (int o = 16; o > 0; o >>= 1) {
            nb.lox = fminf(nb.lox, __shfl_xor_sync(0xffffffffu, nb.lox, o)); nb.loy = fminf(nb.loy, __shfl_xor_sync(0xffffffffu, nb.loy, o));
            nb.loz = fminf(nb.loz, __shfl_xor_sync(0xffffffffu, nb.loz, o)); nb.hix = fmaxf(nb.hix, __shfl_xor_sync(0xffffffffu, nb.hix, o));
            nb.hiy = fmaxf(nb.hiy, __shfl_xor_sync(0xffffffffu, nb.hiy, o)); nb.hiz = fmaxf(nb.hiz, __shfl_xor_sync(0xffffffffu, nb.hiz, o));
            cb.lox = fminf(cb.lox, __shfl_xor_sync(0xffffffffu, cb.lox, o)); cb.loy = fminf(cb.loy, __shfl_xor_sync(0xffffffffu, cb.loy, o));
            cb.loz = fminf(cb.loz, __shfl_xor_sync(0xffffffffu, cb.loz, o)); cb.hix = fmaxf(cb.hix, __shfl_xor_sync(0xffffffffu, cb.hix, o));
            cb.hiy = fmaxf(cb.hiy, __shfl_xor_sync(0xffffffffu, cb.hiy, o)); cb.hiz = fmaxf(cb.hiz, __shfl_xor_sync(0xffffffffu, cb.hiz, o));
        }
        if ((tid & 31) == 0) {
            smem_box_grow(sNode, nb.lox, nb.loy, nb.loz, nb.hix, nb.hiy, nb.hiz);
            smem_box_grow(sCen, cb.lox, cb.loy, cb.loz, cb.hix, cb.hiy, cb.hiz);
        }
    }
    __syncthreads();
    const bld::Box nodeBox = smem_box_load(sNode), cenBox = smem_box_load(sCen);
    const float cmin[3] = {cenBox.lox, cenBox.loy, cenBox.loz};
    const float ext[3] = {cenBox.hix - cenBox.lox, cenBox.hiy - cenBox.loy, cenBox.hiz - cenBox.loz};
    // 2. bin the primitives on all three axes
    if (tk.count > 1) {
        for (int i = tid; i < tk.count; i += SAH_THREADS) {
            const uint32_t id = __ldcg(&idxIn[tk.first + i]);
            const float4 lo = pLo[id], hi = pHi[id];
            const float c[3] = {0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z)};
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const int b = bld::sah_bin_of(c[a], cmin[a], ext[a]);
                smem_box_grow(sBinBox[a][b], lo.x, lo.y, lo.z, hi.x, hi.y, hi.z);
                atomicAdd(&sBinCnt[a][b], 1);
            }
        }
    }
    __syncthreads();
    // 3. evaluate the 3 x 15 candidate planes, decide
    if (tid < 3 * (bld::SAH_BINS - 1) && tk.count > 1) {
        const int a = tid / (bld::SAH_BINS - 1), sidx = tid % (bld::SAH_BINS - 1);
        bld::SahBin bins[bld::SAH_BINS];
        for (int b = 0; b < bld::SAH_BINS; ++b) { bins[b].box = smem_box_load(sBinBox[a][b]); bins[b].count = sBinCnt[a][b]; }
        int lc;
        sCost[tid] = bld::sah_split_cost(bins, sidx, &lc);
        sLeft[tid] = lc;
    }
    __syncthreads();
    if (tid == 0) {
        const bld::SahDecision d = tk.count == 1 ? bld::SahDecision{-1, 0, 0} : bld::sah_decide(sCost, sLeft, tk.count, bld::box_half_area(nodeBox), sp, tk.depth);
        sDec = d;
        t.lo[tk.node] = make_float4(nodeBox.lox, nodeBox.loy, nodeBox.loz, 0.0f);
        t.first[tk.node] = tk.first;
        if (d.axis < 0) {
            t.hi[tk.node] = make_float4(nodeBox.hix, nodeBox.hiy, nodeBox.hiz, ex::u2f((uint32_t)(-tk.count)));
        } else {
            t.hi[tk.node] = make_float4(nodeBox.hix, nodeBox.hiy, nodeBox.hiz, ex::u2f((uint32_t)tk.count));
            const int base = (int)atomicAdd(nodeCounter, 2u);
            t.left[tk.node] = base;
            t.right[tk.node] = base + 1;
            const uint32_t q = atomicAdd(outCount, 2u);
            outQ[q] = SahTask{base, tk.first, d.leftCount, tk.depth + 1};
            outQ[q + 1] = SahTask{base + 1, tk.first + d.leftCount, tk.count - d.leftCount, tk.depth + 1};
        }
    }
    __syncthreads();
    // 4. leaf: the range is final.  split: partition into the other index buffer.
    const bld::SahDecision d = sDec;
    for (int i = tid; i < tk.count; i += SAH_THREADS) {
        const uint32_t id = __ldcg(&idxIn[tk.first + i]);
        if (d.axis < 0) { primFinal[tk.first + i] = id; continue; }
        bool goLeft;
        if (d.axis == 3) goLeft = i < d.leftCount;
        else {
            const float4 lo = pLo[id], hi = pHi[id];
            const float c = d.axis == 0 ? 0.5f * (lo.x + hi.x) : d.axis == 1 ? 0.5f * (lo.y + hi.y) : 0.5f * (lo.z + hi.z);
            goLeft = bld::sah_bin_of(c, cmin[d.axis], ext[d.axis]) <= d.split;
        }
        if (goLeft) idxOut[tk.first + atomicAdd(&sNl, 1)] = id;
        else idxOut[tk.first + tk.count - 1 - atomicAdd(&sNr, 1)] = id;
    }
}

// one level per launch (the host reads the task count back between levels): the fallback form
__global__ void __launch_bounds__(SAH_THREADS) k_sah_level(bld::BinTree t, const float4* __restrict__ pLo, const float4* __restrict__ pHi,
                                                           const uint32_t* __restrict__ idxIn, uint32_t* __restrict__ idxOut,
                                                           uint32_t* __restrict__ primFinal, const SahTask* __restrict__ inQ,
                                                           SahTask* __restrict__ outQ, uint32_t* __restrict__ outCount,
                                                           uint32_t* __restrict__ nodeCounter, bld::SahParams sp) {
    sah_task(inQ[blockIdx.x], t, pLo, pHi, idxIn, idxOut, primFinal, outQ, outCount, nodeCounter, sp);
}

// The whole top-down build in ONE cooperative launch: resident CTAs loop over the tasks of a level, a grid-wide barrier
// separates the levels.  (With one launch per level the build of a 66 k-triangle scene spent 3.4 ms in kernels and
// 3-10 ms in ~30 host round trips.)  Three task counters rotate: level L reads counts[L % 3], appends to
// counts[(L+1) % 3] and clears counts[(L+2) % 3], so one barrier per level is enough.  The index and task buffers
// alternate with the level's parity exactly as in the host loop.
__global__ void __launch_bounds__(SAH_THREADS) k_sah_build(bld::BinTree t, const float4* __restrict__ pLo, const float4* __restrict__ pHi,
                                                           uint32_t* idxA, uint32_t* idxB, uint32_t* __restrict__ primFinal, SahTask* qA, SahTask* qB,
                                                           uint32_t* counts, uint32_t* __restrict__ nodeCounter, bld::SahParams sp, int maxLevels,
                                                           uint32_t* status) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    for (int level = 0;; ++level) {
        const uint32_t cnt = *(volatile uint32_t*)&counts[level % 3];
        if (cnt == 0) break;
        if (level >= maxLevels) {
            if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(status, 2u);  // did not terminate
            break;
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) counts[(level + 2) % 3] = 0u;
        const uint32_t* idxIn = (level & 1) ? idxB : idxA;
        uint32_t* idxOut = (level & 1) ? idxA : idxB;
        const SahTask* inQ = (level & 1) ? qB : qA;
        SahTask* outQ = (level & 1) ? qA : qB;
        for (uint32_t k = blockIdx.x; k < cnt; k += gridDim.x) {
            const SahTask tk{__ldcg(&inQ[k].node), __ldcg(&inQ[k].first), __ldcg(&inQ[k].count), __ldcg(&inQ[k].depth)};
            sah_task(tk, t, pLo, pHi, idxIn, idxOut, primFinal, outQ, &counts[(level + 1) % 3], nodeCounter, sp);
            __syncthreads();  // the task's shared arrays are reused by the next one
        }
        grid.sync();
    }
}

__global__ void k_collapse(bld::BinTree t, bld::WideOut w, const bld::WorkItem* __restrict__ inQueue, const uint32_t* __restrict__ inCount,
                           bld::WorkItem* __restrict__ outQueue, uint32_t* __restrict__ outCount) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= *inCount) return;
    bld::collapse_node(t, w, inQueue[i], outQueue, outCount);
}
// the collapse, level by level, in one cooperative launch (same counter rotation as k_sah_build)
__global__ void __launch_bounds__(128) k_collapse_all(bld::BinTree t, bld::WideOut w, bld::WorkItem* qA, bld::WorkItem* qB, uint32_t* counts) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nthreads = gridDim.x * blockDim.x;
    for (int level = 0;; ++level) {
        const uint32_t cnt = *(volatile uint32_t*)&counts[level % 3];
        if (cnt == 0) break;
        if (tid == 0) counts[(level + 2) % 3] = 0u;
        const bld::WorkItem* inQ = (level & 1) ? qB : qA;
        bld::WorkItem* outQ = (level & 1) ? qA : qB;
        for (uint32_t i = tid; i < cnt; i += nthreads) {
            const bld::WorkItem it{__ldcg(&inQ[i].bnode), __ldcg(&inQ[i].wide), __ldcg(&inQ[i].depth)};  // written by other SMs a level ago
            bld::collapse_node(t, w, it, outQ, &counts[(level + 1) % 3]);
        }
        grid.sync();
    }
}
// ---- refit (tmpt_scene_refit): bottom-up over the wide tree, one thread per node that has only leaf children; the last
// thread to arrive at a parent (atomic countdown of its inner children) carries on upwards ----
struct LoadNodeRowCg {  // a row of ANOTHER node, written by another thread of the refit: bypass the non-coherent L1
    const float4* nodes;
    __device__ float4 operator()(uint32_t n, int row) const { return __ldcg(nodes + (size_t)n * bvh::NODE_F4 + row); }
};
__global__ void k_refit_pending(const float4* __restrict__ nodes, uint32_t count, uint32_t* __restrict__ pending) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) pending[i] = (uint32_t)bld::wide_inner_children(nodes, i);
}
__global__ void k_refit_wide(float4* nodes, float4* tris, const float* __restrict__ tris9, const uint32_t* __restrict__ parent, uint32_t* pending,
                             uint32_t count, const uint32_t* __restrict__ bounds) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count || bld::wide_inner_children(nodes, i) != 0) return;
    const bld::Box scene = load_scene_box(bounds);
    const float maxAbs = fmaxf(fmaxf(fmaxf(fabsf(scene.lox), fabsf(scene.hix)), fmaxf(fabsf(scene.loy), fabsf(scene.hiy))),
                               fmaxf(fabsf(scene.loz), fabsf(scene.hiz)));
    uint32_t node = i;
    for (;;) {
        bld::refit_wide_node(nodes, tris, tris9, node, maxAbs, LoadNodeRowCg{nodes});
        if (node == 0) break;
        __threadfence();
        const uint32_t p = parent[node];
        if (atomicSub(&pending[p], 1u) != 1u) break;  // a sibling subtree is still on its way
        node = p;
    }
}
__global__ void k_quantize_nodes(const float4* __restrict__ nodesF, uint4* __restrict__ qnodes, uint32_t count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) bld::quantize_node(nodesF, qnodes, i);
}
__global__ void k_collapse_root_leaf(bld::BinTree t, bld::WideOut w, int rootNode) { bld::emit_single_leaf_root(t, w, rootNode); }

// ------------------------------------------------------------------------------------------
// K2/K3: batched HitScene
// ------------------------------------------------------------------------------------------
// stats[0] rays, [1] wide-node visits, [2] triangle tests, [3] hits, [4..9] lane / warp iteration counters (include/tmpt.h)
__device__ __forceinline__ void flush_stats(unsigned long long* stats, unsigned long long rays, const bvh::TravStats& ts, unsigned long long hits) {
    unsigned long long v[16] = {rays, ts.nodes, ts.tris, hits, ts.iters, ts.culledPops, ts.leafWaits, ts.nodeWarps, ts.triWarps, ts.warpIters,
                                ts.overflows, ts.depthOver[0], ts.depthOver[1], ts.depthOver[2], ts.depthOver[3], ts.depthOver[4]};
    for (int k = 0; k < 16; ++k) {
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
        if ((threadIdx.x & 31) == 0 && v[k]) atomicAdd(&stats[k], v[k]);
    }
}

template <int MODE, bool STATS>
__global__ void __launch_bounds__(128) k_hit_scene(bvh::SceneView sc, const float* __restrict__ rays6, long long nRays, float tMin, float tMax,
                                                    int* __restrict__ outID, float* __restrict__ outT, float* __restrict__ outPos,
                                                    float* __restrict__ outNormal, unsigned long long* __restrict__ stats) {
    bvh::TravStats ts;
    unsigned long long nr = 0, nh = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nRays; i += (long long)gridDim.x * blockDim.x) {
        const float* r = rays6 + i * 6;
        const ex::V3 o = ex::v3(r[0], r[1], r[2]), d = ex::v3(r[3], r[4], r[5]);
        bvh::HitRec h;
        if (MODE == TMPT_HIT_BRUTE) h = bvh::brute_force(sc, o, d, tMin, tMax);
        else if (MODE == TMPT_HIT_SUN) {  // the integrator's shadow query: the ray's own direction is NOT read, the sun's is used
            h.id = sc.sun.n > 0 && bvh::sun_query<STATS>(sc, o, tMin, tMax, &ts) ? 1 : -1;  // (no grid: an empty scene)
            h.t = 0.0f; h.u = 0.0f; h.v = 0.0f;
        } else if (MODE == TMPT_HIT_ANY) h = bvh::traverse<true, STATS>(sc, o, d, tMin, tMax, &ts);
        else h = bvh::traverse<false, STATS>(sc, o, d, tMin, tMax, &ts);
        if (STATS) { ++nr; nh += h.id >= 0; }
        if (MODE == TMPT_HIT_ANY || MODE == TMPT_HIT_SUN) { outID[i] = h.id < 0 ? -1 : 1; continue; }
        outID[i] = h.id;
        if (h.id >= 0) {
            if (outT) outT[i] = h.t;
            if (outPos || outNormal) {
                ex::V3 pos, nrm;
                bvh::hit_payload(sc, h.id, h.u, h.v, pos, nrm);
                if (outPos) { outPos[i * 3] = pos.x; outPos[i * 3 + 1] = pos.y; outPos[i * 3 + 2] = pos.z; }
                if (outNormal) { outNormal[i * 3] = nrm.x; outNormal[i * 3 + 1] = nrm.y; outNormal[i * 3 + 2] = nrm.z; }
            }
        }
    }
    if (STATS) flush_stats(stats, nr, ts, nh);
}


#if TMPT_EXPERIMENTS
// K2/K3 with per-lane ray REFILL (experiment: -DTMPT_EXPERIMENTS=1 and TMPT_HIT_REFILL=gate; measured in round 2: 5244 -> 4843 Mrays/s
// at the best gate, profiles/r2_tuning_sweeps.txt): a lane whose ray has ended takes the next ray of the batch instead of
// waiting for the warp's longest ray; the fetch code runs when at least GATE lanes are idle (or nothing else is left to do).
template <int MODE, int GATE>
__global__ void __launch_bounds__(128) k_hit_scene_refill(bvh::SceneView sc, const float* __restrict__ rays6, long long nRays, float tMin, float tMax,
                                                           int* __restrict__ outID, float* __restrict__ outT, float* __restrict__ outPos,
                                                           float* __restrict__ outNormal, unsigned long long* __restrict__ counter) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    bvh::LocalStack stack;
    bvh::WalkState w;
    long long ray = -1;
    bool exhausted = false;
    for (;;) {
        const unsigned idle = __ballot_sync(FULL, ray < 0);
        if (idle && !exhausted && (__popc(idle) >= GATE || idle == FULL)) {
            const int cnt = __popc(idle);
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(counter, (unsigned long long)cnt);
            base = __shfl_sync(FULL, base, 0);
            exhausted = base + (unsigned long long)cnt >= (unsigned long long)nRays;
            if (ray < 0) {
                const long long i = (long long)base + __popc(idle & ((1u << lane) - 1u));
                if (i < nRays) {
                    const float* r = rays6 + i * 6;
                    bvh::walk_start(w, sc, ex::v3(r[0], r[1], r[2]), ex::v3(r[3], r[4], r[5]), tMax, MODE == TMPT_HIT_ANY);
                    ray = i;
                }
            }
        }
        if (__all_sync(FULL, ray < 0)) break;
        if (ray >= 0 && bvh::walk_step<false>(w, sc, tMin, tMax, stack, nullptr)) {
            const bvh::HitRec h = w.best;
            if (MODE == TMPT_HIT_ANY) outID[ray] = h.id < 0 ? -1 : 1;
            else {
                outID[ray] = h.id;
                if (h.id >= 0) {
                    if (outT) outT[ray] = h.t;
                    if (outPos || outNormal) {
                        ex::V3 pos, nrm;
                        bvh::hit_payload(sc, h.id, h.u, h.v, pos, nrm);
                        if (outPos) { outPos[ray * 3] = pos.x; outPos[ray * 3 + 1] = pos.y; outPos[ray * 3 + 2] = pos.z; }
                        if (outNormal) { outNormal[ray * 3] = nrm.x; outNormal[ray * 3 + 1] = nrm.y; outNormal[ray * 3 + 2] = nrm.z; }
                    }
                }
            }
            ray = -1;
        }
    }
}
#endif  // TMPT_EXPERIMENTS

// ------------------------------------------------------------------------------------------
// K4: path tracing.  Work unit = (8x4 pixel tile, one chunk of chunk_len(spp) samples) per warp, fetched from a
// global counter (persistent CTAs); a lane runs the samples of its pixel's chunk serially
// because the chunk's XorShift32 stream flows through them (DESIGN.md "RNG").  With more than
// one chunk per pixel the chunk sums go to an accumulation buffer and k_resolve adds them in
// chunk order; this keeps ~10x more work items than resident lanes even when a 1080p frame is
// split over 8 GPUs.
// ------------------------------------------------------------------------------------------
struct RenderParams {
    bvh::SceneView sc;
    integ::Camera cam;
    ex::V3 lightDir;
    int width, height, spp;
    int stripeRows, rank, world, ownedRows;  // stripeRows == 0: tile-interleaved partition (see local_to_global)
    int localWidth;      // width of this rank's LOCAL image: the frame's width (row stripes) or its share of every row (tile interleave)
    int tilesX, numTiles;
    int chunks;          // sample chunks per pixel rendered by this launch
    int chunk0, chunkLen; // first chunk index (progressive passes continue where the last one stopped), samples per chunk
    int useAccum;        // chunk sums go through `accum` + k_resolve (more than one chunk, a progressive pass, or float outputs)
    float4* sumBuf;      // progressive: running per-pixel sums of the whole frame (null for a one-shot frame)
    int bandRow0, bandRows;  // first owned row and row count of the band being rendered (the accumulation buffer covers one band)
    float4* accum;       // [chunks][bandRows][width] chunk sums (chunk-major planes: full-line stores, no read-modify-write in HBM); AOV
                         // kernels: .w = the chunk's camera-ray hits, followed by [chunks][bandRows][width] (normal sum, t sum)
    uchar4* outStripes;  // packed owned rows, or
    uchar4* frame;       // full frame (possibly peer memory)
    float4* radiance;    // tmpt_outputs' float buffers (full frame, device memory; null = not produced): written by k_resolve
    float4* normal;
    float* depth;
    int32_t* triangle;   // stored by the lane that traces chunk 0 of the pixel (AOV kernels)
    unsigned long long* rayCount;
    uint32_t* tileCounter;
    unsigned long long* laneCounter;  // k_render_regen: next lane item
    unsigned long long* stats;  // instrumented pass only
    const uint2* list;   // LIST kernels (adaptive passes): the band's entries of the active list, {x | y << 16, first chunk n_i}
    int listLen;         // entries in the band; accum = [chunks][listLen]
};

__device__ __forceinline__ int owned_row_to_global(int r, int stripeRows, int rank, int world) {
    const int ls = r / stripeRows;
    return (ls * world + rank) * stripeRows + (r - ls * stripeRows);
}
// The two partitions of a frame over `world` ranks, both as a map from a rank's LOCAL image (ownedRows x localWidth, the
// layout of its accumulation planes and of its packed output) to frame pixels:
//   row stripes (stripeRows > 0): stripe k = rows [k * stripeRows, (k+1) * stripeRows) belongs to rank k % world; a local row
//     is an owned row, local x = x.
//   tile interleave (stripeRows == 0): the 8x4-pixel tile (tx, ty) belongs to rank (tx + ty) % world -- every rank owns every
//     world-th tile of every tile row, shifted by one from row to row, i.e. exactly 1/world of the tiles, spread evenly over
//     the frame: the partition is balanced in tile COUNT whatever the frame height (row stripes of four rows give two of
//     eight ranks 33 instead of 34 stripes of a 1080-row frame) and in COST, because every rank samples the whole frame.
//     Local row = frame row; local tile ltx of tile row ty is frame tile ((rank - ty) mod world) + ltx * world.
// Returns false for local pixels that fall outside the frame (the last local tile of a row, when tilesX % world != 0).
__device__ __forceinline__ bool local_to_global(int xl, int r, int stripeRows, int rank, int world, int width, int& x, int& y) {
    if (stripeRows > 0) {
        x = xl;
        y = owned_row_to_global(r, stripeRows, rank, world);
        return true;
    }
    y = r;
    int t0 = (rank - (r >> 2)) % world;
    t0 += t0 < 0 ? world : 0;
    x = ((t0 + (xl >> 3) * world) << 3) + (xl & 7);
    return x < width;
}

// SSTACK = traversal-stack entries per lane kept in shared memory (0: the whole stack is a local-memory array); the launch
// passes SSTACK * THREADS * 8 bytes of dynamic shared memory.
template <int SSTACK, int THREADS>
struct RenderStack {
    using type = bvh::SmemStack<SSTACK, THREADS>;
    static __device__ __forceinline__ type make() {
        extern __shared__ unsigned long long smemStack[];
        return type::make(smemStack, threadIdx.x);
    }
};
template <int THREADS>
struct RenderStack<0, THREADS> {
    using type = bvh::LocalStack;
    static __device__ __forceinline__ type make() { return type(); }
};

#ifndef TMPT_SSTACK
#define TMPT_SSTACK 0
#endif
#ifndef TMPT_TUNE_CFG
#define TMPT_TUNE_CFG 0
#endif
constexpr int kSStack = TMPT_SSTACK;

// What a render launch writes (one mode per instantiation of k_render and k_render_paths):
//   Frame: the RGBA frame, or chunk sums for k_resolve (and the radiance it writes);
//   Aov:   the frame has AOV outputs (tmpt_outputs normal / depth / triangle): the same paths, plus each sample's camera-ray hit;
//   List:  an adaptive pass: work item (list tile t, k) is entry list[t * 32 + lane] of the band, its chunk n_i + k of 8 samples.
enum class OutMode { Frame, Aov, List };

// FAR = the camera stands beyond the scene's far limit (bvh.cuh: ray_is_far): rays are checked and, if far, answered by the
// exact all-triangle scan.  Only the 256-thread configuration has that instantiation (a camera sixteen scene sizes away sees
// a few pixels of scene).
template <bool STATS, int THREADS, int MINB, int SSTACK, bool FAR = false, OutMode MODE = OutMode::Frame>
__global__ void __launch_bounds__(THREADS, MINB) k_render(const RenderParams p) {
    constexpr bool AOV = MODE == OutMode::Aov, LIST = MODE == OutMode::List;
    const int lane = threadIdx.x & 31;
    unsigned long long rays = 0;
    bvh::TravStats ts;
    typename RenderStack<SSTACK, THREADS>::type stack = RenderStack<SSTACK, THREADS>::make();
    for (;;) {
        uint32_t tile = 0;
        if (lane == 0) tile = atomicAdd(p.tileCounter, 1u);
        tile = __shfl_sync(0xffffffffu, tile, 0);
        if (tile >= (uint32_t)p.numTiles * (uint32_t)p.chunks) break;
        const int chunk = (int)(tile / (uint32_t)p.numTiles);
        tile -= (uint32_t)chunk * (uint32_t)p.numTiles;
        if (LIST) {
            const uint32_t e = tile * 32u + (uint32_t)lane;
            if (e < (uint32_t)p.listLen) {
                const uint2 en = p.list[e];
                const ex::V3 sum = integ::render_chunk<STATS, FAR>(stack, p.sc, p.cam, (int)(en.x & 0xFFFFu), (int)(en.x >> 16), (int)en.y + chunk, p.width,
                                                                   p.height, 0x7FFFFFFF, integ::kMaxChunkSamples, p.lightDir, rays, &ts);
                __stcs(&p.accum[(size_t)chunk * p.listLen + e], make_float4(sum.x, sum.y, sum.z, 0.0f));
            }
            continue;
        }
        const int tx = (int)(tile % (uint32_t)p.tilesX), ty = (int)(tile / (uint32_t)p.tilesX);
        const int xl = tx * 8 + (lane & 7), rb = ty * 4 + (lane >> 3), r = p.bandRow0 + rb;
        int x, y;
        if (xl < p.localWidth && r < p.ownedRows && local_to_global(xl, r, p.stripeRows, p.rank, p.world, p.width, x, y)) {
            integ::AovSums aov;
            const ex::V3 sum = integ::render_chunk<STATS, FAR, AOV>(stack, p.sc, p.cam, x, y, p.chunk0 + chunk, p.width, p.height, p.spp, p.chunkLen, p.lightDir, rays, &ts, &aov);
            if (AOV && p.triangle && p.chunk0 + chunk == 0) p.triangle[(size_t)y * p.width + x] = aov.id0;
            if (p.useAccum) {
                const size_t a = ((size_t)chunk * p.bandRows + rb) * p.localWidth + xl;
                __stcs(&p.accum[a], make_float4(sum.x, sum.y, sum.z, AOV ? aov.hits : 0.0f));  // streaming: read once, by k_resolve
                if (AOV) __stcs(&p.accum[a + (size_t)p.chunks * p.bandRows * p.localWidth], make_float4(aov.normal.x, aov.normal.y, aov.normal.z, aov.t));
            } else {
                const uchar4 px = integ::resolve_pixel(sum, ex::divf(1.0f, (float)p.spp));
                if (p.frame) p.frame[(size_t)y * p.width + x] = px;
                else p.outStripes[(size_t)r * p.localWidth + xl] = px;
            }
        }
    }
    if (STATS) flush_stats(p.stats, rays, ts, 0);
    for (int o = 16; o > 0; o >>= 1) rays += __shfl_xor_sync(0xffffffffu, rays, o);
    if (lane == 0 && rays) atomicAdd(p.rayCount, rays);
}

#if TMPT_EXPERIMENTS
// K4': the same frame with per-lane RAY REGENERATION.  In k_render a warp's lanes trace their rays in lockstep: a lane whose
// ray ends early idles until the warp's longest ray is done (about half of all lane slots of the walk).  Here every lane
// is a small state machine over its own path -- closest-hit walk -> shade -> shadow walk -> next bounce ... -> next sample
// -> next work item -- and the warp's loop body is ONE walk step for whichever ray each lane currently has.  The
// transitions between rays (payload + scatter, unwind + next camera ray, work fetch) are divergent by nature, so they are
// GATED: lanes that finished a ray wait until TA of them (TB for the rarer end-of-path work) can make the transition
// together, or until nobody in the warp is walking.  The per-lane arithmetic and its order are those of
// integ::render_chunk, so the frame is byte-identical to k_render's (tests/test_gpu_parity.py).
// Work item = one (pixel, chunk) per LANE from a global counter; consecutive items are the pixels of one 8x4 tile.
enum : int { ST_WALK = 0, ST_HIT = 1, ST_SHADOW_DONE = 2, ST_PATH_END = 3, ST_NEED_ITEM = 4, ST_IDLE = 5 };

template <bool STATS, int THREADS, int MINB, int TA, int TB>
__global__ void __launch_bounds__(THREADS, MINB) k_render_regen(const RenderParams p) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    bvh::LocalStack stack;
    float kk[integ::kMaxDepth];
    bvh::WalkState w;
    bvh::TravStats ts;
    w.any = false; w.best.id = -1;
    unsigned long long rays = 0;
    int state = ST_NEED_ITEM;
    bool exhausted = false;
    uint32_t rng = 0;
    int depth = 0, s = 0, sEnd = 0, x = 0, y = 0, xl = 0, rb = 0, chunk = 0;
    ex::V3 sum = ex::v3(0.0f, 0.0f, 0.0f), nd = ex::v3(0.0f, 0.0f, 0.0f);
    float sunk = 0.0f;
    const float invW = ex::divf(1.0f, (float)p.width), invH = ex::divf(1.0f, (float)p.height);
    const unsigned long long totalItems = (unsigned long long)p.numTiles * (unsigned long long)p.chunks * 32ull;
    for (;;) {
        const unsigned notWalking = __ballot_sync(FULL, state != ST_WALK);
        if (notWalking) {
            bool newRay = false, newAny = false;
            ex::V3 no = ex::v3(0.0f, 0.0f, 0.0f), ndir = no;
            // ---- A: a closest-hit walk found a hit (payload, sun term, scatter, shadow ray) or a shadow walk ended (next bounce)
            const unsigned adv = __ballot_sync(FULL, state == ST_HIT || state == ST_SHADOW_DONE);
            if (adv && (__popc(adv) >= TA || notWalking == FULL)) {
                if (state == ST_HIT) {
                    ex::V3 pos, normal;
                    bvh::hit_payload(p.sc, w.best.id, w.best.u, w.best.v, pos, normal);
                    sunk = integ::sun_term(normal, w.d, p.lightDir);
                    nd = integ::scatter_dir(pos, normal, rng);  // drawn before the shadow walk: that walk draws nothing
                    no = pos; ndir = p.lightDir; newRay = true; newAny = true;
                } else if (state == ST_SHADOW_DONE) {
                    kk[depth] = w.best.id < 0 ? sunk : 0.0f;
                    ++depth;
                    if (depth < integ::kMaxDepth) { no = w.o; ndir = nd; newRay = true; newAny = false; }
                    else state = ST_PATH_END;  // w.any stays true: "ended by depth", colour starts at 0
                }
            }
            // ---- B: end of a path (unwind, add the sample), next camera ray or next work item
            const unsigned endp = __ballot_sync(FULL, state == ST_PATH_END || state == ST_NEED_ITEM);
            const unsigned busy = __ballot_sync(FULL, state == ST_WALK || newRay);
            if (endp && (__popc(endp) >= TB || busy == 0)) {
                if (state == ST_PATH_END) {
                    ex::V3 color = w.any ? ex::v3(0.0f, 0.0f, 0.0f) : integ::sky(w.d);
                    for (int i = depth - 1; i >= 0; --i) color = integ::unwind_step(kk[i], color);
                    sum = ex::add(sum, color);
                    if (++s == sEnd) {
                        if (p.useAccum) {
                            __stcs(&p.accum[((size_t)chunk * p.bandRows + rb) * p.localWidth + xl], make_float4(sum.x, sum.y, sum.z, 0.0f));  // streaming: read once, by k_resolve
                        } else {
                            const uchar4 px = integ::resolve_pixel(sum, ex::divf(1.0f, (float)p.spp));
                            if (p.frame) p.frame[(size_t)y * p.width + x] = px;
                            else p.outStripes[(size_t)(p.bandRow0 + rb) * p.localWidth + xl] = px;
                        }
                        state = ST_NEED_ITEM;
                    }
                }
                const unsigned want = __ballot_sync(FULL, state == ST_NEED_ITEM);
                if (want) {
                    if (exhausted) {
                        if (state == ST_NEED_ITEM) state = ST_IDLE;
                    } else {
                        const int cnt = __popc(want);
                        unsigned long long base = 0;
                        if (lane == 0) base = atomicAdd(p.laneCounter, (unsigned long long)cnt);
                        base = __shfl_sync(FULL, base, 0);
                        exhausted = base + (unsigned long long)cnt >= totalItems;
                        if (state == ST_NEED_ITEM) {
                            const unsigned long long item = base + (unsigned long long)__popc(want & ((1u << lane) - 1u));
                            if (item >= totalItems) {
                                state = ST_IDLE;
                            } else {
                                const uint32_t wi = (uint32_t)(item >> 5), li = (uint32_t)item & 31u;
                                chunk = (int)(wi / (uint32_t)p.numTiles);
                                const uint32_t tile = wi - (uint32_t)chunk * (uint32_t)p.numTiles;
                                const int tx = (int)(tile % (uint32_t)p.tilesX), ty = (int)(tile / (uint32_t)p.tilesX);
                                xl = tx * 8 + (int)(li & 7u); rb = ty * 4 + (int)(li >> 3);
                                const int r = p.bandRow0 + rb;
                                if (xl < p.localWidth && r < p.ownedRows && local_to_global(xl, r, p.stripeRows, p.rank, p.world, p.width, x, y)) {  // (an item outside the frame is simply dropped: the lane asks again)
                                    const int gchunk = p.chunk0 + chunk;  // progressive passes continue the chunk numbering; `chunk` stays the accum plane
                                    rng = ex::chunk_seed((uint32_t)gchunk, (uint32_t)y * (uint32_t)p.width + (uint32_t)x, (uint32_t)p.width * (uint32_t)p.height);
                                    const int len = p.chunkLen;
                                    s = gchunk * len;
                                    sEnd = s + len < p.spp ? s + len : p.spp;
                                    sum = ex::v3(0.0f, 0.0f, 0.0f);
                                    state = ST_PATH_END;  // marks "has an item, needs a camera ray" for the block below
                                    depth = -1;
                                }
                            }
                        }
                    }
                }
                if (state == ST_PATH_END) {  // next sample of the item
                    integ::primary_ray(p.cam, x, y, invW, invH, rng, no, ndir);
                    depth = 0; newRay = true; newAny = false;
                }
            }
            if (newRay) {
                ++rays;
                bvh::walk_start(w, p.sc, no, ndir, integ::kMaxT, newAny);
                state = ST_WALK;
            }
            if (__all_sync(FULL, state == ST_IDLE)) break;
        }
        if (state == ST_WALK) {
            if (bvh::walk_step<STATS>(w, p.sc, integ::kMinT, integ::kMaxT, stack, &ts))
                state = w.any ? ST_SHADOW_DONE : w.best.id < 0 ? ST_PATH_END : ST_HIT;
        }
    }
    if (STATS) flush_stats(p.stats, rays, ts, 0);
    for (int o = 16; o > 0; o >>= 1) rays += __shfl_xor_sync(FULL, rays, o);
    if (lane == 0 && rays) atomicAdd(p.rayCount, rays);
}

#endif  // TMPT_EXPERIMENTS

// K4'': PATH-level regeneration.  k_render's lanes trace the samples of one tile in lockstep: when a lane's path leaves the scene
// early (sky), the lane idles until the longest path of the warp has used up its ten bounces -- nothing in the closed Sponza hall,
// most of the lane slots in open scenes (cube, suzanne, teapot: 2.6 rays per camera sample).  Here a lane whose path has ended takes
// the next sample of its item, or the next (pixel, chunk) item from a global counter (warp-aggregated: ballot / popc / shfl), at the
// next BOUNCE BOUNDARY, where the warp is synchronous anyway: the traversals themselves stay lockstep (per-ray regeneration inside a
// traversal was measured twice and loses, DESIGN.md 5), the regeneration code runs when at least GATE lanes need it or nobody is
// tracing.  Work item = one (pixel, chunk) per lane; consecutive items are the pixels of one 8x4 tile, so a warp starts with a
// whole tile.  The per-lane arithmetic and its order are those of integ::render_chunk: the frame is byte-identical to k_render's.
// AOV (as in k_render): the camera ray's hit of each sample is added to nsum / tsum and counted in cl's top byte.
// LIST (as in k_render): item (list tile t, k, lane) is entry list[t * 32 + lane], chunk n_i + k; loc holds the entry index.
template <int THREADS, int MINB, int GATE, OutMode MODE = OutMode::Frame>
__global__ void __launch_bounds__(THREADS, MINB) k_render_paths(const RenderParams p) {
    constexpr bool AOV = MODE == OutMode::Aov, LIST = MODE == OutMode::List;
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    bvh::LocalStack stack;
    float kk[integ::kMaxDepth];
    unsigned long long rays = 0;
    bool havePath = false, done = false, exhausted = false;
    // a lane's item, packed (the kernel lives at 64 registers): pixel x | y << 16 (both < 10000), packed position xl | rb << 16,
    // chunk << 8 | samples left in the chunk (<= integ::kMaxChunkSamples); hasItem = the lane owes a store when `left` reaches 0.
    // AOV: camera-ray hits of the item so far << 24 (chunk < 2^16)
    uint32_t rng = 0, pix = 0, loc = 0, cl = 0;
    bool hasItem = false;
    int depth = 0;
    ex::V3 sum = ex::v3(0.0f, 0.0f, 0.0f), o = sum, d = sum, nsum = sum;
    float tsum = 0.0f;
    const float invW = ex::divf(1.0f, (float)p.width), invH = ex::divf(1.0f, (float)p.height);
    const unsigned long long totalItems = (unsigned long long)p.numTiles * (unsigned long long)p.chunks * 32ull;
    for (;;) {
        // ---- regeneration: lanes without a path get their item's next sample, or a new item
        const unsigned need = __ballot_sync(FULL, !havePath && !done);
        const unsigned tracing = __ballot_sync(FULL, havePath);
        if (need && (__popc(need) >= GATE || tracing == 0)) {
            // (a) items that are finished: store the chunk sum, ask for a new item
            bool wantItem = !havePath && !done && (cl & 0xFFu) == 0u;
            if (wantItem && hasItem) {
                const int xl = (int)(loc & 0xFFFFu), rb = (int)(loc >> 16);
                if (LIST) {
                    __stcs(&p.accum[(size_t)(cl >> 8) * p.listLen + loc], make_float4(sum.x, sum.y, sum.z, 0.0f));
                } else if (p.useAccum) {
                    const size_t a = ((size_t)(AOV ? (cl >> 8) & 0xFFFFu : cl >> 8) * p.bandRows + rb) * p.localWidth + xl;
                    __stcs(&p.accum[a], make_float4(sum.x, sum.y, sum.z, AOV ? (float)(cl >> 24) : 0.0f));
                    if (AOV) __stcs(&p.accum[a + (size_t)p.chunks * p.bandRows * p.localWidth], make_float4(nsum.x, nsum.y, nsum.z, tsum));
                } else {
                    const uchar4 px = integ::resolve_pixel(sum, ex::divf(1.0f, (float)p.spp));
                    if (p.frame) p.frame[(size_t)(pix >> 16) * p.width + (pix & 0xFFFFu)] = px;
                    else p.outStripes[(size_t)(p.bandRow0 + rb) * p.localWidth + xl] = px;
                }
                hasItem = false;
            }
            while (__any_sync(FULL, wantItem)) {  // (a lane whose item fell outside the frame asks again)
                const unsigned want = __ballot_sync(FULL, wantItem);
                if (exhausted) { if (wantItem) { done = true; wantItem = false; } break; }
                const int cnt = __popc(want);
                unsigned long long base = 0;
                if (lane == __ffs((int)want) - 1) base = atomicAdd(p.laneCounter, (unsigned long long)cnt);
                base = __shfl_sync(FULL, base, __ffs((int)want) - 1);
                exhausted = base + (unsigned long long)cnt >= totalItems;
                if (wantItem) {
                    const unsigned long long item = base + (unsigned long long)__popc(want & ((1u << lane) - 1u));
                    if (item >= totalItems) { done = true; wantItem = false; }
                    else {
                        const uint32_t wi = (uint32_t)(item >> 5), li = (uint32_t)item & 31u;
                        const int chunk = (int)(wi / (uint32_t)p.numTiles);
                        const uint32_t tile = wi - (uint32_t)chunk * (uint32_t)p.numTiles;
                        if (LIST) {
                            const uint32_t e = tile * 32u + li;
                            if (e < (uint32_t)p.listLen) {
                                const uint2 en = p.list[e];
                                rng = ex::chunk_seed(en.y + (uint32_t)chunk, (en.x >> 16) * (uint32_t)p.width + (en.x & 0xFFFFu),
                                                     (uint32_t)p.width * (uint32_t)p.height);
                                pix = en.x;
                                loc = e;
                                cl = ((uint32_t)chunk << 8) | (uint32_t)integ::kMaxChunkSamples;
                                sum = ex::v3(0.0f, 0.0f, 0.0f);
                                hasItem = true;
                                wantItem = false;
                            }
                            continue;
                        }
                        const int tx = (int)(tile % (uint32_t)p.tilesX), ty = (int)(tile / (uint32_t)p.tilesX);
                        const int xl = tx * 8 + (int)(li & 7u), rb = ty * 4 + (int)(li >> 3);
                        const int r = p.bandRow0 + rb;
                        int x, y;
                        if (xl < p.localWidth && r < p.ownedRows && local_to_global(xl, r, p.stripeRows, p.rank, p.world, p.width, x, y)) {
                            const int gchunk = p.chunk0 + chunk;
                            rng = ex::chunk_seed((uint32_t)gchunk, (uint32_t)y * (uint32_t)p.width + (uint32_t)x, (uint32_t)p.width * (uint32_t)p.height);
                            const int s0 = gchunk * p.chunkLen;
                            const int left = (s0 + p.chunkLen < p.spp ? s0 + p.chunkLen : p.spp) - s0;
                            pix = (uint32_t)x | ((uint32_t)y << 16);
                            loc = (uint32_t)xl | ((uint32_t)rb << 16);
                            cl = ((uint32_t)chunk << 8) | (uint32_t)left;
                            sum = ex::v3(0.0f, 0.0f, 0.0f);
                            if (AOV) { nsum = sum; tsum = 0.0f; }
                            hasItem = true;
                            wantItem = false;
                        }
                    }
                }
            }
            // (b) the next camera ray of every lane that has an item and no path
            if (!havePath && !done && (cl & 0xFFu) != 0u) {
                integ::primary_ray(p.cam, (int)(pix & 0xFFFFu), (int)(pix >> 16), invW, invH, rng, o, d);
                depth = 0;
                havePath = true;
            }
        }
        if (__all_sync(FULL, done)) break;
        // ---- one bounce of every lane that has a path (lockstep traversals)
        bool hit = false;
        bvh::HitRec h;
        h.id = -1;
        if (havePath) {
            ++rays;
            h = bvh::traverse_with<false, false, false>(stack, p.sc, o, d, integ::kMinT, integ::kMaxT);
            hit = h.id >= 0;
        }
        ex::V3 pos = ex::v3(0.0f, 0.0f, 0.0f), normal = pos;
        bool shadowed = false;
        if (hit) {
            bvh::hit_payload(p.sc, h.id, h.u, h.v, pos, normal);
            ++rays;
            shadowed = p.sc.sun.n > 0 ? bvh::sun_occluded<false>(p.sc, pos, p.lightDir, integ::kMinT, integ::kMaxT, nullptr)
                                      : bvh::traverse_with<true, false, false>(stack, p.sc, pos, p.lightDir, integ::kMinT, integ::kMaxT).id >= 0;
        }
        if (havePath) {
            bool ended = false;
            ex::V3 color = ex::v3(0.0f, 0.0f, 0.0f);
            if (AOV && depth == 0) {  // the sample's camera ray (integ::render_chunk's AovSums, in the same order)
                if (p.triangle && p.chunk0 == 0 && cl == (uint32_t)min(p.chunkLen, p.spp))  // chunk 0's first sample
                    p.triangle[(size_t)(pix >> 16) * p.width + (pix & 0xFFFFu)] = h.id;
                if (hit) { nsum = ex::add(nsum, normal); tsum = ex::add(tsum, h.t); cl += 1u << 24; }
            }
            if (hit) {
                kk[depth] = shadowed ? 0.0f : integ::sun_term(normal, d, p.lightDir);
                d = integ::scatter_dir(pos, normal, rng);
                o = pos;
                ++depth;
                ended = depth == integ::kMaxDepth;  // out of bounces: the path's colour starts at 0 (main.cpp:84, 112-116)
            } else {
                color = integ::sky(d);
                ended = true;
            }
            if (ended) {
                for (int i = depth - 1; i >= 0; --i) color = integ::unwind_step(kk[i], color);
                sum = ex::add(sum, color);
                --cl;  // one sample less to go (low byte)
                havePath = false;
            }
        }
    }
    for (int k = 16; k > 0; k >>= 1) rays += __shfl_xor_sync(FULL, rays, k);
    if (lane == 0 && rays) atomicAdd(p.rayCount, rays);
}

// ---- K7: the sun grid (sungrid.cuh), built on the device after the tree ---------------------------------------------------------
// One WARP per triangle slot walks the cells of the triangle's padded bounding box (lanes stride over them) and, where the
// projection touches the cell, counts (FILL = false) or writes (FILL = true) an entry.  A triangle whose box spans more than
// kSunBigCells cells (the floor's two triangles cover every cell) is put on a list instead and binned by the whole grid of
// k_sun_bin_big: one warp walking a million cells, an atomic's round trip per step, took 25 ms.
constexpr long long kSunBigCells = 2048;
__device__ __forceinline__ void sun_bin_cell(const sun::View& g, const sun::Tri2& t, int slot, int cx, int cy, bool fill, uint32_t* cellCount,
                                             const uint32_t* cellStart, uint2* entries) {
    if (!sun::touches_cell(g, t, cx, cy)) return;
    const uint32_t c = (uint32_t)cy * (uint32_t)g.n + (uint32_t)cx;
    const uint32_t k = atomicAdd(&cellCount[c], 1u);
    if (fill) entries[cellStart[c] + k] = make_uint2((uint32_t)slot, ex::f2u(sun::far_depth(g, t, cx, cy)));
}
template <bool FILL>
__global__ void __launch_bounds__(256) k_sun_bin(sun::View g, const float4* __restrict__ tris, const float* __restrict__ tris9, int nSlots,
                                                 uint32_t* __restrict__ cellCount, const uint32_t* __restrict__ cellStart, uint2* __restrict__ entries,
                                                 uint32_t* __restrict__ bigList, uint32_t* __restrict__ bigCount) {
    const int slot = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (slot >= nSlots) return;
    const int id = (int)ex::f2u(__ldg(&tris[(size_t)slot * 3]).w);
    const sun::Tri2 t = sun::project_tri(g, tris9 + (size_t)id * 9);
    int x0, x1, y0, y1;
    sun::cell_range(g, t, x0, x1, y0, y1);
    const int wx = x1 - x0 + 1;
    const long long cells = (long long)wx * (y1 - y0 + 1);
    if (cells > kSunBigCells) {
        if (!FILL && lane == 0) bigList[atomicAdd(bigCount, 1u)] = (uint32_t)slot;  // (the fill pass reads the list the count pass made)
        return;
    }
    for (long long i = lane; i < cells; i += 32) sun_bin_cell(g, t, slot, x0 + (int)(i % wx), y0 + (int)(i / wx), FILL, cellCount, cellStart, entries);
}
template <bool FILL>
__global__ void __launch_bounds__(256) k_sun_bin_big(sun::View g, const float4* __restrict__ tris, const float* __restrict__ tris9,
                                                     uint32_t* __restrict__ cellCount, const uint32_t* __restrict__ cellStart, uint2* __restrict__ entries,
                                                     const uint32_t* __restrict__ bigList, const uint32_t* __restrict__ bigCount) {
    const uint32_t nBig = *bigCount;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    for (uint32_t j = 0; j < nBig; ++j) {
        const int slot = (int)bigList[j];
        const int id = (int)ex::f2u(__ldg(&tris[(size_t)slot * 3]).w);
        const sun::Tri2 t = sun::project_tri(g, tris9 + (size_t)id * 9);
        int x0, x1, y0, y1;
        sun::cell_range(g, t, x0, x1, y0, y1);
        const int wx = x1 - x0 + 1;
        const long long cells = (long long)wx * (y1 - y0 + 1);
        for (long long i = tid; i < cells; i += stride) sun_bin_cell(g, t, slot, x0 + (int)(i % wx), y0 + (int)(i / wx), FILL, cellCount, cellStart, entries);
    }
}

// exclusive scan of the cell counts, three small kernels: per-block totals, scan of the totals (one block), per-block scan + offset
constexpr int kScanBlock = 1024;
__global__ void __launch_bounds__(kScanBlock) k_scan_totals(const uint32_t* __restrict__ in, long long n, uint32_t* __restrict__ totals) {
    __shared__ uint32_t sh[kScanBlock / 32];
    const long long i = (long long)blockIdx.x * kScanBlock + threadIdx.x;
    uint32_t v = i < n ? in[i] : 0u;
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t w = sh[threadIdx.x];
        for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
        if (threadIdx.x == 0) totals[blockIdx.x] = w;
    }
}
__global__ void __launch_bounds__(kScanBlock) k_scan_of_totals(uint32_t* __restrict__ totals, int nBlocks, uint32_t* __restrict__ grandTotal) {
    // one block; every thread owns a contiguous run of the totals
    __shared__ uint32_t sh[kScanBlock];
    const int per = (nBlocks + kScanBlock - 1) / kScanBlock, b0 = threadIdx.x * per, b1 = min(nBlocks, b0 + per);
    uint32_t sum = 0;
    for (int b = b0; b < b1; ++b) sum += totals[b];
    sh[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 1; o < kScanBlock; o <<= 1) {  // Hillis-Steele inclusive scan
        const uint32_t add = threadIdx.x >= o ? sh[threadIdx.x - o] : 0u;
        __syncthreads();
        sh[threadIdx.x] += add;
        __syncthreads();
    }
    uint32_t run = sh[threadIdx.x] - sum;  // exclusive prefix of this thread's run
    for (int b = b0; b < b1; ++b) { const uint32_t tot = totals[b]; totals[b] = run; run += tot; }
    if (threadIdx.x == kScanBlock - 1) *grandTotal = sh[threadIdx.x];
}
__global__ void __launch_bounds__(kScanBlock) k_scan_apply(const uint32_t* __restrict__ in, long long n, const uint32_t* __restrict__ totals,
                                                            const uint32_t* __restrict__ grandTotal, uint32_t* __restrict__ out) {
    __shared__ uint32_t sh[kScanBlock];
    const long long i = (long long)blockIdx.x * kScanBlock + threadIdx.x;
    const uint32_t v = i < n ? in[i] : 0u;
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < kScanBlock; o <<= 1) {
        const uint32_t add = threadIdx.x >= o ? sh[threadIdx.x - o] : 0u;
        __syncthreads();
        sh[threadIdx.x] += add;
        __syncthreads();
    }
    if (i < n) out[i] = totals[blockIdx.x] + sh[threadIdx.x] - v;
    if (i == n - 1) out[n] = *grandTotal;
}
// every cell's list into its order (sun::entry_before): one thread per cell, insertion sort in place (lists are short)
__global__ void __launch_bounds__(128) k_sun_sort(const uint32_t* __restrict__ cellStart, long long nCells, uint2* __restrict__ entries) {
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nCells) return;
    const uint32_t b = cellStart[c], e = cellStart[c + 1];
    if (e - b > sun::kSortMax) {  // (thousands of triangles over one cell: no order, no early exit)
        for (uint32_t i = b; i < e; ++i) entries[i].y = ex::f2u(sun::kFarthest);
        return;
    }
    for (uint32_t i = b + 1; i < e; ++i) {
        const uint2 x = entries[i];
        uint32_t j = i;
        while (j > b && sun::entry_before(x, entries[j - 1])) { entries[j] = entries[j - 1]; --j; }
        entries[j] = x;
    }
}

// Which render kernel?  k_render_paths wins where paths leave the scene early (+13..25 % on cube / suzanne / teapot), k_render where
// they do not (Sponza: +8 %).  The probe traces 4096 camera rays on a 64 x 64 grid over the frame and one diffuse bounce from each
// hit: out[0] = camera rays that hit, out[1] = bounce rays traced, out[2] = bounce rays that escaped to the sky.  ~10 us; the
// decision is cached with the scene for as long as camera and frame size stay the same (launch_render).
__global__ void __launch_bounds__(128) k_probe_paths(bvh::SceneView sc, integ::Camera cam, int width, int height, unsigned int* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // 4096 lanes
    const int gx = i & 63, gy = i >> 6;
    const int x = (int)(((long long)gx * 2 + 1) * width / 128), y = (int)(((long long)gy * 2 + 1) * height / 128);
    uint32_t rng = ex::pixel_seed(0x50524F42u + (uint32_t)i);  // "PROB": the probe's own streams, no relation to a frame's
    ex::V3 o, d;
    integ::primary_ray(cam, x, y, ex::divf(1.0f, (float)width), ex::divf(1.0f, (float)height), rng, o, d);
    bvh::HitRec h = bvh::traverse<false>(sc, o, d, integ::kMinT, integ::kMaxT);
    unsigned hit0 = h.id >= 0 ? 1u : 0u, esc = 0u;
    if (hit0) {
        ex::V3 pos, normal;
        bvh::hit_payload(sc, h.id, h.u, h.v, pos, normal);
        d = integ::scatter_dir(pos, normal, rng);
        esc = bvh::traverse<false>(sc, pos, d, integ::kMinT, integ::kMaxT).id < 0 ? 1u : 0u;
    }
    const unsigned nHit = __popc(__ballot_sync(0xffffffffu, hit0 != 0u)), nEsc = __popc(__ballot_sync(0xffffffffu, esc != 0u));
    if ((threadIdx.x & 31) == 0) { atomicAdd(&out[0], nHit); atomicAdd(&out[1], nHit); atomicAdd(&out[2], nEsc); }
}

// pixel = in-order sum of its chunk sums, then mean / sqrt / quantise (main.cpp:221-233), and the float outputs the frame asks
// for (integ::radiance_of ...).  AOV: the planes hold the hit counts and the second plane set (k_render<AOV>).
template <bool AOV>
__global__ void k_resolve(const RenderParams p, int bandRows) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)bandRows * p.localWidth) return;
    const int rb = (int)(i / p.localWidth), xl = (int)(i - (long long)rb * p.localWidth), r = p.bandRow0 + rb;
    int x, y;
    if (!local_to_global(xl, r, p.stripeRows, p.rank, p.world, p.width, x, y)) return;
    const size_t pix = (size_t)y * p.width + x;
    const size_t plane = (size_t)bandRows * p.localWidth;  // chunk-major planes: a warp's stores and these loads cover whole lines
    const float4* a = p.accum + i;
    ex::V3 sum = ex::v3(0.0f, 0.0f, 0.0f), nsum = sum;
    float tsum = 0.0f, hits = 0.0f;
    if (p.sumBuf) { const float4 v = p.sumBuf[pix]; sum = ex::v3(v.x, v.y, v.z); }  // progressive: the chunks before this pass
    for (int c = 0; c < p.chunks; ++c) {
        const float4 v = __ldcs(&a[(size_t)c * plane]);
        sum = ex::add(sum, ex::v3(v.x, v.y, v.z));
        if (AOV) {
            const float4 n = __ldcs(&a[(size_t)(p.chunks + c) * plane]);
            hits = ex::add(hits, v.w);
            nsum = ex::add(nsum, ex::v3(n.x, n.y, n.z));
            tsum = ex::add(tsum, n.w);
        }
    }
    if (p.sumBuf) p.sumBuf[pix] = make_float4(sum.x, sum.y, sum.z, 0.0f);
    const float sppRecip = ex::divf(1.0f, (float)p.spp);
    const uchar4 px = integ::resolve_pixel(sum, sppRecip);
    if (p.frame) p.frame[pix] = px;
    else p.outStripes[(size_t)r * p.localWidth + xl] = px;
    if (p.radiance) p.radiance[pix] = integ::radiance_of(sum, sppRecip);
    if (AOV) {
        if (p.normal) p.normal[pix] = integ::normal_of(nsum, hits, sppRecip);
        if (p.depth) p.depth[pix] = integ::depth_of(tsum, hits);
    }
}

// ---- K8: adaptive progressive passes (tmpt_progressive_pass_adaptive) ------------------------------------------------------------
// The active list is in tile order: slot i = tile (i >> 5) of the frame's 8x4 tiles in row-major tile order, lane i & 31 =
// (x & 7) + 8 (y & 3).  flags[i] = 1 for a pixel of the frame that the pass's params do not call converged; k_scan_* turn the flags
// into list positions and k_adaptive_compact writes each active pixel's entry {x | y << 16, n_i} there.  With every pixel of a
// frame whose size is a multiple of 8 x 4 active, list tile t is frame tile t: a LIST kernel's warp traces what k_render's does.
__global__ void k_adaptive_select(const uint32_t* __restrict__ n, const float2* __restrict__ stat, int width, int height, int tilesX,
                                  long long slots, float tolerance, int minChunks, uint32_t* __restrict__ flags) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= slots) return;
    const int tile = (int)(i >> 5), lane = (int)(i & 31);
    const int x = (tile % tilesX) * 8 + (lane & 7), y = (tile / tilesX) * 4 + (lane >> 3);
    uint32_t f = 0u;
    if (x < width && y < height) {
        const size_t pix = (size_t)y * width + x;
        const float2 st = stat[pix];
        f = integ::adaptive_converged(n[pix], st.x, st.y, tolerance, minChunks) ? 0u : 1u;
    }
    flags[i] = f;
}
__global__ void k_adaptive_compact(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ offs, const uint32_t* __restrict__ n,
                                   int width, int tilesX, long long slots, uint2* __restrict__ list) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= slots || !flags[i]) return;
    const int tile = (int)(i >> 5), lane = (int)(i & 31);
    const int x = (tile % tilesX) * 8 + (lane & 7), y = (tile / tilesX) * 4 + (lane >> 3);
    list[offs[i]] = make_uint2((uint32_t)x | ((uint32_t)y << 16), n[(size_t)y * width + x]);
}
// The band's chunk sums ([chunks][listLen]) into each entry's pixel in chunk order: the colour sum, n and the Welford state, then
// the pixels left unconverged under the pass's params are counted (the others were converged before the pass and are unchanged)
// into counters[0], and counters[1] keeps the session's largest n.
__global__ void k_resolve_adaptive(const RenderParams p, float4* __restrict__ sumBuf, uint32_t* __restrict__ n, float2* __restrict__ stat,
                                   float tolerance, int minChunks, unsigned int* __restrict__ counters) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    bool open = false;
    uint32_t nn = 0u;
    if (e < p.listLen) {
        const uint2 en = p.list[e];
        const size_t pix = (size_t)(en.x >> 16) * p.width + (en.x & 0xFFFFu);
        const float4 s0 = sumBuf[pix];
        ex::V3 sum = ex::v3(s0.x, s0.y, s0.z);
        nn = n[pix];
        float2 st = stat[pix];
        for (int c = 0; c < p.chunks; ++c) {
            const float4 v = __ldcs(&p.accum[(size_t)c * p.listLen + e]);
            const ex::V3 cs = ex::v3(v.x, v.y, v.z);
            sum = ex::add(sum, cs);
            integ::adaptive_add_chunk(cs, nn, st.x, st.y);
        }
        sumBuf[pix] = make_float4(sum.x, sum.y, sum.z, 0.0f);
        n[pix] = nn;
        stat[pix] = st;
        open = !integ::adaptive_converged(nn, st.x, st.y, tolerance, minChunks);
    }
    const unsigned b = __ballot_sync(0xffffffffu, open), mx = __reduce_max_sync(0xffffffffu, nn);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(&counters[0], (unsigned)__popc(b));
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(&counters[1], mx);
}
// The whole frame after an adaptive pass: every pixel is its mean over its own 8 n_i samples (as k_resolve resolves a uniform pass).
__global__ void k_adaptive_write(const float4* __restrict__ sumBuf, const uint32_t* __restrict__ n, long long pixels, uchar4* __restrict__ frame,
                                 float4* __restrict__ radiance, int32_t* __restrict__ samples) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pixels) return;
    const float4 v = sumBuf[i];
    const ex::V3 sum = ex::v3(v.x, v.y, v.z);
    const int spp = (int)n[i] * integ::kMaxChunkSamples;
    const float sppRecip = ex::divf(1.0f, (float)spp);
    frame[i] = integ::resolve_pixel(sum, sppRecip);
    if (radiance) radiance[i] = integ::radiance_of(sum, sppRecip);
    if (samples) samples[i] = spp;
}

// ---- K9: denoiser (tmpt_denoise) -----------------------------------------------------------------------------------------------
// One thread per pixel over 32 x 8 blocks, through denoise.cuh's per-pixel functions.  A warp is one row segment of 32 pixels, so
// every tap's loads are 32 consecutive float4s at any step; no shared-memory tile: from step 2 on the 5 x 5 taps reach 2 .. 128
// pixels away, far outside any tile of a 256-thread block, and at step 1 the overlapping windows of a block are L1 hits.
constexpr int kDenoiseBX = 32, kDenoiseBY = 8;
__global__ void __launch_bounds__(kDenoiseBX * kDenoiseBY) k_denoise_prep(const float4* __restrict__ radiance, const float4* __restrict__ normal,
                                                                        const float* __restrict__ depth, int width, int height,
                                                                        float4* __restrict__ state, float4* __restrict__ guideA,
                                                                        float4* __restrict__ guideB) {
    const int x = blockIdx.x * kDenoiseBX + threadIdx.x, y = blockIdx.y * kDenoiseBY + threadIdx.y;
    if (x >= width || y >= height) return;
    const size_t p = (size_t)y * width + x;
    float4 st, a, b;
    dn::prep_pixel(radiance, normal, depth, width, height, x, y, st, a, b);
    state[p] = st;
    guideA[p] = a;
    guideB[p] = b;
}
// One iteration: state `in` -> `out`; the LAST one writes the outputs instead of a state (the epilogue fused).
template <bool LAST>
__global__ void __launch_bounds__(kDenoiseBX * kDenoiseBY) k_denoise_atrous(const float4* __restrict__ in, float4* __restrict__ out,
                                                                          const float4* __restrict__ guideA, const float4* __restrict__ guideB,
                                                                          int width, int height, int step, dn::Params prm,
                                                                          uchar4* __restrict__ rgba, float4* __restrict__ radiance) {
    const int x = blockIdx.x * kDenoiseBX + threadIdx.x, y = blockIdx.y * kDenoiseBY + threadIdx.y;
    if (x >= width || y >= height) return;
    const size_t p = (size_t)y * width + x;
    const float4 s = dn::atrous_pixel(in, guideA, guideB, width, height, x, y, step, prm);
    if (!LAST) { out[p] = s; return; }
    if (rgba) rgba[p] = dn::rgba_of(s);
    if (radiance) radiance[p] = dn::radiance_of(s);
}
// No iteration: the outputs of the input radiance (radiance out may be radiance in: each thread reads its pixel before it writes it).
__global__ void k_denoise_copy(const float4* radianceIn, long long pixels, uchar4* __restrict__ rgba, float4* radiance) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pixels) return;
    const float4 c = radianceIn[i];
    if (rgba) rgba[i] = dn::rgba_of(c);
    if (radiance) radiance[i] = dn::radiance_of(c);
}

// K5: rank 0 scatters the gathered, rank-major packed stripes into the frame
__global__ void k_unpack_stripes(const uchar4* __restrict__ gathered, int width, int height, int stripeRows, int world, int maxRowsPerRank,
                                 uchar4* __restrict__ frame) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)width * height) return;
    const int y = (int)(i / width), x = (int)(i - (long long)y * width);
    if (stripeRows == 0) {  // tile interleave (local_to_global): tile (tx, ty) is local tile tx / world of rank (tx + ty) % world
        const int tx = x >> 3, ty = y >> 2, rank = (tx + ty) % world, localWidth = ((width + 7) / 8 + world - 1) / world * 8;
        frame[i] = gathered[((size_t)rank * maxRowsPerRank + y) * localWidth + ((tx / world) << 3) + (x & 7)];
        return;
    }
    const int gs = y / stripeRows, rank = gs % world, ls = gs / world;
    const int r = ls * stripeRows + (y - gs * stripeRows);
    frame[i] = gathered[((size_t)rank * maxRowsPerRank + r) * width + x];
}

// ------------------------------------------------------------------------------------------
// host side of the build
// ------------------------------------------------------------------------------------------
namespace {
// rays that start beyond 16 x the scene's largest |coordinate| are answered by the all-triangle scan (bvh.cuh: ray_is_far)
float bvh_far_limit(const tmpt_scene_info& info) {
    float m = 0.0f;
    for (int k = 0; k < 3; ++k) m = std::max(m, std::max(std::fabs(info.bounds_min[k]), std::fabs(info.bounds_max[k])));
    return 16.0f * m;
}

constexpr int kTreeTooDeep = -100;  // internal: tmpt_scene_create falls back to the depth-bounded default builder

int build_bvh(tmpt_scene* s, unsigned flags) {
    const int n = s->triCount;
    cudaStream_t st = s->stream;
    // SAH constants: one binary inner node vs one exact triangle test (TMPT_SAH_CI / TMPT_SAH_MAXLEAF: tuning overrides)
    const float cInner = getenv("TMPT_SAH_CI") ? (float)atof(getenv("TMPT_SAH_CI")) : 1.0f, cTri = 1.0f;
    // the level loops of the SAH build and of the collapse run inside one cooperative launch each; TMPT_BUILD_HOSTLOOP=1 (or a
    // device without cooperative launch) keeps them on the host, one launch and one read-back per level
    int coopAttr = 0;
    CU_TRY(cudaDeviceGetAttribute(&coopAttr, cudaDevAttrCooperativeLaunch, s->device));
    const bool coop = coopAttr != 0 && !(getenv("TMPT_BUILD_HOSTLOOP") && atoi(getenv("TMPT_BUILD_HOSTLOOP")) != 0);
    const int maxLeaf = getenv("TMPT_SAH_MAXLEAF") ? std::max(1, std::min(bvh::MAX_LEAF_TRIS, atoi(getenv("TMPT_SAH_MAXLEAF")))) : bvh::MAX_LEAF_TRIS;

    // every build scratch array comes out of ONE allocation (a dozen cudaMalloc/cudaFree pairs cost more than the kernels)
    struct Arr { void* p = nullptr; };
    Arr bounds, primA, primB, visits, counters, qCount, keysA, keysB, left, right, parent, first, lo, hi, sah, qA, qB, pLo, pHi, primFinal, nodeCounter, tqA, tqB;
    DevBuf<char> arena;
    {
        const size_t N = (size_t)n;
        struct Req { Arr* a; size_t bytes; };
        const Req reqs[] = {{&bounds, 6 * 4}, {&primA, N * 4}, {&primB, N * 4}, {&visits, N * 4}, {&counters, 4 * 4}, {&qCount, 4 * 4}, {&keysA, N * 8},
                            {&keysB, N * 8}, {&left, 2 * N * 4}, {&right, 2 * N * 4}, {&parent, 2 * N * 4}, {&first, 2 * N * 4}, {&lo, 2 * N * 16},
                            {&hi, 2 * N * 16}, {&sah, 2 * 4}, {&qA, N * sizeof(bld::WorkItem)}, {&qB, N * sizeof(bld::WorkItem)}, {&pLo, N * 16},
                            {&pHi, N * 16}, {&primFinal, N * 4}, {&nodeCounter, 4}, {&tqA, N * sizeof(SahTask)}, {&tqB, N * sizeof(SahTask)}};
        size_t total = 0;
        for (const Req& r : reqs) total += (r.bytes + 255) & ~(size_t)255;
        CU_TRY(arena.grow(total, st));
        size_t off = 0;
        for (const Req& r : reqs) { r.a->p = arena.p + off; off += (r.bytes + 255) & ~(size_t)255; }
    }
    // nodes, slots and hit payload share one allocation (each cudaMalloc costs as much as a build kernel)
    CU_TRY(s->d_nodes.grow((size_t)n * (bvh::NODE_F4 + 3 + 3) + div_up((long long)n * 2 + 8, sizeof(float4) / sizeof(uint32_t)), st));
    s->d_tris = s->d_nodes.p + (size_t)n * bvh::NODE_F4;
    s->d_hitdata = s->d_tris + (size_t)n * 3;
    s->d_parent = (uint32_t*)(s->d_hitdata + (size_t)n * 3);
    s->d_pending = s->d_parent + n;
    s->d_bounds = s->d_pending + n;
    CU_TRY(cudaMemsetAsync(s->d_parent, 0, sizeof(uint32_t), st));  // the root is its own parent

    uint32_t* const d_bounds = (uint32_t*)bounds.p; uint32_t* const d_primA = (uint32_t*)primA.p; uint32_t* const d_primB = (uint32_t*)primB.p;
    uint32_t* const d_visits = (uint32_t*)visits.p; uint32_t* const d_counters = (uint32_t*)counters.p; uint32_t* const d_qCount = (uint32_t*)qCount.p;
    uint64_t* const d_keysA = (uint64_t*)keysA.p; uint64_t* const d_keysB = (uint64_t*)keysB.p;
    int* const d_left = (int*)left.p; int* const d_right = (int*)right.p; int* const d_parent = (int*)parent.p; int* const d_first = (int*)first.p;
    float4* const d_lo = (float4*)lo.p; float4* const d_hi = (float4*)hi.p; float* const d_sah = (float*)sah.p;
    bld::WorkItem* const d_qA = (bld::WorkItem*)qA.p; bld::WorkItem* const d_qB = (bld::WorkItem*)qB.p;
    const uint32_t initBounds[6] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u};
    CU_TRY(cudaMemcpyAsync(d_bounds, initBounds, sizeof initBounds, cudaMemcpyHostToDevice, st));
    CU_TRY(cudaMemsetAsync(d_visits, 0, (size_t)n * sizeof(uint32_t), st));
    CU_TRY(cudaMemsetAsync(d_counters, 0, 4 * sizeof(uint32_t), st));
    CU_TRY(cudaMemsetAsync(d_sah, 0, 2 * sizeof(float), st));
    CU_TRY(cudaMemsetAsync(d_parent, 0xFF, 2 * (size_t)n * sizeof(int), st));

    const int B = 256, G = div_up(n, B);
    LAUNCH(k_prim_bounds, G, B, 0, st, s->d_tris9.p, n, d_bounds);
    LAUNCH(k_hitdata, G, B, 0, st, s->d_tris9.p, n, s->d_hitdata);
    bld::BinTree t{n, d_keysA, d_left, d_right, d_parent, d_lo, d_hi, d_first, d_visits};
    bld::SahParams sp{cInner, cTri, maxLeaf};
    const uint32_t* primOrder = d_primA;
    int rootIsLeaf = (n == 1);
    if (flags & TMPT_BUILD_LBVH) {
        LAUNCH(k_morton, G, B, 0, st, s->d_tris9.p, n, d_bounds, d_keysA, d_primA);
        const int passes = 16;  // 63-bit keys, 4 bits per pass; an even count leaves the result in A
        const int sortSmem = 16 * SORT_THREADS * (int)sizeof(uint32_t);
        CU_TRY(cudaFuncSetAttribute(k_radix_sort, cudaFuncAttributeMaxDynamicSharedMemorySize, sortSmem));
        LAUNCH(k_radix_sort, 1, SORT_THREADS, sortSmem, st, d_keysA, d_primA, d_keysB, d_primB, n, passes);
        LAUNCH(k_leaf_boxes, G, B, 0, st, s->d_tris9.p, d_primA, n, d_bounds, cTri, d_lo, d_hi, d_first);
        if (n > 1) {
            LAUNCH(k_karras, div_up(n - 1, B), B, 0, st, t);
            LAUNCH(k_refit, G, B, 0, st, t, sp);
        }
        s->info.builder = TMPT_BUILD_LBVH;
    } else {
        // binned SAH, level by level; tasks double-buffer in the collapse queues' memory
        float4* const d_pLo = (float4*)pLo.p; float4* const d_pHi = (float4*)pHi.p;
        uint32_t* const d_primFinal = (uint32_t*)primFinal.p; uint32_t* const d_nodeCounter = (uint32_t*)nodeCounter.p;
        SahTask* const d_tqA = (SahTask*)tqA.p; SahTask* const d_tqB = (SahTask*)tqB.p;
        LAUNCH(k_prim_boxes, G, B, 0, st, s->d_tris9.p, n, d_bounds, d_pLo, d_pHi, d_primA);
        const SahTask rootTask{0, 0, n, 0};
        const uint32_t one = 1, zero = 0;
        CU_TRY(cudaMemcpyAsync(d_tqA, &rootTask, sizeof rootTask, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(d_nodeCounter, &one, 4, cudaMemcpyHostToDevice, st));
        bool sahDone = false;
        if (coop) {
            // one cooperative launch for all levels (k_sah_build); d_qCount = three rotating task counters
            const uint32_t counts0[3] = {1u, 0u, 0u};
            CU_TRY(cudaMemcpyAsync(d_qCount, counts0, sizeof counts0, cudaMemcpyHostToDevice, st));
            int perSM = 0;
            CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_sah_build, SAH_THREADS, 0));
            const int grid = std::max(1, std::min(s->smCount * std::max(perSM, 1), n));
            uint32_t* idxA = d_primA; uint32_t* idxB = d_primB;
            SahTask* qA = d_tqA; SahTask* qB = d_tqB;
            uint32_t* countsP = d_qCount; uint32_t* nodeCounterP = d_nodeCounter; uint32_t* primFinalP = d_primFinal;
            const float4* pLoP = d_pLo; const float4* pHiP = d_pHi;
            int maxLevels = 4096;
            uint32_t* statusP = s->d_status.p + 1;
            void* args[] = {&t, &pLoP, &pHiP, &idxA, &idxB, &primFinalP, &qA, &qB, &countsP, &nodeCounterP, &sp, &maxLevels, &statusP};
            // (a refused cooperative launch -- e.g. the device is shared and the grid cannot be co-resident -- is not an error:
            //  nothing has run yet, the per-level loop below does the same work)
            if (cudaLaunchCooperativeKernel((void*)k_sah_build, dim3(grid), dim3(SAH_THREADS), args, 0, st) == cudaSuccess) {
                tmpt::count_launch();
                sahDone = true;
            } else {
                cudaGetLastError();
            }
        }
        if (!sahDone) {
            uint32_t* idxIn = d_primA; uint32_t* idxOut = d_primB;
            SahTask* qin = d_tqA; SahTask* qout = d_tqB;
            uint32_t count = 1;
            int levels = 0;
            while (count > 0) {
                CU_TRY(cudaMemcpyAsync(d_qCount, &zero, 4, cudaMemcpyHostToDevice, st));
                LAUNCH(k_sah_level, count, SAH_THREADS, 0, st, t, d_pLo, d_pHi, idxIn, idxOut, d_primFinal, qin, qout, d_qCount, d_nodeCounter, sp);
                CU_TRY(cudaMemcpyAsync(&count, d_qCount, 4, cudaMemcpyDeviceToHost, st));
                CU_TRY(cudaStreamSynchronize(st));
                std::swap(idxIn, idxOut);
                std::swap(qin, qout);
                if (++levels > 4096) return tmpt::fail(TMPT_ERR_CUDA, "SAH build did not terminate");
            }
        }
        // the final order lives in primFinal; keep it in primA for the collapse (same stream, device copy)
        CU_TRY(cudaMemcpyAsync(d_primA, d_primFinal, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
        s->info.builder = TMPT_BUILD_DEFAULT;
    }
    bld::WideOut w{s->d_nodes.p, s->d_tris, s->d_tris9.p, primOrder, d_counters, d_sah, s->d_parent};
    if (n > 1) {
        float4 rootHi;
        uint32_t bst = 0;
        CU_TRY(cudaMemcpyAsync(&rootHi, d_hi, sizeof rootHi, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaMemcpyAsync(&bst, s->d_status.p + 1, 4, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        if (bst & 2u) return tmpt::fail(TMPT_ERR_CUDA, "SAH build did not terminate");
        int c; memcpy(&c, &rootHi.w, 4);
        rootIsLeaf = c < 0;
    }
    if (rootIsLeaf) {
        const uint32_t one = 1;
        CU_TRY(cudaMemcpyAsync(d_counters, &one, 4, cudaMemcpyHostToDevice, st));
        LAUNCH(k_collapse_root_leaf, 1, 1, 0, st, t, w, 0);
    } else {
        const bld::WorkItem root{0, 0u, 0};
        const uint32_t one = 1, zero = 0;
        CU_TRY(cudaMemcpyAsync(d_qA, &root, sizeof root, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(d_counters, &one, 4, cudaMemcpyHostToDevice, st));   // wide node 0 is taken
        CU_TRY(cudaMemcpyAsync(d_qCount, &one, 4, cudaMemcpyHostToDevice, st));
        bool collapseDone = false;
        if (coop) {
            const uint32_t counts0[3] = {1u, 0u, 0u};
            CU_TRY(cudaMemcpyAsync(d_qCount, counts0, sizeof counts0, cudaMemcpyHostToDevice, st));
            int perSM = 0;
            CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_collapse_all, 128, 0));
            const int grid = std::max(1, std::min(s->smCount * std::max(perSM, 1), div_up(n, 128)));
            bld::WorkItem* qA = d_qA; bld::WorkItem* qB = d_qB;
            uint32_t* countsP = d_qCount;
            void* args[] = {&t, &w, &qA, &qB, &countsP};
            if (cudaLaunchCooperativeKernel((void*)k_collapse_all, dim3(grid), dim3(128), args, 0, st) == cudaSuccess) {
                tmpt::count_launch();
                collapseDone = true;
            } else {
                cudaGetLastError();
            }
        }
        if (!collapseDone) {
            CU_TRY(cudaMemcpyAsync(d_qCount, &one, 4, cudaMemcpyHostToDevice, st));
            bld::WorkItem* qin = d_qA; bld::WorkItem* qout = d_qB;
            int cin = 0;
            uint32_t count = 1;
            while (count > 0) {
                CU_TRY(cudaMemcpyAsync(d_qCount + (1 - cin), &zero, 4, cudaMemcpyHostToDevice, st));
                LAUNCH(k_collapse, div_up(count, 128), 128, 0, st, t, w, qin, d_qCount + cin, qout, d_qCount + (1 - cin));
                CU_TRY(cudaMemcpyAsync(&count, d_qCount + (1 - cin), 4, cudaMemcpyDeviceToHost, st));
                CU_TRY(cudaStreamSynchronize(st));
                cin = 1 - cin;
                bld::WorkItem* tq = qin; qin = qout; qout = tq;
            }
        }
    }
    uint32_t hc[4]; float hs[2]; uint32_t hb[6];
    CU_TRY(cudaMemcpyAsync(hc, d_counters, sizeof hc, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(hs, d_sah, sizeof hs, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaMemcpyAsync(hb, d_bounds, sizeof hb, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    CU_TRY(cudaGetLastError());
    s->info.node_count = (int)hc[0];
    s->info.leaf_count = (int)hc[2];
    s->info.max_depth = (int)hc[3] + 1;
    s->info.max_leaf_tris = bvh::MAX_LEAF_TRIS;
    for (int k = 0; k < 3; ++k) {
        s->info.bounds_min[k] = bld::ordered_to_float(hb[k]);
        s->info.bounds_max[k] = bld::ordered_to_float(hb[3 + k]);
    }
    {
        const float dx = s->info.bounds_max[0] - s->info.bounds_min[0], dy = s->info.bounds_max[1] - s->info.bounds_min[1],
                    dz = s->info.bounds_max[2] - s->info.bounds_min[2];
        const float rootArea = dx * dy + dy * dz + dz * dx;
        s->info.sah_cost = rootArea > 0.0f ? (cInner * hs[0] + cTri * hs[1]) / rootArea : 0.0f;
    }
    if ((int)hc[1] != n) return tmpt::fail(TMPT_ERR_CUDA, "BVH build lost triangles: %u slots for %d triangles", hc[1], n);
#if TMPT_QNODES
    CU_TRY(s->d_qnodes.grow((size_t)hc[0] * bvh::QNODE_STRIDE, st));
    LAUNCH(k_quantize_nodes, div_up((int)hc[0], 128), 128, 0, st, s->d_nodes.p, s->d_qnodes.p, hc[0]);
#endif
    // the traversal stack holds at most 3 entries per level (bvh::wide_node_step): refuse what it could not hold.  The default
    // builder cannot get here (bld::sah_must_halve bounds its depth for any input); a Morton tree over many coincident centres can.
    if (3 * s->info.max_depth + 4 > bvh::STACK_SIZE) {
        tmpt::fail(TMPT_ERR_ARG, "BVH is %d levels deep; the traversal stack (%d entries) supports %d", s->info.max_depth, bvh::STACK_SIZE,
                   (bvh::STACK_SIZE - 4) / 3);
        return kTreeTooDeep;
    }
    s->info.device_bytes = (uint64_t)n * 9 * 4 + (uint64_t)hc[0] * (bvh::NODE_F4 + (TMPT_QNODES ? bvh::QNODE_STRIDE : 0)) * 16 + (uint64_t)n * 48 + (uint64_t)n * 48;
    s->view.nodes = s->d_nodes.p;
    s->view.qnodes = s->d_qnodes.p;
    s->view.tris = s->d_tris;
    s->view.tris9 = s->d_tris9.p;
    s->view.hitdata = s->d_hitdata;
    s->view.rootRef = 0u;
    s->view.triCount = n;
    s->view.status = s->d_status.p;
    s->view.farLimit = bvh_far_limit(s->info);
    return TMPT_OK;
}

// The sun grid of a scene (sungrid.cuh): basis and projected bounds on the host (doubles, from the caller's triangles), binning on the
// device.  TMPT_SUN_GRID=0 turns it off (shadow rays walk the tree), =n forces n cells per side.  If the lists would need more
// than kSunMaxEntries entries (a scene of huge overlapping triangles) the grid is halved, and dropped below 32 cells per side.
constexpr unsigned long long kSunMaxEntries = 256ull << 20;
static ex::V3 host_light_dir() { return ex::normalize(ex::v3(-0.7f, 1.0f, 0.5f)); }  // main.cpp:36
static int build_sun_grid(tmpt_scene* s, int n, cudaStream_t st) {  // (after the tree: needs s->info.bounds_min / max)
    static const int forced = getenv("TMPT_SUN_GRID") ? atoi(getenv("TMPT_SUN_GRID")) : -1;
    s->view.sun = sun::View{};
    s->info.device_bytes -= s->sunBytes;
    s->sunBytes = 0; s->sunEntries = 0;
    if (forced == 0 || n <= 0) return TMPT_OK;
    static const bool trace = getenv("TMPT_SUN_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    sun::View g;
    if (!sun::setup_view(s->info.bounds_min, s->info.bounds_max, host_light_dir(), g)) return TMPT_OK;  // NaN / infinite vertices: no grid, the tree copes
    const double t1 = now();
    int cells = forced > 0 ? std::min(std::max(forced, 1), 8192) : sun::default_cells_per_side(n);
    for (;; cells /= 2) {
        if (cells < (forced > 0 ? 1 : 32)) return TMPT_OK;  // (no grid)
        sun::set_resolution(g, cells);
        const long long nCells = (long long)cells * cells;
        const int nBlocks = (int)((nCells + kScanBlock - 1) / kScanBlock);
        const size_t needStart = (size_t)nCells + 1, needCount = (size_t)nCells + nBlocks + 2 + n;
        CU_TRY(s->d_sunStart.grow(needStart, st));  // (a refit finds its buffers in place)
        CU_TRY(s->d_sunCount.grow(needCount, st));
        uint32_t* totals = s->d_sunCount.p + nCells;
        uint32_t* grand = totals + nBlocks;
        uint32_t* bigCount = grand + 1;
        uint32_t* bigList = bigCount + 1;  // up to n slots
        CU_TRY(cudaMemsetAsync(s->d_sunCount.p, 0, (size_t)(nCells + nBlocks + 2) * sizeof(uint32_t), st));
        const int binGrid = (int)(((long long)n * 32 + 255) / 256), bigGrid = s->smCount * 8;
        LAUNCH((k_sun_bin<false>), binGrid, 256, 0, st, g, s->d_tris, s->d_tris9.p, n, s->d_sunCount.p, nullptr, nullptr, bigList, bigCount);
        LAUNCH((k_sun_bin_big<false>), bigGrid, 256, 0, st, g, s->d_tris, s->d_tris9.p, s->d_sunCount.p, nullptr, nullptr, bigList, bigCount);
        LAUNCH(k_scan_totals, nBlocks, kScanBlock, 0, st, s->d_sunCount.p, nCells, totals);
        LAUNCH(k_scan_of_totals, 1, kScanBlock, 0, st, totals, nBlocks, grand);
        LAUNCH(k_scan_apply, nBlocks, kScanBlock, 0, st, s->d_sunCount.p, nCells, totals, grand, s->d_sunStart.p);
        uint32_t total = 0;
        const double t2 = now();
        CU_TRY(cudaMemcpyAsync(&total, grand, sizeof total, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        const double t3 = now();
        if ((unsigned long long)total > kSunMaxEntries) continue;  // halve the grid
        CU_TRY(s->d_sunEntries.grow(total, st));
        CU_TRY(cudaMemsetAsync(s->d_sunCount.p, 0, (size_t)nCells * sizeof(uint32_t), st));
        LAUNCH((k_sun_bin<true>), binGrid, 256, 0, st, g, s->d_tris, s->d_tris9.p, n, s->d_sunCount.p, s->d_sunStart.p, s->d_sunEntries.p, bigList, bigCount);
        LAUNCH((k_sun_bin_big<true>), bigGrid, 256, 0, st, g, s->d_tris, s->d_tris9.p, s->d_sunCount.p, s->d_sunStart.p, s->d_sunEntries.p, bigList, bigCount);
        LAUNCH(k_sun_sort, (int)((nCells + 127) / 128), 128, 0, st, s->d_sunStart.p, nCells, s->d_sunEntries.p);
        if (trace) {
            CU_TRY(cudaStreamSynchronize(st));
            fprintf(stderr, "[sun grid] n %d entries %u: host setup %.2f ms, alloc + count launches %.2f ms, wait for the stream %.2f ms, alloc + fill + sort %.2f ms\n",
                    cells, total, t1 - t0, t2 - t1, t3 - t2, now() - t3);
        }
        g.cellStart = s->d_sunStart.p;
        g.entries = s->d_sunEntries.p;
        s->view.sun = g;
        s->sunBytes = (uint64_t)(nCells + 1) * 4 + (uint64_t)total * 8;
        s->info.device_bytes += s->sunBytes;
        s->sunEntries = total;
        return TMPT_OK;
    }
}

struct DeviceGuard {
    int prev = -1;
    bool ok = false;
    explicit DeviceGuard(int dev) { ok = cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
}  // namespace

// ------------------------------------------------------------------------------------------
// C ABI: scene
// ------------------------------------------------------------------------------------------
extern "C" int tmpt_scene_create(const float* tris9, int triCount, int device, unsigned flags, tmpt_scene** outScene) {
    if (!outScene) return tmpt::fail(TMPT_ERR_ARG, "tmpt_scene_create: outScene is NULL");
    *outScene = nullptr;
    if (triCount < 0 || triCount >= (1 << 28) - 1 || (triCount > 0 && !tris9))
        return tmpt::fail(TMPT_ERR_ARG, "tmpt_scene_create: bad triangle array (count %d)", triCount);
    int nDev = 0;
    if (cudaGetDeviceCount(&nDev) != cudaSuccess || nDev == 0) {
        cudaGetLastError();
        return tmpt::fail(TMPT_ERR_CUDA, "tmpt_scene_create: no CUDA device (this library has no CPU path)");
    }
    if (device < 0 || device >= nDev) return tmpt::fail(TMPT_ERR_ARG, "tmpt_scene_create: device %d of %d", device, nDev);
    DeviceGuard guard(device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_scene_create: cudaSetDevice(%d) failed", device);

    tmpt_scene* s = new (std::nothrow) tmpt_scene();
    if (!s) return tmpt::fail(TMPT_ERR_OOM, "tmpt_scene_create: out of host memory");
    s->device = device;
    s->triCount = triCount;
    s->info.abi_version = TMPT_ABI_VERSION;
    s->info.device = device;
    s->info.tri_count = triCount;
    int rc = TMPT_OK;
    auto body = [&]() -> int {
        cudaDeviceProp prop;
        CU_TRY(cudaGetDeviceProperties(&prop, device));
        s->smCount = prop.multiProcessorCount;
        CU_TRY(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
        CU_TRY(cudaEventCreate(&s->ev0));
        CU_TRY(cudaEventCreate(&s->ev1));
        CU_TRY(s->d_status.grow(4, s->stream));
        CU_TRY(cudaMemsetAsync(s->d_status.p, 0, 4 * sizeof(uint32_t), s->stream));
        CU_TRY(s->d_tileCounter.grow(1, s->stream));
        CU_TRY(s->d_rayCount.grow(1, s->stream));
        CU_TRY(s->d_fetchCounter.grow(1, s->stream));
        CU_TRY(cudaEventRecord(s->ev0, s->stream));
        if (triCount > 0) {
            CU_TRY(s->d_tris9.grow((size_t)triCount * 9, s->stream));
            CU_TRY(cudaMemcpyAsync(s->d_tris9.p, tris9, (size_t)triCount * 9 * sizeof(float), cudaMemcpyHostToDevice, s->stream));
            int brc = build_bvh(s, flags);
            if (brc == kTreeTooDeep && (flags & TMPT_BUILD_LBVH)) {
                // a Morton tree can be arbitrarily deep (many coincident centres); the SAH builder bounds its depth for any input
                CU_TRY(cudaStreamSynchronize(s->stream));
                s->d_nodes.reset();
                s->d_qnodes.reset();
                brc = build_bvh(s, flags & ~(unsigned)TMPT_BUILD_LBVH);
            }
            if (brc != TMPT_OK) return brc == kTreeTooDeep ? TMPT_ERR_ARG : brc;
            brc = build_sun_grid(s, triCount, s->stream);
            if (brc != TMPT_OK) return brc;
        } else {
            s->view = bvh::SceneView{nullptr, nullptr, nullptr, nullptr, bvh::NONE, 0, s->d_status.p, nullptr, 0.0f};
        }
        CU_TRY(cudaEventRecord(s->ev1, s->stream));
        CU_TRY(cudaStreamSynchronize(s->stream));
        float ms = 0.0f;
        CU_TRY(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
        s->info.build_ms = ms;
        return TMPT_OK;
    };
    rc = body();
    if (rc != TMPT_OK) { tmpt_scene_destroy(s); return rc; }
    *outScene = s;
    return TMPT_OK;
}

// Animated vertices: same triangle count and order, new positions.  The tree keeps its topology; boxes, slots and hit
// payload are recomputed on the device (k_refit_wide).  Results stay exact for any motion -- the tree only culls --
// but a tree built for the old positions gets slower the further the vertices move.
extern "C" int tmpt_scene_refit(tmpt_scene* s, const float* tris9, int triCount, double* seconds) {
    if (!s || (triCount > 0 && !tris9)) return tmpt::fail(TMPT_ERR_ARG, "tmpt_scene_refit: NULL scene / triangles");
    if (triCount != s->triCount) return tmpt::fail(TMPT_ERR_ARG, "tmpt_scene_refit: %d triangles, the scene was built with %d", triCount, s->triCount);
    if (seconds) *seconds = 0.0;
    if (triCount == 0) return TMPT_OK;
    std::lock_guard<std::mutex> lock(s->hostCallMutex);
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_scene_refit: cudaSetDevice(%d) failed", s->device);
    cudaStream_t st = s->stream;
    const int n = triCount, B = 256, G = div_up(n, B), nodes = s->info.node_count;
    CU_TRY(cudaEventRecord(s->ev0, st));
    CU_TRY(cudaMemcpyAsync(s->d_tris9.p, tris9, (size_t)n * 9 * sizeof(float), cudaMemcpyHostToDevice, st));
    const uint32_t initBounds[6] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u};
    CU_TRY(cudaMemcpyAsync(s->d_bounds, initBounds, sizeof initBounds, cudaMemcpyHostToDevice, st));
    LAUNCH(k_prim_bounds, G, B, 0, st, s->d_tris9.p, n, s->d_bounds);
    LAUNCH(k_hitdata, G, B, 0, st, s->d_tris9.p, n, s->d_hitdata);
    LAUNCH(k_refit_pending, div_up(nodes, 128), 128, 0, st, s->d_nodes.p, (uint32_t)nodes, s->d_pending);
    LAUNCH(k_refit_wide, div_up(nodes, 128), 128, 0, st, s->d_nodes.p, s->d_tris, s->d_tris9.p, s->d_parent, s->d_pending, (uint32_t)nodes, s->d_bounds);
#if TMPT_QNODES
    LAUNCH(k_quantize_nodes, div_up(nodes, 128), 128, 0, st, s->d_nodes.p, s->d_qnodes.p, (uint32_t)nodes);
#endif
    uint32_t hb[6];
    CU_TRY(cudaMemcpyAsync(hb, s->d_bounds, sizeof hb, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    CU_TRY(cudaGetLastError());
    for (int k = 0; k < 3; ++k) {
        s->info.bounds_min[k] = bld::ordered_to_float(hb[k]);
        s->info.bounds_max[k] = bld::ordered_to_float(hb[3 + k]);
    }
    {  // the shadow rays' grid is rebuilt for the new positions and bounds (inside the timed window)
        const int grc = build_sun_grid(s, n, st);
        if (grc != TMPT_OK) return grc;
    }
    CU_TRY(cudaEventRecord(s->ev1, st));
    CU_TRY(cudaStreamSynchronize(st));
    CU_TRY(cudaGetLastError());
    s->view.farLimit = bvh_far_limit(s->info);
    s->probeW = 0;  // moved geometry: the next frame probes again (k_probe_paths)
    float ms = 0.0f;
    CU_TRY(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    if (seconds) *seconds = ms * 1e-3;
    return TMPT_OK;
}

extern "C" void tmpt_scene_destroy(tmpt_scene* s) {
    if (!s) return;
    DeviceGuard guard(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    if (s->probeDone) cudaEventDestroy(s->probeDone);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;  // (its buffers free their memory while the guard holds the scene's device)
}

extern "C" int tmpt_scene_get_info(const tmpt_scene* s, tmpt_scene_info* out) {
    if (!s || !out) return tmpt::fail(TMPT_ERR_ARG, "tmpt_scene_get_info: NULL argument");
    *out = s->info;
    return TMPT_OK;
}

static int check_status(const tmpt_scene* s, cudaStream_t st) {
    uint32_t status = 0;
    CU_TRY(cudaMemcpyAsync(&status, s->d_status.p, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    if (status & bvh::STACK_OVERFLOW) return tmpt::fail(TMPT_ERR_CUDA, "traversal stack overflow (BVH depth %d)", s->info.max_depth);
    return TMPT_OK;
}

// ------------------------------------------------------------------------------------------
// C ABI: HitScene
// ------------------------------------------------------------------------------------------
extern "C" int tmpt_hit_scene(const tmpt_scene* s, const float* rays6, int64_t nRays, float tMin, float tMax, int mode, int mem,
                              int32_t* outID, float* outT, float* outPos3, float* outNormal3, void* stream) {
    if (!s || nRays < 0 || (nRays > 0 && (!rays6 || !outID))) return tmpt::fail(TMPT_ERR_ARG, "tmpt_hit_scene: NULL scene / rays / outID");
    if (mode != TMPT_HIT_CLOSEST && mode != TMPT_HIT_ANY && mode != TMPT_HIT_BRUTE && mode != TMPT_HIT_SUN) return tmpt::fail(TMPT_ERR_ARG, "tmpt_hit_scene: mode %d", mode);
    if (mode == TMPT_HIT_SUN && s->triCount > 0 && s->view.sun.n == 0) return tmpt::fail(TMPT_ERR_ARG, "tmpt_hit_scene: TMPT_HIT_SUN, but this scene has no sun grid");
    if (mem != TMPT_HOST && mem != TMPT_DEVICE) return tmpt::fail(TMPT_ERR_ARG, "tmpt_hit_scene: mem %d", mem);
    if (nRays == 0) return TMPT_OK;
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_hit_scene: cudaSetDevice(%d) failed", s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;

    const float* dRays = rays6; int* dID = outID; float* dT = outT; float* dPos = outPos3; float* dNrm = outNormal3;
    // TMPT_HOST: [rays 6n | id n | t n | pos 3n | normal 3n] floats / ints in the scene's staging buffers.  The outputs start
    // from the caller's contents, because entries of rays that miss must stay untouched (scene.cpp:86-97 writes outHit only on a hit).
    std::unique_lock<std::mutex> lock(const_cast<tmpt_scene*>(s)->hostCallMutex, std::defer_lock);
    const size_t n = (size_t)nRays;
    const size_t offID = 6 * n * 4, offT = offID + n * 4, offPos = offT + (outT ? n * 4 : 0), offNrm = offPos + (outPos3 ? 3 * n * 4 : 0),
                 total = offNrm + (outNormal3 ? 3 * n * 4 : 0);
    if (mem == TMPT_HOST) {
        lock.lock();
        tmpt_scene* ms = const_cast<tmpt_scene*>(s);  // scratch only
        CU_TRY(ms->d_stage.grow(total, ms->stream, total + total / 4));
        CU_TRY(ms->h_stage.grow(total, ms->stream, total + total / 4));
        char* h = ms->h_stage.p; char* d = ms->d_stage.p;
        memcpy(h, rays6, 6 * n * 4);
        if (outT) memcpy(h + offT, outT, n * 4);
        if (outPos3) memcpy(h + offPos, outPos3, 3 * n * 4);
        if (outNormal3) memcpy(h + offNrm, outNormal3, 3 * n * 4);
        CU_TRY(cudaMemcpyAsync(d, h, 6 * n * 4, cudaMemcpyHostToDevice, st));                                     // rays
        if (total > offT) CU_TRY(cudaMemcpyAsync(d + offT, h + offT, total - offT, cudaMemcpyHostToDevice, st));  // outputs' initial contents
        dRays = (const float*)d; dID = (int*)(d + offID);
        dT = outT ? (float*)(d + offT) : nullptr; dPos = outPos3 ? (float*)(d + offPos) : nullptr; dNrm = outNormal3 ? (float*)(d + offNrm) : nullptr;
    }
    const int B = 128;
    const int G = (int)std::min<long long>(div_up(nRays, B), (long long)s->smCount * 64);
    if (getenv("TMPT_HIT_KERNEL") && atoi(getenv("TMPT_HIT_KERNEL")) > 0)
        return tmpt::fail(TMPT_ERR_ARG, "TMPT_HIT_KERNEL: the experimental HitScene kernels of round 1 were removed (see profiles/r1_hit_scene_variants_ncu.txt)");
#if TMPT_EXPERIMENTS
    static const int refillGate = getenv("TMPT_HIT_REFILL") ? atoi(getenv("TMPT_HIT_REFILL")) : 0;
    if (refillGate > 0 && mode != TMPT_HIT_BRUTE) {
        CU_TRY(cudaMemsetAsync(s->d_fetchCounter.p, 0, sizeof(unsigned long long), st));
        int perSM = 0;
#define REFILL_CASE(M, GT)                                                                                                     \
        if (mode == M && refillGate == GT) {                                                                                   \
            CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSM, k_hit_scene_refill<M, GT>, B, 0));                    \
            const int GP = (int)std::min<long long>(div_up(nRays, B), (long long)s->smCount * std::max(perSM, 1));            \
            LAUNCH((k_hit_scene_refill<M, GT>), GP, B, 0, st, s->view, dRays, (long long)nRays, tMin, tMax, dID, dT, dPos, dNrm, s->d_fetchCounter.p); \
        } else
        REFILL_CASE(TMPT_HIT_CLOSEST, 1) REFILL_CASE(TMPT_HIT_CLOSEST, 4) REFILL_CASE(TMPT_HIT_CLOSEST, 8) REFILL_CASE(TMPT_HIT_CLOSEST, 16)
        REFILL_CASE(TMPT_HIT_ANY, 1) REFILL_CASE(TMPT_HIT_ANY, 4) REFILL_CASE(TMPT_HIT_ANY, 8) REFILL_CASE(TMPT_HIT_ANY, 16)
#undef REFILL_CASE
        return tmpt::fail(TMPT_ERR_ARG, "TMPT_HIT_REFILL=%d: gates are 1, 4, 8, 16", refillGate);
    } else
#endif
    if (mode == TMPT_HIT_CLOSEST) LAUNCH((k_hit_scene<TMPT_HIT_CLOSEST, false>), G, B, 0, st, s->view, dRays, (long long)nRays, tMin, tMax, dID, dT, dPos, dNrm, nullptr);
    else if (mode == TMPT_HIT_ANY) LAUNCH((k_hit_scene<TMPT_HIT_ANY, false>), G, B, 0, st, s->view, dRays, (long long)nRays, tMin, tMax, dID, dT, dPos, dNrm, nullptr);
    else if (mode == TMPT_HIT_SUN) LAUNCH((k_hit_scene<TMPT_HIT_SUN, false>), G, B, 0, st, s->view, dRays, (long long)nRays, tMin, tMax, dID, dT, dPos, dNrm, nullptr);
    else LAUNCH((k_hit_scene<TMPT_HIT_BRUTE, false>), G, B, 0, st, s->view, dRays, (long long)nRays, tMin, tMax, dID, dT, dPos, dNrm, nullptr);
    CU_TRY(cudaGetLastError());
    if (mem == TMPT_HOST) {
        const char* d = s->d_stage.p; char* h = s->h_stage.p;
        CU_TRY(cudaMemcpyAsync(h + offID, d + offID, total - offID, cudaMemcpyDeviceToHost, st));  // id | t | pos | normal in one copy
        CU_TRY(cudaStreamSynchronize(st));
        memcpy(outID, h + offID, n * 4);
        if (outT) memcpy(outT, h + offT, n * 4);
        if (outPos3) memcpy(outPos3, h + offPos, 3 * n * 4);
        if (outNormal3) memcpy(outNormal3, h + offNrm, 3 * n * 4);
        return check_status(s, st);
    }
    return TMPT_OK;
}

// ------------------------------------------------------------------------------------------
// C ABI: render
// ------------------------------------------------------------------------------------------
extern "C" int tmpt_local_width(int width, int stripeRows, int worldSize) {
    if (width <= 0 || stripeRows < 0 || worldSize <= 0) return 0;
    return stripeRows > 0 ? width : ((width + 7) / 8 + worldSize - 1) / worldSize * 8;
}
extern "C" int tmpt_stripe_rows(int height, int stripeRows, int rank, int worldSize) {
    if (height <= 0 || stripeRows < 0 || worldSize <= 0 || rank < 0 || rank >= worldSize) return 0;
    if (stripeRows == 0) return height;  // tile interleave: every rank owns tiles in every row
    const int stripes = (height + stripeRows - 1) / stripeRows;
    int rows = 0;
    for (int k = rank; k < stripes; k += worldSize) rows += std::min(stripeRows, height - k * stripeRows);
    return rows;
}


// samples per chunk / chunks per pixel of a one-shot frame (TMPT_CHUNK_LEN: tuning override, changes the RNG layout)
static int host_chunk_len(int spp) {
    static const int forced = getenv("TMPT_CHUNK_LEN") ? atoi(getenv("TMPT_CHUNK_LEN")) : 0;
    return forced > 0 ? std::min(forced, integ::kMaxChunkSamples) : integ::chunk_len(spp);
}
static int host_chunk_count(int spp) { const int c = host_chunk_len(spp); return (spp + c - 1) / c; }

// One pass of a progressive render: chunks [chunk0, chunk0 + nChunks) of kMaxChunkSamples samples, added to `sum`.  An adaptive
// pass (adaptive != nullptr) traces chunks [n_i, n_i + nChunks) of the pixels on its active list instead (chunk0 unused).
struct AdaptivePass {
    float tolerance;
    int minChunks;
    int32_t* samples;  // the caller's buffer of the frame's samples per pixel (in the call's `mem`), or null
};
struct ProgressivePass {
    int chunk0, nChunks;
    float4* sum;
    const AdaptivePass* adaptive = nullptr;
};
// What render_frame reports of an adaptive pass: the active pixels it traced, then the pixels left unconverged and the session's
// largest n.
struct AdaptiveResult {
    int listLen = 0;
    unsigned int counters[2] = {0u, 0u};
};

// The float outputs of a single-GPU frame (tmpt_outputs, device pointers; null = not produced).
struct FrameOutputs {
    float4* radiance = nullptr;
    float4* normal = nullptr;
    float* depth = nullptr;
    int32_t* triangle = nullptr;
    bool aov() const { return normal || depth || triangle; }    // the render kernels' AOV instantiations run
    bool accum() const { return radiance || normal || depth; }  // k_resolve writes them: chunk sums go through the planes even at one chunk
};

// Everything a frame's or a pass's launches depend on besides the kernel choice, from its arguments alone.
struct RenderPlan {
    OutMode mode;
    int chunks, chunk0, chunkLen;
    int spp;            // the samples the mean divides by (progressive: the samples so far)
    bool useAccum;      // chunk sums go through the accumulation planes and a resolve kernel
    int planes;         // plane sets per chunk: 2 with AOV outputs (the normal and t sums behind the colour's)
    int granule;        // bands are multiples of it: 4 rows (a tile row), or 32 list entries (a list tile)
    int units;          // what is banded: owned rows, or the entries of an adaptive pass's active list
    int unitWidth;      // pixels per unit: the local width, or 1
};
static RenderPlan plan_render(int localWidth, int ownedRows, int spp, const ProgressivePass* prog, const FrameOutputs* outs, int listLen) {
    RenderPlan pl;
    pl.mode = prog && prog->adaptive ? OutMode::List : outs && outs->aov() ? OutMode::Aov : OutMode::Frame;
    pl.chunks = prog ? prog->nChunks : host_chunk_count(spp);
    pl.chunk0 = prog ? prog->chunk0 : 0;
    pl.chunkLen = prog ? integ::kMaxChunkSamples : host_chunk_len(spp);
    pl.spp = prog ? integ::kMaxChunkSamples * (prog->chunk0 + prog->nChunks) : spp;
    pl.useAccum = pl.chunks > 1 || prog || (outs && outs->accum());
    pl.planes = pl.mode == OutMode::Aov ? 2 : 1;
    const bool list = pl.mode == OutMode::List;
    pl.granule = list ? 32 : 4;
    pl.units = list ? listLen : ownedRows;
    pl.unitWidth = list ? 1 : localWidth;
    return pl;
}

// The accumulation buffer of a plan: the chunk sums of one band of units, the band sized so that the buffer stays within a fixed
// budget (a whole 1080p x 64 spp frame, 32 chunks per pixel, is 1.06 GB; the budget is 4 GB).  Allocation happens here so that
// callers can do it before their timed window starts.
static int prepare_accum(tmpt_scene* s, const RenderPlan& pl, cudaStream_t st, int* outBandUnits) {
    int band = pl.units;
    if (pl.useAccum && pl.units > 0) {
        const size_t unitBytes = (size_t)pl.unitWidth * pl.chunks * pl.planes * sizeof(float4), budget = (size_t)4 << 30;
        band = (int)std::min<size_t>((size_t)pl.units, std::max<size_t>(pl.granule, (budget / unitBytes) & ~(size_t)(pl.granule - 1)));
        const size_t need = (size_t)band * unitBytes;
        CU_TRY(s->d_accum.grow(need / sizeof(float4), st));
    }
    if (outBandUnits) *outBandUnits = band;
    return TMPT_OK;
}

// k_render or k_render_paths for this frame?  TMPT_RENDER_PATHS=0 / 1 forces the choice (tests, A/B).  Otherwise k_probe_paths
// decides: a frame whose first diffuse bounce escapes to the sky more than kOpenFrame of the time is an "open" frame.  The probe
// runs when camera or frame size change, on the frame's stream, WITHOUT stalling the host: its result is picked up by the first
// later frame that finds it complete, so a moving camera renders with a decision that is a frame or two old (both kernels produce
// the same bytes, the choice is about speed only).  Only the very first frame of a scene waits for its probe.
static constexpr float kOpenFrame = 0.15f;
static int choose_render_kernel(tmpt_scene* s, const tmpt_camera* camera, const integ::Camera& cam, int width, int height, cudaStream_t st,
                                bool* usePaths) {
    static const int pathsEnv = getenv("TMPT_RENDER_PATHS") ? atoi(getenv("TMPT_RENDER_PATHS")) : -1;
    *usePaths = pathsEnv > 0;
    if (pathsEnv >= 0 || s->triCount == 0) return TMPT_OK;
    if (!s->probeDone) {
        CU_TRY(s->d_probe.grow(4, st));
        CU_TRY(s->h_probe.grow(4, st));
        CU_TRY(cudaEventCreateWithFlags(&s->probeDone, cudaEventDisableTiming));
    }
    auto consume = [&]() {
        s->probeEscape = s->h_probe.p[1] ? (float)s->h_probe.p[2] / (float)s->h_probe.p[1] : 1.0f;  // (no camera ray hits anything: open)
        s->probeUsePaths = s->probeEscape > kOpenFrame ? 1 : 0;
        s->probePending = false;
    };
    if (s->probePending && cudaEventQuery(s->probeDone) == cudaSuccess) consume();
    if (!s->probePending && (s->probeUsePaths < 0 || s->probeW != width || s->probeH != height || memcmp(&s->probeCam, camera, sizeof(tmpt_camera)) != 0)) {
        CU_TRY(cudaMemsetAsync(s->d_probe.p, 0, 4 * sizeof(unsigned int), st));
        LAUNCH(k_probe_paths, 32, 128, 0, st, s->view, cam, width, height, s->d_probe.p);
        CU_TRY(cudaMemcpyAsync(s->h_probe.p, s->d_probe.p, 4 * sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaEventRecord(s->probeDone, st));
        s->probeCam = *camera; s->probeW = width; s->probeH = height;
        s->probePending = true;
        if (s->probeUsePaths < 0) { CU_TRY(cudaEventSynchronize(s->probeDone)); consume(); }
    }
    *usePaths = s->probeUsePaths == 1;
    return TMPT_OK;
}

extern "C" int tmpt_render_kernel_choice(const tmpt_scene* s, int* kernel, float* escapeFraction) {
    if (!s) return tmpt::fail(TMPT_ERR_ARG, "tmpt_render_kernel_choice: NULL scene");
    if (kernel) *kernel = s->lastUsedPaths;
    if (escapeFraction) *escapeFraction = s->probeEscape;
    return TMPT_OK;
}

// A render kernel as the host launches it.
struct RenderKernel {
    void (*fn)(const RenderParams);
    int threads;
    size_t smem;  // dynamic shared memory: k_render's traversal stacks, kSStack entries x 8 bytes per thread
};
template <OutMode MODE>
static RenderKernel shipped_render_kernel(bool paths, int cfg, bool far) {
    constexpr size_t b = kSStack * sizeof(unsigned long long);
    if (paths) return cfg == 3 ? RenderKernel{k_render_paths<1024, 1, 8, MODE>, 1024, 0} : RenderKernel{k_render_paths<256, 4, 8, MODE>, 256, 0};
    if (far) return {k_render<false, 256, 4, kSStack, true, MODE>, 256, 256 * b};
    if (cfg == 3) return {k_render<false, 1024, 1, kSStack, false, MODE>, 1024, 1024 * b};
    if (cfg == 2) return {k_render<false, 512, 2, kSStack, false, MODE>, 512, 512 * b};
    return {k_render<false, 256, 4, kSStack, false, MODE>, 256, 256 * b};
}
// The shipped render instantiation of a launch: k_render_paths (configurations 1 = 256 x 4 and 3 = 1024 x 1) or k_render
// (1, 2 = 512 x 2, 3, and the far-camera one at 256 x 4) in the launch's output mode, or the instrumented pass (frame mode only).
static RenderKernel render_kernel(OutMode mode, bool paths, int cfg, bool far, bool stats) {
    if (stats) return {k_render<true, 256, 4, kSStack>, 256, 256 * kSStack * sizeof(unsigned long long)};
    switch (mode) {
        case OutMode::Aov: return shipped_render_kernel<OutMode::Aov>(paths, cfg, far);
        case OutMode::List: return shipped_render_kernel<OutMode::List>(paths, cfg, far);
        default: return shipped_render_kernel<OutMode::Frame>(paths, cfg, far);
    }
}
// *perSM = the kernel's CTAs per SM, unless already known (>= 0).  The query first allows the kernel's dynamic shared memory beyond
// the default 48 KB (a per-device function attribute: set on every launch path, it costs microseconds); launch_render queries
// every render kernel before its first launch.
static int render_blocks_per_sm(const RenderKernel& k, int* perSM) {
    if (*perSM >= 0) return TMPT_OK;
    if (k.smem > 48 * 1024) CU_TRY(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k.smem));
    CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(perSM, k.fn, k.threads, k.smem));
    return TMPT_OK;
}

static int launch_render(const tmpt_scene* cs, const tmpt_camera* camera, int width, int height, int spp, int stripeRows, int rank, int world,
                         uint8_t* outStripes, uint8_t* frame, unsigned long long* rayCountDev, cudaStream_t st,
                         unsigned long long* statsDev = nullptr, const ProgressivePass* prog = nullptr, const FrameOutputs* outs = nullptr,
                         int listLen = 0) {
    tmpt_scene* s = const_cast<tmpt_scene*>(cs);  // scratch buffers only; the scene data is immutable
    RenderParams p;
    p.sc = s->view;
    static_assert(sizeof(integ::Camera) == sizeof(tmpt_camera), "camera layout");
    memcpy(&p.cam, camera, sizeof p.cam);
    p.lightDir = host_light_dir();
    p.width = width; p.height = height;
    p.stripeRows = stripeRows; p.rank = rank; p.world = world;
    p.ownedRows = tmpt_stripe_rows(height, stripeRows, rank, world);
    p.localWidth = tmpt_local_width(width, stripeRows, world);
    p.tilesX = div_up(p.localWidth, 8);
    const RenderPlan pl = plan_render(p.localWidth, p.ownedRows, spp, prog, outs, listLen);
    p.spp = pl.spp; p.chunks = pl.chunks; p.chunk0 = pl.chunk0; p.chunkLen = pl.chunkLen; p.useAccum = pl.useAccum ? 1 : 0;
    p.radiance = outs ? outs->radiance : nullptr;
    p.normal = outs ? outs->normal : nullptr;
    p.depth = outs ? outs->depth : nullptr;
    p.triangle = outs ? outs->triangle : nullptr;
    p.sumBuf = prog ? prog->sum : nullptr;
    p.outStripes = (uchar4*)outStripes;
    p.frame = (uchar4*)frame;
    p.rayCount = rayCountDev;
    p.tileCounter = s->d_tileCounter.p;
    p.laneCounter = s->d_fetchCounter.p;
    p.stats = statsDev;
    p.accum = nullptr;
    p.list = nullptr;
    p.listLen = 0;
    if (pl.units == 0) return TMPT_OK;  // (an adaptive pass with an empty list traces nothing: the kernel choice stays the last frame's)
    int band = 0;
    TRY(prepare_accum(s, pl, st, &band));
    p.accum = s->d_accum.p;
    // 32 warps per SM at 64 registers (sweep in profiles/r1_tuning_sweeps.txt: 24 warps at 77 registers is 10 % slower, 40
    // warps at 48 registers spills and is 3 % slower), as ONE 1024-thread CTA per SM when the band has work for every SM
    // several times over (+1.6 % over four 256-thread CTAs: 5016 vs 4937 Mrays/s), as 256-thread CTAs for small frames, whose
    // few hundred warp items would otherwise land on a few SMs.  TMPT_RENDER_CFG (tuning): 1 = 256 x 4, 2 = 512 x 2, 3 = 1024 x 1.
    static const int cfgEnv = getenv("TMPT_RENDER_CFG") ? atoi(getenv("TMPT_RENDER_CFG")) : 0;
    // TMPT_RENDER_KERNEL (experiments build only): 0 = lockstep lanes (k_render), 1.. = per-lane ray regeneration with gate sizes (TA, TB)
    static const int rk = getenv("TMPT_RENDER_KERNEL") ? atoi(getenv("TMPT_RENDER_KERNEL")) : 0;
#if !TMPT_EXPERIMENTS
    if (rk > 0) return tmpt::fail(TMPT_ERR_ARG, "TMPT_RENDER_KERNEL is set, but this library was built without -DTMPT_EXPERIMENTS=1");
#endif
    if (pl.mode == OutMode::Aov && (statsDev || rk > 0 || (TMPT_TUNE_CFG && cfgEnv >= 4)))
        return tmpt::fail(TMPT_ERR_ARG, "render: AOV outputs need the shipped render kernels (no instrumented pass, TMPT_RENDER_KERNEL or tuning configuration)");
    if (pl.mode == OutMode::List && (rk > 0 || (TMPT_TUNE_CFG && cfgEnv >= 4)))
        return tmpt::fail(TMPT_ERR_ARG, "render: adaptive passes need the shipped render kernels (no TMPT_RENDER_KERNEL or tuning configuration)");
    // (lens offsets are at most lensRadius from the origin: add it to the test)
    const bool farCamera = s->view.farLimit > 0.0f &&
        std::max(std::max(std::fabs(camera->origin[0]), std::fabs(camera->origin[1])), std::fabs(camera->origin[2])) + std::fabs(camera->lensRadius) >
            0.5f * s->view.farLimit;
    bool usePaths = false;  // (the instrumented pass and far cameras stay with k_render)
    if (!statsDev && !farCamera && rk == 0 && cfgEnv == 0) TRY(choose_render_kernel(s, camera, p.cam, width, height, st, &usePaths));
    if (!statsDev) s->lastUsedPaths = usePaths ? 1 : 0;
    int perSM[4] = {-1, -1, -1, -1};  // CTAs per SM of configuration 1..3's kernel, queried when a band first needs it
    for (int b0 = 0; b0 < pl.units; b0 += band) {
        const int here = std::min(band, pl.units - b0);
        if (pl.mode == OutMode::List) {
            p.list = s->d_adList.p + b0;
            p.listLen = here;
            p.numTiles = div_up(here, 32);
        } else {
            p.bandRow0 = b0;
            p.bandRows = here;
            p.numTiles = p.tilesX * div_up(here, 4);
        }
        const long long items = (long long)p.numTiles * p.chunks;
        if (items >= 0xFFFFFFFFll) return tmpt::fail(TMPT_ERR_ARG, "render: too many work items in one band");
        CU_TRY(cudaMemsetAsync(s->d_tileCounter.p, 0, sizeof(uint32_t), st));
#if TMPT_TUNE_CFG
        if (cfgEnv >= 4 && cfgEnv <= 8) {  // tuning only (-DTMPT_TUNE_CFG=1): other resident-warp / register-budget points
            if (cfgEnv == 4) LAUNCH((k_render<false, 768, 1, 0>), s->smCount, 768, 0, st, p);           // 24 warps, 85 registers
            else if (cfgEnv == 5) LAUNCH((k_render<false, 576, 2, 0>), 2 * s->smCount, 576, 0, st, p);  // 36 warps, 56 registers
            else if (cfgEnv == 6) LAUNCH((k_render<false, 640, 2, 0>), 2 * s->smCount, 640, 0, st, p);  // 40 warps, 48 registers
            else if (cfgEnv == 7) LAUNCH((k_render<false, 896, 1, 0>), s->smCount, 896, 0, st, p);      // 28 warps, 72 registers
            else LAUNCH((k_render<false, 384, 3, 0>), 3 * s->smCount, 384, 0, st, p);                    // 36 warps, 56 registers, three CTAs
        } else
#endif
#if TMPT_EXPERIMENTS
        if (rk > 0 && !statsDev) {
            CU_TRY(cudaMemsetAsync(s->d_fetchCounter.p, 0, sizeof(unsigned long long), st));
            int perSMr = 0;
#define REGEN_CASE(V, TA, TB)                                                                                        \
            if (rk == V) {                                                                                           \
                CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSMr, k_render_regen<false, 256, 4, TA, TB>, 256, 0)); \
                const int gridR = (int)std::min<long long>((long long)s->smCount * std::max(perSMr, 1), (items * 32 + 255) / 256); \
                LAUNCH((k_render_regen<false, 256, 4, TA, TB>), gridR, 256, 0, st, p);                                 \
            } else
            REGEN_CASE(1, 8, 4) REGEN_CASE(2, 4, 2) REGEN_CASE(3, 12, 6) REGEN_CASE(4, 16, 4)
#undef REGEN_CASE
#define PATHS_CASE(V, T, MB, GT)                                                                                       \
            if (rk == V) {                                                                                           \
                CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSMr, k_render_paths<T, MB, GT>, T, 0));     \
                const int gridR = (int)std::min<long long>((long long)s->smCount * std::max(perSMr, 1), (items * 32 + T - 1) / T); \
                LAUNCH((k_render_paths<T, MB, GT>), gridR, T, 0, st, p);                                              \
            } else
            PATHS_CASE(5, 256, 4, 1) PATHS_CASE(6, 256, 4, 8) PATHS_CASE(7, 256, 4, 16) PATHS_CASE(8, 1024, 1, 8) PATHS_CASE(9, 1024, 1, 16)
#undef PATHS_CASE
            return tmpt::fail(TMPT_ERR_ARG, "TMPT_RENDER_KERNEL=%d: no such render kernel", rk);
        } else
#endif
        {
            int cfg = (statsDev || rk > 0 || farCamera) ? 1 : cfgEnv;
            if (cfg <= 0) {
                TRY(render_blocks_per_sm(render_kernel(pl.mode, usePaths, 3, false, false), &perSM[3]));
                cfg = items >= (long long)s->smCount * 32 * 8 && perSM[3] > 0 ? 3 : 1;
            } else if (cfg != 2 && cfg != 3) {
                cfg = 1;
            }
            const RenderKernel k = render_kernel(pl.mode, usePaths, cfg, farCamera, statsDev != nullptr);
            TRY(render_blocks_per_sm(k, &perSM[cfg]));
            if (usePaths) CU_TRY(cudaMemsetAsync(s->d_fetchCounter.p, 0, sizeof(unsigned long long), st));  // one (pixel, chunk) item per lane
            // every SM's resident CTAs, or fewer when a warp per (tile, chunk) item (k_render) or a lane per (pixel, chunk) item
            // (k_render_paths, 32 per tile) needs fewer
            const int warps = k.threads / 32;
            const int grid = (int)std::min<long long>((long long)s->smCount * std::max(perSM[cfg], 1), (items + warps - 1) / warps);
            LAUNCH(k.fn, grid, k.threads, k.smem, st, p);
        }
        if (pl.mode == OutMode::List)
            LAUNCH(k_resolve_adaptive, div_up(here, 256), 256, 0, st, p, prog->sum, s->d_adN.p, s->d_adStat.p, prog->adaptive->tolerance,
                   prog->adaptive->minChunks, s->d_adActive.p);
        else if (p.useAccum && pl.mode == OutMode::Aov) LAUNCH(k_resolve<true>, div_up((long long)here * p.localWidth, 256), 256, 0, st, p, here);
        else if (p.useAccum) LAUNCH(k_resolve<false>, div_up((long long)here * p.localWidth, 256), 256, 0, st, p, here);
    }
    CU_TRY(cudaGetLastError());
    return TMPT_OK;
}

// The reference's own frame-size range (main.cpp:263-279), shared by every entry point that takes a frame size.
static bool frame_size_ok(int width, int height) { return width >= 1 && width <= 10000 && height >= 1 && height <= 10000; }

static int check_render_args(const tmpt_scene* s, const tmpt_camera* camera, int width, int height, int spp) {
    if (!s || !camera) return tmpt::fail(TMPT_ERR_ARG, "render: NULL scene / camera");
    if (!frame_size_ok(width, height) || spp < 1 || spp > 1024)
        return tmpt::fail(TMPT_ERR_ARG, "render: width %d height %d spp %d out of range", width, height, spp);
    return TMPT_OK;
}

// A float parameter that must be finite and > 0 (or >= 0 when zeroOk); NaN fails both comparisons.
static int check_finite(const char* fn, const char* name, float v, bool zeroOk) {
    if ((zeroOk ? v >= 0.0f : v > 0.0f) && v <= 3.4028235e38f) return TMPT_OK;
    return tmpt::fail(TMPT_ERR_ARG, "%s: %s %g is not a finite value %s 0", fn, name, (double)v, zeroOk ? ">=" : ">");
}

extern "C" int tmpt_render_stripes(const tmpt_scene* s, const tmpt_camera* camera, int width, int height, int spp, int stripeRows, int rank,
                                   int worldSize, uint8_t* outStripes, uint8_t* peerFrame, uint64_t* rayCountDev, void* stream) {
    TRY(check_render_args(s, camera, width, height, spp));
    if (stripeRows < 0 || worldSize < 1 || rank < 0 || rank >= worldSize || (!outStripes && !peerFrame) || !rayCountDev)
        return tmpt::fail(TMPT_ERR_ARG, "tmpt_render_stripes: bad stripe arguments");
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_render_stripes: cudaSetDevice(%d) failed", s->device);
    return launch_render(s, camera, width, height, spp, stripeRows, rank, worldSize, outStripes, peerFrame,
                         (unsigned long long*)rayCountDev, stream ? (cudaStream_t)stream : s->stream);
}

// The checks the output entry points share: a NULL `out`, no buffer requested or a bad `mem` is an argument error.
static int check_outputs(const char* fn, const tmpt_outputs* out, int mem) {
    if (!out) return tmpt::fail(TMPT_ERR_ARG, "%s: out is NULL", fn);
    if (!out->rgba && !out->radiance && !out->normal && !out->depth && !out->triangle) return tmpt::fail(TMPT_ERR_ARG, "%s: no output requested", fn);
    if (mem != TMPT_HOST && mem != TMPT_DEVICE) return tmpt::fail(TMPT_ERR_ARG, "%s: mem %d", fn, mem);
    return TMPT_OK;
}

// The buffers rgba, radiance, normal, depth, triangle of a call as the kernels see them.  With TMPT_HOST each buffer the caller gave
// is staged in the scene's device scratch (one buffer per kind, kept with the scene), and the caller copies it in or out inside its
// timed window; with TMPT_DEVICE the kernels use the caller's buffers.
struct Staging {
    void* user[5];
    void* dev[5] = {};
    size_t bytes[5] = {};
    // frame: the kernels write an RGBA frame even when the caller asks for none (into the scene's scratch frame)
    int stage(tmpt_scene* s, size_t pixels, int mem, bool frame, cudaStream_t st) {
        const size_t sizes[5] = {pixels * 4, pixels * sizeof(float4), pixels * sizeof(float4), pixels * sizeof(float), pixels * sizeof(int32_t)};
        for (int k = 0; k < 5; ++k) {
            dev[k] = user[k];
            bytes[k] = sizes[k];
            if ((mem == TMPT_HOST && user[k]) || (k == 0 && frame && !user[k])) {
                CU_TRY(s->staged[k].grow(sizes[k], st));
                dev[k] = s->staged[k].p;
            }
        }
        return TMPT_OK;
    }
    int copy(int mem, cudaMemcpyKind dir, cudaStream_t st) const {  // (TMPT_DEVICE: nothing to copy)
        for (int k = 0; k < 5; ++k)
            if (mem == TMPT_HOST && user[k])
                CU_TRY(dir == cudaMemcpyHostToDevice ? cudaMemcpyAsync(dev[k], user[k], bytes[k], dir, st) : cudaMemcpyAsync(user[k], dev[k], bytes[k], dir, st));
        return TMPT_OK;
    }
};

// The end of a timed window that began with s->ev0 on `st`: records s->ev1, then (outside the window) copies the device counter
// `countDev` to *count if given, waits for the stream and returns the window's length in *seconds.
static int end_timed_window(tmpt_scene* s, cudaStream_t st, double* seconds, const unsigned long long* countDev = nullptr,
                            unsigned long long* count = nullptr) {
    CU_TRY(cudaEventRecord(s->ev1, st));
    if (countDev) CU_TRY(cudaMemcpyAsync(count, countDev, sizeof *count, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    float ms = 0.0f;
    CU_TRY(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    if (seconds) *seconds = (double)ms * 1.0e-3;
    return TMPT_OK;
}

// One single-GPU frame (prog == nullptr) or progressive pass into the buffers `out` names: with TMPT_HOST each requested buffer is
// staged in the scene's device scratch and copied out inside the timed window; the kernels always write an RGBA frame (the scene's
// scratch frame when the caller asks for none).  An adaptive pass reports into *adOut.  The caller holds hostCallMutex and the device.
static int render_frame(tmpt_scene* s, const tmpt_camera* camera, int width, int height, int spp, int mem, const tmpt_outputs* out,
                        const ProgressivePass* prog, cudaStream_t st, uint64_t* rayCount, double* seconds, AdaptiveResult* adOut = nullptr) {
    const size_t pixels = (size_t)width * height;
    Staging g{{out->rgba, out->radiance, out->normal, out->depth, out->triangle}};
    TRY(g.stage(s, pixels, mem, true, st));
    FrameOutputs f;
    f.radiance = (float4*)g.dev[1]; f.normal = (float4*)g.dev[2]; f.depth = (float*)g.dev[3]; f.triangle = (int32_t*)g.dev[4];
    const AdaptivePass* ad = prog ? prog->adaptive : nullptr;
    int32_t* samples = ad ? ad->samples : nullptr;  // (device buffer)
    if (samples && mem == TMPT_HOST) {
        CU_TRY(s->d_samples.grow(pixels, st));
        samples = s->d_samples.p;
    }
    // (scratch allocation stays outside the timed window; an adaptive pass allocates for a list of every pixel)
    TRY(prepare_accum(s, plan_render(width, height, spp, prog, &f, (int)pixels), st, nullptr));
    CU_TRY(cudaEventRecord(s->ev0, st));
    CU_TRY(cudaMemsetAsync(s->d_rayCount.p, 0, sizeof(unsigned long long), st));
    uint32_t listLen = 0;
    if (ad) {  // select + compact: the active list and its length (one small copy)
        const int tilesX = div_up(width, 8);
        const long long slots = (long long)tilesX * div_up(height, 4) * 32;
        const int nBlocks = div_up(slots, kScanBlock);
        LAUNCH(k_adaptive_select, div_up(slots, 256), 256, 0, st, s->d_adN.p, s->d_adStat.p, width, height, tilesX, slots, ad->tolerance, ad->minChunks,
               s->d_adFlags.p);
        LAUNCH(k_scan_totals, nBlocks, kScanBlock, 0, st, s->d_adFlags.p, slots, s->d_adTotals.p);
        LAUNCH(k_scan_of_totals, 1, kScanBlock, 0, st, s->d_adTotals.p, nBlocks, s->d_adTotals.p + nBlocks);
        LAUNCH(k_scan_apply, nBlocks, kScanBlock, 0, st, s->d_adFlags.p, slots, s->d_adTotals.p, s->d_adTotals.p + nBlocks, s->d_adOffs.p);
        LAUNCH(k_adaptive_compact, div_up(slots, 256), 256, 0, st, s->d_adFlags.p, s->d_adOffs.p, s->d_adN.p, width, tilesX, slots, s->d_adList.p);
        CU_TRY(cudaMemsetAsync(s->d_adActive.p, 0, sizeof(unsigned int), st));
        CU_TRY(cudaMemcpyAsync(&listLen, s->d_adTotals.p + nBlocks, sizeof listLen, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
    }
    TRY(launch_render(s, camera, width, height, spp, height, 0, 1, nullptr, (uint8_t*)g.dev[0], s->d_rayCount.p, st, nullptr, prog, &f, (int)listLen));
    if (ad) LAUNCH(k_adaptive_write, div_up((long long)pixels, 256), 256, 0, st, prog->sum, s->d_adN.p, (long long)pixels, (uchar4*)g.dev[0], f.radiance,
                   samples);
    TRY(g.copy(mem, cudaMemcpyDeviceToHost, st));
    if (samples && mem == TMPT_HOST) CU_TRY(cudaMemcpyAsync(ad->samples, samples, pixels * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (ad) {
        adOut->listLen = (int)listLen;
        CU_TRY(cudaMemcpyAsync(adOut->counters, s->d_adActive.p, sizeof adOut->counters, cudaMemcpyDeviceToHost, st));
    }
    unsigned long long rays = 0;
    TRY(end_timed_window(s, st, seconds, s->d_rayCount.p, &rays));
    if (rayCount) *rayCount = rays;
    return TMPT_OK;
}

extern "C" int tmpt_render_outputs(const tmpt_scene* cs, const tmpt_camera* camera, int width, int height, int spp, int mem,
                                   const tmpt_outputs* out, uint64_t* rayCount, double* seconds, void* stream) {
    TRY(check_render_args(cs, camera, width, height, spp));
    TRY(check_outputs("tmpt_render_outputs", out, mem));
    tmpt_scene* s = const_cast<tmpt_scene*>(cs);  // scratch buffers only; the scene data is immutable
    std::lock_guard<std::mutex> lock(s->hostCallMutex);  // concurrent callers take turns (the reference's HitScene is lock-free const; a frame here owns the scene's scratch)
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_render_outputs: cudaSetDevice(%d) failed", s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    TRY(render_frame(s, camera, width, height, spp, mem, out, nullptr, st, rayCount, seconds));
    return check_status(s, st);
}

extern "C" int tmpt_render(const tmpt_scene* cs, const tmpt_camera* camera, int width, int height, int spp, int mem, uint8_t* rgba,
                           uint64_t* rayCount, double* seconds, void* stream) {
    if (!rgba) return tmpt::fail(TMPT_ERR_ARG, "tmpt_render: rgba is NULL");
    tmpt_outputs out{};
    out.rgba = rgba;
    return tmpt_render_outputs(cs, camera, width, height, spp, mem, &out, rayCount, seconds, stream);
}

// Progressive rendering (beyond the reference): the running per-pixel sums live with the scene.
extern "C" int tmpt_progressive_begin(tmpt_scene* s, int width, int height) {
    if (!s) return tmpt::fail(TMPT_ERR_ARG, "tmpt_progressive_begin: NULL scene");
    if (!frame_size_ok(width, height)) return tmpt::fail(TMPT_ERR_ARG, "tmpt_progressive_begin: %d x %d out of range", width, height);
    std::lock_guard<std::mutex> lock(s->hostCallMutex);
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_progressive_begin: cudaSetDevice(%d) failed", s->device);
    const size_t pixels = (size_t)width * height;
    CU_TRY(s->d_sum.grow(pixels, s->stream));
    CU_TRY(cudaMemsetAsync(s->d_sum.p, 0, pixels * sizeof(float4), s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    s->progW = width; s->progH = height; s->progChunks = 0; s->progAdaptive = -1;
    return TMPT_OK;
}

// The checks of both pass kinds that do not read the scene: camera and outputs (passes have no AOV buffers).
static int check_pass_args(const char* fn, const tmpt_scene* s, const tmpt_camera* camera, const tmpt_outputs* out, int mem) {
    if (!s || !camera) return tmpt::fail(TMPT_ERR_ARG, "%s: NULL scene / camera", fn);
    TRY(check_outputs(fn, out, mem));
    if (out->normal || out->depth || out->triangle) return tmpt::fail(TMPT_ERR_ARG, "%s: passes produce rgba and radiance only (no running AOV sums)", fn);
    return TMPT_OK;
}
// The session's checks (the caller holds hostCallMutex): a begun session whose passes are of this kind, with room for nChunks
// more chunks (adaptive: progChunks is the session's largest n; a pixel is traced at most once per pass).
static int check_pass_session(const char* fn, const tmpt_scene* s, int nChunks, bool adaptive) {
    if (s->progChunks < 0) return tmpt::fail(TMPT_ERR_ARG, "%s: call tmpt_progressive_begin first", fn);
    if (s->progAdaptive == (adaptive ? 0 : 1))
        return tmpt::fail(TMPT_ERR_ARG, "%s: this session's passes are %s (tmpt_progressive_begin starts a new one)", fn, adaptive ? "uniform" : "adaptive");
    if (nChunks < 1 || nChunks > 128 || (long long)(s->progChunks + nChunks) * integ::kMaxChunkSamples > (1 << 24))
        return tmpt::fail(TMPT_ERR_ARG, "%s: %d chunks after %d", fn, nChunks, s->progChunks);
    return TMPT_OK;
}

extern "C" int tmpt_progressive_pass_outputs(tmpt_scene* s, const tmpt_camera* camera, int nChunks, int mem, const tmpt_outputs* out,
                                             uint64_t* rayCount, double* seconds, int* samplesSoFar, void* stream) {
    static const char* fn = "tmpt_progressive_pass_outputs";
    TRY(check_pass_args(fn, s, camera, out, mem));
    std::lock_guard<std::mutex> lock(s->hostCallMutex);
    TRY(check_pass_session(fn, s, nChunks, false));
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "%s: cudaSetDevice(%d) failed", fn, s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    const ProgressivePass pass{s->progChunks, nChunks, s->d_sum.p};
    TRY(render_frame(s, camera, s->progW, s->progH, 0, mem, out, &pass, st, rayCount, seconds));
    s->progChunks += nChunks;
    s->progAdaptive = 0;
    if (samplesSoFar) *samplesSoFar = s->progChunks * integ::kMaxChunkSamples;
    return check_status(s, st);
}

// The per-pixel state of adaptive passes, for a progW x progH session: zeroed with the session's first adaptive pass.
static int begin_adaptive(tmpt_scene* s, cudaStream_t st) {
    const int tilesX = div_up(s->progW, 8);
    const size_t slots = (size_t)tilesX * div_up(s->progH, 4) * 32, pixels = (size_t)s->progW * s->progH;
    CU_TRY(s->d_adN.grow(slots, st));
    CU_TRY(s->d_adStat.grow(slots, st));
    CU_TRY(s->d_adFlags.grow(slots, st));
    CU_TRY(s->d_adOffs.grow(slots + 1, st));
    CU_TRY(s->d_adTotals.grow(slots / kScanBlock + 2, st));
    CU_TRY(s->d_adList.grow(slots, st));
    CU_TRY(s->d_adActive.grow(2, st));
    CU_TRY(cudaMemsetAsync(s->d_adN.p, 0, pixels * sizeof(uint32_t), st));
    CU_TRY(cudaMemsetAsync(s->d_adStat.p, 0, pixels * sizeof(float2), st));
    CU_TRY(cudaMemsetAsync(s->d_adActive.p, 0, 2 * sizeof(unsigned int), st));
    return TMPT_OK;
}

extern "C" int tmpt_progressive_pass_adaptive(tmpt_scene* s, const tmpt_camera* camera, int nChunks, const tmpt_adaptive* params, int mem,
                                              const tmpt_outputs* out, int32_t* samples, uint64_t* rayCount, double* seconds,
                                              int64_t* activePixels, void* stream) {
    static const char* fn = "tmpt_progressive_pass_adaptive";
    TRY(check_pass_args(fn, s, camera, out, mem));
    if (!params) return tmpt::fail(TMPT_ERR_ARG, "%s: params is NULL", fn);
    TRY(check_finite(fn, "tolerance", params->tolerance, true));
    if (params->minChunks < 2 || params->minChunks > (1 << 21)) return tmpt::fail(TMPT_ERR_ARG, "%s: minChunks %d out of range 2..2^21", fn, params->minChunks);
    if (nChunks < 1 || nChunks > 128) return tmpt::fail(TMPT_ERR_ARG, "%s: nChunks %d out of range 1..128", fn, nChunks);
    std::lock_guard<std::mutex> lock(s->hostCallMutex);
    TRY(check_pass_session(fn, s, nChunks, true));
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "%s: cudaSetDevice(%d) failed", fn, s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (s->progAdaptive < 0) TRY(begin_adaptive(s, st));
    const AdaptivePass ad{params->tolerance, params->minChunks, samples};
    const ProgressivePass pass{0, nChunks, s->d_sum.p, &ad};
    AdaptiveResult res;
    TRY(render_frame(s, camera, s->progW, s->progH, 0, mem, out, &pass, st, rayCount, seconds, &res));
    s->progAdaptive = 1;
    if (res.listLen > 0) s->progChunks = (int)res.counters[1];
    if (activePixels) *activePixels = (int64_t)res.counters[0];
    return check_status(s, st);
}

extern "C" int tmpt_progressive_pass(tmpt_scene* s, const tmpt_camera* camera, int nChunks, int mem, uint8_t* rgba, uint64_t* rayCount,
                                     double* seconds, int* samplesSoFar, void* stream) {
    if (!s || !camera || !rgba) return tmpt::fail(TMPT_ERR_ARG, "tmpt_progressive_pass: NULL scene / camera / rgba");
    tmpt_outputs out{};
    out.rgba = rgba;
    return tmpt_progressive_pass_outputs(s, camera, nChunks, mem, &out, rayCount, seconds, samplesSoFar, stream);
}

// One process, several devices: stripes of rank i on scenes[i], pixels stored into device 0's frame by peer access.
// The denoiser (beyond the reference): include/tmpt.h documents the filter; denoise.cuh holds its arithmetic.
extern "C" int tmpt_denoise(tmpt_scene* s, int width, int height, int mem, const tmpt_outputs* in, const tmpt_denoise_params* params,
                            const tmpt_outputs* out, double* seconds, void* stream) {
    static const char* fn = "tmpt_denoise";
    if (!s) return tmpt::fail(TMPT_ERR_ARG, "%s: NULL scene", fn);
    if (!in) return tmpt::fail(TMPT_ERR_ARG, "%s: in is NULL", fn);
    if (!params) return tmpt::fail(TMPT_ERR_ARG, "%s: params is NULL", fn);
    if (!out) return tmpt::fail(TMPT_ERR_ARG, "%s: out is NULL", fn);
    if (!in->radiance || !in->normal || !in->depth) return tmpt::fail(TMPT_ERR_ARG, "%s: in->radiance, in->normal and in->depth are required", fn);
    if (!out->rgba && !out->radiance) return tmpt::fail(TMPT_ERR_ARG, "%s: no output requested", fn);
    if (out->normal || out->depth || out->triangle) return tmpt::fail(TMPT_ERR_ARG, "%s: out takes rgba and radiance only", fn);
    if (mem != TMPT_HOST && mem != TMPT_DEVICE) return tmpt::fail(TMPT_ERR_ARG, "%s: mem %d", fn, mem);
    if (!frame_size_ok(width, height)) return tmpt::fail(TMPT_ERR_ARG, "%s: %d x %d out of range", fn, width, height);
    if (params->iterations < 0 || params->iterations > dn::kMaxIterations)
        return tmpt::fail(TMPT_ERR_ARG, "%s: iterations %d out of range 0..%d", fn, params->iterations, dn::kMaxIterations);
    if (params->normalPowerLog2 < 0 || params->normalPowerLog2 > dn::kMaxNormalPowerLog2)
        return tmpt::fail(TMPT_ERR_ARG, "%s: normalPowerLog2 %d out of range 0..%d", fn, params->normalPowerLog2, dn::kMaxNormalPowerLog2);
    TRY(check_finite(fn, "sigmaLuminance", params->sigmaLuminance, false));
    TRY(check_finite(fn, "sigmaDepth", params->sigmaDepth, false));
    std::lock_guard<std::mutex> lock(s->hostCallMutex);
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "%s: cudaSetDevice(%d) failed", fn, s->device);
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    const size_t pixels = (size_t)width * height;
    // (scratch allocation stays outside the timed window; with TMPT_HOST an output radiance is staged where the input radiance is:
    // the prologue, or the copy, reads that before it is written)
    Staging gin{{nullptr, in->radiance, in->normal, in->depth, nullptr}}, gout{{out->rgba, out->radiance, nullptr, nullptr, nullptr}};
    TRY(gin.stage(s, pixels, mem, false, st));
    TRY(gout.stage(s, pixels, mem, false, st));
    uchar4* rgba = (uchar4*)gout.dev[0];
    float4* radiance = (float4*)gout.dev[1];
    if (params->iterations > 0) CU_TRY(s->d_denoise.grow(4 * pixels, st));
    CU_TRY(cudaEventRecord(s->ev0, st));
    TRY(gin.copy(mem, cudaMemcpyHostToDevice, st));
    const float4* rin = (const float4*)gin.dev[1];
    if (params->iterations == 0) {
        LAUNCH(k_denoise_copy, div_up((long long)pixels, 256), 256, 0, st, rin, (long long)pixels, rgba, radiance);
    } else {
        float4 *state[2] = {s->d_denoise.p, s->d_denoise.p + pixels}, *guideA = s->d_denoise.p + 2 * pixels, *guideB = s->d_denoise.p + 3 * pixels;
        const dim3 grid(div_up(width, kDenoiseBX), div_up(height, kDenoiseBY)), block(kDenoiseBX, kDenoiseBY);
        const dn::Params prm{params->iterations, params->sigmaLuminance, params->sigmaDepth, params->normalPowerLog2};
        LAUNCH(k_denoise_prep, grid, block, 0, st, rin, (const float4*)gin.dev[2], (const float*)gin.dev[3], width, height, state[0], guideA, guideB);
        for (int i = 0; i < params->iterations; ++i) {
            if (i + 1 < params->iterations)
                LAUNCH(k_denoise_atrous<false>, grid, block, 0, st, state[i & 1], state[(i + 1) & 1], guideA, guideB, width, height, 1 << i, prm,
                       nullptr, nullptr);
            else
                LAUNCH(k_denoise_atrous<true>, grid, block, 0, st, state[i & 1], nullptr, guideA, guideB, width, height, 1 << i, prm, rgba, radiance);
        }
    }
    CU_TRY(cudaGetLastError());
    TRY(gout.copy(mem, cudaMemcpyDeviceToHost, st));
    return end_timed_window(s, st, seconds);
}

extern "C" int tmpt_render_multi(tmpt_scene* const* scenes, int nScenes, const tmpt_camera* camera, int width, int height, int spp, uint8_t* rgba,
                                 uint64_t* rayCount, double* seconds) {
    if (!scenes || nScenes < 1 || nScenes > 64) return tmpt::fail(TMPT_ERR_ARG, "tmpt_render_multi: bad scene list");
    for (int i = 0; i < nScenes; ++i) {
        TRY(check_render_args(scenes[i], camera, width, height, spp));
        for (int j = 0; j < i; ++j)
            if (scenes[j]->device == scenes[i]->device) return tmpt::fail(TMPT_ERR_ARG, "tmpt_render_multi: two scenes on device %d", scenes[i]->device);
        if (scenes[i]->triCount != scenes[0]->triCount) return tmpt::fail(TMPT_ERR_ARG, "tmpt_render_multi: scenes are not replicas");
    }
    if (!rgba) return tmpt::fail(TMPT_ERR_ARG, "tmpt_render_multi: rgba is NULL");
    if (nScenes == 1) return tmpt_render(scenes[0], camera, width, height, spp, TMPT_HOST, rgba, rayCount, seconds, nullptr);
    tmpt_scene* s0 = scenes[0];
    const size_t bytes = (size_t)width * height * 4;
    int prev = 0;
    CU_TRY(cudaGetDevice(&prev));
    struct Restore { int d; ~Restore() { cudaSetDevice(d); } } restore{prev};
    // the frame lives on device 0; every other device needs peer access to it
    CU_TRY(cudaSetDevice(s0->device));
    CU_TRY(s0->staged[0].grow(bytes, s0->stream));
    std::vector<unsigned long long*> counters(nScenes);
    for (int i = 0; i < nScenes; ++i) {
        CU_TRY(cudaSetDevice(scenes[i]->device));
        if (i > 0) {
            int can = 0;
            CU_TRY(cudaDeviceCanAccessPeer(&can, scenes[i]->device, s0->device));
            if (!can) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_render_multi: device %d cannot access device %d", scenes[i]->device, s0->device);
            const cudaError_t e = cudaDeviceEnablePeerAccess(s0->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CU_TRY(e);
            cudaGetLastError();
        }
        counters[i] = scenes[i]->d_rayCount.p;
        CU_TRY(cudaMemsetAsync(counters[i], 0, sizeof(unsigned long long), scenes[i]->stream));
        TRY(prepare_accum(scenes[i], plan_render(tmpt_local_width(width, 0, nScenes), height, spp, nullptr, nullptr, 0), scenes[i]->stream,
                          nullptr));  // tile interleave
        CU_TRY(cudaStreamSynchronize(scenes[i]->stream));
    }
    // window: from the first launch to the frame in host memory (main.cpp:319-333)
    CU_TRY(cudaSetDevice(s0->device));
    CU_TRY(cudaStreamSynchronize(s0->stream));
    const auto t0 = std::chrono::steady_clock::now();
    for (int i = 0; i < nScenes; ++i) {
        CU_TRY(cudaSetDevice(scenes[i]->device));
        TRY(launch_render(scenes[i], camera, width, height, spp, 0, i, nScenes, nullptr, (uint8_t*)s0->staged[0].p, counters[i], scenes[i]->stream));
    }
    unsigned long long total = 0;
    for (int i = nScenes - 1; i >= 0; --i) {  // device 0 last: its stream then copies the completed frame out
        CU_TRY(cudaSetDevice(scenes[i]->device));
        unsigned long long rays = 0;
        CU_TRY(cudaMemcpyAsync(&rays, counters[i], sizeof rays, cudaMemcpyDeviceToHost, scenes[i]->stream));
        CU_TRY(cudaStreamSynchronize(scenes[i]->stream));
        total += rays;
    }
    CU_TRY(cudaMemcpyAsync(rgba, s0->staged[0].p, bytes, cudaMemcpyDeviceToHost, s0->stream));
    CU_TRY(cudaStreamSynchronize(s0->stream));
    const double sec = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (rayCount) *rayCount = total;
    if (seconds) *seconds = sec;
    for (int i = 0; i < nScenes; ++i) TRY(check_status(scenes[i], scenes[i]->stream));
    return TMPT_OK;
}

// ------------------------------------------------------------------------------------------
// C ABI: peer-writable frame (CUDA IPC)
// ------------------------------------------------------------------------------------------
extern "C" int tmpt_frame_alloc(int device, size_t bytes, void** outPtr, unsigned char outHandle[64]) {
    if (!outPtr || !outHandle || bytes == 0) return tmpt::fail(TMPT_ERR_ARG, "tmpt_frame_alloc: bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DeviceGuard guard(device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_frame_alloc: cudaSetDevice(%d) failed", device);
    void* p = nullptr;
    CU_TRY(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return tmpt::fail(TMPT_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
    memcpy(outHandle, &h, 64);
    *outPtr = p;
    return TMPT_OK;
}
extern "C" int tmpt_frame_open(int device, const unsigned char handle[64], void** outPtr) {
    if (!handle || !outPtr) return tmpt::fail(TMPT_ERR_ARG, "tmpt_frame_open: bad arguments");
    DeviceGuard guard(device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_frame_open: cudaSetDevice(%d) failed", device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CU_TRY(cudaIpcOpenMemHandle(outPtr, h, cudaIpcMemLazyEnablePeerAccess));
    return TMPT_OK;
}
extern "C" int tmpt_frame_close(int device, void* ptr) {
    if (!ptr) return TMPT_OK;
    DeviceGuard guard(device);
    CU_TRY(cudaIpcCloseMemHandle(ptr));
    return TMPT_OK;
}
extern "C" int tmpt_frame_free(int device, void* ptr) {
    if (!ptr) return TMPT_OK;
    DeviceGuard guard(device);
    CU_TRY(cudaFree(ptr));
    return TMPT_OK;
}

// Instrumented passes (same kernels compiled with counters; never part of a timed run).
extern "C" int tmpt_render_stats(const tmpt_scene* cs, const tmpt_camera* camera, int width, int height, int spp, uint64_t outStats[TMPT_STATS_COUNT]) {
    TRY(check_render_args(cs, camera, width, height, spp));
    if (!outStats) return tmpt::fail(TMPT_ERR_ARG, "tmpt_render_stats: outStats is NULL");
    tmpt_scene* s = const_cast<tmpt_scene*>(cs);
    std::lock_guard<std::mutex> lock(s->hostCallMutex);
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_render_stats: cudaSetDevice(%d) failed", s->device);
    cudaStream_t st = s->stream;
    const size_t bytes = (size_t)width * height * 4;
    DevBuf<uint8_t> frame;
    DevBuf<unsigned long long> stats;
    CU_TRY(frame.grow(bytes, st));
    CU_TRY(stats.grow(TMPT_STATS_COUNT, st));
    CU_TRY(cudaMemsetAsync(stats.p, 0, TMPT_STATS_COUNT * sizeof(unsigned long long), st));
    CU_TRY(cudaMemsetAsync(s->d_rayCount.p, 0, sizeof(unsigned long long), st));
    TRY(launch_render(s, camera, width, height, spp, height, 0, 1, nullptr, frame.p, s->d_rayCount.p, st, stats.p));
    CU_TRY(cudaMemcpyAsync(outStats, stats.p, TMPT_STATS_COUNT * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return TMPT_OK;
}

extern "C" int tmpt_hit_scene_stats(const tmpt_scene* s, const float* rays6Dev, int64_t nRays, float tMin, float tMax, int mode, uint64_t outStats[TMPT_STATS_COUNT]) {
    if (!s || !rays6Dev || nRays <= 0 || !outStats || (mode != TMPT_HIT_CLOSEST && mode != TMPT_HIT_ANY && mode != TMPT_HIT_SUN) ||
        (mode == TMPT_HIT_SUN && s->view.sun.n == 0))
        return tmpt::fail(TMPT_ERR_ARG, "tmpt_hit_scene_stats: bad arguments");
    DeviceGuard guard(s->device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_hit_scene_stats: cudaSetDevice(%d) failed", s->device);
    cudaStream_t st = s->stream;
    DevBuf<unsigned long long> stats;
    DevBuf<int> ids;
    CU_TRY(stats.grow(TMPT_STATS_COUNT, st));
    CU_TRY(ids.grow((size_t)nRays, st));
    CU_TRY(cudaMemsetAsync(stats.p, 0, TMPT_STATS_COUNT * sizeof(unsigned long long), st));
    const int B = 128;
    const int G = (int)std::min<long long>(div_up(nRays, B), (long long)s->smCount * 64);
    if (mode == TMPT_HIT_CLOSEST) LAUNCH((k_hit_scene<TMPT_HIT_CLOSEST, true>), G, B, 0, st, s->view, rays6Dev, (long long)nRays, tMin, tMax, ids.p, nullptr, nullptr, nullptr, stats.p);
    else if (mode == TMPT_HIT_SUN) LAUNCH((k_hit_scene<TMPT_HIT_SUN, true>), G, B, 0, st, s->view, rays6Dev, (long long)nRays, tMin, tMax, ids.p, nullptr, nullptr, nullptr, stats.p);
    else LAUNCH((k_hit_scene<TMPT_HIT_ANY, true>), G, B, 0, st, s->view, rays6Dev, (long long)nRays, tMin, tMax, ids.p, nullptr, nullptr, nullptr, stats.p);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(outStats, stats.p, TMPT_STATS_COUNT * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    return TMPT_OK;
}

extern "C" int tmpt_unpack_stripes(const uint8_t* gathered, int width, int height, int stripeRows, int worldSize, int device, uint8_t* frame,
                                   void* stream) {
    if (!gathered || !frame || width < 1 || height < 1 || stripeRows < 0 || worldSize < 1)
        return tmpt::fail(TMPT_ERR_ARG, "tmpt_unpack_stripes: bad arguments");
    DeviceGuard guard(device);
    if (!guard.ok) return tmpt::fail(TMPT_ERR_CUDA, "tmpt_unpack_stripes: cudaSetDevice(%d) failed", device);
    int maxRows = 0;
    for (int r = 0; r < worldSize; ++r) maxRows = std::max(maxRows, tmpt_stripe_rows(height, stripeRows, r, worldSize));  // (tile interleave: height)
    const long long n = (long long)width * height;
    LAUNCH(k_unpack_stripes, div_up(n, 256), 256, 0, (cudaStream_t)stream, (const uchar4*)gathered, width, height, stripeRows, worldSize, maxRows,
           (uchar4*)frame);
    CU_TRY(cudaGetLastError());
    return TMPT_OK;
}

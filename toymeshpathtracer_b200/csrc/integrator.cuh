// integrator.cuh -- the per-sample arithmetic of the Trace() loop: camera rays, sky,
// direct light, diffuse scatter, the back-to-front unwind and the pixel resolve.
//
// Replaces Camera::GetRay (maths.h:93-104), Scatter (main.cpp:44-73), Trace (main.cpp:82-119)
// and the pixel epilogue of TraceImageBody::operator() (main.cpp:209-233).  Every value is
// formed with the reference's operation order and one rounding per operation (exact.cuh), so
// a pixel computed here equals, bit for bit, the same pixel computed by the CPU checker with
// the same RNG stream.  Pure per-lane functions: the kernels in kernels.cu decide how lanes
// are scheduled; __host__ __device__ so tests/emu can run them without a GPU.
#pragma once
#include "bvh.cuh"

namespace integ {

constexpr int kMaxDepth = 10;        // main.cpp:33
constexpr float kMinT = 0.001f;      // main.cpp:30
constexpr float kMaxT = 1.0e7f;      // main.cpp:31

// Camera (maths.h:106-111), 22 floats, same order as tmpt_camera
struct Camera {
    ex::V3 origin, lowerLeftCorner, horizontal, vertical, u, v, w;
    float lensRadius;
};

// maths.h:93-104
TMPT_HD void camera_get_ray(const Camera& c, float s, float t, uint32_t& rng, ex::V3& o, ex::V3& d) {
    float px, py;
    ex::random_in_unit_disk(rng, px, py);
    const float rdx = ex::mul(c.lensRadius, px), rdy = ex::mul(c.lensRadius, py);  // lensRadius * disk
    const ex::V3 offset = ex::add(ex::muls(c.u, rdx), ex::muls(c.v, rdy));
    o = ex::add(c.origin, offset);
    d = ex::normalize(ex::sub(ex::sub(ex::add(ex::add(c.lowerLeftCorner, ex::muls(c.horizontal, s)), ex::muls(c.vertical, t)), c.origin), offset));
}

// main.cpp:214-215 as the reference build evaluates it (v drawn before u), then GetRay
TMPT_HD void primary_ray(const Camera& c, int x, int y, float invW, float invH, uint32_t& rng, ex::V3& o, ex::V3& d) {
    const float fv = ex::mul(ex::add((float)y, ex::random_float01(rng)), invH);
    const float fu = ex::mul(ex::add((float)x, ex::random_float01(rng)), invW);
    camera_get_ray(c, fu, fv, rng, o, d);
}

// main.cpp:106-107: ((1-t)*(1,1,1) + t*(0.5,0.7,1.0)) * 0.5
TMPT_HD ex::V3 sky(ex::V3 dir) {
    const float t = ex::mul(0.5f, ex::add(dir.y, 1.0f));
    const float a = ex::sub(1.0f, t);
    return ex::muls(ex::add(ex::v3(ex::mul(1.0f, a), ex::mul(1.0f, a), ex::mul(1.0f, a)), ex::muls(ex::v3(0.5f, 0.7f, 1.0f), t)), 0.5f);
}

// main.cpp:62-68: the scalar that multiplies albedo*kLightColor when the sun is visible
TMPT_HD float sun_term(ex::V3 normal, ex::V3 rayDir, ex::V3 lightDir) {
    const ex::V3 nl = ex::dot(normal, rayDir) < 0.0f ? normal : ex::neg(normal);
    return fmaxf(0.0f, ex::dot(lightDir, nl));
}

// main.cpp:71-72: normalize((pos + normal + RandomUnitVector) - pos), GEOMETRIC normal
TMPT_HD ex::V3 scatter_dir(ex::V3 pos, ex::V3 normal, uint32_t& rng) {
    const ex::V3 target = ex::add(ex::add(pos, normal), ex::random_unit_vector(rng));
    return ex::normalize(ex::sub(target, pos));
}

// main.cpp:112-116 with light[i] = (albedo*kLightColor)*k_i (+ 0, main.cpp:48, 68) and atten = albedo
TMPT_HD ex::V3 unwind_step(float k, ex::V3 color) {
    const ex::V3 albedo = ex::v3(0.7f, 0.7f, 0.7f);
    const ex::V3 kLightColor = ex::v3(0.7f, 0.6f, 0.5f);
    const ex::V3 light = ex::add(ex::v3(0.0f, 0.0f, 0.0f), ex::muls(ex::mulv(albedo, kLightColor), k));
    return ex::add(light, ex::mulv(albedo, color));
}
// (a shadowed bounce has light = (0,0,0) exactly, which is what k = 0 produces: finite * 0 = +0)

// main.cpp:221-233: mean, sqrt, quantise
TMPT_HD uchar4 resolve_pixel(ex::V3 sum, float sppRecip) {
    const ex::V3 c = ex::muls(sum, sppRecip);
    uchar4 px;
    px.x = ex::quantise(ex::sqrt_rn(c.x));
    px.y = ex::quantise(ex::sqrt_rn(c.y));
    px.z = ex::quantise(ex::sqrt_rn(c.z));
    px.w = 255;
    return px;
}

// What the camera ray of one sample hit (AOV = true): the depth-0 HitScene answer.  id = -1 for the sky; t / normal are
// valid for hits only (normal = hit_payload's geometric normal, as tmpt_hit_scene reports it).
struct FirstHit {
    int id;
    float t;
    ex::V3 normal;
};

// One whole pixel, serially: the straightforward form used by the host emulation and by the
// first (non-wavefront) render kernel.  kk[] holds the per-bounce sun term (0 for a
// shadowed bounce).  AOV: `first` receives the camera ray's hit; the path is the same.
template <bool STATS = false, bool FAR = true, bool AOV = false, class Stack, class Scene>
TMPT_HD ex::V3 trace_path(Stack& stack, const Scene& sc, const Camera& cam, ex::V3 o, ex::V3 d, ex::V3 lightDir, uint32_t& rng,
                          unsigned long long& rays, bvh::TravStats* stats = nullptr, FirstHit* first = nullptr) {
    float kk[kMaxDepth];
    int depth = 0;
    ex::V3 color = ex::v3(0.0f, 0.0f, 0.0f);
    if (AOV) first->id = -1;
    while (depth < kMaxDepth) {
        ++rays;
        const bvh::HitRec h = bvh::traverse_with<false, STATS, FAR>(stack, sc, o, d, kMinT, kMaxT, stats);
        if (h.id < 0) { color = sky(d); break; }
        ex::V3 pos, normal;
        bvh::hit_payload(sc, h.id, h.u, h.v, pos, normal);
        if (AOV && depth == 0) { first->id = h.id; first->t = h.t; first->normal = normal; }
        ++rays;
        // the shadow ray (main.cpp:59): through the sun grid when the scene has one (sungrid.cuh), else through the tree
#if defined(TMPT_SUN_ONLY) && TMPT_SUN_ONLY  // (experiment: what the tree fallback in the same kernel costs)
        const bool shadowed = bvh::sun_occluded<STATS>(sc, pos, lightDir, kMinT, kMaxT, stats);
#else
        const bool shadowed = sc.sun.n > 0 ? bvh::sun_occluded<STATS>(sc, pos, lightDir, kMinT, kMaxT, stats)
                                           : bvh::traverse_with<true, STATS, FAR>(stack, sc, pos, lightDir, kMinT, kMaxT, stats).id >= 0;
#endif
        kk[depth] = shadowed ? 0.0f : sun_term(normal, d, lightDir);
        d = scatter_dir(pos, normal, rng);
        o = pos;
        ++depth;
    }
    for (int i = depth - 1; i >= 0; --i) color = unwind_step(kk[i], color);
    return color;
}

// The unit of parallel work: one CHUNK of a pixel's samples.  A chunk owns an XorShift32 stream
// seeded from (chunk, pixel) and adds its samples in order; a pixel is the in-order sum of its
// chunk sums (DESIGN.md "RNG").  The chunk length depends on spp only -- spp/32 clamped to
// [1, 8] -- so a frame does not depend on how it is split over lanes or GPUs.  Short chunks keep
// the work items short: 2 samples at the headline 64 spp (with 8-sample chunks an item ran for
// 4.4 ms, and on an 8-GPU split, 60 ms per frame, every GPU lost half an item at the end of its
// share: 3.4 % of the frame), one sample below 64 spp (a 640x360x4 frame with four-sample items
// has 1.5 of them per resident warp), 8 samples from 256 spp on, where chunk sums per pixel
// would otherwise cost more memory than they save time.
constexpr int kMaxChunkSamples = 8;
TMPT_HD int chunk_len(int spp) {
    const int c = spp / 32;
    return c < 1 ? 1 : c > kMaxChunkSamples ? kMaxChunkSamples : c;
}
TMPT_HD int chunk_count(int spp) { const int c = chunk_len(spp); return (spp + c - 1) / c; }
// Chunk `chunk` of pixel (x, y) with `len` samples per chunk: its samples [s0, s1) = [chunk * len, min(chunk * len + len, spp)),
// and (returned) the seed of its stream.  render_chunk and the kernels that run their own sample loop all start a chunk here.
TMPT_HD uint32_t chunk_start(int x, int y, int chunk, int width, int height, int spp, int len, int& s0, int& s1) {
    s0 = chunk * len;
    s1 = s0 + len < spp ? s0 + len : spp;
    return ex::chunk_seed((uint32_t)chunk, (uint32_t)y * (uint32_t)width + (uint32_t)x, (uint32_t)width * (uint32_t)height);
}

// AOV sums of one chunk or pixel (AOV = true), each from +0 in sample order, chunk sums added in chunk order like the colour:
// over the samples whose camera ray hits, the hit count, the sum of their normals and of their t.  id0 = the camera-ray hit of
// the first sample (tmpt_outputs.triangle reports chunk 0's).
struct AovSums {
    ex::V3 normal;
    float t, hits;
    int id0;
};
TMPT_HD void aov_clear(AovSums& a) { a.normal = ex::v3(0.0f, 0.0f, 0.0f); a.t = 0.0f; a.hits = 0.0f; a.id0 = -1; }
TMPT_HD void aov_add_hit(AovSums& a, ex::V3 normal, float t) { a.normal = ex::add(a.normal, normal); a.t = ex::add(a.t, t); a.hits = ex::add(a.hits, 1.0f); }

// The float outputs of a pixel (include/tmpt.h, tmpt_outputs) from its sums: radiance = colour sum * (1/spp) with A = 1 (the
// value resolve_pixel takes the square root of), normal = (normal sum, hit count) * (1/spp), depth = t sum / hit count, +inf
// where no camera ray hit.  NaN stays NaN.
TMPT_HD float4 radiance_of(ex::V3 sum, float sppRecip) {
    const ex::V3 c = ex::muls(sum, sppRecip);
    return make_float4(c.x, c.y, c.z, 1.0f);
}
TMPT_HD float4 normal_of(ex::V3 normalSum, float hits, float sppRecip) {
    const ex::V3 n = ex::muls(normalSum, sppRecip);
    return make_float4(n.x, n.y, n.z, ex::mul(hits, sppRecip));
}
TMPT_HD float depth_of(float tSum, float hits) { return hits > 0.0f ? ex::divf(tSum, hits) : ex::u2f(0x7F800000u); }

// `len` = samples per chunk: chunk_len(spp) for a one-shot frame, kMaxChunkSamples for a progressive pass
template <bool STATS = false, bool FAR = true, bool AOV = false, class Stack, class Scene>
TMPT_HD ex::V3 render_chunk(Stack& stack, const Scene& sc, const Camera& cam, int x, int y, int chunk, int width, int height, int spp, int len, ex::V3 lightDir,
                            unsigned long long& rays, bvh::TravStats* stats = nullptr, AovSums* aov = nullptr) {
    const float invW = ex::divf(1.0f, (float)width), invH = ex::divf(1.0f, (float)height);
    int s0, s1;
    uint32_t rng = chunk_start(x, y, chunk, width, height, spp, len, s0, s1);
    ex::V3 sum = ex::v3(0.0f, 0.0f, 0.0f);
    if (AOV) aov_clear(*aov);
    for (int s = s0; s < s1; ++s) {
        ex::V3 o, d;
        primary_ray(cam, x, y, invW, invH, rng, o, d);
        FirstHit fh;
        sum = ex::add(sum, trace_path<STATS, FAR, AOV>(stack, sc, cam, o, d, lightDir, rng, rays, stats, &fh));
        if (AOV) {
            if (s == s0) aov->id0 = fh.id;
            if (fh.id >= 0) aov_add_hit(*aov, fh.normal, fh.t);
        }
    }
    return sum;
}

// Adaptive progressive passes (include/tmpt.h, tmpt_progressive_pass_adaptive): a pixel's chunk count n and the Welford mean / M2
// of its chunk-mean luminance, updated per chunk sum in chunk order.  One rounding per operation, no contraction.
TMPT_HD void adaptive_add_chunk(ex::V3 chunkSum, uint32_t& n, float& mean, float& m2) {
    const float y = ex::mul(ex::add(ex::add(ex::mul(0.2126f, chunkSum.x), ex::mul(0.7152f, chunkSum.y)), ex::mul(0.0722f, chunkSum.z)), 0.125f);
    n += 1u;
    const float delta = ex::sub(y, mean);
    mean = ex::add(mean, ex::divf(delta, (float)n));
    m2 = ex::add(m2, ex::mul(delta, ex::sub(y, mean)));
}
// The stop rule: the standard error of the mean luminance, through the sqrt display curve, in 8-bit codes, is at most
// `tolerance` -- se = sqrt(M2 / (n (n-1))), codes = 255 * se / (2 sqrt(mean)) -- squared and multiplied out (no sqrt, no division).
// NaN state compares false, so such a pixel stops at minChunks.  Tolerance 0 stops nothing: the explicit test keeps a pixel with
// M2 = 0 (then a = b = 0) tracing.
TMPT_HD bool adaptive_converged(uint32_t n, float mean, float m2, float tolerance, int minChunks) {
    if (tolerance == 0.0f || n < (uint32_t)minChunks) return false;
    const float a = ex::mul(m2, 65025.0f);
    const float b = ex::mul(ex::mul(ex::mul((float)n, (float)(n - 1u)), ex::mul(4.0f, fmaxf(mean, 0x1p-16f))), ex::mul(tolerance, tolerance));
    return !(a > b);
}

// One whole pixel, serially (host emulation; the kernels spread the chunks over lanes).  AOV: `aov` receives the pixel's sums.
template <bool STATS = false, bool AOV = false, class Scene>
TMPT_HD uchar4 render_pixel(const Scene& sc, const Camera& cam, int x, int y, int width, int height, int spp, ex::V3 lightDir,
                            unsigned long long& rays, ex::V3* outLinear = nullptr, bvh::TravStats* stats = nullptr, AovSums* aov = nullptr) {
    const float sppRecip = ex::divf(1.0f, (float)spp);
    ex::V3 sum = ex::v3(0.0f, 0.0f, 0.0f);
    bvh::LocalStack stack;
    if (AOV) aov_clear(*aov);
    for (int c = 0; c < chunk_count(spp); ++c) {
        AovSums ca;
        sum = ex::add(sum, render_chunk<STATS, true, AOV>(stack, sc, cam, x, y, c, width, height, spp, chunk_len(spp), lightDir, rays, stats, &ca));
        if (AOV) {
            if (c == 0) aov->id0 = ca.id0;
            aov->normal = ex::add(aov->normal, ca.normal); aov->t = ex::add(aov->t, ca.t); aov->hits = ex::add(aov->hits, ca.hits);
        }
    }
    if (outLinear) *outLinear = ex::muls(sum, sppRecip);
    return resolve_pixel(sum, sppRecip);
}

}  // namespace integ

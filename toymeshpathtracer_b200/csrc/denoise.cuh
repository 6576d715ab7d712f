// denoise.cuh -- the per-pixel arithmetic of tmpt_denoise (include/tmpt.h): an edge-avoiding a-trous wavelet filter
// (Dammertz et al. 2010) with the variance-guided luminance weights of SVGF's spatial filter (Schied et al. 2017), guided by
// the first-hit normal, coverage and depth AOVs of tmpt_render_outputs.
//
// Every value is formed with one rounding per operation (exact.cuh), every sum runs in the fixed tap order below from +0.0f
// and e^(-x) is ex::expneg_spec, so a filtered frame is bit-exact against a serial restatement.  Pure per-pixel functions over
// whole-frame buffers: kernels.cu runs them one thread per pixel (k_denoise_prep, k_denoise_atrous, k_denoise_copy);
// __host__ __device__ so tests/denoise can run the same code without a GPU.
//
// Buffers, [height][width] with row 0 = bottom like the AOVs:
//   state  float4 (c.xyz, variance): the colour being filtered and its luminance variance (ping-pong between iterations)
//   guideA float4 (n.xyz, z): the unit normal (0 where there is none) and the depth
//   guideB float4 (gx, gy, cov, 0): the depth gradient and the coverage of a hit pixel; 0 marks the sky class
#pragma once
#include "integrator.cuh"

// the tap loops unrolled on the device: the kernel-weight tables become constants and the taps' loads are independent
#ifdef __CUDA_ARCH__
#define DN_UNROLL _Pragma("unroll")
#else
#define DN_UNROLL
#endif

namespace dn {

constexpr int kMaxIterations = 8;
constexpr int kMaxNormalPowerLog2 = 8;

struct Params {
    int iterations;
    float sigmaLuminance, sigmaDepth;
    int normalPowerLog2;
};

// adaptive_add_chunk's luminance expression
TMPT_HD float luminance(float x, float y, float z) {
    return ex::add(ex::add(ex::mul(0.2126f, x), ex::mul(0.7152f, y)), ex::mul(0.0722f, z));
}
TMPT_HD bool finite1(float v) { return (ex::f2u(v) & 0x7F800000u) != 0x7F800000u; }
TMPT_HD bool finite3(float4 c) { return finite1(c.x) && finite1(c.y) && finite1(c.z); }

// Prologue of pixel (x, y): the initial state and the guides.
//   hit       normal.w > 0 (coverage); every other pixel (NaN coverage included) is sky.  Classes never mix.
//   n         ex::normalize(normal.xyz) for a hit pixel whose dot(N, N) is finite and > 0, else 0
//   gx / gy   central differences of depth, (z[x+1] - z[x-1]) * 0.5, over in-frame hit neighbours; one-sided (z[x+1] - z or
//             z - z[x-1]) where only one qualifies; 0 where none does and for sky pixels
//   variance  two-pass variance of the luminance of the valid (finite colour) pixels of p's class in the 3 x 3 window,
//             dy outer and dx inner: count and sum, mean = sum / count, then the sum of (l - mean)^2 over the same pixels
//             divided by count; 0 if no pixel qualifies
TMPT_HD void prep_pixel(const float4* radiance, const float4* normal, const float* depth, int w, int h, int x, int y, float4& state,
                        float4& guideA, float4& guideB) {
    const size_t p = (size_t)y * w + x;
    const float4 c = radiance[p], N = normal[p];
    const bool hit = N.w > 0.0f;
    const float z = depth[p];
    ex::V3 n = ex::v3(0.0f, 0.0f, 0.0f);
    float gx = 0.0f, gy = 0.0f;
    if (hit) {
        const ex::V3 nv = ex::v3(N.x, N.y, N.z);
        const float d = ex::dot(nv, nv);
        if (d > 0.0f && finite1(d)) n = ex::normalize(nv);
        const bool l = x > 0 && normal[p - 1].w > 0.0f, r = x + 1 < w && normal[p + 1].w > 0.0f;
        gx = l && r ? ex::mul(ex::sub(depth[p + 1], depth[p - 1]), 0.5f) : r ? ex::sub(depth[p + 1], z) : l ? ex::sub(z, depth[p - 1]) : 0.0f;
        const bool b = y > 0 && normal[p - w].w > 0.0f, t = y + 1 < h && normal[p + w].w > 0.0f;
        gy = b && t ? ex::mul(ex::sub(depth[p + w], depth[p - w]), 0.5f) : t ? ex::sub(depth[p + w], z) : b ? ex::sub(z, depth[p - w]) : 0.0f;
    }
    float count = 0.0f, sum = 0.0f;
    for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
            const int qx = x + dx, qy = y + dy;
            if (qx < 0 || qx >= w || qy < 0 || qy >= h) continue;
            const size_t q = (size_t)qy * w + qx;
            const float4 cq = radiance[q];
            if (!finite3(cq) || (normal[q].w > 0.0f) != hit) continue;
            count = ex::add(count, 1.0f);
            sum = ex::add(sum, luminance(cq.x, cq.y, cq.z));
        }
    float var = 0.0f;
    if (count > 0.0f) {
        const float mean = ex::divf(sum, count);
        float ss = 0.0f;
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx) {
                const int qx = x + dx, qy = y + dy;
                if (qx < 0 || qx >= w || qy < 0 || qy >= h) continue;
                const size_t q = (size_t)qy * w + qx;
                const float4 cq = radiance[q];
                if (!finite3(cq) || (normal[q].w > 0.0f) != hit) continue;
                const float d = ex::sub(luminance(cq.x, cq.y, cq.z), mean);
                ss = ex::add(ss, ex::mul(d, d));
            }
        var = ex::divf(ss, count);
    }
    state = make_float4(c.x, c.y, c.z, var);
    guideA = make_float4(n.x, n.y, n.z, z);
    guideB = make_float4(gx, gy, hit ? N.w : 0.0f, 0.0f);
}

// One a-trous iteration at pixel p = (x, y) with tap spacing `step` (2^i in iteration i) -> p's new state.
//   v_p    the variance prefiltered by the 3 x 3 kernel {1/4, 1/2, 1/4}^2 at spacing 1 over the valid pixels of p's class, dy
//          outer, dx inner: kw = sum k, kv = sum k * var_q, v_p = kv / kw (0 if kw == 0)
//   taps   q = p + step (dx, dy), dy outer and dx inner over -2..2, counted if q is in the frame, valid and of p's class:
//            h    = h1[dx] * h1[dy], h1 = {1/16, 1/4, 3/8, 1/4, 1/16}
//            w_n  = |dot(n_p, n_q)| squared normalPowerLog2 times for a hit pixel (the AOV normal is the geometric e1 x e2 and
//                   the mesh winding is not consistent, hence the absolute value); 1 for sky
//            e_z  = |z_p - z_q| / (sigmaDepth * (|gx dx + gy dy| * step + 0.01 z_p)) for a hit pixel; 0 for sky
//            e_c  = 16 |cov_p - cov_q| for a hit pixel (a silhouette pixel is a blend of surface and sky: it is filtered with
//                   pixels of like coverage, and interior pixels leave it out); 0 for sky
//            e_l  = |l_p - l_q| / (sigmaLuminance * sqrt(v_p) + 1e-10) where p is valid; 0 where it is not
//            w    = (h * w_n) * expneg((e_z + e_c) + e_l)
//          W = sum w, C = sum w * c_q (per channel), V = sum (w * w) * var_q
//   out    (C / W per channel, V / (W * W)); p keeps its state if W == 0 (an invalid pixel without valid neighbours)
TMPT_HD float4 atrous_pixel(const float4* state, const float4* guideA, const float4* guideB, int w, int h, int x, int y, int step,
                            const Params& prm) {
    const float kH[5] = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};
    const float kG[3] = {0.25f, 0.5f, 0.25f};
    const size_t p = (size_t)y * w + x;
    const float4 sp = state[p], ap = guideA[p], bp = guideB[p];
    const bool hit = bp.z > 0.0f, valid = finite3(sp);
    float kw = 0.0f, kv = 0.0f;
    DN_UNROLL for (int dy = -1; dy <= 1; ++dy)
        DN_UNROLL for (int dx = -1; dx <= 1; ++dx) {
            const int qx = x + dx, qy = y + dy;
            if (qx < 0 || qx >= w || qy < 0 || qy >= h) continue;
            const size_t q = (size_t)qy * w + qx;
            const float4 sq = state[q];
            if (!finite3(sq) || (guideB[q].z > 0.0f) != hit) continue;
            const float k = ex::mul(kG[dx + 1], kG[dy + 1]);
            kw = ex::add(kw, k);
            kv = ex::add(kv, ex::mul(k, sq.w));
        }
    const float v = kw > 0.0f ? ex::divf(kv, kw) : 0.0f;
    const float lp = luminance(sp.x, sp.y, sp.z);
    const float lDen = ex::add(ex::mul(prm.sigmaLuminance, ex::sqrt_rn(v)), 1e-10f);
    const ex::V3 np = ex::v3(ap.x, ap.y, ap.z);
    const float zOff = ex::mul(0.01f, ap.w);
    float W = 0.0f, V = 0.0f;
    ex::V3 C = ex::v3(0.0f, 0.0f, 0.0f);
    DN_UNROLL for (int dy = -2; dy <= 2; ++dy)
        DN_UNROLL for (int dx = -2; dx <= 2; ++dx) {
            const int qx = x + step * dx, qy = y + step * dy;
            if (qx < 0 || qx >= w || qy < 0 || qy >= h) continue;
            const size_t q = (size_t)qy * w + qx;
            const float4 sq = state[q];
            const float covq = guideB[q].z;
            if (!finite3(sq) || (covq > 0.0f) != hit) continue;
            float wn = 1.0f, ez = 0.0f, ec = 0.0f, el = 0.0f;
            if (hit) {
                const float4 aq = guideA[q];
                ec = ex::mul(16.0f, fabsf(ex::sub(bp.z, covq)));
                wn = fabsf(ex::dot(np, ex::v3(aq.x, aq.y, aq.z)));
                for (int k = 0; k < prm.normalPowerLog2; ++k) wn = ex::mul(wn, wn);
                const float g = fabsf(ex::add(ex::mul(bp.x, (float)dx), ex::mul(bp.y, (float)dy)));
                ez = ex::divf(fabsf(ex::sub(ap.w, aq.w)), ex::mul(prm.sigmaDepth, ex::add(ex::mul(g, (float)step), zOff)));
            }
            if (valid) el = ex::divf(fabsf(ex::sub(lp, luminance(sq.x, sq.y, sq.z))), lDen);
            const float wt = ex::mul(ex::mul(ex::mul(kH[dx + 2], kH[dy + 2]), wn), ex::expneg_spec(ex::add(ex::add(ez, ec), el)));
            W = ex::add(W, wt);
            C = ex::add(C, ex::v3(ex::mul(wt, sq.x), ex::mul(wt, sq.y), ex::mul(wt, sq.z)));
            V = ex::add(V, ex::mul(ex::mul(wt, wt), sq.w));
        }
    if (W == 0.0f) return sp;
    return make_float4(ex::divf(C.x, W), ex::divf(C.y, W), ex::divf(C.z, W), ex::divf(V, ex::mul(W, W)));
}

// The outputs of a filtered colour c: rgba = integ::resolve_pixel's quantise(sqrt(c)) per channel with A = 255 (NaN -> 0), so
// with no iteration it is tmpt_render's frame byte for byte; radiance = (c, 1.0f).
TMPT_HD uchar4 rgba_of(float4 c) { return integ::resolve_pixel(ex::v3(c.x, c.y, c.z), 1.0f); }
TMPT_HD float4 radiance_of(float4 c) { return make_float4(c.x, c.y, c.z, 1.0f); }

}  // namespace dn

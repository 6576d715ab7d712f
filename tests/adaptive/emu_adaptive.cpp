// tests/adaptive/emu_adaptive.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// tests/emu/emu.cpp (the product's __host__ __device__ integrator compiled for the host) plus one adaptive progressive pass
// (include/tmpt.h, tmpt_progressive_pass_adaptive) over caller-owned per-pixel state, through the helpers the kernels use:
// integ::adaptive_converged (k_adaptive_select), integ::render_chunk with 8-sample chunks (the LIST render kernels),
// integ::adaptive_add_chunk (k_resolve_adaptive), integ::resolve_pixel / radiance_of (k_adaptive_write).  State layout as
// tests/adaptive/oracle_adaptive.c's.
#include "../emu/emu.cpp"

extern "C" int emu_adaptive_converged(uint32_t n, float mean, float m2, float tolerance, int minChunks) {
    return integ::adaptive_converged(n, mean, m2, tolerance, minChunks) ? 1 : 0;
}

extern "C" void emu_pass_adaptive(void* h, const float cam22[22], int w, int hgt, int nChunks, float tolerance, int minChunks, int row0, int row1,
                                  uint32_t* n, float* sum4, float* mean, float* m2, uint8_t* rgba, float* radiance4, int32_t* samples,
                                  long long* activePixels, long long* rayCount) {
    EmuScene* s = (EmuScene*)h;
    integ::Camera cam;
    memcpy(&cam, cam22, sizeof cam);
    const ex::V3 lightDir = ex::normalize(ex::v3(-0.7f, 1.0f, 0.5f));
    unsigned long long total = 0;
    long long active = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : total, active)
    for (int y = row0; y < row1; ++y) {
        unsigned long long rays = 0;
        bvh::LocalStack stack;
        for (int x = 0; x < w; ++x) {
            const size_t p = (size_t)y * w + x;
            ex::V3 sum = ex::v3(sum4[p * 4], sum4[p * 4 + 1], sum4[p * 4 + 2]);
            if (!integ::adaptive_converged(n[p], mean[p], m2[p], tolerance, minChunks)) {
                const int n0 = (int)n[p];
                for (int k = 0; k < nChunks; ++k) {
                    const ex::V3 cs = integ::render_chunk(stack, s->view, cam, x, y, n0 + k, w, hgt, 0x7FFFFFFF, integ::kMaxChunkSamples, lightDir, rays);
                    sum = ex::add(sum, cs);
                    integ::adaptive_add_chunk(cs, n[p], mean[p], m2[p]);
                }
            }
            sum4[p * 4] = sum.x; sum4[p * 4 + 1] = sum.y; sum4[p * 4 + 2] = sum.z; sum4[p * 4 + 3] = 0.0f;
            if (!integ::adaptive_converged(n[p], mean[p], m2[p], tolerance, minChunks)) ++active;
            const int spp = (int)n[p] * integ::kMaxChunkSamples;
            const float sppRecip = ex::divf(1.0f, (float)spp);
            const uchar4 px = integ::resolve_pixel(sum, sppRecip);
            const float4 r = integ::radiance_of(sum, sppRecip);
            rgba[p * 4] = px.x; rgba[p * 4 + 1] = px.y; rgba[p * 4 + 2] = px.z; rgba[p * 4 + 3] = px.w;
            radiance4[p * 4] = r.x; radiance4[p * 4 + 1] = r.y; radiance4[p * 4 + 2] = r.z; radiance4[p * 4 + 3] = r.w;
            samples[p] = spp;
        }
        total += rays;
    }
    if (rayCount) *rayCount = (long long)total;
    if (activePixels) *activePixels = active;
}

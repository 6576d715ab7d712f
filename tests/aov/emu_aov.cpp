// tests/aov/emu_aov.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// tests/emu/emu.cpp (the product's __host__ __device__ integrator compiled for the host) plus one entry point: a frame with
// the buffers of tmpt_outputs (include/tmpt.h), through integ::render_pixel's AOV instantiation and the same
// integ::normal_of / depth_of that k_resolve applies.
#include "../emu/emu.cpp"

extern "C" void emu_render_aov(void* h, const float cam22[22], int w, int hgt, int spp, int row0, int row1, uint8_t* rgba,
                               float* radiance4, float* normal4, float* depth, int32_t* triangle, long long* rayCount) {
    EmuScene* s = (EmuScene*)h;
    integ::Camera cam;
    memcpy(&cam, cam22, sizeof cam);
    const ex::V3 lightDir = ex::normalize(ex::v3(-0.7f, 1.0f, 0.5f));
    const float sppRecip = ex::divf(1.0f, (float)spp);
    unsigned long long total = 0;
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : total)
    for (int y = row0; y < row1; ++y) {
        unsigned long long rays = 0;
        for (int x = 0; x < w; ++x) {
            ex::V3 lin;
            integ::AovSums aov;
            const uchar4 px = integ::render_pixel<false, true>(s->view, cam, x, y, w, hgt, spp, lightDir, rays, &lin, nullptr, &aov);
            const size_t p = (size_t)y * w + x;
            rgba[p * 4] = px.x; rgba[p * 4 + 1] = px.y; rgba[p * 4 + 2] = px.z; rgba[p * 4 + 3] = px.w;
            radiance4[p * 4] = lin.x; radiance4[p * 4 + 1] = lin.y; radiance4[p * 4 + 2] = lin.z; radiance4[p * 4 + 3] = 1.0f;  // lin = sum * (1/spp)
            const float4 n = integ::normal_of(aov.normal, aov.hits, sppRecip);
            normal4[p * 4] = n.x; normal4[p * 4 + 1] = n.y; normal4[p * 4 + 2] = n.z; normal4[p * 4 + 3] = n.w;
            depth[p] = integ::depth_of(aov.t, aov.hits);
            triangle[p] = aov.id0;
        }
        total += rays;
    }
    if (rayCount) *rayCount = (long long)total;
}

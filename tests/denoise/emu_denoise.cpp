// tests/denoise/emu_denoise.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// The product's denoise.cuh (and ex::expneg_spec from exact.cuh) compiled for the host and run serially, pixel by pixel, the way
// kernels.cu's k_denoise_prep / k_denoise_atrous / k_denoise_copy run it one thread per pixel.  Buffers as tmpt_denoise's.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>
#include <vector>

#include "../../toymeshpathtracer_b200/csrc/denoise.cuh"

extern "C" float emu_expneg(float x) { return ex::expneg_spec(x); }

extern "C" void emu_denoise(int w, int h, const float* radiance4, const float* normal4, const float* depth, int iterations, float sigmaL,
                            float sigmaZ, int normalPowerLog2, uint8_t* rgba, float* radianceOut4) {
    const size_t n = (size_t)w * h;
    const float4* rad = (const float4*)radiance4;
    std::vector<float4> state[2] = {std::vector<float4>(n), std::vector<float4>(n)}, ga(n), gb(n);
    const float4* fin = rad;
    if (iterations > 0) {
        for (int y = 0; y < h; ++y)
            for (int x = 0; x < w; ++x) {
                const size_t p = (size_t)y * w + x;
                dn::prep_pixel(rad, (const float4*)normal4, depth, w, h, x, y, state[0][p], ga[p], gb[p]);
            }
        const dn::Params prm{iterations, sigmaL, sigmaZ, normalPowerLog2};
        for (int i = 0; i < iterations; ++i)
            for (int y = 0; y < h; ++y)
                for (int x = 0; x < w; ++x)
                    state[(i + 1) & 1][(size_t)y * w + x] = dn::atrous_pixel(state[i & 1].data(), ga.data(), gb.data(), w, h, x, y, 1 << i, prm);
        fin = state[iterations & 1].data();
    }
    for (size_t p = 0; p < n; ++p) {
        const float4 c = fin[p];
        if (rgba) { const uchar4 px = dn::rgba_of(c); rgba[p * 4] = px.x; rgba[p * 4 + 1] = px.y; rgba[p * 4 + 2] = px.z; rgba[p * 4 + 3] = px.w; }
        if (radianceOut4) { const float4 r = dn::radiance_of(c); memcpy(radianceOut4 + p * 4, &r, sizeof r); }
    }
}

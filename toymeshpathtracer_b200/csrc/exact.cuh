// exact.cuh -- device arithmetic that must reproduce the reference bit for bit.
//
// The reference's results are defined by IEEE binary32 operations rounded ONE AT A TIME
// in the order glm 0.9.9.5's scalar path writes them (external/glm/detail/
// func_geometric.inl:48-90).  nvcc contracts a*b+c into FFMA by default, which changes
// the last bit, so everything here is spelled with the __f*_rn intrinsics: they are never
// contracted, whatever -fmad says.  Division and square root use the correctly rounded
// forms (__fdiv_rn / __frcp_rn / __fsqrt_rn).
//
// Every function is __host__ __device__: tests/emu compiles these same headers for the
// host (g++ -ffp-contract=off, where plain float operators are already one-rounding IEEE)
// so the CPU test suite can run the identical logic without a GPU.  The shipped library
// only ever runs the __CUDA_ARCH__ branches.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>

#define TMPT_HD __host__ __device__ __forceinline__

namespace ex {

#ifdef __CUDA_ARCH__
TMPT_HD float mul(float a, float b) { return __fmul_rn(a, b); }
TMPT_HD float add(float a, float b) { return __fadd_rn(a, b); }
TMPT_HD float sub(float a, float b) { return __fsub_rn(a, b); }
TMPT_HD float divf(float a, float b) { return __fdiv_rn(a, b); }
TMPT_HD float rcp(float a) { return __frcp_rn(a); }  // correctly rounded 1/a == 1.0f / a
TMPT_HD float sqrt_rn(float a) { return __fsqrt_rn(a); }
TMPT_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
TMPT_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
TMPT_HD double dsub(double a, double b) { return __dsub_rn(a, b); }
TMPT_HD float d2f(double a) { return __double2float_rn(a); }
TMPT_HD int f2i_rz(float a) { return __float2int_rz(a); }
#else
TMPT_HD float mul(float a, float b) { return a * b; }
TMPT_HD float add(float a, float b) { return a + b; }
TMPT_HD float sub(float a, float b) { return a - b; }
TMPT_HD float divf(float a, float b) { return a / b; }
TMPT_HD float rcp(float a) { return 1.0f / a; }
TMPT_HD float sqrt_rn(float a) { return sqrtf(a); }
TMPT_HD double dmul(double a, double b) { return a * b; }
TMPT_HD double dadd(double a, double b) { return a + b; }
TMPT_HD double dsub(double a, double b) { return a - b; }
TMPT_HD float d2f(double a) { return (float)a; }
TMPT_HD int f2i_rz(float a) { return (int)a; }
#endif

// bit casts usable on both sides
TMPT_HD uint32_t f2u(float f) {
#ifdef __CUDA_ARCH__
    return __float_as_uint(f);
#else
    uint32_t u; memcpy(&u, &f, 4); return u;
#endif
}
TMPT_HD float u2f(uint32_t u) {
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    float f; memcpy(&f, &u, 4); return f;
#endif
}

struct V3 {
    float x, y, z;
};

TMPT_HD V3 v3(float x, float y, float z) { return V3{x, y, z}; }

TMPT_HD V3 add(V3 a, V3 b) { return v3(add(a.x, b.x), add(a.y, b.y), add(a.z, b.z)); }
TMPT_HD V3 sub(V3 a, V3 b) { return v3(sub(a.x, b.x), sub(a.y, b.y), sub(a.z, b.z)); }
TMPT_HD V3 mulv(V3 a, V3 b) { return v3(mul(a.x, b.x), mul(a.y, b.y), mul(a.z, b.z)); }
TMPT_HD V3 muls(V3 a, float s) { return v3(mul(a.x, s), mul(a.y, s), mul(a.z, s)); }
TMPT_HD V3 neg(V3 a) { return v3(-a.x, -a.y, -a.z); }

// func_geometric.inl:48-55: tmp = a*b; (tmp.x + tmp.y) + tmp.z
TMPT_HD float dot(V3 a, V3 b) {
    return add(add(mul(a.x, b.x), mul(a.y, b.y)), mul(a.z, b.z));
}
// func_geometric.inl:68-79
TMPT_HD V3 cross(V3 x, V3 y) {
    return v3(sub(mul(x.y, y.z), mul(y.y, x.z)), sub(mul(x.z, y.x), mul(y.z, x.x)), sub(mul(x.x, y.y), mul(y.x, x.y)));
}
// func_geometric.inl:82-90 + func_exponential.inl:136-139: v * (1 / sqrt(dot(v, v)))
TMPT_HD V3 normalize(V3 v) {
    float s = divf(1.0f, sqrt_rn(dot(v, v)));
    return muls(v, s);
}

// ---- RNG: maths.cpp:5-18 (shift triple 13/17/15) ----
TMPT_HD uint32_t xorshift32(uint32_t& state) {
    uint32_t x = state;
    x ^= x << 13;
    x ^= x >> 17;
    x ^= x << 15;
    state = x;
    return x;
}
TMPT_HD float random_float01(uint32_t& state) {
    // 24-bit integer -> float is exact; the division by 2^24 is exact too
    return divf((float)(xorshift32(state) & 0xFFFFFF), 16777216.0f);
}

// Per-pixel stream seed (DESIGN.md "RNG"): main.cpp:204's expression on the pixel index,
// scrambled by Wang's hash, never 0.
TMPT_HD uint32_t pixel_seed(uint32_t pixelIndex) {
    uint32_t s = pixelIndex * 9781u + 1u;
    s = (s ^ 61u) ^ (s >> 16);
    s *= 9u;
    s ^= s >> 4;
    s *= 0x27d4eb2du;
    s ^= s >> 15;
    return s ? s : 1u;
}

// Seed of the stream of chunk `chunk` of pixel `pixel` in a frame of `pixels` pixels: pixel_seed of the stream index
// chunk * pixels + pixel.  The index is formed in 64 bits (a 10000 x 10000 frame passes 2^32 at chunk 43, a long
// progressive 1080p render after 2071 chunks) and its high word is folded in before the hash, so that later streams do
// not repeat the first 2^32 in order; below 2^32 the seeds are exactly pixel_seed(index).
TMPT_HD uint32_t chunk_seed(uint32_t chunk, uint32_t pixel, uint32_t pixels) {
    const uint64_t idx = (uint64_t)chunk * (uint64_t)pixels + (uint64_t)pixel;
    uint32_t s = ((uint32_t)idx * 9781u + 1u) ^ ((uint32_t)(idx >> 32) * 0x9E3779B9u);
    s = (s ^ 61u) ^ (s >> 16);
    s *= 9u;
    s ^= s >> 4;
    s *= 0x27d4eb2du;
    s ^= s >> 15;
    return s ? s : 1u;
}

// maths.cpp:20-28.  vec3(R(), R(), 0): the reference build (g++) draws the SECOND
// component first; the oracle pins that order and this follows it.
TMPT_HD void random_in_unit_disk(uint32_t& state, float& px, float& py) {
    float d;
    do {
        float ry = random_float01(state);
        float rx = random_float01(state);
        px = sub(mul(2.0f, rx), 1.0f);
        py = sub(mul(2.0f, ry), 1.0f);
        d = add(add(mul(px, px), mul(py, py)), 0.0f);  // + p.z*p.z with p.z = 0
    } while (d >= 1.0f);
}

// "Trig spec" (DESIGN.md): sin/cos of a in [0, 8) in binary64 with unfused multiply/add,
// one final rounding to binary32.  Same operation sequence as the CPU checker so both
// produce identical bits; glibc's sinf/cosf (what the reference binary calls) differ from
// it by at most one ulp.
TMPT_HD void sincos_spec(float a, float& s, float& c) {
    const double TWO_OVER_PI = 0.63661977236758134308;
    const double P1 = 1.57079632673412561417e+00;  // 0x3FF921FB54400000
    const double P2 = 6.07710050650619224932e-11;
    double x = (double)a;
    double kd = floor(dadd(dmul(x, TWO_OVER_PI), 0.5));
    double y = dsub(dsub(x, dmul(kd, P1)), dmul(kd, P2));
    double z = dmul(y, y);
    double ps = -1.0 / 1307674368000.0;
    ps = dadd(dmul(ps, z), 1.0 / 6227020800.0);
    ps = dadd(dmul(ps, z), -1.0 / 39916800.0);
    ps = dadd(dmul(ps, z), 1.0 / 362880.0);
    ps = dadd(dmul(ps, z), -1.0 / 5040.0);
    ps = dadd(dmul(ps, z), 1.0 / 120.0);
    ps = dadd(dmul(ps, z), -1.0 / 6.0);
    double sy = dadd(y, dmul(y, dmul(z, ps)));
    double pc = 1.0 / 20922789888000.0;
    pc = dadd(dmul(pc, z), -1.0 / 87178291200.0);
    pc = dadd(dmul(pc, z), 1.0 / 479001600.0);
    pc = dadd(dmul(pc, z), -1.0 / 3628800.0);
    pc = dadd(dmul(pc, z), 1.0 / 40320.0);
    pc = dadd(dmul(pc, z), -1.0 / 720.0);
    pc = dadd(dmul(pc, z), 1.0 / 24.0);
    pc = dadd(dmul(pc, z), -0.5);
    double cy = dadd(1.0, dmul(z, pc));
    int q = (int)kd & 3;
    double sv = (q == 0) ? sy : (q == 1) ? cy : (q == 2) ? -sy : -cy;
    double cv = (q == 0) ? cy : (q == 1) ? -sy : (q == 2) ? -cy : sy;
    s = d2f(sv);
    c = d2f(cv);
}

// "Exp spec": e^(-x) for the denoiser's edge-stopping weights (denoise.cuh), written like sincos_spec: binary64 with unfused
// multiply / add and one final rounding to binary32, so the host restatement gives identical bits; within 1 ulp of the
// correctly rounded value.  x <= 0 (and -0) gives 1, so a weight never exceeds its kernel weight; x >= 104 (where e^(-x) is
// below half the smallest subnormal), +inf and NaN give 0, so a bad weight drops out of a sum instead of poisoning it.
// Reduction: x = k ln2 + r with ln2 split Cody-Waite style (k <= 150, so k * LN2_HI is exact), |r| <= ln2 / 2; e^(-r) is the
// degree-13 Taylor polynomial (truncation below 1e-17) in Horner form, scaled by 2^-k exactly (the double has the range).
TMPT_HD float expneg_spec(float x) {
    if (!(x < 104.0f)) return 0.0f;
    if (x <= 0.0f) return 1.0f;
    const double INV_LN2 = 1.44269504088896338700e+00;
    const double LN2_HI = 6.93147180369123816490e-01;  // 0x3FE62E42FEE00000
    const double LN2_LO = 1.90821492927058770002e-10;  // 0x3DEA39EF35793C76
    const double xd = (double)x;
    const double kd = floor(dadd(dmul(xd, INV_LN2), 0.5));
    const double y = -dsub(dsub(xd, dmul(kd, LN2_HI)), dmul(kd, LN2_LO));  // -r
    double p = 1.0 / 6227020800.0;                                          // 1/13!
    p = dadd(dmul(p, y), 1.0 / 479001600.0);
    p = dadd(dmul(p, y), 1.0 / 39916800.0);
    p = dadd(dmul(p, y), 1.0 / 3628800.0);
    p = dadd(dmul(p, y), 1.0 / 362880.0);
    p = dadd(dmul(p, y), 1.0 / 40320.0);
    p = dadd(dmul(p, y), 1.0 / 5040.0);
    p = dadd(dmul(p, y), 1.0 / 720.0);
    p = dadd(dmul(p, y), 1.0 / 120.0);
    p = dadd(dmul(p, y), 1.0 / 24.0);
    p = dadd(dmul(p, y), 1.0 / 6.0);
    p = dadd(dmul(p, y), 0.5);
    p = dadd(dmul(p, y), 1.0);
    p = dadd(dmul(p, y), 1.0);
    const uint64_t bits = (uint64_t)(1023 - (int)kd) << 52;  // 2^-k
    double scale;
#ifdef __CUDA_ARCH__
    scale = __longlong_as_double((long long)bits);
#else
    memcpy(&scale, &bits, 8);
#endif
    return d2f(dmul(p, scale));
}

// maths.cpp:30-38
TMPT_HD V3 random_unit_vector(uint32_t& state) {
    const float kPI = 3.1415926f;  // maths.h:14
    float z = sub(mul(random_float01(state), 2.0f), 1.0f);
    float a = mul(mul(random_float01(state), 2.0f), kPI);
    float r = sqrt_rn(sub(1.0f, mul(z, z)));
    float sa, ca;
    sincos_spec(a, sa, ca);
    return v3(mul(r, ca), mul(r, sa), z);
}

// glm::min / glm::max / clamp (func_common.inl:17-30, 504-508) -- NaN-propagating in x
TMPT_HD float glm_min(float x, float y) { return (y < x) ? y : x; }
TMPT_HD float glm_max(float x, float y) { return (x < y) ? y : x; }

// uint8_t(saturate(c) * 255.0f) (maths.h:16-19, main.cpp:230-232); NaN -> 0 as g++/x86-64
TMPT_HD unsigned char quantise(float c) {
    float s = mul(glm_min(glm_max(c, 0.0f), 1.0f), 255.0f);
    if (s != s) return 0;
    return (unsigned char)f2i_rz(s);
}

}  // namespace ex

/* tests/denoise/oracle_denoise.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * orc_denoise: tmpt_denoise (include/tmpt.h) restated serially in plain C from the header's definition, without the product's
 * headers: prologue, a-trous iterations, outputs; orc_expneg: the header's e^(-x).  One rounding per float operation (build
 * with -ffp-contract=off, as tests/denoise_binding.py does); every sum in the header's tap order.  Rows are spread over
 * threads; every pixel of an iteration depends only on the previous state, so the result does not depend on the split. */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

float orc_expneg(float x);
void orc_denoise(int w, int h, const float* radiance4, const float* normal4, const float* depth, int iterations, float sigmaL,
                 float sigmaZ, int normalPowerLog2, uint8_t* rgba, float* radianceOut4, int threads);

/* e^(-x): binary64, unfused, Cody-Waite reduction by ln2, degree-13 Taylor polynomial, exact scaling, one rounding */
float orc_expneg(float x) {
    if (isnan(x) || x >= 104.0f) return 0.0f;
    if (x <= 0.0f) return 1.0f;
    const double ln2hi = 6.93147180369123816490e-01, ln2lo = 1.90821492927058770002e-10, invln2 = 1.44269504088896338700e+00;
    double xd = (double)x;
    double k = floor(xd * invln2 + 0.5);
    double r = (xd - k * ln2hi) - k * ln2lo;
    double y = -r;
    static const double fact[14] = {1.0, 1.0, 2.0, 6.0, 24.0, 120.0, 720.0, 5040.0, 40320.0, 362880.0, 3628800.0, 39916800.0,
                                    479001600.0, 6227020800.0};
    double p = 1.0 / fact[13];
    for (int i = 12; i >= 0; --i) p = p * y + (i == 2 ? 0.5 : 1.0 / fact[i]);
    return (float)(p * ldexp(1.0, -(int)k));
}

static float lum(const float* c) { return (0.2126f * c[0] + 0.7152f * c[1]) + 0.0722f * c[2]; }
static int fin3(const float* c) { return isfinite(c[0]) && isfinite(c[1]) && isfinite(c[2]); }
static uint8_t quant(float v) {
    v = sqrtf(v);
    if (v != v) return 0;
    if (v < 0.0f) v = 0.0f;
    if (v > 1.0f) v = 1.0f;
    return (uint8_t)(int)(v * 255.0f);
}

typedef struct {
    int w, h, step, npow, last;
    float sigmaL, sigmaZ;
    const float *radiance, *normal, *depth;
    float *cur, *next;      /* state: [w*h][4] = c.xyz, variance */
    float *nrm, *z, *grad;  /* n_p [3], z_p, (gx, gy) */
    const float* cov;       /* normal.w */
    uint8_t* cls;           /* 1 hit, 0 sky */
    uint8_t* rgba;
    float* radOut;
    int phase;              /* 0 prologue, 1 iteration */
    int nextRow;
    pthread_mutex_t mu;
} job_t;

static void prologue_row(job_t* j, int y) {
    const int w = j->w, h = j->h;
    for (int x = 0; x < w; ++x) {
        const size_t p = (size_t)y * w + x;
        const float* N = j->normal + 4 * p;
        const int hit = j->cls[p];
        float n[3] = {0.0f, 0.0f, 0.0f}, gx = 0.0f, gy = 0.0f;
        if (hit) {
            float d = (N[0] * N[0] + N[1] * N[1]) + N[2] * N[2];
            if (d > 0.0f && isfinite(d)) {
                float s = 1.0f / sqrtf(d);
                n[0] = N[0] * s; n[1] = N[1] * s; n[2] = N[2] * s;
            }
            const float* z = j->depth;
            int l = x > 0 && j->cls[p - 1], r = x < w - 1 && j->cls[p + 1];
            if (l && r) gx = (z[p + 1] - z[p - 1]) * 0.5f;
            else if (r) gx = z[p + 1] - z[p];
            else if (l) gx = z[p] - z[p - 1];
            int b = y > 0 && j->cls[p - w], t = y < h - 1 && j->cls[p + w];
            if (b && t) gy = (z[p + w] - z[p - w]) * 0.5f;
            else if (t) gy = z[p + w] - z[p];
            else if (b) gy = z[p] - z[p - w];
        }
        float ls[9];
        int m = 0;
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx) {
                int qx = x + dx, qy = y + dy;
                if (qx < 0 || qy < 0 || qx >= w || qy >= h) continue;
                size_t q = (size_t)qy * w + qx;
                if (!fin3(j->radiance + 4 * q) || j->cls[q] != hit) continue;
                ls[m++] = lum(j->radiance + 4 * q);
            }
        float var = 0.0f;
        if (m > 0) {
            float cnt = 0.0f, sum = 0.0f;
            for (int i = 0; i < m; ++i) { cnt = cnt + 1.0f; sum = sum + ls[i]; }
            float mean = sum / cnt, ss = 0.0f;
            for (int i = 0; i < m; ++i) { float d = ls[i] - mean; ss = ss + d * d; }
            var = ss / cnt;
        }
        memcpy(j->cur + 4 * p, j->radiance + 4 * p, 3 * sizeof(float));
        j->cur[4 * p + 3] = var;
        memcpy(j->nrm + 3 * p, n, sizeof n);
        j->z[p] = j->depth[p];
        j->grad[2 * p] = gx; j->grad[2 * p + 1] = gy;
    }
}

static void iteration_row(job_t* j, int y) {
    static const float h1[5] = {1.0f / 16.0f, 1.0f / 4.0f, 3.0f / 8.0f, 1.0f / 4.0f, 1.0f / 16.0f};
    static const float g1[3] = {0.25f, 0.5f, 0.25f};
    const int w = j->w, h = j->h, s = j->step;
    for (int x = 0; x < w; ++x) {
        const size_t p = (size_t)y * w + x;
        const float* sp = j->cur + 4 * p;
        const int hit = j->cls[p], valid = fin3(sp);
        float kw = 0.0f, kv = 0.0f;
        for (int dy = -1; dy <= 1; ++dy)
            for (int dx = -1; dx <= 1; ++dx) {
                int qx = x + dx, qy = y + dy;
                if (qx < 0 || qy < 0 || qx >= w || qy >= h) continue;
                size_t q = (size_t)qy * w + qx;
                if (!fin3(j->cur + 4 * q) || j->cls[q] != hit) continue;
                float k = g1[dx + 1] * g1[dy + 1];
                kw = kw + k;
                kv = kv + k * j->cur[4 * q + 3];
            }
        float vp = kw > 0.0f ? kv / kw : 0.0f;
        float lp = lum(sp), lden = j->sigmaL * sqrtf(vp) + 1e-10f;
        float W = 0.0f, C[3] = {0.0f, 0.0f, 0.0f}, V = 0.0f;
        for (int dy = -2; dy <= 2; ++dy)
            for (int dx = -2; dx <= 2; ++dx) {
                int qx = x + s * dx, qy = y + s * dy;
                if (qx < 0 || qy < 0 || qx >= w || qy >= h) continue;
                size_t q = (size_t)qy * w + qx;
                const float* sq = j->cur + 4 * q;
                if (!fin3(sq) || j->cls[q] != hit) continue;
                float wn = 1.0f, ez = 0.0f, ec = 0.0f, el = 0.0f;
                if (hit) {
                    const float *a = j->nrm + 3 * p, *b = j->nrm + 3 * q;
                    wn = fabsf((a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]);
                    for (int k = 0; k < j->npow; ++k) wn = wn * wn;
                    float g = fabsf(j->grad[2 * p] * (float)dx + j->grad[2 * p + 1] * (float)dy);
                    ez = fabsf(j->z[p] - j->z[q]) / (j->sigmaZ * (g * (float)s + 0.01f * j->z[p]));
                    ec = 16.0f * fabsf(j->cov[4 * p] - j->cov[4 * q]);
                }
                if (valid) el = fabsf(lp - lum(sq)) / lden;
                float wt = ((h1[dx + 2] * h1[dy + 2]) * wn) * orc_expneg((ez + ec) + el);
                W = W + wt;
                for (int c = 0; c < 3; ++c) C[c] = C[c] + wt * sq[c];
                V = V + (wt * wt) * sq[3];
            }
        float* out = j->next + 4 * p;
        if (W == 0.0f) {
            memcpy(out, sp, 4 * sizeof(float));
        } else {
            for (int c = 0; c < 3; ++c) out[c] = C[c] / W;
            out[3] = V / (W * W);
        }
    }
}

static void* worker(void* arg) {
    job_t* j = (job_t*)arg;
    for (;;) {
        pthread_mutex_lock(&j->mu);
        int y = j->nextRow++;
        pthread_mutex_unlock(&j->mu);
        if (y >= j->h) break;
        if (j->phase == 0) prologue_row(j, y);
        else iteration_row(j, y);
    }
    return NULL;
}

static void run(job_t* j, int threads) {
    j->nextRow = 0;
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    pthread_t t[256];
    for (int i = 1; i < threads; ++i) pthread_create(&t[i], NULL, worker, j);
    worker(j);
    for (int i = 1; i < threads; ++i) pthread_join(t[i], NULL);
}

void orc_denoise(int w, int h, const float* radiance4, const float* normal4, const float* depth, int iterations, float sigmaL,
                 float sigmaZ, int normalPowerLog2, uint8_t* rgba, float* radianceOut4, int threads) {
    const size_t n = (size_t)w * h;
    job_t j;
    memset(&j, 0, sizeof j);
    j.w = w; j.h = h; j.npow = normalPowerLog2; j.sigmaL = sigmaL; j.sigmaZ = sigmaZ;
    j.radiance = radiance4; j.normal = normal4; j.depth = depth; j.cov = normal4 + 3;
    j.cur = malloc(n * 4 * sizeof(float)); j.next = malloc(n * 4 * sizeof(float));
    j.nrm = malloc(n * 3 * sizeof(float)); j.z = malloc(n * sizeof(float)); j.grad = malloc(n * 2 * sizeof(float));
    j.cls = malloc(n);
    for (size_t p = 0; p < n; ++p) j.cls[p] = normal4[4 * p + 3] > 0.0f;
    pthread_mutex_init(&j.mu, NULL);
    j.phase = 0;
    run(&j, threads);
    for (int i = 0; i < iterations; ++i) {
        j.phase = 1; j.step = 1 << i;
        run(&j, threads);
        float* t = j.cur; j.cur = j.next; j.next = t;
    }
    for (size_t p = 0; p < n; ++p) {
        const float* c = j.cur + 4 * p;
        if (rgba) { rgba[4 * p] = quant(c[0]); rgba[4 * p + 1] = quant(c[1]); rgba[4 * p + 2] = quant(c[2]); rgba[4 * p + 3] = 255; }
        if (radianceOut4) { memcpy(radianceOut4 + 4 * p, c, 3 * sizeof(float)); radianceOut4[4 * p + 3] = 1.0f; }
    }
    pthread_mutex_destroy(&j.mu);
    free(j.cur); free(j.next); free(j.nrm); free(j.z); free(j.grad); free(j.cls);
}

/* tests/adaptive/oracle_adaptive.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * orc_pass_adaptive: one adaptive progressive pass (include/tmpt.h, tmpt_progressive_pass_adaptive) restated serially with
 * oracle/oracle.c's own functions, over caller-owned per-pixel state: n (chunks so far), the colour sum, the Welford mean and M2
 * of the chunk-mean luminance.  This file includes oracle.c, so the pinned restatement itself stays as it is.
 *
 * Chunk c of pixel (x, y) is 8 samples from the stream orc_stream_seed(c * w * h + y * w + x), as in orc_render's ORC_RNG_PIXEL
 * mode from 256 spp on; chunk sums are added in chunk order.  Rows [row0, row1) only, so a large frame can be checked at a few
 * rows.  Build with -ffp-contract=off, like oracle.c (tests/adaptive_binding.py does). */
#include "../../oracle/oracle.c"

void orc_pass_adaptive(const float* tris9, int nTris, const float cam22[22], int w, int h, int nChunks, float tolerance, int minChunks,
                       int row0, int row1, uint32_t* n, float* sum4, float* mean, float* m2, uint8_t* rgba, float* radiance4,
                       int32_t* samples, int64_t* activePixels, int64_t* rayCount, int threads);
int orc_adaptive_converged(uint32_t n, float mean, float m2, float tolerance, int minChunks);

int orc_adaptive_converged(uint32_t n, float mean, float m2, float tolerance, int minChunks) {
    if (tolerance == 0.0f || n < (uint32_t)minChunks) return 0;
    const float a = m2 * 65025.0f;
    const float b = (((float)n * (float)(n - 1u)) * (4.0f * fmaxf(mean, 0x1p-16f))) * (tolerance * tolerance);
    return !(a > b);
}

typedef struct {
    render_job base; /* scene, camera, frame size, rows, rgba, ray total, row counter */
    int nChunks, minChunks;
    float tolerance;
    uint32_t* n;
    float *sum4, *mean, *m2, *radiance4;
    int32_t* samples;
    int64_t active;
} adaptive_job;

static void pass_row(adaptive_job* a, int y, int64_t* rayCount, int64_t* active) {
    render_job* j = &a->base;
    const float invWidth = 1.0f / (float)j->w, invHeight = 1.0f / (float)j->h;
    for (int x = 0; x < j->w; ++x) {
        const size_t p = (size_t)y * (size_t)j->w + (size_t)x;
        v3 col = V(a->sum4[p * 4], a->sum4[p * 4 + 1], a->sum4[p * 4 + 2]);
        if (!orc_adaptive_converged(a->n[p], a->mean[p], a->m2[p], a->tolerance, a->minChunks)) {
            for (int k = 0; k < a->nChunks; ++k) {
                const uint64_t c = (uint64_t)a->n[p];
                uint32_t rng = orc_stream_seed(c * ((uint64_t)j->w * (uint64_t)j->h) + (uint64_t)y * (uint64_t)j->w + (uint64_t)x);
                v3 chunk = V(0.0f, 0.0f, 0.0f);
                for (int s = 0; s < 8; ++s) {
                    float fv = ((float)y + random_float01(&rng)) * invHeight;
                    float fu = ((float)x + random_float01(&rng)) * invWidth;
                    ray_t ray = camera_get_ray(&j->cam, fu, fv, &rng);
                    chunk = add(chunk, trace(&j->sc, ray, &rng, rayCount));
                }
                col = add(col, chunk);
                /* the Welford update of the chunk-mean luminance */
                const float Y = ((0.2126f * chunk.x + 0.7152f * chunk.y) + 0.0722f * chunk.z) * 0.125f;
                a->n[p] += 1u;
                const float delta = Y - a->mean[p];
                a->mean[p] = a->mean[p] + delta / (float)a->n[p];
                a->m2[p] = a->m2[p] + delta * (Y - a->mean[p]);
            }
        }
        a->sum4[p * 4] = col.x; a->sum4[p * 4 + 1] = col.y; a->sum4[p * 4 + 2] = col.z; a->sum4[p * 4 + 3] = 0.0f;
        if (!orc_adaptive_converged(a->n[p], a->mean[p], a->m2[p], a->tolerance, a->minChunks)) ++*active;
        const int spp = (int)a->n[p] * 8;
        const float sppRecip = 1.0f / (float)spp;
        col = muls(col, sppRecip);
        if (a->samples) a->samples[p] = spp;
        if (a->radiance4) { a->radiance4[p * 4] = col.x; a->radiance4[p * 4 + 1] = col.y; a->radiance4[p * 4 + 2] = col.z; a->radiance4[p * 4 + 3] = 1.0f; }
        col = V(sqrtf(col.x), sqrtf(col.y), sqrtf(col.z));
        j->rgba[p * 4 + 0] = quantise(col.x);
        j->rgba[p * 4 + 1] = quantise(col.y);
        j->rgba[p * 4 + 2] = quantise(col.z);
        j->rgba[p * 4 + 3] = 255;
    }
}

static void* pass_worker(void* arg) {
    adaptive_job* a = (adaptive_job*)arg;
    render_job* j = &a->base;
    int64_t rays = 0, active = 0;
    for (;;) {
        pthread_mutex_lock(&j->mu);
        int y = j->next_row++;
        pthread_mutex_unlock(&j->mu);
        if (y >= j->row1) break;
        pass_row(a, y, &rays, &active);
    }
    pthread_mutex_lock(&j->mu);
    j->rays += rays;
    a->active += active;
    pthread_mutex_unlock(&j->mu);
    return NULL;
}

void orc_pass_adaptive(const float* tris9, int nTris, const float cam22[22], int w, int h, int nChunks, float tolerance, int minChunks,
                       int row0, int row1, uint32_t* n, float* sum4, float* mean, float* m2, uint8_t* rgba, float* radiance4,
                       int32_t* samples, int64_t* activePixels, int64_t* rayCount, int threads) {
    adaptive_job a;
    render_job* j = &a.base;
    j->sc.tris9 = tris9; j->sc.nTris = nTris; j->sc.lightDir = light_dir(); j->sc.trig = ORC_TRIG_SPEC;
    j->cam = camera_from22(cam22);
    j->w = w; j->h = h; j->spp = 8; j->rngMode = ORC_RNG_PIXEL; j->row1 = row1;
    j->rgba = rgba; j->linear = NULL; j->next_row = row0; j->rays = 0;
    a.nChunks = nChunks; a.minChunks = minChunks; a.tolerance = tolerance;
    a.n = n; a.sum4 = sum4; a.mean = mean; a.m2 = m2; a.radiance4 = radiance4; a.samples = samples; a.active = 0;
    pthread_mutex_init(&j->mu, NULL);
    run_threads(pass_worker, &a, threads);
    pthread_mutex_destroy(&j->mu);
    if (rayCount) *rayCount = j->rays;
    if (activePixels) *activePixels = a.active;
}

/* tests/aov/oracle_aov.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * orc_render_aov: orc_render (oracle/oracle.c) plus the buffers of tmpt_outputs (include/tmpt.h) -- the linear radiance and
 * the camera rays' first-hit normal, coverage, depth and triangle -- restated with the oracle's own functions.  This file
 * includes oracle.c, so the pinned restatement itself stays as it is.  The first hit of a sample is hit_scene() on its
 * camera ray, the same query trace() starts with: paths, RNG streams, ray count and rgba are orc_render's.
 *
 * Summation order (what the GPU path follows, include/tmpt.h): inside a chunk the sums run in sample order from +0.0f and a
 * sample whose camera ray misses adds nothing; chunk sums are added in chunk order from +0.0f.  Build with
 * -ffp-contract=off, like oracle.c (tests/aov_binding.py does). */
#include "../../oracle/oracle.c"

void orc_render_aov(const float* tris9, int nTris, const float cam22[22], int w, int h, int spp, int rngMode, int trig,
                    int row0, int row1, uint8_t* rgba, float* outRadiance4, float* outNormal4, float* outDepth,
                    int32_t* outTriangle, int64_t* rayCount, int threads);

typedef struct {
    render_job base;  /* scene, camera, frame size, rows, rgba, ray total, row counter */
    float *radiance, *normal, *depth;
    int32_t* triangle;
} aov_job;

static void render_row_aov(aov_job* a, int y, int64_t* rayCount) { /* render_row with the AOV sums */
    render_job* j = &a->base;
    const float invWidth = 1.0f / (float)j->w, invHeight = 1.0f / (float)j->h;
    const float sppRecip = 1.0f / (float)j->spp;
    uint32_t rng = (uint32_t)y * 9781u + 1u; /* main.cpp:204 */
    for (int x = 0; x < j->w; ++x) {
        v3 col = V(0.0f, 0.0f, 0.0f), nrm = V(0.0f, 0.0f, 0.0f);
        float tSum = 0.0f, hits = 0.0f;
        int id0 = -1;
        const int chunkLen = j->rngMode == ORC_RNG_PIXEL ? ORC_CHUNK_SAMPLES(j->spp) : j->spp;
        for (int s0 = 0, c = 0; s0 < j->spp; s0 += chunkLen, ++c) {
            if (j->rngMode == ORC_RNG_PIXEL)
                rng = orc_stream_seed((uint64_t)c * ((uint64_t)j->w * (uint64_t)j->h) + (uint64_t)y * (uint64_t)j->w + (uint64_t)x);
            v3 chunk = V(0.0f, 0.0f, 0.0f), chunkN = V(0.0f, 0.0f, 0.0f);
            float chunkT = 0.0f, chunkHits = 0.0f;
            const int s1 = s0 + chunkLen < j->spp ? s0 + chunkLen : j->spp;
            for (int s = s0; s < s1; ++s) {
                float fv = ((float)y + random_float01(&rng)) * invHeight;
                float fu = ((float)x + random_float01(&rng)) * invWidth;
                ray_t ray = camera_get_ray(&j->cam, fu, fv, &rng);
                hit_t first;
                memset(&first, 0, sizeof first);
                const int id = hit_scene(j->sc.tris9, j->sc.nTris, &ray, kMinT, kMaxT, 0, &first); /* draws nothing from rng */
                if (s == 0) id0 = id;
                if (id != -1) {
                    chunkN = add(chunkN, first.normal);
                    chunkT = chunkT + first.t;
                    chunkHits = chunkHits + 1.0f;
                }
                chunk = add(chunk, trace(&j->sc, ray, &rng, rayCount));
            }
            if (j->rngMode == ORC_RNG_PIXEL) {
                col = add(col, chunk); nrm = add(nrm, chunkN); tSum = tSum + chunkT; hits = hits + chunkHits;
            } else {
                col = chunk; nrm = chunkN; tSum = chunkT; hits = chunkHits;
            }
        }
        col = muls(col, sppRecip);
        const size_t p = (size_t)y * (size_t)j->w + (size_t)x;
        if (a->radiance) { a->radiance[p * 4] = col.x; a->radiance[p * 4 + 1] = col.y; a->radiance[p * 4 + 2] = col.z; a->radiance[p * 4 + 3] = 1.0f; }
        if (a->normal) {
            const v3 n = muls(nrm, sppRecip);
            a->normal[p * 4] = n.x; a->normal[p * 4 + 1] = n.y; a->normal[p * 4 + 2] = n.z; a->normal[p * 4 + 3] = hits * sppRecip;
        }
        if (a->depth) a->depth[p] = hits > 0.0f ? tSum / hits : INFINITY;
        if (a->triangle) a->triangle[p] = id0;
        col = V(sqrtf(col.x), sqrtf(col.y), sqrtf(col.z));
        j->rgba[p * 4 + 0] = quantise(col.x);
        j->rgba[p * 4 + 1] = quantise(col.y);
        j->rgba[p * 4 + 2] = quantise(col.z);
        j->rgba[p * 4 + 3] = 255;
    }
}

static void* render_worker_aov(void* arg) {
    aov_job* a = (aov_job*)arg;
    render_job* j = &a->base;
    int64_t rays = 0;
    for (;;) {
        pthread_mutex_lock(&j->mu);
        int y = j->next_row++;
        pthread_mutex_unlock(&j->mu);
        if (y >= j->row1) break;
        render_row_aov(a, y, &rays);
    }
    pthread_mutex_lock(&j->mu);
    j->rays += rays;
    pthread_mutex_unlock(&j->mu);
    return NULL;
}

void orc_render_aov(const float* tris9, int nTris, const float cam22[22], int w, int h, int spp, int rngMode, int trig,
                    int row0, int row1, uint8_t* rgba, float* outRadiance4, float* outNormal4, float* outDepth,
                    int32_t* outTriangle, int64_t* rayCount, int threads) {
    aov_job a;
    render_job* j = &a.base;
    j->sc.tris9 = tris9; j->sc.nTris = nTris; j->sc.lightDir = light_dir(); j->sc.trig = trig;
    j->cam = camera_from22(cam22);
    j->w = w; j->h = h; j->spp = spp; j->rngMode = rngMode; j->row1 = row1;
    j->rgba = rgba; j->linear = NULL; j->next_row = row0; j->rays = 0;
    a.radiance = outRadiance4; a.normal = outNormal4; a.depth = outDepth; a.triangle = outTriangle;
    pthread_mutex_init(&j->mu, NULL);
    run_threads(render_worker_aov, &a, threads);
    pthread_mutex_destroy(&j->mu);
    if (rayCount) *rayCount = j->rays;
}

/* include/tmpt.h -- C ABI of the B200-native Trace() hot path ("tmpt" = toy mesh path tracer).
 *
 * The reference (pr0g/ToyMeshPathTracer) has no plugin / FFI layer: its seam is the
 * C++ `Scene` class plus the row functor that main() hands to TBB.  Every entry point
 * below names the reference interface it stands in for (paths relative to
 * /root/reference/source).  INTEGRATION.md shows the binding a reference maintainer
 * would add.  Plain pointers and sizes only; no C++ or torch types cross this line;
 * nothing throws.  All functions return TMPT_OK (0) or a negative tmpt_status and
 * leave a message for tmpt_last_error() (thread-local).
 *
 * There is NO CPU fallback: without a CUDA device, or if a kernel launch fails, the
 * compute entry points return TMPT_ERR_CUDA.
 */
#ifndef TMPT_H
#define TMPT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TMPT_ABI_VERSION 3

typedef enum tmpt_status {
    TMPT_OK = 0,
    TMPT_ERR_ARG = -1,   /* bad argument (null pointer, size out of range)            */
    TMPT_ERR_CUDA = -2,  /* CUDA runtime / launch failure, or no device               */
    TMPT_ERR_IO = -3,    /* file could not be read / written                          */
    TMPT_ERR_OOM = -4
} tmpt_status;

/* Opaque scene: triangle replica + BVH resident on ONE device.
 * Stands in for `Scene` (scene.h:17-43). */
typedef struct tmpt_scene tmpt_scene;

/* The reference's Camera fields in declaration order (maths.h:106-111): 22 floats, 88 bytes. */
typedef struct tmpt_camera {
    float origin[3];
    float lowerLeftCorner[3];
    float horizontal[3];
    float vertical[3];
    float u[3], v[3], w[3];
    float lensRadius;
} tmpt_camera;

/* Where a caller-supplied buffer lives. */
typedef enum tmpt_mem { TMPT_HOST = 0, TMPT_DEVICE = 1 } tmpt_mem;

/* tmpt_scene_create flags */
#define TMPT_BUILD_DEFAULT 0u /* binned-SAH top-down build on the device (16 bins per axis)     */
#define TMPT_BUILD_LBVH 1u    /* Morton codes + radix sort + Karras hierarchy: faster build,
                                 ~40 % more node visits per ray                                */

/* tmpt_hit_scene modes */
#define TMPT_HIT_CLOSEST 0 /* nearest hit through the BVH                                  */
#define TMPT_HIT_ANY 1     /* shadow-ray early out: outID is 1 / -1 (any triangle in range) */
#define TMPT_HIT_BRUTE 2   /* nearest hit by scanning every triangle on the GPU (upstream's
                              HitScene); used to cross-check the BVH at sizes the CPU oracle
                              cannot reach                                                  */
#define TMPT_HIT_SUN 3     /* the integrator's own shadow query (main.cpp:59): any hit along
                              the SUN direction (main.cpp:36) from each ray's origin, through
                              the scene's sun grid; the rays' directions are not read.  outID
                              is 1 / -1.  Equals TMPT_HIT_ANY with direction = the sun's.   */

typedef struct tmpt_scene_info {
    int32_t abi_version;
    int32_t device;
    int32_t tri_count;
    int32_t node_count;      /* wide BVH nodes                                             */
    int32_t leaf_count;
    int32_t max_leaf_tris;
    int32_t max_depth;       /* deepest wide node; the traversal stack is sized from it    */
    int32_t builder;         /* TMPT_BUILD_* actually used                                 */
    float bounds_min[3];     /* bounds of all input triangles                              */
    float bounds_max[3];
    float sah_cost;          /* SAH cost of the wide tree (Cnode = Ctri = 1, root-relative) */
    float build_ms;          /* upload + build, device time                                */
    uint64_t device_bytes;   /* triangles + nodes resident in HBM                          */
} tmpt_scene_info;

/* ---- scene: Scene::Scene(const Triangle*, int) (scene.h:19, scene.cpp:54-57) followed by
 * BuildOctree (scene.h:26, scene.cpp:75-83; called from main.cpp:312).  Upstream spells it
 * InitializeScene(triCount, tris).  tris9 = triCount x 9 floats, AoS v0.xyz v1.xyz v2.xyz,
 * bit-identical to the reference's Triangle[] (maths.h:56-59).  The input is copied to
 * `device` and the BVH is built there; the caller keeps ownership of tris9. */
int tmpt_scene_create(const float* tris9, int triCount, int device, unsigned flags, tmpt_scene** outScene);
void tmpt_scene_destroy(tmpt_scene* scene); /* Scene::~Scene (scene.cpp:59) */
int tmpt_scene_get_info(const tmpt_scene* scene, tmpt_scene_info* outInfo);
/* Beyond the reference (SURVEY.md 8(f) rank 4): the same triangles, moved.  `tris9` has the layout and the count the
 * scene was created with; the BVH keeps its topology and is refitted on the device (boxes, Moller-Trumbore slots, hit
 * payload).  Every query after the call answers for the NEW positions, exactly as a freshly created scene would (the
 * tree only culls); traversal gets slower the further the vertices move from where the tree was built.
 * `seconds` (may be NULL): upload + device time.  Not to be called while a query or a render of the scene is in flight. */
int tmpt_scene_refit(tmpt_scene* scene, const float* tris9, int triCount, double* seconds);

/* ---- query: int Scene::HitScene(const Ray&, float tMin, float tMax, Hit&) const
 * (scene.h:36-37, scene.cpp:86-97), batched over nRays.
 *   rays6      nRays x 6 floats: orig.xyz dir.xyz (Ray, maths.h:31-40; dir assumed unit)
 *   outID      -1 on a miss; else the ORIGINAL index of the nearest triangle (the contract
 *              scene.h:35 documents and upstream implements; the fork itself returns 1).
 *              Tie rule: lowest index among triangles whose t is bit-equal nearest.
 *              Range rule: tMin <= t <= tMax and t < tMax (maths.cpp:371 + scene.cpp:34, 90).
 *   outT / outPos3 / outNormal3   Hit fields (maths.h:46-51), written ONLY for hits, may be
 *              NULL.  pos is the barycentric point (maths.cpp:374), normal the normalised
 *              e1 x e2 (maths.cpp:375); bit-exact with the reference's arithmetic.
 *   mem        TMPT_HOST: all pointers are host memory (copies are made inside the call);
 *              TMPT_DEVICE: all are device pointers on the scene's device.
 *   stream     a cudaStream_t (NULL = the scene's own stream); with TMPT_DEVICE the call is
 *              asynchronous on that stream.
 *   tMin may be 0 (a ray that starts ON a surface then hits it at t = +-0; ties between the triangles around a vertex go
 *   to the lowest index) or negative.  Origins beyond 16 x the scene's largest |coordinate| are answered by the all-triangle
 *   scan (same answers, slower).  The one case in which the answer differs from a scan over all triangles -- and from the
 *   reference's octree, and the octree from the scan -- is a "hit" that is rounding noise of maths.cpp:350's determinant test
 *   (a ray in the plane of a zero-area or very long thin triangle), reported far from the triangle itself: DESIGN.md 2.1. */
int tmpt_hit_scene(const tmpt_scene* scene, const float* rays6, int64_t nRays, float tMin, float tMax,
                   int mode, int mem, int32_t* outID, float* outT, float* outPos3, float* outNormal3,
                   void* stream);

/* ---- render: the row functor TraceImageBody (main.cpp:180-246) with Trace (:82-119) and
 * Scatter (:44-73) inside, over image rows [0, height) -- the tbb::parallel_for of
 * main.cpp:329-331.
 *   rgba       width*height*4 bytes, row 0 = bottom of the picture (main.cpp:229), A = 255
 *   rayCount   one count per HitScene-equivalent query (main.cpp:57, 91), 64-bit
 *   seconds    device time of the render window (main.cpp:319-333): kernel(s) plus, for
 *              TMPT_HOST, the device-to-host copy of the frame
 * RNG: one XorShift32 stream (maths.cpp:5-13) per PIXEL and per chunk of spp/32 (clamped to 1..8)
 * samples, seeded from (chunk, pixel index) (DESIGN.md "RNG"); the reference seeds one per row (main.cpp:204).
 * A scene renders one frame at a time (its scratch buffers are per scene). */
int tmpt_render(const tmpt_scene* scene, const tmpt_camera* camera, int width, int height, int spp,
                int mem, uint8_t* rgba, uint64_t* rayCount, double* seconds, void* stream);

/* Beyond the reference: the linear radiance and first-hit AOVs ("arbitrary output variables") of a frame, for denoisers,
 * tone mapping, compositing and picking.  Each pointer may be NULL (not produced); at least one must be set.  All buffers
 * are [height][width] with row 0 = bottom (as tmpt_render's rgba), in the memory space `mem` names. */
typedef struct tmpt_outputs {
    uint8_t* rgba;      /* width*height*4 bytes: tmpt_render's frame, byte for byte                                        */
    float* radiance;    /* width*height*4: the linear per-pixel mean BEFORE sqrt / quantise, sum * (1/spp); A = 1.0f        */
    float* normal;      /* width*height*4: xyz = sum over the samples of the camera ray's first-hit geometric normal (as
                           tmpt_hit_scene's outNormal3) * (1/spp); w = hits * (1/spp), the coverage.  Albedo is 0.7 at
                           every hit (main.cpp:48), so 0.7 * w is the albedo AOV                                            */
    float* depth;       /* width*height: sum of the first-hit t / hits (IEEE division); +INFINITY where no sample hit        */
    int32_t* triangle;  /* width*height: ORIGINAL index of the triangle that sample 0's camera ray hits, -1 for the sky     */
} tmpt_outputs;

/* One frame of tmpt_render with the outputs `out` names.  The paths do not change: RNG streams, rays, rayCount and rgba
 * are those of tmpt_render with the same arguments; the AOVs are recorded from the camera rays the integrator traces
 * anyway.  Summation order (what makes every buffer bit-exact against a serial restatement): inside a chunk the colour and
 * the AOV sums run in sample order from +0.0f, a sample whose camera ray misses adds nothing to the AOV sums; the chunk
 * sums are then added in chunk order from +0.0f; the divisions by spp are multiplications by the float 1/spp.  NaN stays
 * NaN: `radiance` keeps a NaN the reference arithmetic makes (such pixels are 0 in rgba); nothing is sanitised.
 * TMPT_HOST: each requested buffer is staged in device scratch owned by the scene; `seconds` covers the kernels and every
 * device-to-host copy.  Errors: TMPT_ERR_ARG for a NULL `out`, no buffer requested, a bad `mem`, or the range checks of
 * tmpt_render.  Single GPU. */
int tmpt_render_outputs(const tmpt_scene* scene, const tmpt_camera* camera, int width, int height, int spp, int mem,
                        const tmpt_outputs* out, uint64_t* rayCount, double* seconds, void* stream);

/* Beyond the reference: nViews frames of one size, one camera each, in one call (orbits, cube-map faces, stereo pairs,
 * light-field grids).  The views share one work queue and one launch sequence, so small views keep the GPU busy.
 *   cameras    a HOST array of nViews cameras (as tmpt_render's camera is a host pointer); the call uploads it into scratch
 *              owned by the scene.
 *   out        as tmpt_render_outputs, every buffer view-major: [nViews][height][width] with the per-pixel layout of
 *              tmpt_render_outputs, row 0 = the bottom of each view.  View v of a buffer starts at v * width * height pixels,
 *              so tmpt_denoise can run on one view of a batch through plain pointer offsets.
 *   rayCount   the sum of the counts of the nViews single frames below.
 *   mem / stream / seconds   as tmpt_render_outputs; with TMPT_HOST the buffers are staged in the scene's scratch, sized for
 *              the whole batch.  A batch uses the scene's scratch like a frame does (calls take turns).
 * Equality: view v of every buffer equals tmpt_render_outputs(cameras[v], width, height, spp) with the same outputs: bytes for
 * rgba and triangle, bits for radiance, normal and depth, NaN included.
 * RNG: every view uses the pixel streams of a single frame, seeded from (chunk, pixel index in its view).  Two views with the
 * same camera are therefore identical, and the noise of different views is correlated.  This is deliberate: it is the price
 * of the equality above.
 * Errors, before any device work: TMPT_ERR_ARG for a NULL scene or cameras, nViews outside 1..65536, nViews * width * height
 * above 10^8 (the reference's largest single frame), the range checks of tmpt_render, or the checks of tmpt_render_outputs'
 * `out` and `mem`.  Single GPU; no progressive or adaptive form. */
int tmpt_render_views(const tmpt_scene* scene, const tmpt_camera* cameras, int nViews, int width, int height, int spp,
                      int mem, const tmpt_outputs* out, uint64_t* rayCount, double* seconds, void* stream);

/* Progressive rendering (beyond the reference, SURVEY.md 8(f) rank 4): the frame converges over calls.
 * tmpt_progressive_begin fixes the frame size and clears the running per-pixel sums kept with the scene; every
 * tmpt_progressive_pass traces `nChunks` (1..128) more chunks of 8 samples per pixel with the SAME camera, adds them to
 * the sums in chunk order and writes the mean over all samples so far (quantised like tmpt_render's frame).  Chunk c of
 * a pixel is the same XorShift32 stream whether it is traced by a one-shot frame or by a pass, so after P chunks in total
 * the frame equals tmpt_render(spp = 8 * P) byte for byte whenever P >= 32 (a one-shot frame uses 8-sample chunks from
 * 256 spp on).  rayCount / seconds: this pass only.  samplesSoFar (may be NULL): 8 * chunks so far.  Single GPU. */
int tmpt_progressive_begin(tmpt_scene* scene, int width, int height);
int tmpt_progressive_pass(tmpt_scene* scene, const tmpt_camera* camera, int nChunks, int mem, uint8_t* rgba,
                          uint64_t* rayCount, double* seconds, int* samplesSoFar, void* stream);
/* A pass with tmpt_outputs: rgba and radiance only, both the mean over all samples so far (after P >= 32 chunks in total,
 * radiance equals tmpt_render_outputs' at spp = 8 * P bit for bit).  A normal, depth or triangle pointer is TMPT_ERR_ARG:
 * passes keep no running AOV sums. */
int tmpt_progressive_pass_outputs(tmpt_scene* scene, const tmpt_camera* camera, int nChunks, int mem, const tmpt_outputs* out,
                                  uint64_t* rayCount, double* seconds, int* samplesSoFar, void* stream);

/* Adaptive progressive passes (beyond the reference): a pass traces only the pixels whose estimated error is still above a
 * tolerance.  A session (tmpt_progressive_begin, which also clears the adaptive state) becomes uniform or adaptive with its
 * first pass; a uniform pass in an adaptive session, or an adaptive pass in a uniform one, is TMPT_ERR_ARG.
 * Per pixel the session keeps n (chunks so far), the colour sum and a Welford mean and M2 of the chunk-mean luminance.  For
 * each new chunk sum S, in chunk order, with one rounding per float operation and no contraction:
 *     Y = ((0.2126f*S.x + 0.7152f*S.y) + 0.0722f*S.z) * 0.125f;   n = n + 1;   delta = Y - mean;
 *     mean = mean + delta / (float)n;   M2 = M2 + delta * (Y - mean)
 * Stop rule -- the standard error of the mean luminance, taken through the sqrt display curve, in 8-bit codes, at most
 * `tolerance` -- written without sqrt or division:
 *     a = M2 * 65025.0f;   b = (((float)n * (float)(n - 1)) * (4.0f * fmaxf(mean, 0x1p-16f))) * (tolerance * tolerance)
 *     converged = tolerance != 0 && n >= minChunks && !(a > b)
 * A pixel whose state became NaN is therefore converged once n >= minChunks (more samples cannot remove a NaN from a sum).
 * A pass: every pixel not converged under this pass's params traces exactly nChunks more 8-sample chunks, chunk indices
 * n .. n + nChunks - 1, and updates its state as above; converged pixels are not traced.  Chunk c of a pixel is the stream a
 * uniform pass traces as that pixel's chunk c, so every pixel equals, bit for bit in rgba and radiance, the same pixel of a
 * uniform session after n of its chunks (and tmpt_render_outputs at spp = 8 n once n >= 32); with tolerance 0 a pass equals
 * tmpt_progressive_pass_outputs with the same nChunks in bytes, radiance and rayCount.
 *   out          rgba and / or radiance (other pointers: TMPT_ERR_ARG), written for the whole frame: sum * (1 / (8 n))
 *   samples      (may be NULL) width*height int32: 8 n per pixel
 *   rayCount     the rays traced in this pass only
 *   activePixels (may be NULL) pixels not converged under this pass's params after the pass: 0 = the next identical pass
 *                traces nothing
 *   seconds      device time of select, compaction, render, resolve and copies
 * Errors (TMPT_ERR_ARG, with a message): nChunks outside 1..128, a NULL params, a negative, NaN or infinite tolerance,
 * minChunks outside 2..2^21, and the limits of tmpt_progressive_pass_outputs (8 x the session's most chunks of a pixel at
 * most 2^24).  Single GPU. */
typedef struct tmpt_adaptive {
    float tolerance;   /* 8-bit display codes; 0 = adaptivity off (every pixel is traced) */
    int32_t minChunks; /* no pixel stops before it has this many chunks; 2 .. 2^21 */
} tmpt_adaptive;
int tmpt_progressive_pass_adaptive(tmpt_scene* scene, const tmpt_camera* camera, int nChunks, const tmpt_adaptive* params, int mem,
                                   const tmpt_outputs* out, int32_t* samples, uint64_t* rayCount, double* seconds,
                                   int64_t* activePixels, void* stream);

/* Denoising (beyond the reference): an edge-avoiding a-trous wavelet filter (Dammertz et al. 2010) with the variance-guided
 * luminance weights of SVGF's spatial filter (Schied et al. 2017) over a frame's linear radiance, guided by its first-hit normal,
 * coverage and depth.  Bit-exact against a serial restatement: one rounding per float operation, no contraction, every sum in
 * the order below from +0.0f, and e^(-x) is expneg (binary64 with unfused operations, one rounding to binary32, within 1 ulp of
 * the correctly rounded value; 1 for x <= 0; 0 for x >= 104, +inf and NaN).
 * Per pixel p: c = radiance.xyz, N = normal.xyz, z = depth; l(c) = ((0.2126f c.x + 0.7152f c.y) + 0.0722f c.z).
 *   class      p is a hit pixel if normal.w > 0, else sky; pixels of different classes never mix
 *   valid      all three channels of p's current colour are finite; an invalid pixel is never a tap, so a NaN pixel becomes the
 *              weighted mean of its valid neighbours (it keeps its input if it has none)
 *   prologue   n_p = N * (1 / sqrt(dot(N, N))) for a hit pixel with dot(N, N) finite and > 0, else 0.
 *              (gx, gy): (z[x+1] - z[x-1]) * 0.5 over in-frame hit neighbours, z[x+1] - z or z - z[x-1] where only one is,
 *              0 where none is (likewise in y with the rows above and below); 0 for sky.
 *              var_p: over the valid pixels of p's class in the 3 x 3 window (dy outer, dx inner), count and sum of l, then
 *              mean = sum / count and var = (sum of (l - mean) * (l - mean)) / count; 0 if none qualifies.  State = (c, var).
 *   iteration  i = 0 .. iterations - 1 with step s = 2^i, each from the previous state into a new one:
 *              v_p = (sum k var_q) / (sum k) over the valid pixels of p's class in the 3 x 3 window at spacing 1, k =
 *                    g[dx] * g[dy] with g = {1/4, 1/2, 1/4}; 0 if none qualifies
 *              taps q = p + s (dx, dy), dy outer and dx inner over -2..2, counted if in the frame, valid and of p's class:
 *                h   = h1[dx] * h1[dy], h1 = {1/16, 1/4, 3/8, 1/4, 1/16}
 *                w_n = |dot(n_p, n_q)| squared normalPowerLog2 times (hit); 1 (sky)
 *                e_z = |z_p - z_q| / (sigmaDepth * (|gx dx + gy dy| * s + 0.01f z_p)) (hit); 0 (sky)
 *                e_c = 16 |cov_p - cov_q| with cov = normal.w (hit): silhouette pixels, blends of surface and sky, are
 *                      filtered with pixels of like coverage and left out of the interior's sums; 0 (sky)
 *                e_l = |l_p - l_q| / (sigmaLuminance * sqrt(v_p) + 1e-10f) for a valid p; 0 for an invalid one
 *                w   = (h * w_n) * expneg((e_z + e_c) + e_l)
 *              W = sum w, C = sum w c_q per channel, V = sum (w w) var_q; new state (C / W, V / (W W)), or the old one if W == 0
 *   outputs    rgba = quantise(sqrt(c)) per channel as tmpt_render (NaN -> 0), A = 255; radiance = (c, 1.0f).  With
 *              iterations = 0 both come straight from the input: rgba is tmpt_render's frame for the same radiance, byte for byte.
 *   in         tmpt_render_outputs' buffers: radiance, normal and depth are required; rgba and triangle are not read.  The guides
 *              may come from a frame at another spp than the radiance: e.g. normal and depth from tmpt_render_outputs at spp 8,
 *              radiance from an adaptive session (tmpt_progressive_pass_adaptive) of the same camera and size.
 *   out        rgba and / or radiance (other pointers: TMPT_ERR_ARG); out->radiance may be in->radiance (filters in place).
 *   mem / stream / seconds as tmpt_render_outputs: with TMPT_HOST the inputs and outputs are staged in device scratch owned by
 *              the scene; seconds = device time of the kernels and copies.  The scene supplies the device, the stream, its
 *              host-call lock and scratch (4 x 16 bytes per pixel); its triangles are not read.  Single GPU.
 * Errors (TMPT_ERR_ARG, with a message, before any device work): a NULL scene, in, params or out; a missing in->radiance,
 * in->normal or in->depth; no output requested or an AOV pointer in `out`; a bad mem; width or height outside 1..10000;
 * iterations outside 0..8, normalPowerLog2 outside 0..8, or a sigma that is not a finite value > 0. */
typedef struct tmpt_denoise_params {
    int32_t iterations;      /* 0..8 a-trous passes; pass i's taps are 2^i pixels apart; 0 = the output is the input     */
    float sigmaLuminance;    /* > 0, finite: luminance edge-stop in units of the local standard deviation (SVGF: 4)     */
    float sigmaDepth;        /* > 0, finite: depth edge-stop (SVGF: 1)                                                   */
    int32_t normalPowerLog2; /* 0..8: the normal weight is |n_p . n_q|^(2^k) (SVGF's 128 = 7)                           */
} tmpt_denoise_params;
int tmpt_denoise(tmpt_scene* scene, int width, int height, int mem, const tmpt_outputs* in, const tmpt_denoise_params* params,
                 const tmpt_outputs* out, double* seconds, void* stream);

/* Multi-GPU form: this rank renders only its share of the frame and writes it packed into
 * outStripes (device memory on the scene's device, tmpt_stripe_rows(...) *
 * tmpt_local_width(...) * 4 bytes).  Two partitions:
 *   stripeRows > 0   row stripes: stripe k (rows [k*stripeRows, (k+1)*stripeRows)) belongs to
 *                    rank k % worldSize; packed = owned rows, stripe after stripe;
 *   stripeRows == 0  tile interleave (the default of multigpu.py and tmpt_render_multi): the
 *                    8x4-pixel tile (tx, ty) belongs to rank (tx + ty) % worldSize, so every
 *                    rank owns 1/worldSize of the tiles spread evenly over the frame; packed =
 *                    [height][localWidth] with local tile tx / worldSize of each tile row.
 * The frame does not depend on the partition (per-pixel RNG streams).  Asynchronous on `stream`.  rayCountDev is a
 * device uint64 the kernel adds to.  If peerFrame is non-NULL the pixels are written
 * straight into that full-size frame (width*height*4, possibly peer / IPC-mapped memory
 * on another GPU) instead -- the gather fused into the render epilogue. */
int tmpt_render_stripes(const tmpt_scene* scene, const tmpt_camera* camera, int width, int height, int spp,
                        int stripeRows, int rank, int worldSize, uint8_t* outStripes, uint8_t* peerFrame,
                        uint64_t* rayCountDev, void* stream);
int tmpt_stripe_rows(int height, int stripeRows, int rank, int worldSize); /* rows of the rank's packed output */
int tmpt_local_width(int width, int stripeRows, int worldSize);            /* pixels per row of it */
/* Rank 0 after a gather: scatter worldSize packed stripe buffers (each padded to
 * maxRowsPerRank*width*4 bytes, rank-major) into the final frame.  Device pointers. */
int tmpt_unpack_stripes(const uint8_t* gathered, int width, int height, int stripeRows, int worldSize,
                        int device, uint8_t* frame, void* stream);

/* One frame on several GPUs from ONE process: scenes[i] is a replica of the same triangles on its
 * own device (tmpt_scene_create per device).  Device i renders the row stripes of rank i of
 * nScenes (as tmpt_render_stripes) and stores its pixels straight into the frame that lives on
 * scenes[0]'s device -- peer access over NVLink / NVSwitch -- which is then copied to `rgba`
 * (host memory, width*height*4).  The multi-GPU form of the tbb::parallel_for of main.cpp:329-331
 * for the command line (TMPT_GPUS=n); multi-process callers use tmpt_render_stripes + tmpt_frame_*. */
int tmpt_render_multi(tmpt_scene* const* scenes, int nScenes, const tmpt_camera* camera, int width, int height, int spp,
                      uint8_t* rgba, uint64_t* rayCount, double* seconds);

/* Frame memory that other ranks (processes) on the same node can write: rank 0 allocates
 * the full-size frame and exports a 64-byte CUDA IPC handle; every other rank opens it and
 * passes the mapped pointer as `peerFrame` to tmpt_render_stripes, so its pixels travel over
 * NVLink / NVSwitch as plain stores in the render kernel's epilogue -- no gather step, no copy. */
int tmpt_frame_alloc(int device, size_t bytes, void** outPtr, unsigned char outHandle[64]);
int tmpt_frame_open(int device, const unsigned char handle[64], void** outPtr);
int tmpt_frame_close(int device, void* ptr);   /* for pointers from tmpt_frame_open  */
int tmpt_frame_free(int device, void* ptr);    /* for pointers from tmpt_frame_alloc */

/* Instrumented passes: the same kernels compiled with work counters, for the roofline's
 * per-ray figures (never part of a timed run).  outStats (TMPT_STATS_COUNT entries): [0] rays
 * (HitScene-equivalent queries), [1] wide BVH nodes visited (4 box tests each), [2] exact
 * triangle tests, [3] hits (tmpt_hit_scene_stats only), [4] walk iterations summed over lanes,
 * [5] pops of entries the best t had already culled, [6] lane iterations spent waiting at a
 * leaf while the parked one was tested, [7] warp iterations with a node step, [8] with a
 * triangle test, [9] warp iterations in all ([4] / (32 * [9]) = share of lane slots that held
 * an unfinished ray), [10] rays traced twice because their shared-memory stack overflowed,
 * [11..15] rays whose stack held more than 4 / 8 / 12 / 16 / 24 entries at some point.
 * rays6Dev is a DEVICE pointer. */
#define TMPT_STATS_COUNT 16
int tmpt_render_stats(const tmpt_scene* scene, const tmpt_camera* camera, int width, int height, int spp, uint64_t outStats[TMPT_STATS_COUNT]);
int tmpt_hit_scene_stats(const tmpt_scene* scene, const float* rays6Dev, int64_t nRays, float tMin, float tMax, int mode,
                         uint64_t outStats[TMPT_STATS_COUNT]);

/* ---- host glue that main() does around the hot path ---- */
/* LoadScene (main.cpp:122-170): parse the OBJ like external/objparser.cpp, build Triangle[]
 * plus the two floor triangles, report model bounds.  *outTris9 is malloc'ed; tmpt_free it. */
int tmpt_load_obj(const char* path, float** outTris9, int* outTriCount, float boundsMin[3], float boundsMax[3]);
void tmpt_free(void* p);
/* Camera::Camera (maths.cpp:40-59). */
void tmpt_camera_make(const float lookFrom[3], const float lookAt[3], const float vup[3], float vfovDeg,
                      float aspect, float aperture, float focusDist, tmpt_camera* out);
/* Camera placement of main() (main.cpp:296-307), including the "sponza.obj" special case. */
void tmpt_camera_for_scene(const char* objPath, const float boundsMin[3], const float boundsMax[3],
                           int width, int height, tmpt_camera* out);
/* stbi_write_png + stbi_flip_vertically_on_write (main.cpp:341-342): 8-bit RGBA PNG. */
int tmpt_write_png(const char* path, int width, int height, const uint8_t* rgba, int flipVertically);

/* The whole CLI (main.cpp:248-345): `<width> <height> <spp> <datafile>` -> output.png and the
 * three report lines; returns the process exit code. */
int tmpt_main(int argc, const char** argv);

/* Which render kernel the last frame of this scene used (kernels.cu: choose_render_kernel):
 * *kernel = 0 lockstep tiles (k_render), 1 path regeneration (k_render_paths, frames whose paths
 * leave the scene early), -1 no frame decided yet; *escapeFraction = the probe's measure, the
 * share of first diffuse bounces that reach the sky.  Both kernels produce the same bytes.  Either
 * pointer may be NULL. */
int tmpt_render_kernel_choice(const tmpt_scene* scene, int* kernel, float* escapeFraction);

const char* tmpt_last_error(void);
int tmpt_device_count(void);
/* kernels launched by this library since load (bench.py's gpu_launches evidence) */
uint64_t tmpt_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* TMPT_H */

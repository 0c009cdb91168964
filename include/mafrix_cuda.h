/*
 * mafrix_cuda.h -- C ABI of libmafrix_cuda, the B200 (sm_100a) path-tracing backend that
 * drops in behind MafrixRender's IPixelIntegrator seam.
 *
 * Every entry point names the reference interface it replaces (paths under
 * /root/reference/EngineCore/).  The F# P/Invoke stubs a maintainer would add are in
 * INTEGRATION.md.  Plain C types only: no CUDA or torch types cross this boundary.
 *
 * Conventions
 *   - every function returns MFX_OK (0) or a negative MfxStatus; the message is available
 *     from mfx_last_error() (thread-local).  Nothing throws or aborts across the ABI.
 *   - the caller owns every input array (copied during mfx_scene_create; may be freed
 *     afterwards) and every output buffer; the library owns the opaque handles and all
 *     device memory.
 *   - one host thread per handle (the reference calls Sample from its single render thread,
 *     Film.fs:67-73); distinct handles are independent.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     MFX_ERR_NO_DEVICE.
 */
#ifndef MAFRIX_CUDA_H
#define MAFRIX_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MFX_API __attribute__((visibility("default")))

typedef enum {
    MFX_OK = 0,
    MFX_ERR_INVALID_ARGUMENT = -1,
    MFX_ERR_NO_DEVICE = -2,
    MFX_ERR_CUDA = -3,
    MFX_ERR_OUT_OF_MEMORY = -4,
    MFX_ERR_UNSUPPORTED = -5
} MfxStatus;

/* IHitable implementations on the path: Shape/Trangle.fs:98, Shape/Rect.fs:11, Shape/Sphere.fs:9 */
typedef enum { MFX_TRIANGLE = 0, MFX_RECT = 1, MFX_SPHERE = 2 } MfxPrimKind;
/* IMaterial implementations: Materials/Material.fs:39 (Lambertian), :56 (Metal), :98 (SpecularTransmission) */
/* MFX_SKY_TRACER only (RenderTest/Sample/RayTracing.fs): :300-325 Dielectric(ri), :282-290 Lambertian over a
 * CheckerTexture (:54-61) of two constant colours, Lambertian over the NoiseTexture (:96-99). */
typedef enum { MFX_LAMBERT = 0, MFX_METAL = 1, MFX_SPECTRANS = 2,
               MFX_DIELECTRIC = 3, MFX_LAMBERT_CHECKER = 4, MFX_LAMBERT_NOISE = 5 } MfxMaterialKind;
/* IPathTracer implementations: Integrator/Integrators.fs:96 (PathIntegrator, the live one),
 * Tracer/PathTracer.fs:13 (NewPathTracer, where Metal/SpecularTransmission act);
 * MFX_SKY_TRACER = GetColor of the sphere sample (RenderTest/Sample/RayTracing.fs:367-382): no light, sky
 * gradient on a miss, black at the depth limit, closest hit = ListHit over the whole list (:256-258). */
typedef enum { MFX_PATH_INTEGRATOR = 0, MFX_NEW_PATH_TRACER = 1, MFX_SKY_TRACER = 2 } MfxIntegrator;
/* Arithmetic of the device path.
 *   MFX_EXACT_F64: f64, reference operation order, no FMA contraction -- primitive ids, t and
 *                  radiance are bit-identical to the reference algorithm.
 *   MFX_FAST_F32 : f32 wavefront kernels over the compact float4 layout (the throughput path). */
typedef enum { MFX_EXACT_F64 = 0, MFX_FAST_F32 = 1 } MfxPrecision;

/* One IHitable.  Triangle: v[0..8] = v0,v1,v2.  Rect: v[0..11] = v0,v1,v2,v3 (Rect.fs:17-19).
 * Sphere: v[0..2] = center, v[3] = radius (Sphere.fs:15-20).  material indexes the table
 * passed in MfxSceneDesc (the already-resolved MaterialManager table, IMaterial.fs:20-35). */
typedef struct {
    int32_t kind;
    int32_t material;
    double  v[12];
} MfxPrim;

/* One IMaterial: Lambertian(albedo) | Metal(albedo, fuzz) | SpecularTransmission(T=albedo, ei, et).
 * MFX_SKY_TRACER: Lambertian(ConstantTexture albedo) | Metal(albedo, fuzz) | Dielectric(ri = ei) |
 * Lambertian(CheckerTexture(even = albedo, odd = (fuzz, ei, et))) | Lambertian(NoiseTexture) (tables in MfxSkyTracer). */
typedef struct {
    int32_t kind;
    int32_t pad;
    double  albedo[3];
    double  fuzz;
    double  ei;
    double  et;
} MfxMaterial;

/* BvhNode (Accelerate/BvhNode.fs:11-17): bound, first, count; array is heap-indexed
 * (children of i at 2i+1 / 2i+2, BvhNode.fs:40-41) with 2N-1 slots (BvhNode.fs:26). */
typedef struct {
    double  pmin[3];
    double  pmax[3];
    int32_t first;
    int32_t count;
} MfxBvhNode;

/* NewAreaLight (Lights/Light.fs:32-41): quad p0..p3, normal, colour. */
typedef struct {
    double p[12];
    double normal[3];
    double color[3];
} MfxAreaLight;

/* PinholeCamera, already derived (Camera.fs:113-133): position, topleft, coord.right, coord.down. */
typedef struct {
    double pos[3];
    double topleft[3];
    double right[3];
    double down[3];
} MfxCamera;

/* RayTraceCamera, already derived (RayTracing.fs:335-358): origin, lowerLeftCorner, horizontal, vertical, the lens
 * basis u, v and lensRadius = aperture/2.  mfx_camera_lens reproduces the constructor. */
typedef struct {
    double origin[3];
    double lower_left[3];
    double horizontal[3];
    double vertical[3];
    double u[3];
    double v[3];
    double lens_radius;
} MfxLensCamera;

/* What the sphere sample needs beyond prims/materials (RayTracing.fs:384-415).  perlin_* may be NULL when no
 * material is MFX_LAMBERT_NOISE: Perlin's static tables (:81-95) -- ranfloat[256], perm_x|perm_y|perm_z[3*256] --
 * which the reference fills from Random.Shared, so the host supplies them. */
typedef struct {
    MfxLensCamera  camera;
    const double  *perlin_ranfloat;
    const int32_t *perlin_perm;
} MfxSkyTracer;

/* What `new Scene(state)` holds for the path (Scene/Scene.fs:298-313). */
typedef struct {
    const MfxPrim     *prims;          /* state.shapes                                          */
    int32_t            n_prims;
    const MfxMaterial *materials;      /* MaterialManager.GetManager().materials                 */
    int32_t            n_materials;
    const MfxBvhNode  *nodes;          /* Bvh.nodes (BvhNode.fs:22) or NULL: build on the host   */
    int32_t            n_node_slots;   /* 2*n_prims-1 when nodes != NULL                         */
    const int32_t     *indices;        /* Bvh.indices (BvhNode.fs:20) or NULL                    */
    MfxAreaLight       light;          /* state.light                                            */
    MfxCamera          camera;         /* state.camera                                           */
    int32_t            width, height;  /* state.film.Size                                        */
    int32_t            max_depth;      /* PathIntegrator(bvh, maxDepth, light), Scene.fs:304     */
    int32_t            integrator;     /* MfxIntegrator                                          */
    const MfxSkyTracer *sky;           /* MFX_SKY_TRACER: lens camera + noise tables (light and camera above are
                                          ignored, prims must be spheres, max_depth = the `depth < 50` of
                                          RayTracing.fs:373); NULL otherwise                      */
} MfxSceneDesc;

/* Arguments of one IPixelIntegrator.Sample call. */
typedef struct {
    int32_t  precision;      /* MfxPrecision                                                     */
    int32_t  spp;            /* n of Sample(n) (Integrators.fs:161)                               */
    uint64_t seed;           /* key of the counter-based RNG (replaces `new Random()`, :162)      */
    int32_t  first_sample;   /* absolute index of the first sample (progressive frames)          */
    int32_t  tile_size;      /* multi-GPU: interleaved square tiles; 0 = whole frame              */
    int32_t  rank;           /* this process renders tiles with  tile_index % world == rank       */
    int32_t  world;          /* 1 = whole frame                                                   */
    int32_t  flags;          /* MFX_SAMPLE_* bits                                                 */
} MfxSampleParams;

#define MFX_SAMPLE_COUNT_TRAVERSAL 1   /* instrumented kernels: fill node/prim counters in MfxStats */
/* MFX_FAST_F32 only.  By default the fast path draws the hemisphere direction of GetRandomInUnitSphere
 * (Material.fs:9-14) and the light point (Rect.fs:33-38) directly -- same distributions, one RNG call per vertex,
 * no rejection loop.  With this bit it runs the reference's rejection loop on the f32 view of the very random
 * stream MFX_EXACT_F64 uses, so a fast frame can be compared with the exact one sample for sample. */
#define MFX_SAMPLE_REFERENCE_STREAM 2
/* MFX_FAST_F32 only: instrumented run on the library's own tree (what the shipped kernel really fetches):
 * MfxStats.nodes counts 128-byte four-child records, tris / spheres count primitive tests. */
#define MFX_SAMPLE_COUNT_OWN_TREE 4
/* MFX_FAST_F32 only.  By default the closest hits of bounce 0 (the primary rays) are ID-EXACT: same primitive and the
 * same f64 t as Bvh.Hit (BvhNode.fs:62-83) finds, tie rules included -- f32 box tests over conservatively padded boxes
 * of the library's own tree, f64 primitive tests, mfx_hybrid.cu.  With this bit bounce 0 uses f32 primitive tests like
 * the deeper bounces (primary ids then differ from the reference on <= 2e-4 of the rays). */
#define MFX_SAMPLE_F32_PRIMARY 8
/* Multi-GPU ownership by COLUMN STRIPES instead of square tiles: columns [c*tile_size, (c+1)*tile_size) belong to rank
 * c % world.  In the reference's x-major Color[w,h] a stripe is one contiguous block, ownership is arithmetic (no pixel
 * table is built or uploaded).  mfx_multi_sample uses it. */
#define MFX_SAMPLE_STRIPES 16
/* With world > 1: leave the pixels of the other ranks in the output untouched instead of zeroing them (the caller
 * assembles the frame from the owned pixels only). */
#define MFX_SAMPLE_NO_CLEAR 32

typedef struct {
    uint64_t closest_rays;       /* closest-hit queries traced by the last Sample call             */
    uint64_t shadow_rays;        /* shadow queries traced                                          */
    uint64_t paths;              /* camera paths started                                           */
    uint64_t nodes[2];           /* node records touched   [0]=closest [1]=shadow (counting runs)  */
    uint64_t tris[2];            /* triangle records tested                                        */
    uint64_t spheres[2];         /* sphere records tested                                          */
    double   ms_total;           /* device time of the whole call (CUDA events, library stream)    */
    double   ms_extend;          /* summed device time of the closest-hit traversal launches       */
    double   ms_shadow;          /* summed device time of the shadow traversal launches            */
    double   ms_shade;           /* ray generation + shading + resolve launches                    */
    uint32_t launches;           /* kernels launched by the call                                   */
    uint32_t launches_extend;
    uint32_t launches_shadow;
    uint32_t hybrid_fixups;      /* id-exact bounce 0 / seams: rays the hybrid kernel handed to the exact walk */
} MfxStats;

typedef struct MfxScene MfxScene;
typedef struct MfxFilm  MfxFilm;

/* ---- process / device ---------------------------------------------------------------------- */
MFX_API const char *mfx_version(void);
MFX_API const char *mfx_last_error(void);
MFX_API int mfx_device_count(void);
/* Selects the CUDA device for the calling thread's subsequent handles. */
MFX_API int mfx_init(int device);

/* ---- host-side reproductions (no GPU needed) ------------------------------------------------ */
/* PinholeCamera(pos, dir, fov, aspect) constructor, Camera.fs:96-133 (effective FOV = fov/2). */
MFX_API int mfx_camera_pinhole(const double pos[3], const double dir[3], double fov, double aspect,
                               MfxCamera *out);
/* RayTraceCamera(lookfrom, lookat, vup, vfov, aspect, aperture, focus_dist, _, _) constructor,
 * RenderTest/Sample/RayTracing.fs:335-358. */
MFX_API int mfx_camera_lens(const double lookfrom[3], const double lookat[3], const double vup[3], double vfov,
                            double aspect, double aperture, double focus_dist, MfxLensCamera *out);
/* Bvh.Build, BvhNode.fs:24-61: median split on the node bound's longest axis, leaf <= 3,
 * heap-indexed nodes (n_slots must be 2n-1), stable sort (the reference's sort is unstable). */
MFX_API int mfx_bvh_build(const MfxPrim *prims, int32_t n, MfxBvhNode *nodes_out, int32_t n_slots,
                          int32_t *indices_out);

/* Multi-GPU pixel ownership: the frame is cut into tile_size x tile_size tiles numbered row-major;
 * tile k belongs to rank k % world.  Writes this rank's linear pixel ids (y*width+x, tile after
 * tile) to pixels_out (capacity width*height, may be NULL to query) and their number to n_out. */
MFX_API int mfx_tile_map(int32_t width, int32_t height, int32_t tile_size, int32_t rank, int32_t world,
                         int32_t *pixels_out, int32_t *n_out);

/* Column-stripe ownership (MFX_SAMPLE_STRIPES) as a table, in the order the kernels enumerate it: this rank's stripes one
 * after the other, row-major inside a stripe.  pixels_out may be NULL to query the count. */
MFX_API int mfx_stripe_map(int32_t width, int32_t height, int32_t stripe, int32_t rank, int32_t world,
                           int32_t *pixels_out, int32_t *n_out);

/* ---- scene: replaces `new Scene(state)`'s Bvh + PathIntegrator + PixelIntegrator ------------ */
MFX_API int mfx_scene_create(const MfxSceneDesc *desc, MfxScene **out);
MFX_API int mfx_scene_destroy(MfxScene *scene);
/* Builds the device layouts a Sample of this MfxPrecision uses now, not inside the first Sample (a host that pipelines
 * frames calls it while the previous frame renders). */
MFX_API int mfx_scene_prepare(MfxScene *scene, int32_t precision);
/* Copies out the tree the scene traverses (as built or as supplied). */
MFX_API int mfx_scene_get_bvh(const MfxScene *scene, MfxBvhNode *nodes_out, int32_t *indices_out);
/* Bytes of the flattened scene resident in HBM for each precision. */
MFX_API int mfx_scene_device_bytes(const MfxScene *scene, uint64_t *exact_bytes, uint64_t *fast_bytes);

/* ---- finer seams (parity tests) -------------------------------------------------------------- */
/* Bvh.Hit(ray, tMin, tMax), BvhNode.fs:83, for n rays.  origins/dirs: n x 3 doubles.
 * prim = original primitive index or -1; sub = 0/1 (which triangle of a Rect); t = distance.
 * any_hit != 0: only `prim >= 0 ? occluded : clear` is meaningful (shadow query, Integrators.fs:44). */
MFX_API int mfx_bvh_hit(MfxScene *scene, int32_t precision, int32_t any_hit, int64_t n,
                        const double *origins, const double *dirs, double tmin, double tmax,
                        int32_t *prim, int32_t *sub, double *t);
/* cam.GetRay(u,v) (Camera.fs:134-139) + bvh.Hit(ray, 1e-6, 99999999.) (Integrators.fs:108).
 * uv == NULL: pixel centres, n == width*height, ray r = y*width+x. */
MFX_API int mfx_trace_primary(MfxScene *scene, int32_t precision, int64_t n, const double *uv,
                              int32_t *prim, double *t);

/* ---- the drop-in: IPixelIntegrator.Sample : int -> Texture2D<Color>, IIntegrator.fs:35-40 ---- */
/* texture = the reference's Color[w,h] (Texture.fs:21-28): element [x,y] at (x*height+y)*4
 * doubles r,g,b,a; a = 1.  A blittable Array2D<Color> can be pinned and passed directly.
 * With world > 1 only this rank's tiles are written, every other pixel is 0. */
MFX_API int mfx_pixel_integrator_sample(MfxScene *scene, const MfxSampleParams *params, double *texture);
/* Sample without the wait (the reference's loop renders frame after frame, Scene.fs:331-333 from Film.fs:67-73): the
 * kernels and the download are enqueued and the call returns; mfx_pixel_integrator_wait completes the OLDEST frame in
 * flight (texture filled, mfx_get_stats describes it).  Up to two frames per scene may be in flight -- the download of
 * frame k then runs beside the kernels of frame k+1; a third call completes the oldest first.  texture must be pinned
 * (mfx_host_register) and stay untouched until its wait returns; use one texture per frame in flight. */
MFX_API int mfx_pixel_integrator_sample_async(MfxScene *scene, const MfxSampleParams *params, double *texture);
MFX_API int mfx_pixel_integrator_wait(MfxScene *scene);
/* Same call, result left on the device: d_rgba = width*height float4, row-major (y*width+x),
 * mean over spp, zero outside this rank's tiles (so a sum-reduce over ranks assembles the frame). */
MFX_API int mfx_pixel_integrator_sample_device(MfxScene *scene, const MfxSampleParams *params,
                                               void *d_rgba_f32);
/* Same, result left on the device in the reference's own layout: d_color_wh = Color[w,h], width*height*4 doubles,
 * x-major.  With MFX_SAMPLE_STRIPES a rank's share is a set of contiguous blocks: what a multi-process host gathers. */
MFX_API int mfx_pixel_integrator_sample_device_color(MfxScene *scene, const MfxSampleParams *params,
                                                     void *d_color_wh_f64);
/* Same, host output as float RGBA row-major (PFM/PNG writers). */
MFX_API int mfx_pixel_integrator_sample_f32(MfxScene *scene, const MfxSampleParams *params, float *rgba);
MFX_API int mfx_get_stats(const MfxScene *scene, MfxStats *out);
/* Pin (cudaHostRegister) / unpin a caller buffer that will receive textures repeatedly. */
MFX_API int mfx_host_register(void *ptr, uint64_t bytes);
MFX_API int mfx_host_unregister(void *ptr);

/* ---- multi-GPU behind the same seam ------------------------------------------------------------
 * The reference host is one process with one render thread (Film.fs:67-73 -> Scene.Render -> Integrators.fs:160-172);
 * its only parallelism is Array.Parallel.iter over pixels (:164).  mfx_multi_* is that loop over GPUs: the scene is
 * replicated on every listed device, one worker thread per device lives inside the library, and the caller's single
 * thread gets IPixelIntegrator.Sample back with the whole frame.  Ownership: column stripes of 16 pixels, stripe c ->
 * devices[c % n]; every device writes its stripes straight into the caller's texture over its own PCIe link (no
 * collective: the path has no exchange step).  The frame is bit-identical to the one-GPU frame. */
typedef struct MfxMulti MfxMulti;
/* devices == NULL: the first n_devices CUDA devices (n_devices <= 0: all of them).  desc->nodes == NULL: Bvh.Build runs
 * once on the host and every replica takes that tree. */
MFX_API int mfx_multi_create(const MfxSceneDesc *desc, const int32_t *devices, int32_t n_devices, MfxMulti **out);
MFX_API int mfx_multi_destroy(MfxMulti *multi);
MFX_API int mfx_multi_device_count(const MfxMulti *multi, int32_t *n_out);
/* IPixelIntegrator.Sample over all devices -> Color[w,h] (pin it once with mfx_host_register: direct DMA from every
 * device).  params->rank / world / tile_size are ignored (the library shards), every other field as in
 * mfx_pixel_integrator_sample. */
MFX_API int mfx_multi_sample(MfxMulti *multi, const MfxSampleParams *params, double *texture);
/* The same call without the wait (one frame in flight per handle): the workers render and download while the caller goes
 * on; mfx_multi_wait completes it.  texture must stay untouched until then. */
MFX_API int mfx_multi_sample_async(MfxMulti *multi, const MfxSampleParams *params, double *texture);
MFX_API int mfx_multi_wait(MfxMulti *multi);
/* mfx_scene_prepare on every replica, side by side. */
MFX_API int mfx_multi_prepare(MfxMulti *multi, int32_t precision);
/* Same, float RGBA row-major. */
MFX_API int mfx_multi_sample_f32(MfxMulti *multi, const MfxSampleParams *params, float *rgba);
/* total: rays / paths / launches summed over the devices, ms_* of the slowest one; per_device: n entries or NULL. */
MFX_API int mfx_multi_get_stats(const MfxMulti *multi, MfxStats *total, MfxStats *per_device);

/* ---- Film (Film.fs:13-34): progressive accumulation, state kept in HBM ----------------------- */
/* Lifetime: a film borrows its scene's stream -- destroy every film BEFORE mfx_scene_destroy of its scene. */
MFX_API int mfx_film_create(MfxScene *scene, MfxFilm **out);
MFX_API int mfx_film_destroy(MfxFilm *film);
MFX_API int mfx_film_reset(MfxFilm *film);                                   /* Film.Reset, :26-30 */
/* Film.GetFrame(integrator, samples), :32-34: frame = Sample(samples); sum += frame;
 * target = sum / frameCount; texture (Color[w,h], may be NULL) receives target. */
MFX_API int mfx_film_get_frame(MfxFilm *film, const MfxSampleParams *params, double *texture);
/* ACESFilmToneMapping + sqrt + int(255.99 c) -> RGBA8 at x*4 + y*width*4 (Scene.fs:273-289,315-330)
 * applied on the device to the film's current target.  Under MFX_SKY_TRACER: the sphere sample's own display
 * transform instead -- sqrt, int(255.99 c), row j of the texture on screen row height-1-j (RayTracing.fs:456-460). */
MFX_API int mfx_film_post_process(MfxFilm *film, uint8_t *rgba8);
MFX_API int mfx_film_frame_count(const MfxFilm *film, double *out);
/* Checkpoint / resume of the only state the reference's renderer carries between frames: Film.texture (the
 * running sum, Color[w,h]) and frameCount (Film.fs:14-17).  With the counter-based RNG a resumed film continues
 * bit-exactly (pass first_sample = frames already rendered x spp). */
MFX_API int mfx_film_export(MfxFilm *film, double *sum_color_wh, double *frame_count);
MFX_API int mfx_film_import(MfxFilm *film, const double *sum_color_wh, double frame_count);

/* ---- Film over several GPUs (Film.fs:13-34 on an MfxMulti handle) --------------------------------
 * Every device accumulates, divides and tone-maps only the column stripes it owns, in its own HBM (a full-frame sum,
 * target and RGBA8 buffer per device, of which only the owned stripes are touched), and copies only its stripes of
 * what the caller asks for.  Every result is bit-identical to the one-GPU mfx_film_* on the same scene, params and seed.
 * Rules: mfx_multi_destroy fails with MFX_ERR_INVALID_ARGUMENT while a film of the handle is alive; a film call while an
 * mfx_multi_sample_async of the handle has not been waited for is refused; a plain mfx_multi_sample between film frames
 * leaves the film untouched. */
typedef struct MfxMultiFilm MfxMultiFilm;
MFX_API int mfx_multi_film_create(MfxMulti *multi, MfxMultiFilm **out);
MFX_API int mfx_multi_film_destroy(MfxMultiFilm *film);
MFX_API int mfx_multi_film_reset(MfxMultiFilm *film);                        /* Film.Reset, Film.fs:26-30 */
/* Film.GetFrame, Film.fs:18-23,32-34: Sample over all devices, sum += frame, target = sum / frameCount; texture
 * (Color[w,h], may be NULL) receives target.  params are read as mfx_multi_sample reads them: rank, world and
 * tile_size are ignored, world > 1 is refused. */
MFX_API int mfx_multi_film_get_frame(MfxMultiFilm *film, const MfxSampleParams *params, double *texture);
/* mfx_film_post_process over the devices' stripes (Scene.fs:315-330; RayTracing.fs:456-460 under MFX_SKY_TRACER),
 * byte for byte the same RGBA8 at x*4 + y*width*4. */
MFX_API int mfx_multi_film_post_process(MfxMultiFilm *film, uint8_t *rgba8);
MFX_API int mfx_multi_film_frame_count(const MfxMultiFilm *film, double *out);
/* The same checkpoint as mfx_film_export / _import (full Color[w,h] running sum + frameCount): a film exported from
 * N devices resumes on M devices or on a one-GPU MfxFilm, and the other way round. */
MFX_API int mfx_multi_film_export(MfxMultiFilm *film, double *sum_color_wh, double *frame_count);
MFX_API int mfx_multi_film_import(MfxMultiFilm *film, const double *sum_color_wh, double frame_count);

#ifdef __cplusplus
}
#endif
#endif /* MAFRIX_CUDA_H */

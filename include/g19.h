/* g19.h -- C ABI of lib2019global_b200 (the B200 radiance-loop engine).
 *
 * This is the drop-in boundary for the ONE hot path of preon7/2019global:
 * RayTracer::run and everything it calls (reference include/raytracer.h:23-87).
 * The reference has no FFI of its own; its seam is the public surface of the
 * header-only classes RayTracer / Octree / Entity / Material / Camera / Image.
 * Every entry point below names the reference interface it replaces.
 *
 * Conventions: plain C, no C++ types, no exceptions across the boundary.
 * Every function returns an int status (G19_OK == 0) unless stated otherwise.
 * Caller owns all input buffers; the library copies what it keeps.
 * One g19_ctx serves one render at a time; g19_cancel / g19_progress are the
 * only calls that may be made concurrently with a running g19_render*.
 * There is NO CPU fallback: without a CUDA device g19_create fails loudly.
 */
#ifndef G19_H
#define G19_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define G19_ABI_VERSION 6

/* ---- status codes ------------------------------------------------------- */
enum {
    G19_OK = 0,
    G19_ERR_INVALID = 1,   /* bad argument                                   */
    G19_ERR_NO_DEVICE = 2, /* no usable CUDA device (there is no CPU path)   */
    G19_ERR_CUDA = 3,      /* CUDA runtime error, see g19_last_error         */
    G19_ERR_NO_SCENE = 4,  /* render before g19_upload_scene                 */
    G19_ERR_CANCELLED = 5, /* g19_cancel observed; output is partial         */
    G19_ERR_LIMIT = 6,     /* scene exceeds a documented device-side limit   */
    G19_ERR_REJECTED = 7,  /* entity rejected by the root-overlap test       */
    G19_ERR_TIMEOUT = 8    /* shared frame: a device-side wait gave up (lost rank); the frame is dead */
};

/* ---- entities (reference include/entities.h) ---------------------------- */
/* One value per concrete reference class. A composite is ONE entity id.     */
enum g19_entity_kind {
    G19_IMP_SPHERE = 0,    /* ImpSphere(pos, radius, color)      entities.h:43-133  */
    G19_IMP_TRIANGLE = 1,  /* ImpTriangle(p1,p2,p3)              entities.h:136-306 */
    G19_EXP_RECTANGLE = 2, /* ExpRectangle(p1,p2,p3)             entities.h:308-377 */
    G19_EXP_BOX = 3,       /* ExpBox(min,max)                    entities.h:379-454 */
    G19_EXP_SPHERE = 4,    /* ExpSphere(pos, radius, color)      entities.h:457-575 */
    G19_EXP_QUAD = 5,      /* ExpQuad(pos,width,length,alpha,c)  entities.h:579-647 */
    G19_EXP_CUBE = 6,      /* ExpCube(pos,w,l,h,color)           entities.h:650-818 */
    G19_EXP_CONE = 7       /* ExpCone(pos,dir,height,radius,c)   entities.h:821-967 */
};

/* Bounce model used by G19_MODE_PATH only (the reference has no bounces;
 * reference Material, material.h:12-107, only feeds G19_MODE_REF shading). */
enum g19_bsdf {
    G19_BSDF_DIFFUSE = 0,
    G19_BSDF_MIRROR = 1,
    G19_BSDF_GLASS = 2,
    G19_BSDF_EMITTER = 3
};

/* Constructor arguments of one reference entity, in the reference's own types
 * (double points, float scalars -- the float/double split is part of the
 * bit-exact contract).
 *   kind            p[0..2]   p[3..5]   p[6..8]   f[0]    f[1]    f[2]
 *   IMP_SPHERE      pos                           radius
 *   IMP_TRIANGLE    p1        p2        p3
 *   EXP_RECTANGLE   p1        p2        p3
 *   EXP_BOX         min       max
 *   EXP_SPHERE      pos                           radius
 *   EXP_QUAD        pos                           width   length  alpha
 *   EXP_CUBE        pos                           width   length  height
 *   EXP_CONE        pos       dir                 height  radius
 * color is Material(color) (material.h:13-16). For the kinds whose reference
 * constructor takes no colour (triangle, rectangle, box) it is what a caller
 * assigns to the public Entity::material field afterwards; the reference
 * default is (1,0,0) (entities.h:21). */
typedef struct g19_entity_desc {
    int32_t kind;        /* enum g19_entity_kind */
    int32_t bsdf;        /* enum g19_bsdf (PATH mode) */
    double p[9];
    float f[4];
    double color[3];
    float emission[3];   /* radiance of a G19_BSDF_EMITTER (PATH mode) */
    float ior;           /* index of refraction of G19_BSDF_GLASS (PATH mode) */
    /* The other public fields of the reference's Material (material.h:23-29), consumed by G19_MODE_REF's shade and
     * the depth-0 slice. material_set == 0: they take the values Material(color) gives them (material.h:13-16,27,29)
     * and the fields below are ignored; 1: the caller's values, as after assigning to entity->material.<field>.  */
    int32_t material_set;
    int32_t reserved_;
    double diffuse_color[3];     /* Material::diffuse_color      default color * 0.5 (untextured blinn_phong only) */
    double specular_color[3];    /* Material::specular_color     default (1,1,1)                                   */
    double shader_parameters[3]; /* Material::shader_parameters  default (0.1, 0.7, 1): ambient, diffuse, specular  */
    double specular_power;       /* Material::specular_power     default 5                                         */
} g19_entity_desc;

/* ---- scene = Octree + the entities pushed into it (octree.h:12-68) ------ */
typedef struct g19_scene g19_scene;

/* Octree(min,max)                                            octree.h:14    */
int g19_scene_create(const double min[3], const double max[3], g19_scene** out);
void g19_scene_destroy(g19_scene* scene);
/* new <Entity>(...) followed by Octree::push_back            octree.h:20-30.
 * *out_index (nullable) receives the entity id = construction order. An
 * entity whose bounding box misses the root is still numbered but silently
 * absent from the tree, exactly like the reference; the call then returns
 * G19_ERR_REJECTED (informational). */
int g19_scene_add_entity(g19_scene* scene, const g19_entity_desc* desc, int32_t* out_index);
int g19_scene_entity_count(const g19_scene* scene);
int g19_scene_get_entity(const g19_scene* scene, int32_t index, g19_entity_desc* out);
/* Entity::boundingBox() as the reference computes it (incl. its quirks).    */
int g19_scene_entity_bbox(const g19_scene* scene, int32_t index, double out_min_max[6]);
/* The triangles a composite owns (public `triangles` members), 9 doubles
 * each. Returns the count; writes at most max_tris. IMP_SPHERE returns 0.   */
int g19_scene_entity_triangles(const g19_scene* scene, int32_t index, double* out, int max_tris);

/* Which triangles G19_MODE_PATH extracts from the composite entities (applies at the next g19_upload_scene;
 * G19_MODE_REF always traces the reference's own, bugs included):
 *   G19_SHAPES_REF    what the reference's constructors build -- ExpRectangle's p4 = -p3 (entities.h:319),
 *                     ExpSphere tessellated around -pos and without its first triangle (entities.h:475-482,520),
 *                     ExpQuad's doubled pos.z (entities.h:586), ExpCone's hard-coded direction (entities.h:825)
 *   G19_SHAPES_FIXED  what they were meant to build (csrc/fixed_shapes.cpp), behind the same entity ids          */
enum g19_shapes { G19_SHAPES_REF = 0, G19_SHAPES_FIXED = 1 };
int g19_scene_set_shapes(g19_scene* scene, int shapes);

/* Stateless forms of the two calls above, for one entity outside any scene
 * (what an Entity subclass needs to fill its public members at construction). */
int g19_entity_bbox(const g19_entity_desc* desc, double out_min_max[6]);
int g19_entity_triangles(const g19_entity_desc* desc, double* out, int max_tris);

/* Procedural scenes of BASELINE.json `configs` (SURVEY.md section 8(d)).    */
enum g19_builtin_scene {
    G19_SCENE_DEFAULT = 0,     /* main.cpp:24-57 literal (config 1)             */
    G19_SCENE_CORNELL = 1,     /* diffuse Cornell box + 2 spheres + area light  */
    G19_SCENE_CORNELL_GLASS = 2, /* same, one mirror + one glass sphere         */
    G19_SCENE_HEIGHTFIELD = 3, /* n x n heightfield, 2 n^2 ... triangles        */
    G19_SCENE_HEIGHTFIELD_ROOM = 4 /* the same surface as the far wall of a closed room with a ceiling light */
};
typedef struct g19_camera {
    double pos[3];     /* Camera::pos      camera.h:12 */
    double look_at[3]; /* Camera ctor arg  camera.h:8  */
    double focal;      /* Camera::focalDist camera.h:16 */
} g19_camera;
/* Builds a named scene; `n` is the heightfield grid size (ignored otherwise).
 * w,h select the camera pitch that centres the frame (SURVEY hard part 4).
 * out_camera / out_light (nullable) receive the matching camera and light.  */
int g19_scene_builtin(int which, int n, int w, int h, g19_scene** out,
                      g19_camera* out_camera, double out_light[3]);

/* ---- engine -------------------------------------------------------------- */
typedef struct g19_ctx g19_ctx;

enum g19_mode {
    G19_MODE_REF = 0, /* bug-for-bug reference: 1 primary ray per pixel through
                         the pixel corner, reference octree candidate semantics,
                         LAST intersecting candidate wins, Blinn-Phong + checker,
                         truncating RGB888 store (raytracer.h:23-87).          */
    G19_MODE_PATH = 1 /* path tracing: spp, pixel jitter, bounces, area light,
                         mirror/glass, nearest hit -- NOT in the reference;
                         defined by this repo's oracle (oracle/path_oracle.c). */
};

typedef struct g19_params {
    int32_t width, height; /* RayTracer::run(w,h)  raytracer.h:23 */
    int32_t mode;          /* enum g19_mode */
    int32_t spp;           /* PATH: samples per pixel (REF: ignored, 1) */
    int32_t max_depth;     /* PATH: max ray segments per camera path. 0 = the DEPTH-0 SLICE: one un-jittered
                              ray through each pixel corner (raytracer.h:41-43) traced through PATH mode's own
                              structures (nearest hit), then the reference's direct shade of that hit
                              (getTextureCoord + Material::blinn_phong_texture, material.h:48-62) and its
                              truncating store -- what RayTracer::run computes, through the PATH pipeline   */
    uint32_t seed;         /* PATH: RNG key; counter = (pixel, sample, bounce) */
    /* Image-tile sharding (SURVEY 8(e)): 32x32 tiles, tile t belongs to rank
     * t % world. rank=0, world=1 renders everything. Pixels of other ranks
     * are left untouched in the output buffers.                             */
    int32_t rank, world;
    int32_t spp_per_pass;  /* PATH: samples per wavefront pass (0 = auto)   */
    int32_t profile;       /* 1: time every kernel class with CUDA events   */
    int32_t pixels_per_pass; /* PATH: pixels of this rank per wavefront pass, in whole
                              32x32 tiles (0 = auto: the whole frame, or windows of it when
                              the per-path state would outgrow the L2 cache)            */
} g19_params;

typedef struct g19_stats {
    uint64_t samples;         /* camera paths started                         */
    uint64_t extend_segments; /* rays through traverse+intersect              */
    uint64_t shadow_segments; /* any-hit rays                                 */
    uint64_t kernel_launches; /* kernels of this library launched by the call */
    double render_ms;         /* device time of the whole call (CUDA events)  */
    /* per kernel class, only when params.profile: [raygen+extend (camera
     * segment), bounce (shade + continuation trace), -, accumulate,
     * ref_visibility, ref_shade, other]                                      */
    double class_ms[8];
    uint64_t class_launches[8];
    uint64_t node_tests, prim_tests; /* REF mode, only when profile           */
    uint64_t shade_calls;     /* PATH: surface interactions shaded            */
    uint64_t shade_calls_first; /* ... of which on the camera segment         */
    uint64_t lit_samples;     /* PATH: unoccluded next-event samples          */
    uint64_t radiance_reads;  /* PATH, tree scenes: diffuse vertices past the camera segment
                                 (their light sample reads the slot's radiance so far)        */
    uint64_t radiance_stores; /* PATH, flat scenes: paths that ended in a bounce kernel (one
                                 16-byte radiance store each; bench.py's byte model)          */
    uint64_t shade_calls_folded; /* PATH, flat scenes: last vertices shaded by the launch that found
                                 them (counted in shade_calls; no vertex record written or read) */
} g19_stats;

enum { G19_K_EXTEND = 0, G19_K_SHADE = 1, G19_K_SHADOW = 2, G19_K_ACCUM = 3,
       G19_K_REF_VIS = 4, G19_K_REF_SHADE = 5, G19_K_OTHER = 6 };

/* RayTracer(camera, light) + device selection. devices==NULL,n==0 -> the
 * current CUDA device. Fails with G19_ERR_NO_DEVICE when CUDA is unusable.  */
int g19_create(const int* devices, int n_devices, g19_ctx** out);
void g19_destroy(g19_ctx* ctx);
const char* g19_last_error(const g19_ctx* ctx); /* ctx may be NULL: create errors */

/* RayTracer::setScene(const Octree*)                       raytracer.h:21.
 * Builds the reference octree (octree.h:75-129) and the engine's own linear
 * octree on the host, flattens both and copies them to HBM.                 */
int g19_upload_scene(g19_ctx* ctx, const g19_scene* scene);

/* RayTracer::run(w,h)                                      raytracer.h:23-87.
 * Blocking; HOST pointers, each nullable:
 *   rgb888_out   w*h*3 bytes, row-major, row 0 = top (Image / QImage RGB888,
 *                image.h:9-16)
 *   hit_id_out   w*h int32: primary-hit entity id (push order), -1 = miss. REF mode: the reference's
 *                front object (last intersecting candidate). PATH mode: the NEAREST hit of the un-jittered
 *                ray through the pixel corner -- the same ray, through PATH mode's own structures; equal to
 *                REF's wherever "last hit" and "nearest hit" coincide (tests/test_path_link.py)
 *   radiance_out w*h*3 float: linear radiance (REF: the shaded colour)       */
int g19_render(g19_ctx* ctx, const g19_camera* camera, const double light[3],
               const g19_params* params, uint8_t* rgb888_out, int32_t* hit_id_out,
               float* radiance_out);
/* Progressive form of g19_render -- the reference's "incremental rendering" intent
 * (raytracer.h:31): the Qt viewer repaints from getImage() every 32 ms while run() is in flight
 * (viewer.h:18-21,36-43). After a wavefront pass, once at least min_interval_ms have gone by
 * since the last refresh, the image of the samples so far is resolved into rgb888_out and
 * on_pass(user, fraction, rgb888_out) is called on the calling thread; a non-zero return cancels
 * like g19_cancel (latency: one pass). The last call has fraction 1.0 and the final image. REF
 * mode is a single pass: one call. radiance_out (nullable) receives the final radiance only.   */
typedef int (*g19_pass_fn)(void* user, double fraction, const uint8_t* rgb888);
int g19_render_progressive(g19_ctx* ctx, const g19_camera* camera, const double light[3],
                           const g19_params* params, uint8_t* rgb888_out, float* radiance_out,
                           g19_pass_fn on_pass, void* user, int min_interval_ms);

/* Same with DEVICE pointers (HBM-resident outputs) on `stream` (a
 * cudaStream_t, NULL = legacy default). Asynchronous w.r.t. the host unless
 * params->profile; stats (nullable) are complete after the stream is synced. */
int g19_render_device(g19_ctx* ctx, const g19_camera* camera, const double light[3],
                      const g19_params* params, uint8_t* d_rgb888, int32_t* d_hit_id,
                      float* d_radiance, void* stream);
int g19_get_stats(g19_ctx* ctx, g19_stats* out);

/* Noise-targeted adaptive sampling (PATH mode): samples go where the frame is still noisy, a 32x32 tile at a time. No
 * counterpart in the reference (one sample per pixel).
 *   mode        G19_MODE_PATH only. params->spp is the most samples a pixel takes; rank / world, spp_per_pass,
 *               pixels_per_pass, profile and the g19_tune knobs mean what they mean for g19_render. Pixels of other
 *               ranks are left untouched
 *   rounds      round 0 gives every owned tile samples [0, min_spp). After each round every active tile is tested: one
 *               whose error E <= noise_target stops; any other with n samples takes samples [n, min(2n, spp)) in the next
 *               round. The render ends when no tile is active: counts are min_spp * 2^k, capped at spp
 *   error       per sample Y = 0.2126 R + 0.7152 G + 0.0722 B (FP32, of the radiance g19_render averages); per pixel
 *               S2 = sum of Y^2 (FP32, in sample order), m = 0.2126 sum(R)/n + 0.7152 sum(G)/n + 0.0722 sum(B)/n (the
 *               radiance output's means), v = max(S2 - n m^2, 0) / (n (n - 1)) -- the variance of the pixel's mean --
 *               and e = sqrt(v) / max(m, 0.05) (below 5 % of display white the test is absolute); E = the largest e
 *               over the tile's in-frame pixels
 *   outputs     all nullable, full frame, row-major. rgb888 (w*h*3 bytes) and radiance (w*h*3 floats): exactly what
 *               g19_render gives at spp = the pixel's count, so a tile that stopped at n samples holds the bytes of a
 *               uniform render at n; variance (w*h floats): v at that count; spp (w*h int32): that count
 *   stats       samples = the sum over owned in-frame pixels of their count (g19_render's count when every tile
 *               reaches spp); the other fields as for g19_render
 *   errors      G19_ERR_INVALID: ctx, params or adaptive NULL, REF mode, noise_target not finite or <= 0, min_spp < 2
 *               or > spp, max_depth < 1 (and whatever g19_render refuses); G19_ERR_NO_SCENE before an upload;
 *               G19_ERR_CANCELLED: g19_cancel, seen between passes -- the outputs are then left as they were
 *   device form stream-ordered on `stream` (a cudaStream_t, NULL = legacy default), but it synchronises `stream` once
 *               per round to read how many tiles are still active (a pinned word): one host round trip per round,
 *               and there are at most ceil(log2(spp / min_spp)) + 1 rounds. The host form blocks.                  */
typedef struct g19_adaptive {
    float noise_target; /* tau > 0, finite: a tile stops once its error E <= tau                   */
    int32_t min_spp;    /* samples every owned pixel takes before the first test, 2 <= min_spp <= spp */
} g19_adaptive;
int g19_render_adaptive(g19_ctx* ctx, const g19_camera* camera, const double light[3], const g19_params* params,
                        const g19_adaptive* adaptive, uint8_t* rgb888_out, float* radiance_out, float* variance_out,
                        int32_t* spp_out);
int g19_render_adaptive_device(g19_ctx* ctx, const g19_camera* camera, const double light[3], const g19_params* params,
                               const g19_adaptive* adaptive, uint8_t* d_rgb888, float* d_radiance, float* d_variance,
                               int32_t* d_spp, void* stream);

/* Batched ray queries: what does each ray hit first, or is anything in its way (Embree's rtcIntersect /
 * rtcOccluded, OptiX's closest-hit / any-hit). No counterpart in the reference: its Octree::intersect
 * (octree.h:46-68) returns candidates, not hits.
 *   scene       the PATH view of the last g19_upload_scene, with the shapes that upload used (G19_SHAPES_REF /
 *               G19_SHAPES_FIXED); REF mode's octree and its "last candidate wins" rule are not involved
 *   rays        n x 8 floats (ox, oy, oz, tmax, dx, dy, dz, 0), 16-byte aligned. The direction need not be unit
 *               length: it is normalised, and t is the distance along the unit direction
 *   invalid     a non-finite origin or direction, a zero direction, or tmax not > 0 (NaN included): a miss,
 *               nothing traversed
 *   hit         the nearest primitive with 0 <= t < tmax, by the render's own hit functions. A ray that starts on a
 *               surface may hit it at t = 0: offset origins off surfaces (the engine offsets by 1e-3 along the normal)
 *   outputs     out_entity n int32 (required): the entity id (push order; a merged parallelogram reports the
 *               triangle the hit lies in, as hit_id_out of g19_render does); out_t n floats and out_normal n x 3
 *               floats (both nullable): t and the normal -- the geometric normal turned against the ray for
 *               triangles, (p - c) / r for spheres. A miss is entity -1, t = +inf, normal (0, 0, 0)
 *   G19_CAST_ANY_HIT  occlusion query: out_entity = an entity hit with t < tmax (which one is unspecified), or -1;
 *               out_t and out_normal must be NULL
 *   G19_CAST_COUNT    tally node / primitive tests into g19_stats (tree scenes, with walks that count: 1 and 4)
 *   structure   flat scenes: the packed pair loops over the staged scene; tree scenes: the walk g19_tune("walk")
 *               selects, with the render's knobs (walk_steps, bvh_stack, coop_leaf, refill, trace_occ)
 *   stats       g19_get_stats then reports the cast: extend_segments = n (nearest hit) or shadow_segments = n
 *               (any hit), kernel_launches, render_ms (device time), node_tests / prim_tests with G19_CAST_COUNT
 *   errors      G19_ERR_INVALID: ctx NULL, n < 0, rays or out_entity NULL with n > 0, rays not 16-byte aligned,
 *               out_t / out_normal with G19_CAST_ANY_HIT, unknown flag bits; G19_ERR_NO_SCENE before any upload.
 *               n == 0 returns G19_OK and launches nothing
 * A cast touches no render buffer: a render's output does not depend on casts before it. One call per context at a
 * time, as for renders.
 * g19_cast_rays: HOST pointers, blocking; the rays are staged in a device buffer the context keeps (grown on demand).
 * g19_cast_rays_device: DEVICE pointers, asynchronous on `stream` (a cudaStream_t, NULL = legacy default).     */
#define G19_CAST_ANY_HIT 1u
#define G19_CAST_COUNT 2u
int g19_cast_rays(g19_ctx* ctx, int32_t n, const float* rays, uint32_t flags,
                  int32_t* out_entity, float* out_t, float* out_normal);
int g19_cast_rays_device(g19_ctx* ctx, int32_t n, const float* d_rays, uint32_t flags,
                         int32_t* d_entity, float* d_t, float* d_normal, void* stream);

/* Multi-GPU (SURVEY.md 8(e)): one process and one g19_ctx per GPU, image
 * tiles interleaved by params->rank/world. A rank's pixels form a compact
 * "local pixel" array: local tile j is global tile j*world+rank (row-major
 * tile order), 1024 pixels per tile, row-major inside the tile, out-of-frame
 * positions of edge tiles included as padding.
 *   g19_tile_pixels          entries in that array for (w,h,rank,world)
 *   g19_render_tiles_device  like g19_render_device, but fills the compact
 *                            arrays (rgb: 3 B, ids: int32, rad: 3 floats per
 *                            entry) -- the payload a rank sends to rank 0
 *   g19_untile_device        scatters one rank's compact arrays into the
 *                            full row-major frame (what rank 0 runs on each
 *                            received payload; other pixels untouched)      */
int64_t g19_tile_pixels(int width, int height, int rank, int world);
int g19_render_tiles_device(g19_ctx* ctx, const g19_camera* camera, const double light[3],
                            const g19_params* params, uint8_t* d_tile_rgb, int32_t* d_tile_ids,
                            float* d_tile_rad, void* stream);
int g19_untile_device(g19_ctx* ctx, int width, int height, int rank, int world,
                      const uint8_t* d_tile_rgb, const int32_t* d_tile_ids, const float* d_tile_rad,
                      uint8_t* d_rgb888, int32_t* d_hit_id, float* d_radiance, void* stream);

/* Shared frame: the same exchange WITHOUT a collective call or a staging copy. Rank 0 owns a
 * frame in its HBM; the other ranks map it (CUDA IPC, reached over NVLink / NVSwitch) and their
 * resolve kernel stores each finished pixel straight into place (RGB888 + float radiance), then
 * signals a system-scope counter in the owner's memory. No counterpart in the reference (one
 * process, one thread); the frame plays the role of RayTracer::_image (raytracer.h:25,93).
 *   g19_frame_create    owner (rank 0) allocates                 -> Image(w,h), image.h:9
 *   g19_frame_export    fills a G19_FRAME_BLOB_BYTES blob to ship to the other ranks (any transport)
 *   g19_frame_import    another rank maps the owner's frame
 *   g19_render_to_frame every rank, same (camera, params) except params->rank: render my tiles into
 *                       the frame; asynchronous on `stream`; frames must be rendered in lockstep
 *   g19_frame_wait      owner: enqueue a wait on `stream` until all `world` ranks have delivered the
 *                       frame last passed to g19_render_to_frame; work enqueued behind it sees it whole
 *   g19_frame_release   owner: enqueue "done reading this frame"; the other ranks' next resolve waits
 *                       for it (device side, never the host) before overwriting pixels
 *   g19_frame_read      owner: enqueue copies of the frame into host (pinned) or device buffers
 *   g19_frame_pointers  owner's device pointers (row-major, row 0 = top)
 *   g19_frame_timeouts  device-side spins that gave up after 5 s (a lost rank); 0 in a healthy run
 *   g19_frame_status    synchronises `stream`, then G19_OK or G19_ERR_TIMEOUT. A spin that gives up raises a sticky
 *                       word in the calling process's mapped host memory; from then on EVERY g19_frame_* /
 *                       g19_render_to_frame call on that frame returns G19_ERR_TIMEOUT (its pixels may be
 *                       incomplete and a late arrival of the lost rank would count towards a later frame): destroy
 *                       it and create a new one. Call g19_frame_status before trusting what g19_frame_read copied. */
typedef struct g19_frame g19_frame;
#define G19_FRAME_BLOB_BYTES 128
int g19_frame_create(g19_ctx* ctx, int width, int height, g19_frame** out);
int g19_frame_export(g19_ctx* ctx, g19_frame* frame, void* blob, size_t blob_bytes);
int g19_frame_import(g19_ctx* ctx, const void* blob, size_t blob_bytes, g19_frame** out);
void g19_frame_destroy(g19_frame* frame);
int g19_frame_pointers(g19_frame* frame, uint8_t** d_rgb888, float** d_radiance);
int g19_render_to_frame(g19_ctx* ctx, const g19_camera* camera, const double light[3],
                        const g19_params* params, g19_frame* frame, void* stream);
int g19_frame_wait(g19_ctx* ctx, g19_frame* frame, int world, void* stream);
int g19_frame_release(g19_ctx* ctx, g19_frame* frame, void* stream);
int g19_frame_read(g19_ctx* ctx, g19_frame* frame, uint8_t* rgb888_out, float* radiance_out, void* stream);
int g19_frame_timeouts(g19_ctx* ctx, g19_frame* frame, unsigned* out);
int g19_frame_status(g19_ctx* ctx, g19_frame* frame, void* stream);

/* Tuning knobs (DESIGN.md section 9): "lanes", "pass_slots", "leaf_max", "refill", "coop_leaf", "walk_steps",
 * "leaf_batch", "walk", "tree_build", "debug_tree", ... g19_create reads them ONCE from the
 * environment (G19_LANES, ...); this call changes one afterwards (value NULL = back to the default). Nothing
 * on the render path reads the environment. No counterpart in the reference (it has no knobs, SURVEY.md 5). */
int g19_tune(g19_ctx* ctx, const char* key, const char* value);

/* RayTracer::stop()/running()                              raytracer.h:89-91 */
int g19_cancel(g19_ctx* ctx);
/* Fraction of the current render already enqueued+finished, 0..1.            */
int g19_progress(g19_ctx* ctx, double* out_fraction);

/* Unit-level probes (used by the parity tests; they run the SAME device
 * functions as the render kernels, one thread per ray).
 * Entity::intersect(ray, point, normal)                    entities.h:26    */
int g19_probe_intersect(g19_ctx* ctx, int32_t entity, int n, const double* origins,
                        const double* dirs, int32_t* out_hit, double* out_points,
                        double* out_normals);
/* Octree::intersect(ray) candidate list                    octree.h:46-68.
 * Writes up to max_out entity ids for ONE ray, returns the count in *out_n. */
int g19_probe_candidates(g19_ctx* ctx, const double origin[3], const double dir[3],
                         int32_t* out_ids, int max_out, int* out_n);

/* The linear octree PATH mode traverses (the engine's own build of what Octree::push_back,
 * octree.h:20-43,75-129, builds for the reference; large scenes build it on the GPU): node records
 * (first, count|leaf bit31) as 2 x uint32 each, and the concatenated leaf primitive lists. Pass
 * NULL / 0 to query the sizes.                                                                  */
int g19_probe_path_tree(g19_ctx* ctx, uint32_t* nodes_out, uint32_t max_nodes, uint32_t* index_out,
                        uint32_t max_index, uint32_t* n_nodes, uint32_t* n_index);

/* Entity::getTextureCoord(point)                           entities.h:32    */
int g19_probe_texcoord(g19_ctx* ctx, int32_t entity, int n, const double* points, int32_t* out_uv);
/* Material::blinn_phong_texture / blinn_phong              material.h:31-62.
 * One call per point: ray direction, light, hit point, normal, (u,v);
 * textured=0 selects the untextured variant. out_rgb: 3 doubles in [0,1].   */
int g19_probe_shade(g19_ctx* ctx, int32_t entity, int textured, const double ray_dir[3],
                    const double light[3], const double point[3], const double normal[3], int u, int v,
                    double out_rgb[3]);

#ifdef __cplusplus
}
#endif
#endif /* G19_H */

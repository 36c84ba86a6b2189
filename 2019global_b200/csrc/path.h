// path.h -- G19_MODE_PATH: host-side driver of the wavefront path tracer.
//
// Nothing here has a counterpart in the reference (it casts one primary ray
// per pixel and shades directly, raytracer.h:32-86). The transport model is
// defined by this repo and pinned by oracle/path_oracle.c (FP64, brute force):
//   * camera: the reference's pinhole (raytracer.h:26-30) with a uniform
//     jitter in [0,1)^2 added to the integer pixel corner
//   * geometry: the primitives each entity would test in REF mode, intersected
//     properly (nearest hit, t > 0, Moller-Trumbore / analytic sphere)
//   * BSDFs: lambert (albedo = clamp(Material::color,0,1)), mirror, dielectric
//   * light: triangle emitters, next-event estimation at diffuse hits, emission
//     counted on camera rays and after specular bounces only
//   * max_depth = maximum number of ray segments along the camera path
//   * RNG: Philox4x32-7, counter (pixel, sample, bounce, stream), key (seed, K)
#pragma once

#include <atomic>
#include <cstdint>
#include <string>

#include <cuda_runtime.h>

#include "g19.h"
#include "kernels.h"
#include "scene.h"

namespace g19 {

constexpr int kMaxPathDepth = 64;    // segments per path
constexpr int kMaxTreeDepth = 14;    // linear-octree levels below the root
constexpr int kBvhSmemStack = 12;    // BVH walks: levels of the postponed-children stack kept in shared memory (8 / 12 / 16 / 24 / 32: 358 / 358 / 363 / 363 / 373 ms: the L1 is what the carve-out leaves)
constexpr int kNumQueues = 6;        // (diffuse, mirror, glass) x two bounce parities
// Queue entries are reserved in warp-private chunks; a launch can leave at most one partly used
// chunk per warp and queue behind (padded with an invalid marker): 2 Mi entries of slack cover
// 148 SMs x 64 warps x 64 entries x 3 producer kernels.
constexpr size_t kQueueSlack = size_t(2) << 20;
enum { Q_RAYS = 0, Q_DIFFUSE = 1, Q_MIRROR = 2, Q_GLASS = 3 }; // column of PassArgs::counts (material = g19_bsdf + 1)

struct PathSceneD {
    const PathNodeD* nodes;
    const uint32_t* index;   // leaf lists: n_index primitive ids (a primitive appears in every leaf it overlaps)
    const PrimHot* hot;      // 64-byte intersection records by primitive id
    const PrimCold* cold;
    const MaterialD* materials;
    const LightD* lights;
    int32_t n_nodes, n_index, n_prims, n_lights, tree_depth;
    int32_t n_par, n_tri;    // flat scenes: primitives sorted parallelograms | triangles | spheres
    const float* pairs;      // flat scenes: the same primitives as PAIRS for the packed-FP32 loops (path.cu build_pairs)
    int32_t pairs_bytes;
    const int32_t* prim_entity; // 2 per primitive: the entity id REF mode would report (both halves of a merged parallelogram)
    float root_lo[3], root_size[3];
    float grid_scale[3];     // 2^kMaxTreeDepth / root_size: world position -> coordinate on the finest octree grid
    const uint2* top;        // direct index over the first top_level levels (tree_build.cu top_table_kernel), or nullptr
    int32_t top_level;
    // bounding-volume hierarchy (bvh_build.cu), the structure tune walk=3 traverses; nullptr = not built
    const float4* bvh_nodes; // 4 x float4 per internal node: both children's boxes and references
    const uint4* bvh4_nodes; // the 4-wide form (walk=4): 64 B per node, boxes quantised to 16 bits on the root box's grid
    const float4* bvh_prims; // the hot records in leaf order, original primitive id in row 3 .w
    const uint32_t* bvh_big; // primitives kept out of the hierarchy (much larger than the rest): tested up front,
    int32_t n_big;           // kind-sorted (big_par parallelograms, big_tri triangles, spheres) ...
    const float* bvh_big_pairs; // ... as primitive PAIRS through the packed-FP32 loops of the flat scenes
    int32_t big_par, big_tri;
    uint32_t bvh_root;       // node index, leaf reference, or 0xffffffff (nothing in the hierarchy)
};

// A flat scene's primitive pairs (PathSceneD::pairs, same record layout), passed to the flat bounce kernels as a launch
// parameter of their own when every kind group fits: their pair loops are then unrolled to these capacities and read the
// coefficients as constant-bank (uniform) operands instead of per-thread registers loaded from shared memory. Not a
// __constant__ symbol: several contexts and lanes render concurrently. 1664 B of the 32 KB parameter space; not in
// PassArgs, which every other kernel gets too.
constexpr int kUniPlanarPairs = 8; // per planar kind (parallelograms, triangles)
constexpr int kUniSpherePairs = 4;
struct FlatPairsU {
    ulonglong2 par[kUniPlanarPairs][6]; // rows a, b, c of two parallelograms, every coefficient a float2
    ulonglong2 tri[kUniPlanarPairs][6];
    ulonglong2 sph[kUniSpherePairs][2]; // (-centre, radius^2) of two spheres
};

struct PathCamera { // float copies of the reference basis (RefCamera)
    float pos[3], top_left[3], left[3], up[3];
};

struct DeviceArray {
    void* p = nullptr;
    size_t bytes = 0;
    cudaError_t ensure(size_t need);
    void release();
};

// A temporary of the scene builders, from the device's stream-ordered memory pool (cudaMallocAsync / cudaFreeAsync on the
// builder's stream): no device synchronisation per allocation, and the pool keeps the memory for the next upload.
struct PoolArray {
    void* p = nullptr;
    size_t bytes = 0;
    cudaStream_t stream = nullptr;
    cudaError_t ensure(size_t need, cudaStream_t s);
    void release();
};
void path_pool_keep(); // raise the release threshold of the current device's default pool (idempotent)

struct PathSceneBuffers {
    DeviceArray nodes, prim_index, hot, cold, materials, lights, pairs, prim_entity, top;
    DeviceArray bvh_nodes, bvh4_nodes, bvh_prims, bvh_big, bvh_big_pairs;
    PathSceneD view{};
    FlatPairsU upairs{};       // view.pairs again, for the flat bounce kernels' FlatPairsU parameter
    bool upairs_fit = false;   // the scene is flat and its kind groups fit FlatPairsU
    bool has_bsdf[4] = {false, false, false, false};
    unsigned long long upload_serial = 0; // counts path_upload calls: a new number = a different scene
};

// Wavefront state of ONE pass in flight (P path slots, slot = sample_in_pass * window + pixel_in_window).
struct PathLane {
    size_t capacity = 0;       // slots
    bool L_written_whole = false; // the last pass on this lane was a flat scene's: L holds its radiance, not zeros
    DeviceArray hp, dw, tp;    // tree scenes: float4[P] vertex state by slot (hit point+primitive, direction+pixel, throughput+sample)
    DeviceArray L;             // radiance of the slot's path: float4[P] (flat scenes) / float[3][P] (tree scenes)
    DeviceArray queues;        // tree scenes: uint32[6][P + slack]: (diffuse, mirror, glass) of even / odd bounces
    DeviceArray recs;          // flat scenes: float4[4][2][(P + slack) + (P + 2 slack | 0)] dense vertex records
    DeviceArray rays;          // float4[3][2P + slack]: ray queue of one bounce (tree scenes only)
    DeviceArray rkeys, perm, sort_tmp; // ray_sort.cu: uint16[2][2P + slack] keys (in | sorted), uint32[2P + slack] fetch order, CUB scratch
    DeviceArray counts;        // uint32[kMaxPathDepth+1][5]: queue lengths per bounce + ray fetch cursors
};

// Up to kMaxLanes passes are kept in flight, each on its own stream with its own PathLane: a pass is a chain of
// 7-40 dependent kernels, every one of which ends in a tail where SMs idle (ncu: sm__cycles_active
// 84-95 % of elapsed; the deep bounces of tree scenes run a handful of long rays at 15 % issue
// utilisation) -- the other pass's kernels fill those holes. Only `accumulate` is ordered across
// the lanes (events), so the per-pixel sums are still taken in sample order.
constexpr int kMaxLanes = 8;
struct PathWork {
    PathLane lane[kMaxLanes];
    cudaStream_t side[kMaxLanes] = {}; // streams of lanes 1.. (lane 0 runs on the caller's; side[0] unused)
    cudaEvent_t ev_fork = nullptr, ev_join[kMaxLanes] = {}, ev_acc[kMaxLanes] = {};
    // Frames in a row (tune overlap_frames): the side lanes of frame k + 1 need not wait for frame k's join, resolve and
    // gather -- their passes touch lane-private buffers only; what they share with the caller's stream is the statistics
    // block (two of them, by frame parity, the next frame's zeroed at this frame's start: ev_start) and `accum` (only the
    // accumulate launches touch it, and those are chained behind the frame's memset through pass 0 on the caller's stream).
    cudaEvent_t ev_start[2] = {nullptr, nullptr};
    unsigned long long frame_serial = 0;
    unsigned long long overlap_key = 0; // (scene, pass size, lanes, depth ...) of the last frame that completed its enqueue, 0 = none
    int totals_parity = 0;
    DeviceArray totals;        // uint64[8]: extend segments, shadow segments, ...
    DeviceArray accum;         // float[3][n_local_pix]; adaptive renders: float[4][n_local_pix] (+ sum of Y^2 per pixel)
    // adaptive renders only (path_render_adaptive), allocated by the first one: per local tile its sample count, the active
    // flag the tile test sets, two compacted lists of active local tiles (this round's, the next round's) with their length
    // at [0], and pinned host memory for the next list's length and the counts (read once per round)
    DeviceArray tile_n, tile_flag, tile_list;
    int32_t* tile_h = nullptr; // [0] active tiles, [1 ..] tile_n
    size_t tile_h_n = 0;
    DeviceArray rad_l, rgb_l;  // resolved local-pixel outputs
    DeviceArray iota;          // uint32[2P + slack] 0, 1, 2, ...: the values the ray sort permutes
    size_t iota_n = 0;
    // How many rays each bounce queued the last time this workload was rendered: the ray sort covers that many entries
    // (+ a margin) instead of the queue's capacity. Kept as a running maximum on the device (trace_kernel), copied to
    // pinned host memory at the end of a frame; a stale or missing hint costs speed, never correctness.
    DeviceArray ray_hint_d;    // uint32[kMaxPathDepth + 1]
    uint32_t* ray_hint_h = nullptr;
    unsigned long long hint_key = 0; // (scene, pass size, depth) the hints belong to
    // event pool for params.profile
    cudaEvent_t* events = nullptr;
    int n_events = 0, used_events = 0;
    int event_class[32768];
    bool totals_pending = false;
    cudaStream_t totals_stream = nullptr;
};

// Tuning knobs (DESIGN.md section 9). Read ONCE from the environment at g19_create (G19_LANES, G19_PASS_SLOTS, ...),
// changed afterwards only through g19_tune: no getenv on the render path.
struct PathTuning {
    int lanes = 4;            // passes kept in flight
    long long pass_slots = 0; // path slots per pass (0 = auto)
    int leaf_max = 8;         // primitives per octree leaf (read at scene upload)
    int refill = 8;           // trace_kernel: idle lanes per warp that trigger a ray fetch
    int coop_leaf = 1;        // warp-cooperative leaf tests
    int walk_steps = 0;       // cell moves / node visits per round of the tree walk (0 = auto: 2 for the octree walk, 8 / 5 for the binary / 4-wide BVH)
    int leaf_batch = 0;       // primitives per ray and round (0 = auto: 16 cooperative, 4 sequential)
    int tree_build = -1;      // -1 auto (device from 4096 primitives), 0 host, 1 device
    int debug_tree = 0;       // print octree statistics at upload
    int walk = 4;             // tree walk: 4 = 4-wide quantised bounding-volume hierarchy (Bvh4Walk, bvh_build.cu), 3 = its binary form (BvhWalk),
                              // 1 = point-location restart walk over the linear octree (TreeWalk2); 0 and 2 are taken as 1.
                              // Room scene, 1080p x 64 spp: 566 / 378 / 345 ms for 1 / 3 / 4 (866 for round 1's parametric stack walk)
    int trace_occ = 4;        // CTAs per SM of trace_kernel (4 = 64 registers, 114 bytes of spills: the walk is bound by memory
                              // latency, a third more warps in flight buys more than the spills cost -- room scene 775 -> 687 ms)
    int top_level = 7;        // levels covered by the walk's direct-index table (0 = none; capped at tree depth - 2): 16 MB at 7; ROOM 668 / 630 / 611 ms at 0 / 6 / 7
    int overlap_frames = 1;   // frames rendered back to back: the side lanes start the next frame's passes behind their own, not behind the join
    int flat_uniform = 1;     // flat scenes whose pairs fit FlatPairsU: the bounce kernels' pair loops read them from the launch parameters
    int bvh_stack = kBvhSmemStack; // walk=3/4: levels of the postponed-children stack in shared memory (1 KB per level and CTA)
    int bvh_spec = 1;         // walk=3: a lane that reaches a leaf postpones it and keeps descending
    int bvh_leaf = 4;         // walk=3: primitives per BVH leaf at most (1..8; read at scene upload)
    int upload_threads = 0;   // host threads of the primitive extraction at scene upload (0 = auto: one below 32 Ki entities, else up to 16)
    int sort_rays = -1;       // tree scenes: reorder each bounce's ray queue by origin cell / kind / octant before the walk (ray_sort.cu).
                              // -1 = auto: on for the octree walks (room scene 611 -> 566 ms), off for the BVH walk (397 with, 378 without:
                              // its walk is short enough for the sort to cost more than the coherence brings)
    int ref_heavy = 128;      // REF mode: node expansions after which a ray is spread over many warps (ref_heavy_kernel; 0 = never)
};
void path_tuning_from_env(PathTuning& t);
bool path_tuning_set(PathTuning& t, const char* key, const char* value); // false: unknown key

struct PathRenderArgs {
    PathTuning tune;
    RefCamera cam;
    g19_params params;
    TileMap map;
    uint8_t* d_rgb;   // full-frame outputs (nullable)
    float* d_rad;
    int32_t* d_ids;
    uint8_t* t_rgb;   // compact local-pixel outputs (nullable)
    float* t_rad;
    // primary-hit AOV (nullable): entity id / hit point / facing normal of the UN-jittered ray through each pixel
    // corner -- the ray the reference casts (raytracer.h:41-43) -- by local pixel; points/normals as three FP64 planes
    int32_t* ids_l = nullptr;
    double* points_l = nullptr;
    double* normals_l = nullptr;
    // shared frame (possibly a peer mapping of rank 0's memory): resolve stores straight into it
    uint8_t* frame_rgb = nullptr;
    float* frame_rad = nullptr;
    unsigned* frame_flags = nullptr;
    unsigned* frame_status = nullptr; // mapped host word raised by a device-side wait that gives up
    unsigned frame_need_consumed = 0;
    // progressive refresh (g19_render_progressive): d_rgb is resolved and copied to h_rgb between passes
    g19_pass_fn on_pass = nullptr;
    void* pass_user = nullptr;
    uint8_t* h_rgb = nullptr;
    int min_interval_ms = 0;
    cudaStream_t stream;
    int sm_count;
    std::atomic<int>* cancel;
    std::atomic<int>* progress_milli;
    cudaEvent_t cls0, cls1;
};

// tree_build.cu: the linear octree built level by level on the device (same rules as path.cu's host builder)
int path_build_tree_device(const float* d_boxes, uint32_t n_prims, const float root_lo[3], const float root_size[3],
                           int leaf_max, int max_depth, cudaStream_t s, PathNodeD** d_nodes, uint32_t* n_nodes,
                           uint32_t** d_index, uint32_t* n_index, int* tree_depth, std::string& err);
// bvh_build.cu
int path_build_bvh_device(const float* d_boxes, const uint32_t* d_ids, uint32_t n, const float root_lo[3], const float root_size[3],
                          const PrimHot* d_hot, int leaf_max, cudaStream_t s, DeviceArray& nodes, DeviceArray& nodes4, DeviceArray& prims,
                          uint32_t* root, std::string& err);
int path_build_top_table(const PathNodeD* d_nodes, int top_level, uint2* d_table, cudaStream_t s);
int path_upload(PathSceneBuffers& b, const g19_scene& scene, const PathTuning& tune, cudaStream_t stream, std::string& err);
int path_render(PathSceneBuffers& b, PathWork& w, const PathRenderArgs& a, g19_stats& stats, std::string& err);
int path_finish_stats(PathWork& w, g19_stats& stats, std::string& err);
// Noise-targeted adaptive render (g19_render_adaptive, include/g19.h): rounds of passes over the compacted list of the
// tiles whose error is still above tau; a.params.spp is the most samples a tile takes. Full-frame outputs (nullable): rgb and
// radiance as path_render gives them at each tile's count, the variance of each pixel's mean, the tile's count.
// Synchronises a.stream once per round. Host-pointer forms, progressive refresh and the shared frame are not served here.
int path_render_adaptive(PathSceneBuffers& b, PathWork& w, const PathRenderArgs& a, float tau, int min_spp, float* d_var,
                         int32_t* d_spp, g19_stats& stats, std::string& err);
// Batched ray queries (g19_cast_rays) against the PATH view, on `stream`. Their state is their own, so a cast leaves every
// render buffer as it was.
struct PathCastWork {
    DeviceArray counters;        // uint64[10]: walk tallies at [7] / [8] (where flush_walk_counts adds them), ray cursor at [9]
    bool counts_pending = false; // the last call was a counting cast whose tallies g19_get_stats has not read yet
};
int path_cast(const PathSceneBuffers& b, PathCastWork& cw, const PathTuning& tune, int32_t n, const float* d_rays, uint32_t flags,
              int32_t* d_ids, float* d_t, float* d_normals, cudaStream_t stream, int sm_count, g19_stats& stats, std::string& err);
int path_cast_finish_stats(PathCastWork& cw, g19_stats& stats, std::string& err);
void path_release(PathSceneBuffers& b, PathWork& w);

// ---- path_kernels.cu -------------------------------------------------------
struct PassArgs {
    PathSceneD scene;
    PathCamera cam;
    TileMap map;
    uint32_t seed;
    int32_t spp_pass;      // samples in this pass
    int32_t sample_base;   // first sample index of this pass
    int32_t max_depth;
    uint32_t n_slots;      // spp_pass * pix_count
    uint32_t pix_base;     // the pass covers local pixels [pix_base, pix_base + pix_count)
    uint32_t pix_count;
    float4* hp;            // vertex: hit point, primitive
    float4* dw;            // vertex: incoming direction, pixel
    float4* tp;            // throughput, sample (not written for the camera segment: 1, slot / n_local_pix)
    float* L;              // radiance of the slot's path: tree scenes 3 planes of `plane` floats (added to as the path
                           // goes), flat scenes float4[plane] (stored once, when the path ends)
    size_t plane;          // slots per plane (capacity)
    uint32_t* q[6];        // [bounce parity * 3 + (kind - 1)]
    uint32_t kind_mask;    // bit (kind - 1): the scene has a material of that class
    size_t queue_cap;      // entries per queue (P + chunk slack); flat scenes: of the diffuse record array
    size_t spec_cap;       // flat scenes: entries of the array mirror and glass share (P + 2 x slack), 0 = no specular material
    // flat scenes: the queues hold the vertex records themselves (dense, 64 B per vertex) in four float4
    // planes of 2 x (queue_cap + spec_cap) entries: per bounce parity the diffuse array, then the array mirror
    // (upwards) and glass (downwards) share -- path_kernels.cu rec_queue. A padding entry has slot kInvalid.
    // hp/dw/tp/q above then serve tree scenes only (slot-indexed).
    float4* rec_ls;        // radiance so far, slot
    float4* rec_hp;        // hit point, primitive
    float4* rec_dw;        // incoming direction, pixel
    float4* rec_tp;        // throughput, sample
    float4* ray0;          // tree scenes: the bounce's ray queue (origin, tmax)
    float4* ray1;          //   (direction, slot | flags)
    float4* ray2;          //   (light sample rgb) of shadow rays
    uint16_t* rkey;        //   sort key per queued ray (ray_sort.cu), nullptr = rays are walked in queue order
    const uint32_t* perm;  //   the order trace_kernel fetches the first perm_n rays in (sorted by key); the rest in queue order
    uint32_t perm_n;
    uint32_t* ray_hint;    //   [bounce] running maximum of the rays queued (nullable)
    uint32_t* counts;      // [kMaxPathDepth+1][4] queue lengths (column 0: rays) + [kMaxPathDepth+1] fetch cursors
    unsigned long long* totals;
    float* accum;          // 3 planes of n_local_pix
    // shared-memory staging (see path_kernels.cu stage_scene)
    int32_t stage_nodes, stage_prims, stage_cold, stage_lights, stack_levels;
    int32_t refill;        // trace_kernel: idle lanes per warp that trigger a fetch of new rays
    int32_t walk_steps, leaf_batch; // tree walk: cell moves / primitives tested per round (TreeWalk2::step)
    int32_t coop_leaf;     // tree walk: leaf tests spread over the whole warp (default; G19_COOP_LEAF=0: sequential)
    int32_t trace_occ;     // CTAs per SM of trace_kernel (3 or 4)
    int32_t bvh_spec;      // BvhWalk: speculative traversal (PathTuning::bvh_spec)
    int32_t fold_last;     // this launch shades the path's last vertex in place (flat scenes, bounce max_depth - 2)
    int32_t walk;          // tree walk variant (PathTuning::walk); +2 when the walk counts its node / primitive tests
    int32_t flat_uniform;  // the flat bounce kernels trace through their FlatPairsU parameter (unrolled pair loops)
    const FlatPairsU* upairs; // host memory (PathSceneBuffers::upairs): what the launchers pass as that parameter
    // adaptive passes (path_render_adaptive), nullptr otherwise: the window positions [pix_base, pix_base + pix_count) index
    // a compacted list of local tiles, position pos = local pixel (tiles[pos >> 10] << 10) | (pos & 1023); the camera
    // segment and accumulate run their LIST forms, and accumulate adds the per-sample luminance squared to accum's fourth plane
    const uint32_t* tiles;
};

// path.cu: the PassArgs fields that follow from the scene and the tuning alone (staging sizes, walk and its knobs);
// count = the walk tallies its node / primitive tests
PassArgs path_pass_setup(const PathSceneBuffers& b, const PathTuning& tune, bool count);
// tree scenes: the camera segment
void launch_raygen_extend(const PassArgs& a, int sm_count, cudaStream_t s);
// tree scenes: one material queue; false = nothing to launch for this (bounce, kind): specular vertices on the last segment
bool launch_bounce(const PassArgs& a, int bounce, int kind, int sm_count, cudaStream_t s);
void launch_trace(const PassArgs& a, int bounce, int sm_count, cudaStream_t s); // tree scenes: after the bounce's shade launches
// ray_sort.cu
size_t ray_sort_temp_bytes(size_t n);
void launch_iota(uint32_t* out, size_t n, cudaStream_t s);
cudaError_t launch_ray_sort(void* temp, size_t temp_bytes, const uint16_t* keys_in, uint16_t* keys_out, const uint32_t* iota,
                            uint32_t* perm, size_t n, cudaStream_t s);
bool path_scene_is_flat(const PassArgs& a);
// flat scenes, bounce 0: the camera segment and the first vertex in ONE launch (at max_depth 1 the only one)
void launch_bounce_first_fused(const PassArgs& a, int sm_count, cudaStream_t s);
// flat scenes, a bounce before the last (bounce 0 only with mirror / glass, whose camera hits the fused launch queued):
// one launch for all material queues; false = no launch (the scene has no surface a path goes on from)
bool launch_bounce_flat(const PassArgs& a, int bounce, int sm_count, cudaStream_t s);
void launch_accumulate(const PassArgs& a, cudaStream_t s);
void launch_primary(const PassArgs& a, int32_t* ids_l, double* points_l, double* normals_l, int sm_count, cudaStream_t s);
// batched ray queries (g19_cast_rays): n ray records of two float4 (origin, tmax) (direction, -) -> entity id per ray and,
// when non-null, t and the normal (3 floats); cursor = the tree kernel's ray fetch counter (zeroed by the caller)
struct CastArgs {
    const float4* rays;
    int32_t* ids;
    float* t;
    float* normals;
    uint32_t n;
    uint32_t* cursor;
};
void launch_cast(const PassArgs& a, const CastArgs& c, bool any, int sm_count, cudaStream_t s);
void launch_resolve(const TileMap& map, const float* accum, int spp, float* rad_l, uint8_t* rgb_l, cudaStream_t s);
// Adaptive renders. Tile test: one warp per entry of list[0 .. n_active): the tile's error E over its in-frame pixels at
// n samples; tile_n[tile] = n, flag[entry] = E > tau and n < spp.
void launch_tile_test(const TileMap& map, const float* accum, const uint32_t* list, uint32_t n_active, int n, int spp, float tau,
                      int32_t* tile_n, uint32_t* flag, cudaStream_t s);
// One CTA: the entries of list[0 .. n_active) whose flag is set, in order, to list_out; their number to *count_out.
void launch_tile_compact(const uint32_t* list, uint32_t n_active, const uint32_t* flag, uint32_t* list_out, uint32_t* count_out,
                         cudaStream_t s);
// Per owned in-frame pixel at its tile's count: rgb / radiance (as resolve), variance of the mean, count (all nullable,
// full-frame row-major).
void launch_resolve_adaptive(const TileMap& map, const float* accum, const int32_t* tile_n, uint8_t* rgb, float* rad, float* var,
                             int32_t* spp, cudaStream_t s);
const char* path_launch_error(); // first failed launch/attribute call since the last clear, or nullptr
void path_clear_launch_error();

} // namespace g19

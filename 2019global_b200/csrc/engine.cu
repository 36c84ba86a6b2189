// engine.cu -- g19_ctx: device state, scene flattening/upload, render drivers.
//
// Implements the engine half of include/g19.h. The reference's RayTracer
// (include/raytracer.h:15-101) owns a Camera, a light and a non-owning Octree*
// and renders with run(w,h); here the ctx owns the flattened scene in HBM and
// g19_render* is run(). There is no CPU path: every entry point that computes
// launches CUDA kernels, and g19_create fails when no device is usable.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <cuda_runtime.h>

#include "g19.h"
#include "kernels.h"
#include "path.h"
#include "scene.h"

using namespace g19;

namespace {

thread_local std::string g_create_error; // g19_last_error(NULL) reports the calling thread's last g19_create failure

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    cudaError_t ensure(size_t need) {
        if (need <= bytes) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
        cudaError_t e = cudaMalloc(&p, need);
        if (e == cudaSuccess) bytes = need;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

} // namespace

struct ProgressHook { // g19_render_progressive -> render_any
    g19_pass_fn fn = nullptr;
    void* user = nullptr;
    uint8_t* h_rgb = nullptr;
    int min_interval_ms = 0;
};

struct g19_ctx {
    ProgressHook hook;
    int device = 0;
    cudaStream_t stream = nullptr; // used by the host-pointer entry points
    std::string err;
    std::atomic<int> cancel{0};
    std::atomic<int> progress_milli{0};
    int sm_count = 148;
    bool has_scene = false;
    bool host_call = false; // inside g19_render / g19_render_progressive: the caller blocks, so REF mode may render in bands

    // REF view
    DevBuf ref_nodes, ref_ents, ref_entities, ref_tris;
    RefSceneD ref{};
    int ref_depth = 0;
    // PATH view
    PathSceneBuffers path;
    PathTuning tune; // environment read once in g19_create; g19_tune afterwards

    // per-render work buffers (local-pixel indexed)
    DevBuf ids_l, points_l, normals_l, rgb_l, colour_l, counters;
    DevBuf heavy; // REF mode: heavy-ray lists, one set per band in flight (RefHeavyD)
    // frame buffers for the host-pointer entry point
    DevBuf rgb_f, ids_f, rad_f, var_f, spp_f; // (variance and sample counts: g19_render_adaptive)
    PathWork work;
    // ray queries (g19_cast_rays*): their own state, no render buffer
    PathCastWork cast;
    DevBuf cast_io; // g19_cast_rays: the rays and the outputs staged on the device

    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    cudaEvent_t cls0 = nullptr, cls1 = nullptr;
    cudaStream_t side = nullptr;                   // REF mode: the second band in flight
    cudaEvent_t ev_band[2] = {nullptr, nullptr}, ev_ready = nullptr;
    g19_stats stats{};
    bool stats_pending = false;
};

// A frame that several ranks write (include/g19.h "shared frame"): owner = the process that
// allocated it (rank 0), importers map it through CUDA IPC and reach it over NVLink.
struct g19_frame {
    int device = 0;
    bool owner = false;
    int32_t w = 0, h = 0;
    void* base = nullptr; // [flags 512 B][radiance w*h*3 floats, 256-aligned][rgb888 w*h*3]
    size_t bytes = 0;
    unsigned* flags = nullptr;
    float* rad = nullptr;
    uint8_t* rgb = nullptr;
    unsigned epoch = 0; // frames rendered into it by THIS process (all ranks advance in lockstep)
    cudaIpcMemHandle_t handle{};
    // sticky "a device-side wait gave up" word: pinned host memory of THIS process, mapped into the device
    unsigned* h_status = nullptr;
    unsigned* d_status = nullptr;
};

namespace {

struct FrameBlob { // what g19_frame_export ships to the other ranks
    uint32_t magic;
    int32_t w, h;
    uint64_t bytes;
    cudaIpcMemHandle_t handle;
};
constexpr uint32_t kFrameMagic = 0x46393147u; // "G19F"

void frame_layout(g19_frame* f) {
    size_t npx = size_t(f->w) * size_t(f->h);
    size_t rad_off = 512, rgb_off = (rad_off + npx * 12 + 255) & ~size_t(255);
    f->bytes = rgb_off + ((npx * 3 + 255) & ~size_t(255));
    if (f->base) {
        f->flags = static_cast<unsigned*>(f->base);
        f->rad = reinterpret_cast<float*>(static_cast<char*>(f->base) + rad_off);
        f->rgb = reinterpret_cast<uint8_t*>(static_cast<char*>(f->base) + rgb_off);
    }
}

int frame_status_alloc(g19_frame* f) {
    if (cudaHostAlloc(reinterpret_cast<void**>(&f->h_status), 64, cudaHostAllocMapped) != cudaSuccess) return G19_ERR_CUDA;
    *f->h_status = 0;
    if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&f->d_status), f->h_status, 0) != cudaSuccess) return G19_ERR_CUDA;
    return G19_OK;
}
// A frame on which a device-side wait timed out is dead: its pixels may be incomplete and a late signal of the
// lost rank would count towards a later frame, so every further call refuses it.
bool frame_dead(g19_ctx* ctx, const g19_frame* f) {
    if (!f->h_status || *reinterpret_cast<volatile unsigned*>(f->h_status) == 0) return false;
    ctx->err = "shared frame: a device-side wait gave up after 5 s (a rank was lost or fell behind); the frame may be "
               "incomplete -- destroy it and create a new one";
    return true;
}

#define G19_CUDA(ctx, call)                                                                              \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e__);                            \
            return G19_ERR_CUDA;                                                                         \
        }                                                                                                \
    } while (0)

template <typename T> cudaError_t upload(DevBuf& b, const std::vector<T>& v, cudaStream_t s) {
    size_t bytes = v.size() * sizeof(T);
    cudaError_t e = b.ensure(bytes ? bytes : sizeof(T));
    if (e != cudaSuccess || !bytes) return e;
    return cudaMemcpyAsync(b.p, v.data(), bytes, cudaMemcpyHostToDevice, s);
}

void copy3(double* dst, V3 v) {
    dst[0] = v.x;
    dst[1] = v.y;
    dst[2] = v.z;
}

// ---- flatten the reference octree (SURVEY.md section 7 step 5) ---------------
// fn(begin, end) over [0, n) on the host's cores: scene flattening of a 1 M-entity mesh is a few hundred MB of
// independent per-entity writes (single-threaded it was 0.3 s of the 0.8 s upload)
template <typename F> void host_parallel_for(size_t n, F fn) {
    unsigned hw = std::thread::hardware_concurrency();
    const size_t threads = n < (size_t(1) << 15) ? 1 : std::min<size_t>(hw ? hw : 4, 16);
    if (threads <= 1) { fn(size_t(0), n); return; }
    std::vector<std::thread> pool;
    const size_t chunk = (n + threads - 1) / threads;
    for (size_t t = 0; t < threads; ++t) {
        const size_t b = t * chunk, e = std::min(n, b + chunk);
        if (b < e) pool.emplace_back([=] { fn(b, e); });
    }
    for (std::thread& th : pool) th.join();
}

int flatten_ref(g19_ctx* ctx, const g19_scene& s) {
    std::vector<RefNodeD> nodes(s.nodes.size());
    // offsets first (a running sum), then every record is filled independently
    std::vector<int32_t> list_offset(s.nodes.size());
    size_t n_list = 0;
    for (size_t i = 0; i < s.nodes.size(); ++i) {
        list_offset[i] = int32_t(n_list);
        if (s.nodes[i].first_child < 0) n_list += s.nodes[i].ents.size(); // only leaf lists are ever returned (octree.h:133-135)
    }
    std::vector<int32_t> lists(n_list);
    host_parallel_for(s.nodes.size(), [&](size_t b, size_t e) {
        for (size_t i = b; i < e; ++i) {
            const HostNode& h = s.nodes[i];
            RefNodeD& d = nodes[i];
            copy3(d.mn, h.mn);
            copy3(d.mx, h.mx);
            d.first_child = h.first_child;
            d.ent_count = int32_t(h.ents.size());
            d.ent_offset = 0;
            d.pad = 0;
            if (h.first_child < 0) {
                d.ent_offset = list_offset[i];
                std::copy(h.ents.begin(), h.ents.end(), lists.begin() + list_offset[i]);
            }
        }
    });
    std::vector<RefEntityD> ents(s.ents.size());
    std::vector<int32_t> tri_offset(s.ents.size());
    size_t ntri = 0;
    for (size_t i = 0; i < s.ents.size(); ++i) {
        tri_offset[i] = int32_t(ntri);
        ntri += s.ents[i].tris.size();
    }
    std::vector<RefTriD> tris(ntri);
    host_parallel_for(s.ents.size(), [&](size_t b, size_t e) {
        for (size_t i = b; i < e; ++i) {
            const HostEntity& h = s.ents[i];
            RefEntityD& d = ents[i];
            std::memset(&d, 0, sizeof d);
            d.kind = h.kind;
            d.combine = h.combine;
            d.tri_offset = tri_offset[i];
            d.tri_count = int32_t(h.tris.size());
            d.first_tested = h.first_tested;
            d.radius = h.radius;
            std::memcpy(d.f, h.desc.f, sizeof d.f);
            copy3(d.pos, h.pos);
            d.color[0] = h.desc.color[0];
            d.color[1] = h.desc.color[1];
            d.color[2] = h.desc.color[2];
            copy3(d.aux0, h.aux0);
            copy3(d.aux1, h.aux1);
            // Material(color) defaults (material.h:13-16,27,29) unless the caller assigned the fields
            const g19_entity_desc& ed = h.desc;
            for (int k = 0; k < 3; ++k) {
                d.diffuse_color[k] = ed.material_set ? ed.diffuse_color[k] : ed.color[k] * 0.5;
                d.specular_color[k] = ed.material_set ? ed.specular_color[k] : 1.0;
            }
            d.shader[0] = ed.material_set ? ed.shader_parameters[0] : 0.1;
            d.shader[1] = ed.material_set ? ed.shader_parameters[1] : 0.7;
            d.shader[2] = ed.material_set ? ed.shader_parameters[2] : 1.0;
            d.specular_power = ed.material_set ? ed.specular_power : 5.0;
            RefTriD* out = tris.data() + tri_offset[i];
            for (const HostTri& t : h.tris) {
                RefTriD& r = *out++;
                std::memset(&r, 0, sizeof r);
                copy3(r.p1, t.p1);
                copy3(r.p2, t.p2);
                copy3(r.p3, t.p3);
                copy3(r.pos, t.pos);
                copy3(r.normal, t.normal);
                r.e1[0] = float(t.edge1.x); r.e1[1] = float(t.edge1.y); r.e1[2] = float(t.edge1.z);
                r.e2[0] = float(t.edge2.x); r.e2[1] = float(t.edge2.y); r.e2[2] = float(t.edge2.z);
            }
        }
    });
    const auto t_host = std::chrono::steady_clock::now();
    ctx->ref_depth = max_depth(s);
    if (ctx->ref_depth >= 39) {
        ctx->err = "reference octree deeper than the device traversal stack (39 levels)";
        return G19_ERR_LIMIT;
    }
    G19_CUDA(ctx, upload(ctx->ref_nodes, nodes, ctx->stream));
    G19_CUDA(ctx, upload(ctx->ref_ents, lists, ctx->stream));
    G19_CUDA(ctx, upload(ctx->ref_entities, ents, ctx->stream));
    G19_CUDA(ctx, upload(ctx->ref_tris, tris, ctx->stream));
    G19_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); // host vectors die at scope exit
    if (ctx->tune.debug_tree)
        std::fprintf(stderr, "[g19] REF view: %zu nodes, %zu entities, %zu triangles; copies %.1f ms (%.0f MB)\n", nodes.size(), ents.size(),
                     tris.size(), std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host).count(),
                     double(nodes.size() * sizeof(RefNodeD) + lists.size() * 4 + ents.size() * sizeof(RefEntityD) + tris.size() * sizeof(RefTriD)) / 1e6);
    ctx->ref.nodes = ctx->ref_nodes.as<RefNodeD>();
    ctx->ref.ents = ctx->ref_ents.as<int32_t>();
    ctx->ref.entities = ctx->ref_entities.as<RefEntityD>();
    ctx->ref.tris = ctx->ref_tris.as<RefTriD>();
    ctx->ref.n_nodes = int32_t(nodes.size());
    ctx->ref.n_entities = int32_t(ents.size());
    return G19_OK;
}

// Camera basis, raytracer.h:26-30 and camera.h:8-10, in the reference's order.
V3 add(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
V3 sub(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
V3 mul(V3 a, double s) { return {a.x * s, a.y * s, a.z * s}; }
double dotv(V3 a, V3 b) {
    double tx = a.x * b.x, ty = a.y * b.y, tz = a.z * b.z;
    return tx + ty + tz;
}
V3 crossv(V3 a, V3 b) { return {a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y}; }
V3 unitv(V3 v) { return mul(v, 1.0 / std::sqrt(dotv(v, v))); }

RefCamera make_camera(const g19_camera& c, const double light[3], int w) {
    V3 pos = {c.pos[0], c.pos[1], c.pos[2]};
    V3 look = {c.look_at[0], c.look_at[1], c.look_at[2]};
    V3 up = {0, 0, 1.0};
    V3 forward = unitv(sub(look, pos));
    V3 left = unitv(crossv(up, forward));
    V3 fwd = {c.focal * forward.x, c.focal * forward.y, c.focal * forward.z}; // scalar * vec
    V3 t = add(pos, fwd);
    t = add(t, mul(mul(mul(left, double(w)), 0.5), 0.0002));
    t = add(t, mul(mul(mul(up, double(w)), 0.5), 0.0002)); // the WIDTH, also vertically (raytracer.h:30)
    V3 top_left = sub(t, pos);
    RefCamera r;
    copy3(r.pos, pos);
    copy3(r.up, up);
    copy3(r.left, left);
    copy3(r.top_left, top_left);
    r.light[0] = light ? light[0] : 0;
    r.light[1] = light ? light[1] : 0;
    r.light[2] = light ? light[2] : 0;
    return r;
}

int check_params(g19_ctx* ctx, const g19_camera* cam, const g19_params* p) {
    if (!ctx) return G19_ERR_INVALID;
    if (!cam || !p || p->width < 0 || p->height < 0 || p->world < 1 || p->rank < 0 || p->rank >= p->world ||
        (p->mode != G19_MODE_REF && p->mode != G19_MODE_PATH)) {
        ctx->err = "invalid camera/params";
        return G19_ERR_INVALID;
    }
    // validated BEFORE anything is launched or signalled (a failed render must not leave a shared frame's
    // arrival counter ahead of its epoch)
    if (p->mode == G19_MODE_PATH && (p->spp < 1 || p->max_depth < 0 || p->max_depth > kMaxPathDepth)) {
        ctx->err = "PATH mode needs spp >= 1 and 0 <= max_depth <= 64";
        return G19_ERR_INVALID;
    }
    if ((long long)p->width * p->height > (1ll << 30)) {
        ctx->err = "image larger than 2^30 pixels";
        return G19_ERR_LIMIT;
    }
    if (!ctx->has_scene) {
        ctx->err = "g19_render before g19_upload_scene";
        return G19_ERR_NO_SCENE;
    }
    return G19_OK;
}

uint64_t owned_pixels(const TileMap& map) { // in-frame pixels owned by this rank
    uint64_t owned = 0;
    for (int lt = 0; lt < map.n_local_tiles; ++lt) {
        int tile = lt * map.world + map.rank;
        int ty = tile / map.tiles_x, tx = tile % map.tiles_x;
        owned += uint64_t(std::min(kTile, map.w - tx * kTile)) * uint64_t(std::min(kTile, map.h - ty * kTile));
    }
    return owned;
}

struct ClassTimer { // CUDA-event timing of one kernel class (params.profile)
    g19_ctx* ctx;
    cudaStream_t s;
    bool on;
    void begin() {
        if (on) cudaEventRecord(ctx->cls0, s);
    }
    void end(int cls, int launches) {
        ctx->stats.class_launches[cls] += launches;
        ctx->stats.kernel_launches += launches;
        if (!on) return;
        cudaEventRecord(ctx->cls1, s);
        cudaEventSynchronize(ctx->cls1);
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->cls0, ctx->cls1);
        ctx->stats.class_ms[cls] += ms;
        if (ctx->tune.debug_tree && cls == G19_K_REF_VIS) std::fprintf(stderr, "[g19] REF visibility launch: %.2f ms\n", ms);
    }
};

int render_ref(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p, const TileMap& map,
               uint8_t* d_rgb, int32_t* d_ids, float* d_rad, uint8_t* t_rgb, int32_t* t_ids, float* t_rad,
               cudaStream_t s, g19_frame* frame = nullptr) {
    RefCamera rc = make_camera(*cam, light, p->width);
    size_t n = size_t(map.n_local_pix);
    G19_CUDA(ctx, ctx->ids_l.ensure(n * sizeof(int32_t)));
    G19_CUDA(ctx, ctx->points_l.ensure(n * 3 * sizeof(double)));
    G19_CUDA(ctx, ctx->normals_l.ensure(n * 3 * sizeof(double)));
    G19_CUDA(ctx, ctx->rgb_l.ensure(n * 3));
    G19_CUDA(ctx, ctx->colour_l.ensure(n * 3 * sizeof(float)));
    G19_CUDA(ctx, ctx->counters.ensure(8 * sizeof(unsigned long long))); // [node tests, primitive tests, work counter, max per ray, work counter of the second band in flight, ...]
    unsigned long long* counters = nullptr;
    if (p->profile) {
        counters = ctx->counters.as<unsigned long long>();
        G19_CUDA(ctx, cudaMemsetAsync(counters, 0, 8 * sizeof(unsigned long long), s));
    }
    unsigned* next = reinterpret_cast<unsigned*>(ctx->counters.as<unsigned long long>() + 2);
    // heavy-ray lists (ref_heavy_kernel), one set per band in flight
    constexpr int kHeavyCap = 4096;
    RefHeavyD heavy[2] = {};
    if (ctx->tune.ref_heavy > 0 && ctx->ref.n_nodes > 1) {
        const size_t set = (ref_heavy_bytes(kHeavyCap) + 255) / 256 * 256;
        G19_CUDA(ctx, ctx->heavy.ensure(2 * set));
        for (int k = 0; k < 2; ++k) {
            char* base = static_cast<char*>(ctx->heavy.p) + k * set;
            heavy[k].count = reinterpret_cast<unsigned*>(base);
            heavy[k].lp = reinterpret_cast<int32_t*>(base + 64);
            heavy[k].best = reinterpret_cast<unsigned*>(base + 64 + size_t(kHeavyCap) * 4);
            heavy[k].lock = reinterpret_cast<int*>(base + 64 + size_t(kHeavyCap) * 8);
            heavy[k].masks = reinterpret_cast<unsigned short*>(base + 64 + size_t(kHeavyCap) * 12);
            heavy[k].cap = kHeavyCap;
            heavy[k].budget = ctx->tune.ref_heavy;
        }
    }
    ClassTimer t{ctx, s, p->profile != 0};
    // The reference fills its Image pixel by pixel and polls _running per pixel (raytracer.h:32-33), so stop() and
    // the viewer's 32 ms repaint see a frame in progress. On a heavy scene (the 1 M-entity heightfield takes seconds)
    // the host-pointer entry points therefore render BAND by band of whole tile rows: between bands the host
    // checks the cancel flag, publishes progress and -- for g19_render_progressive -- refreshes the caller's image.
    // Light scenes and the device-pointer entry points (asynchronous by contract) stay one launch.
    const bool banded = ctx->host_call && !frame && map.n_local_tiles >= 64 && (ctx->ref.n_nodes > 512 || ctx->ref.n_entities > 4096);
    int rc_band = G19_OK;
    if (!banded) {
        t.begin();
        launch_ref_visibility(ctx->ref, rc, map, ctx->ids_l.as<int32_t>(), ctx->points_l.as<double>(),
                              ctx->normals_l.as<double>(), counters, s, 0, -1, next, &heavy[0]);
        t.end(G19_K_REF_VIS, heavy[0].budget > 0 ? 2 : 1);
        t.begin();
        launch_ref_shade(ctx->ref, rc, map, ctx->ids_l.as<int32_t>(), ctx->points_l.as<double>(),
                         ctx->normals_l.as<double>(), ctx->rgb_l.as<uint8_t>(), ctx->colour_l.as<float>(), s);
        t.end(G19_K_REF_SHADE, 1);
    } else {
        // pixels a cancelled render never reaches stay "no hit, black" (Image(w,h) starts black, image.h:9)
        G19_CUDA(ctx, cudaMemsetAsync(ctx->ids_l.p, 0xff, n * sizeof(int32_t), s));
        G19_CUDA(ctx, cudaMemsetAsync(ctx->rgb_l.p, 0, n * 3, s));
        G19_CUDA(ctx, cudaMemsetAsync(ctx->colour_l.p, 0, n * 3 * sizeof(float), s));
        // About an eighth of the frame per band. Every band ends in a tail that waits for its most expensive ray (on the
        // 1 M-entity heightfield ONE ray tests 318 932 child boxes while the average ray tests 10), so two bands are kept
        // in flight on two streams: the tail of one hides under the bulk of the next, and the host -- which handles
        // cancel / progress / refresh for a band once its event has fired -- is at most two bands ahead of the device.
        const int tiles_per_band = std::max(map.tiles_x / std::max(1, map.world), (map.n_local_tiles + 7) / 8);
        // (one band at a time under params.profile -- its per-class event brackets need one launch at a time -- and while a
        // refresh hook is installed: a progressive caller is shown whole bands in order, never half of the next one)
        const bool overlap = !p->profile && !ctx->hook.fn;
        if (overlap) {
            if (!ctx->side) G19_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->side, cudaStreamNonBlocking));
            for (cudaEvent_t* e : {&ctx->ev_band[0], &ctx->ev_band[1], &ctx->ev_ready})
                if (!*e) G19_CUDA(ctx, cudaEventCreateWithFlags(e, cudaEventDisableTiming));
            G19_CUDA(ctx, cudaEventRecord(ctx->ev_ready, s)); // the clears above
            G19_CUDA(ctx, cudaStreamWaitEvent(ctx->side, ctx->ev_ready, 0));
        }
        auto last_refresh = std::chrono::steady_clock::now();
        // what the host does once band `done_lp1` is complete: progress, refresh, cancel from the hook
        auto after_band = [&](int done_lp1) -> int {
            ctx->progress_milli.store(int(1000.0 * double(done_lp1) / double(map.n_local_pix)));
            const auto now = std::chrono::steady_clock::now();
            if (ctx->hook.fn && d_rgb && ctx->hook.h_rgb && done_lp1 < map.n_local_pix &&
                std::chrono::duration<double, std::milli>(now - last_refresh).count() >= double(ctx->hook.min_interval_ms)) {
                last_refresh = now;
                launch_untile(map, ctx->rgb_l.as<uint8_t>(), nullptr, nullptr, d_rgb, nullptr, nullptr, s);
                G19_CUDA(ctx, cudaMemcpyAsync(ctx->hook.h_rgb, d_rgb, size_t(map.w) * size_t(map.h) * 3, cudaMemcpyDeviceToHost, s));
                G19_CUDA(ctx, cudaStreamSynchronize(s));
                ctx->stats.kernel_launches += 1;
                if (ctx->hook.fn(ctx->hook.user, double(done_lp1) / double(map.n_local_pix), ctx->hook.h_rgb) != 0) ctx->cancel.store(1);
            }
            return G19_OK;
        };
        int band = 0, pending_lp1[2] = {0, 0};
        bool pending[2] = {false, false};
        for (int t0 = 0; t0 < map.n_local_tiles; t0 += tiles_per_band, ++band) {
            if (ctx->cancel.load()) { // RayTracer::stop()
                rc_band = G19_ERR_CANCELLED;
                break;
            }
            const int lp0 = t0 * kTilePix, lp1 = std::min(map.n_local_tiles, t0 + tiles_per_band) * kTilePix;
            const int slot = overlap ? (band & 1) : 0;
            cudaStream_t bs = slot ? ctx->side : s;
            if (overlap && pending[slot]) { // this stream's previous band (two bands ago) must be done before its slot is reused
                G19_CUDA(ctx, cudaEventSynchronize(ctx->ev_band[slot]));
                pending[slot] = false;
                int rc2 = after_band(pending_lp1[slot]);
                if (rc2 != G19_OK) return rc2;
                if (ctx->cancel.load()) { rc_band = G19_ERR_CANCELLED; break; }
            }
            t.s = bs;
            t.begin();
            launch_ref_visibility(ctx->ref, rc, map, ctx->ids_l.as<int32_t>(), ctx->points_l.as<double>(),
                                  ctx->normals_l.as<double>(), counters, bs, lp0, lp1, next + 4 * slot, &heavy[slot]);
            t.end(G19_K_REF_VIS, heavy[slot].budget > 0 ? 2 : 1);
            t.begin();
            launch_ref_shade(ctx->ref, rc, map, ctx->ids_l.as<int32_t>(), ctx->points_l.as<double>(),
                             ctx->normals_l.as<double>(), ctx->rgb_l.as<uint8_t>(), ctx->colour_l.as<float>(), bs, lp0, lp1);
            t.end(G19_K_REF_SHADE, 1);
            if (overlap) {
                G19_CUDA(ctx, cudaEventRecord(ctx->ev_band[slot], bs));
                pending[slot] = true;
                pending_lp1[slot] = lp1;
            } else {
                G19_CUDA(ctx, cudaStreamSynchronize(s)); // the host stays one band ahead at most: that is the cancel latency
                int rc2 = after_band(lp1);
                if (rc2 != G19_OK) return rc2;
            }
        }
        t.s = s;
        if (overlap) { // drain in band order, then let the caller's stream continue behind both
            for (int k = 0; k < 2; ++k) {
                const int slot = (band + k) & 1;
                if (!pending[slot]) continue;
                G19_CUDA(ctx, cudaEventSynchronize(ctx->ev_band[slot]));
                pending[slot] = false;
                after_band(pending_lp1[slot]);
            }
            G19_CUDA(ctx, cudaEventRecord(ctx->ev_ready, ctx->side));
            G19_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev_ready, 0));
        }
    }
    t.begin();
    if (frame) { // shared frame: wait for the owner, scatter this rank's pixels into it, signal
        launch_frame_acquire(frame->flags, frame->epoch - 1, frame->d_status, s);
        launch_untile(map, ctx->rgb_l.as<uint8_t>(), nullptr, ctx->colour_l.as<float>(), frame->rgb, nullptr, frame->rad, s);
        launch_frame_signal(frame->flags, s);
        t.end(G19_K_OTHER, 3);
    } else {
        launch_untile(map, d_rgb ? ctx->rgb_l.as<uint8_t>() : nullptr, d_ids ? ctx->ids_l.as<int32_t>() : nullptr,
                      d_rad ? ctx->colour_l.as<float>() : nullptr, d_rgb, d_ids, d_rad, s);
        t.end(G19_K_OTHER, 1);
    }
    G19_CUDA(ctx, cudaGetLastError());
    if (t_rgb) G19_CUDA(ctx, cudaMemcpyAsync(t_rgb, ctx->rgb_l.p, n * 3, cudaMemcpyDeviceToDevice, s));
    if (t_ids) G19_CUDA(ctx, cudaMemcpyAsync(t_ids, ctx->ids_l.p, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    if (t_rad) G19_CUDA(ctx, cudaMemcpyAsync(t_rad, ctx->colour_l.p, n * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    ctx->stats.samples = 0;
    if (p->profile) {
        unsigned long long h[8] = {};
        G19_CUDA(ctx, cudaMemcpyAsync(h, counters, sizeof h, cudaMemcpyDeviceToHost, s));
        G19_CUDA(ctx, cudaStreamSynchronize(s));
        ctx->stats.node_tests = h[0];
        ctx->stats.prim_tests = h[1];
        if (ctx->tune.debug_tree)
            std::fprintf(stderr, "[g19] REF: the most expensive single-warp walk tested %llu child boxes; %llu heavy rays were spread over many warps\n", h[3], h[5]);
    }
    // in-frame pixels owned by this rank
    uint64_t owned = 0;
    for (int lt = 0; lt < map.n_local_tiles; ++lt) {
        int tile = lt * map.world + map.rank;
        int ty = tile / map.tiles_x, tx = tile % map.tiles_x;
        int wx = std::min(kTile, map.w - tx * kTile), wy = std::min(kTile, map.h - ty * kTile);
        owned += uint64_t(wx) * uint64_t(wy);
    }
    ctx->stats.samples = owned;
    ctx->stats.extend_segments = owned;
    return rc_band;
}

} // namespace

extern "C" {

int g19_create(const int* devices, int n_devices, g19_ctx** out) {
    if (!out) return G19_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_create_error = std::string("no usable CUDA device (") + cudaGetErrorString(e) +
                         "); lib2019global_b200 has no CPU path";
        return G19_ERR_NO_DEVICE;
    }
    int dev = 0;
    if (devices && n_devices > 0) dev = devices[0];
    else cudaGetDevice(&dev);
    if (dev < 0 || dev >= count) {
        g_create_error = "device index out of range";
        return G19_ERR_INVALID;
    }
    if (n_devices > 1) {
        g_create_error = "one g19_ctx drives one device; run one process (rank) per GPU and shard tiles with "
                         "g19_params.rank/world";
        return G19_ERR_INVALID;
    }
    e = cudaSetDevice(dev);
    if (e != cudaSuccess) {
        g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
        return G19_ERR_NO_DEVICE;
    }
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) {
        g_create_error = std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e);
        return G19_ERR_NO_DEVICE;
    }
    if (prop.major != 10) {
        g_create_error = "lib2019global_b200 is built for sm_100a only; device is sm_" + std::to_string(prop.major) +
                         std::to_string(prop.minor);
        return G19_ERR_NO_DEVICE;
    }
    g19_ctx* ctx = new (std::nothrow) g19_ctx();
    if (!ctx) return G19_ERR_INVALID;
    ctx->device = dev;
    ctx->sm_count = prop.multiProcessorCount;
    path_tuning_from_env(ctx->tune);
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
        cudaEventCreate(&ctx->cls0) != cudaSuccess || cudaEventCreate(&ctx->cls1) != cudaSuccess) {
        g_create_error = "stream/event creation failed";
        delete ctx;
        return G19_ERR_CUDA;
    }
    *out = ctx;
    return G19_OK;
}

void g19_destroy(g19_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (DevBuf* b : {&ctx->heavy, &ctx->ref_nodes, &ctx->ref_ents, &ctx->ref_entities, &ctx->ref_tris, &ctx->ids_l, &ctx->points_l,
                      &ctx->normals_l, &ctx->rgb_l, &ctx->colour_l, &ctx->counters, &ctx->rgb_f, &ctx->ids_f,
                      &ctx->rad_f, &ctx->var_f, &ctx->spp_f, &ctx->cast_io})
        b->release();
    path_release(ctx->path, ctx->work);
    ctx->cast.counters.release();
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->cls0) cudaEventDestroy(ctx->cls0);
    if (ctx->cls1) cudaEventDestroy(ctx->cls1);
    for (cudaEvent_t e : {ctx->ev_band[0], ctx->ev_band[1], ctx->ev_ready})
        if (e) cudaEventDestroy(e);
    if (ctx->side) cudaStreamDestroy(ctx->side);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* g19_last_error(const g19_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int g19_upload_scene(g19_ctx* ctx, const g19_scene* scene) {
    if (!ctx || !scene) return G19_ERR_INVALID;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    ctx->has_scene = false;
    // The two views are independent (REF: the reference's octree and FP64 records; PATH: primitives, octree, BVH): a large
    // scene flattens the REF view on a second host thread while this one builds the PATH view (1 M triangles: 0.22 s and
    // 0.32 s, 0.54 s one after the other).
    const auto t0 = std::chrono::steady_clock::now();
    const bool two_threads = scene->ents.size() >= (size_t(1) << 15);
    int rc_ref = G19_OK;
    double ms_ref = 0;
    std::thread ref_thread;
    auto do_ref = [&] {
        cudaSetDevice(ctx->device);
        rc_ref = flatten_ref(ctx, *scene);
        ms_ref = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    if (two_threads) ref_thread = std::thread(do_ref);
    else do_ref();
    if (!two_threads && rc_ref != G19_OK) return rc_ref;
    const auto t1 = std::chrono::steady_clock::now();
    std::string perr;
    int rc = path_upload(ctx->path, *scene, ctx->tune, ctx->stream, perr);
    const double ms_path = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count();
    if (two_threads) ref_thread.join();
    if (ctx->tune.debug_tree)
        std::fprintf(stderr, "[g19] upload: REF view %.1f ms, PATH view %.1f ms%s, together %.1f ms\n", ms_ref, ms_path,
                     two_threads ? " (side by side)" : "", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    if (rc_ref != G19_OK) return rc_ref;
    if (rc != G19_OK) {
        ctx->err = perr;
        return rc;
    }
    ctx->has_scene = true;
    return G19_OK;
}

// What path_render / path_render_adaptive get from the context and the call.
static PathRenderArgs path_args(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p, const TileMap& map,
                                cudaStream_t s) {
    PathRenderArgs a;
    a.tune = ctx->tune;
    a.cam = make_camera(*cam, light, p->width);
    a.params = *p;
    a.map = map;
    a.d_rgb = nullptr;
    a.d_rad = nullptr;
    a.d_ids = nullptr;
    a.t_rgb = nullptr;
    a.t_rad = nullptr;
    a.stream = s;
    a.sm_count = ctx->sm_count;
    a.cancel = &ctx->cancel;
    a.progress_milli = &ctx->progress_milli;
    a.cls0 = ctx->cls0;
    a.cls1 = ctx->cls1;
    return a;
}

static int render_any(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p,
                      uint8_t* d_rgb, int32_t* d_ids, float* d_rad, uint8_t* t_rgb, int32_t* t_ids, float* t_rad,
                      void* stream, g19_frame* frame = nullptr) {
    int rc = check_params(ctx, cam, p);
    if (rc != G19_OK) return rc;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    ctx->cancel.store(0);
    ctx->progress_milli.store(0);
    ctx->stats = g19_stats{};
    ctx->cast.counts_pending = false; // (the statistics now belong to this render)
    TileMap map = make_tile_map(p->width, p->height, p->rank, p->world);
    G19_CUDA(ctx, cudaEventRecord(ctx->ev0, s));
    if (p->mode == G19_MODE_REF) {
        if (frame && map.n_local_pix == 0) launch_frame_signal(frame->flags, s); // no tiles: still counted
        else rc = render_ref(ctx, cam, light, p, map, d_rgb, d_ids, d_rad, t_rgb, t_ids, t_rad, s, frame);
    } else {
        PathRenderArgs a = path_args(ctx, cam, light, p, map, s);
        const RefCamera& rc64 = a.cam;
        a.d_rgb = d_rgb;
        a.d_rad = d_rad;
        a.d_ids = d_ids;
        a.t_rgb = t_rgb;
        a.t_rad = t_rad;
        if (ctx->hook.fn) {
            a.on_pass = ctx->hook.fn;
            a.pass_user = ctx->hook.user;
            a.h_rgb = ctx->hook.h_rgb;
            a.min_interval_ms = ctx->hook.min_interval_ms;
        }
        if (frame) {
            a.frame_rgb = frame->rgb;
            a.frame_rad = frame->rad;
            a.frame_flags = frame->flags;
            a.frame_status = frame->d_status;
            a.frame_need_consumed = frame->epoch - 1;
        }
        // primary-hit AOV (hit_id_out in PATH mode) and the depth-0 slice (max_depth = 0: the reference's own
        // direct shade of the PATH primary hit, material.h:48-62) share REF mode's work buffers
        const bool depth0 = p->max_depth == 0;
        const size_t n = size_t(map.n_local_pix);
        if ((d_ids || t_ids || depth0) && n > 0) {
            G19_CUDA(ctx, ctx->ids_l.ensure(n * sizeof(int32_t)));
            a.ids_l = ctx->ids_l.as<int32_t>();
            if (depth0) {
                G19_CUDA(ctx, ctx->points_l.ensure(n * 3 * sizeof(double)));
                G19_CUDA(ctx, ctx->normals_l.ensure(n * 3 * sizeof(double)));
                G19_CUDA(ctx, ctx->rgb_l.ensure(n * 3));
                G19_CUDA(ctx, ctx->colour_l.ensure(n * 3 * sizeof(float)));
                a.points_l = ctx->points_l.as<double>();
                a.normals_l = ctx->normals_l.as<double>();
                a.frame_flags = nullptr; // the shade below delivers into the frame, not path_render's resolve
            }
        }
        std::string perr;
        rc = path_render(ctx->path, ctx->work, a, ctx->stats, perr);
        if (rc != G19_OK) ctx->err = perr;
        if (rc == G19_OK && n > 0 && depth0) {
            launch_ref_shade(ctx->ref, rc64, map, ctx->ids_l.as<int32_t>(), ctx->points_l.as<double>(),
                             ctx->normals_l.as<double>(), ctx->rgb_l.as<uint8_t>(), ctx->colour_l.as<float>(), s);
            if (frame) {
                launch_frame_acquire(frame->flags, frame->epoch - 1, frame->d_status, s);
                launch_untile(map, ctx->rgb_l.as<uint8_t>(), nullptr, ctx->colour_l.as<float>(), frame->rgb, nullptr, frame->rad, s);
                launch_frame_signal(frame->flags, s);
                ctx->stats.kernel_launches += 2;
            } else {
                launch_untile(map, d_rgb ? ctx->rgb_l.as<uint8_t>() : nullptr, d_ids ? ctx->ids_l.as<int32_t>() : nullptr,
                              d_rad ? ctx->colour_l.as<float>() : nullptr, d_rgb, d_ids, d_rad, s);
            }
            ctx->stats.kernel_launches += 2;
            G19_CUDA(ctx, cudaGetLastError());
            if (t_rgb) G19_CUDA(ctx, cudaMemcpyAsync(t_rgb, ctx->rgb_l.p, n * 3, cudaMemcpyDeviceToDevice, s));
            if (t_rad) G19_CUDA(ctx, cudaMemcpyAsync(t_rad, ctx->colour_l.p, n * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
            if (t_ids) G19_CUDA(ctx, cudaMemcpyAsync(t_ids, ctx->ids_l.p, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
            ctx->stats.samples = ctx->stats.extend_segments = owned_pixels(map); // as REF mode: one depth-0 sample per owned pixel
        } else if ((rc == G19_OK || rc == G19_ERR_CANCELLED) && n > 0 && (d_ids || t_ids)) {
            if (d_ids) {
                launch_untile(map, nullptr, ctx->ids_l.as<int32_t>(), nullptr, nullptr, d_ids, nullptr, s);
                ctx->stats.kernel_launches += 1;
            }
            if (t_ids) G19_CUDA(ctx, cudaMemcpyAsync(t_ids, ctx->ids_l.p, n * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        }
        // a rank without tiles still counts as arrived -- signalled only once the render call has succeeded
        if ((rc == G19_OK || rc == G19_ERR_CANCELLED) && frame && map.n_local_pix == 0) launch_frame_signal(frame->flags, s);
    }
    if (rc != G19_OK && rc != G19_ERR_CANCELLED) return rc;
    G19_CUDA(ctx, cudaEventRecord(ctx->ev1, s));
    ctx->stats_pending = true;
    if (rc == G19_OK) ctx->progress_milli.store(1000);
    return rc;
}

int g19_render_device(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p,
                      uint8_t* d_rgb, int32_t* d_ids, float* d_rad, void* stream) {
    return render_any(ctx, cam, light, p, d_rgb, d_ids, d_rad, nullptr, nullptr, nullptr, stream);
}

int64_t g19_tile_pixels(int w, int h, int rank, int world) {
    if (w < 0 || h < 0 || world < 1 || rank < 0 || rank >= world) return -1;
    return make_tile_map(w, h, rank, world).n_local_pix;
}

int g19_render_tiles_device(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p,
                            uint8_t* t_rgb, int32_t* t_ids, float* t_rad, void* stream) {
    return render_any(ctx, cam, light, p, nullptr, nullptr, nullptr, t_rgb, t_ids, t_rad, stream);
}

int g19_untile_device(g19_ctx* ctx, int w, int h, int rank, int world, const uint8_t* t_rgb, const int32_t* t_ids,
                      const float* t_rad, uint8_t* d_rgb, int32_t* d_ids, float* d_rad, void* stream) {
    if (!ctx || w < 0 || h < 0 || world < 1 || rank < 0 || rank >= world) return G19_ERR_INVALID;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    launch_untile(make_tile_map(w, h, rank, world), t_rgb, t_ids, t_rad, d_rgb, d_ids, d_rad,
                  static_cast<cudaStream_t>(stream));
    G19_CUDA(ctx, cudaGetLastError());
    return G19_OK;
}

int g19_render(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p, uint8_t* rgb,
               int32_t* ids, float* rad) {
    int rc = check_params(ctx, cam, p);
    if (rc != G19_OK) return rc;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    size_t npx = size_t(p->width) * size_t(p->height);
    if (npx == 0) return G19_OK;
    cudaStream_t s = ctx->stream;
    if (rgb) G19_CUDA(ctx, ctx->rgb_f.ensure(npx * 3));
    if (ids) G19_CUDA(ctx, ctx->ids_f.ensure(npx * sizeof(int32_t)));
    if (rad) G19_CUDA(ctx, ctx->rad_f.ensure(npx * 3 * sizeof(float)));
    // pixels owned by other ranks stay as the caller left them: seed the device
    // copies from the caller's buffers when sharded, else clear (Image::clear, image.h:24)
    if (p->world > 1) {
        if (rgb) G19_CUDA(ctx, cudaMemcpyAsync(ctx->rgb_f.p, rgb, npx * 3, cudaMemcpyHostToDevice, s));
        if (ids) G19_CUDA(ctx, cudaMemcpyAsync(ctx->ids_f.p, ids, npx * 4, cudaMemcpyHostToDevice, s));
        if (rad) G19_CUDA(ctx, cudaMemcpyAsync(ctx->rad_f.p, rad, npx * 12, cudaMemcpyHostToDevice, s));
    }
    ctx->host_call = true;
    rc = g19_render_device(ctx, cam, light, p, rgb ? ctx->rgb_f.as<uint8_t>() : nullptr,
                           ids ? ctx->ids_f.as<int32_t>() : nullptr, rad ? ctx->rad_f.as<float>() : nullptr, s);
    ctx->host_call = false;
    if (rc != G19_OK && rc != G19_ERR_CANCELLED) return rc;
    if (rgb) G19_CUDA(ctx, cudaMemcpyAsync(rgb, ctx->rgb_f.p, npx * 3, cudaMemcpyDeviceToHost, s));
    if (ids) G19_CUDA(ctx, cudaMemcpyAsync(ids, ctx->ids_f.p, npx * 4, cudaMemcpyDeviceToHost, s));
    if (rad) G19_CUDA(ctx, cudaMemcpyAsync(rad, ctx->rad_f.p, npx * 12, cudaMemcpyDeviceToHost, s));
    G19_CUDA(ctx, cudaStreamSynchronize(s));
    return rc;
}

// ---- adaptive sampling (PATH mode) -------------------------------------------------------------
static int check_adaptive(g19_ctx* ctx, const g19_camera* cam, const g19_params* p, const g19_adaptive* ad) {
    if (!ctx) return G19_ERR_INVALID;
    const char* bad = nullptr;
    if (!p || !ad) bad = "params and adaptive are required";
    else if (p->mode != G19_MODE_PATH) bad = "only G19_MODE_PATH renders adaptively";
    else if (!(ad->noise_target > 0.0f) || !std::isfinite(ad->noise_target)) bad = "noise_target must be finite and > 0";
    else if (ad->min_spp < 2 || ad->min_spp > p->spp) bad = "min_spp must be in [2, spp]";
    else if (p->max_depth < 1) bad = "max_depth must be >= 1";
    if (bad) {
        ctx->err = std::string("g19_render_adaptive: ") + bad;
        return G19_ERR_INVALID;
    }
    return check_params(ctx, cam, p);
}

int g19_render_adaptive_device(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p,
                               const g19_adaptive* ad, uint8_t* d_rgb, float* d_rad, float* d_var, int32_t* d_spp, void* stream) {
    int rc = check_adaptive(ctx, cam, p, ad);
    if (rc != G19_OK) return rc;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    ctx->cancel.store(0);
    ctx->progress_milli.store(0);
    ctx->stats = g19_stats{};
    ctx->cast.counts_pending = false; // (the statistics now belong to this render)
    const TileMap map = make_tile_map(p->width, p->height, p->rank, p->world);
    G19_CUDA(ctx, cudaEventRecord(ctx->ev0, s));
    PathRenderArgs a = path_args(ctx, cam, light, p, map, s);
    a.d_rgb = d_rgb;
    a.d_rad = d_rad;
    std::string perr;
    rc = path_render_adaptive(ctx->path, ctx->work, a, ad->noise_target, ad->min_spp, d_var, d_spp, ctx->stats, perr);
    if (rc != G19_OK && rc != G19_ERR_CANCELLED) {
        ctx->err = perr;
        return rc;
    }
    G19_CUDA(ctx, cudaEventRecord(ctx->ev1, s));
    ctx->stats_pending = true;
    if (rc == G19_OK) ctx->progress_milli.store(1000);
    return rc;
}

int g19_render_adaptive(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p, const g19_adaptive* ad,
                        uint8_t* rgb, float* rad, float* var, int32_t* spp) {
    int rc = check_adaptive(ctx, cam, p, ad);
    if (rc != G19_OK) return rc;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t npx = size_t(p->width) * size_t(p->height);
    if (npx == 0) return G19_OK;
    cudaStream_t s = ctx->stream;
    if (rgb) G19_CUDA(ctx, ctx->rgb_f.ensure(npx * 3));
    if (rad) G19_CUDA(ctx, ctx->rad_f.ensure(npx * 3 * sizeof(float)));
    if (var) G19_CUDA(ctx, ctx->var_f.ensure(npx * sizeof(float)));
    if (spp) G19_CUDA(ctx, ctx->spp_f.ensure(npx * sizeof(int32_t)));
    // pixels owned by other ranks stay as the caller left them (as g19_render)
    if (p->world > 1) {
        if (rgb) G19_CUDA(ctx, cudaMemcpyAsync(ctx->rgb_f.p, rgb, npx * 3, cudaMemcpyHostToDevice, s));
        if (rad) G19_CUDA(ctx, cudaMemcpyAsync(ctx->rad_f.p, rad, npx * 12, cudaMemcpyHostToDevice, s));
        if (var) G19_CUDA(ctx, cudaMemcpyAsync(ctx->var_f.p, var, npx * 4, cudaMemcpyHostToDevice, s));
        if (spp) G19_CUDA(ctx, cudaMemcpyAsync(ctx->spp_f.p, spp, npx * 4, cudaMemcpyHostToDevice, s));
    }
    rc = g19_render_adaptive_device(ctx, cam, light, p, ad, rgb ? ctx->rgb_f.as<uint8_t>() : nullptr, rad ? ctx->rad_f.as<float>() : nullptr,
                                    var ? ctx->var_f.as<float>() : nullptr, spp ? ctx->spp_f.as<int32_t>() : nullptr, s);
    if (rc != G19_OK) {
        if (rc == G19_ERR_CANCELLED) G19_CUDA(ctx, cudaStreamSynchronize(s));
        return rc;
    }
    if (rgb) G19_CUDA(ctx, cudaMemcpyAsync(rgb, ctx->rgb_f.p, npx * 3, cudaMemcpyDeviceToHost, s));
    if (rad) G19_CUDA(ctx, cudaMemcpyAsync(rad, ctx->rad_f.p, npx * 12, cudaMemcpyDeviceToHost, s));
    if (var) G19_CUDA(ctx, cudaMemcpyAsync(var, ctx->var_f.p, npx * 4, cudaMemcpyDeviceToHost, s));
    if (spp) G19_CUDA(ctx, cudaMemcpyAsync(spp, ctx->spp_f.p, npx * 4, cudaMemcpyDeviceToHost, s));
    G19_CUDA(ctx, cudaStreamSynchronize(s));
    return G19_OK;
}

// ---- shared frame (multi-GPU, fused gather) ---------------------------------------------------
int g19_frame_create(g19_ctx* ctx, int w, int h, g19_frame** out) {
    if (!ctx || !out || w < 0 || h < 0) return G19_ERR_INVALID;
    *out = nullptr;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    g19_frame* f = new (std::nothrow) g19_frame();
    if (!f) return G19_ERR_INVALID;
    f->device = ctx->device;
    f->owner = true;
    f->w = w;
    f->h = h;
    frame_layout(f);
    cudaError_t e = cudaMalloc(&f->base, f->bytes);
    if (e == cudaSuccess) e = cudaMemset(f->base, 0, f->bytes);
    if (e != cudaSuccess) {
        ctx->err = std::string("g19_frame_create: ") + cudaGetErrorString(e);
        if (f->base) cudaFree(f->base);
        delete f;
        return G19_ERR_CUDA;
    }
    frame_layout(f);
    if (frame_status_alloc(f) != G19_OK) {
        ctx->err = "g19_frame_create: cudaHostAlloc of the status word failed";
        cudaFree(f->base);
        delete f;
        return G19_ERR_CUDA;
    }
    *out = f;
    return G19_OK;
}

int g19_frame_export(g19_ctx* ctx, g19_frame* f, void* blob, size_t blob_bytes) {
    if (!ctx || !f || !blob || !f->owner) return G19_ERR_INVALID;
    if (blob_bytes < sizeof(FrameBlob)) {
        ctx->err = "g19_frame_export: blob buffer smaller than G19_FRAME_BLOB_BYTES";
        return G19_ERR_INVALID;
    }
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    G19_CUDA(ctx, cudaIpcGetMemHandle(&f->handle, f->base));
    FrameBlob b;
    std::memset(&b, 0, sizeof b);
    b.magic = kFrameMagic;
    b.w = f->w;
    b.h = f->h;
    b.bytes = f->bytes;
    b.handle = f->handle;
    std::memset(blob, 0, blob_bytes);
    std::memcpy(blob, &b, sizeof b);
    return G19_OK;
}

int g19_frame_import(g19_ctx* ctx, const void* blob, size_t blob_bytes, g19_frame** out) {
    if (!ctx || !blob || !out || blob_bytes < sizeof(FrameBlob)) return G19_ERR_INVALID;
    *out = nullptr;
    FrameBlob b;
    std::memcpy(&b, blob, sizeof b);
    if (b.magic != kFrameMagic) {
        ctx->err = "g19_frame_import: not a frame blob";
        return G19_ERR_INVALID;
    }
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    g19_frame* f = new (std::nothrow) g19_frame();
    if (!f) return G19_ERR_INVALID;
    f->device = ctx->device;
    f->owner = false;
    f->w = b.w;
    f->h = b.h;
    cudaError_t e = cudaIpcOpenMemHandle(&f->base, b.handle, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        ctx->err = std::string("g19_frame_import: cudaIpcOpenMemHandle: ") + cudaGetErrorString(e) +
                   " (peer access over NVLink between the two devices is required)";
        delete f;
        return G19_ERR_CUDA;
    }
    frame_layout(f);
    if (f->bytes != b.bytes) {
        ctx->err = "g19_frame_import: layout mismatch";
        cudaIpcCloseMemHandle(f->base);
        delete f;
        return G19_ERR_INVALID;
    }
    if (frame_status_alloc(f) != G19_OK) {
        ctx->err = "g19_frame_import: cudaHostAlloc of the status word failed";
        cudaIpcCloseMemHandle(f->base);
        delete f;
        return G19_ERR_CUDA;
    }
    *out = f;
    return G19_OK;
}

void g19_frame_destroy(g19_frame* f) {
    if (!f) return;
    cudaSetDevice(f->device);
    cudaDeviceSynchronize();
    if (f->base) {
        if (f->owner) cudaFree(f->base);
        else cudaIpcCloseMemHandle(f->base);
    }
    if (f->h_status) cudaFreeHost(f->h_status);
    delete f;
}

int g19_frame_pointers(g19_frame* f, uint8_t** d_rgb, float** d_rad) {
    if (!f) return G19_ERR_INVALID;
    if (d_rgb) *d_rgb = f->rgb;
    if (d_rad) *d_rad = f->rad;
    return G19_OK;
}

int g19_render_to_frame(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p, g19_frame* f,
                        void* stream) {
    if (!ctx || !f || !p) return G19_ERR_INVALID;
    if (p->width != f->w || p->height != f->h) {
        ctx->err = "g19_render_to_frame: params do not match the frame size";
        return G19_ERR_INVALID;
    }
    if (frame_dead(ctx, f)) return G19_ERR_TIMEOUT;
    ++f->epoch;
    int rc = render_any(ctx, cam, light, p, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, stream, f);
    if (rc != G19_OK && rc != G19_ERR_CANCELLED) --f->epoch;
    return rc;
}

int g19_frame_wait(g19_ctx* ctx, g19_frame* f, int world, void* stream) {
    if (!ctx || !f || !f->owner || world < 1) return G19_ERR_INVALID;
    if (frame_dead(ctx, f)) return G19_ERR_TIMEOUT;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    launch_frame_wait(f->flags, f->epoch * unsigned(world), f->d_status, static_cast<cudaStream_t>(stream));
    G19_CUDA(ctx, cudaGetLastError());
    return G19_OK;
}

int g19_frame_release(g19_ctx* ctx, g19_frame* f, void* stream) {
    if (!ctx || !f || !f->owner) return G19_ERR_INVALID;
    if (frame_dead(ctx, f)) return G19_ERR_TIMEOUT;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    launch_frame_release(f->flags, f->epoch, static_cast<cudaStream_t>(stream));
    G19_CUDA(ctx, cudaGetLastError());
    return G19_OK;
}

int g19_frame_read(g19_ctx* ctx, g19_frame* f, uint8_t* rgb_out, float* rad_out, void* stream) {
    if (!ctx || !f || !f->owner) return G19_ERR_INVALID;
    if (frame_dead(ctx, f)) return G19_ERR_TIMEOUT;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    size_t npx = size_t(f->w) * size_t(f->h);
    if (rgb_out && npx) G19_CUDA(ctx, cudaMemcpyAsync(rgb_out, f->rgb, npx * 3, cudaMemcpyDefault, s));
    if (rad_out && npx) G19_CUDA(ctx, cudaMemcpyAsync(rad_out, f->rad, npx * 12, cudaMemcpyDefault, s));
    return G19_OK;
}

int g19_frame_timeouts(g19_ctx* ctx, g19_frame* f, unsigned* out) {
    if (!ctx || !f || !out) return G19_ERR_INVALID;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    G19_CUDA(ctx, cudaMemcpy(out, f->flags + 64, sizeof(unsigned), cudaMemcpyDeviceToHost));
    return G19_OK;
}

int g19_frame_status(g19_ctx* ctx, g19_frame* f, void* stream) {
    if (!ctx || !f) return G19_ERR_INVALID;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    G19_CUDA(ctx, cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    return frame_dead(ctx, f) ? G19_ERR_TIMEOUT : G19_OK;
}

int g19_tune(g19_ctx* ctx, const char* key, const char* value) {
    if (!ctx || !key) return G19_ERR_INVALID;
    if (!path_tuning_set(ctx->tune, key, value)) {
        ctx->err = std::string("g19_tune: unknown key '") + key + "'";
        return G19_ERR_INVALID;
    }
    return G19_OK;
}

int g19_render_progressive(g19_ctx* ctx, const g19_camera* cam, const double light[3], const g19_params* p,
                           uint8_t* rgb, float* rad, g19_pass_fn on_pass, void* user, int min_interval_ms) {
    if (!ctx || !rgb) return G19_ERR_INVALID;
    ctx->hook.fn = on_pass;
    ctx->hook.user = user;
    ctx->hook.h_rgb = rgb;
    ctx->hook.min_interval_ms = min_interval_ms < 0 ? 0 : min_interval_ms;
    int rc = g19_render(ctx, cam, light, p, rgb, nullptr, rad);
    ctx->hook = ProgressHook{};
    if ((rc == G19_OK || rc == G19_ERR_CANCELLED) && on_pass) {
        double done = 1.0;
        if (rc == G19_ERR_CANCELLED) g19_progress(ctx, &done);
        on_pass(user, rc == G19_OK ? 1.0 : done, rgb); // the final (or last complete) image
    }
    return rc;
}

int g19_get_stats(g19_ctx* ctx, g19_stats* out) {
    if (!ctx || !out) return G19_ERR_INVALID;
    if (ctx->stats_pending) {
        G19_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
        float ms = 0;
        G19_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        ctx->stats.render_ms = ms;
        std::string perr;
        int rc = path_finish_stats(ctx->work, ctx->stats, perr);
        if (rc == G19_OK) rc = path_cast_finish_stats(ctx->cast, ctx->stats, perr);
        if (rc != G19_OK) {
            ctx->err = perr;
            return rc;
        }
        ctx->stats_pending = false;
    }
    *out = ctx->stats;
    return G19_OK;
}

// ---- ray queries ------------------------------------------------------------------------------------
static int check_cast(g19_ctx* ctx, int32_t n, const float* rays, uint32_t flags, const int32_t* ids, const float* t,
                      const float* normals) {
    if (!ctx) return G19_ERR_INVALID;
    const char* bad = nullptr;
    if (n < 0) bad = "n < 0";
    else if (n > 0 && (!rays || !ids)) bad = "rays and out_entity are required";
    else if (reinterpret_cast<uintptr_t>(rays) % 16 != 0) bad = "rays must be 16-byte aligned";
    else if ((flags & ~(G19_CAST_ANY_HIT | G19_CAST_COUNT)) != 0u) bad = "unknown flag bits";
    else if ((flags & G19_CAST_ANY_HIT) && (t || normals)) bad = "an any-hit cast has no t or normal outputs";
    if (bad) {
        ctx->err = std::string("g19_cast_rays: ") + bad;
        return G19_ERR_INVALID;
    }
    if (!ctx->has_scene) return G19_ERR_NO_SCENE;
    return G19_OK;
}

int g19_cast_rays_device(g19_ctx* ctx, int32_t n, const float* d_rays, uint32_t flags, int32_t* d_entity, float* d_t,
                         float* d_normal, void* stream) {
    int rc = check_cast(ctx, n, d_rays, flags, d_entity, d_t, d_normal);
    if (rc != G19_OK || n == 0) return rc;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    ctx->stats = g19_stats{};
    ctx->stats_pending = false;
    ctx->work.totals_pending = false; // (the statistics now belong to this cast)
    G19_CUDA(ctx, cudaEventRecord(ctx->ev0, s));
    std::string perr;
    rc = path_cast(ctx->path, ctx->cast, ctx->tune, n, d_rays, flags, d_entity, d_t, d_normal, s, ctx->sm_count, ctx->stats, perr);
    if (rc != G19_OK) {
        ctx->err = perr;
        return rc;
    }
    G19_CUDA(ctx, cudaEventRecord(ctx->ev1, s));
    ctx->stats_pending = true;
    return G19_OK;
}

int g19_cast_rays(g19_ctx* ctx, int32_t n, const float* rays, uint32_t flags, int32_t* out_entity, float* out_t,
                  float* out_normal) {
    int rc = check_cast(ctx, n, rays, flags, out_entity, out_t, out_normal);
    if (rc != G19_OK || n == 0) return rc;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    // one buffer: rays (32 B per ray) | ids | t | normals
    const size_t un = size_t(n), b_rays = un * 32, b_ids = (un * 4 + 15) & ~size_t(15), b_t = (un * 4 + 15) & ~size_t(15);
    G19_CUDA(ctx, ctx->cast_io.ensure(b_rays + b_ids + b_t + un * 12));
    char* base = ctx->cast_io.as<char>();
    float* d_rays = reinterpret_cast<float*>(base);
    int32_t* d_ids = reinterpret_cast<int32_t*>(base + b_rays);
    float* d_t = out_t ? reinterpret_cast<float*>(base + b_rays + b_ids) : nullptr;
    float* d_nrm = out_normal ? reinterpret_cast<float*>(base + b_rays + b_ids + b_t) : nullptr;
    cudaStream_t s = ctx->stream;
    G19_CUDA(ctx, cudaMemcpyAsync(d_rays, rays, b_rays, cudaMemcpyHostToDevice, s));
    rc = g19_cast_rays_device(ctx, n, d_rays, flags, d_ids, d_t, d_nrm, s);
    if (rc != G19_OK) return rc;
    G19_CUDA(ctx, cudaMemcpyAsync(out_entity, d_ids, un * 4, cudaMemcpyDeviceToHost, s));
    if (out_t) G19_CUDA(ctx, cudaMemcpyAsync(out_t, d_t, un * 4, cudaMemcpyDeviceToHost, s));
    if (out_normal) G19_CUDA(ctx, cudaMemcpyAsync(out_normal, d_nrm, un * 12, cudaMemcpyDeviceToHost, s));
    G19_CUDA(ctx, cudaStreamSynchronize(s));
    return G19_OK;
}

int g19_cancel(g19_ctx* ctx) {
    if (!ctx) return G19_ERR_INVALID;
    ctx->cancel.store(1);
    return G19_OK;
}

int g19_progress(g19_ctx* ctx, double* out) {
    if (!ctx || !out) return G19_ERR_INVALID;
    *out = ctx->progress_milli.load() / 1000.0;
    return G19_OK;
}

int g19_probe_intersect(g19_ctx* ctx, int32_t entity, int n, const double* origins, const double* dirs, int32_t* hit,
                        double* points, double* normals) {
    if (!ctx || !origins || !dirs || !hit || !points || !normals || n < 0) return G19_ERR_INVALID;
    if (!ctx->has_scene) return G19_ERR_NO_SCENE;
    if (entity < 0 || entity >= ctx->ref.n_entities) return G19_ERR_INVALID;
    if (n == 0) return G19_OK;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf o, d, h, p, nn;
    size_t v = size_t(n) * 3 * sizeof(double);
    cudaStream_t s = ctx->stream;
    int rc = G19_OK;
    auto fail = [&](cudaError_t e, const char* what) {
        ctx->err = std::string(what) + ": " + cudaGetErrorString(e);
        rc = G19_ERR_CUDA;
    };
    cudaError_t e;
    if ((e = o.ensure(v)) != cudaSuccess || (e = d.ensure(v)) != cudaSuccess ||
        (e = h.ensure(size_t(n) * 4)) != cudaSuccess || (e = p.ensure(v)) != cudaSuccess ||
        (e = nn.ensure(v)) != cudaSuccess) {
        fail(e, "probe alloc");
    } else {
        cudaMemcpyAsync(o.p, origins, v, cudaMemcpyHostToDevice, s);
        cudaMemcpyAsync(d.p, dirs, v, cudaMemcpyHostToDevice, s);
        launch_probe_intersect(ctx->ref, entity, n, o.as<double>(), d.as<double>(), h.as<int32_t>(), p.as<double>(),
                               nn.as<double>(), s);
        cudaMemcpyAsync(hit, h.p, size_t(n) * 4, cudaMemcpyDeviceToHost, s);
        cudaMemcpyAsync(points, p.p, v, cudaMemcpyDeviceToHost, s);
        cudaMemcpyAsync(normals, nn.p, v, cudaMemcpyDeviceToHost, s);
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) fail(e, "probe_intersect");
    }
    for (DevBuf* b : {&o, &d, &h, &p, &nn}) b->release();
    return rc;
}

int g19_probe_texcoord(g19_ctx* ctx, int32_t entity, int n, const double* points, int32_t* out_uv) {
    if (!ctx || !points || !out_uv || n < 0) return G19_ERR_INVALID;
    if (!ctx->has_scene) return G19_ERR_NO_SCENE;
    if (entity < 0 || entity >= ctx->ref.n_entities) return G19_ERR_INVALID;
    if (n == 0) return G19_OK;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf p, uv;
    cudaStream_t s = ctx->stream;
    cudaError_t e;
    int rc = G19_OK;
    if ((e = p.ensure(size_t(n) * 24)) != cudaSuccess || (e = uv.ensure(size_t(n) * 8)) != cudaSuccess) {
        ctx->err = std::string("probe alloc: ") + cudaGetErrorString(e);
        rc = G19_ERR_CUDA;
    } else {
        cudaMemcpyAsync(p.p, points, size_t(n) * 24, cudaMemcpyHostToDevice, s);
        launch_probe_texcoord(ctx->ref, entity, n, p.as<double>(), uv.as<int32_t>(), s);
        cudaMemcpyAsync(out_uv, uv.p, size_t(n) * 8, cudaMemcpyDeviceToHost, s);
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) {
            ctx->err = std::string("probe_texcoord: ") + cudaGetErrorString(e);
            rc = G19_ERR_CUDA;
        }
    }
    p.release();
    uv.release();
    return rc;
}

int g19_probe_shade(g19_ctx* ctx, int32_t entity, int textured, const double ray_dir[3], const double light[3],
                    const double point[3], const double normal[3], int u, int v, double out_rgb[3]) {
    if (!ctx || !ray_dir || !light || !point || !normal || !out_rgb) return G19_ERR_INVALID;
    if (!ctx->has_scene) return G19_ERR_NO_SCENE;
    if (entity < 0 || entity >= ctx->ref.n_entities) return G19_ERR_INVALID;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf in, out;
    cudaStream_t s = ctx->stream;
    double h[15] = {ray_dir[0], ray_dir[1], ray_dir[2], light[0], light[1], light[2], point[0], point[1],
                    point[2],   normal[0],  normal[1],  normal[2], 0,       0,        0};
    cudaError_t e;
    int rc = G19_OK;
    if ((e = in.ensure(sizeof h)) != cudaSuccess || (e = out.ensure(24)) != cudaSuccess) {
        ctx->err = std::string("probe alloc: ") + cudaGetErrorString(e);
        rc = G19_ERR_CUDA;
    } else {
        cudaMemcpyAsync(in.p, h, sizeof h, cudaMemcpyHostToDevice, s);
        launch_probe_shade(ctx->ref, entity, textured, in.as<double>(), u, v, out.as<double>(), s);
        cudaMemcpyAsync(out_rgb, out.p, 24, cudaMemcpyDeviceToHost, s);
        if ((e = cudaStreamSynchronize(s)) != cudaSuccess) {
            ctx->err = std::string("probe_shade: ") + cudaGetErrorString(e);
            rc = G19_ERR_CUDA;
        }
    }
    in.release();
    out.release();
    return rc;
}

int g19_probe_path_tree(g19_ctx* ctx, uint32_t* nodes_out, uint32_t max_nodes, uint32_t* index_out, uint32_t max_index,
                        uint32_t* n_nodes, uint32_t* n_index) {
    if (!ctx || !n_nodes || !n_index) return G19_ERR_INVALID;
    if (!ctx->has_scene) return G19_ERR_NO_SCENE;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    const PathSceneD& v = ctx->path.view;
    *n_nodes = uint32_t(v.n_nodes);
    *n_index = uint32_t(v.n_index);
    if (nodes_out && max_nodes >= *n_nodes)
        G19_CUDA(ctx, cudaMemcpy(nodes_out, v.nodes, size_t(v.n_nodes) * sizeof(PathNodeD), cudaMemcpyDeviceToHost));
    if (index_out && max_index >= *n_index && v.n_index > 0)
        G19_CUDA(ctx, cudaMemcpy(index_out, v.index, size_t(v.n_index) * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return G19_OK;
}

int g19_probe_candidates(g19_ctx* ctx, const double origin[3], const double dir[3], int32_t* out_ids, int max_out,
                         int* out_n) {
    if (!ctx || !origin || !dir || !out_n || max_out < 0) return G19_ERR_INVALID;
    if (!ctx->has_scene) return G19_ERR_NO_SCENE;
    G19_CUDA(ctx, cudaSetDevice(ctx->device));
    DevBuf od, ids, cnt;
    cudaStream_t s = ctx->stream;
    double h[6] = {origin[0], origin[1], origin[2], dir[0], dir[1], dir[2]};
    int rc = G19_OK;
    cudaError_t e;
    if ((e = od.ensure(sizeof h)) != cudaSuccess || (e = ids.ensure(size_t(max_out ? max_out : 1) * 4)) != cudaSuccess ||
        (e = cnt.ensure(4)) != cudaSuccess) {
        ctx->err = std::string("probe alloc: ") + cudaGetErrorString(e);
        rc = G19_ERR_CUDA;
    } else {
        cudaMemcpyAsync(od.p, h, sizeof h, cudaMemcpyHostToDevice, s);
        launch_probe_candidates(ctx->ref, od.as<double>(), ids.as<int32_t>(), max_out, cnt.as<int32_t>(), s);
        int32_t n = 0;
        cudaMemcpyAsync(&n, cnt.p, 4, cudaMemcpyDeviceToHost, s);
        e = cudaStreamSynchronize(s);
        if (e == cudaSuccess && out_ids && max_out > 0) {
            int m = n < max_out ? n : max_out;
            e = cudaMemcpy(out_ids, ids.p, size_t(m) * 4, cudaMemcpyDeviceToHost);
        }
        if (e != cudaSuccess) {
            ctx->err = std::string("probe_candidates: ") + cudaGetErrorString(e);
            rc = G19_ERR_CUDA;
        }
        *out_n = n;
    }
    for (DevBuf* b : {&od, &ids, &cnt}) b->release();
    return rc;
}

} // extern "C"

// path_kernels.cu -- the wavefront path tracer on sm_100a (G19_MODE_PATH).
//
// One pass traces P = spp_pass * window camera paths, bounce by bounce; up to four passes are in
// flight on their own streams (path.cu). Two families of kernels share the shading code:
//
// FLAT scenes (the whole scene is one leaf of <= 192 primitives, staged in shared memory):
//   bounce_flat_fused    camera ray from the pixel index, nearest hit, and the first vertex shaded
//                        in place; camera hits on mirror / glass go to their material's queue
//   bounce_flat          one bounce of a diffuse-only scene (scenes with specular materials run
//                        the three queues of a bounce in ONE launch, bounce_flat_all): next-event
//                        estimation, BSDF sample, the shadow ray and the continuation ray traced in
//                        one loop over primitive PAIRS (packed FP32), the new vertex record written
//                        into the next bounce's queue. The queues hold the records themselves (four
//                        float4 planes), the path's radiance rides in the record and is stored once
//                        when the path ends. The bounce before the last shades the last vertex in
//                        place (FOLD): the last bounce has no launch.
// TREE scenes (linear octree in HBM / L2):
//   raygen_extend        camera ray + ordered octree walk (all 32 lanes of a warp in fixed-trip rounds)
//   bounce<KIND>         shades a queue of slot indices and queues the vertex's rays
//   trace                persistent walk over the bounce's ray queue with dynamic ray fetch
// Both:
//   accumulate           per pixel, in sample order, radiance -> accumulation buffer
//   resolve              mean, clamp, truncating RGB888 store (Image::setPixel, reference include/image.h:14-16)
//
// There is no separate extend launch after the camera segment: a queue entry always produces
// exactly one continuation ray, so compacting between "shade" and "extend" would only re-read what
// the thread already holds in registers. Every launch is a persistent grid (SM count x resident
// CTAs) that reads its queue length from device memory and is chained to its predecessor by
// programmatic dependent launch, so a frame is enqueued without a single host round trip. The RNG
// is Philox4x32-7 keyed on (global pixel, sample, bounce, stream): results do not depend on
// queue order, pass size, passes in flight or how tiles are split across GPUs.
//
// What the ncu captures drove (profiles/r01_tuning_log.md has the numbers):
//   session 1  * the kernels are issue-bound, not HBM-bound -> triangle test by a precomputed affine
//                map (6 dot products, one MUFU reciprocal, no branches), coplanar triangle pairs
//                merged into parallelograms by the builder
//              * barrier stalls from block-level compaction -> queue space is reserved in
//                warp-private 64-entry chunks: one atomic per 64 outputs, no __syncthreads
//              * long-scoreboard stalls on queue -> state dependent loads -> cp.async prefetch of
//                the next record into shared memory
//   session 2  * shade + extend fused; (pixel, sample) ride in the spare words of the vertex record
//              * flat scenes: the shadow ray and the continuation ray leave the same point, so ONE
//                loop over the primitives tests both (shared origin half, shared loads)
//              * tree scenes: while-while walk in converged rounds, dynamic ray fetch
//   session 3  * slot-indexed state cost the same time per launch whatever the number of live
//                paths (sector waste) -> dense vertex records in the queues
//              * 40 % of the instructions FP32 at 70 % issue utilisation -> primitive pairs through
//                FFMA2 / FMUL2 / FADD2
//              * every kernel ends in a tail -> several passes in flight
//
// Scene access: flat scenes stage everything (records, pairs, shading records, lights) into shared
// memory at kernel start with cp.async.bulk (TMA bulk copy, one mbarrier); tree scenes stage the
// breadth-first prefix of the node array and read the rest through L2 with read-only loads.
#include "path.h"

#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstdlib>
#include <mutex>

namespace g19 {
namespace {

constexpr int kThreads = 256;
constexpr uint32_t kFull = 0xffffffffu;
constexpr uint32_t kInvalid = 0xffffffffu; // padding entry of a queue / "no primitive"
constexpr uint32_t kChunk = 64;            // queue entries reserved per atomic (>= 32)
constexpr float kRayEps = 1.0e-3f;         // origin offset along the normal (scene units)
constexpr float kPi = 3.14159265358979323846f;
constexpr uint32_t kRayShadow = 0x80000000u;   // ray record flags riding on the slot index (< 2^30)
constexpr uint32_t kRaySpecular = 0x40000000u; // the continuation ray leaves a specular vertex
constexpr uint32_t kRaySlotMask = 0x3fffffffu;

__device__ __forceinline__ unsigned warp_sum_u(unsigned v) {
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
    return v;
}

// Streaming (evict-first) 16-byte accesses for data that is written once and read once far later (ray queue records).
// Through INTEGER registers: the records carry slot indices and flags in the bit patterns of their w words, which look
// like denormals -- the float4 overloads of __ldcs / __stcs are free to flush them (measured: every shadow ray then
// delivered to slot 0).
__device__ __forceinline__ void st_stream(float4* p, float x, float y, float z, uint32_t w_bits) {
    __stcs(reinterpret_cast<uint4*>(p), make_uint4(__float_as_uint(x), __float_as_uint(y), __float_as_uint(z), w_bits));
}
__device__ __forceinline__ float4 ld_stream(const float4* p) {
    const uint4 v = __ldcs(reinterpret_cast<const uint4*>(p));
    return make_float4(__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w));
}

// ---- Philox4x32-7 (Salmon et al. 2011: the fewest rounds that pass BigCrush; three rounds = 36 instructions per vertex
// fewer than the -10 variant of round 1); identical integer stream in oracle/path_oracle.c
__device__ __forceinline__ uint4 philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0) {
    uint32_t k1 = 0x32303139u; // "2019"
#pragma unroll
    for (int r = 0; r < 7; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01(uint32_t v) { return float(v >> 8) * (1.0f / 16777216.0f); }

// ---- small float3 kit -------------------------------------------------------
__device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float dot(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ float3 normalize(float3 v) { return v * rsqrtf(dot(v, v)); }

// ---- shared-memory scene prefix ----------------------------------------------
// Dynamic shared memory, sized on the host to what the scene needs (PassArgs::stage_*):
//   [nodes: stage_nodes x 8 B][hot primitive records: stage_prims x 64 B (flat scenes only)]
//   [cold records: stage_cold x 32 B][lights: stage_lights x 80 B]   (flat scenes only)
//   [traversal stack: stack_levels x kThreads x 4 B][mbarrier: 8 B]
// A Cornell box stages whole (about 0.8 KB) and leaves the SM free for more CTAs.
extern __shared__ __align__(16) unsigned char g19_dyn_smem[];

template <bool ALL> struct SceneAccess {
    const PathSceneD* g;
    const uint2* nodes_s;
    const float4* hot_s;
    const float4* cold_s;
    const float4* lights_s;
    const ulonglong2* pairs_s; // flat scenes: primitive PAIRS, one float2 per coefficient (trace_flat)
    const FlatPairsU* upairs;  // the same pairs in the flat bounce kernels' launch parameters (trace_flat<UNI>; set by those kernels)
    uint32_t* stack;
    int n_nodes_s;
    int walk_steps;      // tree walk: cell moves per round
    uint32_t leaf_batch; // tree walk: primitives tested per round
    int bvh_stack;       // BvhWalk: levels of the postponed-children stack in shared memory (= PassArgs::stack_levels)
    int bvh_spec;        // BvhWalk: a lane that reaches a leaf postpones it and keeps descending (speculative traversal)
    unsigned long long* coop; // tree walk, cooperative leaf tests: this warp's 32 result slots, or nullptr
    __device__ __forceinline__ uint2 node(uint32_t i) const {
        if (ALL || i < (uint32_t)n_nodes_s) return nodes_s[i];
        return __ldg(reinterpret_cast<const uint2*>(g->nodes) + i);
    }
    // shading record of primitive id `prim`: (normal, ior), (albedo, material)
    __device__ __forceinline__ void cold(uint32_t prim, float4& c0, float4& c1) const {
        if (ALL) {
            c0 = cold_s[2 * prim]; c1 = cold_s[2 * prim + 1];
        } else {
            const float4* p = reinterpret_cast<const float4*>(g->cold) + 2 * (size_t)prim;
            c0 = __ldg(p); c1 = __ldg(p + 1);
        }
    }
    // area-light record = 5 x float4: (v0, area) (e1, pdf_pick) (e2, -) (n, -) (emission, -)
    __device__ __forceinline__ const float4* light(int li) const {
        if (ALL) return lights_s + 5 * li;
        return reinterpret_cast<const float4*>(g->lights) + 5 * (size_t)li;
    }
    // row 0 / row 3 of the hot record BY PRIMITIVE ID (flat scenes: leaf order == id order)
    __device__ __forceinline__ float4 hot_row(uint32_t prim, int row) const {
        if (ALL) return hot_s[4 * prim + row];
        return __ldg(reinterpret_cast<const float4*>(g->hot) + 4 * (size_t)prim + row);
    }
};

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// Programmatic dependent launch: a pass is a chain of 7 to 40 short persistent kernels, each
// depending on the previous one's queues. Every kernel lets its successor be scheduled as soon as
// CTAs retire (launch_dependents, first instruction), does whatever does not depend on earlier
// kernels (staging the scene into shared memory), and only then waits for the predecessor's
// memory (griddepcontrol.wait): launch latency and prologue hide under the predecessor's tail.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Stage the scene prefix with TMA bulk copies (cp.async.bulk) completing on one mbarrier.
template <bool ALL> __device__ __forceinline__ SceneAccess<ALL> stage_scene(const PassArgs& a) {
    const PathSceneD& g = a.scene;
    SceneAccess<ALL> acc;
    acc.g = &a.scene;
    acc.n_nodes_s = a.stage_nodes;
    acc.walk_steps = a.walk_steps;
    acc.leaf_batch = uint32_t(a.leaf_batch);
    acc.bvh_spec = a.bvh_spec;
    acc.bvh_stack = a.stack_levels;
    acc.coop = nullptr;
    // byte counts rounded up to 16 (the device arrays are padded, see DeviceArray::ensure)
    const uint32_t nb = (uint32_t(a.stage_nodes) * 8u + 15u) & ~15u;
    const uint32_t pb = uint32_t(a.stage_prims) * 64u;
    const uint32_t cb = ALL ? uint32_t(a.stage_cold) * 32u : 0u;
    const uint32_t lb = ALL ? uint32_t(a.stage_lights) * 80u : 0u;
    const uint32_t qb = ALL ? uint32_t(g.pairs_bytes) : 0u;
    unsigned char* base = g19_dyn_smem;
    acc.nodes_s = reinterpret_cast<const uint2*>(base);
    acc.hot_s = reinterpret_cast<const float4*>(base + nb);
    acc.cold_s = reinterpret_cast<const float4*>(base + nb + pb);
    acc.lights_s = reinterpret_cast<const float4*>(base + nb + pb + cb);
    acc.pairs_s = reinterpret_cast<const ulonglong2*>(base + nb + pb + cb + lb);
    acc.stack = reinterpret_cast<uint32_t*>(base + nb + pb + cb + lb + qb) + threadIdx.x;
    unsigned long long* barp =
        reinterpret_cast<unsigned long long*>(base + nb + pb + cb + lb + qb + uint32_t(a.stack_levels) * kThreads * 4u);
    const uint32_t bar = smem_addr(barp);
    if (!ALL && a.coop_leaf) acc.coop = barp + 2 + (threadIdx.x >> 5) * 32; // [barrier 8 B, pad 8 B][8 warps x 32 slots x 8 B]
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(nb + pb + cb + lb + qb) : "memory");
        if (nb)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             smem_addr(base)),
                         "l"(g.nodes), "r"(nb), "r"(bar)
                         : "memory");
        if (pb)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             smem_addr(base + nb)),
                         "l"(g.hot), "r"(pb), "r"(bar)
                         : "memory");
        if (cb)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             smem_addr(base + nb + pb)),
                         "l"(g.cold), "r"(cb), "r"(bar)
                         : "memory");
        if (lb)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             smem_addr(base + nb + pb + cb)),
                         "l"(g.lights), "r"(lb), "r"(bar)
                         : "memory");
        if (qb)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             smem_addr(base + nb + pb + cb + lb)),
                         "l"(g.pairs), "r"(qb), "r"(bar)
                         : "memory");
    }
    uint32_t done = 0; // everyone waits for phase 0 of the barrier
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done)
                     : "r"(bar)
                     : "memory");
    }
    return acc;
}

// ---- primitive intersection ---------------------------------------------------
// Triangles / parallelograms: the ray is mapped into the primitive's own (b1, b2, h) frame by
// the precomputed affine rows -- the ORIGIN half (three 4-term dot products) is shared by every
// ray that leaves the same point, the DIRECTION half costs 9 FMAs, one fast division and 2 FMAs
// per ray. The accept test is built for the ALU pipe, the busiest one (ncu: 50 % of its peak):
//   * t in (0, tmax): ONE unsigned compare of the float bit patterns -- negative values, -0 and
//     NaN all have larger patterns than any positive bound; a switched-off ray has bound 0
//   * parallelogram (kind 2): the builder centres the coordinates, inside <=> max(|u|,|v|) <= 1/2
//   * triangle (kind 1): inside <=> min(u, v, 1 - u - v) >= 0
// Spheres: unit direction, discriminant from the perpendicular offset; the nearer root ahead of
// the origin is the unsigned minimum of the two roots' bit patterns.
struct PlaneOrigin {
    float ox, oy, oz;
};
__device__ __forceinline__ PlaneOrigin plane_origin(float4 a, float4 b, float4 c, float3 o) {
    PlaneOrigin r;
    r.oz = fmaf(c.x, o.x, fmaf(c.y, o.y, fmaf(c.z, o.z, c.w)));
    r.ox = fmaf(a.x, o.x, fmaf(a.y, o.y, fmaf(a.z, o.z, a.w)));
    r.oy = fmaf(b.x, o.x, fmaf(b.y, o.y, fmaf(b.z, o.z, b.w)));
    return r;
}
// KIND 2 parallelogram, 1 triangle. Returns "hit inside and nearer than lim"; t_bits = pattern of t.
template <int KIND>
__device__ __forceinline__ bool plane_hit(float4 a, float4 b, float4 c, PlaneOrigin po, float3 d, uint32_t lim, uint32_t& t_bits) {
    const float dz = fmaf(c.x, d.x, fmaf(c.y, d.y, c.z * d.z));
    const float t = __fdividef(-po.oz, dz);
    const float dx = fmaf(a.x, d.x, fmaf(a.y, d.y, a.z * d.z));
    const float dy = fmaf(b.x, d.x, fmaf(b.y, d.y, b.z * d.z));
    const float u = fmaf(t, dx, po.ox), v = fmaf(t, dy, po.oy);
    t_bits = __float_as_uint(t);
    if (KIND == 2) return (fmaxf(fabsf(u), fabsf(v)) <= 0.5f) & (t_bits < lim);
    return (fminf(fminf(u, v), 1.0f - (u + v)) >= 0.0f) & (t_bits < lim);
}
__device__ __forceinline__ bool sphere_hit(float3 oc, float radius, float3 d, uint32_t lim, uint32_t& t_bits) {
    const float bq = dot(oc, d);
    const float3 l = oc - d * bq;
    const float disc = fmaf(radius, radius, -dot(l, l));
    const float sq = sqrtf(disc); // NaN when the ray misses: fails the range test below
    t_bits = min(__float_as_uint(-bq - sq), __float_as_uint(sq - bq));
    return t_bits < lim;
}
__device__ __forceinline__ uint32_t range_limit(float tmax) { return tmax > 0.0f ? __float_as_uint(tmax) : 0u; }

// generic form for the mixed leaves of a tree: t in (0, tmax) or -1
__device__ __forceinline__ float hit_prim(float4 a, float4 b, float4 c, float4 tag, float3 o, float3 d, float tmax) {
    uint32_t tb;
    bool ok;
    const uint32_t lim = __float_as_uint(tmax); // callers pass tmax > 0
    if (tag.z != 0.0f) {
        const PlaneOrigin po = plane_origin(a, b, c, o);
        ok = tag.z > 1.5f ? plane_hit<2>(a, b, c, po, d, lim, tb) : plane_hit<1>(a, b, c, po, d, lim, tb);
    } else {
        ok = sphere_hit(o - f3(a.x, a.y, a.z), a.w, d, lim, tb);
    }
    return ok ? __uint_as_float(tb) : -1.0f;
}

// ---- packed FP32 pairs (sm_100: FFMA2 / FMUL2 / FADD2) -----------------------------------
// One issue slot carries two FP32 lanes; an operand built as pk(x, x) compiles to the scalar
// broadcast form (R.F32), so only the primitive coefficients need to be stored as pairs. Measured
// here (tools/ubench/ffma2.cu): 0.98 FFMA or 0.49 FFMA2 per cycle and scheduler, same 4-cycle
// dependent latency -- the FMA pipe does the same work, the ISSUE slots halve, and issue slots are
// what bounds these kernels (ncu: issue 71 %, FMA pipe 34 %, 40 % of the instructions FP32).
typedef unsigned long long f2;
__device__ __forceinline__ f2 pk(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void upk(f2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f2 bc(float x) { return pk(x, x); }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 r; asm("fma.rn.ftz.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 r; asm("mul.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 r; asm("add.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 sub2(f2 a, f2 b) { f2 r; asm("sub.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ float rcp_fast(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// A ray as the pair loops want it: direction and negated direction as scalars (broadcast operands).
struct RayDir {
    float x, y, z, nx, ny, nz;
};
__device__ __forceinline__ RayDir ray_dir(float3 d) { return RayDir{d.x, d.y, d.z, -d.x, -d.y, -d.z}; }

// Two planar primitives at once. Pair record = 6 x ulonglong2: row a = (x,y | z,w), row b, row c,
// every coefficient a float2 (primitive 2j, primitive 2j+1). Same operation order per lane as
// plane_origin / plane_hit above, so the results are bit-identical to the scalar form.
struct PlaneOrigin2 {
    f2 ox, oy, oz;
};
__device__ __forceinline__ PlaneOrigin2 plane_origin2(const ulonglong2* r, float3 o) {
    const f2 ox = bc(o.x), oy = bc(o.y), oz = bc(o.z);
    const ulonglong2 a0 = r[0], a1 = r[1], b0 = r[2], b1 = r[3], c0 = r[4], c1 = r[5];
    PlaneOrigin2 p;
    p.oz = fma2(c0.x, ox, fma2(c0.y, oy, fma2(c1.x, oz, c1.y)));
    p.ox = fma2(a0.x, ox, fma2(a0.y, oy, fma2(a1.x, oz, a1.y)));
    p.oy = fma2(b0.x, ox, fma2(b0.y, oy, fma2(b1.x, oz, b1.y)));
    return p;
}
// t = -h(o) / h'(d) is formed as h(o) * rcp(h'(-d)): no negation of a pair is needed.
__device__ __forceinline__ void plane_uvt2(const ulonglong2* r, const PlaneOrigin2& po, const RayDir& d, f2& u, f2& v, f2& t) {
    const ulonglong2 a0 = r[0], a1 = r[1], b0 = r[2], b1 = r[3], c0 = r[4], c1 = r[5];
    const f2 ndz = fma2(c0.x, bc(d.nx), fma2(c0.y, bc(d.ny), mul2(c1.x, bc(d.nz))));
    float z0, z1;
    upk(ndz, z0, z1);
    t = mul2(po.oz, pk(rcp_fast(z0), rcp_fast(z1)));
    const f2 dx = fma2(a0.x, bc(d.x), fma2(a0.y, bc(d.y), mul2(a1.x, bc(d.z))));
    const f2 dy = fma2(b0.x, bc(d.x), fma2(b0.y, bc(d.y), mul2(b1.x, bc(d.z))));
    u = fma2(t, dx, po.ox);
    v = fma2(t, dy, po.oy);
}
template <int KIND> __device__ __forceinline__ bool plane_inside(float u, float v) {
    if (KIND == 2) return fmaxf(fabsf(u), fabsf(v)) <= 0.5f;
    return fminf(fminf(u, v), 1.0f - (u + v)) >= 0.0f;
}

// Flat scene (ONE leaf, fully staged, primitives sorted parallelograms | triangles | spheres by
// the builder): nearest hit of ray (o, d1) within tmax1 and, when DUAL, any hit of ray (o, d0)
// within tmax0 -- both leave the same point, so one pass over the primitives serves both. A ray
// with tmax <= 0 is switched off. Three branch-free loops over primitive PAIRS (each kind group is
// padded to an even count with a NaN record that can never be hit); the position in its group IS
// the primitive id.
template <int KIND, bool DUAL>
__device__ __forceinline__ void plane_pair(const ulonglong2* rec, uint32_t id, float3 o, const RayDir& d1, const RayDir& d0,
                                           uint32_t& lim1, uint32_t& lim0, uint32_t& hit_k) {
    const PlaneOrigin2 po = plane_origin2(rec, o);
    f2 u, v, t;
    plane_uvt2(rec, po, d1, u, v, t);
    float ua, ub, va, vb, ta, tb;
    upk(u, ua, ub); upk(v, va, vb); upk(t, ta, tb);
    if (plane_inside<KIND>(ua, va) & (__float_as_uint(ta) < lim1)) { lim1 = __float_as_uint(ta); hit_k = id; }
    if (plane_inside<KIND>(ub, vb) & (__float_as_uint(tb) < lim1)) { lim1 = __float_as_uint(tb); hit_k = id + 1u; }
    if (DUAL) {
        plane_uvt2(rec, po, d0, u, v, t);
        upk(u, ua, ub); upk(v, va, vb); upk(t, ta, tb);
        if ((plane_inside<KIND>(ua, va) & (__float_as_uint(ta) < lim0)) | (plane_inside<KIND>(ub, vb) & (__float_as_uint(tb) < lim0)))
            lim0 = 0u;
    }
}
template <int KIND, bool DUAL>
__device__ __forceinline__ void plane_pairs(const ulonglong2* rec, uint32_t n_pairs, uint32_t id0, float3 o, const RayDir& d1,
                                            const RayDir& d0, uint32_t& lim1, uint32_t& lim0, uint32_t& hit_k) {
#pragma unroll 1
    for (uint32_t j = 0; j < n_pairs; ++j, rec += 6) plane_pair<KIND, DUAL>(rec, id0 + 2u * j, o, d1, d0, lim1, lim0, hit_k);
}
// The pairs of the launch parameters (FlatPairsU): the loop is unrolled to the capacity and left at the group's count (warp-uniform), so
// every coefficient sits at a fixed constant-bank offset and is read as a uniform operand of the FFMA2s -- no per-thread
// registers and no shared-memory loads for the 24 coefficients of a pair, no loop counter or record pointer.
template <int KIND, bool DUAL>
__device__ __forceinline__ void plane_pairs_u(const ulonglong2 (&rec)[kUniPlanarPairs][6], uint32_t n_pairs, uint32_t id0, float3 o,
                                              const RayDir& d1, const RayDir& d0, uint32_t& lim1, uint32_t& lim0, uint32_t& hit_k) {
#pragma unroll
    for (uint32_t j = 0; j < uint32_t(kUniPlanarPairs); ++j) {
        if (j >= n_pairs) break;
        plane_pair<KIND, DUAL>(rec[j], id0 + 2u * j, o, d1, d0, lim1, lim0, hit_k);
    }
}
// Sphere pair record = 2 x ulonglong2: (-cx, -cy | -cz, r^2). Unit direction, discriminant from the
// perpendicular offset; the nearer root ahead of the origin is the unsigned minimum of the roots.
__device__ __forceinline__ void sphere_roots2(f2 ocx, f2 ocy, f2 ocz, f2 rr, const RayDir& d, uint32_t& ta, uint32_t& tb) {
    const f2 bq = fma2(ocz, bc(d.z), fma2(ocy, bc(d.y), mul2(ocx, bc(d.x))));
    const f2 lx = fma2(bq, bc(d.nx), ocx), ly = fma2(bq, bc(d.ny), ocy), lz = fma2(bq, bc(d.nz), ocz);
    const f2 disc = sub2(rr, fma2(lz, lz, fma2(ly, ly, mul2(lx, lx))));
    float b0, b1, q0, q1;
    upk(bq, b0, b1);
    upk(disc, q0, q1);
    const float s0 = sqrtf(q0), s1 = sqrtf(q1); // NaN when the ray misses: fails the range test
    ta = min(__float_as_uint(-b0 - s0), __float_as_uint(s0 - b0));
    tb = min(__float_as_uint(-b1 - s1), __float_as_uint(s1 - b1));
}
template <bool DUAL>
__device__ __forceinline__ void sphere_pair(const ulonglong2* rec, uint32_t id, float3 o, const RayDir& r1, const RayDir& r0,
                                            uint32_t& lim1, uint32_t& lim0, uint32_t& hit_k) {
    const ulonglong2 c0 = rec[0], c1 = rec[1];
    const f2 ocx = add2(c0.x, bc(o.x)), ocy = add2(c0.y, bc(o.y)), ocz = add2(c1.x, bc(o.z));
    uint32_t ta, tb;
    sphere_roots2(ocx, ocy, ocz, c1.y, r1, ta, tb);
    if (ta < lim1) { lim1 = ta; hit_k = id; }
    if (tb < lim1) { lim1 = tb; hit_k = id + 1u; }
    if (DUAL) {
        sphere_roots2(ocx, ocy, ocz, c1.y, r0, ta, tb);
        if ((ta < lim0) | (tb < lim0)) lim0 = 0u;
    }
}
// UNI: the pairs come from the launch parameters (S.upairs; the scene fits FlatPairsU: PassArgs::flat_uniform) instead of
// shared memory.
template <bool DUAL, bool UNI = false>
__device__ __forceinline__ void trace_flat(const SceneAccess<true>& S, float3 o, float3 d1, float tmax1, float3 d0,
                                           float tmax0, float& best, uint32_t& best_k, bool& occluded) {
    uint32_t lim1 = range_limit(tmax1), lim0 = DUAL ? range_limit(tmax0) : 0u;
    uint32_t hit_k = kInvalid;
    const uint32_t n_par = uint32_t(S.g->n_par), n_tri = uint32_t(S.g->n_tri), n = uint32_t(S.g->n_prims);
    const uint32_t p_par = (n_par + 1u) >> 1, p_tri = (n_tri + 1u) >> 1, p_sph = (n - n_par - n_tri + 1u) >> 1;
    const RayDir r1 = ray_dir(d1), r0 = ray_dir(d0);
    if (UNI) {
        const FlatPairsU& P = *S.upairs;
        plane_pairs_u<2, DUAL>(P.par, p_par, 0u, o, r1, r0, lim1, lim0, hit_k);
        plane_pairs_u<1, DUAL>(P.tri, p_tri, n_par, o, r1, r0, lim1, lim0, hit_k);
#pragma unroll
        for (uint32_t j = 0; j < uint32_t(kUniSpherePairs); ++j) {
            if (j >= p_sph) break;
            sphere_pair<DUAL>(P.sph[j], n_par + n_tri + 2u * j, o, r1, r0, lim1, lim0, hit_k);
        }
    } else {
        const ulonglong2* rec = S.pairs_s;
        plane_pairs<2, DUAL>(rec, p_par, 0u, o, r1, r0, lim1, lim0, hit_k);
        rec += 6u * p_par;
        plane_pairs<1, DUAL>(rec, p_tri, n_par, o, r1, r0, lim1, lim0, hit_k);
        rec += 6u * p_tri;
#pragma unroll 1
        for (uint32_t j = 0; j < p_sph; ++j, rec += 2) sphere_pair<DUAL>(rec, n_par + n_tri + 2u * j, o, r1, r0, lim1, lim0, hit_k);
    }
    best = __uint_as_float(lim1);
    best_k = hit_k;
    occluded = DUAL && tmax0 > 0.0f && lim0 == 0u;
}

// ---- octree walk (tree scenes) ---------------------------------------------------------------
// What the ncu capture of the 1M-triangle heightfield drove (profiles/r01b_heightfield_*):
//   * 4.4 of 32 threads active per instruction: the one-big-loop form serialised "step",
//     "descend", "test leaf" and "pop" branches -> WHILE-WHILE form: every lane first walks to
//     its next non-empty leaf (lanes that found one wait at the reconvergence point), then all
//     lanes test their leaves together
//   * 443 MB of leaf-ordered primitive copies (6.9 references per primitive) streamed from DRAM
//     -> leaves hold 4-byte indices into the 64-byte records: nodes + indices + records = 108 MB,
//     L2-resident on B200 (126 MB)
// The walk is a resumable state machine: init() places the ray at the root, step() advances it
// to its next non-empty leaf and tests that leaf (one while-while round), returning true when
// the ray is finished. traverse() below runs it to completion; trace_kernel interleaves the
// steps of 32 rays per warp and hands a finished lane the next ray of the queue.

// The leaf test of the octree walk's sequential form and of a scene that is one whole leaf: the ray (o, d) against up to
// `limit` primitives of the leaf list [first, first + n), nearest hit within `best`, two per step (independent FMA chains,
// all loads of the step issued up front). `any` = stop at the first hit (shadow rays).
struct LeafTest {
    float3 o, d;
    float best;
    uint32_t best_prim;
    bool any;

    __device__ __forceinline__ void run(const PathSceneD& g, uint32_t first, uint32_t n, uint32_t limit) {
        const uint32_t* __restrict__ index = g.index;
        const float4* __restrict__ hot = reinterpret_cast<const float4*>(g.hot);
        if (n > limit) n = limit;
        uint32_t id0 = __ldg(index + first), id1 = n > 1 ? __ldg(index + first + 1) : id0;
        for (uint32_t k = 0; k < n; k += 2) {
            const float4* p0 = hot + 4 * (size_t)id0;
            const float4* p1 = hot + 4 * (size_t)id1;
            const float4 a0 = __ldg(p0), b0 = __ldg(p0 + 1), c0 = __ldg(p0 + 2), g0 = __ldg(p0 + 3);
            const float4 a1 = __ldg(p1), b1 = __ldg(p1 + 1), c1 = __ldg(p1 + 2), g1 = __ldg(p1 + 3);
            const uint32_t cur0 = id0, cur1 = id1;
            const bool second = k + 1 < n;
            if (k + 2 < n) id0 = __ldg(index + first + k + 2); // next step's indices while this one computes
            if (k + 3 < n) id1 = __ldg(index + first + k + 3);
            else id1 = id0;
            const float t0 = hit_prim(a0, b0, c0, g0, o, d, best);
            if (t0 >= 0.0f) { best = t0; best_prim = cur0; }
            const float t1 = second ? hit_prim(a1, b1, c1, g1, o, d, best) : -1.0f;
            if (t1 >= 0.0f) { best = t1; best_prim = cur1; }
            if (any && best_prim != kInvalid) break;
        }
    }
};

// ---- TreeWalk2: point-location restart walk ---------------------------------------------------
// What the round-1 capture of the walk this one replaced, a parametric front-to-back walk after Revelles et al. 2000
// (profiles/r01f_tree_kernels_ncu.json), showed: ~870 warp
// instructions per ray at 13.7 of 32 lanes, 62 % of them cell MOVES at ~130 instructions each -- every move
// recomputes nine plane parameters, edits a 64-bit code word with variable shifts and runs a four-way
// leave / descend / skip / arrive decision, and going from one leaf to a neighbour under another ancestor costs one
// move per level up plus one per level down. This walk keeps the ray's position as INTEGER coordinates (X, Y, Z) on
// the finest grid of the octree (2^14 cells per axis; node boxes are implicit, so a cell of level l is the top l
// bits) and does three cheap things per visited cell:
//   descend   from the deepest ancestor still valid for (X, Y, Z) -- its child base sits on the per-thread stack in
//             shared memory -- follow the coordinate bits down to the leaf or empty cell: three bit extracts, one
//             8-byte node record, ~12 instructions per level, typically 1-3 levels
//   exit      the parameter at which the ray leaves the cell: one FMA per axis on the linear plane form
//             t(i) = A + i * (B * 2^-level), A = (root_lo - o) / d and B = root_size / d per axis (the planes a cell
//             shares with its parent get bit-identical parameters: same exact product), minimum of three
//   advance   step the exit axis' coordinate to the neighbouring cell (exact integer arithmetic: no epsilon nudging),
//             re-derive the other two from the exit point clamped to the current cell's range, and find the common
//             ancestor with one XOR + CLZ
// -- no plane registers, no code word, no pops. Cells are visited strictly in ray order, so the walk still stops at
// the first leaf whose hit lies inside its own cell. COUNT: node records visited and primitives tested are tallied
// for the issue-roofline model (SURVEY.md 8(d)); instantiated only under params.profile.
template <bool COUNT> struct TreeWalk2 {
    float3 o, d, A, B;
    float best;
    uint32_t best_prim;
    uint32_t X, Y, Z;            // position on the finest grid
    uint32_t lv;                 // deepest level whose stack entry (child base) is valid for (X, Y, Z)
    float t_exit;                // where the ray leaves the current cell (valid while an advance is pending)
    uint32_t leaf_first, leaf_n; // the part of the current leaf's list still to be tested
    float leaf_exit;
    uint32_t state;              // bit 0: any-hit ray; bit 1: advance pending; bits 2-3: exit axis
    uint32_t n_node, n_prim;     // COUNT only

    template <bool ALL>
    __device__ __forceinline__ bool init(const SceneAccess<ALL>& S, float3 o_, float3 d_, float tmax, bool any_) {
        const PathSceneD& g = *S.g;
        o = o_;
        d = d_;
        best = tmax;
        best_prim = kInvalid;
        state = any_ ? 1u : 0u;
        leaf_n = 0;
        const uint2 root = S.node(0);
        if (root.y & kLeafBit) { // the whole scene is one leaf (but not staged as a flat scene)
            LeafTest w0 = {}; // (set member by member: aggregate initialisation compiles the same arithmetic to other SASS)
            w0.o = o; w0.d = d; w0.best = best; w0.best_prim = kInvalid; w0.any = any_;
            w0.run(g, root.x, root.y & ~kLeafBit, 0x7fffffffu);
            best = w0.best;
            best_prim = w0.best_prim;
            return true;
        }
        // slab clip against the root box; an axis the ray (almost) does not move along never produces an exit
        float tn = 0.0f, tf = best;
        bool miss = false;
        const float inf = __int_as_float(0x7f800000);
#define G19_AXIS(c, k)                                                                  \
        if (fabsf(d.c) < 1.0e-12f) {                                                    \
            miss |= o.c < g.root_lo[k] || o.c > g.root_lo[k] + g.root_size[k];          \
            A.c = inf; B.c = 0.0f;                                                      \
        } else {                                                                        \
            const float inv = __fdividef(1.0f, d.c);                                    \
            A.c = (g.root_lo[k] - o.c) * inv;                                           \
            B.c = g.root_size[k] * inv;                                                 \
            const float t1 = A.c + B.c;                                                 \
            tn = fmaxf(tn, fminf(A.c, t1));                                             \
            tf = fminf(tf, fmaxf(A.c, t1));                                             \
        }
        G19_AXIS(x, 0) G19_AXIS(y, 1) G19_AXIS(z, 2)
#undef G19_AXIS
        if (miss || tn > tf + 1.0e-5f) return true;
        const int hi = (1 << kMaxTreeDepth) - 1;
        X = uint32_t(min(max(__float2int_rd((fmaf(d.x, tn, o.x) - g.root_lo[0]) * g.grid_scale[0]), 0), hi));
        Y = uint32_t(min(max(__float2int_rd((fmaf(d.y, tn, o.y) - g.root_lo[1]) * g.grid_scale[1]), 0), hi));
        Z = uint32_t(min(max(__float2int_rd((fmaf(d.z, tn, o.z) - g.root_lo[2]) * g.grid_scale[2]), 0), hi));
        lv = 0;
        S.stack[0] = root.x;
        if (COUNT) n_node = n_prim = 0;
        return false;
    }

    // One ROUND for the 32 rays of a warp (MUST be called by all lanes, `active` = this lane has a ray): walk_steps
    // times [advance out of the finished cell, descend to the next leaf / empty cell, compute its exit], then one
    // batch of at most leaf_batch primitives of the lanes that stand in a leaf. Returns true when the lane's ray is
    // finished. The fixed-trip loop re-converges the warp at every move: with `continue` / `break` in a data-dependent
    // loop the lanes drifted apart and ran the loop body in ~2.5 separate groups of 5.6 lanes (ncu,
    // profiles/r01_tuning_log.md).
    template <bool ALL, bool COOP> __device__ __forceinline__ bool step(const SceneAccess<ALL>& S, bool active) {
        uint32_t* const stack = S.stack;
        const PathSceneD& g = *S.g;
        bool done = false;
        const int kWalkSteps = S.walk_steps;
        const uint32_t kLeafBatch = S.leaf_batch;
#pragma unroll 1
        for (int it = 0; it < kWalkSteps; ++it) {
            __syncwarp();
            bool walking = active && !done && leaf_n == 0u;
            if (walking && (state & 2u)) {
                // ---- advance: out of the current cell through its exit face ----
                const uint32_t s = uint32_t(kMaxTreeDepth - 1) - lv; // the cell is at level lv + 1: it spans 2^s fine cells per axis
                const uint32_t axis = (state >> 2) & 3u;
                const uint32_t mask = (1u << s) - 1u;
                const int hi = (1 << kMaxTreeDepth) - 1;
                // the exit point on the finest grid, held inside the current cell (it IS on the cell's boundary)
                int nx = __float2int_rd((fmaf(d.x, t_exit, o.x) - g.root_lo[0]) * g.grid_scale[0]);
                int ny = __float2int_rd((fmaf(d.y, t_exit, o.y) - g.root_lo[1]) * g.grid_scale[1]);
                int nz = __float2int_rd((fmaf(d.z, t_exit, o.z) - g.root_lo[2]) * g.grid_scale[2]);
                const int x0 = int(X & ~mask), y0 = int(Y & ~mask), z0 = int(Z & ~mask);
                nx = min(max(nx, x0), x0 + int(mask));
                ny = min(max(ny, y0), y0 + int(mask));
                nz = min(max(nz, z0), z0 + int(mask));
                // ... and one cell further along the exit axis
                if (axis == 0u) nx = d.x > 0.0f ? x0 + int(mask) + 1 : x0 - 1;
                else if (axis == 1u) ny = d.y > 0.0f ? y0 + int(mask) + 1 : y0 - 1;
                else nz = d.z > 0.0f ? z0 + int(mask) + 1 : z0 - 1;
                if ((nx | ny | nz) < 0 || nx > hi || ny > hi || nz > hi) {
                    done = true; // left the root box
                    walking = false;
                } else {
                    const uint32_t diff = (X ^ uint32_t(nx)) | (Y ^ uint32_t(ny)) | (Z ^ uint32_t(nz));
                    // highest differing bit h = 31 - clz: the level-m ancestors agree for m <= kMaxTreeDepth - 1 - h
                    lv = min(lv, uint32_t(__clz(int(diff))) - uint32_t(32 - kMaxTreeDepth));
                    X = uint32_t(nx); Y = uint32_t(ny); Z = uint32_t(nz);
                }
                state &= ~2u;
            }
            // ---- descend to the leaf / empty cell that holds (X, Y, Z) ----
            bool desc = walking;
            uint32_t k = lv;
            uint2 rec = make_uint2(0u, kLeafBit);
            // a descent that would start above the top table's level starts IN the table: one load instead of a
            // chain of top_level dependent ones
            const uint32_t top_level = uint32_t(g.top_level);
            if (desc && k < top_level) {
                const uint32_t sh = uint32_t(kMaxTreeDepth) - top_level;
                rec = __ldg(g.top + ((((size_t(Z >> sh) << top_level) | (Y >> sh)) << top_level) | (X >> sh)));
                if (COUNT) ++n_node;
                if (rec.y & kLeafBit) {
                    k = ((rec.y >> 24) & 0xfu) - 1u; // the covering leaf / empty cell sits at that (coarser) level
                    rec.y &= 0x80ffffffu;
                    desc = false;
                } else {
                    k = top_level;
                    stack[k * kThreads] = rec.x;
                }
            }
            while (__any_sync(kFull, desc)) {
                if (desc) {
                    const uint32_t sh = uint32_t(kMaxTreeDepth - 1) - k;
                    const uint32_t c = ((X >> sh) & 1u) | (((Y >> sh) & 1u) << 1) | (((Z >> sh) & 1u) << 2);
                    rec = S.node(stack[k * kThreads] + c);
                    if (COUNT) ++n_node;
                    if ((rec.y & kLeafBit) || k + 1u >= uint32_t(kMaxTreeDepth)) {
                        desc = false;
                    } else {
                        ++k;
                        stack[k * kThreads] = rec.x;
                    }
                }
            }
            if (walking) {
                lv = k;
                // ---- exit parameter of the cell (level lv + 1): the far plane per axis, linear in the plane index ----
                const uint32_t sh = uint32_t(kMaxTreeDepth - 1) - k;
                const float s1 = __int_as_float((127 - int(k + 1u)) << 23); // 2^-(level), exact
                const float fx = float((X >> sh) + (d.x > 0.0f ? 1u : 0u)), fy = float((Y >> sh) + (d.y > 0.0f ? 1u : 0u)),
                            fz = float((Z >> sh) + (d.z > 0.0f ? 1u : 0u));
                const float tx = fmaf(fx, B.x * s1, A.x), ty = fmaf(fy, B.y * s1, A.y), tz = fmaf(fz, B.z * s1, A.z);
                const uint32_t axis = (tx <= ty && tx <= tz) ? 0u : (ty <= tz ? 1u : 2u);
                t_exit = fminf(fminf(tx, ty), tz);
                state = (state & 1u) | 2u | (axis << 2);
                if (rec.y != kLeafBit) { // a leaf with primitives
                    leaf_first = rec.x;
                    leaf_n = rec.y & ~kLeafBit;
                    leaf_exit = t_exit;
                } else if (t_exit >= best) {
                    done = true; // empty cell, and everything beyond it is farther than the hit / the ray's end
                }
            }
        }
        __syncwarp();
        // ---- test: the next batch of the current leaf's primitives ----
        const bool any = (state & 1u) != 0u;
        if constexpr (COOP) {
            // COOPERATIVE form (default; coop_leaf = 0 selects the sequential one): ncu showed the leaf batches running at
            // ~8 of 32 lanes (only the lanes that stand in a leaf) for 28 % of trace_kernel's instructions. Here the warp's
            // pending (ray, primitive) pairs are spread over all 32 lanes: a lane looks up which ray task j belongs to
            // (binary search over the inclusive prefix sum of the batch sizes), fetches that ray by shuffle, tests ONE
            // primitive, and the nearest hit per ray is reduced with a 64-bit atomicMin on (t bits << 32 | primitive) in
            // the warp's shared-memory slots. Same hits as the sequential form; a tie in t goes to the lower primitive id.
            const uint32_t lane = threadIdx.x & 31u;
            const bool mine = active && !done && leaf_n != 0u;
            const uint32_t cnt = mine ? (leaf_n < kLeafBatch ? leaf_n : kLeafBatch) : 0u;
            if (__ballot_sync(kFull, cnt != 0u) != 0u) {
                uint32_t inc = cnt; // inclusive prefix sum over the lanes
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const uint32_t v = __shfl_up_sync(kFull, inc, off);
                    if (lane >= uint32_t(off)) inc += v;
                }
                const uint32_t total = __shfl_sync(kFull, inc, 31);
                const uint32_t exc = inc - cnt;
                S.coop[lane] = ~0ull;
                __syncwarp();
                const uint32_t* __restrict__ index = g.index;
                const float4* __restrict__ hot = reinterpret_cast<const float4*>(g.hot);
                for (uint32_t base = 0; base < total; base += 32u) {
                    const uint32_t j = base + lane;
                    uint32_t own = 0; // number of lanes whose tasks all lie before j = the owner of task j
#pragma unroll
                    for (int stepw = 16; stepw > 0; stepw >>= 1) {
                        const uint32_t probe = __shfl_sync(kFull, inc, int(own) + stepw - 1);
                        if (probe <= j) own += uint32_t(stepw);
                    }
                    const bool valid = j < total;
                    if (!valid) own = 0;
                    const uint32_t kk = j - __shfl_sync(kFull, exc, int(own));
                    const uint32_t lf = __shfl_sync(kFull, leaf_first, int(own));
                    const float rox = __shfl_sync(kFull, o.x, int(own)), roy = __shfl_sync(kFull, o.y, int(own)), roz = __shfl_sync(kFull, o.z, int(own));
                    const float rdx = __shfl_sync(kFull, d.x, int(own)), rdy = __shfl_sync(kFull, d.y, int(own)), rdz = __shfl_sync(kFull, d.z, int(own));
                    const float rbest = __shfl_sync(kFull, best, int(own));
                    if (valid) {
                        const uint32_t id = __ldg(index + lf + kk);
                        const float4* pp = hot + 4 * (size_t)id;
                        const float4 a0 = __ldg(pp), b0 = __ldg(pp + 1), c0 = __ldg(pp + 2), g0 = __ldg(pp + 3);
                        const float t = hit_prim(a0, b0, c0, g0, f3(rox, roy, roz), f3(rdx, rdy, rdz), rbest);
                        if (t >= 0.0f) atomicMin(S.coop + own, ((unsigned long long)__float_as_uint(t) << 32) | id);
                    }
                }
                __syncwarp();
                if (cnt != 0u) {
                    const unsigned long long r = S.coop[lane];
                    if (r != ~0ull) { best = __uint_as_float(uint32_t(r >> 32)); best_prim = uint32_t(r); }
                    if (COUNT) n_prim += cnt;
                    leaf_first += cnt;
                    leaf_n -= cnt;
                    if (any && best_prim != kInvalid) done = true;
                    else if (leaf_n == 0u && leaf_exit >= best) done = true; // the hit lies inside this cell / the ray ends here
                }
                __syncwarp();
            }
        } else if (active && !done && leaf_n != 0u) { // sequential form: every lane tests its own leaf's primitives
            LeafTest w0 = {};
            w0.o = o; w0.d = d; w0.best = best; w0.best_prim = best_prim; w0.any = any;
            w0.run(g, leaf_first, leaf_n, kLeafBatch);
            best = w0.best;
            best_prim = w0.best_prim;
            const uint32_t tested = leaf_n < kLeafBatch ? leaf_n : kLeafBatch;
            if (COUNT) n_prim += tested;
            leaf_first += tested;
            leaf_n -= tested;
            if (any && best_prim != kInvalid) done = true;
            else if (leaf_n == 0u && leaf_exit >= best) done = true;
        }
        __syncwarp();
        return done;
    }
};

// ---- BvhWalk: bounding-volume hierarchy (bvh_build.cu) --------------------------------------------------
// Same resumable interface as the octree walks (init / step / best / best_prim), so trace_kernel's dynamic ray fetch and
// the camera-ray kernel use it unchanged. A round = walk_steps node visits (a node record is both children's boxes: two
// slab tests against [0, nearest hit so far], descend into the nearer child that is hit, push the other) followed by one
// leaf visit for the lanes that stand at a leaf (1-4 primitives, contiguous 64-byte records in leaf order: one load
// chain). Fixed-trip and predicated like the octree rounds, so the warp re-converges after every visit. The stack of
// postponed children lives in local memory (L1): an LBVH over 30-bit Morton codes is at most ~40 levels deep.
// The few primitives the host kept out of the hierarchy (walls around a mesh: their boxes would cover every level above
// them) are tested first -- which also gives the walk a finite nearest-hit bound from its first node on.
// The primitives the host kept out of the hierarchy, nearest hit within `best`: the flat scenes' pair loops (two
// primitives per packed-FP32 instruction, kind-sorted, no branch per primitive) over records every lane reads from the
// same addresses. Round 2 capture: the room's seven big primitives were 2/3 of all primitive tests of the BVH walk.
__device__ __forceinline__ void bvh_big_hits(const PathSceneD& g, float3 o, float3 d, float& best, uint32_t& best_prim) {
    if (g.n_big == 0) return;
    uint32_t lim1 = range_limit(best), lim0 = 0u, hit_k = kInvalid;
    const uint32_t n_par = uint32_t(g.big_par), n_tri = uint32_t(g.big_tri), n = uint32_t(g.n_big);
    const uint32_t p_par = (n_par + 1u) >> 1, p_tri = (n_tri + 1u) >> 1, p_sph = (n - n_par - n_tri + 1u) >> 1;
    const RayDir r1 = ray_dir(d);
    const ulonglong2* rec = reinterpret_cast<const ulonglong2*>(g.bvh_big_pairs);
    plane_pairs<2, false>(rec, p_par, 0u, o, r1, r1, lim1, lim0, hit_k);
    rec += 6u * p_par;
    plane_pairs<1, false>(rec, p_tri, n_par, o, r1, r1, lim1, lim0, hit_k);
    rec += 6u * p_tri;
#pragma unroll 1
    for (uint32_t j = 0; j < p_sph; ++j, rec += 2) {
        const ulonglong2 c0 = rec[0], c1 = rec[1];
        const f2 ocx = add2(c0.x, bc(o.x)), ocy = add2(c0.y, bc(o.y)), ocz = add2(c1.x, bc(o.z));
        uint32_t ta, tb;
        sphere_roots2(ocx, ocy, ocz, c1.y, r1, ta, tb);
        const uint32_t id = n_par + n_tri + 2u * j;
        if (ta < lim1) { lim1 = ta; hit_k = id; }
        if (tb < lim1) { lim1 = tb; hit_k = id + 1u; }
    }
    if (hit_k != kInvalid) {
        best = __uint_as_float(lim1);
        best_prim = __ldg(g.bvh_big + hit_k);
    }
}

constexpr uint32_t kBvhLeaf = 0x80000000u, kBvhDone = 0xffffffffu;
// Entries beyond the shared-memory levels live in local memory (rarely touched). Together they can hold the deepest walk
// there is: Karras' tree over (30-bit code, 32-bit position) keys is at most 62 levels deep, the binary walk postpones at
// most one child per level, the 4-wide walk (31 levels) at most three.
constexpr int kBvhLocalStack = 96;
struct BvhWalk {
    float3 o, d, idir, ood;
    float best;
    uint32_t best_prim;
    uint32_t cur;  // node index, kBvhLeaf | (count - 1) << 28 | first, or kBvhDone
    uint32_t pend; // a leaf reached but not tested yet (speculative traversal), 0 = none
    uint32_t any;
    int sp, cap; // cap: stack levels in shared memory
    uint32_t stk[kBvhLocalStack];

    // The postponed children: the first kBvhSmemStack levels in the thread's column of shared memory (the capture of the
    // all-local form had 22 % of trace_kernel's stall samples on the push / pop lines), deeper ones in local memory.
    __device__ __forceinline__ void push(uint32_t* __restrict__ smem, uint32_t v) {
        if (sp < cap) smem[sp * kThreads] = v;
        else if (sp < cap + kBvhLocalStack) stk[sp - cap] = v;
        else return;
        ++sp;
    }
    __device__ __forceinline__ void pop(const uint32_t* __restrict__ smem) {
        if (sp == 0) { cur = kBvhDone; return; }
        --sp;
        cur = sp < cap ? smem[sp * kThreads] : stk[sp - cap];
    }

    template <bool ALL>
    __device__ __forceinline__ bool init(const SceneAccess<ALL>& S, float3 o_, float3 d_, float tmax, bool any_) {
        const PathSceneD& g = *S.g;
        o = o_;
        d = d_;
        best = tmax;
        best_prim = kInvalid;
        any = any_ ? 1u : 0u;
        sp = 0;
        cap = S.bvh_stack;
        pend = 0u;
        bvh_big_hits(g, o, d, best, best_prim);
        if (any_ && best_prim != kInvalid) return true;
        float3 dd = d;
        if (fabsf(dd.x) < 1.0e-20f) dd.x = copysignf(1.0e-20f, dd.x);
        if (fabsf(dd.y) < 1.0e-20f) dd.y = copysignf(1.0e-20f, dd.y);
        if (fabsf(dd.z) < 1.0e-20f) dd.z = copysignf(1.0e-20f, dd.z);
        idir = f3(__fdividef(1.0f, dd.x), __fdividef(1.0f, dd.y), __fdividef(1.0f, dd.z));
        ood = f3(o.x * idir.x, o.y * idir.y, o.z * idir.z);
        cur = g.bvh_root;
        return cur == kBvhDone;
    }

    template <bool ALL, bool COOP> __device__ __forceinline__ bool step(const SceneAccess<ALL>& S, bool active) {
        const PathSceneD& g = *S.g;
        const int kWalkSteps = S.walk_steps;
        const float4* __restrict__ nodes = g.bvh_nodes;
#pragma unroll 1
        const bool spec = (S.bvh_spec & 1) != 0;
        for (int it = 0; it < kWalkSteps; ++it) {
            __syncwarp();
            // Speculative traversal (Aila & Laine 2009): a lane that arrives at a leaf while the others still descend
            // puts the leaf aside and goes on with its next postponed node instead of idling until the leaf step. The
            // nearest-hit bound is then one leaf behind, which can only cost visits, never a hit.
            if (spec && active && pend == 0u && cur >= kBvhLeaf && cur != kBvhDone) {
                pend = cur;
                pop(S.stack);
            }
            if (active && cur < kBvhLeaf) { // an internal node: both children's slabs
                const float4* __restrict__ np = nodes + 4 * (size_t)cur;
                const float4 n0 = __ldg(np), n1 = __ldg(np + 1), n2 = __ldg(np + 2), n3 = __ldg(np + 3);
                // slightly widened: a hit ON a box face must not be lost to rounding (the primitive test decides)
                const float hi = best * 1.000002f + 1.0e-6f;
                const float c0lox = fmaf(n0.x, idir.x, -ood.x), c0hix = fmaf(n0.y, idir.x, -ood.x);
                const float c0loy = fmaf(n0.z, idir.y, -ood.y), c0hiy = fmaf(n0.w, idir.y, -ood.y);
                const float c0loz = fmaf(n2.x, idir.z, -ood.z), c0hiz = fmaf(n2.y, idir.z, -ood.z);
                const float c1lox = fmaf(n1.x, idir.x, -ood.x), c1hix = fmaf(n1.y, idir.x, -ood.x);
                const float c1loy = fmaf(n1.z, idir.y, -ood.y), c1hiy = fmaf(n1.w, idir.y, -ood.y);
                const float c1loz = fmaf(n2.z, idir.z, -ood.z), c1hiz = fmaf(n2.w, idir.z, -ood.z);
                const float t0n = fmaxf(fmaxf(fminf(c0lox, c0hix), fminf(c0loy, c0hiy)), fmaxf(fminf(c0loz, c0hiz), 0.0f));
                const float t0f = fminf(fminf(fmaxf(c0lox, c0hix), fmaxf(c0loy, c0hiy)), fminf(fmaxf(c0loz, c0hiz), hi));
                const float t1n = fmaxf(fmaxf(fminf(c1lox, c1hix), fminf(c1loy, c1hiy)), fmaxf(fminf(c1loz, c1hiz), 0.0f));
                const float t1f = fminf(fminf(fmaxf(c1lox, c1hix), fmaxf(c1loy, c1hiy)), fminf(fmaxf(c1loz, c1hiz), hi));
                // (1 + 3 ulp on the far side: the products above round independently)
                const bool h0 = t0n <= t0f * 1.0000004f, h1 = t1n <= t1f * 1.0000004f;
                const uint32_t r0 = __float_as_uint(n3.x), r1 = __float_as_uint(n3.y);
                const bool both = h0 && h1, swap = both && t1n < t0n; // swap: child 1 is entered first
                if (both) push(S.stack, swap ? r0 : r1);
                if (h0 || h1) cur = (h0 && !swap) ? r0 : r1;
                else pop(S.stack);
            }
        }
        __syncwarp();
        if (active && pend == 0u && cur >= kBvhLeaf && cur != kBvhDone) { // the leaf the lane stands at
            pend = cur;
            pop(S.stack);
        }
        if (active && pend != 0u) { // a leaf: its primitives, nearest so far kept
            const uint32_t first = pend & 0x0fffffffu, cnt = ((pend >> 28) & 7u) + 1u;
            pend = 0u;
            const float4* __restrict__ pp = g.bvh_prims + 4 * (size_t)first;
#pragma unroll 1
            for (uint32_t k = 0; k < cnt; ++k, pp += 4) {
                const float4 a0 = __ldg(pp), b0 = __ldg(pp + 1), c0 = __ldg(pp + 2), g0 = __ldg(pp + 3);
                const float t = hit_prim(a0, b0, c0, g0, o, d, best);
                if (t >= 0.0f) { best = t; best_prim = __float_as_uint(g0.w); }
            }
            if (any && best_prim != kInvalid) cur = kBvhDone;
        }
        __syncwarp();
        return active && cur == kBvhDone;
    }
};

// ---- Bvh4Walk: the 4-wide, quantised form of the same hierarchy ---------------------------------------------
// What the capture of the binary walk showed (profiles/r02m_*): issue 37 %, but the L1 data pipe at 81 % of its peak --
// every lane pulls its own 64-byte node record through L1, four wavefronts per visit. Here the same four wavefronts
// carry FOUR children (boxes as 16-bit coordinates on the root box's grid, bvh_build.cu), and a ray makes half as many
// dependent visits. A coordinate q becomes a float with one byte permute and one subtraction (0x4B000000 | q is the
// float 2^23 + q), the grid scale and the ray's origin are folded into the per-ray slab constants (sc, of), the hit
// children are ordered by entry distance with a five-exchange network on (distance bits | slot) keys, nearest entered,
// the others pushed farthest first.
template <bool COUNT> struct Bvh4Walk { // COUNT: box and primitive tests are tallied (params.profile: the issue-roofline model)
    float3 o, d, sc, of; // slab parameter of grid coordinate q along x: q * sc.x + of.x
    uint32_t n_node, n_prim; // COUNT only
    float best;
    uint32_t best_prim;
    uint32_t cur, pend, any;
    int sp, cap; // cap: stack levels in shared memory
    uint32_t stk[kBvhLocalStack];

    __device__ __forceinline__ void push(uint32_t* __restrict__ smem, uint32_t v) {
        if (sp < cap) smem[sp * kThreads] = v;
        else if (sp < cap + kBvhLocalStack) stk[sp - cap] = v;
        else return;
        ++sp;
    }
    __device__ __forceinline__ void pop(const uint32_t* __restrict__ smem) {
        if (sp == 0) { cur = kBvhDone; return; }
        --sp;
        cur = sp < cap ? smem[sp * kThreads] : stk[sp - cap];
    }

    template <bool ALL>
    __device__ __forceinline__ bool init(const SceneAccess<ALL>& S, float3 o_, float3 d_, float tmax, bool any_) {
        const PathSceneD& g = *S.g;
        o = o_;
        d = d_;
        best = tmax;
        best_prim = kInvalid;
        any = any_ ? 1u : 0u;
        sp = 0;
        cap = S.bvh_stack;
        pend = 0u;
        if (COUNT) { n_node = 0; n_prim = uint32_t(g.n_big); }
        bvh_big_hits(g, o, d, best, best_prim);
        if (any_ && best_prim != kInvalid) return true;
        float3 dd = d;
        if (fabsf(dd.x) < 1.0e-20f) dd.x = copysignf(1.0e-20f, dd.x);
        if (fabsf(dd.y) < 1.0e-20f) dd.y = copysignf(1.0e-20f, dd.y);
        if (fabsf(dd.z) < 1.0e-20f) dd.z = copysignf(1.0e-20f, dd.z);
        const float3 idir = f3(__fdividef(1.0f, dd.x), __fdividef(1.0f, dd.y), __fdividef(1.0f, dd.z));
        sc = f3(g.root_size[0] * (1.0f / 65535.0f) * idir.x, g.root_size[1] * (1.0f / 65535.0f) * idir.y, g.root_size[2] * (1.0f / 65535.0f) * idir.z);
        of = f3((g.root_lo[0] - o.x) * idir.x, (g.root_lo[1] - o.y) * idir.y, (g.root_lo[2] - o.z) * idir.z);
        cur = g.bvh_root;
        return cur == kBvhDone;
    }

    // 16-bit grid coordinate (low / high half of w) as a float: exact
    __device__ __forceinline__ static float q_lo(uint32_t w) { return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7610)) - 8388608.0f; }
    __device__ __forceinline__ static float q_hi(uint32_t w) { return __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7632)) - 8388608.0f; }

    // entry distance of one child as an orderable key: distance bits with the slot number in the two lowest bits, or
    // 0xffffffff when the slab test fails
    __device__ __forceinline__ uint32_t child_key(float lox, float hix, float loy, float hiy, float loz, float hiz, float hi, uint32_t slot) const {
        const float ax = fmaf(lox, sc.x, of.x), bx = fmaf(hix, sc.x, of.x);
        const float ay = fmaf(loy, sc.y, of.y), by = fmaf(hiy, sc.y, of.y);
        const float az = fmaf(loz, sc.z, of.z), bz = fmaf(hiz, sc.z, of.z);
        const float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fmaxf(fminf(az, bz), 0.0f));
        const float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fminf(fmaxf(az, bz), hi));
        return tn <= tf * 1.0000004f ? ((__float_as_uint(tn) & ~3u) | slot) : 0xffffffffu;
    }

    template <bool ALL, bool COOP> __device__ __forceinline__ bool step(const SceneAccess<ALL>& S, bool active) {
        const PathSceneD& g = *S.g;
        const int kWalkSteps = S.walk_steps;
        const uint4* __restrict__ nodes = g.bvh4_nodes;
        const bool spec = (S.bvh_spec & 1) != 0;
#pragma unroll 1
        for (int it = 0; it < kWalkSteps; ++it) {
            __syncwarp();
            if (spec && active && pend == 0u && cur >= kBvhLeaf && cur != kBvhDone) { // speculative traversal, see BvhWalk
                pend = cur;
                pop(S.stack);
            }
            if (active && cur < kBvhLeaf) {
                const uint4* __restrict__ np = nodes + 4 * (size_t)cur;
                const uint4 bx = __ldg(np), by = __ldg(np + 1), bz = __ldg(np + 2), rf = __ldg(np + 3);
                const float hi = best * 1.000002f + 1.0e-6f;
                if (COUNT) n_node += 2u + (rf.z != kBvhDone ? 1u : 0u) + (rf.w != kBvhDone ? 1u : 0u);
                // (slots 0 and 1 are always filled; an empty slot 2 / 3 carries the reference kBvhDone)
                uint32_t k0 = child_key(q_lo(bx.x), q_lo(bx.z), q_lo(by.x), q_lo(by.z), q_lo(bz.x), q_lo(bz.z), hi, 0u);
                uint32_t k1 = child_key(q_hi(bx.x), q_hi(bx.z), q_hi(by.x), q_hi(by.z), q_hi(bz.x), q_hi(bz.z), hi, 1u);
                uint32_t k2 = rf.z != kBvhDone ? child_key(q_lo(bx.y), q_lo(bx.w), q_lo(by.y), q_lo(by.w), q_lo(bz.y), q_lo(bz.w), hi, 2u) : 0xffffffffu;
                uint32_t k3 = rf.w != kBvhDone ? child_key(q_hi(bx.y), q_hi(bx.w), q_hi(by.y), q_hi(by.w), q_hi(bz.y), q_hi(bz.w), hi, 3u) : 0xffffffffu;
                // ascending order (misses last): five compare-exchanges
                uint32_t t;
                t = min(k0, k1); k1 = max(k0, k1); k0 = t;
                t = min(k2, k3); k3 = max(k2, k3); k2 = t;
                t = min(k0, k2); k2 = max(k0, k2); k0 = t;
                t = min(k1, k3); k3 = max(k1, k3); k1 = t;
                t = min(k1, k2); k2 = max(k1, k2); k1 = t;
                auto ref_of = [&](uint32_t key) {
                    const uint32_t sl = key & 3u;
                    return sl == 0u ? rf.x : (sl == 1u ? rf.y : (sl == 2u ? rf.z : rf.w));
                };
                // The hits are k0 .. k(n-1). Enter k0, postpone the others farthest first. Written without branches for
                // the common case (the capture of the branchy form ran these lines at 4-7 of 32 lanes, 15 % of the kernel's
                // instructions): three unconditional stores above the stack pointer -- what lies above it is never read.
                const int n = int(k0 != 0xffffffffu) + int(k1 != 0xffffffffu) + int(k2 != 0xffffffffu) + int(k3 != 0xffffffffu);
                const uint32_t e1 = ref_of(k1), e2 = ref_of(k2), e3 = ref_of(k3);
                if (S.bvh_spec & 2) { // A/B knob: the branchy form
                    if (n == 4) push(S.stack, e3);
                    if (n >= 3) push(S.stack, e2);
                    if (n >= 2) push(S.stack, e1);
                    if (n > 0) cur = ref_of(k0);
                    else pop(S.stack);
                    continue;
                }
                if (sp + 3 <= cap) {
                    uint32_t* __restrict__ at = S.stack + sp * kThreads;
                    at[0] = n == 4 ? e3 : (n == 3 ? e2 : e1);
                    at[kThreads] = n == 4 ? e2 : e1;
                    at[2 * kThreads] = e1;
                    sp += max(n - 1, 0);
                } else { // deep in the stack: the general form (entries beyond the shared-memory levels live in local memory)
                    if (n == 4) push(S.stack, e3);
                    if (n >= 3) push(S.stack, e2);
                    if (n >= 2) push(S.stack, e1);
                }
                if (n > 0) {
                    cur = ref_of(k0);
                } else if (sp <= cap) { // pop from the shared-memory levels: one predicated load
                    const int at = max(sp - 1, 0);
                    const uint32_t top = S.stack[at * kThreads];
                    cur = sp > 0 ? top : kBvhDone;
                    sp = at;
                } else {
                    pop(S.stack);
                }
            }
        }
        __syncwarp();
        if (active && pend == 0u && cur >= kBvhLeaf && cur != kBvhDone) {
            pend = cur;
            pop(S.stack);
        }
        if (active && pend != 0u) {
            const uint32_t first = pend & 0x0fffffffu, cnt = ((pend >> 28) & 7u) + 1u;
            pend = 0u;
            if (COUNT) n_prim += cnt;
            const float4* __restrict__ pp = g.bvh_prims + 4 * (size_t)first;
#pragma unroll 1
            for (uint32_t k = 0; k < cnt; ++k, pp += 4) {
                const float4 a0 = __ldg(pp), b0 = __ldg(pp + 1), c0 = __ldg(pp + 2), g0 = __ldg(pp + 3);
                const float t = hit_prim(a0, b0, c0, g0, o, d, best);
                if (t >= 0.0f) { best = t; best_prim = __float_as_uint(g0.w); }
            }
            if (any && best_prim != kInvalid) cur = kBvhDone;
        }
        __syncwarp();
        return active && cur == kBvhDone;
    }
};

template <int WALK> struct WalkOf;
template <> struct WalkOf<1> { using type = TreeWalk2<false>; };
template <> struct WalkOf<2> { using type = TreeWalk2<true>; };
template <> struct WalkOf<3> { using type = BvhWalk; };
template <> struct WalkOf<5> { using type = Bvh4Walk<false>; };
template <> struct WalkOf<6> { using type = Bvh4Walk<true>; };
template <typename W> __device__ __forceinline__ void walk_counts(const W&, unsigned&, unsigned&) {}
template <> __device__ __forceinline__ void walk_counts(const TreeWalk2<true>& w, unsigned& nodes, unsigned& prims) {
    nodes += w.n_node;
    prims += w.n_prim;
}
template <> __device__ __forceinline__ void walk_counts(const Bvh4Walk<true>& w, unsigned& nodes, unsigned& prims) {
    nodes += w.n_node;
    prims += w.n_prim;
}
// tallies of finished rays -> totals[7] (node records visited), totals[8] (primitive tests)
__device__ __forceinline__ void flush_walk_counts(const PassArgs& a, unsigned nodes, unsigned prims) {
    nodes = warp_sum_u(nodes);
    prims = warp_sum_u(prims);
    if ((threadIdx.x & 31u) == 0u && (nodes | prims)) {
        atomicAdd(a.totals + 7, (unsigned long long)nodes);
        atomicAdd(a.totals + 8, (unsigned long long)prims);
    }
}

// Runs the walks of a whole warp to completion; MUST be called by all 32 lanes (`active` = this
// lane has a ray). Used for camera rays; secondary rays go through trace_kernel.
template <bool ALL, bool COOP, int WALK>
__device__ bool traverse(const SceneAccess<ALL>& S, bool active, float3 o, float3 d, float tmax, bool any, float& t_hit,
                         uint32_t& prim_hit, unsigned* n_node = nullptr, unsigned* n_prim = nullptr) {
    typename WalkOf<WALK>::type w = {};
    w.best_prim = kInvalid;
    bool busy = active && !w.init(S, o, d, tmax, any);
    const bool walked = busy;
    while (__any_sync(kFull, busy))
        if (w.template step<ALL, COOP>(S, busy)) busy = false;
    t_hit = w.best;
    prim_hit = w.best_prim;
    if ((WALK == 2 || WALK == 6) && walked && n_node) walk_counts(w, *n_node, *n_prim);
    return active && w.best_prim != kInvalid;
}

// ---- per-slot helpers ------------------------------------------------------------
// n / d without the 32-bit integer-division sequence: float estimate + one exact correction.
__device__ __forceinline__ uint32_t fast_div(uint32_t n, uint32_t d, uint32_t& rem) {
    uint32_t q = (uint32_t)__fdividef(__uint2float_rz(n), __uint2float_rn(d));
    int32_t r = (int32_t)(n - q * d);
    if (r < 0) { --q; r += (int32_t)d; }
    else if ((uint32_t)r >= d) { ++q; r -= (int32_t)d; }
    rem = (uint32_t)r;
    return q;
}

// LIST (adaptive passes): the window runs over a compacted list of local tiles (PassArgs::tiles)
template <bool LIST = false>
__device__ __forceinline__ bool slot_pixel(const PassArgs& a, uint32_t slot, int& x, int& y, uint32_t& sample) {
    uint32_t lp, tx;
    uint32_t s = fast_div(slot, a.pix_count, lp); // slot = sample in pass * window size + pixel in window
    lp += a.pix_base;
    if (LIST) lp = (a.tiles[lp >> 10] << 10) | (lp & 1023u);
    sample = (uint32_t)a.sample_base + s;
    uint32_t lt = lp >> 10, in = lp & 1023u;
    uint32_t t = lt * (uint32_t)a.map.world + (uint32_t)a.map.rank;
    uint32_t ty = fast_div(t, (uint32_t)a.map.tiles_x, tx);
    x = int(tx * kTile + (in & 31u));
    y = int(ty * kTile + (in >> 5));
    return x < a.map.w && y < a.map.h;
}

// The reference pinhole (raytracer.h:26-30,41) with a uniform jitter inside the pixel.
__device__ __forceinline__ void camera_ray(const PassArgs& a, int x, int y, uint32_t pixel, uint32_t sample, float3& o,
                                           float3& d) {
    uint4 r = philox(pixel, sample, 0u, 0u, a.seed);
    float fx = (float(x) + u01(r.x)) * 0.0002f, fy = (float(y) + u01(r.y)) * 0.0002f;
    const PathCamera& c = a.cam;
    o = f3(c.pos[0], c.pos[1], c.pos[2]);
    float3 v = f3(c.top_left[0] - c.left[0] * fx - c.up[0] * fy, c.top_left[1] - c.left[1] * fx - c.up[1] * fy,
                  c.top_left[2] - c.left[2] * fx - c.up[2] * fy);
    d = normalize(v);
}

// Warp-ballot compaction into a queue whose space the warp reserves in private chunks of
// kChunk entries: one atomic per kChunk outputs, no block barrier. Must be called by all
// 32 lanes of a converged warp.
struct WarpCursor {
    uint32_t pos, end; // warp-uniform
    uint32_t next;     // lane 0: base of the chunk reserved ahead of time (warp_reserve)
    bool has_next;     // warp-uniform
};

__device__ __forceinline__ void warp_append(WarpCursor& c, bool want, uint32_t value, uint32_t* __restrict__ queue,
                                            uint32_t* __restrict__ counter) {
    const uint32_t m = __ballot_sync(kFull, want);
    if (m == 0) return;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t n = __popc(m), rank = __popc(m & ((1u << lane) - 1u));
    const uint32_t room = c.end - c.pos, base0 = c.pos;
    uint32_t base1 = 0;
    if (n > room) { // the tail goes to a fresh chunk
        if (lane == 0) base1 = atomicAdd(counter, kChunk);
        base1 = __shfl_sync(kFull, base1, 0);
        c.pos = base1 + (n - room);
        c.end = base1 + kChunk;
    } else {
        c.pos += n;
    }
    if (want) queue[rank < room ? base0 + rank : base1 + (rank - room)] = value;
}

// Same reservation, for records wider than a queue entry: returns the lane's position (kInvalid
// for lanes that do not want one); the caller writes the record.
// The chunk a warp will need NEXT is reserved ahead of time, as soon as an append could overflow
// the current one (room < 32): ncu attributed 5.5 % of the bounce kernel's stall samples to the 16
// instructions around this atomic -- its round trip to L2 was exposed once per 64 records. Now the
// atomic is in flight during the ~800 instructions of the next vertex and its result is only read
// at the next overflow. A warp that appends sparsely never gets close to the end of its chunk and
// prefetches nothing; a dense producer leaves at most one unused chunk behind (warp_flush pads it).
template <bool AHEAD = true, uint32_t CHUNK = kChunk>
__device__ __forceinline__ uint32_t warp_reserve(WarpCursor& c, bool want, uint32_t* __restrict__ counter) {
    static_assert(CHUNK >= 32u, "one append of a full warp must fit a fresh chunk");
    const uint32_t m = __ballot_sync(kFull, want);
    if (m == 0) return kInvalid;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t n = __popc(m), rank = __popc(m & ((1u << lane) - 1u));
    const uint32_t room = c.end - c.pos, base0 = c.pos;
    uint32_t base1 = 0;
    if (n > room) {
        if (!c.has_next && lane == 0) c.next = atomicAdd(counter, CHUNK); // first chunk, or a sparse producer
        base1 = __shfl_sync(kFull, c.next, 0);
        c.has_next = false;
        c.pos = base1 + (n - room);
        c.end = base1 + CHUNK;
    } else {
        c.pos += n;
    }
    if (AHEAD && !c.has_next && c.end - c.pos < 32u) { // the next append may overflow: fetch its chunk now
        if (lane == 0) c.next = atomicAdd(counter, CHUNK);
        c.has_next = true;
    }
    return want ? (rank < room ? base0 + rank : base1 + (rank - room)) : kInvalid;
}

// Pad what is left of the warp's last chunk so that consumers can skip it.
__device__ __forceinline__ void warp_flush(const WarpCursor& c, uint32_t* __restrict__ queue) {
    for (uint32_t i = c.pos + (threadIdx.x & 31u); i < c.end; i += 32u) queue[i] = kInvalid;
    if (c.has_next) { // a chunk reserved ahead of time and never used
        const uint32_t base = __shfl_sync(kFull, c.next, 0);
        for (uint32_t i = threadIdx.x & 31u; i < kChunk; i += 32u) queue[base + i] = kInvalid;
    }
}

__device__ __forceinline__ unsigned warp_sum(unsigned v) {
    for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(kFull, v, off);
    return v;
}

// A slot's radiance is only ever touched by the one thread that owns the slot in a launch.
__device__ __forceinline__ void add_radiance(const PassArgs& a, uint32_t slot, float3 v) {
    // (measured: RED.ADD.F32 here costs 1.7x the whole shade kernel -- 1.2 G L2 atomics per
    // frame; the plain read-modify-write is exclusive to the slot's thread anyway)
    float* L = a.L;
    const float l0 = L[slot], l1 = L[a.plane + slot], l2 = L[2 * a.plane + slot];
    L[slot] = l0 + v.x;
    L[a.plane + slot] = l1 + v.y;
    L[2 * a.plane + slot] = l2 + v.z;
}

// The three material queues a launch feeds (the next bounce's), one warp-private cursor each.
struct Sorter {
    WarpCursor cur[3];
    uint32_t* q[3];
    uint32_t* counters; // diffuse, mirror, glass are adjacent
    uint32_t mask;      // material classes the scene has
    __device__ __forceinline__ void init(const PassArgs& a, int next_bounce) {
        const int set = (next_bounce & 1) * 3;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            cur[k] = WarpCursor{0, 0, 0, false};
            q[k] = a.q[set + k];
        }
        counters = a.counts + next_bounce * 4 + Q_DIFFUSE;
        mask = a.kind_mask;
    }
    // kind: G19_BSDF_DIFFUSE / MIRROR / GLASS, or -1 for "path ended"
    __device__ __forceinline__ void push(int kind, uint32_t slot) {
        if (mask & 1u) warp_append(cur[0], kind == G19_BSDF_DIFFUSE, slot, q[0], counters + 0);
        if (mask & 2u) warp_append(cur[1], kind == G19_BSDF_MIRROR, slot, q[1], counters + 1);
        if (mask & 4u) warp_append(cur[2], kind == G19_BSDF_GLASS, slot, q[2], counters + 2);
    }
    __device__ __forceinline__ void flush() {
#pragma unroll
        for (int k = 0; k < 3; ++k)
            if (mask & (1u << k)) warp_flush(cur[k], q[k]);
    }
};

// Nearest hit of one ray, flat or tree. Called by all 32 lanes; `active` = the lane has a ray.
template <bool ALL, bool COOP, int WALK>
__device__ __forceinline__ bool nearest(const SceneAccess<ALL>& S, bool active, float3 o, float3 d, float& t, uint32_t& prim,
                                        unsigned* n_node = nullptr, unsigned* n_prim = nullptr) {
    if constexpr (ALL) {
        bool occ;
        trace_flat<false>(S, o, d, active ? FLT_MAX : -1.0f, d, -1.0f, t, prim, occ);
        return prim != kInvalid;
    } else {
        return traverse<ALL, COOP, WALK>(S, active, o, d, FLT_MAX, false, t, prim, n_node, n_prim);
    }
}

// What a new path vertex leaves behind for the next bounce (32 B + 16 B + queue entry).
__device__ __forceinline__ void store_vertex(const PassArgs& a, uint32_t slot, float3 p, uint32_t prim, float3 d,
                                             uint32_t pixel) {
    a.hp[slot] = make_float4(p.x, p.y, p.z, __uint_as_float(prim));
    a.dw[slot] = make_float4(d.x, d.y, d.z, __uint_as_float(pixel));
}

// ---- raygen + extend (camera segment), tree scenes: slot-indexed state ----------------------
// 3 CTAs per SM at 80 registers (68 bytes of spills) beat 2 at 95 on the octree walk: 23.8 vs 26.4 ms per 66 M camera rays
template <bool COOP, int WALK, bool LIST = false> __global__ void __launch_bounds__(kThreads, 3) raygen_extend_kernel(const PassArgs a) {
    pdl_launch_dependents();
    const uint32_t n = a.n_slots;
    if (blockIdx.x * kThreads >= n) return;
    const SceneAccess<false> S = stage_scene<false>(a);
    pdl_wait(); // the previous pass's accumulate cleared the queue lengths and the radiance planes
    Sorter out;
    out.init(a, 0);
    unsigned cnt_node = 0, cnt_prim = 0;
    const uint32_t stride = gridDim.x * kThreads;
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t q = blockIdx.x * kThreads + threadIdx.x; q - lane < n; q += stride) { // warp-uniform trip count
        const uint32_t slot = q;
        int kind = -1;
        bool live = false;
        uint32_t pixel = 0;
        float3 o = f3(0.f, 0.f, 0.f), d = f3(0.f, 0.f, 1.f);
        if (q < n) {
            int x, y;
            uint32_t sample;
            live = slot_pixel<LIST>(a, slot, x, y, sample);
            if (live) {
                pixel = uint32_t(y) * uint32_t(a.map.w) + uint32_t(x);
                camera_ray(a, x, y, pixel, sample, o, d);
            }
        }
        float t;
        uint32_t prim;
        if (nearest<false, COOP, WALK>(S, live, o, d, t, prim, &cnt_node, &cnt_prim)) { // all 32 lanes walk together
            const float4 tag = S.hot_row(prim, 3);
            const int bsdf = __float_as_int(tag.y); // material class rides in the hot record
            if (bsdf == G19_BSDF_EMITTER) {          // directly visible light: the path ends here
                const MaterialD& m = a.scene.materials[__float_as_int(tag.x)];
                add_radiance(a, slot, f3(m.emission[0], m.emission[1], m.emission[2]));
            } else if (bsdf == G19_BSDF_DIFFUSE || a.max_depth > 1) {
                kind = bsdf;
                store_vertex(a, slot, o + d * t, prim, d, pixel);
            }
        }
        out.push(kind, slot);
    }
    out.flush();
    if (WALK == 2 || WALK == 6) flush_walk_counts(a, cnt_node, cnt_prim);
}

// ---- bounce: shade + trace the continuation ray ------------------------------------------
__device__ __forceinline__ void onb(float3 n, float3& t, float3& b) { // Duff et al. 2017
    float s = copysignf(1.0f, n.z);
    float a = -1.0f / (s + n.z);
    float bb = n.x * n.y * a;
    t = f3(1.0f + s * n.x * n.x * a, s * bb, -s * n.x);
    b = f3(bb, s + n.y * n.y * a, -n.y);
}

__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- shading of one path vertex (shared by the flat-scene and the tree-scene bounce kernels) ----
// In: the vertex (hit point p on primitive prim, arrival direction d, throughput T). Out: the
// next-event sample (direction w, length tmax_s, radiance lit_rgb if it turns out unoccluded) and
// the continuation ray (origin no, direction nd, throughput T updated). flags bit 0: specular.
struct Shaded {
    float3 no, nd, w, lit_rgb, T;
    float tmax_s;
    bool want_shadow;
    uint32_t flags;
};
template <int KIND, bool LAST, bool ALL>
__device__ __forceinline__ Shaded shade_vertex(const PassArgs& a, const SceneAccess<ALL>& S, int bounce, float3 p, float3 d,
                                               float3 T, uint32_t prim, uint32_t pixel, uint32_t sample) {
    constexpr bool kDiffuse = KIND == Q_DIFFUSE;
    Shaded o;
    float4 c0, c1; // (normal, ior), (albedo, material)
    S.cold(prim, c0, c1);
    float3 ng = f3(c0.x, c0.y, c0.z);
    if (c0.x == 0.0f && c0.y == 0.0f && c0.z == 0.0f) { // spheres store no normal: (p - centre) / r
        const float4 q0 = S.hot_row(prim, 0);
        ng = (p - f3(q0.x, q0.y, q0.z)) * __fdividef(1.0f, q0.w);
    }
    const float ior = c0.w;
    const bool entering = dot(ng, d) < 0.0f;
    const float3 nf = entering ? ng : -ng; // normal on the side the ray arrives from
    const float3 albedo = f3(c1.x, c1.y, c1.z);
    const uint4 r = philox(pixel, sample, uint32_t(bounce), 1u, a.seed);
    o.nd = f3(0.f, 0.f, 1.f);
    o.flags = 0;
    o.want_shadow = false;
    o.w = f3(0.f, 0.f, 1.f);
    o.lit_rgb = f3(0.f, 0.f, 0.f);
    o.tmax_s = -1.0f;
    if (kDiffuse) {
        // next-event estimation (diffuse only): one light, one uniformly sampled point
        if (a.scene.n_lights > 0) {
            float pick = u01(r.x) * float(a.scene.n_lights);
            int li = min(int(pick), a.scene.n_lights - 1);
            float u1 = pick - float(li), u2 = u01(r.y);
            const float4* lt = S.light(li);
            const float4 l0 = lt[0], l1 = lt[1], l2 = lt[2], l3 = lt[3];
            float su = sqrtf(u1);
            float b1 = su * (1.0f - u2), b2 = su * u2;
            float3 yl = f3(l0.x + l1.x * b1 + l2.x * b2, l0.y + l1.y * b1 + l2.y * b2, l0.z + l1.z * b1 + l2.z * b2);
            float3 w = yl - p;
            float dist2 = dot(w, w);
            float inv_dist = rsqrtf(dist2);
            float dist = dist2 * inv_dist;
            w = w * inv_dist;
            o.w = w;
            float cs = dot(nf, w);
            float cl = fabsf(dot(f3(l3.x, l3.y, l3.z), w));
            if (cs > 0.0f && cl > 0.0f && dist > 2.0f * kRayEps) {
                o.want_shadow = true;
                o.tmax_s = dist - 2.0f * kRayEps;
                const float4 l4 = lt[4];
                float gterm = cs * cl * l0.w * __fdividef(1.0f, dist2 * l1.w) * (1.0f / kPi);
                o.lit_rgb = f3(T.x * albedo.x * l4.x * gterm, T.y * albedo.y * l4.y * gterm, T.z * albedo.z * l4.z * gterm);
            }
        }
        o.no = p + nf * kRayEps;
        if (!LAST) { // cosine-weighted bounce: pdf cancels cos/pi, throughput *= albedo
            float u3 = u01(r.z), u4 = u01(r.w);
            float rr = sqrtf(u3), phi = 2.0f * kPi * u4 - kPi; // [-pi, pi): MUFU range
            float sp, cp;
            __sincosf(phi, &sp, &cp);
            sp = -sp; cp = -cp; // shift back by pi
            float3 tx, ty;
            onb(nf, tx, ty);
            o.nd = normalize(tx * (rr * cp) + ty * (rr * sp) + nf * sqrtf(fmaxf(0.0f, 1.0f - u3)));
        }
        o.T = T * albedo;
    } else if (KIND == Q_MIRROR) {
        o.nd = normalize(d - nf * (2.0f * dot(d, nf)));
        o.no = p + nf * kRayEps;
        o.T = T * albedo;
        o.flags = 1u;
    } else { // dielectric
        float etai = entering ? 1.0f : ior, etat = entering ? ior : 1.0f;
        float eta = etai / etat;
        float cosi = fminf(1.0f, -dot(d, nf));
        float sin2t = eta * eta * fmaxf(0.0f, 1.0f - cosi * cosi);
        float F = 1.0f;
        float cost = 0.0f;
        if (sin2t < 1.0f) {
            cost = sqrtf(1.0f - sin2t);
            float rs = (etai * cosi - etat * cost) / (etai * cosi + etat * cost);
            float rp = (etai * cost - etat * cosi) / (etai * cost + etat * cosi);
            F = 0.5f * (rs * rs + rp * rp);
        }
        if (u01(r.x) < F) {
            o.nd = normalize(d + nf * (2.0f * cosi));
            o.no = p + nf * kRayEps;
        } else {
            o.nd = normalize(d * eta + nf * (eta * cosi - cost));
            o.no = p - nf * kRayEps;
        }
        o.T = T * albedo;
        o.flags = 1u;
    }
    return o;
}

// ---- flat scenes: dense vertex records --------------------------------------------------
// What the ncu capture of the slot-indexed state showed (profiles/r01c_ncu_pass_summary.json): the four
// diffuse bounce launches of a Cornell pass execute 100 / 93 / 83 / 73 M warp instructions but all
// take ~128 us -- as paths end, the survivors' slots thin out, every 16-byte state record still
// costs a 32-byte sector (global load sectors per launch stay at 8 M), DRAM channel load becomes
// uneven and long-scoreboard stalls grow 0.55 -> 1.97 per issue. So the QUEUES now hold the records
// themselves: a vertex is written at the position its warp reserved in the next bounce's material
// queue (slot, hit point + primitive, direction + pixel, throughput + sample, radiance so far --
// 64 bytes, all planes coalesced) and read back from consecutive addresses; the path's radiance
// travels with it and is stored to the slot's accumulator input exactly once, when the path ends.
// A bounce holds at most P vertices over its three material queues together, so the queues of a bounce parity share
// storage instead of being P entries each (VERDICT r01: 16 GB reserved for a 14-primitive scene): the diffuse queue has
// an array of its own (P + slack entries), mirror and glass share ONE array of P + 2 x slack entries -- mirror grows
// from its bottom, glass from its top downwards (entry q of the glass queue lives at top - q: consecutive lanes still
// touch consecutive 16-byte words). A diffuse-only scene allocates no specular array at all.
struct RecView { // one queue: four float4 planes; entry q is at plane[q * dir]
    float4 *ls, *hp, *dw, *tp; // (radiance so far | slot) (hit point | primitive) (direction | pixel) (throughput | sample)
    int dir;
    __device__ __forceinline__ ptrdiff_t at(uint32_t q) const { return dir > 0 ? ptrdiff_t(q) : -ptrdiff_t(q); }
};
__device__ __forceinline__ RecView rec_queue(const PassArgs& a, int qi) { // qi = bounce parity * 3 + (kind - 1)
    RecView r;
    const int parity = qi >= 3 ? 1 : 0, kind = qi - 3 * parity;
    size_t off = size_t(parity) * (a.queue_cap + a.spec_cap);
    r.dir = 1;
    if (kind != 0) {
        off += a.queue_cap;                                      // the shared specular array of this parity
        if (kind == 2) { off += a.spec_cap - 1; r.dir = -1; }   // glass: from the top, downwards
    }
    r.ls = a.rec_ls + off;
    r.hp = a.rec_hp + off;
    r.dw = a.rec_dw + off;
    r.tp = a.rec_tp + off;
    return r;
}

// The record queues a launch feeds (the next bounce's). SPEC = the scene has mirror or glass
// materials; a diffuse-only scene keeps one cursor (registers: the three-cursor form spilled).
template <bool SPEC> struct RecSorter {
    WarpCursor cur[SPEC ? 3 : 1];
    uint32_t* counters;
    uint32_t mask;
    int set;
    __device__ __forceinline__ void init(const PassArgs& a, int next_bounce) {
#pragma unroll
        for (int k = 0; k < (SPEC ? 3 : 1); ++k) cur[k] = WarpCursor{0, 0, 0, false};
        set = (next_bounce & 1) * 3;
        counters = a.counts + next_bounce * 4 + Q_DIFFUSE;
        mask = SPEC ? a.kind_mask : 1u;
    }
    // kind: G19_BSDF_DIFFUSE / MIRROR / GLASS, or -1 for "path ended". Returns the lane's position in
    // its kind's queue (kInvalid for ended paths). Called by all 32 lanes.
    __device__ __forceinline__ uint32_t reserve(int kind) {
        if (!SPEC) return warp_reserve(cur[0], kind == 0, counters);
        uint32_t pos = kInvalid;
#pragma unroll
        for (int k = 0; k < (SPEC ? 3 : 1); ++k)
            if (mask & (1u << k)) {
                // the specular queues fill slowly (a few entries per warp and launch): no chunk ahead of
                // time and 32-entry chunks, or their consumers would run on mostly padding
                const uint32_t p = k == 0 ? warp_reserve<true>(cur[k], kind == k, counters + k)
                                          : warp_reserve<false, 32u>(cur[k], kind == k, counters + k);
                if (kind == k) pos = p;
            }
        return pos;
    }
    // pad what is left of the warp's chunks: an entry whose slot word is kInvalid is skipped by the consumer
    __device__ __forceinline__ void flush(const PassArgs& a) {
        const uint32_t lane = threadIdx.x & 31u;
        const float4 pad = make_float4(0.f, 0.f, 0.f, __uint_as_float(kInvalid));
#pragma unroll
        for (int k = 0; k < (SPEC ? 3 : 1); ++k)
            if (mask & (1u << k)) {
                const RecView r = rec_queue(a, set + k);
                const WarpCursor& c = cur[k];
                for (uint32_t i = c.pos + lane; i < c.end; i += 32u) r.ls[r.at(i)] = pad;
                if (c.has_next) { // a chunk reserved ahead of time and never used
                    const uint32_t base = __shfl_sync(kFull, c.next, 0);
                    for (uint32_t i = lane; i < kChunk; i += 32u) r.ls[r.at(base + i)] = pad;
                }
            }
    }
};

// Asynchronous prefetch of the NEXT record into shared memory (LDGSTS): a register prefetch gets
// sunk to its first use by the compiler (ncu: 20 % of the kernel's stall samples sat on that one
// instruction); a cp.async cannot be, and it holds no registers while in flight. Two buffers per
// thread, each thread only ever touches its own column. The records are dense, so the address of
// the next one is known without loading anything first.
template <bool FULL> struct RecStage {
    float4 ls[2][kThreads]; // radiance so far, slot
    float4 hp[2][kThreads];
    float4 dw[2][kThreads];
    float4 tp[FULL ? 2 : 1][FULL ? kThreads : 1];
};
template <bool FULL>
__device__ __forceinline__ void prefetch_rec(const RecView& r, uint32_t pos, bool valid, RecStage<FULL>& st, int buf) {
    const int t = threadIdx.x;
    if (valid) {
        const ptrdiff_t at = r.at(pos);
        cp_async16(&st.ls[buf][t], r.ls + at);
        cp_async16(&st.hp[buf][t], r.hp + at);
        cp_async16(&st.dw[buf][t], r.dw + at);
        if (FULL) cp_async16(&st.tp[buf][t], r.tp + at);
    }
    cp_async_commit();
}

// One material queue of one bounce: next-event estimation, BSDF sample, the trace of BOTH rays in one loop over the
// staged primitives, and the new vertex record written straight into the next bounce's material queue.
// KIND: Q_DIFFUSE / Q_MIRROR / Q_GLASS. FIRST: the queue holds the 48-byte records of camera hits. SPEC: the scene has
// mirror / glass queues to feed.
// FUSED (the first bounce): the camera segment of each path slot of the pass is traced right here, so the vertex record
// of a diffuse camera hit (48 B written, 48 B read back, a fifth of the frame's HBM traffic), its queue reservation and
// a camera launch per pass do not exist; `n` is then the number of path slots of the pass. LAST (FUSED at max_depth 1):
// the camera segment ended at the path's last vertex -- next-event estimation only, no continuation.
// FOLD (the bounce before the last): the vertex the continuation ray finds would be the path's
// last one -- next-event estimation only. It is shaded right here (light sample + shadow ray) instead of being written as a
// 64-byte record for a launch of its own to read back: same arithmetic in the same order, one launch per pass fewer.
template <int KIND, bool FIRST, bool LAST, bool SPEC, bool FUSED, bool FOLD, bool UNI, bool LIST = false>
__device__ __forceinline__ void bounce_flat_body(const PassArgs& a, const int bounce, const SceneAccess<true>& S, const uint32_t n,
                                                 const uint32_t cta, const uint32_t n_cta, RecStage<!FIRST>& stage) {
    constexpr bool kDiffuse = KIND == Q_DIFFUSE;
    const RecView in = rec_queue(a, (bounce & 1) * 3 + (KIND - 1));
    RecSorter<SPEC> out;
    if (!LAST && !FOLD) out.init(a, bounce + 1);
    // statistics (g19_stats), two 16-bit counters per register (a thread runs < 2^16 iterations: the grid
    // has > 10^5 threads and a queue < 2^32 entries): calls | traced << 16, shadow rays | lit << 16
    uint32_t cnt_a = 0, cnt_b = 0, stored = 0, folded = 0;
    const uint32_t stride = n_cta * kThreads;
    const uint32_t lane = threadIdx.x & 31u;
    const int tid = threadIdx.x;
    const bool next_last = bounce + 2 >= a.max_depth;

    uint32_t q = cta * kThreads + threadIdx.x;
    int buf = 0;
    if (!FUSED) prefetch_rec(in, q, q < n, stage, 0);
    for (; q - lane < n; q += stride) {
        uint32_t slot = kInvalid;
        float4 ls = make_float4(0.f, 0.f, 0.f, 0.f);
        float3 p = f3(0.f, 0.f, 0.f), d = f3(0.f, 0.f, 1.f);
        uint32_t prim = kInvalid, pixel = 0, sample = 0;
        if (FUSED) {
            // ---- the camera segment of path slot q ----
            bool live = false;
            float3 o = f3(0.f, 0.f, 0.f);
            if (q < n) {
                int x, y;
                live = slot_pixel<LIST>(a, q, x, y, sample);
                if (live) {
                    pixel = uint32_t(y) * uint32_t(a.map.w) + uint32_t(x);
                    camera_ray(a, x, y, pixel, sample, o, d);
                }
            }
            float t = 0.0f;
            uint32_t pr = kInvalid;
            int spec_kind = -1; // SPEC: the camera ray met a mirror / glass surface: that vertex goes to its material's queue
            float4 seen = make_float4(0.f, 0.f, 0.f, 0.f); // what a path that ends on the camera segment delivers
            bool unused_occ;
            trace_flat<false, UNI>(S, o, d, live ? FLT_MAX : -1.0f, d, -1.0f, t, pr, unused_occ); // = nearest's flat form
            if (pr != kInvalid) {
                const float4 tag = S.hot_row(pr, 3);
                const int bsdf = __float_as_int(tag.y);
                if (bsdf == G19_BSDF_EMITTER) { // directly visible light: the path ends here
                    const MaterialD& m = a.scene.materials[__float_as_int(tag.x)];
                    seen = make_float4(m.emission[0], m.emission[1], m.emission[2], 0.0f);
                } else if (bsdf == G19_BSDF_DIFFUSE) {
                    slot = q;
                    prim = pr;
                    p = o + d * t;
                } else if (SPEC && a.max_depth > 1) {
                    spec_kind = bsdf;
                }
            }
            if (q < n && slot == kInvalid && spec_kind < 0) reinterpret_cast<float4*>(a.L)[q] = seen; // miss, emitter, or a slot outside the frame
            if (SPEC) {
                // The few camera hits on mirror / glass (the two spheres of the glass Cornell box: a tenth of the pixels) keep
                // the material queues: their 48-byte camera records go to bounce 0's queue of their kind, reserved with one
                // atomic per warp and kind -- no cursor state carried through the loop -- for the launch that follows this one.
#pragma unroll
                for (int k = G19_BSDF_MIRROR; k <= G19_BSDF_GLASS; ++k) {
                    const uint32_t m = __ballot_sync(kFull, spec_kind == k);
                    if (m == 0u) continue;
                    uint32_t base = 0;
                    if (lane == uint32_t(__ffs(int(m)) - 1)) base = atomicAdd(a.counts + Q_DIFFUSE + k, uint32_t(__popc(m)));
                    base = __shfl_sync(kFull, base, __ffs(int(m)) - 1);
                    if (spec_kind == k) {
                        const RecView r = rec_queue(a, k); // bounce 0, parity 0
                        const ptrdiff_t at = r.at(base + uint32_t(__popc(m & ((1u << lane) - 1u))));
                        const float3 ph = o + d * t;
                        r.ls[at] = make_float4(__uint_as_float(sample), 0.f, 0.f, __uint_as_float(q));
                        r.hp[at] = make_float4(ph.x, ph.y, ph.z, __uint_as_float(pr));
                        r.dw[at] = make_float4(d.x, d.y, d.z, __uint_as_float(pixel));
                    }
                }
            }
        } else {
            const uint32_t qn = q + stride;
            prefetch_rec(in, qn, qn < n && qn > q, stage, buf ^ 1); // next record, in flight during this body
            cp_async_wait<1>();                                     // this record has landed
            ls = stage.ls[buf][tid];
            slot = q < n ? __float_as_uint(ls.w) : kInvalid;
        }
        int kind_next = -1;
        float3 p_next = f3(0.f, 0.f, 0.f), d_next = f3(0.f, 0.f, 1.f), T = f3(1.f, 1.f, 1.f), Lp = f3(0.f, 0.f, 0.f);
        uint32_t prim_next = kInvalid;
        if (slot != kInvalid) {
            if (!FUSED) {
                const float4 hp = stage.hp[buf][tid], dw = stage.dw[buf][tid];
                p = f3(hp.x, hp.y, hp.z);
                d = f3(dw.x, dw.y, dw.z);
                prim = __float_as_uint(hp.w);
                pixel = __float_as_uint(dw.w);
            }
            if (FUSED) {
                // throughput 1, no radiance yet: nothing to load
            } else if (FIRST) {
                sample = __float_as_uint(ls.x); // the camera record: no radiance yet, x carries the sample index
            } else {
                const float4 tp = stage.tp[buf][tid];
                T = f3(tp.x, tp.y, tp.z);
                sample = __float_as_uint(tp.w);
                Lp = f3(ls.x, ls.y, ls.z);
            }
            const Shaded sh = shade_vertex<KIND, LAST, true>(a, S, bounce, p, d, T, prim, pixel, sample);
            T = sh.T;
            const bool cont = !LAST && (T.x > 0.0f || T.y > 0.0f || T.z > 0.0f);
            cnt_a += 1u + (cont ? 0x10000u : 0u);
            // ---- the rays of this vertex: shadow (any hit) and continuation (nearest hit) ----
            bool blocked = false;
            float t_hit = FLT_MAX;
            uint32_t prim_hit = kInvalid;
            if (kDiffuse && !LAST) {
                if (sh.want_shadow || cont)
                    trace_flat<true, UNI>(S, sh.no, sh.nd, cont ? FLT_MAX : -1.0f, sh.w, sh.tmax_s, t_hit, prim_hit, blocked);
            } else if (kDiffuse) { // LAST: the shadow ray alone
                if (sh.want_shadow) {
                    bool unused;
                    trace_flat<false, UNI>(S, sh.no, sh.w, sh.tmax_s, sh.w, -1.0f, t_hit, prim_hit, unused);
                    blocked = prim_hit != kInvalid;
                }
            } else if (cont) {
                bool unused;
                trace_flat<false, UNI>(S, sh.no, sh.nd, FLT_MAX, sh.nd, -1.0f, t_hit, prim_hit, unused);
            }
            const bool hit = cont && prim_hit != kInvalid;
            const bool lit = kDiffuse && sh.want_shadow && !blocked;
            if (kDiffuse) cnt_b += (sh.want_shadow ? 1u : 0u) + (lit ? 0x10000u : 0u);
            if (lit) Lp = Lp + sh.lit_rgb;
            if (hit) {
                const float4 tag = S.hot_row(prim_hit, 3);
                const int bsdf = __float_as_int(tag.y);
                if (bsdf == G19_BSDF_EMITTER) {
                    // emission counts after specular bounces only (NEE covers the diffuse ones)
                    if (sh.flags & 1u) {
                        const MaterialD& m = a.scene.materials[__float_as_int(tag.x)];
                        Lp = Lp + f3(T.x * m.emission[0], T.y * m.emission[1], T.z * m.emission[2]);
                    }
                } else if (bsdf == G19_BSDF_DIFFUSE || !next_last) { // a specular vertex on the last segment adds nothing
                    kind_next = bsdf;
                    p_next = sh.no + sh.nd * t_hit;
                    d_next = sh.nd;
                    prim_next = prim_hit;
                }
            }
            if (FOLD && kind_next == G19_BSDF_DIFFUSE) { // the path's last vertex, shaded in place (next_last holds for this launch)
                const Shaded s2 = shade_vertex<Q_DIFFUSE, true, true>(a, S, bounce + 1, p_next, d_next, T, prim_next, pixel, sample);
                cnt_a += 1u;
                ++folded;
                if (s2.want_shadow) {
                    bool unused;
                    float t2;
                    uint32_t k2;
                    trace_flat<false, UNI>(S, s2.no, s2.w, s2.tmax_s, s2.w, -1.0f, t2, k2, unused);
                    const bool lit2 = k2 == kInvalid;
                    cnt_b += 1u + (lit2 ? 0x10000u : 0u);
                    if (lit2) Lp = Lp + s2.lit_rgb;
                }
                kind_next = -1;
            }
            if (kind_next < 0) {
                // the path ends here: its radiance goes to the slot's accumulator input, once (zero or not:
                // accumulate does not clear what it read)
                ++stored;
                // (slots are scattered by now: ONE 16-byte store, not three 4-byte stores into three planes --
                // the last bounce of the depth-12 glass box spent 148 us on 37 M instructions doing those)
                reinterpret_cast<float4*>(a.L)[slot] = make_float4(Lp.x, Lp.y, Lp.z, 0.0f);
            }
        }
        if (!LAST && !FOLD) {
            const uint32_t pos = out.reserve(kind_next);
            if (pos != kInvalid) {
                const RecView r = rec_queue(a, out.set + kind_next);
                const ptrdiff_t at = r.at(pos);
                r.ls[at] = make_float4(Lp.x, Lp.y, Lp.z, __uint_as_float(slot));
                r.hp[at] = make_float4(p_next.x, p_next.y, p_next.z, __uint_as_float(prim_next));
                r.dw[at] = make_float4(d_next.x, d_next.y, d_next.z, __uint_as_float(pixel));
                r.tp[at] = make_float4(T.x, T.y, T.z, __uint_as_float(sample));
            }
        }
        buf ^= 1;
    }
    cp_async_wait<0>();
    if (!LAST && !FOLD) out.flush(a);
    const unsigned calls = warp_sum(cnt_a & 0xffffu), traced = warp_sum(cnt_a >> 16);
    const unsigned shadow_rays = warp_sum(cnt_b & 0xffffu), lit = warp_sum(cnt_b >> 16);
    stored = warp_sum(stored);
    if (lane == 0 && calls) {
        atomicAdd(a.totals + 2, (unsigned long long)calls);
        if (FIRST) atomicAdd(a.totals + 3, (unsigned long long)calls);
        if (traced) atomicAdd(a.totals + 0, (unsigned long long)traced);
        if (shadow_rays) atomicAdd(a.totals + 1, (unsigned long long)shadow_rays);
        if (lit) atomicAdd(a.totals + 4, (unsigned long long)lit);
        if (stored) atomicAdd(a.totals + 6, (unsigned long long)stored);
    }
    if (FOLD) {
        folded = warp_sum(folded);
        if (lane == 0 && folded) atomicAdd(a.totals + 9, (unsigned long long)folded);
    }
}

// A bounce after the first of a diffuse-only scene: its one material queue.
template <bool FOLD, bool UNI>
__global__ void __launch_bounds__(kThreads, 3) bounce_flat_kernel(const PassArgs a, const int bounce, const __grid_constant__ FlatPairsU up) {
    pdl_launch_dependents();
    SceneAccess<true> S = stage_scene<true>(a); // does not depend on earlier kernels: overlaps their tail
    S.upairs = &up;
    pdl_wait();
    const uint32_t n = a.counts[bounce * 4 + Q_DIFFUSE];
    if (blockIdx.x * kThreads >= n) return; // short queue: surplus CTAs leave
    __shared__ RecStage<true> stage;
    bounce_flat_body<Q_DIFFUSE, false, false, false, false, FOLD, UNI>(a, bounce, S, n, blockIdx.x, gridDim.x, stage);
}

// The first bounce: camera segment + first vertex in one launch (bounce_flat_body<FUSED>), over the path slots of the pass
// instead of a queue. LIST: an adaptive pass (slot_pixel).
template <bool LAST, bool FOLD, bool SPEC, bool UNI, bool LIST = false>
__global__ void __launch_bounds__(kThreads, 3) bounce_flat_fused_kernel(const PassArgs a, const __grid_constant__ FlatPairsU up) {
    pdl_launch_dependents();
    const uint32_t n = a.n_slots;
    if (blockIdx.x * kThreads >= n) return;
    SceneAccess<true> S = stage_scene<true>(a);
    S.upairs = &up;
    pdl_wait(); // the previous pass's accumulate cleared the queue lengths
    RecStage<false>& unused = *reinterpret_cast<RecStage<false>*>(g19_dyn_smem); // (the fused body prefetches no records)
    bounce_flat_body<Q_DIFFUSE, true, LAST, SPEC, true, FOLD, UNI, LIST>(a, 0, S, n, blockIdx.x, gridDim.x, unused);
}

// All three material queues of one bounce in ONE launch (scenes with mirror / glass). The mirror and
// glass queues of a Cornell box hold a few per cent of the vertices: as launches of their own they
// ran 1-2 records per thread at 50-60 % issue utilisation with nothing to overlap their latency
// (ncu, profiles/r01c: 25 + 35 us next to the diffuse launch's 216 us, 21 of 34 launches per pass).
// Here the grid's CTAs are split between the queues in proportion to their estimated work, so the
// specular vertices fill issue slots beside the diffuse ones and a pass is 13 launches, not 34.
// The per-material queues and kernels' code are unchanged: a CTA runs exactly one KIND.
template <bool FIRST, bool FOLD, bool UNI>
__global__ void __launch_bounds__(kThreads, 3) bounce_flat_all_kernel(const PassArgs a, const int bounce, const __grid_constant__ FlatPairsU up) {
    pdl_launch_dependents();
    SceneAccess<true> S = stage_scene<true>(a);
    S.upairs = &up;
    pdl_wait();
    const uint32_t n1 = a.counts[bounce * 4 + Q_DIFFUSE], n2 = a.counts[bounce * 4 + Q_MIRROR], n3 = a.counts[bounce * 4 + Q_GLASS];
    // estimated work per queue entry relative to a diffuse vertex (two rays, light sample): measured
    // instructions per entry, padding of the sparsely filled specular chunks included
    const float w1 = float(n1), w2 = 0.45f * float(n2), w3 = 0.6f * float(n3);
    const float total = w1 + w2 + w3;
    if (total <= 0.0f) return;
    const uint32_t G = gridDim.x;
    uint32_t g2 = n2 ? max(1u, min(uint32_t(float(G) * w2 / total + 0.5f), (n2 + kThreads - 1) / kThreads)) : 0u;
    uint32_t g3 = n3 ? max(1u, min(uint32_t(float(G) * w3 / total + 0.5f), (n3 + kThreads - 1) / kThreads)) : 0u;
    if (g2 + g3 >= G) { g2 = min(g2, G / 3); g3 = min(g3, G / 3); }
    const uint32_t g1 = n1 ? min(G - g2 - g3, (n1 + kThreads - 1) / kThreads) : 0u;
    __shared__ RecStage<!FIRST> stage;
    const uint32_t b = blockIdx.x;
    if (b < g1) bounce_flat_body<Q_DIFFUSE, FIRST, false, true, false, FOLD, UNI>(a, bounce, S, n1, b, g1, stage);
    else if (b < g1 + g2) bounce_flat_body<Q_MIRROR, FIRST, false, true, false, FOLD, UNI>(a, bounce, S, n2, b - g1, g2, stage);
    else if (b < g1 + g2 + g3) bounce_flat_body<Q_GLASS, FIRST, false, true, false, FOLD, UNI>(a, bounce, S, n3, b - g1 - g2, g3, stage);
}

// ---- bounce, tree scenes: shade and queue the rays -----------------------------------------
// Asynchronous prefetch of the NEXT slot's state into shared memory (see prefetch_rec); here the
// state is indexed by slot, so the queue entry is loaded two iterations ahead.
template <bool TP> struct VertexStage {
    float4 hp[2][kThreads];
    float4 dw[2][kThreads];
    float4 tp[TP ? 2 : 1][TP ? kThreads : 1];
};
template <bool TP> __device__ __forceinline__ void prefetch_vertex(const PassArgs& a, uint32_t slot, VertexStage<TP>& st, int buf) {
    const int t = threadIdx.x;
    if (slot != kInvalid) {
        cp_async16(&st.hp[buf][t], a.hp + slot);
        cp_async16(&st.dw[buf][t], a.dw + slot);
        if (TP) cp_async16(&st.tp[buf][t], a.tp + slot);
    }
    cp_async_commit();
}

// Tree scenes only shade here: the rays go to the bounce's ray queue and trace_kernel walks them
// with dynamic fetch (a heavy tail of long walks would otherwise hold the other 31 lanes of the
// warp -- ncu: 3.4 of 32 lanes active); trace_kernel also adds the light sample and delivers the
// continuation vertex into the slot-indexed state and the next bounce's material queues.
// Sort key of a queued ray (ray_sort.cu): where it starts, on a 32^3 grid over the root box, in Morton order.
// Shadow rays (they all aim at the lights): 1 | 15 bits; continuation rays: 0 | 12 bits (16^3 cells) | direction octant.
__device__ __forceinline__ uint32_t spread5(uint32_t x) { // bit k -> bit 3k
    x = (x | (x << 8)) & 0x100fu;
    x = (x | (x << 4)) & 0x10c3u;
    x = (x | (x << 2)) & 0x1249u;
    return x;
}
__device__ __forceinline__ uint32_t ray_sort_key(const PathSceneD& g, float3 o, float3 d, bool shadow) {
    const int sh = kMaxTreeDepth - 5;
    const uint32_t x = uint32_t(min(max(__float2int_rd((o.x - g.root_lo[0]) * g.grid_scale[0]) >> sh, 0), 31));
    const uint32_t y = uint32_t(min(max(__float2int_rd((o.y - g.root_lo[1]) * g.grid_scale[1]) >> sh, 0), 31));
    const uint32_t z = uint32_t(min(max(__float2int_rd((o.z - g.root_lo[2]) * g.grid_scale[2]) >> sh, 0), 31));
    const uint32_t m = spread5(x) | (spread5(y) << 1) | (spread5(z) << 2);
    if (shadow) return 0x8000u | m;
    const uint32_t oct = (d.x < 0.0f ? 1u : 0u) | (d.y < 0.0f ? 2u : 0u) | (d.z < 0.0f ? 4u : 0u);
    return ((m >> 3) << 3) | oct;
}

template <int KIND, bool FIRST, bool LAST>
__global__ void __launch_bounds__(kThreads, KIND != Q_DIFFUSE ? 4 : 3) bounce_kernel(const PassArgs a, const int bounce) {
    constexpr bool kDiffuse = KIND == Q_DIFFUSE;
    pdl_launch_dependents();
    if (LAST && !kDiffuse) return; // a specular vertex on the last segment contributes nothing
    SceneAccess<false> S;
    S.g = &a.scene;
    pdl_wait();
    const uint32_t n = a.counts[bounce * 4 + KIND];
    if (blockIdx.x * kThreads >= n) return; // short queue: surplus CTAs leave
    const uint32_t* __restrict__ qin = a.q[(bounce & 1) * 3 + (KIND - 1)];
    WarpCursor ray_cur = {0, 0, 0, false};
    uint32_t* const ray_counter = a.counts + bounce * 4 + Q_RAYS;
    unsigned traced = 0, shadow_rays = 0, calls = 0;
    const uint32_t stride = gridDim.x * kThreads;
    const uint32_t lane = threadIdx.x & 31u;

    __shared__ VertexStage<!FIRST> stage;
    uint32_t q = blockIdx.x * kThreads + threadIdx.x;
    uint32_t s_cur = kInvalid, s_nxt = kInvalid;
    if (q < n) s_cur = qin[q];
    if (q + stride < n && q + stride >= q) s_nxt = qin[q + stride];
    int buf = 0;
    prefetch_vertex(a, s_cur, stage, 0);
    for (; q - lane < n; q += stride) {
        uint32_t s_nn = kInvalid;
        {
            const uint32_t q2 = q + 2u * stride;
            if (q2 < n && q2 > q) s_nn = qin[q2];
        }
        prefetch_vertex(a, s_nxt, stage, buf ^ 1); // next slot's state, in flight during this body
        cp_async_wait<1>();                        // this slot's state has landed
        const uint32_t slot = s_cur;
        bool ray_shadow = false, ray_cont = false; // rays to enqueue
        float3 ray_o = f3(0.f, 0.f, 0.f), ray_w = f3(0.f, 0.f, 1.f), ray_d = f3(0.f, 0.f, 1.f), ray_rgb = f3(0.f, 0.f, 0.f);
        float ray_tmax = 0.0f;
        uint32_t ray_flags = 0;
        if (slot != kInvalid) {
            ++calls;
            const int tid = threadIdx.x;
            const float4 hp = stage.hp[buf][tid], dw = stage.dw[buf][tid];
            const float3 p = f3(hp.x, hp.y, hp.z), d = f3(dw.x, dw.y, dw.z);
            const uint32_t prim = __float_as_uint(hp.w), pixel = __float_as_uint(dw.w);
            float3 T = f3(1.f, 1.f, 1.f);
            uint32_t sample;
            if (FIRST) {
                uint32_t lp;
                sample = uint32_t(a.sample_base) + fast_div(slot, a.pix_count, lp);
            } else {
                const float4 tp = stage.tp[buf][tid];
                T = f3(tp.x, tp.y, tp.z);
                sample = __float_as_uint(tp.w);
            }
            const Shaded sh = shade_vertex<KIND, LAST, false>(a, S, bounce, p, d, T, prim, pixel, sample);
            T = sh.T;
            const bool cont = !LAST && (T.x > 0.0f || T.y > 0.0f || T.z > 0.0f);
            if (cont) ++traced;
            if (sh.want_shadow) ++shadow_rays;
            ray_o = sh.no; ray_w = sh.w; ray_d = sh.nd; ray_rgb = sh.lit_rgb; ray_tmax = sh.tmax_s;
            ray_flags = (sh.flags & 1u) ? kRaySpecular : 0u;
            // the continuation vertex's direction / pixel / throughput / sample are known now;
            // trace_kernel adds the hit point and primitive (or ends the path)
            ray_shadow = kDiffuse && sh.want_shadow;
            ray_cont = cont;
            if (cont) {
                a.dw[slot] = make_float4(sh.nd.x, sh.nd.y, sh.nd.z, __uint_as_float(pixel));
                a.tp[slot] = make_float4(T.x, T.y, T.z, __uint_as_float(sample));
            }
        }
        // ray records: (origin, tmax) (direction, slot | kRayShadow | kRaySpecular) (light sample rgb)
        const uint32_t is = warp_reserve(ray_cur, ray_shadow, ray_counter);
        if (is != kInvalid) {
            st_stream(a.ray0 + is, ray_o.x, ray_o.y, ray_o.z, __float_as_uint(ray_tmax));
            st_stream(a.ray1 + is, ray_w.x, ray_w.y, ray_w.z, slot | kRayShadow);
            st_stream(a.ray2 + is, ray_rgb.x, ray_rgb.y, ray_rgb.z, 0u);
            if (a.rkey) a.rkey[is] = (uint16_t)ray_sort_key(a.scene, ray_o, ray_w, true);
        }
        const uint32_t ic = warp_reserve(ray_cur, ray_cont, ray_counter);
        if (ic != kInvalid) {
            st_stream(a.ray0 + ic, ray_o.x, ray_o.y, ray_o.z, __float_as_uint(FLT_MAX));
            st_stream(a.ray1 + ic, ray_d.x, ray_d.y, ray_d.z, slot | ray_flags);
            if (a.rkey) a.rkey[ic] = (uint16_t)ray_sort_key(a.scene, ray_o, ray_d, false);
        }
        s_cur = s_nxt; s_nxt = s_nn;
        buf ^= 1;
    }
    cp_async_wait<0>();
    for (uint32_t i = ray_cur.pos + lane; i < ray_cur.end; i += 32u) a.ray1[i] = make_float4(0.f, 0.f, 0.f, __uint_as_float(kInvalid));
    if (ray_cur.has_next) { // a chunk reserved ahead of time and never used
        const uint32_t base = __shfl_sync(kFull, ray_cur.next, 0);
        for (uint32_t i = lane; i < kChunk; i += 32u) a.ray1[base + i] = make_float4(0.f, 0.f, 0.f, __uint_as_float(kInvalid));
    }
    calls = warp_sum(calls);
    traced = warp_sum(traced);
    shadow_rays = warp_sum(shadow_rays);
    if (lane == 0 && calls) {
        atomicAdd(a.totals + 2, (unsigned long long)calls);
        if (FIRST) atomicAdd(a.totals + 3, (unsigned long long)calls);
        if (traced) atomicAdd(a.totals + 0, (unsigned long long)traced);
        if (shadow_rays) atomicAdd(a.totals + 1, (unsigned long long)shadow_rays);
        if (!FIRST && kDiffuse) atomicAdd(a.totals + 5, (unsigned long long)calls); // diffuse vertices whose light sample may read L
    }
}

// ---- trace (tree scenes): persistent walk with dynamic ray fetch -----------------------------
// One launch per bounce over the ray queue the bounce kernels filled. Every lane owns at most one
// ray; a round = every lane with a ray walks to its next non-empty leaf and tests it (TreeWalk2::step).
// Lanes whose ray finished deliver the result -- shadow ray: add the light sample unless occluded;
// continuation ray: hit point + primitive into the vertex record, slot into its material queue --
// and, once PassArgs::refill lanes are idle, the warp pulls that many new rays with ONE atomic. A warp's
// time is then the sum of its rays' rounds / 32, not 32 x the longest walk.

template <bool COOP, int WALK, int OCC = 3> __global__ void __launch_bounds__(kThreads, OCC) trace_kernel(const PassArgs a, const int bounce) {
    pdl_launch_dependents();
    const SceneAccess<false> S = stage_scene<false>(a);
    pdl_wait();
    const uint32_t n = a.counts[bounce * 4 + Q_RAYS];
    if (a.ray_hint && blockIdx.x == 0 && threadIdx.x == 0) atomicMax(a.ray_hint + bounce, n);
    if (n == 0) return;
    const bool sort = bounce + 1 < a.max_depth;
    const bool next_last = bounce + 2 >= a.max_depth;
    Sorter out;
    out.init(a, bounce + 1);
    uint32_t* const fetch = a.counts + (kMaxPathDepth + 1) * 4 + bounce;
    const uint32_t lane = threadIdx.x & 31u;
    typename WalkOf<WALK>::type w = {};
    unsigned cnt_node = 0, cnt_prim = 0;
    bool have = false, more = true;
    uint32_t tag = 0; // slot | flags of the lane's ray
    float3 rgb = f3(0.f, 0.f, 0.f);
    int pend_kind = -1;
    uint32_t pend_slot = 0;
    unsigned lit = 0;
    while (true) {
        // (converged) deliver the slots whose continuation ray found a surface
        if (sort && __any_sync(kFull, pend_kind >= 0)) {
            out.push(pend_kind, pend_slot);
            pend_kind = -1;
        }
        const uint32_t idle = __ballot_sync(kFull, !have);
        if (more && idle != 0u && (__popc(idle) >= a.refill || idle == kFull)) {
            const uint32_t cnt = __popc(idle);
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(fetch, cnt);
            base = __shfl_sync(kFull, base, 0);
            if (base + cnt >= n) more = false; // the queue is drained (warp-uniform)
            const uint32_t at = base + __popc(idle & ((1u << lane) - 1u));
            if (!have && at < n) {
                const uint32_t i = at < a.perm_n ? __ldg(a.perm + at) : at; // sorted by origin cell (ray_sort.cu) / queue order
                const float4 r1 = ld_stream(a.ray1 + i); // streamed: read once (evict first, the scene stays in L2)
                tag = __float_as_uint(r1.w);
                if (tag != kInvalid) { // not the padding of a producer's last chunk
                    const float4 r0 = ld_stream(a.ray0 + i);
                    const bool shadow = (tag & kRayShadow) != 0u;
                    if (shadow) {
                        const float4 r2 = ld_stream(a.ray2 + i);
                        rgb = f3(r2.x, r2.y, r2.z);
                    }
                    have = true;
                    if (w.init(S, f3(r0.x, r0.y, r0.z), f3(r1.x, r1.y, r1.z), r0.w, shadow)) have = false, pend_kind = -2; // finished at once
                }
            }
        }
        // a ray that finished inside init() (missed the root box / one-leaf scene) is delivered like any other
        bool finished = pend_kind == -2;
        if (finished) pend_kind = -1;
        if (__ballot_sync(kFull, have || finished) == 0u) {
            if (!more) break;
            continue;
        }
        if (w.template step<false, COOP>(S, have)) { // all 32 lanes: one round
            finished = true;
            have = false;
        }
        if (finished) {
            if (WALK == 2 || WALK == 6) walk_counts(w, cnt_node, cnt_prim);
            const uint32_t slot = tag & kRaySlotMask;
            if (tag & kRayShadow) {
                if (w.best_prim == kInvalid) { // unoccluded: the light sample counts
                    ++lit;
                    add_radiance(a, slot, rgb);
                }
            } else if (w.best_prim != kInvalid) {
                const float4 t4 = S.hot_row(w.best_prim, 3);
                const int bsdf = __float_as_int(t4.y);
                if (bsdf == G19_BSDF_EMITTER) {
                    // emission counts after specular bounces only (NEE covers the diffuse ones)
                    if (tag & kRaySpecular) {
                        const float4 T = a.tp[slot];
                        const MaterialD& m = a.scene.materials[__float_as_int(t4.x)];
                        add_radiance(a, slot, f3(T.x * m.emission[0], T.y * m.emission[1], T.z * m.emission[2]));
                    }
                } else if (bsdf == G19_BSDF_DIFFUSE || !next_last) {
                    const float3 p = w.o + w.d * w.best;
                    a.hp[slot] = make_float4(p.x, p.y, p.z, __uint_as_float(w.best_prim));
                    pend_kind = bsdf;
                    pend_slot = slot;
                }
            }
        }
    }
    if (sort) out.flush();
    lit = warp_sum(lit);
    if (lane == 0 && lit) atomicAdd(a.totals + 4, (unsigned long long)lit);
    if (WALK == 2 || WALK == 6) flush_walk_counts(a, cnt_node, cnt_prim);
}

// ---- primary-hit AOV ------------------------------------------------------------------------
// The ray the REFERENCE casts -- through the integer pixel corner, no jitter (raytracer.h:41-43) -- traced
// through THIS engine's structures (flat pair loops / linear octree, nearest hit): entity id (push order, the
// numbering REF mode reports), hit point and the normal turned towards the ray (what ImpTriangle::intersect
// returns, entities.h:239-246; spheres: (p - centre) / r, entities.h:94). Ties PATH mode back to the pinned
// mode: the ids must equal REF's wherever "last hit wins" coincides with "nearest hit" (tests/test_path_link.py),
// and with max_depth = 0 these three arrays feed the reference's own shade (ref_shade_kernel), so the default
// scene closes the loop through the PATH pipeline.

// The entity a hit on primitive `prim` at p (ray direction d) reports, and its normal: for a triangle or parallelogram
// the geometric normal turned against the ray, for a sphere (p - c) / r. primary_kernel and cast_kernel share it.
template <bool ALL>
__device__ __forceinline__ int32_t hit_entity(const SceneAccess<ALL>& S, uint32_t prim, float3 p, float3 d, float3& ng) {
    const float4 r0 = S.hot_row(prim, 0), tag = S.hot_row(prim, 3);
    float4 c0, c1;
    S.cold(prim, c0, c1);
    ng = f3(c0.x, c0.y, c0.z);
    int half = 0;
    if (tag.z == 0.0f) {
        ng = (p - f3(r0.x, r0.y, r0.z)) * __fdividef(1.0f, r0.w);
    } else {
        if (tag.z > 1.5f) { // merged parallelogram: which of its two triangles (the builder's b1 >= b2 rule)
            const float4 r1 = S.hot_row(prim, 1);
            const float b1 = fmaf(r0.x, p.x, fmaf(r0.y, p.y, fmaf(r0.z, p.z, r0.w)));
            const float b2 = fmaf(r1.x, p.x, fmaf(r1.y, p.y, fmaf(r1.z, p.z, r1.w)));
            half = b1 >= b2 ? 0 : 1;
        }
        if (dot(ng, d) > 0.0f) ng = -ng;
    }
    return S.g->prim_entity[2 * size_t(prim) + half];
}

template <bool ALL>
__global__ void __launch_bounds__(kThreads, 2) primary_kernel(const PassArgs a, int32_t* __restrict__ ids, double* __restrict__ points,
                                                              double* __restrict__ normals) {
    const SceneAccess<ALL> S = stage_scene<ALL>(a);
    const uint32_t n = uint32_t(a.map.n_local_pix);
    const uint32_t stride = gridDim.x * kThreads;
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t lp = blockIdx.x * kThreads + threadIdx.x; lp - lane < n; lp += stride) { // warp-uniform trip count
        bool live = false;
        float3 o = f3(0.f, 0.f, 0.f), d = f3(0.f, 0.f, 1.f);
        if (lp < n) {
            const uint32_t lt = lp >> 10, in = lp & 1023u;
            uint32_t tx;
            const uint32_t t = lt * uint32_t(a.map.world) + uint32_t(a.map.rank);
            const uint32_t ty = fast_div(t, uint32_t(a.map.tiles_x), tx);
            const int x = int(tx * kTile + (in & 31u)), y = int(ty * kTile + (in >> 5));
            live = x < a.map.w && y < a.map.h;
            if (live) {
                const PathCamera& c = a.cam;
                const float fx = float(x) * 0.0002f, fy = float(y) * 0.0002f;
                o = f3(c.pos[0], c.pos[1], c.pos[2]);
                d = normalize(f3(c.top_left[0] - c.left[0] * fx - c.up[0] * fy, c.top_left[1] - c.left[1] * fx - c.up[1] * fy,
                                 c.top_left[2] - c.left[2] * fx - c.up[2] * fy));
            }
        }
        float t;
        uint32_t prim;
        const bool hit = nearest<ALL, false, 1>(S, live, o, d, t, prim); // all 32 lanes walk together
        if (lp < n) {
            int32_t id = -1;
            double px = DBL_MAX, py = DBL_MAX, pz = DBL_MAX, nx = 0, ny = 0, nz = 0; // a miss looks like REF's (ref_visibility_kernel)
            if (hit) {
                const float3 p = o + d * t;
                float3 ng;
                id = hit_entity(S, prim, p, d, ng);
                px = double(p.x); py = double(p.y); pz = double(p.z);
                nx = double(ng.x); ny = double(ng.y); nz = double(ng.z);
            }
            ids[lp] = id;
            if (points) { points[lp] = px; points[size_t(n) + lp] = py; points[2 * size_t(n) + lp] = pz; }
            if (normals) { normals[lp] = nx; normals[size_t(n) + lp] = ny; normals[2 * size_t(n) + lp] = nz; }
        }
    }
}

// ---- batched ray queries (g19_cast_rays) ---------------------------------------------------------
// Rays in, hits out, through the render's own structures: the pair loops of a flat scene, the selected walk of a tree
// scene. A ray record is two float4, (origin, tmax) and (direction, -). It is invalid -- a miss, never walked -- when
// its origin or direction is not finite, its direction is zero or its tmax is not > 0 (NaN included).
__device__ __forceinline__ bool finite_f(float x) { return (__float_as_uint(x) & 0x7f800000u) != 0x7f800000u; }
__device__ __forceinline__ bool cast_ray(const CastArgs& c, uint32_t i, float3& o, float3& d, float& tmax) {
    const float4 r0 = ld_stream(c.rays + 2 * size_t(i)), r1 = ld_stream(c.rays + 2 * size_t(i) + 1);
    o = f3(r0.x, r0.y, r0.z);
    d = f3(r1.x, r1.y, r1.z);
    tmax = fminf(r0.w, FLT_MAX); // (an infinite bound is FLT_MAX, the bound of the render's camera rays)
    const float m = fmaxf(fabsf(d.x), fmaxf(fabsf(d.y), fabsf(d.z)));
    if (!(finite_f(o.x) && finite_f(o.y) && finite_f(o.z) && finite_f(d.x) && finite_f(d.y) && finite_f(d.z) && m > 0.0f &&
          r0.w > 0.0f))
        return false;
    // sphere_hit assumes a unit direction; a power-of-two prescale keeps dot(d, d) clear of overflow and of flushed
    // denormals (and is exact, so an ordinary direction normalises exactly as the render's do)
    d = normalize(d * (m > 0x1p32f ? 0x1p-80f : (m < 0x1p-32f ? 0x1p80f : 1.0f)));
    return true;
}
// Outputs of ray i: entity id (push order) and, where asked for, t along the unit direction and the normal
// (hit_entity's rule); a miss is -1, +inf, (0, 0, 0).
template <bool ALL>
__device__ __forceinline__ void cast_store(const CastArgs& c, const SceneAccess<ALL>& S, uint32_t i, uint32_t prim, float3 o, float3 d,
                                           float t) {
    int32_t id = -1;
    float3 ng = f3(0.f, 0.f, 0.f);
    if (prim != kInvalid) id = hit_entity(S, prim, o + d * t, d, ng);
    else t = __int_as_float(0x7f800000);
    c.ids[i] = id;
    if (c.t) c.t[i] = t;
    if (c.normals) {
        c.normals[3 * size_t(i)] = ng.x;
        c.normals[3 * size_t(i) + 1] = ng.y;
        c.normals[3 * size_t(i) + 2] = ng.z;
    }
}

// Flat scenes: one ray per thread over the staged scene. An any-hit query takes the nearest-hit loop with the ray's own
// bound: a hit below tmax exists exactly when the nearest one is below it, and the shadow half of trace_flat<true> runs
// the same arithmetic per ray (its other half would test a switched-off ray for nothing).
__global__ void __launch_bounds__(kThreads, 4) cast_flat_kernel(const PassArgs a, const CastArgs c) {
    const SceneAccess<true> S = stage_scene<true>(a);
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < c.n; i += gridDim.x * kThreads) {
        float3 o, d;
        float tmax, t = 0.0f;
        uint32_t prim = kInvalid;
        bool occ;
        if (cast_ray(c, i, o, d, tmax)) trace_flat<false>(S, o, d, tmax, d, -1.0f, t, prim, occ);
        cast_store(c, S, i, prim, o, d, t);
    }
}

// Tree scenes: trace_kernel's persistent scheme over the caller's rays -- the warp interleaves the walks of 32 rays in
// rounds, a lane that finishes writes its ray's outputs, and once PassArgs::refill lanes are idle the warp pulls that many
// new rays with one atomic on the cast's cursor. ANY = occlusion query: the walks stop at the first hit below tmax.
template <bool COOP, int WALK, bool ANY, int OCC = 3>
__global__ void __launch_bounds__(kThreads, OCC) cast_kernel(const PassArgs a, const CastArgs c) {
    const SceneAccess<false> S = stage_scene<false>(a);
    const uint32_t lane = threadIdx.x & 31u;
    typename WalkOf<WALK>::type w = {};
    unsigned cnt_node = 0, cnt_prim = 0;
    bool have = false, more = true;
    uint32_t ray = 0; // index of the lane's ray
    while (true) {
        bool finished = false;
        const uint32_t idle = __ballot_sync(kFull, !have);
        if (more && idle != 0u && (__popc(idle) >= a.refill || idle == kFull)) {
            const uint32_t cnt = __popc(idle);
            uint32_t base = 0;
            if (lane == 0) base = atomicAdd(c.cursor, cnt);
            base = __shfl_sync(kFull, base, 0);
            if (base + cnt >= c.n) more = false; // all rays handed out (warp-uniform)
            const uint32_t at = base + __popc(idle & ((1u << lane) - 1u));
            if (!have && at < c.n) {
                ray = at;
                float3 o, d;
                float tmax;
                if (!cast_ray(c, at, o, d, tmax)) cast_store(c, S, at, kInvalid, o, d, 0.0f);
                else if (w.init(S, o, d, tmax, ANY)) finished = true; // missed the root box / one-leaf scene / a big primitive
                else have = true;
            }
        }
        if (__ballot_sync(kFull, have || finished) == 0u) {
            if (!more) break;
            continue;
        }
        if (w.template step<false, COOP>(S, have)) { // all 32 lanes: one round
            finished = true;
            have = false;
            if (WALK == 2 || WALK == 6) walk_counts(w, cnt_node, cnt_prim); // (rays that walked, as traverse() counts)
        }
        if (finished) cast_store(c, S, ray, w.best_prim, w.o, w.d, w.best);
    }
    if (WALK == 2 || WALK == 6) flush_walk_counts(a, cnt_node, cnt_prim);
}

// ---- accumulate / resolve ---------------------------------------------------------------
// FLAT: the finished paths' radiance is a float4 per slot, stored once for EVERY slot of the pass by the kernel
// that ended its path, so it is only read here; otherwise three planes that paths add to and this kernel clears.
// ADAPT (adaptive passes): the window positions go through the tile list (PassArgs::tiles), and a fourth plane of accum
// takes the sum of Y^2 per pixel, Y = 0.2126 R + 0.7152 G + 0.0722 B of each sample, in the same sample order.
__device__ __forceinline__ float luminance(float r, float g, float b) {
    return __fmaf_rn(0.0722f, b, __fmaf_rn(0.7152f, g, __fmul_rn(0.2126f, r)));
}
template <bool ADAPT> struct Moment {
    __device__ __forceinline__ void add(float, float, float) {}
};
template <> struct Moment<true> {
    float s2;
    __device__ __forceinline__ void add(float r, float g, float b) {
        const float y = luminance(r, g, b);
        s2 = __fmaf_rn(y, y, s2);
    }
};
template <bool FLAT, bool ADAPT = false> __global__ void __launch_bounds__(kThreads) accumulate_kernel(const PassArgs a) {
    pdl_launch_dependents();
    pdl_wait();
    const uint32_t npix = (uint32_t)a.map.n_local_pix, nwin = a.pix_count;
    const uint32_t wp = blockIdx.x * kThreads + threadIdx.x; // pixel within the pass's window
    if (wp < nwin) {
        uint32_t lp = a.pix_base + wp;
        if (ADAPT) lp = (a.tiles[lp >> 10] << 10) | (lp & 1023u);
        float acc0 = a.accum[lp], acc1 = a.accum[(size_t)npix + lp], acc2 = a.accum[2 * (size_t)npix + lp];
        Moment<ADAPT> mo;
        if constexpr (ADAPT) mo.s2 = a.accum[3 * (size_t)npix + lp];
        // strictly in sample order (independent of the pass split); loads batched four samples deep
        if constexpr (FLAT) {
            float4* L = reinterpret_cast<float4*>(a.L) + wp;
            int s = 0;
            for (; s + 4 <= a.spp_pass; s += 4) {
                float4 v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] = L[(size_t)(s + k) * nwin];
#pragma unroll
                for (int k = 0; k < 4; ++k) { acc0 += v[k].x; acc1 += v[k].y; acc2 += v[k].z; mo.add(v[k].x, v[k].y, v[k].z); }
            }
            for (; s < a.spp_pass; ++s) {
                const float4 v = L[(size_t)s * nwin];
                acc0 += v.x; acc1 += v.y; acc2 += v.z;
                mo.add(v.x, v.y, v.z);
            }
        } else {
            float* L0 = a.L + wp;
            float* L1 = a.L + a.plane + wp;
            float* L2 = a.L + 2 * a.plane + wp;
            int s = 0;
            for (; s + 4 <= a.spp_pass; s += 4) {
                float v0[4], v1[4], v2[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    size_t i = (size_t)(s + k) * nwin;
                    v0[k] = L0[i]; v1[k] = L1[i]; v2[k] = L2[i];
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    size_t i = (size_t)(s + k) * nwin;
                    acc0 += v0[k]; acc1 += v1[k]; acc2 += v2[k];
                    mo.add(v0[k], v1[k], v2[k]);
                    if (v0[k] != 0.0f) L0[i] = 0.0f;
                    if (v1[k] != 0.0f) L1[i] = 0.0f;
                    if (v2[k] != 0.0f) L2[i] = 0.0f;
                }
            }
            for (; s < a.spp_pass; ++s) {
                size_t i = (size_t)s * nwin;
                float v0 = L0[i], v1 = L1[i], v2 = L2[i];
                acc0 += v0; acc1 += v1; acc2 += v2;
                mo.add(v0, v1, v2);
                if (v0 != 0.0f) L0[i] = 0.0f;
                if (v1 != 0.0f) L1[i] = 0.0f;
                if (v2 != 0.0f) L2[i] = 0.0f;
            }
        }
        a.accum[lp] = acc0;
        a.accum[(size_t)npix + lp] = acc1;
        a.accum[2 * (size_t)npix + lp] = acc2;
        if constexpr (ADAPT) a.accum[3 * (size_t)npix + lp] = mo.s2;
    }
    // the pass is over: clear its queue lengths for the next one
    if (blockIdx.x == 0)
        for (int i = threadIdx.x; i < (kMaxPathDepth + 1) * 5; i += kThreads) a.counts[i] = 0; // queue lengths + fetch cursors
}

__global__ void __launch_bounds__(kThreads) resolve_kernel(TileMap map, const float* __restrict__ accum, int spp,
                                                           float* __restrict__ rad_l, uint8_t* __restrict__ rgb_l) {
    const uint32_t npix = (uint32_t)map.n_local_pix;
    uint32_t lp = blockIdx.x * kThreads + threadIdx.x;
    if (lp >= npix) return;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float v = __fdiv_rn(accum[(size_t)c * npix + lp], float(spp));
        rad_l[3 * (size_t)lp + c] = v;
        float cl = fminf(fmaxf(v, 0.0f), 1.0f);
        rgb_l[3 * (size_t)lp + c] = (uint8_t)(int)(255.0f * cl); // truncation, as Image::setPixel
    }
}

// ---- adaptive renders: tile test, compaction, resolve at each tile's count -----------------------------------
// The variance of a pixel's mean after n samples, from its sums (accum planes 0-2: R, G, B; plane 3: Y^2):
// m = 0.2126 R/n + 0.7152 G/n + 0.0722 B/n with the means resolve stores, v = max(S2 - n m^2, 0) / (n (n - 1)).
__device__ __forceinline__ float pixel_variance(const float* __restrict__ accum, size_t npix, uint32_t lp, int n, float& m) {
    const float fn = float(n);
    m = luminance(__fdiv_rn(accum[lp], fn), __fdiv_rn(accum[npix + lp], fn), __fdiv_rn(accum[2 * npix + lp], fn));
    const float d = __fsub_rn(accum[3 * npix + lp], __fmul_rn(fn, __fmul_rn(m, m)));
    return __fdiv_rn(fmaxf(d, 0.0f), __fmul_rn(fn, fn - 1.0f));
}

// One warp per active tile; lane = column, 32 rows. Every pixel's error e = sqrt(v) / max(m, 0.05) is computed alone and
// max is exact, so E does not depend on the reduction order.
__global__ void __launch_bounds__(kThreads) tile_test_kernel(TileMap map, const float* __restrict__ accum, const uint32_t* __restrict__ list,
                                                             uint32_t n_active, int n, int spp, float tau, int32_t* __restrict__ tile_n,
                                                             uint32_t* __restrict__ flag) {
    const uint32_t entry = (blockIdx.x * kThreads + threadIdx.x) >> 5, lane = threadIdx.x & 31u;
    if (entry >= n_active) return;
    const uint32_t lt = list[entry];
    const uint32_t t = lt * (uint32_t)map.world + (uint32_t)map.rank;
    const uint32_t ty = t / (uint32_t)map.tiles_x, tx = t - ty * (uint32_t)map.tiles_x;
    const int x = int(tx * kTile + lane);
    float E = 0.0f;
    if (x < map.w)
        for (int row = 0; row < kTile && int(ty * kTile) + row < map.h; ++row) {
            float m;
            const float v = pixel_variance(accum, (size_t)map.n_local_pix, (lt << 10) | (uint32_t(row) << 5) | lane, n, m);
            E = fmaxf(E, __fdiv_rn(__fsqrt_rn(v), fmaxf(m, 0.05f)));
        }
    for (int off = 16; off > 0; off >>= 1) E = fmaxf(E, __shfl_xor_sync(kFull, E, off));
    if (lane == 0) {
        tile_n[lt] = n;
        flag[entry] = (E > tau && n < spp) ? 1u : 0u;
    }
}

// One CTA of 1024 threads walks the list in blocks of 1024 entries: warp ballots + a scan of the 32 warp totals. The
// order of the list is kept (ascending local tile).
__global__ void __launch_bounds__(1024) tile_compact_kernel(const uint32_t* __restrict__ list, uint32_t n_active,
                                                            const uint32_t* __restrict__ flag, uint32_t* __restrict__ list_out,
                                                            uint32_t* __restrict__ count_out) {
    __shared__ uint32_t warp_base[32], block_total;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t base = 0;
    for (uint32_t i0 = 0; i0 < n_active; i0 += 1024u) {
        const uint32_t i = i0 + threadIdx.x;
        const bool keep = i < n_active && flag[i] != 0u;
        const uint32_t m = __ballot_sync(kFull, keep);
        if (lane == 0) warp_base[warp] = __popc(m);
        __syncthreads();
        if (warp == 0) { // exclusive scan of the warp totals
            const uint32_t c = warp_base[lane];
            uint32_t inc = c;
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t o = __shfl_up_sync(kFull, inc, off);
                if (lane >= uint32_t(off)) inc += o;
            }
            warp_base[lane] = inc - c;
            if (lane == 31) block_total = inc;
        }
        __syncthreads();
        if (keep) list_out[base + warp_base[warp] + __popc(m & ((1u << lane) - 1u))] = list[i];
        base += block_total;
        __syncthreads();
    }
    if (threadIdx.x == 0) *count_out = base;
}

__global__ void __launch_bounds__(kThreads) resolve_adaptive_kernel(TileMap map, const float* __restrict__ accum,
                                                                    const int32_t* __restrict__ tile_n, uint8_t* rgb, float* rad,
                                                                    float* var, int32_t* spp) {
    const uint32_t lp = blockIdx.x * kThreads + threadIdx.x;
    if (lp >= (uint32_t)map.n_local_pix) return;
    const uint32_t lt = lp >> 10, in = lp & 1023u;
    const uint32_t t = lt * (uint32_t)map.world + (uint32_t)map.rank;
    const uint32_t ty = t / (uint32_t)map.tiles_x, tx = t - ty * (uint32_t)map.tiles_x;
    const int x = int(tx * kTile + (in & 31u)), y = int(ty * kTile + (in >> 5));
    if (y >= map.h || x >= map.w) return;
    const int n = tile_n[lt];
    const size_t npix = (size_t)map.n_local_pix, gpx = (size_t)y * map.w + x;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float v = __fdiv_rn(accum[c * npix + lp], float(n));
        if (rad) rad[3 * gpx + c] = v;
        const float cl = fminf(fmaxf(v, 0.0f), 1.0f);
        if (rgb) rgb[3 * gpx + c] = (uint8_t)(int)(255.0f * cl); // truncation, as Image::setPixel
    }
    if (var) {
        float m;
        var[gpx] = pixel_variance(accum, npix, lp, n, m);
    }
    if (spp) spp[gpx] = n;
}

// Persistent grids: SM count x the CTAs the occupancy calculator says are resident.
template <typename K> static int resident_grid(K kernel, size_t smem, int sm_count) {
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, smem) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    return per_sm * sm_count;
}

static bool all_staged(const PassArgs& a) { // one leaf, everything in shared memory
    return a.scene.n_nodes == 1 && a.stage_nodes >= 1 && a.stage_prims >= a.scene.n_index &&
           a.scene.n_index == a.scene.n_prims && a.stage_cold >= a.scene.n_prims && a.stage_lights >= a.scene.n_lights;
}

size_t path_smem_bytes(const PassArgs& a) {
    size_t nb = (size_t(a.stage_nodes) * 8 + 15) & ~size_t(15);
    size_t cb = all_staged(a) ? size_t(a.stage_cold) * 32 + size_t(a.stage_lights) * 80 + size_t(a.scene.pairs_bytes) : 0;
    return nb + size_t(a.stage_prims) * 64 + cb + size_t(a.stack_levels) * kThreads * 4 + 16 +
           (a.coop_leaf ? size_t(kThreads / 32) * 32 * 8 : 0);
}

// per thread: launches are issued and their errors collected on the thread inside path_render, so several
// g19_ctx driven from several threads never see (or race on) each other's failures
static thread_local char g_launch_error[256] = "";
static void note_launch_error(const char* what, cudaError_t e, size_t smem, int grid) {
    if (!g_launch_error[0])
        snprintf(g_launch_error, sizeof g_launch_error, "%s: %s (dynamic smem %zu B, grid %d)", what, cudaGetErrorString(e),
                 smem, grid);
}

// The grid of a persistent kernel = SM count x resident CTAs, cached per (device, kernel, smem size):
// function attributes are per device, and one process may drive several (one g19_ctx each).
template <typename K> static int persistent_grid(K kernel, size_t smem, int sm_count) {
    struct Entry { int device; const void* fn; size_t smem; int grid; };
    static Entry cache[256];
    static int n_cache = 0;
    static std::mutex lock;
    int device = 0;
    cudaGetDevice(&device);
    std::lock_guard<std::mutex> guard(lock);
    for (int i = 0; i < n_cache; ++i)
        if (cache[i].device == device && cache[i].fn == (const void*)kernel && cache[i].smem == smem) return cache[i].grid;
    // static (prefetch stage) + dynamic (scene prefix, stack) shared memory may exceed 48 KB.
    // The attribute is a CAP: always raise it to the same ceiling, never to this scene's size
    // (a smaller later scene would otherwise lower it under a cached larger launch).
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024);
    if (e != cudaSuccess) note_launch_error("cudaFuncSetAttribute(MaxDynamicSharedMemorySize)", e, smem, 0);
    const int grid = resident_grid(kernel, smem, sm_count);
    if (n_cache < 256) cache[n_cache++] = Entry{device, (const void*)kernel, smem, grid};
    return grid;
}

// Launch with programmatic stream serialization: the kernel may start while its predecessor in
// the stream drains; it synchronises with pdl_wait() itself.
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, size_t smem, cudaStream_t s, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(unsigned(grid));
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// What the flat bounce kernels get as their FlatPairsU parameter.
static const FlatPairsU& launch_pairs(const PassArgs& a) {
    static const FlatPairsU none{};
    return a.flat_uniform ? *a.upairs : none;
}

// Flat scenes, a bounce after the camera segment's: the three material queues in one launch when the scene has mirror /
// glass (at bounce 0 only their queues hold records: the fused launch shaded the diffuse camera hits), else the diffuse
// queue (bounces >= 1).
template <bool FOLD, bool UNI> static void (*flat_bounce_kernel(const PassArgs& a, bool first))(PassArgs, int, FlatPairsU) {
    if (a.kind_mask & 6u) return first ? bounce_flat_all_kernel<true, FOLD, UNI> : bounce_flat_all_kernel<false, FOLD, UNI>;
    return bounce_flat_kernel<FOLD, UNI>;
}

// Tree scenes only shade here: no scene staging, no dynamic shared memory.
template <int KIND, bool FIRST, bool LAST> static void launch_bounce_k(const PassArgs& a, int bounce, int sm_count, cudaStream_t s) {
    void (*kernel)(PassArgs, int) = bounce_kernel<KIND, FIRST, LAST>;
    const int grid = persistent_grid(kernel, 0, sm_count);
    cudaError_t e = launch_pdl(kernel, grid, 0, s, a, bounce);
    if (e != cudaSuccess) note_launch_error("bounce kernel launch", e, 0, grid);
}

template <int KIND> static void launch_bounce_fl(const PassArgs& a, int bounce, int sm_count, cudaStream_t s) {
    const bool first = bounce == 0, last = bounce + 1 >= a.max_depth;
    if (first && last) launch_bounce_k<KIND, true, true>(a, bounce, sm_count, s);
    else if (first) launch_bounce_k<KIND, true, false>(a, bounce, sm_count, s);
    else if (last) launch_bounce_k<KIND, false, true>(a, bounce, sm_count, s);
    else launch_bounce_k<KIND, false, false>(a, bounce, sm_count, s);
}

} // namespace

template <bool LIST> static void (*raygen_extend_k(const PassArgs& a))(PassArgs) {
    if (a.walk == 6) return raygen_extend_kernel<false, 6, LIST>;
    if (a.walk == 5) return raygen_extend_kernel<false, 5, LIST>;
    if (a.walk == 3) return raygen_extend_kernel<false, 3, LIST>;
    if (a.walk == 2) return a.coop_leaf ? raygen_extend_kernel<true, 2, LIST> : raygen_extend_kernel<false, 2, LIST>;
    return a.coop_leaf ? raygen_extend_kernel<true, 1, LIST> : raygen_extend_kernel<false, 1, LIST>;
}

void launch_raygen_extend(const PassArgs& a, int sm_count, cudaStream_t s) {
    const size_t smem = path_smem_bytes(a);
    void (*kernel)(PassArgs) = a.tiles ? raygen_extend_k<true>(a) : raygen_extend_k<false>(a);
    const int grid = persistent_grid(kernel, smem, sm_count);
    const cudaError_t e = launch_pdl(kernel, grid, smem, s, a);
    if (e != cudaSuccess) note_launch_error("raygen_extend kernel launch", e, smem, grid);
}

void launch_trace(const PassArgs& a, int bounce, int sm_count, cudaStream_t s) {
    const size_t smem = path_smem_bytes(a);
    void (*kernel)(PassArgs, int);
    if (a.walk == 6) kernel = trace_kernel<false, 6, 3>;
    else if (a.walk == 5) kernel = a.trace_occ == 4 ? trace_kernel<false, 5, 4> : trace_kernel<false, 5, 3>;
    else if (a.walk == 3) kernel = a.trace_occ == 4 ? trace_kernel<false, 3, 4> : trace_kernel<false, 3, 3>;
    else if (a.walk == 2) kernel = a.coop_leaf ? trace_kernel<true, 2> : trace_kernel<false, 2>;
    else kernel = a.coop_leaf ? (a.trace_occ == 4 ? trace_kernel<true, 1, 4> : trace_kernel<true, 1, 3>) : trace_kernel<false, 1>;
    const int grid = persistent_grid(kernel, smem, sm_count);
    cudaError_t e = launch_pdl(kernel, grid, smem, s, a, bounce);
    if (e != cudaSuccess) note_launch_error("trace kernel launch", e, smem, grid);
}

bool path_scene_is_flat(const PassArgs& a) { return all_staged(a); }

template <bool LIST> static void (*first_fused_k(const PassArgs& a))(PassArgs, FlatPairsU) {
    const bool u = a.flat_uniform != 0;
    if (a.kind_mask & 6u) // mirror / glass in the scene: diffuse camera hits shaded in place, specular ones queued
        return a.max_depth <= 1 ? (u ? bounce_flat_fused_kernel<true, false, true, true, LIST> : bounce_flat_fused_kernel<true, false, true, false, LIST>)
               : a.fold_last    ? (u ? bounce_flat_fused_kernel<false, true, true, true, LIST> : bounce_flat_fused_kernel<false, true, true, false, LIST>)
                                : (u ? bounce_flat_fused_kernel<false, false, true, true, LIST> : bounce_flat_fused_kernel<false, false, true, false, LIST>);
    return a.max_depth <= 1 ? (u ? bounce_flat_fused_kernel<true, false, false, true, LIST> : bounce_flat_fused_kernel<true, false, false, false, LIST>)
           : a.fold_last    ? (u ? bounce_flat_fused_kernel<false, true, false, true, LIST> : bounce_flat_fused_kernel<false, true, false, false, LIST>)
                            : (u ? bounce_flat_fused_kernel<false, false, false, true, LIST> : bounce_flat_fused_kernel<false, false, false, false, LIST>);
}

void launch_bounce_first_fused(const PassArgs& a, int sm_count, cudaStream_t s) {
    const size_t smem = path_smem_bytes(a);
    void (*kernel)(PassArgs, FlatPairsU) = a.tiles ? first_fused_k<true>(a) : first_fused_k<false>(a);
    const int grid = persistent_grid(kernel, smem, sm_count);
    cudaError_t e = launch_pdl(kernel, grid, smem, s, a, launch_pairs(a));
    if (e != cudaSuccess) note_launch_error("fused first bounce kernel launch", e, smem, grid);
}

bool launch_bounce_flat(const PassArgs& a, int bounce, int sm_count, cudaStream_t s) {
    if (!(a.kind_mask & 7u)) return false; // no surface a path goes on from
    const size_t smem = path_smem_bytes(a);
    const bool first = bounce == 0;
    void (*kernel)(PassArgs, int, FlatPairsU);
    if (a.fold_last) kernel = a.flat_uniform ? flat_bounce_kernel<true, true>(a, first) : flat_bounce_kernel<true, false>(a, first);
    else kernel = a.flat_uniform ? flat_bounce_kernel<false, true>(a, first) : flat_bounce_kernel<false, false>(a, first);
    const int grid = persistent_grid(kernel, smem, sm_count);
    cudaError_t e = launch_pdl(kernel, grid, smem, s, a, bounce, launch_pairs(a));
    if (e != cudaSuccess) note_launch_error("flat bounce kernel launch", e, smem, grid);
    return true;
}

bool launch_bounce(const PassArgs& a, int bounce, int kind, int sm_count, cudaStream_t s) {
    const bool last = bounce + 1 >= a.max_depth;
    if (last && kind != Q_DIFFUSE) return false; // nothing to do: no launch
    switch (kind) {
    case Q_DIFFUSE: launch_bounce_fl<Q_DIFFUSE>(a, bounce, sm_count, s); break;
    case Q_MIRROR: launch_bounce_fl<Q_MIRROR>(a, bounce, sm_count, s); break;
    default: launch_bounce_fl<Q_GLASS>(a, bounce, sm_count, s); break;
    }
    return true;
}

const char* path_launch_error() { return g_launch_error[0] ? g_launch_error : nullptr; }
void path_clear_launch_error() { g_launch_error[0] = 0; }

void launch_accumulate(const PassArgs& a, cudaStream_t s) {
    int blocks = int((a.pix_count + kThreads - 1) / kThreads);
    if (blocks < 1) blocks = 1;
    void (*kernel)(PassArgs) = all_staged(a) ? (a.tiles ? accumulate_kernel<true, true> : accumulate_kernel<true, false>)
                                             : (a.tiles ? accumulate_kernel<false, true> : accumulate_kernel<false, false>);
    cudaError_t e = launch_pdl(kernel, blocks, 0, s, a);
    if (e != cudaSuccess) note_launch_error("accumulate kernel launch", e, 0, blocks);
}

void launch_primary(const PassArgs& a, int32_t* ids_l, double* points_l, double* normals_l, int sm_count, cudaStream_t s) {
    if (a.map.n_local_pix == 0) return;
    PassArgs b = a;
    b.coop_leaf = 0; // sequential leaf tests: no cooperative result slots needed
    b.leaf_batch = 4;
    const size_t smem = path_smem_bytes(b);
    void (*kernel)(PassArgs, int32_t*, double*, double*) = all_staged(b) ? primary_kernel<true> : primary_kernel<false>;
    int grid = persistent_grid(kernel, smem, sm_count);
    grid = std::min(grid, (a.map.n_local_pix + kThreads - 1) / kThreads);
    kernel<<<grid, kThreads, smem, s>>>(b, ids_l, points_l, normals_l);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) note_launch_error("primary kernel launch", e, smem, grid);
}

// The same walk, leaf mode and occupancy launch_trace picks for the render, in its any-hit or nearest-hit form.
template <bool ANY> static void (*cast_tree_kernel(const PassArgs& a))(PassArgs, CastArgs) {
    if (a.walk == 6) return cast_kernel<false, 6, ANY, 3>;
    if (a.walk == 5) return a.trace_occ == 4 ? cast_kernel<false, 5, ANY, 4> : cast_kernel<false, 5, ANY, 3>;
    if (a.walk == 3) return a.trace_occ == 4 ? cast_kernel<false, 3, ANY, 4> : cast_kernel<false, 3, ANY, 3>;
    if (a.walk == 2) return a.coop_leaf ? cast_kernel<true, 2, ANY> : cast_kernel<false, 2, ANY>;
    return a.coop_leaf ? (a.trace_occ == 4 ? cast_kernel<true, 1, ANY, 4> : cast_kernel<true, 1, ANY, 3>) : cast_kernel<false, 1, ANY>;
}

void launch_cast(const PassArgs& a, const CastArgs& c, bool any, int sm_count, cudaStream_t s) {
    if (c.n == 0) return;
    const size_t smem = path_smem_bytes(a);
    void (*kernel)(PassArgs, CastArgs) = all_staged(a) ? cast_flat_kernel : (any ? cast_tree_kernel<true>(a) : cast_tree_kernel<false>(a));
    int grid = persistent_grid(kernel, smem, sm_count);
    grid = std::min<int64_t>(grid, (int64_t(c.n) + kThreads - 1) / kThreads);
    kernel<<<grid, kThreads, smem, s>>>(a, c);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) note_launch_error("cast kernel launch", e, smem, grid);
}

void launch_resolve(const TileMap& map, const float* accum, int spp, float* rad_l, uint8_t* rgb_l, cudaStream_t s) {
    if (map.n_local_pix == 0) return;
    resolve_kernel<<<(map.n_local_pix + kThreads - 1) / kThreads, kThreads, 0, s>>>(map, accum, spp, rad_l, rgb_l);
}

void launch_tile_test(const TileMap& map, const float* accum, const uint32_t* list, uint32_t n_active, int n, int spp, float tau,
                      int32_t* tile_n, uint32_t* flag, cudaStream_t s) {
    if (n_active == 0) return;
    const uint32_t blocks = (n_active * 32u + kThreads - 1) / kThreads;
    tile_test_kernel<<<blocks, kThreads, 0, s>>>(map, accum, list, n_active, n, spp, tau, tile_n, flag);
}

void launch_tile_compact(const uint32_t* list, uint32_t n_active, const uint32_t* flag, uint32_t* list_out, uint32_t* count_out,
                         cudaStream_t s) {
    tile_compact_kernel<<<1, 1024, 0, s>>>(list, n_active, flag, list_out, count_out);
}

void launch_resolve_adaptive(const TileMap& map, const float* accum, const int32_t* tile_n, uint8_t* rgb, float* rad, float* var,
                             int32_t* spp, cudaStream_t s) {
    if (map.n_local_pix == 0) return;
    resolve_adaptive_kernel<<<(map.n_local_pix + kThreads - 1) / kThreads, kThreads, 0, s>>>(map, accum, tile_n, rgb, rad, var, spp);
}

} // namespace g19

// path.cu -- host side of G19_MODE_PATH: primitive extraction, the engine's own
// linear octree ("FIXED" semantics of SURVEY.md section 7, hard part 1: true
// bounds, every primitive reachable, nearest hit), and the wavefront driver.
//
// Reference counterpart: the octree build of include/octree.h:75-129 -- which
// loses entities on split and boxes spheres around the origin -- is NOT
// reproduced here; it lives, bug for bug, in scene.cpp for REF mode. This tree
// is what the path tracer traverses:
//   * node boxes are implicit: the root box is Octree::min/max, a node at
//     level l with integer coordinates (ix,iy,iz) spans
//     root_lo + (i, i+1) * root_size * 2^-l per axis (same float expression on
//     host and device, so the boxes tile space without cracks)
//   * records are 8 bytes; the 8 children of a node are contiguous = one 64 B
//     line; nodes are laid out breadth first so the top levels are a prefix
//     that the kernels stage into shared memory
#include "path.h"

#include <algorithm>
#include <cctype>
#include <chrono>
#include <limits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

namespace g19 {

cudaError_t DeviceArray::ensure(size_t need) {
    if (need <= bytes) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    // pad so that 16-byte bulk copies may run past the logical end
    cudaError_t e = cudaMalloc(&p, need + 256);
    if (e == cudaSuccess) bytes = need;
    return e;
}
void DeviceArray::release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
}
cudaError_t PoolArray::ensure(size_t need, cudaStream_t s) {
    if (need <= bytes && p) return cudaSuccess;
    release();
    stream = s;
    cudaError_t e = cudaMallocAsync(&p, need + 256, s);
    if (e == cudaSuccess) bytes = need;
    else p = nullptr;
    return e;
}
void PoolArray::release() {
    if (p) cudaFreeAsync(p, stream);
    p = nullptr;
    bytes = 0;
}
void path_pool_keep() {
    int dev = 0;
    cudaMemPool_t pool;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetDefaultMemPool(&pool, dev) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    unsigned long long keep = 2ull << 30; // what the builders of a 1 M-triangle scene hold at their peak is ~0.5 GB
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    cudaGetLastError();
}

namespace {

struct Box {
    float lo[3], hi[3];
};

struct BuildPrim {
    PrimHot hot;
    PrimCold cold;
    Box box;
    float v[3][3]; // triangle corners (float), for the parallelogram merge
    bool tri;
    int32_t ent[2]; // entity id (push order, as REF mode reports it); a merged parallelogram keeps both triangles' ids:
                    // ent[0] owns the half b1 >= b2 of the parallelogram frame, ent[1] the half b1 < b2
};

// world -> (b1, b2, h) rows for the frame (v0; e1, e2): rows of [e1 e2 n]^-1, n = e1 x e2, translation -M v0
void affine_rows(float* q, const float v0[3], const float e1[3], const float e2[3]) {
    double a[3] = {e1[0], e1[1], e1[2]}, b[3] = {e2[0], e2[1], e2[2]};
    double n[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
    double nn = n[0] * n[0] + n[1] * n[1] + n[2] * n[2];
    for (int k = 0; k < 12; ++k) q[k] = 0.0f; // degenerate: t = 0/0 = NaN -> never hit
    if (!(nn > 0)) return;
    double r0[3] = {(b[1] * n[2] - b[2] * n[1]) / nn, (b[2] * n[0] - b[0] * n[2]) / nn, (b[0] * n[1] - b[1] * n[0]) / nn};
    double r1[3] = {(n[1] * a[2] - n[2] * a[1]) / nn, (n[2] * a[0] - n[0] * a[2]) / nn, (n[0] * a[1] - n[1] * a[0]) / nn};
    double r2[3] = {n[0] / nn, n[1] / nn, n[2] / nn};
    const double* rows[3] = {r0, r1, r2};
    for (int r = 0; r < 3; ++r) {
        for (int k = 0; k < 3; ++k) q[4 * r + k] = float(rows[r][k]);
        q[4 * r + 3] = float(-(rows[r][0] * v0[0] + rows[r][1] * v0[1] + rows[r][2] * v0[2]));
    }
}

float clamp01(double v) { return float(v < 0 ? 0 : (v > 1 ? 1 : v)); }

void add_triangle(std::vector<BuildPrim>& out, const HostTri& t, int material, int entity) {
    BuildPrim p;
    std::memset(&p, 0, sizeof p);
    float v0[3] = {float(t.p1.x), float(t.p1.y), float(t.p1.z)};
    float v1[3] = {float(t.p2.x), float(t.p2.y), float(t.p2.z)};
    float v2[3] = {float(t.p3.x), float(t.p3.y), float(t.p3.z)};
    float e1[3], e2[3];
    for (int k = 0; k < 3; ++k) {
        e1[k] = v1[k] - v0[k];
        e2[k] = v2[k] - v0[k];
    }
    affine_rows(p.hot.q, v0, e1, e2);
    p.hot.q[14] = 1.0f; // kind = triangle
    p.tri = true;
    for (int k = 0; k < 3; ++k) { p.v[0][k] = v0[k]; p.v[1][k] = v1[k]; p.v[2][k] = v2[k]; }
    // geometric normal from the double-precision vertices
    double ax = t.p2.x - t.p1.x, ay = t.p2.y - t.p1.y, az = t.p2.z - t.p1.z;
    double bx = t.p3.x - t.p1.x, by = t.p3.y - t.p1.y, bz = t.p3.z - t.p1.z;
    double nx = ay * bz - az * by, ny = az * bx - ax * bz, nz = ax * by - ay * bx;
    double len = std::sqrt(nx * nx + ny * ny + nz * nz);
    if (len > 0) { nx /= len; ny /= len; nz /= len; }
    p.cold.n[0] = float(nx); p.cold.n[1] = float(ny); p.cold.n[2] = float(nz);
    p.cold.material = material;
    p.ent[0] = p.ent[1] = entity;
    for (int k = 0; k < 3; ++k) {
        p.box.lo[k] = std::min(v0[k], std::min(v1[k], v2[k]));
        p.box.hi[k] = std::max(v0[k], std::max(v1[k], v2[k]));
    }
    out.push_back(p);
}

void add_sphere(std::vector<BuildPrim>& out, const HostEntity& e, int material, int entity) {
    BuildPrim p;
    std::memset(&p, 0, sizeof p);
    float c[3] = {float(e.pos.x), float(e.pos.y), float(e.pos.z)};
    float* q = p.hot.q;
    q[0] = c[0]; q[1] = c[1]; q[2] = c[2]; q[3] = e.radius;
    q[14] = 0.0f; // kind = sphere
    p.tri = false;
    p.cold.material = material;
    p.ent[0] = p.ent[1] = entity;
    for (int k = 0; k < 3; ++k) {
        p.box.lo[k] = c[k] - e.radius;
        p.box.hi[k] = c[k] + e.radius;
    }
    out.push_back(p);
}

struct Pending {
    uint32_t node;
    int level;
    uint32_t ix, iy, iz;
    std::vector<uint32_t> prims;
};

bool overlaps(const Box& a, const float lo[3], const float hi[3]) {
    for (int k = 0; k < 3; ++k)
        if (a.hi[k] < lo[k] || a.lo[k] > hi[k]) return false;
    return true;
}

} // namespace

// Cell bounds: the ONE expression shared with the device (path_kernels.cu cell_lo/cell_hi).
static inline float cell_edge(float root_lo, float root_size, int level, uint32_t i) {
    return root_lo + float(i) * std::ldexp(root_size, -level);
}

void path_tuning_from_env(PathTuning& t) {
    static const char* const keys[] = {"lanes", "pass_slots", "leaf_max", "refill", "coop_leaf", "walk_steps", "leaf_batch",
                                       "tree_build", "debug_tree", "walk", "trace_occ", "top_level", "ref_heavy", "sort_rays", "upload_threads", "bvh_leaf", "bvh_spec", "bvh_stack", "overlap_frames", "flat_uniform"};
    for (const char* k : keys) {
        std::string env = "G19_";
        for (const char* c = k; *c; ++c) env += char(std::toupper(*c));
        if (const char* v = std::getenv(env.c_str())) path_tuning_set(t, k, v);
    }
}

bool path_tuning_set(PathTuning& t, const char* key, const char* value) {
    const PathTuning def;
    const std::string k = key ? key : "";
    auto num = [&](int dflt, int lo, int hi) { return value ? std::max(lo, std::min(hi, std::atoi(value))) : dflt; };
    if (k == "lanes") t.lanes = num(def.lanes, 1, kMaxLanes);
    else if (k == "pass_slots") t.pass_slots = value ? std::max<long long>(kTilePix, std::atoll(value)) : 0;
    else if (k == "leaf_max") t.leaf_max = num(def.leaf_max, 1, 1 << 20);
    else if (k == "refill") t.refill = num(def.refill, 1, 32);
    else if (k == "coop_leaf") t.coop_leaf = num(def.coop_leaf, 0, 1);
    else if (k == "walk_steps") t.walk_steps = num(def.walk_steps, 0, 16);
    else if (k == "leaf_batch") t.leaf_batch = num(def.leaf_batch, 0, 16);
    else if (k == "tree_build") t.tree_build = !value ? -1 : (std::strcmp(value, "device") == 0 ? 1 : (std::strcmp(value, "host") == 0 ? 0 : -1));
    else if (k == "debug_tree") t.debug_tree = value ? 1 : 0;
    else if (k == "walk") { t.walk = num(def.walk, 1, 4); if (t.walk == 2) t.walk = 1; }
    else if (k == "trace_occ") t.trace_occ = num(def.trace_occ, 3, 4);
    else if (k == "top_level") t.top_level = num(def.top_level, 0, 8);
    else if (k == "overlap_frames") t.overlap_frames = num(def.overlap_frames, 0, 1);
    else if (k == "flat_uniform") t.flat_uniform = num(def.flat_uniform, 0, 1);
    else if (k == "bvh_stack") t.bvh_stack = num(def.bvh_stack, 4, 64);
    else if (k == "bvh_spec") t.bvh_spec = num(def.bvh_spec, 0, 3);
    else if (k == "bvh_leaf") t.bvh_leaf = num(def.bvh_leaf, 1, 8);
    else if (k == "upload_threads") t.upload_threads = num(def.upload_threads, 0, 64);
    else if (k == "sort_rays") t.sort_rays = num(def.sort_rays, -1, 1);
    else if (k == "ref_heavy") t.ref_heavy = num(def.ref_heavy, 0, 1 << 30);
    else return false;
    return true;
}

// Primitive PAIRS for the packed-FP32 loops of path_kernels.cu (plane_pairs / sphere_roots2): `hot[first ...]` holds
// n_par parallelograms, then n_tri triangles, then n_sph spheres. Planar pair = rows a, b, c with every coefficient a
// float2 (primitive 2j, 2j+1), 96 B; sphere pair = (-centre, radius^2) as float2s, 32 B. Each kind group is padded to an
// even count with NaNs: every comparison on a NaN fails, so a padding record is never hit.
static void build_pairs(const std::vector<PrimHot>& hot, size_t first, size_t n_par, size_t n_tri, size_t n_sph, std::vector<float>& pairs) {
    const float nan = std::numeric_limits<float>::quiet_NaN();
    auto planar = [&](size_t f, size_t count) {
        for (size_t k = 0; k < count; k += 2)
            for (int c = 0; c < 12; ++c)
                for (size_t e = 0; e < 2; ++e) pairs.push_back(k + e < count ? hot[f + k + e].q[c] : nan);
    };
    planar(first, n_par);
    planar(first + n_par, n_tri);
    const size_t s0 = first + n_par + n_tri;
    for (size_t k = 0; k < n_sph; k += 2)
        for (int c = 0; c < 4; ++c)
            for (size_t e = 0; e < 2; ++e) {
                float v = nan;
                if (k + e < n_sph) v = c < 3 ? -hot[s0 + k + e].q[c] : hot[s0 + k + e].q[3] * hot[s0 + k + e].q[3];
                pairs.push_back(v);
            }
}

int path_upload(PathSceneBuffers& b, const g19_scene& scene, const PathTuning& tune, cudaStream_t stream, std::string& err) {
    const auto t_start = std::chrono::steady_clock::now();
    ++b.upload_serial;
    path_pool_keep();
    // Extraction runs on the host's cores, a contiguous range of entities per thread with its own primitive, material
    // and light lists (a 1 M-triangle mesh: 0.26 s single-threaded); the ranges are then joined in entity order, with the
    // "same material as the previous entity" rule applied across the seams too, so the result does not depend on the
    // number of threads.
    struct Extracted {
        std::vector<BuildPrim> prims;
        std::vector<MaterialD> materials;
        std::vector<LightD> lights;
        bool has_bsdf[4] = {false, false, false, false};
    };
    auto extract = [&](size_t eb, size_t ee, Extracted& out) {
        std::vector<BuildPrim>& prims = out.prims;
        std::vector<MaterialD>& materials = out.materials;
        std::vector<LightD>& lights = out.lights;
        bool* has_bsdf = out.has_bsdf;
        for (size_t ei = eb; ei < ee; ++ei) {
            const HostEntity& e = scene.ents[ei];
            if (!e.in_tree) continue; // rejected by Octree::push_back: not part of the scene
            MaterialD m;
            m.albedo[0] = clamp01(e.desc.color[0]);
            m.albedo[1] = clamp01(e.desc.color[1]);
            m.albedo[2] = clamp01(e.desc.color[2]);
            m.bsdf = e.desc.bsdf;
            if (m.bsdf < 0 || m.bsdf > 3) m.bsdf = G19_BSDF_DIFFUSE;
            m.emission[0] = e.desc.emission[0];
            m.emission[1] = e.desc.emission[1];
            m.emission[2] = e.desc.emission[2];
            m.ior = e.desc.ior > 0 ? e.desc.ior : 1.5f;
            // one material per entity, deduplicated against the previous one (meshes)
            int mi;
            if (!materials.empty() && std::memcmp(&materials.back(), &m, sizeof m) == 0) mi = int(materials.size()) - 1;
            else { materials.push_back(m); mi = int(materials.size()) - 1; }
            has_bsdf[m.bsdf] = true;
            // material index and class ride in the spare words of the hot record
            auto tag = [&](BuildPrim& p) {
                int32_t mat_bits = mi, bsdf_bits = m.bsdf;
                p.cold.ior = m.ior;
                p.cold.albedo[0] = m.albedo[0]; p.cold.albedo[1] = m.albedo[1]; p.cold.albedo[2] = m.albedo[2];
                std::memcpy(&p.hot.q[12], &mat_bits, 4);
                std::memcpy(&p.hot.q[13], &bsdf_bits, 4);
            };
            if (e.combine == COMBINE_SPHERE) {
                add_sphere(prims, e, mi, int(ei));
                tag(prims.back());
            } else {
                // the triangles REF mode tests (from `first_tested`: ExpSphere skips its first one) -- or, with
                // G19_SHAPES_FIXED, the triangles the constructor meant to build (fixed_shapes.cpp)
                std::vector<HostTri> fixed;
                const bool use_fixed = scene.shapes == G19_SHAPES_FIXED && fixed_triangles(e.desc, fixed);
                const std::vector<HostTri>& tris = use_fixed ? fixed : e.tris;
                for (size_t t = use_fixed ? 0 : size_t(e.first_tested); t < tris.size(); ++t) {
                    add_triangle(prims, tris[t], mi, int(ei));
                    tag(prims.back());
                    if (m.bsdf == G19_BSDF_EMITTER) {
                        const BuildPrim& p = prims.back();
                        LightD l;
                        std::memset(&l, 0, sizeof l);
                        const HostTri& ht = tris[t];
                        const float fv0[3] = {float(ht.p1.x), float(ht.p1.y), float(ht.p1.z)};
                        const float fv1[3] = {float(ht.p2.x), float(ht.p2.y), float(ht.p2.z)};
                        const float fv2[3] = {float(ht.p3.x), float(ht.p3.y), float(ht.p3.z)};
                        for (int k = 0; k < 3; ++k) {
                            l.v0[k] = fv0[k];
                            l.e1[k] = fv1[k] - fv0[k];
                            l.e2[k] = fv2[k] - fv0[k];
                        }
                        float cx = l.e1[1] * l.e2[2] - l.e1[2] * l.e2[1];
                        float cy = l.e1[2] * l.e2[0] - l.e1[0] * l.e2[2];
                        float cz = l.e1[0] * l.e2[1] - l.e1[1] * l.e2[0];
                        l.area = 0.5f * std::sqrt(cx * cx + cy * cy + cz * cz);
                        l.prim = -1; // (unused: primitive ids are final only after the merge / kind sort below)
                        l.n[0] = p.cold.n[0]; l.n[1] = p.cold.n[1]; l.n[2] = p.cold.n[2];
                        l.emission[0] = m.emission[0]; l.emission[1] = m.emission[1]; l.emission[2] = m.emission[2];
                        if (l.area > 0) lights.push_back(l);
                    }
                }
            }
        }
    };
    const size_t n_ents = scene.ents.size();
    unsigned hw = std::thread::hardware_concurrency();
    size_t n_threads = n_ents < (size_t(1) << 15) ? 1 : std::min<size_t>(hw ? hw : 4, 16);
    if (tune.upload_threads > 0) n_threads = std::min<size_t>(size_t(tune.upload_threads), std::max<size_t>(1, n_ents)); // tuning / test knob
    std::vector<Extracted> parts(n_threads);
    {
        const size_t chunk = (n_ents + n_threads - 1) / n_threads;
        std::atomic<bool> failed{false}; // an exception (out of host memory) must not escape a worker thread
        auto guarded = [&](size_t eb, size_t ee, Extracted& out) {
            try {
                extract(eb, ee, out);
            } catch (...) {
                failed.store(true);
            }
        };
        std::vector<std::thread> pool;
        for (size_t t = 1; t < n_threads; ++t) {
            const size_t eb = std::min(n_ents, t * chunk), ee = std::min(n_ents, eb + chunk);
            pool.emplace_back([&, eb, ee, t] { guarded(eb, ee, parts[t]); });
        }
        guarded(0, std::min(n_ents, chunk), parts[0]);
        for (std::thread& th : pool) th.join();
        if (failed.load()) {
            err = "path_upload: out of host memory while extracting primitives";
            return G19_ERR_LIMIT;
        }
    }
    std::vector<BuildPrim> prims;
    std::vector<MaterialD> materials;
    std::vector<LightD> lights;
    for (bool& h : b.has_bsdf) h = false;
    if (n_threads == 1) {
        prims.swap(parts[0].prims);
        materials.swap(parts[0].materials);
        lights.swap(parts[0].lights);
        for (int k = 0; k < 4; ++k) b.has_bsdf[k] = parts[0].has_bsdf[k];
    } else {
        size_t total = 0;
        std::vector<size_t> prim_at(n_threads);
        std::vector<int> mat_shift(n_threads);
        for (size_t t = 0; t < n_threads; ++t) {
            Extracted& e = parts[t];
            prim_at[t] = total;
            total += e.prims.size();
            for (int k = 0; k < 4; ++k) b.has_bsdf[k] = b.has_bsdf[k] || e.has_bsdf[k];
            // local material i becomes global i + shift; the first local one folds into the previous part's last when equal
            size_t first = 0;
            if (!materials.empty() && !e.materials.empty() && std::memcmp(&materials.back(), &e.materials[0], sizeof(MaterialD)) == 0) first = 1;
            mat_shift[t] = int(materials.size()) - int(first);
            materials.insert(materials.end(), e.materials.begin() + first, e.materials.end());
            lights.insert(lights.end(), e.lights.begin(), e.lights.end());
        }
        prims.resize(total);
        std::vector<std::thread> pool;
        for (size_t t = 0; t < n_threads; ++t)
            pool.emplace_back([&, t] {
                const int shift = mat_shift[t];
                BuildPrim* out = prims.data() + prim_at[t];
                for (BuildPrim p : parts[t].prims) {
                    p.cold.material += shift;
                    int32_t mat_bits;
                    std::memcpy(&mat_bits, &p.hot.q[12], 4);
                    mat_bits += shift;
                    std::memcpy(&p.hot.q[12], &mat_bits, 4);
                    *out++ = p;
                }
                std::vector<BuildPrim>().swap(parts[t].prims);
            });
        for (std::thread& th : pool) th.join();
    }
    for (LightD& l : lights) l.pdf_pick = 1.0f / float(lights.size());

    // ---- merge coplanar triangle pairs into parallelograms --------------------------------
    // Two consecutive triangles with the same material that share an edge s1-s2 and whose
    // other corners u, v satisfy s1 + s2 = u + v tile the parallelogram (s1; u-s1, v-s1): one
    // primitive test (b1, b2 in [0,1]) instead of two. Walls, floors and light panels built
    // as triangle pairs (the Cornell configs) halve their test count; a curved mesh keeps
    // its triangles. The oracle still tests the triangles: the union is the same point set.
    {
        std::vector<BuildPrim> merged;
        merged.reserve(prims.size());
        for (size_t i = 0; i < prims.size(); ++i) {
            bool done = false;
            if (i + 1 < prims.size() && prims[i].tri && prims[i + 1].tri &&
                prims[i].cold.material == prims[i + 1].cold.material) {
                const BuildPrim &A = prims[i], &B = prims[i + 1];
                int sa[2], sb[2], ns = 0;
                for (int x = 0; x < 3; ++x)
                    for (int y = 0; y < 3; ++y)
                        if (ns < 2 && A.v[x][0] == B.v[y][0] && A.v[x][1] == B.v[y][1] && A.v[x][2] == B.v[y][2]) {
                            sa[ns] = x; sb[ns] = y; ++ns;
                        }
                if (ns == 2 && sa[0] != sa[1] && sb[0] != sb[1]) {
                    const float* s1 = A.v[sa[0]];
                    const float* s2 = A.v[sa[1]];
                    const float* u = A.v[3 - sa[0] - sa[1]];
                    const float* v = B.v[3 - sb[0] - sb[1]];
                    double scale = 0, gap = 0;
                    for (int k = 0; k < 3; ++k) {
                        gap = std::max(gap, std::fabs(double(s1[k]) + s2[k] - u[k] - v[k]));
                        scale = std::max(scale, std::fabs(double(s2[k]) - s1[k]));
                    }
                    if (gap <= 1e-6 * scale && scale > 0) {
                        BuildPrim q = A;
                        float e1[3], e2[3];
                        for (int k = 0; k < 3; ++k) { e1[k] = u[k] - s1[k]; e2[k] = v[k] - s1[k]; }
                        affine_rows(q.hot.q, s1, e1, e2);
                        q.hot.q[14] = 2.0f; // kind = parallelogram
                        q.hot.q[3] -= 0.5f; // centred coordinates: inside <=> max(|b1|, |b2|) <= 1/2
                        q.hot.q[7] -= 0.5f;
                        for (int k = 0; k < 3; ++k) {
                            q.box.lo[k] = std::min(A.box.lo[k], B.box.lo[k]);
                            q.box.hi[k] = std::max(A.box.hi[k], B.box.hi[k]);
                        }
                        q.tri = false;
                        q.ent[0] = A.ent[0]; // A = (s1, s2, u): u sits at (b1, b2) = (1, 0), so A is the half b1 >= b2
                        q.ent[1] = B.ent[0];
                        merged.push_back(q);
                        ++i;
                        done = true;
                    }
                }
            }
            if (!done) merged.push_back(prims[i]);
        }
        prims.swap(merged);
    }
    if (prims.size() >= 0x7fffffffu) {
        err = "too many primitives";
        return G19_ERR_LIMIT;
    }

    const auto t_prims = std::chrono::steady_clock::now();
    // ---- linear octree, breadth first ------------------------------------------
    // measured on the 1M-triangle heightfield, ms per 1080p x 32 spp frame at 4 / 6 / 8 / 12 / 16 / 32: 107.3 / 107.7 / 107.6 /
    // 110.6 / 114.6 / 141.3 (an earlier walk, before the fixed-trip rounds, preferred 16)
    const int kLeafMax = tune.leaf_max;
    float root_lo[3] = {float(scene.rmin.x), float(scene.rmin.y), float(scene.rmin.z)};
    float root_hi[3] = {float(scene.rmax.x), float(scene.rmax.y), float(scene.rmax.z)};
    for (int k = 0; k < 3; ++k) { // the root box must enclose every primitive
        for (const BuildPrim& p : prims) {
            root_lo[k] = std::min(root_lo[k], p.box.lo[k]);
            root_hi[k] = std::max(root_hi[k], p.box.hi[k]);
        }
    }
    float root_size[3] = {root_hi[0] - root_lo[0], root_hi[1] - root_lo[1], root_hi[2] - root_lo[2]};
    for (int k = 0; k < 3; ++k) { // nudge up so that lo + 1 * size >= hi after rounding
        while (root_lo[k] + root_size[k] < root_hi[k]) root_size[k] = std::nextafter(root_size[k], INFINITY);
        if (!(root_size[k] > 0)) root_size[k] = 1.0f;
    }
    // Large scenes build the tree on the device (tree_build.cu: same rules, bit-identical result);
    // small ones -- and G19_TREE_BUILD=host -- here. The host builder is also the test's checker.
    bool on_device = prims.size() >= 4096;
    if (tune.tree_build >= 0) on_device = tune.tree_build == 1;
    PathNodeD* dev_nodes = nullptr;
    uint32_t* dev_index = nullptr;
    uint32_t dev_n_nodes = 0, dev_n_index = 0;
    int dev_depth = 0;
    if (on_device) {
        std::vector<float> boxes(prims.size() * 6);
        for (size_t i = 0; i < prims.size(); ++i)
            for (int k = 0; k < 3; ++k) {
                boxes[6 * i + k] = prims[i].box.lo[k];
                boxes[6 * i + 3 + k] = prims[i].box.hi[k];
            }
        PoolArray d_boxes;
        cudaError_t be = d_boxes.ensure(boxes.size() * sizeof(float) + 16, stream);
        if (be == cudaSuccess) be = cudaMemcpyAsync(d_boxes.p, boxes.data(), boxes.size() * sizeof(float), cudaMemcpyHostToDevice, stream);
        if (be == cudaSuccess) be = cudaStreamSynchronize(stream);
        if (be != cudaSuccess) {
            err = std::string("path_upload (boxes): ") + cudaGetErrorString(be);
            d_boxes.release();
            return G19_ERR_CUDA;
        }
        int rc = path_build_tree_device(static_cast<const float*>(d_boxes.p), uint32_t(prims.size()), root_lo, root_size, kLeafMax,
                                        kMaxTreeDepth, stream, &dev_nodes, &dev_n_nodes, &dev_index, &dev_n_index, &dev_depth, err);
        d_boxes.release();
        if (rc != G19_OK) return rc;
        if (dev_n_nodes == 1) { // a flat scene after all: the host path sorts it by kind
            cudaFree(dev_nodes);
            cudaFree(dev_index);
            dev_nodes = nullptr;
            dev_index = nullptr;
            on_device = false;
        }
    }
    std::vector<PathNodeD> nodes(1);
    std::vector<uint32_t> index;
    std::vector<Pending> frontier, next;
    if (!on_device) { // the host builder starts from the root; a device-built tree leaves the frontier empty
        Pending root;
        root.node = 0;
        root.level = 0;
        root.ix = root.iy = root.iz = 0;
        root.prims.resize(prims.size());
        for (size_t i = 0; i < prims.size(); ++i) root.prims[i] = uint32_t(i);
        frontier.push_back(std::move(root));
    }
    int tree_depth = 0;
    while (!frontier.empty()) {
        next.clear();
        for (Pending& n : frontier) {
            bool leaf = int(n.prims.size()) <= kLeafMax || n.level >= kMaxTreeDepth;
            std::vector<uint32_t> child[8];
            if (!leaf) {
                size_t refs = 0;
                for (int c = 0; c < 8; ++c) {
                    uint32_t cx = 2 * n.ix + (c & 1), cy = 2 * n.iy + ((c >> 1) & 1), cz = 2 * n.iz + ((c >> 2) & 1);
                    float lo[3] = {cell_edge(root_lo[0], root_size[0], n.level + 1, cx),
                                   cell_edge(root_lo[1], root_size[1], n.level + 1, cy),
                                   cell_edge(root_lo[2], root_size[2], n.level + 1, cz)};
                    float hi[3] = {cell_edge(root_lo[0], root_size[0], n.level + 1, cx + 1),
                                   cell_edge(root_lo[1], root_size[1], n.level + 1, cy + 1),
                                   cell_edge(root_lo[2], root_size[2], n.level + 1, cz + 1)};
                    for (uint32_t pi : n.prims)
                        if (overlaps(prims[pi].box, lo, hi)) child[c].push_back(pi);
                    refs += child[c].size();
                }
                // splitting must pay: stop when the children mostly duplicate the parent
                if (refs >= 3 * n.prims.size()) leaf = true;
            }
            if (leaf) {
                nodes[n.node].first = uint32_t(index.size());
                nodes[n.node].count = uint32_t(n.prims.size()) | kLeafBit;
                index.insert(index.end(), n.prims.begin(), n.prims.end());
                continue;
            }
            uint32_t base = uint32_t(nodes.size());
            nodes[n.node].first = base;
            nodes[n.node].count = 0;
            nodes.resize(nodes.size() + 8);
            tree_depth = std::max(tree_depth, n.level + 1);
            for (int c = 0; c < 8; ++c) {
                Pending ch;
                ch.node = base + c;
                ch.level = n.level + 1;
                ch.ix = 2 * n.ix + (c & 1);
                ch.iy = 2 * n.iy + ((c >> 1) & 1);
                ch.iz = 2 * n.iz + ((c >> 2) & 1);
                ch.prims = std::move(child[c]);
                next.push_back(std::move(ch));
            }
        }
        frontier.swap(next);
    }

    const auto t_tree = std::chrono::steady_clock::now();
    if (tune.debug_tree && on_device) { // statistics need the arrays on the host
        nodes.resize(dev_n_nodes);
        index.resize(dev_n_index);
        cudaMemcpy(nodes.data(), dev_nodes, size_t(dev_n_nodes) * sizeof(PathNodeD), cudaMemcpyDeviceToHost);
        cudaMemcpy(index.data(), dev_index, size_t(dev_n_index) * sizeof(uint32_t), cudaMemcpyDeviceToHost);
        tree_depth = dev_depth;
    }
    if (tune.debug_tree) {
        std::fprintf(stderr, "[g19] path_upload: %zu primitives extracted in %.1f ms, tree built on the %s in %.1f ms\n", prims.size(),
                     std::chrono::duration<double, std::milli>(t_prims - t_start).count(), on_device ? "device" : "host",
                     std::chrono::duration<double, std::milli>(t_tree - t_prims).count());
        size_t leaves = 0, empty = 0, biggest = 0;
        for (const PathNodeD& n : nodes)
            if (n.count & kLeafBit) {
                size_t c = n.count & ~kLeafBit;
                if (c) { ++leaves; biggest = std::max(biggest, c); } else ++empty;
            }
        std::fprintf(stderr, "[g19] path octree: %zu prims, %zu nodes, depth %d, %zu leaves (+%zu empty), %zu refs "
                             "(%.2f per prim, %.1f per leaf, max %zu)\n",
                     prims.size(), nodes.size(), tree_depth, leaves, empty, index.size(),
                     double(index.size()) / double(std::max<size_t>(1, prims.size())),
                     double(index.size()) / double(std::max<size_t>(1, leaves)), biggest);
    }
    // A flat scene (the whole scene is one leaf) is sorted parallelograms | triangles | spheres so
    // that the kernels walk three branch-free loops; the leaf position stays the primitive id.
    int n_par = 0, n_tri = 0;
    if (!on_device && nodes.size() == 1) {
        auto rank = [](const BuildPrim& p) { return p.hot.q[14] == 2.0f ? 0 : (p.hot.q[14] == 1.0f ? 1 : 2); };
        std::stable_sort(prims.begin(), prims.end(), [&](const BuildPrim& x, const BuildPrim& y) { return rank(x) < rank(y); });
        for (const BuildPrim& p : prims) {
            if (rank(p) == 0) ++n_par;
            else if (rank(p) == 1) ++n_tri;
        }
        for (size_t i = 0; i < index.size(); ++i) index[i] = uint32_t(i);
    }
    std::vector<PrimHot> hot(prims.size());
    std::vector<PrimCold> cold(prims.size());
    std::vector<int32_t> prim_entity(2 * prims.size());
    for (size_t i = 0; i < prims.size(); ++i) {
        hot[i] = prims[i].hot;
        cold[i] = prims[i].cold;
        prim_entity[2 * i] = prims[i].ent[0];
        prim_entity[2 * i + 1] = prims[i].ent[1];
    }
    // Flat scenes: the same records as primitive PAIRS for the packed-FP32 (FFMA2) loops of
    // trace_flat -- planar pair = rows a, b, c with every coefficient a float2 (primitive 2j, 2j+1),
    // 96 B; sphere pair = (-centre, radius^2) as float2s, 32 B. Each kind group is padded to an even
    // count with NaNs: every comparison on a NaN fails, so a padding record is never hit.
    std::vector<float> pairs;
    if (!on_device && nodes.size() == 1) build_pairs(hot, 0, size_t(n_par), size_t(n_tri), hot.size() - size_t(n_par) - size_t(n_tri), pairs);
    {
        const size_t p_par = (size_t(n_par) + 1) / 2, p_tri = (size_t(n_tri) + 1) / 2;
        const size_t p_sph = (hot.size() - size_t(n_par) - size_t(n_tri) + 1) / 2;
        b.upairs = FlatPairsU{};
        b.upairs_fit = !pairs.empty() && p_par <= size_t(kUniPlanarPairs) && p_tri <= size_t(kUniPlanarPairs) &&
                       p_sph <= size_t(kUniSpherePairs);
        if (b.upairs_fit) {
            const float* src = pairs.data();
            std::memcpy(b.upairs.par, src, p_par * sizeof b.upairs.par[0]);
            src += p_par * 24;
            std::memcpy(b.upairs.tri, src, p_tri * sizeof b.upairs.tri[0]);
            src += p_tri * 24;
            std::memcpy(b.upairs.sph, src, p_sph * sizeof b.upairs.sph[0]);
        }
    }
    auto up = [&](DeviceArray& d, const void* src, size_t bytes) -> cudaError_t {
        cudaError_t e = d.ensure(bytes ? bytes : 16);
        if (e != cudaSuccess || !bytes) return e;
        return cudaMemcpyAsync(d.p, src, bytes, cudaMemcpyHostToDevice, stream);
    };
    cudaError_t e;
    if (on_device) { // the arrays are already in HBM: adopt them
        b.nodes.release();
        b.prim_index.release();
        b.nodes.p = dev_nodes;
        b.nodes.bytes = size_t(dev_n_nodes) * sizeof(PathNodeD);
        b.prim_index.p = dev_index;
        b.prim_index.bytes = size_t(dev_n_index) * sizeof(uint32_t);
    }
    if ((!on_device && ((e = up(b.nodes, nodes.data(), nodes.size() * sizeof(PathNodeD))) != cudaSuccess ||
                        (e = up(b.prim_index, index.data(), index.size() * sizeof(uint32_t))) != cudaSuccess)) ||
        (e = up(b.hot, hot.data(), hot.size() * sizeof(PrimHot))) != cudaSuccess ||
        (e = up(b.cold, cold.data(), cold.size() * sizeof(PrimCold))) != cudaSuccess ||
        (e = up(b.pairs, pairs.data(), pairs.size() * sizeof(float))) != cudaSuccess ||
        (e = up(b.prim_entity, prim_entity.data(), prim_entity.size() * sizeof(int32_t))) != cudaSuccess ||
        (e = up(b.materials, materials.data(), materials.size() * sizeof(MaterialD))) != cudaSuccess ||
        (e = up(b.lights, lights.data(), lights.size() * sizeof(LightD))) != cudaSuccess ||
        (e = cudaStreamSynchronize(stream)) != cudaSuccess) {
        err = std::string("path_upload: ") + cudaGetErrorString(e);
        return G19_ERR_CUDA;
    }
    if (tune.debug_tree)
        std::fprintf(stderr, "[g19] path_upload: record arrays uploaded %.1f ms after the tree\n",
                     std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_tree).count());
    PathSceneD& v = b.view;
    v.nodes = static_cast<const PathNodeD*>(b.nodes.p);
    v.index = static_cast<const uint32_t*>(b.prim_index.p);
    v.hot = static_cast<const PrimHot*>(b.hot.p);
    v.cold = static_cast<const PrimCold*>(b.cold.p);
    v.materials = static_cast<const MaterialD*>(b.materials.p);
    v.lights = static_cast<const LightD*>(b.lights.p);
    v.prim_entity = static_cast<const int32_t*>(b.prim_entity.p);
    v.n_nodes = on_device ? int32_t(dev_n_nodes) : int32_t(nodes.size());
    v.n_index = on_device ? int32_t(dev_n_index) : int32_t(index.size());
    if (on_device) tree_depth = dev_depth;
    v.n_prims = int32_t(prims.size());
    v.n_lights = int32_t(lights.size());
    v.tree_depth = tree_depth;
    // direct index over the first levels for the walk's descents (only worth it for a deep tree)
    v.top = nullptr;
    v.top_level = std::min(tune.top_level, tree_depth - 2);
    if (v.top_level >= 3) {
        cudaError_t te = b.top.ensure((size_t(1) << (3 * v.top_level)) * sizeof(uint2));
        if (te == cudaSuccess && path_build_top_table(v.nodes, v.top_level, static_cast<uint2*>(b.top.p), stream) == G19_OK &&
            cudaStreamSynchronize(stream) == cudaSuccess) {
            v.top = static_cast<const uint2*>(b.top.p);
        } else {
            cudaGetLastError();
            v.top_level = 0;
        }
    } else {
        v.top_level = 0;
    }
    // bounding-volume hierarchy for tune walk=3 (tree scenes only)
    v.bvh_nodes = nullptr;
    v.bvh4_nodes = nullptr;
    v.bvh_prims = nullptr;
    v.bvh_big = nullptr;
    v.bvh_big_pairs = nullptr;
    v.n_big = v.big_par = v.big_tri = 0;
    v.bvh_root = 0xffffffffu;
    if (tune.walk >= 3 && v.n_nodes > 1) {
        const auto t_bvh = std::chrono::steady_clock::now();
        // primitives much larger than the rest stay out of the hierarchy: at most 64, larger than 1/32 of the root box
        float root_max = std::max(root_size[0], std::max(root_size[1], root_size[2]));
        std::vector<std::pair<float, uint32_t>> large;
        for (size_t i = 0; i < prims.size(); ++i) {
            const Box& bx = prims[i].box;
            const float ext = std::max(bx.hi[0] - bx.lo[0], std::max(bx.hi[1] - bx.lo[1], bx.hi[2] - bx.lo[2]));
            if (ext > root_max * (1.0f / 32.0f)) large.emplace_back(ext, uint32_t(i));
        }
        std::sort(large.begin(), large.end(), [](const std::pair<float, uint32_t>& x, const std::pair<float, uint32_t>& y) {
            return x.first > y.first || (x.first == y.first && x.second < y.second);
        });
        if (large.size() > 64) large.resize(64);
        std::vector<uint32_t> big_ids;
        std::vector<char> is_big(prims.size(), 0);
        for (auto& l : large) { big_ids.push_back(l.second); is_big[l.second] = 1; }
        // kind-sorted (parallelograms | triangles | spheres, by id inside a kind) for the pair loops that test them
        auto kind_rank = [&](uint32_t id) { return prims[id].hot.q[14] == 2.0f ? 0 : (prims[id].hot.q[14] == 1.0f ? 1 : 2); };
        std::sort(big_ids.begin(), big_ids.end(), [&](uint32_t x, uint32_t y) {
            const int rx = kind_rank(x), ry = kind_rank(y);
            return rx < ry || (rx == ry && x < y);
        });
        std::vector<PrimHot> big_hot;
        size_t big_par = 0, big_tri = 0;
        for (uint32_t id : big_ids) {
            big_hot.push_back(hot[id]);
            if (kind_rank(id) == 0) ++big_par;
            else if (kind_rank(id) == 1) ++big_tri;
        }
        std::vector<float> big_pairs;
        build_pairs(big_hot, 0, big_par, big_tri, big_hot.size() - big_par - big_tri, big_pairs);
        std::vector<uint32_t> small_ids;
        small_ids.reserve(prims.size());
        for (size_t i = 0; i < prims.size(); ++i)
            if (!is_big[i]) small_ids.push_back(uint32_t(i));
        std::vector<float> boxes(prims.size() * 6);
        for (size_t i = 0; i < prims.size(); ++i)
            for (int k = 0; k < 3; ++k) {
                boxes[6 * i + k] = prims[i].box.lo[k];
                boxes[6 * i + 3 + k] = prims[i].box.hi[k];
            }
        PoolArray d_boxes, d_small;
        cudaError_t be = d_boxes.ensure(boxes.size() * sizeof(float) + 16, stream);
        if (be == cudaSuccess) be = d_small.ensure(small_ids.size() * sizeof(uint32_t) + 16, stream);
        if (be == cudaSuccess) be = cudaMemcpyAsync(d_boxes.p, boxes.data(), boxes.size() * sizeof(float), cudaMemcpyHostToDevice, stream);
        if (be == cudaSuccess && !small_ids.empty())
            be = cudaMemcpyAsync(d_small.p, small_ids.data(), small_ids.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, stream);
        if (be == cudaSuccess) be = up(b.bvh_big, big_ids.data(), big_ids.size() * sizeof(uint32_t));
        if (be == cudaSuccess) be = up(b.bvh_big_pairs, big_pairs.data(), big_pairs.size() * sizeof(float));
        if (be == cudaSuccess) be = cudaStreamSynchronize(stream);
        int rc = G19_OK;
        if (be != cudaSuccess) {
            err = std::string("path_upload (bvh): ") + cudaGetErrorString(be);
            rc = G19_ERR_CUDA;
        } else {
            rc = path_build_bvh_device(static_cast<const float*>(d_boxes.p), static_cast<const uint32_t*>(d_small.p), uint32_t(small_ids.size()),
                                       root_lo, root_size, v.hot, tune.bvh_leaf, stream, b.bvh_nodes, b.bvh4_nodes, b.bvh_prims, &v.bvh_root, err);
        }
        d_boxes.release();
        d_small.release();
        if (rc != G19_OK) return rc;
        v.bvh_nodes = static_cast<const float4*>(b.bvh_nodes.p);
        v.bvh4_nodes = static_cast<const uint4*>(b.bvh4_nodes.p);
        v.bvh_prims = static_cast<const float4*>(b.bvh_prims.p);
        v.bvh_big = static_cast<const uint32_t*>(b.bvh_big.p);
        v.n_big = int32_t(big_ids.size());
        v.bvh_big_pairs = static_cast<const float*>(b.bvh_big_pairs.p);
        v.big_par = int32_t(big_par);
        v.big_tri = int32_t(big_tri);
        if (tune.debug_tree)
            std::fprintf(stderr, "[g19] path bvh: %zu primitives in the hierarchy, %zu kept out (big), built in %.1f ms\n", small_ids.size(),
                         big_ids.size(), std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_bvh).count());
    }
    v.n_par = n_par;
    v.n_tri = n_tri;
    v.pairs = static_cast<const float*>(b.pairs.p);
    v.pairs_bytes = int32_t(pairs.size() * sizeof(float));
    for (int k = 0; k < 3; ++k) {
        v.root_lo[k] = root_lo[k];
        v.root_size[k] = root_size[k];
        v.grid_scale[k] = float(double(1 << kMaxTreeDepth) / double(root_size[k]));
    }
    return G19_OK;
}

void path_release(PathSceneBuffers& b, PathWork& w) {
    for (DeviceArray* d : {&b.nodes, &b.prim_index, &b.hot, &b.cold, &b.materials, &b.lights, &b.pairs, &b.prim_entity, &b.top, &b.bvh_nodes, &b.bvh4_nodes, &b.bvh_prims, &b.bvh_big, &b.bvh_big_pairs, &w.totals, &w.accum,
                           &w.rad_l, &w.rgb_l, &w.iota})
        d->release();
    w.iota_n = 0;
    w.tile_n.release();
    w.tile_flag.release();
    w.tile_list.release();
    if (w.tile_h) cudaFreeHost(w.tile_h);
    w.tile_h = nullptr;
    w.tile_h_n = 0;
    w.ray_hint_d.release();
    if (w.ray_hint_h) cudaFreeHost(w.ray_hint_h);
    w.ray_hint_h = nullptr;
    w.hint_key = 0;
    for (PathLane& l : w.lane) {
        for (DeviceArray* d : {&l.hp, &l.dw, &l.tp, &l.L, &l.queues, &l.recs, &l.rays, &l.counts, &l.rkeys, &l.perm, &l.sort_tmp}) d->release();
        l.capacity = 0;
    }
    for (int i = 0; i < kMaxLanes; ++i) {
        if (w.side[i]) cudaStreamDestroy(w.side[i]);
        w.side[i] = nullptr;
        for (cudaEvent_t* e : {&w.ev_join[i], &w.ev_acc[i]}) {
            if (*e) cudaEventDestroy(*e);
            *e = nullptr;
        }
    }
    if (w.ev_fork) cudaEventDestroy(w.ev_fork);
    w.ev_fork = nullptr;
    for (cudaEvent_t& e : w.ev_start) {
        if (e) cudaEventDestroy(e);
        e = nullptr;
    }
    w.overlap_key = 0;
    if (w.events) {
        for (int i = 0; i < w.n_events; ++i) cudaEventDestroy(w.events[i]);
        delete[] w.events;
        w.events = nullptr;
        w.n_events = 0;
    }
}

namespace {

struct ClassClock { // non-blocking CUDA-event bracket around each launch group
    PathWork& w;
    cudaStream_t s;
    bool on;
    void begin() {
        if (!on || w.used_events + 2 > w.n_events) return;
        cudaEventRecord(w.events[w.used_events], s);
    }
    void end(int cls) {
        if (!on || w.used_events + 2 > w.n_events) return;
        cudaEventRecord(w.events[w.used_events + 1], s);
        w.event_class[w.used_events / 2] = cls;
        w.used_events += 2;
    }
};

} // namespace

PassArgs path_pass_setup(const PathSceneBuffers& b, const PathTuning& tune, bool count) {
    PassArgs pa{};
    pa.scene = b.view;
    pa.kind_mask = (b.has_bsdf[G19_BSDF_DIFFUSE] ? 1u : 0u) | (b.has_bsdf[G19_BSDF_MIRROR] ? 2u : 0u) |
                   (b.has_bsdf[G19_BSDF_GLASS] ? 4u : 0u);

    // stage the breadth-first prefix of the tree and the first primitives (<= ~24 KB)
    pa.stage_nodes = std::min(b.view.n_nodes, 1024);
    // flat scene (one leaf, <= 192 primitives): intersection + shading records and lights staged whole;
    // a tree scene reaches its primitives through leaf index lists, so only the node prefix is staged
    const bool flat = b.view.n_nodes == 1 && b.view.n_index == b.view.n_prims && b.view.n_prims <= 192;
    pa.stage_prims = flat ? b.view.n_prims : 0;
    pa.stage_cold = flat ? b.view.n_prims : 0;
    pa.stage_lights = (pa.stage_cold > 0 && b.view.n_lights <= 32) ? b.view.n_lights : 0;
    if (b.view.n_lights > 32) pa.stage_cold = 0; // not a "flat, fully staged" scene: the generic kernels take it
    pa.stack_levels = b.view.tree_depth + 1;
    // tree scenes: the bounce kernels queue their rays (2 per vertex at most) for trace_kernel
    pa.refill = tune.refill;
    // tree walk: leaf tests spread over the whole warp, 8 primitives per ray and round (heightfield 1080p x 32 spp:
    // sequential 4 per round 107.1 ms, cooperative 4 / 8 / 16 per round 115.4 / 104.9 / 105.4)
    pa.coop_leaf = tune.coop_leaf;
    pa.walk_steps = tune.walk_steps > 0 ? tune.walk_steps : 2; // measured (room scene, ms per 1080p x 64 spp): octree walk 2 / 4 / 8 steps = 780 / 838 / 961
    pa.leaf_batch = tune.leaf_batch > 0 ? tune.leaf_batch : (pa.coop_leaf ? 16 : 4); // cooperative: the whole leaf in one go (leaf max 8 / 12 / 16 at batch 16: 97.7 / 96.9 / 97.8 ms)
    pa.trace_occ = tune.trace_occ;
    pa.bvh_spec = tune.bvh_spec;
    pa.fold_last = 0;
    pa.flat_uniform = tune.flat_uniform && b.upairs_fit ? 1 : 0;
    pa.upairs = &b.upairs;
    pa.walk = count ? 2 : 1; // the octree walk counts its node / primitive tests when asked (params.profile)
    if (tune.walk >= 3 && b.view.bvh_root != 0xffffffffu && b.view.bvh_nodes) {
        pa.walk = tune.walk == 4 ? (count ? 6 : 5) : 3; // bounding-volume hierarchy, binary / 4-wide (the latter counts its tests when asked)
        // node visits per round, room scene: binary 4 / 6 / 8 / 12 = 437 / 423 / 418 / 418 ms; 4-wide 4 / 6 / 8 / 12 = 346 / 345 / 364 / 382 ms
        if (tune.walk_steps <= 0) pa.walk_steps = tune.walk == 4 ? 5 : 8;
        pa.stack_levels = std::max(pa.stack_levels, tune.bvh_stack);
        pa.coop_leaf = 0;
        pa.stage_nodes = 0; // no octree prefix in shared memory: the L1 the walk lives off is what the carve-out leaves
    }
    return pa;
}

#define PATH_CUDA(call)                                                        \
    do {                                                                       \
        cudaError_t e__ = (call);                                              \
        if (e__ != cudaSuccess) {                                              \
            err = std::string(#call) + ": " + cudaGetErrorString(e__);         \
            return G19_ERR_CUDA;                                               \
        }                                                                      \
    } while (0)

namespace {

// What the passes of one frame share (path_render, path_render_adaptive): frame_begin sets it up, frame_pass enqueues one
// pass, frame_join puts the caller's stream behind every lane.
struct Frame {
    PassArgs pa0;                        // the frame's arguments; per-lane copies below
    PassArgs lanes[kMaxLanes];
    cudaStream_t lane_stream[kMaxLanes];
    bool fused = false;                  // flat scenes trace the camera segment in the first bounce's launch
    size_t window = 0;                   // local pixels (or tile-list positions) per pass, whole tiles
    int spp_pass = 0;                    // samples per pass
    size_t P = 0;                        // path slots per pass
    int n_lanes = 1, first_side = 1, parity = 0;
    int prev_lane = -1;                  // lane of the previous pass
    size_t pass_index = 0;
    unsigned long long key = 0;          // the frame's shape (PathWork::overlap_key)
};

PassArgs frame_args(const PathSceneBuffers& b, const PathRenderArgs& a) {
    const g19_params& p = a.params;
    PassArgs pa0 = path_pass_setup(b, a.tune, p.profile != 0);
    for (int k = 0; k < 3; ++k) {
        pa0.cam.pos[k] = float(a.cam.pos[k]);
        pa0.cam.top_left[k] = float(a.cam.top_left[k]);
        pa0.cam.left[k] = float(a.cam.left[k]);
        pa0.cam.up[k] = float(a.cam.up[k]);
    }
    pa0.map = a.map;
    pa0.seed = p.seed;
    pa0.max_depth = p.max_depth;
    return pa0;
}

// Pass size, lanes and their buffers, the frame's statistics block and accum (accum_planes planes, zeroed), and the side
// lanes started behind the caller's stream -- or, for a frame behind a frame of the same shape with overlap_frames,
// behind their own previous passes (allow_overlap).
int frame_begin(PathSceneBuffers& b, PathWork& w, const PathRenderArgs& a, Frame& f, int accum_planes, bool allow_overlap,
                std::string& err) {
    const g19_params& p = a.params;
    cudaStream_t s = a.stream;
    const size_t npix = size_t(a.map.n_local_pix);
    // Pass size. Flat scenes keep dense vertex records in their queues, so a bounce streams exactly
    // the live vertices whatever the pass size: bigger passes only amortise launch tails (measured on
    // B200, ms per 1080p x 64 spp frame at 2 / 4 / 8 / 16 M slots, one pass in flight: Cornell depth 5
    // 22.3 / 20.9 / 20.2 / 20.2, glass Cornell depth 12 64.4 / 52.0 / 47.7 / 49.3). Tree scenes index their
    // state by slot; with four passes in flight the 1 M-triangle heightfield at depth 5 still prefers big
    // passes (1 / 2 / 4 / 8 / 16 M slots: 166.9 / 142.8 / 128.0 / 121.0 / 117.4 ms per 1080p x 32 spp): its
    // deep-bounce trace launches are a handful of long rays, and fewer, longer launches waste less.
    // Deep tree renders keep smaller passes (their sparse slot accesses live off the 126 MB L2).
    // A pass covers a WINDOW of the rank's pixels (whole 32x32 tiles) times spp_pass samples; frames
    // larger than the target are rendered window by window.
    const bool flat_scene = b.view.n_nodes == 1 && b.view.n_index == b.view.n_prims && b.view.n_prims <= 192 &&
                            b.view.n_lights <= 32;
    size_t target = flat_scene ? (size_t(1) << 23) : (p.max_depth > 6 ? (size_t(1) << 22) : (size_t(1) << 24));
    if (a.tune.pass_slots > 0) target = size_t(a.tune.pass_slots); // tuning knob
    size_t window = npix;
    if (p.pixels_per_pass > 0) window = std::min(npix, (size_t(p.pixels_per_pass) + kTilePix - 1) / kTilePix * kTilePix);
    else if (npix > target) window = target;
    int spp_pass = p.spp_per_pass;
    if (spp_pass <= 0) spp_pass = int(std::max<size_t>(1, target / window));
    spp_pass = std::min(spp_pass, p.spp);
    // enough passes to keep kMaxLanes of them in flight (PathWork), as long as a pass still fills the machine
    if (p.spp_per_pass <= 0)
        while (spp_pass > 1 && ((npix + window - 1) / window) * size_t((p.spp + spp_pass - 1) / spp_pass) < size_t(std::min(4, a.tune.lanes)) &&
               window * size_t((spp_pass + 1) / 2) >= (size_t(1) << 21))
            spp_pass = (spp_pass + 1) / 2;
    const size_t P = window * size_t(spp_pass);
    if (P > 0xfffffff0ull) {
        err = "pass too large";
        return G19_ERR_LIMIT;
    }
    f.window = window;
    f.spp_pass = spp_pass;
    f.P = P;
    // passes of this frame, and how many are kept in flight (see PathWork)
    const size_t n_windows = (npix + window - 1) / window;
    const size_t n_passes = n_windows * size_t((p.spp + spp_pass - 1) / spp_pass);
    const int n_lanes = (p.profile || a.on_pass) ? 1 : int(std::min<size_t>(size_t(a.tune.lanes), n_passes)); // profiling and progressive refresh: one at a time
    f.n_lanes = n_lanes;
    if (n_lanes > 1 && !w.ev_fork) PATH_CUDA(cudaEventCreateWithFlags(&w.ev_fork, cudaEventDisableTiming));
    for (int i = 0; i < n_lanes; ++i) {
        if ((i > 0 || n_lanes > 1) && !w.side[i]) PATH_CUDA(cudaStreamCreateWithFlags(&w.side[i], cudaStreamNonBlocking));
        if (n_lanes > 1 && !w.ev_acc[i]) {
            PATH_CUDA(cudaEventCreateWithFlags(&w.ev_acc[i], cudaEventDisableTiming));
            PATH_CUDA(cudaEventCreateWithFlags(&w.ev_join[i], cudaEventDisableTiming));
        }
    }
    // Frames in a row with the same buffers may overlap on the side lanes (PathWork::ev_start): anything allocated,
    // resized or reset in this call, profiling, progressive refresh or a single lane switch it off for this frame.
    const size_t bytes_before = w.totals.bytes + w.accum.bytes + w.rad_l.bytes + w.rgb_l.bytes + w.iota.bytes + w.ray_hint_d.bytes;
    size_t lane_bytes_before = 0;
    for (const PathLane& l : w.lane) lane_bytes_before += l.capacity + l.L.bytes + l.recs.bytes + l.rays.bytes + l.queues.bytes + l.counts.bytes + l.rkeys.bytes;
    f.key = ((b.upload_serial + 1) << 44) ^ (static_cast<unsigned long long>(P) << 12) ^
            (static_cast<unsigned long long>(n_lanes) << 8) ^ static_cast<unsigned long long>(p.max_depth) ^
            (static_cast<unsigned long long>(npix) << 20) ^ reinterpret_cast<unsigned long long>(s);
    PATH_CUDA(w.totals.ensure(2 * 10 * sizeof(unsigned long long)));
    PATH_CUDA(w.accum.ensure(npix * accum_planes * sizeof(float)));
    PATH_CUDA(w.rad_l.ensure(npix * 3 * sizeof(float)));
    PATH_CUDA(w.rgb_l.ensure(npix * 3));
    for (cudaEvent_t& e : w.ev_start)
        if (!e) PATH_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    const bool may_overlap = allow_overlap && a.tune.overlap_frames && n_lanes > 1 && w.overlap_key == f.key && !p.profile && !a.on_pass;
    w.overlap_key = 0; // set again once this frame is enqueued whole
    const int parity = int(w.frame_serial & 1ull);
    f.parity = parity;
    unsigned long long* const totals2 = static_cast<unsigned long long*>(w.totals.p);
    if (!may_overlap) PATH_CUDA(cudaMemsetAsync(totals2, 0, 2 * 10 * sizeof(unsigned long long), s));
    else PATH_CUDA(cudaMemsetAsync(totals2 + 10 * (parity ^ 1), 0, 10 * sizeof(unsigned long long), s)); // the NEXT frame's block
    PATH_CUDA(cudaMemsetAsync(w.accum.p, 0, npix * accum_planes * sizeof(float), s));
    if (p.profile && !w.events) {
        w.n_events = 65536;
        w.events = new cudaEvent_t[w.n_events];
        for (int i = 0; i < w.n_events; ++i) PATH_CUDA(cudaEventCreate(&w.events[i]));
    }
    w.used_events = 0;
    PassArgs& pa0 = f.pa0;
    pa0.totals = totals2 + 10 * parity;
    w.totals_parity = parity;
    pa0.accum = static_cast<float*>(w.accum.p);

    // per-lane buffers
    const bool fused = f.fused;
    for (int i = 0; i < kMaxLanes; ++i) {
        f.lanes[i] = pa0;
        f.lane_stream[i] = s;
    }
    // Several lanes: with overlap_frames ALL of them run on streams of their own (the caller's stream only zeroes, joins and
    // resolves), so that the next frame's passes can follow this frame's on every lane; otherwise lane 0 is the caller's stream.
    f.first_side = (n_lanes > 1 && a.tune.overlap_frames) ? 0 : 1;
    for (int i = f.first_side; i < n_lanes; ++i) f.lane_stream[i] = w.side[i];
    for (int li = 0; li < n_lanes; ++li) {
        PathLane& l = w.lane[li];
        PassArgs& pa = f.lanes[li];
        if (P > l.capacity) {
            PATH_CUDA(l.L.ensure(P * 4 * sizeof(float))); // flat scenes: float4 per slot; tree scenes: three planes
            l.capacity = P;
            PATH_CUDA(cudaMemsetAsync(l.L.p, 0, P * 4 * sizeof(float), f.lane_stream[li]));
            l.L_written_whole = false;
        }
        // tree scenes ADD to zeroed planes (accumulate clears what it read); flat scenes store every slot
        // (a lane's own buffers are cleared on the lane's own stream: in order with its passes, whatever the caller's stream is at)
        if (!fused && l.L_written_whole) PATH_CUDA(cudaMemsetAsync(l.L.p, 0, l.capacity * 4 * sizeof(float), f.lane_stream[li]));
        l.L_written_whole = fused;
        const size_t plane = l.capacity;
        PATH_CUDA(l.counts.ensure((kMaxPathDepth + 1) * 5 * sizeof(uint32_t)));
        PATH_CUDA(cudaMemsetAsync(l.counts.p, 0, (kMaxPathDepth + 1) * 5 * sizeof(uint32_t), f.lane_stream[li]));
        pa.L = static_cast<float*>(l.L.p);
        pa.plane = plane;
        pa.queue_cap = plane + kQueueSlack;
        pa.spec_cap = 0;
        for (int k = 0; k < kNumQueues; ++k) pa.q[k] = nullptr;
        pa.counts = static_cast<uint32_t*>(l.counts.p);
        pa.ray0 = pa.ray1 = pa.ray2 = nullptr;
        pa.hp = pa.dw = pa.tp = nullptr;
        pa.rec_ls = pa.rec_hp = pa.rec_dw = pa.rec_tp = nullptr;
        if (fused) {
            // dense vertex records, four float4 planes: per bounce parity the diffuse array and -- only when the scene has
            // mirror or glass -- the array those two share (a bounce holds at most P vertices over its queues together)
            pa.spec_cap = (pa0.kind_mask & 6u) ? plane + 2 * kQueueSlack : 0;
            const size_t per_plane = 2 * (pa.queue_cap + pa.spec_cap);
            PATH_CUDA(l.recs.ensure(per_plane * 4 * sizeof(float4)));
            pa.rec_ls = static_cast<float4*>(l.recs.p);
            pa.rec_hp = pa.rec_ls + per_plane;
            pa.rec_dw = pa.rec_hp + per_plane;
            pa.rec_tp = pa.rec_dw + per_plane;
        } else {
            PATH_CUDA(l.queues.ensure((plane + kQueueSlack) * kNumQueues * sizeof(uint32_t)));
            for (int k = 0; k < kNumQueues; ++k) pa.q[k] = static_cast<uint32_t*>(l.queues.p) + size_t(k) * pa.queue_cap;
            PATH_CUDA(l.hp.ensure(plane * sizeof(float4)));
            PATH_CUDA(l.dw.ensure(plane * sizeof(float4)));
            PATH_CUDA(l.tp.ensure(plane * sizeof(float4)));
            pa.hp = static_cast<float4*>(l.hp.p);
            pa.dw = static_cast<float4*>(l.dw.p);
            pa.tp = static_cast<float4*>(l.tp.p);
            const size_t ray_cap = 2 * plane + kQueueSlack;
            PATH_CUDA(l.rays.ensure(3 * ray_cap * sizeof(float4)));
            pa.ray0 = static_cast<float4*>(l.rays.p);
            pa.ray1 = pa.ray0 + ray_cap;
            pa.ray2 = pa.ray1 + ray_cap;
            pa.rkey = nullptr;
            pa.perm = nullptr;
            pa.perm_n = 0;
            pa.ray_hint = nullptr;
            const bool sort_rays = a.tune.sort_rays < 0 ? pa0.walk < 3 : a.tune.sort_rays != 0;
            if (sort_rays && p.max_depth > 1) {
                PATH_CUDA(l.rkeys.ensure(2 * ray_cap * sizeof(uint16_t)));
                PATH_CUDA(l.perm.ensure(ray_cap * sizeof(uint32_t)));
                PATH_CUDA(l.sort_tmp.ensure(ray_sort_temp_bytes(ray_cap)));
                if (w.iota_n < ray_cap) {
                    PATH_CUDA(w.iota.ensure(ray_cap * sizeof(uint32_t)));
                    launch_iota(static_cast<uint32_t*>(w.iota.p), ray_cap, s);
                    w.iota_n = ray_cap;
                }
                pa.rkey = static_cast<uint16_t*>(l.rkeys.p);
                pa.perm = static_cast<uint32_t*>(l.perm.p);
                // the hints of the last frame of this workload (scene upload, pass size, depth)
                const unsigned long long key = (b.upload_serial << 40) ^ (static_cast<unsigned long long>(P) << 8) ^ static_cast<unsigned long long>(p.max_depth);
                if (!w.ray_hint_h) PATH_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&w.ray_hint_h), (kMaxPathDepth + 1) * sizeof(uint32_t), cudaHostAllocDefault));
                if (!w.ray_hint_d.p || w.hint_key != key) {
                    PATH_CUDA(w.ray_hint_d.ensure((kMaxPathDepth + 1) * sizeof(uint32_t)));
                    PATH_CUDA(cudaStreamSynchronize(s)); // (a copy of the previous workload's hints may still be in flight)
                    PATH_CUDA(cudaMemsetAsync(w.ray_hint_d.p, 0, (kMaxPathDepth + 1) * sizeof(uint32_t), s));
                    std::memset(w.ray_hint_h, 0, (kMaxPathDepth + 1) * sizeof(uint32_t));
                    w.hint_key = key;
                }
                pa.ray_hint = static_cast<uint32_t*>(w.ray_hint_d.p);
            }
        }
    }
    {
        size_t lane_bytes_after = 0;
        for (const PathLane& l : w.lane) lane_bytes_after += l.capacity + l.L.bytes + l.recs.bytes + l.rays.bytes + l.queues.bytes + l.counts.bytes + l.rkeys.bytes;
        const size_t bytes_after = w.totals.bytes + w.accum.bytes + w.rad_l.bytes + w.rgb_l.bytes + w.iota.bytes + w.ray_hint_d.bytes;
        const bool overlap = may_overlap && lane_bytes_after == lane_bytes_before && bytes_after == bytes_before;
        PATH_CUDA(cudaEventRecord(w.ev_start[parity], s)); // the memsets above (this frame's accum, the next frame's statistics)
        if (n_lanes > 1) {
            if (overlap) {
                // a frame behind a frame of the same shape: the side lanes go on behind their own passes; all they need from the
                // caller's stream is last frame's start (their statistics block was zeroed there)
                for (int i = f.first_side; i < n_lanes; ++i) PATH_CUDA(cudaStreamWaitEvent(w.side[i], w.ev_start[parity ^ 1], 0));
            } else { // the other lanes start after everything enqueued so far on the caller's stream
                PATH_CUDA(cudaEventRecord(w.ev_fork, s));
                for (int i = f.first_side; i < n_lanes; ++i) PATH_CUDA(cudaStreamWaitEvent(w.side[i], w.ev_fork, 0));
            }
        }
    }
    return G19_OK;
}

// One pass: samples [base, base + batch_spp) of window positions [pix0, pix0 + pix_count) -- the camera segment, the
// bounces (tree scenes: with their ray sorts and walks), then accumulate, behind the previous pass's accumulate whichever
// lane that ran on, so that the per-pixel sums are taken in sample order.
int frame_pass(const PathSceneBuffers& b, PathWork& w, const PathRenderArgs& a, Frame& f, ClassClock& clk, int base, int batch_spp,
               size_t pix0, size_t pix_count, g19_stats& stats, std::string& err) {
    const g19_params& p = a.params;
    const bool fused = f.fused;
    const int n_lanes = f.n_lanes;
    const int li = int(f.pass_index++ % size_t(n_lanes));
    PassArgs& pa = f.lanes[li];
    cudaStream_t ls = f.lane_stream[li];
    clk.s = ls;
    pa.sample_base = base;
    pa.spp_pass = batch_spp;
    pa.pix_base = uint32_t(pix0);
    pa.pix_count = uint32_t(pix_count);
    pa.n_slots = uint32_t(size_t(pa.pix_count) * size_t(pa.spp_pass));
    if (!fused) { // flat scenes trace the camera segment in the first bounce's launch
        clk.begin();
        launch_raygen_extend(pa, a.sm_count, ls);
        clk.end(G19_K_EXTEND);
        stats.class_launches[G19_K_EXTEND] += 1;
    }
    // flat scenes: the launch before the last shades the last vertex in place, so the last bounce has no launch
    const int n_launch = fused && p.max_depth >= 2 ? p.max_depth - 1 : p.max_depth;
    for (int bounce = 0; bounce < n_launch; ++bounce) {
        clk.begin();
        int n = 0;
        if (fused) {
            pa.fold_last = bounce == p.max_depth - 2 ? 1 : 0;
            if (bounce == 0) {
                launch_bounce_first_fused(pa, a.sm_count, ls);
                ++n;
            }
            // (at bounce 0 with mirror / glass: the camera hits on those, which the fused launch queued)
            if ((bounce > 0 || ((pa.kind_mask & 6u) && p.max_depth > 1)) && launch_bounce_flat(pa, bounce, a.sm_count, ls)) ++n;
            clk.end(G19_K_SHADE);
            stats.class_launches[G19_K_SHADE] += n;
            continue;
        }
        // the first bounce's rays leave the camera rays' hit points in pixel order: coherent as they are
        // ... and a queue that stayed short the last time is walked in a blink: not worth three more launches.
        const size_t ray_cap = 2 * pa.plane + kQueueSlack;
        size_t n_sort = 0;
        if (pa.rkey && bounce > 0) {
            const uint32_t hint = w.ray_hint_h[bounce]; // 0 = not known yet: the whole queue
            n_sort = hint == 0 ? ray_cap : std::min(ray_cap, size_t(hint) + size_t(hint) / 8 + 65536);
            if (hint != 0 && hint < (1u << 19)) n_sort = 0;
        }
        const bool sort_this = n_sort > 0;
        PassArgs pb = pa;
        pb.perm_n = uint32_t(n_sort);
        if (!sort_this) pb.rkey = nullptr, pb.perm = nullptr;
        if (sort_this) PATH_CUDA(cudaMemsetAsync(pa.rkey, 0xff, n_sort * sizeof(uint16_t), ls));
        for (int kind = Q_DIFFUSE; kind <= Q_GLASS; ++kind) {
            if (!b.has_bsdf[kind - 1]) continue; // no such material in the scene: queue is always empty
            if (launch_bounce(pb, bounce, kind, a.sm_count, ls)) ++n;
        }
        if (n > 0) { // one walk over the rays this bounce's vertices produced
            if (sort_this) {
                PATH_CUDA(launch_ray_sort(w.lane[li].sort_tmp.p, w.lane[li].sort_tmp.bytes, pa.rkey, pa.rkey + ray_cap,
                                          static_cast<const uint32_t*>(w.iota.p), static_cast<uint32_t*>(w.lane[li].perm.p), n_sort, ls));
                n += 3; // histogram + two one-sweep passes
            }
            launch_trace(pb, bounce, a.sm_count, ls);
            ++n;
        }
        clk.end(G19_K_SHADE);
        stats.class_launches[G19_K_SHADE] += n;
    }
    // the per-pixel sums are taken in pass order whichever lane a pass ran on
    if (n_lanes > 1 && f.prev_lane >= 0) PATH_CUDA(cudaStreamWaitEvent(ls, w.ev_acc[f.prev_lane], 0));
    else if (n_lanes > 1 && ls != a.stream) PATH_CUDA(cudaStreamWaitEvent(ls, w.ev_start[f.parity], 0)); // the frame's first: behind the memset of accum
    clk.begin();
    launch_accumulate(pa, ls);
    clk.end(G19_K_ACCUM);
    stats.class_launches[G19_K_ACCUM] += 1;
    if (n_lanes > 1) {
        PATH_CUDA(cudaEventRecord(w.ev_acc[li], ls));
        f.prev_lane = li;
    }
    return G19_OK;
}

// The caller's stream continues after the other lanes (and copies the ray-sort hints they raised).
int frame_join(PathWork& w, const PathRenderArgs& a, Frame& f, ClassClock& clk, std::string& err) {
    cudaStream_t s = a.stream;
    for (int i = f.first_side; i < f.n_lanes; ++i) {
        PATH_CUDA(cudaEventRecord(w.ev_join[i], w.side[i]));
        PATH_CUDA(cudaStreamWaitEvent(s, w.ev_join[i], 0));
    }
    clk.s = s;
    if (!f.fused && w.ray_hint_h && w.ray_hint_d.p && f.lanes[0].ray_hint)
        PATH_CUDA(cudaMemcpyAsync(w.ray_hint_h, w.ray_hint_d.p, (kMaxPathDepth + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    return G19_OK;
}

// A launch that failed during the frame: its lanes' radiance planes and queue lengths are dirty -- re-zero them before the
// next render.
int frame_launch_error(PathWork& w, std::string& err) {
    const char* le = path_launch_error();
    if (!le) return G19_OK;
    err = le;
    path_clear_launch_error();
    cudaGetLastError();
    for (PathLane& l : w.lane) l.capacity = 0;
    return G19_ERR_CUDA;
}

uint64_t tile_pixels_in_frame(const TileMap& map, int lt) {
    const int tile = lt * map.world + map.rank;
    const int ty = tile / map.tiles_x, tx = tile % map.tiles_x;
    return uint64_t(std::min(kTile, map.w - tx * kTile)) * uint64_t(std::min(kTile, map.h - ty * kTile));
}

} // namespace

int path_render(PathSceneBuffers& b, PathWork& w, const PathRenderArgs& a, g19_stats& stats, std::string& err) {
    const g19_params& p = a.params;
    if (p.spp < 1 || p.max_depth < 0 || p.max_depth > kMaxPathDepth || (p.max_depth == 0 && !a.ids_l)) {
        err = "PATH mode needs spp >= 1 and 0 <= max_depth <= 64";
        return G19_ERR_INVALID;
    }
    cudaStream_t s = a.stream;
    const size_t npix = size_t(a.map.n_local_pix);
    if (npix == 0) return G19_OK;
    path_clear_launch_error();
    Frame f;
    f.pa0 = frame_args(b, a);
    f.fused = path_scene_is_flat(f.pa0); // flat scenes trace inside the bounce kernels
    // primary-hit AOV: the un-jittered ray of every pixel (the reference's ray) through this engine's structures
    if (a.ids_l) {
        launch_primary(f.pa0, a.ids_l, a.points_l, a.normals_l, a.sm_count, s);
        stats.class_launches[G19_K_EXTEND] += 1;
        stats.kernel_launches += 1;
    }
    if (p.max_depth == 0) { // depth-0 slice: nothing to bounce; the caller shades the primary hits (engine.cu)
        if (const char* le = path_launch_error()) {
            err = le;
            path_clear_launch_error();
            return G19_ERR_CUDA;
        }
        return G19_OK;
    }
    int rc = frame_begin(b, w, a, f, 3, true, err);
    if (rc != G19_OK) return rc;
    const PassArgs& pa0 = f.pa0;
    ClassClock clk{w, s, p.profile != 0};
    auto last_refresh = std::chrono::steady_clock::now();
    int batch_spp = 0;
    for (int base = 0; base < p.spp; base += f.spp_pass) {
        if (a.cancel && a.cancel->load()) { // RayTracer::stop(): honoured between passes
            rc = G19_ERR_CANCELLED;
            break;
        }
        batch_spp = std::min(f.spp_pass, p.spp - base);
        for (size_t pix0 = 0; pix0 < npix; pix0 += f.window) { // the windows of this sample batch
            const int prc = frame_pass(b, w, a, f, clk, base, batch_spp, pix0, std::min(f.window, npix - pix0), stats, err);
            if (prc != G19_OK) return prc;
        }
        stats.samples += uint64_t(batch_spp); // scaled by owned pixels below
        if (a.progress_milli) a.progress_milli->store(int(1000.0 * double(base + batch_spp) / double(p.spp)));
        if (a.on_pass && a.d_rgb && a.h_rgb && base + batch_spp < p.spp) {
            // progressive refresh: the host stays at most one pass ahead of the device (that is also
            // the cancellation latency), and repaints no more often than the caller asked for
            PATH_CUDA(cudaStreamSynchronize(s));
            const auto now = std::chrono::steady_clock::now();
            if (std::chrono::duration<double, std::milli>(now - last_refresh).count() >= double(a.min_interval_ms)) {
                last_refresh = now;
                const int so_far = base + batch_spp;
                launch_resolve(a.map, pa0.accum, so_far, static_cast<float*>(w.rad_l.p), static_cast<uint8_t*>(w.rgb_l.p), s);
                launch_untile(a.map, static_cast<uint8_t*>(w.rgb_l.p), nullptr, nullptr, a.d_rgb, nullptr, nullptr, s);
                PATH_CUDA(cudaMemcpyAsync(a.h_rgb, a.d_rgb, size_t(a.map.w) * size_t(a.map.h) * 3, cudaMemcpyDeviceToHost, s));
                PATH_CUDA(cudaStreamSynchronize(s));
                stats.class_launches[G19_K_OTHER] += 2;
                if (a.on_pass(a.pass_user, double(so_far) / double(p.spp), a.h_rgb) != 0) a.cancel->store(1);
            }
        }
    }
    const int jrc = frame_join(w, a, f, clk, err);
    if (jrc != G19_OK) return jrc;
    const int done_spp = int(stats.samples);
    clk.begin();
    if (a.frame_flags) {
        // fused resolve + untile + gather: wait until the owner is done with the previous frame,
        // store this rank's pixels into the shared frame, then signal arrival
        launch_frame_acquire(a.frame_flags, a.frame_need_consumed, a.frame_status, s);
        launch_resolve_to_frame(a.map, pa0.accum, done_spp > 0 ? done_spp : 1, a.frame_rgb, a.frame_rad, s);
        launch_frame_signal(a.frame_flags, s);
        clk.end(G19_K_OTHER);
        stats.class_launches[G19_K_OTHER] += 3;
    } else {
        launch_resolve(a.map, pa0.accum, done_spp > 0 ? done_spp : 1, static_cast<float*>(w.rad_l.p),
                       static_cast<uint8_t*>(w.rgb_l.p), s);
        const bool to_frame = a.d_rgb || a.d_rad;
        if (to_frame)
            launch_untile(a.map, a.d_rgb ? static_cast<uint8_t*>(w.rgb_l.p) : nullptr, nullptr,
                          a.d_rad ? static_cast<float*>(w.rad_l.p) : nullptr, a.d_rgb, nullptr, a.d_rad, s);
        clk.end(G19_K_OTHER);
        stats.class_launches[G19_K_OTHER] += to_frame ? 2 : 1;
    }
    if (a.t_rad) PATH_CUDA(cudaMemcpyAsync(a.t_rad, w.rad_l.p, npix * 3 * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (a.t_rgb) PATH_CUDA(cudaMemcpyAsync(a.t_rgb, w.rgb_l.p, npix * 3, cudaMemcpyDeviceToDevice, s));
    const int lrc = frame_launch_error(w, err);
    if (lrc != G19_OK) return lrc;
    PATH_CUDA(cudaGetLastError());
    for (int k = 0; k < 8; ++k) stats.kernel_launches += stats.class_launches[k];
    // owned in-frame pixels
    uint64_t owned = 0;
    for (int lt = 0; lt < a.map.n_local_tiles; ++lt) owned += tile_pixels_in_frame(a.map, lt);
    stats.samples = owned * uint64_t(done_spp);
    w.totals_pending = true;
    w.totals_stream = s;
    ++w.frame_serial;
    if (rc == G19_OK) w.overlap_key = f.key; // the next frame of the same shape may start behind this one's passes
    return rc;
}

// Rounds: round 0 gives every local tile samples [0, min_spp); after a round the tile test marks the tiles whose error is
// still above tau (and below spp), the compaction lists them, and the next round gives those [n, min(2n, spp)). A round's
// passes run over windows of the list (PassArgs::tiles), with the pass size and lanes path_render would use for this frame
// at spp samples, so a tile's sums are those of path_render at its count.
int path_render_adaptive(PathSceneBuffers& b, PathWork& w, const PathRenderArgs& a, float tau, int min_spp, float* d_var,
                         int32_t* d_spp, g19_stats& stats, std::string& err) {
    const g19_params& p = a.params;
    if (p.max_depth < 1 || p.max_depth > kMaxPathDepth || min_spp < 2 || min_spp > p.spp || !(tau > 0.0f) || !std::isfinite(tau)) {
        err = "adaptive PATH render needs 1 <= max_depth <= 64, 2 <= min_spp <= spp and a finite noise_target > 0";
        return G19_ERR_INVALID;
    }
    cudaStream_t s = a.stream;
    const TileMap& map = a.map;
    const size_t n_tiles = size_t(map.n_local_tiles);
    w.overlap_key = 0; // this frame's lanes and accum are not what the next g19_render's overlap expects
    if (n_tiles == 0) return G19_OK;
    path_clear_launch_error();
    // per-tile state: [0] the length of the next list, [1 ..] the count of each local tile; the two lists; the flags
    PATH_CUDA(w.tile_n.ensure((n_tiles + 1) * sizeof(int32_t)));
    PATH_CUDA(w.tile_flag.ensure(n_tiles * sizeof(uint32_t)));
    PATH_CUDA(w.tile_list.ensure(2 * n_tiles * sizeof(uint32_t)));
    if (w.tile_h_n < n_tiles + 1) {
        if (w.tile_h) cudaFreeHost(w.tile_h);
        w.tile_h = nullptr;
        w.tile_h_n = 0;
        PATH_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&w.tile_h), (n_tiles + 1) * sizeof(int32_t), cudaHostAllocDefault));
        w.tile_h_n = n_tiles + 1;
    }
    int32_t* const d_tile = static_cast<int32_t*>(w.tile_n.p);
    uint32_t* const d_flag = static_cast<uint32_t*>(w.tile_flag.p);
    uint32_t* list[2] = {static_cast<uint32_t*>(w.tile_list.p), static_cast<uint32_t*>(w.tile_list.p) + n_tiles};
    launch_iota(list[0], n_tiles, s); // round 0: every local tile (ahead of the side lanes' fork in frame_begin)
    stats.class_launches[G19_K_OTHER] += 1;
    Frame f;
    f.pa0 = frame_args(b, a);
    f.fused = path_scene_is_flat(f.pa0);
    int rc = frame_begin(b, w, a, f, 4, false, err);
    if (rc != G19_OK) return rc;
    ClassClock clk{w, s, p.profile != 0};
    uint32_t n_active = uint32_t(n_tiles);
    int cur = 0, done = 0, upto = min_spp;
    for (;;) {
        for (int k = 0; k < f.n_lanes; ++k) f.lanes[k].tiles = list[cur];
        const size_t positions = size_t(n_active) * kTilePix;
        for (int base = done; base < upto; base += f.spp_pass) {
            if (a.cancel && a.cancel->load()) { // g19_cancel: honoured between passes
                rc = G19_ERR_CANCELLED;
                break;
            }
            const int batch_spp = std::min(f.spp_pass, upto - base);
            for (size_t pix0 = 0; pix0 < positions; pix0 += f.window) {
                const int prc = frame_pass(b, w, a, f, clk, base, batch_spp, pix0, std::min(f.window, positions - pix0), stats, err);
                if (prc != G19_OK) return prc;
            }
        }
        const int jrc = frame_join(w, a, f, clk, err);
        if (jrc != G19_OK) return jrc;
        if (rc != G19_OK) break;
        // the tile test sees the round's last accumulate through the join; the host reads the next list's length
        clk.begin();
        launch_tile_test(map, f.pa0.accum, list[cur], n_active, upto, p.spp, tau, d_tile + 1, d_flag, s);
        launch_tile_compact(list[cur], n_active, d_flag, list[cur ^ 1], reinterpret_cast<uint32_t*>(d_tile), s);
        clk.end(G19_K_OTHER);
        stats.class_launches[G19_K_OTHER] += 2;
        PATH_CUDA(cudaMemcpyAsync(w.tile_h, d_tile, (n_tiles + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        PATH_CUDA(cudaStreamSynchronize(s));
        const int lrc = frame_launch_error(w, err);
        if (lrc != G19_OK) return lrc;
        n_active = uint32_t(w.tile_h[0]);
        if (a.progress_milli) a.progress_milli->store(int(1000.0 * double(upto) / double(p.spp)));
        if (n_active == 0) break;
        cur ^= 1;
        done = upto;
        upto = std::min(2 * upto, p.spp);
        if (f.n_lanes > 1) { // the next round's passes read the new list: the side lanes start behind the compaction
            PATH_CUDA(cudaEventRecord(w.ev_fork, s));
            for (int i = f.first_side; i < f.n_lanes; ++i) PATH_CUDA(cudaStreamWaitEvent(w.side[i], w.ev_fork, 0));
        }
    }
    if (rc == G19_OK) {
        clk.begin();
        launch_resolve_adaptive(map, f.pa0.accum, d_tile + 1, a.d_rgb, a.d_rad, d_var, d_spp, s);
        clk.end(G19_K_OTHER);
        stats.class_launches[G19_K_OTHER] += 1;
    }
    const int lrc = frame_launch_error(w, err);
    if (lrc != G19_OK) return lrc;
    PATH_CUDA(cudaGetLastError());
    for (int k = 0; k < 8; ++k) stats.kernel_launches += stats.class_launches[k];
    uint64_t samples = 0; // in-frame owned pixels times their tile's count (complete rounds only)
    if (rc == G19_OK)
        for (int lt = 0; lt < map.n_local_tiles; ++lt) samples += tile_pixels_in_frame(map, lt) * uint64_t(w.tile_h[1 + lt]);
    stats.samples = samples;
    w.totals_pending = true;
    w.totals_stream = s;
    ++w.frame_serial;
    return rc;
}

#undef PATH_CUDA

int path_finish_stats(PathWork& w, g19_stats& stats, std::string& err) {
    if (!w.totals_pending) return G19_OK;
    unsigned long long h[10];
    cudaError_t e = cudaMemcpy(h, static_cast<const unsigned long long*>(w.totals.p) + 10 * w.totals_parity, sizeof h, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
        err = std::string("path_finish_stats: ") + cudaGetErrorString(e);
        return G19_ERR_CUDA;
    }
    stats.extend_segments = h[0] + stats.samples; // bounce 0 has no queue: one segment per camera path
    stats.shadow_segments = h[1];
    stats.shade_calls = h[2];
    stats.shade_calls_first = h[3];
    stats.lit_samples = h[4];
    stats.radiance_reads = h[5];
    stats.radiance_stores = h[6];
    stats.node_tests = h[7]; // tree scenes under params.profile: octree node records visited / primitive tests (TreeWalk2<COUNT>)
    stats.prim_tests = h[8];
    stats.shade_calls_folded = h[9];
    for (int i = 0; i + 1 < w.used_events; i += 2) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, w.events[i], w.events[i + 1]) == cudaSuccess) stats.class_ms[w.event_class[i / 2]] += ms;
    }
    w.totals_pending = false;
    return G19_OK;
}

int path_cast(const PathSceneBuffers& b, PathCastWork& cw, const PathTuning& tune, int32_t n, const float* d_rays, uint32_t flags,
              int32_t* d_ids, float* d_t, float* d_normals, cudaStream_t stream, int sm_count, g19_stats& stats, std::string& err) {
    const bool any = (flags & G19_CAST_ANY_HIT) != 0u, count = (flags & G19_CAST_COUNT) != 0u;
    cudaError_t e = cw.counters.ensure(10 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemsetAsync(cw.counters.p, 0, 10 * sizeof(unsigned long long), stream);
    if (e != cudaSuccess) {
        err = std::string("path_cast: ") + cudaGetErrorString(e);
        return G19_ERR_CUDA;
    }
    PassArgs pa = path_pass_setup(b, tune, count);
    pa.totals = static_cast<unsigned long long*>(cw.counters.p);
    CastArgs c;
    c.rays = reinterpret_cast<const float4*>(d_rays);
    c.ids = d_ids;
    c.t = d_t;
    c.normals = d_normals;
    c.n = uint32_t(n);
    c.cursor = reinterpret_cast<uint32_t*>(pa.totals + 9);
    path_clear_launch_error();
    launch_cast(pa, c, any, sm_count, stream);
    if (const char* le = path_launch_error()) {
        err = le;
        path_clear_launch_error();
        cudaGetLastError();
        return G19_ERR_CUDA;
    }
    (any ? stats.shadow_segments : stats.extend_segments) = uint64_t(n);
    stats.kernel_launches = 1;
    cw.counts_pending = count;
    return G19_OK;
}

int path_cast_finish_stats(PathCastWork& cw, g19_stats& stats, std::string& err) {
    if (!cw.counts_pending) return G19_OK;
    unsigned long long h[2];
    cudaError_t e = cudaMemcpy(h, static_cast<const unsigned long long*>(cw.counters.p) + 7, sizeof h, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
        err = std::string("path_cast_finish_stats: ") + cudaGetErrorString(e);
        return G19_ERR_CUDA;
    }
    stats.node_tests = h[0];
    stats.prim_tests = h[1];
    cw.counts_pending = false;
    return G19_OK;
}

} // namespace g19

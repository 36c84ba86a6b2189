// octree.h -- interface-compatible Octree (reference include/octree.h:12-68).
//
// push_back forwards each entity's descriptor to a g19_scene, where the
// reference's build (partition / push_obj, octree.h:75-129) is mirrored bug for
// bug on the host (csrc/scene.cpp) and later flattened to HBM. intersect() is a
// GPU probe returning the reference's candidate list. Two additions the
// reference does not offer: handle() (its Node/_root are private), the way for
// RayTracer to reach the tree, and nearest(), batched nearest-hit queries
// (g19_cast_rays) for picking.
#pragma once
#include <algorithm>
#include <cstddef>
#include <limits>
#include <memory>
#include <vector>
#include "bbox.h"
#include "entities.h"

class Octree {
  public:
    Octree(glm::dvec3 lo, glm::dvec3 hi) : min(lo), max(hi) {
        const double a[3] = {lo.x, lo.y, lo.z}, b[3] = {hi.x, hi.y, hi.z};
        g19_scene* s = nullptr;
        g19::detail::check(g19_scene_create(a, b, &s), nullptr, "g19_scene_create");
        _scene.reset(s, g19_scene_destroy);
    }

    glm::dvec3 min;
    glm::dvec3 max;

    void push_back(Entity* object) {
        g19_entity_desc d = object->describe();
        // a root-test reject is silent, as in octree.h:22-24 (the engine still numbers the entity); anything else
        // means the engine did NOT number it, and appending it here would shift every later id
        const int rc = g19_scene_add_entity(_scene.get(), &d, nullptr);
        if (rc != G19_OK && rc != G19_ERR_REJECTED) g19::detail::check(rc, nullptr, "g19_scene_add_entity");
        _entities.push_back(object);
        ++_version;
    }

    std::vector<Entity*> intersect(const Ray& ray) const {
        std::lock_guard<std::mutex> lock(g19::detail::probe_mutex());
        g19_ctx* ctx = g19::detail::probe_ctx();
        g19::detail::upload_cached(_scene.get(), _serial, _version);
        const double o[3] = {ray.origin.x, ray.origin.y, ray.origin.z}, d[3] = {ray.dir.x, ray.dir.y, ray.dir.z};
        int n = 0;
        std::vector<int32_t> ids(1 << 16);
        g19::detail::check(g19_probe_candidates(ctx, o, d, ids.data(), int(ids.size()), &n), ctx, "g19_probe_candidates");
        std::vector<Entity*> out;
        for (int i = 0; i < n && i < int(ids.size()); ++i) out.push_back(_entities[size_t(ids[i])]);
        return out;
    }

    // additions
    // What each ray hits first (nearest hit, g19_cast_rays over PATH mode's structures): the entity, or nullptr for a
    // miss; t (nullable) receives the distance along the normalised direction (+inf for a miss). What a viewer needs
    // for picking: the entity under the mouse.
    std::vector<Entity*> nearest(const std::vector<Ray>& rays, std::vector<double>* t = nullptr) const {
        std::lock_guard<std::mutex> lock(g19::detail::probe_mutex());
        g19_ctx* ctx = g19::detail::probe_ctx();
        g19::detail::upload_cached(_scene.get(), _serial, _version);
        const size_t n = rays.size();
        std::vector<float> rec(8 * n, 0.0f); // (origin, tmax | direction, 0) per ray
        for (size_t i = 0; i < n; ++i) {
            const Ray& r = rays[i];
            const float v[8] = {float(r.origin.x), float(r.origin.y), float(r.origin.z), std::numeric_limits<float>::infinity(),
                                float(r.dir.x), float(r.dir.y), float(r.dir.z), 0.0f};
            std::copy(v, v + 8, rec.begin() + std::ptrdiff_t(8 * i));
        }
        std::vector<int32_t> ids(n);
        std::vector<float> tf(t ? n : 0);
        g19::detail::check(g19_cast_rays(ctx, int32_t(n), rec.data(), 0u, ids.data(), t ? tf.data() : nullptr, nullptr), ctx,
                           "g19_cast_rays");
        std::vector<Entity*> out(n, nullptr);
        for (size_t i = 0; i < n; ++i)
            if (ids[i] >= 0) out[i] = _entities[size_t(ids[i])];
        if (t) t->assign(tf.begin(), tf.end());
        return out;
    }
    const g19_scene* handle() const { return _scene.get(); }
    unsigned version() const { return _version; }
    const std::vector<Entity*>& entities() const { return _entities; }

  private:
    std::shared_ptr<g19_scene> _scene;
    std::vector<Entity*> _entities; // id = push order, same numbering as the engine
    unsigned _version = 0;
    unsigned long _serial = g19::detail::next_serial(); // identifies this Octree to the probe upload cache
};

// ref_driver.cpp -- C API over the UNMODIFIED reference headers.
//
// TEST INFRASTRUCTURE ONLY (oracle/): nothing in the product path may link or
// load this. It is compiled by oracle/Makefile from the sources where they lie
// in the reference checkout named by G19_REFERENCE (never copied) into
// oracle/_ref/libg19ref.so.
//
// What it exposes:
//   * g19ref_render      -- RayTracer::run verbatim (reference raytracer.h:23-87)
//   * g19ref_trace       -- the same per-pixel loop restated through the
//                           reference's PUBLIC API only (raytracer.h:28-84), so
//                           that the per-pixel entity id / hit point / normal
//                           (which run() never exposes) can be read. Its RGB
//                           bytes are checked against g19ref_render in
//                           tests/test_oracle_ref.py -- that equality is what
//                           licenses its ids.
//   * per-entity probes  -- intersect / boundingBox / getTextureCoord /
//                           triangles, and Octree::intersect candidate lists.
#include <cstdint>
#include <cstring>
#include <thread>
#include <unordered_map>
#include <vector>

#include "raytracer.h" // the reference's, via -I$G19_REFERENCE/include

#include "g19.h" // descriptor structs only

// `friend class Viewer;` (reference image.h:28) is the one door to Image::_image.
class Viewer {
  public:
    static const QImage& bits(const Image& im) { return im._image; }
};

namespace {

struct RefScene {
    Octree tree;
    std::vector<Entity*> entities;              // construction order = entity id
    std::unordered_map<const Entity*, int> ids;
    RefScene(glm::dvec3 mn, glm::dvec3 mx) : tree(mn, mx) {}
};

glm::dvec3 v3(const double* p) { return glm::dvec3{p[0], p[1], p[2]}; }

Entity* make_entity(const g19_entity_desc& d) {
    glm::dvec3 color = v3(d.color);
    Entity* e = nullptr;
    switch (d.kind) {
    case G19_IMP_SPHERE: e = new ImpSphere(v3(d.p), d.f[0], color); break;
    case G19_IMP_TRIANGLE: e = new ImpTriangle(v3(d.p), v3(d.p + 3), v3(d.p + 6)); break;
    case G19_EXP_RECTANGLE: e = new ExpRectangle(v3(d.p), v3(d.p + 3), v3(d.p + 6)); break;
    case G19_EXP_BOX: e = new ExpBox(v3(d.p), v3(d.p + 3)); break;
    case G19_EXP_SPHERE: e = new ExpSphere(v3(d.p), d.f[0], color); break;
    case G19_EXP_QUAD: e = new ExpQuad(v3(d.p), d.f[0], d.f[1], d.f[2], color); break;
    case G19_EXP_CUBE: e = new ExpCube(v3(d.p), d.f[0], d.f[1], d.f[2], color); break;
    case G19_EXP_CONE: e = new ExpCone(v3(d.p), v3(d.p + 3), d.f[0], d.f[1], color); break;
    default: return nullptr;
    }
    // kinds whose constructor takes no colour: assign the public field
    if (d.kind == G19_IMP_TRIANGLE || d.kind == G19_EXP_RECTANGLE || d.kind == G19_EXP_BOX)
        e->material = Material(color);
    // a caller who assigned the other public Material fields (material.h:24-29) after construction
    if (d.material_set) {
        e->material.diffuse_color = v3(d.diffuse_color);
        e->material.specular_color = v3(d.specular_color);
        e->material.shader_parameters = v3(d.shader_parameters);
        e->material.specular_power = d.specular_power;
    }
    return e;
}

const std::vector<Entity*>* composite_tris(const Entity* e, int kind) {
    switch (kind) {
    case G19_EXP_SPHERE: return &static_cast<const ExpSphere*>(e)->triangles;
    case G19_EXP_QUAD: return &static_cast<const ExpQuad*>(e)->triangles;
    case G19_EXP_CUBE: return &static_cast<const ExpCube*>(e)->triangles;
    case G19_EXP_CONE: return &static_cast<const ExpCone*>(e)->triangles;
    default: return nullptr;
    }
}

void put_tri(const ImpTriangle* t, double* out) {
    for (int k = 0; k < 3; ++k) {
        out[k] = t->p1[k];
        out[3 + k] = t->p2[k];
        out[6 + k] = t->p3[k];
    }
}

// One pixel of raytracer.h:41-84, public API only.
struct PixelOut {
    int id;
    glm::dvec3 point, normal, colour;
};

inline PixelOut trace_pixel(const RefScene& s, const Camera& cam, const glm::dvec3& light,
                            const glm::dvec3& top_left, const glm::dvec3& left, int x, int y,
                            bool shade) {
    glm::dvec2 resolution = {0.0002, 0.0002};
    glm::dvec3 direction = top_left - left * double(x) * resolution.x - cam.up * double(y) * resolution.y;
    Ray r = Ray(cam.pos, direction);
    std::vector<Entity*> objects = s.tree.intersect(r);
    glm::dvec3 intersect = glm::dvec3{DBL_MAX, DBL_MAX, DBL_MAX};
    glm::dvec3 normal = glm::dvec3{0, 0, 0};
    Entity* front = nullptr;
    for (size_t i = 0; i < objects.size(); i++) {
        glm::dvec3 ci = glm::dvec3{0, 0, 0}, cn = glm::dvec3{0, 0, 0};
        // min_dist_square lives INSIDE the loop (raytracer.h:58): every hit wins.
        if (objects[i]->intersect(r, ci, cn)) {
            intersect = ci;
            normal = cn;
            front = objects[i];
        }
    }
    PixelOut o;
    o.id = front ? s.ids.at(front) : -1;
    o.point = intersect;
    o.normal = normal;
    o.colour = glm::dvec3{0, 0, 0};
    if (front && shade) {
        auto coord = front->getTextureCoord(intersect);
        o.colour = front->material.blinn_phong_texture(r, light, intersect, normal, std::get<0>(coord),
                                                       std::get<1>(coord));
    }
    return o;
}

} // namespace

extern "C" {

void* g19ref_scene_create(const double mn[3], const double mx[3]) { return new RefScene(v3(mn), v3(mx)); }

void g19ref_scene_destroy(void* h) { delete static_cast<RefScene*>(h); } // entities leak, like main.cpp

int g19ref_scene_add(void* h, const g19_entity_desc* d) {
    RefScene* s = static_cast<RefScene*>(h);
    Entity* e = make_entity(*d);
    if (!e) return -1;
    int id = int(s->entities.size());
    s->entities.push_back(e);
    s->ids[e] = id;
    s->tree.push_back(e);
    return id;
}

int g19ref_entity_count(void* h) { return int(static_cast<RefScene*>(h)->entities.size()); }

int g19ref_entity_bbox(void* h, int idx, double out[6]) {
    RefScene* s = static_cast<RefScene*>(h);
    BoundingBox b = s->entities.at(idx)->boundingBox();
    for (int k = 0; k < 3; ++k) { out[k] = b.min[k]; out[3 + k] = b.max[k]; }
    return 0;
}

int g19ref_entity_triangles(void* h, int idx, int kind, double* out, int max_tris) {
    RefScene* s = static_cast<RefScene*>(h);
    const Entity* e = s->entities.at(idx);
    if (kind == G19_IMP_TRIANGLE) {
        if (max_tris > 0) put_tri(static_cast<const ImpTriangle*>(e), out);
        return 1;
    }
    if (kind == G19_EXP_RECTANGLE) {
        const ExpRectangle* r = static_cast<const ExpRectangle*>(e);
        if (max_tris > 0) put_tri(&r->t1, out);
        if (max_tris > 1) put_tri(&r->t2, out + 9);
        return 2;
    }
    if (kind == G19_EXP_BOX) {
        const ExpBox* b = static_cast<const ExpBox*>(e);
        int n = 0;
        for (auto& f : b->faces) {
            if (n < max_tris) put_tri(&f->t1, out + 9 * n);
            ++n;
            if (n < max_tris) put_tri(&f->t2, out + 9 * n);
            ++n;
        }
        return n;
    }
    const std::vector<Entity*>* tris = composite_tris(e, kind);
    if (!tris) return 0;
    int n = 0;
    for (Entity* t : *tris) {
        if (n < max_tris) put_tri(static_cast<const ImpTriangle*>(t), out + 9 * n);
        ++n;
    }
    return n;
}

// Derived members of an ImpTriangle built from three points (entities.h:138-148).
int g19ref_triangle_derived(const double p[9], double out_pos_e1_e2_n[12]) {
    ImpTriangle t(v3(p), v3(p + 3), v3(p + 6));
    for (int k = 0; k < 3; ++k) {
        out_pos_e1_e2_n[k] = t.pos[k];
        out_pos_e1_e2_n[3 + k] = t.edge1[k];
        out_pos_e1_e2_n[6 + k] = t.edge2[k];
        out_pos_e1_e2_n[9 + k] = t.normal[k];
    }
    return 0;
}

int g19ref_intersect(void* h, int idx, int n, const double* o, const double* d, int32_t* hit,
                     double* points, double* normals) {
    RefScene* s = static_cast<RefScene*>(h);
    const Entity* e = s->entities.at(idx);
    for (int i = 0; i < n; ++i) {
        Ray r(v3(o + 3 * i), v3(d + 3 * i));
        glm::dvec3 p{0, 0, 0}, nn{0, 0, 0};
        hit[i] = e->intersect(r, p, nn) ? 1 : 0;
        for (int k = 0; k < 3; ++k) { points[3 * i + k] = p[k]; normals[3 * i + k] = nn[k]; }
    }
    return 0;
}

int g19ref_texcoord(void* h, int idx, int n, const double* points, int32_t* uv) {
    RefScene* s = static_cast<RefScene*>(h);
    const Entity* e = s->entities.at(idx);
    for (int i = 0; i < n; ++i) {
        auto c = e->getTextureCoord(v3(points + 3 * i));
        uv[2 * i] = std::get<0>(c);
        uv[2 * i + 1] = std::get<1>(c);
    }
    return 0;
}

int g19ref_shade(void* h, int idx, const double o[3], const double d[3], const double light[3],
                 const double point[3], const double normal[3], int u, int v, double rgb[3]) {
    RefScene* s = static_cast<RefScene*>(h);
    Entity* e = s->entities.at(idx);
    Ray r(v3(o), v3(d));
    glm::dvec3 c = e->material.blinn_phong_texture(r, v3(light), v3(point), v3(normal), u, v);
    rgb[0] = c.x; rgb[1] = c.y; rgb[2] = c.z;
    return 0;
}

int g19ref_candidates(void* h, const double o[3], const double d[3], int32_t* out, int max_out) {
    RefScene* s = static_cast<RefScene*>(h);
    Ray r(v3(o), v3(d));
    std::vector<Entity*> c = s->tree.intersect(r);
    int n = 0;
    for (Entity* e : c) {
        if (n < max_out) out[n] = s->ids.at(e);
        ++n;
    }
    return n;
}

// RayTracer::run, verbatim. rgb = w*h*3 bytes.
int g19ref_render(void* h, const g19_camera* cam, const double light[3], int w, int hgt, uint8_t* rgb) {
    RefScene* s = static_cast<RefScene*>(h);
    Camera camera(v3(cam->pos), v3(cam->look_at), cam->focal);
    RayTracer rt(camera, v3(light));
    rt.setScene(&s->tree);
    rt.start();
    rt.run(w, hgt);
    const QImage& im = Viewer::bits(*rt.getImage());
    std::memcpy(rgb, im.bits(), size_t(w) * size_t(hgt) * 3);
    return 0;
}

// Restated loop over rows [y0,y1), optionally on several threads. Any output
// pointer may be NULL. ids: int32 per pixel; points/normals: 3 doubles per
// pixel; rgb: 3 bytes per pixel; all indexed by the FULL image (y*w+x).
int g19ref_trace(void* h, const g19_camera* cam, const double light_[3], int w, int hgt, int y0, int y1,
                 int32_t* ids, double* points, double* normals, uint8_t* rgb, int nthreads) {
    const RefScene* s = static_cast<RefScene*>(h);
    Camera camera(v3(cam->pos), v3(cam->look_at), cam->focal);
    glm::dvec3 light = v3(light_);
    glm::dvec2 resolution = {0.0002, 0.0002};
    glm::dvec3 left = glm::normalize(glm::cross(camera.up, camera.forward));
    glm::dvec3 top_left = (camera.pos + camera.focalDist * camera.forward + left * double(w) * 0.5 * resolution.x +
                           camera.up * double(w) * 0.5 * resolution.y) -
                          camera.pos;
    if (nthreads < 1) nthreads = 1;
    auto band = [&](int t) {
        for (int y = y0 + t; y < y1; y += nthreads) {
            for (int x = 0; x < w; ++x) {
                PixelOut o = trace_pixel(*s, camera, light, top_left, left, x, y, rgb != nullptr);
                size_t i = size_t(y) * w + x;
                if (ids) ids[i] = o.id;
                if (points) for (int k = 0; k < 3; ++k) points[3 * i + k] = o.point[k];
                if (normals) for (int k = 0; k < 3; ++k) normals[3 * i + k] = o.normal[k];
                if (rgb) {
                    QRgb c = QColor((int)(255 * o.colour.r), (int)(255 * o.colour.g), (int)(255 * o.colour.b)).rgb();
                    rgb[3 * i] = uint8_t(qRed(c));
                    rgb[3 * i + 1] = uint8_t(qGreen(c));
                    rgb[3 * i + 2] = uint8_t(qBlue(c));
                }
            }
        }
    };
    if (nthreads == 1) {
        band(0);
    } else {
        std::vector<std::thread> th;
        for (int t = 0; t < nthreads; ++t) th.emplace_back(band, t);
        for (auto& t : th) t.join();
    }
    return 0;
}

} // extern "C"

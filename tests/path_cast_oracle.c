/* path_cast_oracle.c -- the PATH oracle's answer to batched ray queries (g19_cast_rays), for the tests.
 *
 * TEST INFRASTRUCTURE ONLY. It compiles oracle/path_oracle.c into the same translation unit, so that the queries run
 * through that file's own primitive extraction (build_prims: FIXED shapes included), closest() / occluded() and their
 * uniform-grid acceleration, and answer by g19o_path_primary's id and normal rule. tests/cast_util.py builds it into
 * a temporary directory; the scene handle is one made by oracle/libg19oracle.so (same o_scene layout, same source).
 *
 * g19o_path_cast: n rays (o, d) as row-major triples, bounds tmax; any = occlusion query. The direction is normalised;
 * a ray whose origin or direction is not finite, whose direction is zero or whose tmax is not > 0 is a miss. A hit is
 * the nearest primitive with 0 < t < tmax (closest()); an occlusion query asks occluded() and reports the nearest
 * primitive's entity. A miss is id -1, t = DBL_MAX, normal 0. normals may be NULL.
 */
#include "path_oracle.c"

int g19o_path_cast(void* scene, int n, const double* o, const double* d, const double* tmax, int any, int32_t* ids, double* t,
                   double* normals) {
    p_scene* ps = build_prims((const o_scene*)scene);
    for (int i = 0; i < n; ++i) {
        const v3 oi = V(o[3 * i], o[3 * i + 1], o[3 * i + 2]), di = V(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
        const double m = fmax(fabs(di.x), fmax(fabs(di.y), fabs(di.z)));
        const int valid = isfinite(oi.x) && isfinite(oi.y) && isfinite(oi.z) && isfinite(di.x) && isfinite(di.y) && isfinite(di.z) &&
                          m > 0 && tmax[i] > 0;
        int pi = -1;
        double th = DBL_MAX;
        v3 u = V(0, 0, 1), nn = V(0, 0, 0);
        if (valid) {
            /* vnorm as g19o_path_primary normalises its rays (bit-equal directions for the same input); scaled first
             * only where the squared length would overflow or underflow */
            u = (m > 1e150 || m < 1e-150) ? vnorm(V(di.x / m, di.y / m, di.z / m)) : vnorm(di);
            if (!any || occluded(ps, oi, u, tmax[i])) {
                pi = closest(ps, oi, u, &th);
                if (!any && pi >= 0 && !(th < tmax[i])) pi = -1;
            }
        }
        if (pi >= 0) {
            const p_prim* pr = &ps->prims[pi];
            const v3 p = vadd(oi, vmul(u, th));
            if (pr->is_tri) nn = vdot(pr->n, u) > 0 ? vmul(pr->n, -1) : pr->n;
            else nn = vmul(vsub(p, pr->c), 1.0 / pr->r);
        } else {
            th = DBL_MAX;
        }
        ids[i] = pi >= 0 ? ps->prims[pi].entity : -1;
        if (t) t[i] = th;
        if (normals) { normals[3 * i] = nn.x; normals[3 * i + 1] = nn.y; normals[3 * i + 2] = nn.z; }
    }
    free_prims(ps);
    return 0;
}

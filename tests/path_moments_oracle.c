/* path_moments_oracle.c -- per-pixel sample moments of the PATH oracle, for the adaptive-sampling tests.
 *
 * TEST INFRASTRUCTURE ONLY. It compiles oracle/path_oracle.c into the same translation unit, so that every sample is
 * that file's own trace_path (same Philox counters, same camera, same transport); tests/adaptive_util.py builds it into
 * a temporary directory. The scene handle is one made by oracle/libg19oracle.so (same o_scene layout, same source).
 *
 * g19o_path_moments: for every pixel of the window [x0,x1) x [y0,y1) of a w x h frame, the FP64 sums over samples
 * [s0, s1) of R, G, B and Y^2 (Y = 0.2126 R + 0.7152 G + 0.0722 B), four doubles per pixel, window row-major.
 */
#include "path_oracle.c"

int g19o_path_moments(void* scene, const g19_camera* cam, int w, int h, int s0, int s1, int max_depth, uint32_t seed, int x0,
                      int y0, int x1, int y1, double* out) {
    p_scene* ps = build_prims((const o_scene*)scene);
    v3 cpos, up, left, top_left;
    camera_basis(cam, w, &cpos, &up, &left, &top_left);
    job j = {ps, cpos, up, left, top_left, w, h, s1, max_depth, x0, y0, x1, y1, 0, 1, seed, NULL, 0, 0};
    for (int y = y0; y < y1; ++y)
        for (int x = x0; x < x1; ++x) {
            double r = 0, g = 0, b = 0, y2 = 0;
            for (int s = s0; s < s1; ++s) {
                const v3 L = trace_path(&j, x, y, (uint32_t)s);
                const double lum = 0.2126 * L.x + 0.7152 * L.y + 0.0722 * L.z;
                r += L.x;
                g += L.y;
                b += L.z;
                y2 += lum * lum;
            }
            double* o = out + 4 * ((size_t)(y - y0) * (size_t)(x1 - x0) + (size_t)(x - x0));
            o[0] = r;
            o[1] = g;
            o[2] = b;
            o[3] = y2;
        }
    free_prims(ps);
    return 0;
}

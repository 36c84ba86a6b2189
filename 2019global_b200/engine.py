"""Python front end of lib2019global_b200.so (ctypes over include/g19.h).

Class and method names follow the reference's host interface so that tests read
like a port of its main.cpp (reference main.cpp:24-59):

    scene = Octree((-20,)*3, (20,)*3)            # include/octree.h:14
    scene.push_back(ImpSphere((3,4,4), 2, (1,0,0)))   # octree.h:20
    rt = RayTracer(Camera((-10,0,0), (1,0,0), 0.1), light=(-10,10,10))
    rt.setScene(scene)                            # raytracer.h:21
    rt.start(); image = rt.run(500, 500)          # raytracer.h:23,91

The compute path is the CUDA library; there is no fallback. Importing this
module without the built .so raises, and creating a RayTracer without a B200
raises G19Error(ERR_NO_DEVICE).
"""
import ctypes as C
import os

import numpy as np

from . import abi

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib2019global_b200.so")

# every symbol include/g19.h declares
EXPORTS = [
    "g19_scene_create", "g19_scene_destroy", "g19_scene_add_entity", "g19_scene_entity_count",
    "g19_scene_get_entity", "g19_scene_entity_bbox", "g19_scene_entity_triangles", "g19_scene_builtin",
    "g19_create", "g19_destroy", "g19_last_error", "g19_upload_scene", "g19_render", "g19_render_device",
    "g19_get_stats", "g19_cancel", "g19_progress", "g19_probe_intersect", "g19_probe_candidates",
    "g19_frame_create", "g19_frame_export", "g19_frame_import", "g19_frame_destroy", "g19_frame_pointers",
    "g19_render_to_frame", "g19_frame_wait", "g19_frame_release", "g19_frame_timeouts",
    "g19_frame_read", "g19_render_progressive", "g19_render_tiles_device", "g19_untile_device", "g19_tile_pixels",
    "g19_probe_texcoord", "g19_probe_shade", "g19_probe_path_tree", "g19_entity_bbox", "g19_entity_triangles",
    "g19_frame_status", "g19_tune", "g19_scene_set_shapes", "g19_cast_rays", "g19_cast_rays_device",
    "g19_render_adaptive", "g19_render_adaptive_device",
]


PASS_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_double, C.POINTER(C.c_uint8))  # g19_pass_fn


class G19Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("g19 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    """Load the C-ABI library (fails loudly when it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("lib2019global_b200.so is missing: run `python -c 'import __graft_entry__ as g; g.build()'`"
                              " -- there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.g19_last_error.restype = C.c_char_p
        L.g19_last_error.argtypes = [C.c_void_p]
        L.g19_scene_destroy.restype = None
        L.g19_scene_destroy.argtypes = [C.c_void_p]
        L.g19_destroy.restype = None
        L.g19_destroy.argtypes = [C.c_void_p]
        L.g19_scene_add_entity.argtypes = [C.c_void_p, C.POINTER(abi.EntityDesc), C.POINTER(C.c_int32)]
        L.g19_scene_get_entity.argtypes = [C.c_void_p, C.c_int32, C.POINTER(abi.EntityDesc)]
        L.g19_scene_entity_count.argtypes = [C.c_void_p]
        L.g19_scene_set_shapes.argtypes = [C.c_void_p, C.c_int]
        L.g19_scene_entity_bbox.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.g19_scene_entity_triangles.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int]
        L.g19_upload_scene.argtypes = [C.c_void_p, C.c_void_p]
        L.g19_render.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.c_void_p, C.POINTER(abi.Params), C.c_void_p,
                                 C.c_void_p, C.c_void_p]
        L.g19_render_device.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.c_void_p, C.POINTER(abi.Params),
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.g19_get_stats.argtypes = [C.c_void_p, C.POINTER(abi.Stats)]
        L.g19_cancel.argtypes = [C.c_void_p]
        L.g19_progress.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        L.g19_probe_intersect.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]
        L.g19_probe_path_tree.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32),
                                          C.POINTER(C.c_uint32)]
        L.g19_probe_candidates.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                           C.POINTER(C.c_int)]
        L.g19_probe_texcoord.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_void_p, C.c_void_p]
        L.g19_probe_shade.argtypes = [C.c_void_p, C.c_int32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                      C.c_void_p]
        L.g19_render_progressive.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.c_void_p, C.POINTER(abi.Params),
                                             C.c_void_p, C.c_void_p, PASS_FN, C.c_void_p, C.c_int]
        L.g19_frame_create.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.g19_frame_export.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.g19_frame_import.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
        L.g19_frame_destroy.restype = None
        L.g19_frame_destroy.argtypes = [C.c_void_p]
        L.g19_frame_pointers.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
        L.g19_render_to_frame.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.c_void_p, C.POINTER(abi.Params),
                                          C.c_void_p, C.c_void_p]
        L.g19_frame_wait.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.g19_frame_release.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.g19_frame_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.g19_frame_timeouts.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint)]
        L.g19_frame_status.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.g19_tune.argtypes = [C.c_void_p, C.c_char_p, C.c_char_p]
        L.g19_cast_rays.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.g19_cast_rays_device.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p]
        L.g19_render_adaptive.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.c_void_p, C.POINTER(abi.Params),
                                          C.POINTER(abi.Adaptive), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.g19_render_adaptive_device.argtypes = [C.c_void_p, C.POINTER(abi.Camera), C.c_void_p, C.POINTER(abi.Params),
                                                 C.POINTER(abi.Adaptive), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                 C.c_void_p]
        _lib = L
    return _lib


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


# ---- entities: constructor arguments exactly as the reference's classes take them ----
def ImpSphere(pos, radius, color, **kw):
    return abi.EntityDesc.make(abi.IMP_SPHERE, pos, [radius], color, **kw)


def ImpTriangle(p1, p2, p3, color=(1.0, 0.0, 0.0), **kw):
    return abi.EntityDesc.make(abi.IMP_TRIANGLE, list(p1) + list(p2) + list(p3), [], color, **kw)


def ExpRectangle(p1, p2, p3, color=(1.0, 0.0, 0.0), **kw):
    return abi.EntityDesc.make(abi.EXP_RECTANGLE, list(p1) + list(p2) + list(p3), [], color, **kw)


def ExpBox(mn, mx, color=(1.0, 0.0, 0.0), **kw):
    return abi.EntityDesc.make(abi.EXP_BOX, list(mn) + list(mx), [], color, **kw)


def ExpSphere(pos, radius, color, **kw):
    return abi.EntityDesc.make(abi.EXP_SPHERE, pos, [radius], color, **kw)


def ExpQuad(pos, width, length, alpha, color, **kw):
    return abi.EntityDesc.make(abi.EXP_QUAD, pos, [width, length, alpha], color, **kw)


def ExpCube(pos, width, length, height, color, **kw):
    return abi.EntityDesc.make(abi.EXP_CUBE, pos, [width, length, height], color, **kw)


def ExpCone(pos, direction, height, radius, color, **kw):
    return abi.EntityDesc.make(abi.EXP_CONE, list(pos) + list(direction), [height, radius], color, **kw)


def Camera(pos, look_at=(0.0, 0.0, 0.0), focal=0.04):
    """camera.h:7-10 (the one-argument form looks at the origin with focal 0.04)."""
    return abi.Camera.make(pos, look_at, focal)


class Octree:
    """Octree(min, max) + push_back (include/octree.h:12-30). Host-side only: no GPU needed."""

    def __init__(self, mn, mx, _handle=None):
        self._L = lib()
        if _handle is not None:
            self.h = _handle
        else:
            h = C.c_void_p()
            rc = self._L.g19_scene_create(abi.d3(mn), abi.d3(mx), C.byref(h))
            if rc != abi.OK:
                raise G19Error(rc, "g19_scene_create")
            self.h = h
        self.min, self.max = tuple(mn), tuple(mx)

    @classmethod
    def builtin(cls, which, n=0, w=500, h=500):
        """One of BASELINE.json's procedural configs -> (scene, camera, light)."""
        L = lib()
        hd = C.c_void_p()
        cam = abi.Camera()
        light = (C.c_double * 3)()
        rc = L.g19_scene_builtin(which, n, w, h, C.byref(hd), C.byref(cam), light)
        if rc != abi.OK:
            raise G19Error(rc, "g19_scene_builtin")
        return cls((-20,) * 3, (20,) * 3, _handle=hd), cam, tuple(light[:])

    def __del__(self):
        try:
            self._L.g19_scene_destroy(self.h)
        except Exception:
            pass

    def push_back(self, desc):
        """Returns (entity_id, accepted). A rejected entity is numbered but not in the tree (octree.h:22-24)."""
        idx = C.c_int32(-1)
        rc = self._L.g19_scene_add_entity(self.h, C.byref(desc), C.byref(idx))
        if rc not in (abi.OK, abi.ERR_REJECTED):
            raise G19Error(rc, "g19_scene_add_entity")
        return idx.value, rc == abi.OK

    def set_shapes(self, fixed):
        """g19_scene_set_shapes: PATH mode traces the composites as their constructors meant them (True) or the
        reference's own triangles, bugs included (False, the default). REF mode is unaffected."""
        rc = self._L.g19_scene_set_shapes(self.h, abi.SHAPES_FIXED if fixed else abi.SHAPES_REF)
        if rc != abi.OK:
            raise G19Error(rc, "g19_scene_set_shapes")

    def __len__(self):
        return self._L.g19_scene_entity_count(self.h)

    def entity(self, i):
        d = abi.EntityDesc()
        rc = self._L.g19_scene_get_entity(self.h, i, C.byref(d))
        if rc != abi.OK:
            raise G19Error(rc, "g19_scene_get_entity")
        return d

    def entities(self):
        return [self.entity(i) for i in range(len(self))]

    def bbox(self, i):
        out = np.zeros(6)
        self._L.g19_scene_entity_bbox(self.h, i, _ptr(out))
        return out

    def triangles(self, i, max_tris=256):
        out = np.zeros((max_tris, 9))
        n = self._L.g19_scene_entity_triangles(self.h, i, _ptr(out), max_tris)
        return out[:min(n, max_tris)].copy()


class RayTracer:
    """RayTracer(camera, light) with setScene/run/start/stop/running (include/raytracer.h:15-101)."""

    def __init__(self, camera, light, device=None):
        self._L = lib()
        self.camera, self.light = camera, tuple(light)
        h = C.c_void_p()
        if device is None:
            rc = self._L.g19_create(None, 0, C.byref(h))
        else:
            dev = (C.c_int * 1)(device)
            rc = self._L.g19_create(dev, 1, C.byref(h))
        if rc != abi.OK:
            raise G19Error(rc, self._L.g19_last_error(None).decode())
        self.h = h
        self._running = False
        self._scene = None

    def __del__(self):
        try:
            self._L.g19_destroy(self.h)
        except Exception:
            pass

    def _check(self, rc, allow=()):
        if rc != abi.OK and rc not in allow:
            raise G19Error(rc, self._L.g19_last_error(self.h).decode())
        return rc

    def setScene(self, scene):
        self._scene = scene  # the reference keeps a non-owning pointer; keep the Python object alive
        self._check(self._L.g19_upload_scene(self.h, scene.h))

    def running(self):
        return self._running

    def start(self):
        self._running = True

    def stop(self):
        self._running = False
        self._L.g19_cancel(self.h)

    def params(self, w, h, mode=abi.MODE_REF, spp=1, max_depth=1, seed=0, rank=0, world=1, spp_per_pass=0, profile=0,
               pixels_per_pass=0):
        return abi.Params(w, h, mode, spp, max_depth, seed, rank, world, spp_per_pass, profile, pixels_per_pass)

    def run(self, w, h, mode=abi.MODE_REF, want=("rgb",), out=None, **kw):
        """Blocking render into host arrays (the reference's run(w,h)). Returns a dict of numpy arrays."""
        if not self._running:  # raytracer.h:32: nothing renders before start()
            return {"rgb": np.zeros((h, w, 3), np.uint8)}
        p = self.params(w, h, mode, **kw)
        out = out or {}
        # (a caller's own buffer -- pinned, in bench.py's e2e leg -- is used as it is; a fresh one is only made when none is
        # given: dict.get's default is evaluated on every call, and zeroing 6 MB cost each frame 0.4 ms)
        rgb = (out["rgb"] if "rgb" in out else np.zeros((h, w, 3), np.uint8)) if "rgb" in want else None
        ids = (out["ids"] if "ids" in out else np.full((h, w), -1, np.int32)) if "ids" in want else None
        rad = (out["radiance"] if "radiance" in out else np.zeros((h, w, 3), np.float32)) if "radiance" in want else None
        self._check(self._L.g19_render(self.h, C.byref(self.camera), abi.d3(self.light), C.byref(p), _ptr(rgb),
                                       _ptr(ids), _ptr(rad)), allow=(abi.ERR_CANCELLED,))
        return {"rgb": rgb, "ids": ids, "radiance": rad}

    def run_progressive(self, w, h, on_pass, min_interval_ms=32, mode=abi.MODE_PATH, want_radiance=False, **kw):
        """run() with the viewer's repaint hook (g19_render_progressive): on_pass(fraction, rgb) is called
        with the samples-so-far image (a (h,w,3) uint8 view, valid during the call); return True to cancel."""
        if not self._running:
            return {"rgb": np.zeros((h, w, 3), np.uint8)}
        p = self.params(w, h, mode, **kw)
        rgb = np.zeros((h, w, 3), np.uint8)
        rad = np.zeros((h, w, 3), np.float32) if want_radiance else None

        def hook(_user, fraction, _px):
            return 1 if on_pass(fraction, rgb) else 0
        cb = PASS_FN(hook)
        self._check(self._L.g19_render_progressive(self.h, C.byref(self.camera), abi.d3(self.light), C.byref(p), _ptr(rgb),
                                                   _ptr(rad), cb, None, int(min_interval_ms)), allow=(abi.ERR_CANCELLED,))
        return {"rgb": rgb, "radiance": rad}

    def run_device(self, p, d_rgb=0, d_ids=0, d_rad=0, stream=0):
        """Asynchronous render into device pointers (ints, e.g. torch.Tensor.data_ptr())."""
        return self._check(self._L.g19_render_device(self.h, C.byref(self.camera), abi.d3(self.light), C.byref(p),
                                                     C.c_void_p(d_rgb), C.c_void_p(d_ids), C.c_void_p(d_rad),
                                                     C.c_void_p(stream)), allow=(abi.ERR_CANCELLED,))

    def run_adaptive(self, w, h, noise_target, min_spp, spp, max_depth, seed=0, want=("rgb", "radiance", "variance", "spp"),
                     out=None, **kw):
        """Blocking PATH-mode render with noise-targeted adaptive sampling (g19_render_adaptive): a 32x32 tile stops once
        its worst pixel's relative standard error is <= noise_target; counts are min_spp * 2^k up to spp. Returns a dict of
        numpy arrays: "rgb" (h,w,3) uint8, "radiance" (h,w,3) float32, "variance" (h,w) float32 (variance of each pixel's
        mean luminance), "spp" (h,w) int32 (each pixel's sample count); None for what `want` leaves out. kw: the other
        params() fields (rank, world, spp_per_pass, pixels_per_pass, profile)."""
        p = self.params(w, h, abi.MODE_PATH, spp=spp, max_depth=max_depth, seed=seed, **kw)
        ad = abi.Adaptive(float(noise_target), int(min_spp))
        out = out or {}
        shapes = {"rgb": ((h, w, 3), np.uint8), "radiance": ((h, w, 3), np.float32), "variance": ((h, w), np.float32),
                  "spp": ((h, w), np.int32)}
        res = {k: ((out[k] if k in out else np.zeros(*shapes[k])) if k in want else None) for k in shapes}
        self._check(self._L.g19_render_adaptive(self.h, C.byref(self.camera), abi.d3(self.light), C.byref(p), C.byref(ad),
                                                _ptr(res["rgb"]), _ptr(res["radiance"]), _ptr(res["variance"]), _ptr(res["spp"])),
                    allow=(abi.ERR_CANCELLED,))
        return res

    def run_adaptive_device(self, p, adaptive, d_rgb=0, d_rad=0, d_var=0, d_spp=0, stream=0):
        """g19_render_adaptive_device into device pointers (ints, e.g. torch.Tensor.data_ptr()); p: abi.Params, adaptive:
        abi.Adaptive. Stream-ordered, but synchronises `stream` once per round."""
        return self._check(self._L.g19_render_adaptive_device(self.h, C.byref(self.camera), abi.d3(self.light), C.byref(p),
                                                              C.byref(adaptive), C.c_void_p(d_rgb), C.c_void_p(d_rad),
                                                              C.c_void_p(d_var), C.c_void_p(d_spp), C.c_void_p(stream)),
                           allow=(abi.ERR_CANCELLED,))

    def cast(self, origins, dirs, tmax=None, any_hit=False, want_normals=False, count=False):
        """Batched ray queries against the PATH view of the scene (g19_cast_rays, blocking). origins, dirs: (n, 3);
        tmax: scalar or (n,), None = unbounded. Returns {"ids": (n,) int32 entity ids (-1 = miss), "t": (n,) float32
        distances along the unit direction (+inf = miss; None for any_hit), "normals": (n, 3) float32 or None}.
        any_hit: occlusion query (ids = an entity hit below tmax, or -1)."""
        o = np.asarray(origins, dtype=np.float32).reshape(-1, 3)
        d = np.asarray(dirs, dtype=np.float32).reshape(-1, 3)
        n = o.shape[0]
        if d.shape[0] != n:
            raise ValueError("origins and dirs must both be (n, 3)")
        buf = np.zeros(n * 8 + 4, np.float32)  # the records must start on a 16-byte boundary
        skip = (-buf.ctypes.data % 16) // 4
        rays = buf[skip:skip + n * 8].reshape(n, 8)
        rays[:, 0:3] = o
        rays[:, 3] = np.inf if tmax is None else np.broadcast_to(np.asarray(tmax, dtype=np.float32), (n,))
        rays[:, 4:7] = d
        ids = np.empty(n, np.int32)
        t = None if any_hit else np.empty(n, np.float32)
        nrm = np.empty((n, 3), np.float32) if want_normals and not any_hit else None
        flags = (abi.CAST_ANY_HIT if any_hit else 0) | (abi.CAST_COUNT if count else 0)
        self._check(self._L.g19_cast_rays(self.h, n, _ptr(rays), flags, _ptr(ids), _ptr(t), _ptr(nrm)))
        return {"ids": ids, "t": t, "normals": nrm}

    def cast_device(self, n, d_rays, d_ids, d_t=0, d_normals=0, flags=0, stream=0):
        """Asynchronous g19_cast_rays_device on device pointers (ints, e.g. torch.Tensor.data_ptr()): d_rays n x 8 float32,
        16-byte aligned; d_ids n int32; d_t n float32 and d_normals n x 3 float32 optional (0)."""
        return self._check(self._L.g19_cast_rays_device(self.h, int(n), C.c_void_p(d_rays), int(flags), C.c_void_p(d_ids),
                                                        C.c_void_p(d_t), C.c_void_p(d_normals), C.c_void_p(stream)))

    def tune(self, key, value=None):
        """g19_tune: set one tuning knob ("lanes", "walk", ...); value None = back to the default."""
        v = None if value is None else str(value).encode()
        self._check(self._L.g19_tune(self.h, key.encode(), v))

    def stats(self):
        s = abi.Stats()
        self._check(self._L.g19_get_stats(self.h, C.byref(s)))
        return s

    def progress(self):
        v = C.c_double(0)
        self._L.g19_progress(self.h, C.byref(v))
        return v.value

    # unit-level probes (tests)
    def probe_intersect(self, entity, origins, dirs):
        o = np.ascontiguousarray(origins, dtype=np.float64)
        d = np.ascontiguousarray(dirs, dtype=np.float64)
        n = o.shape[0]
        hit = np.zeros(n, np.int32)
        pts = np.zeros((n, 3))
        nrm = np.zeros((n, 3))
        self._check(self._L.g19_probe_intersect(self.h, entity, n, _ptr(o), _ptr(d), _ptr(hit), _ptr(pts), _ptr(nrm)))
        return hit, pts, nrm

    def probe_texcoord(self, entity, points):
        """Entity::getTextureCoord (entities.h:32) on the device for n points -> (n, 2) int32."""
        p = np.ascontiguousarray(points, dtype=np.float64)
        uv = np.zeros((p.shape[0], 2), np.int32)
        self._check(self._L.g19_probe_texcoord(self.h, entity, p.shape[0], _ptr(p), _ptr(uv)))
        return uv

    def probe_shade(self, entity, ray_dir, light, point, normal, u=0, v=0, textured=True):
        """Material::blinn_phong_texture / blinn_phong (material.h:31-62) on the device for one point -> 3 doubles."""
        out = (C.c_double * 3)()
        self._check(self._L.g19_probe_shade(self.h, entity, 1 if textured else 0, abi.d3(ray_dir), abi.d3(light), abi.d3(point),
                                            abi.d3(normal), int(u), int(v), out))
        return np.array(out[:])

    def path_tree(self):
        """(nodes (n,2) uint32, index (m,) uint32) of the linear octree PATH mode traverses."""
        nn, ni = C.c_uint32(0), C.c_uint32(0)
        self._check(self._L.g19_probe_path_tree(self.h, None, 0, None, 0, C.byref(nn), C.byref(ni)))
        nodes = np.zeros((nn.value, 2), np.uint32)
        index = np.zeros(max(ni.value, 1), np.uint32)
        self._check(self._L.g19_probe_path_tree(self.h, _ptr(nodes), nn.value, _ptr(index), ni.value, C.byref(nn), C.byref(ni)))
        return nodes, index[:ni.value]

    def probe_candidates(self, o, d, max_out=1 << 16):
        out = np.zeros(max_out, np.int32)
        n = C.c_int(0)
        self._check(self._L.g19_probe_candidates(self.h, abi.d3(o), abi.d3(d), _ptr(out), max_out, C.byref(n)))
        return out[:min(n.value, max_out)].copy()


def tile_pixels(w, h, rank, world):
    """Entries in a rank's compact local-pixel arrays (g19_tile_pixels)."""
    L = lib()
    L.g19_tile_pixels.restype = C.c_int64
    return int(L.g19_tile_pixels(w, h, rank, world))


def _render_tiles(self, p, t_rgb=0, t_ids=0, t_rad=0, stream=0):
    """Render this rank's tiles into compact device arrays (the payload sent to rank 0)."""
    return self._check(self._L.g19_render_tiles_device(self.h, C.byref(self.camera), abi.d3(self.light), C.byref(p),
                                                       C.c_void_p(t_rgb), C.c_void_p(t_ids), C.c_void_p(t_rad),
                                                       C.c_void_p(stream)), allow=(abi.ERR_CANCELLED,))


def _untile(self, w, h, rank, world, t_rgb=0, t_ids=0, t_rad=0, d_rgb=0, d_ids=0, d_rad=0, stream=0):
    """Scatter rank `rank`'s compact arrays into the full frame (device pointers)."""
    return self._check(self._L.g19_untile_device(self.h, w, h, rank, world, C.c_void_p(t_rgb), C.c_void_p(t_ids),
                                                 C.c_void_p(t_rad), C.c_void_p(d_rgb), C.c_void_p(d_ids),
                                                 C.c_void_p(d_rad), C.c_void_p(stream)))


RayTracer.render_tiles = _render_tiles
RayTracer.untile = _untile


FRAME_BLOB_BYTES = 128


class SharedFrame:
    """A frame in the owner's HBM that every rank's resolve kernel stores into directly
    (include/g19.h "shared frame"): SharedFrame.create on rank 0, .blob() shipped to the other
    ranks by any transport, SharedFrame.attach there."""

    def __init__(self, rt, handle, w, h, owner):
        self.rt, self.h_, self.w, self.h, self.owner = rt, handle, w, h, owner

    @classmethod
    def create(cls, rt, w, h):
        hd = C.c_void_p()
        rt._check(rt._L.g19_frame_create(rt.h, w, h, C.byref(hd)))
        return cls(rt, hd, w, h, True)

    @classmethod
    def attach(cls, rt, blob, w, h):
        hd = C.c_void_p()
        buf = C.create_string_buffer(bytes(blob), FRAME_BLOB_BYTES)
        rt._check(rt._L.g19_frame_import(rt.h, buf, FRAME_BLOB_BYTES, C.byref(hd)))
        return cls(rt, hd, w, h, False)

    def blob(self):
        buf = C.create_string_buffer(FRAME_BLOB_BYTES)
        self.rt._check(self.rt._L.g19_frame_export(self.rt.h, self.h_, buf, FRAME_BLOB_BYTES))
        return bytes(buf.raw)

    def pointers(self):
        """(rgb888, radiance) device pointers on the owner."""
        a, b = C.c_void_p(), C.c_void_p()
        self.rt._check(self.rt._L.g19_frame_pointers(self.h_, C.byref(a), C.byref(b)))
        return a.value, b.value

    def render(self, p, stream=0):
        """Every rank: render my tiles straight into the frame (asynchronous)."""
        rt = self.rt
        return rt._check(rt._L.g19_render_to_frame(rt.h, C.byref(rt.camera), abi.d3(rt.light), C.byref(p), self.h_,
                                                   C.c_void_p(stream)), allow=(abi.ERR_CANCELLED,))

    def wait(self, world, stream=0):
        """Owner: everything enqueued on `stream` after this sees the complete frame."""
        self.rt._check(self.rt._L.g19_frame_wait(self.rt.h, self.h_, world, C.c_void_p(stream)))

    def read(self, rgb=0, rad=0, stream=0):
        """Owner: enqueue copies of the frame to host (pinned) or device addresses (ints)."""
        self.rt._check(self.rt._L.g19_frame_read(self.rt.h, self.h_, C.c_void_p(rgb), C.c_void_p(rad), C.c_void_p(stream)))

    def release(self, stream=0):
        """Owner: done reading; the ranks may overwrite the frame with the next one."""
        self.rt._check(self.rt._L.g19_frame_release(self.rt.h, self.h_, C.c_void_p(stream)))

    def check(self, stream=0):
        """Synchronise `stream`, then raise G19Error(ERR_TIMEOUT) if any device-side wait on this frame gave up."""
        self.rt._check(self.rt._L.g19_frame_status(self.rt.h, self.h_, C.c_void_p(stream)))

    def timeouts(self):
        v = C.c_uint(0)
        self.rt._check(self.rt._L.g19_frame_timeouts(self.rt.h, self.h_, C.byref(v)))
        return v.value

    def close(self):
        if self.h_ is not None:
            self.rt._L.g19_frame_destroy(self.h_)
            self.h_ = None

"""ctypes mirror of include/g19.h (struct layouts and enum values only)."""
import ctypes as C

ABI_VERSION = 6

# enum g19_entity_kind (reference include/entities.h, one value per class)
IMP_SPHERE, IMP_TRIANGLE, EXP_RECTANGLE, EXP_BOX, EXP_SPHERE, EXP_QUAD, EXP_CUBE, EXP_CONE = range(8)
KIND_NAMES = ["ImpSphere", "ImpTriangle", "ExpRectangle", "ExpBox", "ExpSphere", "ExpQuad", "ExpCube", "ExpCone"]
# enum g19_bsdf
BSDF_DIFFUSE, BSDF_MIRROR, BSDF_GLASS, BSDF_EMITTER = range(4)
# enum g19_mode
MODE_REF, MODE_PATH = 0, 1
# enum g19_shapes
SHAPES_REF, SHAPES_FIXED = 0, 1
# enum g19_builtin_scene
SCENE_DEFAULT, SCENE_CORNELL, SCENE_CORNELL_GLASS, SCENE_HEIGHTFIELD, SCENE_HEIGHTFIELD_ROOM = range(5)
# status
OK, ERR_INVALID, ERR_NO_DEVICE, ERR_CUDA, ERR_NO_SCENE, ERR_CANCELLED, ERR_LIMIT, ERR_REJECTED, ERR_TIMEOUT = range(9)
# g19_cast_rays flags
CAST_ANY_HIT, CAST_COUNT = 1, 2
K_EXTEND, K_SHADE, K_SHADOW, K_ACCUM, K_REF_VIS, K_REF_SHADE, K_OTHER = range(7)
CLASS_NAMES = ["raygen_extend", "bounce", "shadow", "accumulate", "ref_visibility", "ref_shade", "other", "_"]


class EntityDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("bsdf", C.c_int32), ("p", C.c_double * 9), ("f", C.c_float * 4),
                ("color", C.c_double * 3), ("emission", C.c_float * 3), ("ior", C.c_float),
                ("material_set", C.c_int32), ("reserved_", C.c_int32), ("diffuse_color", C.c_double * 3),
                ("specular_color", C.c_double * 3), ("shader_parameters", C.c_double * 3), ("specular_power", C.c_double)]

    @classmethod
    def make(cls, kind, p=(), f=(), color=(1.0, 0.0, 0.0), bsdf=BSDF_DIFFUSE, emission=(0.0, 0.0, 0.0), ior=1.5,
             diffuse_color=None, specular_color=None, shader_parameters=None, specular_power=None):
        d = cls()
        if any(v is not None for v in (diffuse_color, specular_color, shader_parameters, specular_power)):
            # the reference's Material(color) defaults (material.h:13-16,27,29) for whatever the caller left alone
            d.material_set = 1
            for i in range(3):
                d.diffuse_color[i] = (diffuse_color or [0.5 * c for c in color])[i]
                d.specular_color[i] = (specular_color or (1.0, 1.0, 1.0))[i]
                d.shader_parameters[i] = (shader_parameters or (0.1, 0.7, 1.0))[i]
            d.specular_power = 5.0 if specular_power is None else specular_power
        d.kind, d.bsdf, d.ior = kind, bsdf, ior
        for i, v in enumerate(p):
            d.p[i] = v
        for i, v in enumerate(f):
            d.f[i] = v
        for i, v in enumerate(color):
            d.color[i] = v
        for i, v in enumerate(emission):
            d.emission[i] = v
        return d


class Camera(C.Structure):
    _fields_ = [("pos", C.c_double * 3), ("look_at", C.c_double * 3), ("focal", C.c_double)]

    @classmethod
    def make(cls, pos, look_at, focal):
        c = cls()
        c.pos[:] = list(pos)
        c.look_at[:] = list(look_at)
        c.focal = focal
        return c


class Params(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("mode", C.c_int32), ("spp", C.c_int32),
                ("max_depth", C.c_int32), ("seed", C.c_uint32), ("rank", C.c_int32), ("world", C.c_int32),
                ("spp_per_pass", C.c_int32), ("profile", C.c_int32), ("pixels_per_pass", C.c_int32)]


class Adaptive(C.Structure):
    """g19_adaptive: a tile stops once its error is <= noise_target; every owned pixel first takes min_spp samples."""
    _fields_ = [("noise_target", C.c_float), ("min_spp", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("extend_segments", C.c_uint64), ("shadow_segments", C.c_uint64),
                ("kernel_launches", C.c_uint64), ("render_ms", C.c_double), ("class_ms", C.c_double * 8),
                ("class_launches", C.c_uint64 * 8), ("node_tests", C.c_uint64), ("prim_tests", C.c_uint64),
                ("shade_calls", C.c_uint64), ("shade_calls_first", C.c_uint64), ("lit_samples", C.c_uint64),
                ("radiance_reads", C.c_uint64), ("radiance_stores", C.c_uint64), ("shade_calls_folded", C.c_uint64)]


def d3(v):
    return (C.c_double * 3)(*[float(x) for x in v])

"""Ray sets for the batched ray-query tests (g19_cast_rays), all in FP64 and seeded, and the PATH oracle's answer to
them (tests/path_cast_oracle.c)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_cast_lib = None


def _oracle_cast_lib():
    """tests/path_cast_oracle.c (oracle/path_oracle.c plus g19o_path_cast), compiled once per process into a temporary
    directory with the flags of oracle/Makefile."""
    global _cast_lib
    if _cast_lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="g19_cast_oracle_"), "libg19castoracle.so")
        subprocess.run(["/usr/bin/gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread",
                        "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle"), "-Wall", "-Wno-unused-function",
                        os.path.join(HERE, "path_cast_oracle.c"), "-o", out, "-lm"], check=True)
        lib = C.CDLL(out)
        lib.g19o_path_cast.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 3
        _cast_lib = lib
    return _cast_lib


def path_cast(scene, origins, dirs, tmax=None, any_hit=False):
    """PATH oracle's batched ray queries (FP64) on an oracle CheckerScene -> ids (n,) int32, t (n,) (DBL_MAX = miss),
    normals (n, 3)."""
    assert scene.lib.which == "oracle"
    o = np.ascontiguousarray(origins, np.float64).reshape(-1, 3)
    d = np.ascontiguousarray(dirs, np.float64).reshape(-1, 3)
    n = o.shape[0]
    tm = np.ascontiguousarray(np.broadcast_to(np.inf if tmax is None else np.asarray(tmax, np.float64), (n,)), np.float64)
    ids = np.full(n, -2, np.int32)
    t = np.zeros(n)
    nrm = np.zeros((n, 3))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    _oracle_cast_lib().g19o_path_cast(scene.h, n, p(o), p(d), p(tm), 1 if any_hit else 0, p(ids), p(t), p(nrm))
    return ids, t, nrm


def corner_rays(cam, w, h):
    """The un-jittered rays through the integer pixel corners (raytracer.h:41-43; the basis of path_oracle.c's
    camera_basis, the reference's vertical pitch included) -> origins (h*w, 3), directions (h*w, 3), row-major. The
    directions are the ones g19o_path_primary normalises: a cast normalises them the same way."""
    cpos = np.array(cam.pos[:])
    fwd = np.array(cam.look_at[:]) - cpos
    fwd = fwd * (1.0 / np.sqrt(fwd[0] * fwd[0] + fwd[1] * fwd[1] + fwd[2] * fwd[2]))
    up = np.array([0.0, 0.0, 1.0])
    left = np.array([up[1] * fwd[2] - fwd[1] * up[2], up[2] * fwd[0] - fwd[2] * up[0], up[0] * fwd[1] - fwd[0] * up[1]])
    left = left * (1.0 / np.sqrt(left[0] * left[0] + left[1] * left[1] + left[2] * left[2]))
    t = cpos + cam.focal * fwd
    t = t + left * float(w) * 0.5 * 0.0002
    t = t + up * float(w) * 0.5 * 0.0002
    top_left = t - cpos
    ys, xs = np.mgrid[0:h, 0:w]
    fx = (xs.astype(np.float64) * 0.0002).reshape(-1, 1)
    fy = (ys.astype(np.float64) * 0.0002).reshape(-1, 1)
    d = top_left[None, :] - left[None, :] * fx - up[None, :] * fy
    return np.repeat(cpos[None, :], h * w, 0), d


def unit(d):
    return d / np.linalg.norm(d, axis=1, keepdims=True)


def as_cast(o, d):
    """The rays as a cast receives them: origins and directions rounded to FP32 (then held in FP64 for the oracle). A
    ray leaving a surface hits its neighbours at small t, where the rounding of the origin moves the hit further than
    the robustness test's turn of the direction does -- so the oracle is asked about the rays the GPU actually casts."""
    return o.astype(np.float32).astype(np.float64), d.astype(np.float32).astype(np.float64)


def bounce_rays(points, normals, n, seed=0, eps=1e-3):
    """n rays leaving surface points (picked at random from the given hits), offset by eps along the normal (the side the
    hit was seen from), cosine-distributed around it."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, len(points), n)
    p, nn = points[k], normals[k]
    nn = nn / np.linalg.norm(nn, axis=1, keepdims=True)
    a = np.where(np.abs(nn[:, :1]) > 0.9, np.array([[0.0, 1.0, 0.0]]), np.array([[1.0, 0.0, 0.0]]))
    tx = np.cross(nn, a)
    tx /= np.linalg.norm(tx, axis=1, keepdims=True)
    ty = np.cross(nn, tx)
    u1, u2 = rng.random(n), rng.random(n)
    r, phi = np.sqrt(u1), 2 * np.pi * u2
    d = tx * (r * np.cos(phi))[:, None] + ty * (r * np.sin(phi))[:, None] + nn * np.sqrt(np.maximum(0.0, 1 - u1))[:, None]
    return p + eps * nn, d / np.linalg.norm(d, axis=1, keepdims=True)


def box_rays(lo, hi, n, seed=0):
    """n rays with uniform origins inside the box lo..hi and uniform directions."""
    rng = np.random.default_rng(seed)
    o = rng.uniform(np.asarray(lo, float), np.asarray(hi, float), (n, 3))
    d = rng.normal(size=(n, 3))
    return o, d / np.linalg.norm(d, axis=1, keepdims=True)


def perturbed(d, eps=1e-5):
    """Six copies of the directions d turned by eps radians (both ways about two axes and the diagonals between)."""
    d = unit(d)
    a = np.where(np.abs(d[:, :1]) > 0.9, np.array([[0.0, 1.0, 0.0]]), np.array([[1.0, 0.0, 0.0]]))
    t = np.cross(d, a)
    t /= np.linalg.norm(t, axis=1, keepdims=True)
    b = np.cross(d, t)
    out = []
    for e in (t, -t, b, -b, (t + b) / np.sqrt(2), -(t + b) / np.sqrt(2)):
        q = np.cos(eps) * d + np.sin(eps) * e
        out.append(q / np.linalg.norm(q, axis=1, keepdims=True))
    return out


def robust_mask(chk, o, d):
    """Rays whose oracle id does not change under perturbed(): the ones FP32 and FP64 must agree on. Returns (mask, ids,
    t, normals) of the oracle's cast of (o, d)."""
    ids, t, nrm = path_cast(chk, o, d)
    ok = np.ones(len(ids), bool)
    for q in perturbed(d):
        ok &= path_cast(chk, o, q)[0] == ids
    return ok, ids, t, nrm

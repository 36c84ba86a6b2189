"""Shared helpers for the parity tests."""
import contextlib
import hashlib
import math
import os

import numpy as np


@contextlib.contextmanager
def quiet_stdout():
    """The reference prints from ExpRectangle::getTextureCoord (entities.h:362); silence fd 1."""
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    try:
        os.dup2(devnull, 1)
        yield
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
        os.close(saved)


def mirror(checker, octree):
    """The same Octree + entities on a CPU checker, from the product scene's own descriptors."""
    return checker.scene(octree.min, octree.max, octree.entities())


def zoo(g19):
    """One entity of every reference class, in a root that subdivides."""
    E = g19
    sc = g19.Octree((-20,) * 3, (20,) * 3)
    descs = [
        E.ImpSphere((3, 4, 4), 2, (1, 0, 0)),
        E.ImpTriangle((3, -2, 1), (3, 2, -1), (3, -2, -1), (0, 1, 0)),
        E.ExpRectangle((0, 0, 0), (3, 3, 3), (3, 3, 0), (1, 1, 0)),
        E.ExpBox((1, 1, 1), (3, 4, 5), (0, 1, 1)),
        E.ExpSphere((-2, 0, 0), 2, (0, 1, 0)),
        E.ExpQuad((0.5, 0.2, 0.3), 2, 3, 0.7, (1, 2, 3)),
        E.ExpCube((0.3, -0.4, 1), 2, 2.5, 1.5, (1, 0, 0)),
        E.ExpCone((0, 0, 2), (-1, 1, -3), 5, 3, (1, 1, 0)),
        E.ImpSphere((-3, -4, -4), 1.5, (0, 0, 1)),
    ]
    for d in descs:
        sc.push_back(d)
    return sc


def probe_rays(n, seed=0):
    rng = np.random.default_rng(seed)
    o = rng.uniform(-12, 12, (n, 3))
    tgt = rng.uniform(-4, 4, (n, 3))
    d = tgt - o
    k = min(50, n // 8)
    d[:k] = [1, 0, 0]
    d[k:2 * k] = [0, 1, 0]
    d[2 * k:3 * k] = [0, 0, 1]
    d[3 * k:4 * k] = [0, 0, -1]
    return o, d


def rel_rmse(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return math.sqrt(np.mean((a - b) ** 2)) / max(np.mean(b), 1e-12)


# ---- what the comparisons against the reference compute (tests/test_oracle_ref.py), for any CPU checker --------
# The same functions generate tests/golden/ref_live.npz (tests/golden/make_golden_live.py), so a test compares the
# restatement with the stored vectors always and with the compiled reference (oracle/_ref) where it is built.
def sha(b):
    return np.frombuffer(hashlib.sha256(b).digest(), np.uint8)


def live_golden():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_live.npz"))


def reference_checker():
    """The compiled, unmodified reference (oracle/_ref) where it is built, else None."""
    from oracle import binding
    return binding.CheckerLib("ref") if binding.available("ref") else None


def assert_same(got, exp):
    """Byte equality of every array in `exp` with the same key in `got`."""
    for k, v in exp.items():
        a, b = np.asarray(got[k]), np.asarray(v)
        assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes(), k


def live_zoo(checker, z):
    """zoo(): per entity, hits, hit points + normals (hashed) and texture coordinates of 5000 probe rays; triangle_derived
    of 50 random triangles. The points fed to getTextureCoord are the checker's own hits."""
    c = mirror(checker, z)
    out = {}
    for i in range(len(z)):
        o, d = probe_rays(5000, seed=100 + i)
        h, p, n = c.intersect(i, o, d)
        m = h.astype(bool)
        out["zoo_%d_hit" % i] = np.packbits(m)
        out["zoo_%d_ptsha" % i] = sha(p[m].tobytes() + n[m].tobytes())
        with quiet_stdout():  # the reference prints from ExpRectangle::getTextureCoord
            out["zoo_%d_uv" % i] = c.texcoord(i, p[m][:300])
    tri = np.random.default_rng(1).uniform(-5, 5, (50, 9))
    out["tri_derived"] = np.array([c.triangle_derived(t) for t in tri])
    return out


def live_frame_scenes(abi):
    """(scene, n, (w, h)) of the small frames traced through each checker's octree."""
    return ((abi.SCENE_DEFAULT, 0, (120, 120)), (abi.SCENE_CORNELL, 0, (64, 36)), (abi.SCENE_CORNELL_GLASS, 0, (48, 48)),
            (abi.SCENE_HEIGHTFIELD, 20, (48, 27)))


def live_frames(checker, g19, abi):
    """Hashes of ids / points / normals / rgb of the per-pixel trace, and of run()'s own image, per frame scene."""
    out = {}
    for which, n, (w, h) in live_frame_scenes(abi):
        sc, cam, light = g19.Octree.builtin(which, n=n, w=w, h=h)
        c = mirror(checker, sc)
        with quiet_stdout():
            t = c.trace(cam, light, w, h, threads=4)
            run_rgb = c.render(cam, light, w, h)
        for k in ("ids", "points", "normals", "rgb"):
            out["frame_%d_%s" % (which, k)] = sha(t[k].tobytes())
        out["frame_%d_run" % which] = sha(run_rgb.tobytes())
    return out


def material_descs(g19):
    """Two entities whose Material fields beyond `color` are assigned after construction, one left at the defaults."""
    custom = dict(shader_parameters=(0.25, 0.5, 0.6), specular_color=(0.9, 0.4, 0.2), specular_power=9.0, diffuse_color=(0.1, 0.2, 0.3))
    return [g19.ImpSphere((3, 1, 0), 2.0, (1, 0, 2), **custom),
            g19.ImpTriangle((4, -5, -3), (4, 5, -3), (4, 0, 4), (0, 1, 1), **custom),
            g19.ImpSphere((3, -3, 2), 1.5, (0, 1, 0))]


def live_material(checker, g19):
    """Material::blinn_phong_texture of material_descs() at 40 random points each, and a 96x96 frame (ids, rgb)."""
    rng = np.random.default_rng(11)
    sc = checker.scene((-20,) * 3, (20,) * 3, material_descs(g19))
    shades = []
    for i in range(3):
        for _ in range(40):
            o = (-10, 0, 0)
            p = rng.uniform(-3, 3, 3)
            n = rng.normal(size=3)
            n /= np.linalg.norm(n)
            d = p - np.array(o)
            light = rng.uniform(-10, 10, 3)
            u, v = (int(x) for x in rng.integers(0, 200, 2))
            with quiet_stdout():
                shades.append(sc.shade(i, o, d, light, p, n, u, v))
    cam = g19.Camera((-10, 0, 0), (1, 0, 0), 0.02)
    with quiet_stdout():
        f = sc.trace(cam, (-8, 6, 9), 96, 96, want=("rgb", "ids"), threads=2)
    return {"material_shade": np.array(shades), "material_ids": f["ids"], "material_rgb": f["rgb"]}

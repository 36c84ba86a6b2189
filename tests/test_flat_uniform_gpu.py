"""Flat scenes whose primitive pairs fit the flat bounce kernels' FlatPairsU launch parameter (tune flat_uniform, default on) trace
through pair loops unrolled to that capacity, with the coefficients as constant-bank operands, instead of the loops over
the pairs staged in shared memory. Same operations in the same order per lane, so every frame must be bit-identical to
the shared-memory form, with the same segment counts: on the Cornell boxes (diffuse-only; mirror / glass), on flat
scenes just under and just over the capacity (8 parallelogram pairs, 8 triangle pairs, 4 sphere pairs: the larger scene
keeps the shared-memory loops either way), and on odd, even and empty kind groups."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _render(g19, abi, sc, cam, light, w, h, uniform, tune=(), **kw):
    rt = g19.RayTracer(cam, light)
    rt.tune("flat_uniform", uniform)
    for k, v in tune:
        rt.tune(k, v)
    rt.setScene(sc)
    rt.start()
    rad = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), **kw)["radiance"]
    st = rt.stats()
    return rad, int(st.extend_segments), int(st.shadow_segments)


def _same(g19, abi, sc, cam, light, w, h, tune=(), **kw):
    on = _render(g19, abi, sc, cam, light, w, h, 1, tune, **kw)
    off = _render(g19, abi, sc, cam, light, w, h, 0, tune, **kw)
    assert on[0].max() > 0
    assert on[0].tobytes() == off[0].tobytes(), (tune, kw)
    assert on[1:] == off[1:], (tune, kw, on[1:], off[1:])


@pytest.mark.parametrize("depth,spp,spp_pass", [(1, 3, 0), (2, 4, 0), (5, 6, 0), (5, 6, 2)])
def test_cornell_bit_identical(g19, abi, depth, spp, spp_pass):
    w, h = 150, 97  # ragged tiles
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    _same(g19, abi, sc, cam, light, w, h, spp=spp, max_depth=depth, seed=8, spp_per_pass=spp_pass)


@pytest.mark.parametrize("depth", [1, 2, 5, 8])
@pytest.mark.parametrize("spp_pass", [2, 5])  # three passes of 2, 2 and 1 samples / one pass
def test_cornell_glass_bit_identical(g19, abi, depth, spp_pass):
    w, h = 150, 97
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL_GLASS, w=w, h=h)
    _same(g19, abi, sc, cam, light, w, h, spp=5, max_depth=depth, seed=3, spp_per_pass=spp_pass)


def _scene(g19, abi, n_quads, n_tris, n_spheres, seed=4):
    """One leaf (leaf_max raised by the caller): an emitter triangle overhead, n_quads parallelograms (two coplanar
    triangles each, merged by the builder), n_tris triangles and n_spheres spheres (diffuse, mirror, glass in turn)
    scattered in front of the camera."""
    rng = np.random.default_rng(seed)
    sc = g19.Octree((-20,) * 3, (20,) * 3)
    sc.push_back(g19.ImpTriangle((-4, -9, 9), (-4, 9, 9), (8, 0, 9), (1, 1, 1), bsdf=abi.BSDF_EMITTER, emission=(9.0, 8.0, 7.0)))
    sc.push_back(g19.ImpTriangle((9, -12, -12), (9, 12, -12), (9, 12, 12), (0.7, 0.7, 0.7)))  # back wall: 1 parallelogram
    sc.push_back(g19.ImpTriangle((9, -12, -12), (9, 12, 12), (9, -12, 12), (0.7, 0.7, 0.7)))
    for _ in range(n_quads - 1):
        a = rng.uniform((0, -7, -7), (8, 7, 7))
        e1, e2 = rng.uniform(-1.5, 1.5, 3), rng.uniform(-1.5, 1.5, 3)
        col = tuple(rng.uniform(0.3, 0.9, 3))
        b, c, d = a + e1, a + e1 + e2, a + e2
        sc.push_back(g19.ImpTriangle(tuple(a), tuple(b), tuple(c), col))
        sc.push_back(g19.ImpTriangle(tuple(a), tuple(c), tuple(d), col))
    for _ in range(n_tris):
        a = rng.uniform((0, -7, -7), (8, 7, 7))
        sc.push_back(g19.ImpTriangle(tuple(a), tuple(a + rng.uniform(-2, 2, 3)), tuple(a + rng.uniform(-2, 2, 3)),
                                     tuple(rng.uniform(0.3, 0.9, 3))))
    kinds = (abi.BSDF_DIFFUSE, abi.BSDF_MIRROR, abi.BSDF_GLASS)
    for k in range(n_spheres):
        sc.push_back(g19.ImpSphere(tuple(rng.uniform((0, -6, -6), (8, 6, 6))), float(rng.uniform(0.4, 1.2)), (0.9, 0.8, 0.7),
                                   bsdf=kinds[k % 3]))
    return sc


# (parallelograms, triangles besides the emitter, spheres): at the capacity, one pair over it per kind, and odd / even /
# empty groups as in test_path_gpu.py::test_flat_scene_pair_padding
@pytest.mark.parametrize("n_quads,n_tris,n_spheres", [(16, 15, 8), (17, 15, 8), (16, 17, 8), (16, 15, 9),
                                                      (1, 0, 0), (1, 1, 1), (2, 3, 2), (3, 2, 3), (1, 0, 2), (4, 4, 0)])
@pytest.mark.parametrize("depth", [1, 2, 5])
def test_flat_scene_shapes_bit_identical(g19, abi, n_quads, n_tris, n_spheres, depth):
    sc = _scene(g19, abi, n_quads, n_tris, n_spheres)
    cam = g19.Camera((-10, 0, 0), (1, 0, 0), 0.02)
    _same(g19, abi, sc, cam, (0, 0, 0), 96, 64, tune=(("leaf_max", 64),), spp=4, max_depth=depth, seed=5, spp_per_pass=2)

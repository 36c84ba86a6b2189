"""G19_MODE_PATH (wavefront path tracer) on the GPU against the FP64 brute-force oracle.

The reference has no bounce transport (SURVEY.md 8(a) row 14), so the oracle here is this
repo's own definition (oracle/path_oracle.c). Tolerances (SURVEY.md 8(c)):
  (i)  same seed: relRMSE = sqrt(mean((gpu-cpu)^2)) / mean(cpu) <= 1e-2 on linear radiance --
       FP32 vs FP64 paths only part ways at discontinuities;
  (ii) different seeds: relRMSE(gpu, cpu') <= 1.5 x relRMSE(cpu, cpu').
Everything integer is exact: segment counts may differ only by the handful of paths that
diverge at a discontinuity (<= 0.1 %), and the GPU result is bit-identical across runs,
pass sizes and tile sharding.
"""
import numpy as np
import pytest

from oracle import binding
from util import mirror, rel_rmse

pytestmark = pytest.mark.gpu


def _gpu(g19, abi, sc, cam, light, w, h, **kw):
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()
    out = rt.run(w, h, mode=abi.MODE_PATH, want=("rgb", "radiance"), **kw)
    return rt, out, rt.stats()


# Flat scenes trace the camera segment in the first bounce's launch and shade a path's last vertex in the launch before
# the last: the depths below run every form of that schedule -- the first launch alone (1), first launch folding the last
# vertex (2), one middle launch (3) -- also with mirror / glass, whose camera hits on those go to a queue. A wrong random
# number index or a dropped vertex in any of them is noise-level error at these sample counts, far above the bar.
# (which, depth, spp, (w, h, spp per pass) or None = 96 x 54 in one pass)
ORACLE_CASES = [("CORNELL", 5, 16, None), ("CORNELL_GLASS", 12, 16, None), ("CORNELL", 1, 16, None), ("CORNELL", 2, 16, None),
                ("CORNELL", 3, 16, None), ("CORNELL", 5, 6, (150, 97, 2)), ("CORNELL_GLASS", 1, 16, None),
                ("CORNELL_GLASS", 2, 16, None), ("CORNELL_GLASS", 8, 16, None)]


@pytest.mark.parametrize("which,depth,spp,shape", ORACLE_CASES,
                         ids=["%s-%d-%d" % c[:3] + ("-%dx%d-pass%d" % c[3] if c[3] else "") for c in ORACLE_CASES])
def test_same_seed_matches_oracle(g19, abi, oracle, which, depth, spp, shape):
    w, h, spp_pass = shape or (96, 54, 0)
    sc, cam, light = g19.Octree.builtin(getattr(abi, "SCENE_" + which), w=w, h=h)
    rt, got, st = _gpu(g19, abi, sc, cam, light, w, h, spp=spp, max_depth=depth, seed=7, spp_per_pass=spp_pass)
    exp, segs = binding.path_render(mirror(oracle, sc), cam, w, h, spp, depth, seed=7)
    if which == "CORNELL" and shape is None:
        # diffuse-only, one pass, no primary-hit AOV: no camera launch, one launch per bounce but the last
        assert st.class_launches[abi.K_EXTEND] == 0
        assert st.class_launches[abi.K_SHADE] == max(1, depth - 1)
    assert exp.mean() > 0.05
    err = rel_rmse(got["radiance"], exp)
    print("%s: same-seed relRMSE %.3e, segments gpu %d/%d cpu %d/%d" % (which, err, st.extend_segments,
                                                                         st.shadow_segments, segs[0], segs[1]))
    assert err <= 1e-2
    assert st.samples == w * h * spp
    assert abs(int(st.extend_segments) - segs[0]) <= 1e-3 * segs[0] + 2
    assert abs(int(st.shadow_segments) - segs[1]) <= 1e-3 * segs[1] + 2
    # RGB888 is the truncated clamp of the radiance (Image::setPixel)
    q = (255.0 * np.clip(got["radiance"], 0, 1)).astype(np.int32)
    assert np.abs(q - got["rgb"].astype(np.int32)).max() <= 1


def test_independent_seeds_statistical(g19, abi, oracle):
    w, h, spp, depth = 64, 36, 64, 5
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    rt, got, st = _gpu(g19, abi, sc, cam, light, w, h, spp=spp, max_depth=depth, seed=1)
    chk = mirror(oracle, sc)
    a, _ = binding.path_render(chk, cam, w, h, spp, depth, seed=2)
    b, _ = binding.path_render(chk, cam, w, h, spp, depth, seed=3)
    base = rel_rmse(a, b)
    err = rel_rmse(got["radiance"], b)
    print("independent seeds: gpu-vs-cpu %.3f, cpu-vs-cpu %.3f" % (err, base))
    assert err <= 1.5 * base


def test_heightfield_matches_oracle(g19, abi, oracle):
    w, h, spp, depth = 64, 36, 4, 4
    sc, cam, light = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD, n=24, w=w, h=h)
    rt, got, st = _gpu(g19, abi, sc, cam, light, w, h, spp=spp, max_depth=depth, seed=3)
    exp, segs = binding.path_render(mirror(oracle, sc), cam, w, h, spp, depth, seed=3)
    assert exp.mean() > 0.01
    err = rel_rmse(got["radiance"], exp)
    print("heightfield: same-seed relRMSE %.3e segments %d vs %d" % (err, st.extend_segments, segs[0]))
    assert err <= 1e-2
    assert abs(int(st.extend_segments) - segs[0]) <= 1e-3 * segs[0] + 2


def test_large_octree_agrees_with_small_leaves(g19, abi, oracle):
    """A deeper linear octree (n=96: 18 432 triangles) still finds the nearest hit: depth-1 image vs oracle."""
    w, h = 128, 72
    sc, cam, light = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD, n=96, w=w, h=h)
    rt, got, st = _gpu(g19, abi, sc, cam, light, w, h, spp=2, max_depth=2, seed=11)
    exp, segs = binding.path_render(mirror(oracle, sc), cam, w, h, 2, 2, seed=11)
    assert rel_rmse(got["radiance"], exp) <= 1e-2
    assert abs(int(st.extend_segments) - segs[0]) <= 1e-3 * segs[0] + 2


def test_deterministic_and_pass_invariant(g19, abi):
    w, h = 100, 70  # ragged tiles
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL_GLASS, w=w, h=h)
    rt, a, sa = _gpu(g19, abi, sc, cam, light, w, h, spp=12, max_depth=8, seed=5)
    b = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=12, max_depth=8, seed=5)
    assert a["radiance"].tobytes() == b["radiance"].tobytes()
    for spp_pass in (1, 5, 12):
        c = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=12, max_depth=8, seed=5, spp_per_pass=spp_pass)
        assert a["radiance"].tobytes() == c["radiance"].tobytes(), spp_pass
    # ... and of the pixel window a pass covers (whole 32x32 tiles of the rank's pixels)
    for ppp, spp_pass in ((1024, 0), (3000, 5), (4096, 1)):
        c = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=12, max_depth=8, seed=5, spp_per_pass=spp_pass,
                   pixels_per_pass=ppp)
        assert a["radiance"].tobytes() == c["radiance"].tobytes(), (ppp, spp_pass)
    d = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=12, max_depth=8, seed=6)
    assert a["radiance"].tobytes() != d["radiance"].tobytes()


def test_tile_sharding_bit_identical(g19, abi):
    w, h = 130, 75
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    rt, one, st1 = _gpu(g19, abi, sc, cam, light, w, h, spp=8, max_depth=5, seed=9)
    out = {"radiance": np.zeros((h, w, 3), np.float32), "rgb": np.zeros((h, w, 3), np.uint8)}
    total = 0
    for rank in range(4):
        rt.run(w, h, mode=abi.MODE_PATH, want=("rgb", "radiance"), out=out, spp=8, max_depth=5, seed=9, rank=rank,
               world=4)
        total += rt.stats().samples
    assert total == st1.samples == w * h * 8
    assert out["radiance"].tobytes() == one["radiance"].tobytes()
    assert np.array_equal(out["rgb"], one["rgb"])


def test_edge_cases(g19, abi):
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=64, h=64)
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()
    # depth 1: only directly visible emitters contribute
    d1 = rt.run(64, 64, mode=abi.MODE_PATH, want=("radiance",), spp=4, max_depth=1)["radiance"]
    assert ((d1 == 0) | (d1 == 17.0)).all() or np.isclose(d1[d1 > 0].max(), 17.0)
    with pytest.raises(g19.G19Error):
        rt.run(64, 64, mode=abi.MODE_PATH, spp=0, max_depth=5)
    with pytest.raises(g19.G19Error):
        rt.run(64, 64, mode=abi.MODE_PATH, spp=1, max_depth=-1)
    with pytest.raises(g19.G19Error):
        rt.run(64, 64, mode=abi.MODE_PATH, spp=1, max_depth=65)
    # max_depth 0 is the depth-0 slice (the reference's shade of the primary hit, tests/test_path_link.py): no bounce
    d0 = rt.run(64, 64, mode=abi.MODE_PATH, want=("rgb", "ids"), spp=1, max_depth=0)
    assert (d0["ids"] >= 0).mean() > 0.9 and d0["rgb"].max() > 0
    # empty scene: black
    empty = g19.Octree((-1,) * 3, (1,) * 3)
    rt.setScene(empty)
    z = rt.run(40, 24, mode=abi.MODE_PATH, want=("radiance",), spp=2, max_depth=3)["radiance"]
    assert (z == 0).all()


def test_cancel_between_passes(g19, abi):
    import threading
    w, h = 256, 256
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()
    t = threading.Timer(0.05, rt.stop)  # the GUI thread calling stop() (viewer.h:29-34)
    t.start()
    rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=4096, max_depth=5, spp_per_pass=1)
    t.join()
    assert rt.stats().samples < w * h * 4096
    assert 0.0 <= rt.progress() <= 1.0


def test_zoo_every_entity_kind(g19, abi, oracle):
    """PATH mode over one entity of every reference class (analytic spheres, single triangles, the
    rectangle/box pairs with the reference's p4 = -p3 geometry, tessellated sphere/quad/cube/cone),
    one of them emitting: primitive extraction and the octree must agree with the brute-force oracle."""
    from util import zoo
    sc = zoo(g19)
    sc.push_back(g19.ImpTriangle((-6, -9, 9), (-6, 9, 9), (6, 0, 9), (1, 1, 1), bsdf=abi.BSDF_EMITTER,
                                 emission=(6.0, 6.0, 6.0)))
    sc.push_back(g19.ExpQuad((2, 0, -3), 6, 8, 0.2, (0.8, 0.8, 0.8)))
    cam = g19.Camera((-10, 0, 0), (1, 0, 0), 0.1)
    w, h = 120, 120
    rt, got, st = _gpu(g19, abi, sc, cam, (0, 0, 0), w, h, spp=8, max_depth=4, seed=21)
    exp, segs = binding.path_render(mirror(oracle, sc), cam, w, h, 8, 4, seed=21)
    assert exp.mean() > 0.01
    err = rel_rmse(got["radiance"], exp)
    print("zoo: same-seed relRMSE %.3e, segments gpu %d/%d cpu %d/%d" % (err, st.extend_segments, st.shadow_segments,
                                                                          segs[0], segs[1]))
    assert err <= 1e-2
    assert abs(int(st.extend_segments) - segs[0]) <= 1e-3 * segs[0] + 2
    assert abs(int(st.shadow_segments) - segs[1]) <= 1e-3 * segs[1] + 2


def test_progressive_refreshes_and_cancel(g19, abi):
    """g19_render_progressive: the viewer's repaint hook (raytracer.h:31, viewer.h:18-21). Refreshes carry
    growing fractions and ever more converged images; the result equals the plain render; returning
    non-zero from the hook cancels within one pass."""
    w, h = 160, 96
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()
    plain = rt.run(w, h, mode=abi.MODE_PATH, want=("rgb", "radiance"), spp=24, max_depth=4, seed=2, spp_per_pass=2)
    seen = []

    def on_pass(fraction, rgb):
        seen.append((fraction, rgb.copy()))
        return False
    out = rt.run_progressive(w, h, on_pass, min_interval_ms=0, want_radiance=True, spp=24, max_depth=4, seed=2, spp_per_pass=2)
    fr = [f for f, _ in seen]
    assert len(seen) == 12 and fr == sorted(fr) and fr[-1] == 1.0 and abs(fr[0] - 2 / 24) < 1e-9
    assert np.array_equal(out["rgb"], plain["rgb"]) and out["radiance"].tobytes() == plain["radiance"].tobytes()
    assert np.array_equal(seen[-1][1], plain["rgb"])
    err = [np.abs(img.astype(int) - plain["rgb"].astype(int)).mean() for _, img in seen]
    assert err[0] > err[5] > err[-1] == 0
    # a long interval: only the final refresh
    seen.clear()
    rt.run_progressive(w, h, on_pass, min_interval_ms=60000, spp=8, max_depth=3, spp_per_pass=2)
    assert [f for f, _ in seen] == [1.0]
    # cancel from the hook after the second refresh
    seen.clear()

    def stop_after_two(fraction, rgb):
        seen.append(fraction)
        return len(seen) == 2
    rt.run_progressive(w, h, stop_after_two, min_interval_ms=0, spp=64, max_depth=4, spp_per_pass=2)
    assert len(seen) == 3 and seen[1] == 4 / 64 and seen[2] < 0.2  # two refreshes + the closing call
    assert rt.stats().samples < w * h * 64
    # REF mode: one pass, one call
    seen.clear()
    sc1, cam1, light1 = g19.Octree.builtin(abi.SCENE_DEFAULT)
    rt1 = g19.RayTracer(cam1, light1)
    rt1.setScene(sc1)
    rt1.start()
    r = rt1.run_progressive(200, 200, lambda f, rgb: seen.append(f) or False, mode=abi.MODE_REF)
    assert seen == [1.0] and np.array_equal(r["rgb"], rt1.run(200, 200)["rgb"])


@pytest.mark.parametrize("n_quads,n_tris,n_spheres", [(1, 0, 0), (0, 1, 1), (1, 1, 1), (2, 3, 2), (3, 2, 3), (0, 0, 2)])
def test_flat_scene_pair_padding(g19, abi, oracle, n_quads, n_tris, n_spheres):
    """Flat scenes run their primitives two at a time through the packed-FP32 loops; each kind group
    (parallelograms | triangles | spheres) is padded to an even count with a NaN record. Odd and even
    group sizes, empty groups and every BSDF class must agree with the brute-force oracle."""
    sc = g19.Octree((-20,) * 3, (20,) * 3)
    # the emitter: one triangle overhead (always present; counts as a triangle of the scene)
    sc.push_back(g19.ImpTriangle((-4, -6, 7), (-4, 6, 7), (8, 0, 7), (1, 1, 1), bsdf=abi.BSDF_EMITTER, emission=(9.0, 8.0, 7.0)))
    quads = [((6, -8, -8), (6, 8, -8), (6, 8, 8), (6, -8, 8)),      # back wall
             ((-8, -8, -1.5), (6, -8, -1.5), (6, 8, -1.5), (-8, 8, -1.5)),  # floor
             ((-8, 7, -8), (6, 7, -8), (6, 7, 8), (-8, 7, 8))]      # side wall
    for a, b, c, d in quads[:n_quads]:  # two coplanar triangles each: the builder merges them into one parallelogram
        sc.push_back(g19.ImpTriangle(a, b, c, (0.7, 0.6, 0.5)))
        sc.push_back(g19.ImpTriangle(a, c, d, (0.7, 0.6, 0.5)))
    tris = [((2, -3, -1), (2, 3, -1), (2, 0, 4)), ((3, -6, 0), (4, -2, -1), (3, -4, 4)), ((1, 2, -1), (3, 5, 0), (2, 3, 4))]
    for k, (a, b, c) in enumerate(tris[:n_tris]):
        sc.push_back(g19.ImpTriangle(a, b, c, (0.2 + 0.3 * k, 0.8, 0.4)))
    spheres = [((2, 2, 1), 1.5, abi.BSDF_DIFFUSE), ((1, -3, 2), 1.2, abi.BSDF_MIRROR), ((-1, 0, 0.5), 1.0, abi.BSDF_GLASS)]
    for pos, r, bsdf in spheres[:n_spheres]:
        sc.push_back(g19.ImpSphere(pos, r, (0.9, 0.9, 0.9), bsdf=bsdf))
    cam = g19.Camera((-10, 0, 0), (1, 0, 0), 0.02)
    w, h, spp, depth = 96, 64, 8, 6
    rt, got, st = _gpu(g19, abi, sc, cam, (0, 0, 0), w, h, spp=spp, max_depth=depth, seed=5)
    exp, segs = binding.path_render(mirror(oracle, sc), cam, w, h, spp, depth, seed=5)
    assert exp.mean() > 0.005
    err = rel_rmse(got["radiance"], exp)
    print("pairs (%d,%d,%d): same-seed relRMSE %.3e, segments gpu %d/%d cpu %d/%d" % (
        n_quads, n_tris, n_spheres, err, st.extend_segments, st.shadow_segments, segs[0], segs[1]))
    assert err <= 1e-2
    assert abs(int(st.extend_segments) - segs[0]) <= 1e-3 * segs[0] + 2
    assert abs(int(st.shadow_segments) - segs[1]) <= 1e-3 * segs[1] + 2


@pytest.mark.parametrize("which,depth", [("CORNELL", 5), ("CORNELL_GLASS", 9)])
def test_passes_in_flight_bit_identical(g19, abi, which, depth):
    """Up to four passes run concurrently on their own streams (PathWork lanes). That may not change a bit: the
    accumulation stays in pass order (events) and every vertex is shaded by the same code."""
    w, h, spp = 160, 96, 24
    sc, cam, light = g19.Octree.builtin(getattr(abi, "SCENE_" + which), w=w, h=h)
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()

    def render():
        return rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=spp, max_depth=depth, seed=11, spp_per_pass=2)["radiance"]

    base = render()  # default: four lanes
    assert base.mean() > 0.05
    for lanes in ("1", "2", "3"):
        rt.tune("lanes", lanes)
        assert render().tobytes() == base.tobytes(), "lanes=" + lanes


def test_flat_then_tree_scene_on_one_context(g19, abi):
    """Flat scenes store every slot's radiance (accumulate only reads it); tree scenes add to zeroed planes
    that accumulate clears. One context switching between the two must not carry anything over."""
    w, h = 128, 96
    kw = dict(mode=abi.MODE_PATH, want=("radiance",), spp=6, max_depth=4, seed=3, spp_per_pass=2)
    scenes = [g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h), g19.Octree.builtin(abi.SCENE_HEIGHTFIELD, n=48, w=w, h=h)]
    want = []
    for sc, cam, light in scenes:  # each scene on a context of its own
        rt = g19.RayTracer(cam, light)
        rt.setScene(sc)
        rt.start()
        want.append(rt.run(w, h, **kw)["radiance"])
        assert want[-1].mean() > 0.01
    rt = g19.RayTracer(scenes[0][1], scenes[0][2])
    rt.start()
    for k in (0, 1, 0, 1, 1):
        sc, cam, light = scenes[k]
        rt.camera, rt.light = cam, tuple(light)
        rt.setScene(sc)
        assert rt.run(w, h, **kw)["radiance"].tobytes() == want[k].tobytes(), k


@pytest.mark.parametrize("which,n,w,h,spp,depth", [("HEIGHTFIELD", 24, 64, 36, 4, 4), ("HEIGHTFIELD_ROOM", 40, 96, 54, 4, 5),
                                                    ("HEIGHTFIELD_ROOM", 150, 160, 90, 2, 4), ("ZOO", 0, 120, 120, 8, 4)])
def test_bvh_walk_matches_oracle_and_octree(g19, abi, oracle, which, n, w, h, spp, depth):
    """tune walk=3 / 4: the bounding-volume hierarchy (csrc/bvh_build.cu; BvhWalk binary, Bvh4Walk 4-wide) instead of the linear octree. Same
    nearest hits, so the same radiance as the brute-force oracle and as the octree walk (they may part ways only where
    two primitives tie in t along a shared edge), same segment counts. n = 150 builds both trees on the device."""
    if which == "ZOO":
        from util import zoo
        sc = zoo(g19)
        sc.push_back(g19.ImpTriangle((-6, -9, 9), (-6, 9, 9), (6, 0, 9), (1, 1, 1), bsdf=abi.BSDF_EMITTER, emission=(6.0, 6.0, 6.0)))
        sc.push_back(g19.ExpQuad((2, 0, -3), 6, 8, 0.2, (0.8, 0.8, 0.8)))
        cam, light = g19.Camera((-10, 0, 0), (1, 0, 0), 0.1), (0, 0, 0)
    else:
        sc, cam, light = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=n, w=w, h=h)
    outs = {}
    for walk in (1, 3, 4):
        rt = g19.RayTracer(cam, light)
        rt.tune("walk", walk)
        rt.setScene(sc)
        rt.start()
        rad = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=spp, max_depth=depth, seed=17)["radiance"]
        st = rt.stats()
        outs[walk] = (rad, int(st.extend_segments), int(st.shadow_segments))
        again = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=spp, max_depth=depth, seed=17)["radiance"]
        assert rad.tobytes() == again.tobytes()
    exp, segs = binding.path_render(mirror(oracle, sc), cam, w, h, spp, depth, seed=17)
    assert exp.mean() > 0.005
    for walk, (rad, ext, shd) in outs.items():
        err = rel_rmse(rad, exp)
        print("%s walk=%d: same-seed relRMSE %.3e, segments %d/%d vs oracle %d/%d" % (which, walk, err, ext, shd, segs[0], segs[1]))
        assert err <= 1e-2
        assert abs(ext - segs[0]) <= 1e-3 * segs[0] + 2
        assert abs(shd - segs[1]) <= 1e-3 * segs[1] + 2
    assert rel_rmse(outs[3][0], outs[1][0]) <= 2e-3
    assert rel_rmse(outs[4][0], outs[1][0]) <= 2e-3


def test_bvh_deep_stack_on_a_pile_of_overlapping_triangles(g19, abi, oracle):
    """Worst case for the postponed-children stack of the BVH walks: 1500 small triangles piled on one spot (every box
    overlaps every other, equal Morton codes split by position only, so the hierarchy is deep and a ray through the pile
    is inside every box) next to a regular floor. Twelve stack levels live in shared memory, the rest in local memory:
    no child may be dropped -- the nearest hits, hence radiance and segment counts, must equal the oracle's and the
    octree walk's."""
    rng = np.random.default_rng(5)
    sc = g19.Octree((-20,) * 3, (20,) * 3)
    for k in range(1500):
        c = np.array([2.0, 0.0, 0.0]) + rng.uniform(-0.02, 0.02, 3)
        a, b, d = (c + rng.uniform(-0.3, 0.3, 3) for _ in range(3))
        sc.push_back(g19.ImpTriangle(tuple(a), tuple(b), tuple(d), tuple(rng.uniform(0.3, 0.9, 3))))
    for i in range(-8, 8):
        for j in range(-8, 8):
            p = [(i, j, -2.0), (i + 1, j, -2.0), (i + 1, j + 1, -2.0), (i, j + 1, -2.0)]
            sc.push_back(g19.ImpTriangle(p[0], p[1], p[2], (0.7, 0.7, 0.7)))
            sc.push_back(g19.ImpTriangle(p[0], p[2], p[3], (0.7, 0.7, 0.7)))
    sc.push_back(g19.ImpTriangle((-6, -9, 9), (-6, 9, 9), (6, 0, 9), (1, 1, 1), bsdf=abi.BSDF_EMITTER, emission=(8.0, 8.0, 8.0)))
    cam = g19.Camera((-10, 0, 0), (1, 0, 0), 0.1)
    w, h, spp, depth = 96, 96, 2, 3
    outs = {}
    for walk, stack in ((1, 12), (3, 4), (4, 4), (4, 12)):
        rt = g19.RayTracer(cam, (0, 0, 0))
        rt.tune("walk", walk)
        rt.tune("bvh_stack", stack)
        rt.setScene(sc)
        rt.start()
        rad = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=spp, max_depth=depth, seed=2)["radiance"]
        st = rt.stats()
        outs[(walk, stack)] = (rad, int(st.extend_segments), int(st.shadow_segments))
    exp, segs = binding.path_render(mirror(oracle, sc), cam, w, h, spp, depth, seed=2)
    assert exp.mean() > 0.005
    for key, (rad, ext, shd) in outs.items():
        err = rel_rmse(rad, exp)
        print("pile walk/stack %s: relRMSE %.3e segments %d/%d vs %d/%d" % (key, err, ext, shd, segs[0], segs[1]))
        assert err <= 1e-2
        assert abs(ext - segs[0]) <= 1e-3 * segs[0] + 2 and abs(shd - segs[1]) <= 1e-3 * segs[1] + 2


@pytest.mark.parametrize("which,n,depth", [("CORNELL", 0, 5), ("CORNELL_GLASS", 0, 8), ("HEIGHTFIELD_ROOM", 40, 4)])
def test_frames_in_a_row_overlap_and_stay_bit_identical(g19, abi, which, n, depth):
    """Frames enqueued back to back on one stream (tune overlap_frames, default on): the side lanes start frame k + 1's
    passes behind their own passes of frame k instead of behind frame k's join and resolve. Every frame must still be
    what a lone, synchronous render of the same seed produces, bit for bit -- statistics included."""
    import torch
    w, h, spp = 320, 200, 12
    sc, cam, light = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=n, w=w, h=h)
    seeds = [3, 4, 3, 5, 4, 3, 6, 6]
    stream = torch.cuda.current_stream().cuda_stream
    for overlap in (1, 0):
        rt = g19.RayTracer(cam, light)
        rt.tune("overlap_frames", overlap)
        rt.setScene(sc)
        rt.start()
        alone = {}
        for sd in sorted(set(seeds)):
            alone[sd] = rt.run(w, h, mode=abi.MODE_PATH, want=("radiance",), spp=spp, max_depth=depth, seed=sd, spp_per_pass=2)["radiance"]
            alone[sd] = (alone[sd], int(rt.stats().extend_segments))
        bufs = [torch.zeros(h * w * 3, dtype=torch.float32, device="cuda") for _ in seeds]
        for sd, buf in zip(seeds, bufs):  # nothing synchronises between these
            rt.run_device(rt.params(w, h, mode=abi.MODE_PATH, spp=spp, max_depth=depth, seed=sd, spp_per_pass=2), d_rad=buf.data_ptr(), stream=stream)
        torch.cuda.synchronize()
        assert int(rt.stats().extend_segments) == alone[seeds[-1]][1]  # the statistics are the last frame's
        for sd, buf in zip(seeds, bufs):
            got = buf.cpu().numpy().reshape(h, w, 3)
            assert got.tobytes() == alone[sd][0].tobytes(), (overlap, sd)

"""Pins the CPU oracle (oracle/ref_restate.c) to the reference.

Three anchors, strongest first:
  1. the compiled, unmodified reference (oracle/_ref/libg19ref.so) when it is present --
     byte equality on everything the reference's public API exposes;
  2. tests/golden/ref_golden.npz -- outputs of that same compiled reference, committed
     (generator: tests/golden/make_golden.py), so the pin survives without the reference sources;
     tests/golden/ref_live.npz (generator: tests/golden/make_golden_live.py) holds what the comparisons
     with oracle/_ref below compare with, so they run where it is not built;
  3. the vectors SURVEY.md section 4 derived from the reference's own dead test functions
     (main.cpp:90-133) and the config-1 sha256 / hit histogram.
"""
import hashlib
import os

import numpy as np
import pytest

from util import (assert_same, live_frame_scenes, live_frames, live_golden, live_material, live_zoo, material_descs, mirror,
                  probe_rays, reference_checker, zoo)

C1_SHA = "9ab0129419a4c328d4ea865adf74b66e3c91d10c6190cc34373fa2b0187bba85"
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_golden.npz"))
LIVE = live_golden()


def test_config1_sha256_and_histogram(g19, abi, oracle):
    sc, cam, light = g19.Octree.builtin(abi.SCENE_DEFAULT)
    chk = mirror(oracle, sc)
    rgb = chk.render(cam, light, 500, 500)
    assert hashlib.sha256(rgb.tobytes()).hexdigest() == C1_SHA
    assert bytes(GOLD["c1_sha256"]).hex() == C1_SHA
    t = chk.trace(cam, light, 500, 500, want=("ids", "rgb"), threads=8)
    assert np.array_equal(t["rgb"], rgb)  # the id-exposing loop shades the same bytes as run()
    hist = np.bincount(t["ids"].ravel() + 1, minlength=4)
    assert hist.tolist() == [196818, 14702, 20806, 17674] == GOLD["c1_hist"].tolist()


def test_entity_test_vector(g19, oracle):
    """main.cpp:90-104: ImpSphere({2,0,0}, r=10), Ray({-10,0,0},{1,.5,.5})."""
    sc = g19.Octree((-20,) * 3, (20,) * 3)
    sc.push_back(g19.ImpSphere((2, 0, 0), 10, (0, 1, 0)))
    h, p, n = mirror(oracle, sc).intersect(0, [[-10, 0, 0]], [[1, .5, .5]])
    assert h[0] == 1
    assert np.allclose(p[0], (-7.887841, 1.056080, 1.056080), atol=5e-7)
    assert np.allclose(n[0], (-0.988784, 0.105608, 0.105608), atol=5e-7)
    assert p.tobytes() == GOLD["kat_entity_pt"].tobytes() and n.tobytes() == GOLD["kat_entity_nrm"].tobytes()


def test_bbox_test_vector(g19, oracle):
    """main.cpp:125-133 bbox_test(): b1=[0,2]^3 and b2=[-2,1]x[-2,1]x[0,2] overlap -> an entity with
    bbox b2 is accepted by an Octree whose root is b1; one that only touches (strict <) is rejected."""
    sc = g19.Octree((0, 0, 0), (2, 2, 2))
    _, ok = sc.push_back(g19.ExpBox((-2, -2, 0), (1, 1, 2)))
    assert ok
    _, ok = sc.push_back(g19.ExpBox((2, 0, 0), (3, 2, 2)))  # shares only the face x=2
    assert not ok
    chk = mirror(oracle, sc)
    assert len(chk.candidates((-5, .5, .5), (1, 0, 0))) == 1  # the rejected box is not in the tree


@pytest.mark.parametrize("idx", range(9))
def test_zoo_probes_against_golden(g19, oracle, idx):
    z = zoo(g19)
    chk = mirror(oracle, z)
    o, d = probe_rays(20000, seed=idx)
    h, p, n = chk.intersect(idx, o, d)
    m = h.astype(bool)
    assert np.array_equal(np.packbits(m), GOLD["zoo_%d_hit" % idx])
    assert hashlib.sha256(p[m].tobytes() + n[m].tobytes()).digest() == bytes(GOLD["zoo_%d_ptsha" % idx])
    assert np.array_equal(chk.texcoord(idx, p[m][:512]), GOLD["zoo_%d_uv" % idx])
    assert chk.bbox(idx).tobytes() == GOLD["zoo_%d_bbox" % idx].tobytes()
    assert chk.triangles(idx).tobytes() == GOLD["zoo_%d_tris" % idx].tobytes()


def test_frames_against_golden(g19, abi, oracle):
    z = zoo(g19)
    chk = mirror(oracle, z)
    t = chk.trace(g19.Camera((-10, 0, 0), (1, 0, 0), 0.1), (-10, 10, 10), 200, 200, threads=8)
    assert np.array_equal(t["ids"], GOLD["zoo_ids"])
    assert hashlib.sha256(t["points"].tobytes()).digest() == bytes(GOLD["zoo_ptsha"])
    ok = t["ids"] != 4  # ExpSphere's negative texture rows read outside the pattern (undefined)
    assert np.array_equal(t["rgb"][ok], GOLD["zoo_rgb"][ok])
    rng = np.random.default_rng(5)
    flat = []
    for _ in range(64):
        o, d = rng.uniform(-15, 15, 3), rng.uniform(-1, 1, 3)
        c = chk.candidates(o, d)
        flat.append(np.concatenate([[len(c)], c]))
    assert np.array_equal(np.concatenate(flat), GOLD["cand_flat"])
    w, h = 96, 54
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    t = mirror(oracle, sc).trace(cam, light, w, h, want=("ids", "rgb"), threads=8)
    assert np.array_equal(t["ids"], GOLD["cornell_ids"]) and np.array_equal(t["rgb"], GOLD["cornell_rgb"])
    assert len(np.unique(t["ids"])) >= 12
    sc, cam, light = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD, n=32, w=w, h=h)
    t = mirror(oracle, sc).trace(cam, light, w, h, want=("ids",), threads=8)
    assert np.array_equal(t["ids"], GOLD["height_ids"])


# ---- against the reference: tests/golden/ref_live.npz always, oracle/_ref live where it is built -----------
def test_live_reference_zoo(g19, oracle):
    z = zoo(g19)
    got = live_zoo(oracle, z)
    assert_same(got, {k: LIVE[k] for k in got})
    b = mirror(oracle, z)
    for i in range(len(z)):
        assert b.bbox(i).tobytes() == GOLD["zoo_%d_bbox" % i].tobytes()
        assert b.triangles(i).tobytes() == GOLD["zoo_%d_tris" % i].tobytes()
    ref = reference_checker()
    if ref is not None:
        assert_same(live_zoo(ref, z), got)
        a = mirror(ref, z)
        for i in range(len(z)):
            assert a.bbox(i).tobytes() == b.bbox(i).tobytes()
            assert a.triangles(i).tobytes() == b.triangles(i).tobytes()


def test_live_reference_frames(g19, abi, oracle):
    got = live_frames(oracle, g19, abi)
    assert_same(got, {k: LIVE[k] for k in got})
    for which, _, _ in live_frame_scenes(abi):
        assert np.array_equal(got["frame_%d_run" % which], got["frame_%d_rgb" % which])  # run() itself
    ref = reference_checker()
    if ref is not None:
        assert_same(live_frames(ref, g19, abi), got)


def test_live_reference_material_fields(g19, oracle):
    """Material's public fields beyond `color` (reference include/material.h:24-29: diffuse_color, specular_color,
    shader_parameters, specular_power) travel in g19_entity_desc: a caller who assigns them after construction gets
    the reference's own blinn_phong_texture result (material.h:48-62), byte for byte, from the restatement -- and a
    frame shaded with them equals the reference's."""
    descs = material_descs(g19)
    assert descs[0].material_set == 1 and descs[2].material_set == 0
    got = live_material(oracle, g19)
    assert_same(got, {k: LIVE[k] for k in got})
    ref = reference_checker()
    if ref is not None:
        assert_same(live_material(ref, g19), got)
    assert (got["material_ids"] >= 0).sum() > 500
    # the custom fields do change the picture
    cam = g19.Camera((-10, 0, 0), (1, 0, 0), 0.02)
    plain = oracle.scene((-20,) * 3, (20,) * 3, [g19.ImpSphere((3, 1, 0), 2.0, (1, 0, 2)), g19.ImpTriangle((4, -5, -3), (4, 5, -3), (4, 0, 4), (0, 1, 1)),
                                                 descs[2]]).trace(cam, (-8, 6, 9), 96, 96, want=("rgb",), threads=2)
    assert not np.array_equal(plain["rgb"], got["material_rgb"])

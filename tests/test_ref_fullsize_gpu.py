"""G19_MODE_REF at the sizes BASELINE.json states: 1920x1080 on the Cornell box and on the 1 002 528-triangle
heightfield (reference octree ~1.5 M nodes), against ids produced by the UNMODIFIED reference
(oracle/_ref/libg19ref.so -> tests/golden/ref_1080p.npz, generator tests/golden/make_golden_1080p.py).

The north-star's "primary-hit entity IDs must match bit-exactly" is a statement about RayTracer::run's own loop
(reference include/raytracer.h:41-74); round 1 checked it on 480x270 and n = 48 only (VERDICT r01 weak 4).
"""
import os

import numpy as np
import pytest

from util import quiet_stdout

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "ref_1080p.npz")
W, H, N = 1920, 1080, 708


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _rt(g19, sc, cam, light):
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()
    return rt


def test_cornell_1080p_ids_bit_exact_vs_compiled_reference(g19, abi, oracle, gold):
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=W, h=H)
    got = _rt(g19, sc, cam, light).run(W, H, want=("ids", "rgb"))
    exp_ids = gold["cornell_ids"].astype(np.int32)
    assert np.array_equal(got["ids"], exp_ids), "%d of %d ids differ" % (int((got["ids"] != exp_ids).sum()), W * H)
    assert (exp_ids >= 0).mean() > 0.99
    # colours: the restatement (byte-equal to the compiled reference, test_oracle_ref.py) on the whole frame
    from util import mirror
    exp = mirror(oracle, sc).trace(cam, light, W, H, want=("rgb",), threads=os.cpu_count() or 8)["rgb"]
    import hashlib
    assert hashlib.sha256(exp.tobytes()).digest() == bytes(gold["cornell_rgb_sha"])  # the restatement is pinned at this size too
    d = np.abs(got["rgb"].astype(np.int32) - exp.astype(np.int32)).max(2)
    assert (d > 1).sum() <= 0.001 * W * H, "%d pixels off by more than 1 LSB" % int((d > 1).sum())


@pytest.mark.parametrize("which,rows_key,ids_key,drop", [("HEIGHTFIELD", "height_rows", "height_ids", 2),
                                                          ("HEIGHTFIELD_ROOM", "room_rows", "room_ids", 0)])
def test_heightfield_1m_triangles_1080p_ids_bit_exact_vs_compiled_reference(g19, abi, gold, which, rows_key, ids_key, drop):
    full, cam, light = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=N, w=W, h=H)
    if drop:  # the bare surface: without the light panel behind the camera (tests/test_path_link.py explains why)
        sc = g19.Octree(full.min, full.max)
        ents = full.entities()
        for d in ents[:-drop]:
            sc.push_back(d)
    else:
        sc = full
    assert len(sc) >= 2 * N * N
    got = _rt(g19, sc, cam, light).run(W, H, want=("ids",))["ids"]
    rows, exp = gold[rows_key], gold[ids_key]
    assert exp.shape == (rows.size, W)
    sub = got[rows]
    assert np.array_equal(sub, exp), "%d of %d ids differ" % (int((sub != exp).sum()), exp.size)
    assert (exp >= 0).sum() > 1000  # the bands do see the surface


def test_live_reference_band_on_this_box(g19, abi, gold):
    """A band of the 1080p Cornell frame and a small heightfield room on the GPU against the reference directly (not
    through the restatement): ids from ref_1080p.npz, colours and the room's ids from ref_live.npz, and the compiled
    reference run live on this machine where oracle/_ref is built."""
    from util import live_golden, mirror, reference_checker
    live = live_golden()
    reflib = reference_checker()
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=W, h=H)
    got = _rt(g19, sc, cam, light).run(W, H, want=("ids", "rgb"))
    y0, y1 = (int(v) for v in live["band_rows"])
    refs = [{"ids": gold["cornell_ids"][y0:y1].astype(np.int32), "rgb": live["band_cornell_rgb"]}]
    if reflib is not None:
        with quiet_stdout():
            t = mirror(reflib, sc).trace(cam, light, W, H, y0=y0, y1=y1, want=("ids", "rgb"), threads=os.cpu_count() or 8)
        refs.append({"ids": t["ids"][y0:y1], "rgb": t["rgb"][y0:y1]})
    for ref in refs:
        assert np.array_equal(got["ids"][y0:y1], ref["ids"])
        d = np.abs(got["rgb"][y0:y1].astype(np.int32) - ref["rgb"].astype(np.int32)).max(2)
        assert (d > 1).sum() <= 0.001 * d.size
    w, h = 320, 180
    sc, cam, light = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD_ROOM, n=96, w=w, h=h)
    got = _rt(g19, sc, cam, light).run(w, h, want=("ids",))
    assert np.array_equal(got["ids"], live["room96_ids"].astype(np.int32))
    if reflib is not None:
        with quiet_stdout():
            ref = mirror(reflib, sc).trace(cam, light, w, h, want=("ids",), threads=os.cpu_count() or 8)
        assert np.array_equal(got["ids"], ref["ids"])

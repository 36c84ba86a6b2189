"""Batched nearest-hit and occlusion ray queries (g19_cast_rays) on the GPU, against the FP64 PATH oracle."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from cast_util import as_cast, bounce_rays, box_rays, corner_rays, path_cast, robust_mask, unit
from test_path_link import _interior
from util import mirror, zoo

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W, H = 480, 270
FLAT = [("DEFAULT", 0), ("CORNELL", 0), ("CORNELL_GLASS", 0)]
TREE = [("HEIGHTFIELD", 48), ("HEIGHTFIELD_ROOM", 64)]
WALKS = (1, 3, 4)


def _scene(g19, abi, which, n, walk=None):
    """(RayTracer with the scene uploaded under `walk`, scene, oracle scene, camera)."""
    from oracle import binding
    if which == "ZOO":
        sc = zoo(g19)
        sc.set_shapes(True)
        cam = g19.Camera((-15.0, 2.0, 3.0), (0.0, 0.0, 0.0), 0.04)
    else:
        sc, cam, _ = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=n, w=W, h=H)
    rt = g19.RayTracer(cam, (0.0, 0.0, 10.0))
    if walk is not None:
        rt.tune("walk", walk)
    rt.setScene(sc)
    rt.start()
    chk = mirror(binding.CheckerLib("oracle"), sc)
    if which == "ZOO":
        chk.lib.lib.g19o_scene_set_shapes(chk.h, abi.SHAPES_FIXED)
    return rt, sc, chk, cam


def _ray_sets(chk, cam, lo, hi):
    """corner rays, bounce rays off their hits, random rays inside the scene box. The bounce rays leave robust hits only:
    a hit on an edge would put the origin on the adjacent surface, where t = 0 hits are allowed (g19.h) and the oracle's
    t > 0 rule disagrees by design."""
    o, d = as_cast(*corner_rays(cam, W, H))
    ok, ids, t, nrm = robust_mask(chk, o, d)
    hit = ok & (ids >= 0)
    bo, bd = bounce_rays(o[hit] + unit(d[hit]) * t[hit, None], nrm[hit], 4096, seed=1)
    return {"corner": (o, d), "bounce": as_cast(bo, bd), "box": as_cast(*box_rays(lo, hi, 4096, seed=2))}


def _check_vs_oracle(got, ok, ids, t, nrm, what):
    assert ok.mean() >= 0.98, "%s: only %.1f %% of the rays are robust" % (what, 100 * ok.mean())
    assert np.array_equal(got["ids"][ok], ids[ok]), "%s: %d robust rays differ" % (what, int((got["ids"][ok] != ids[ok]).sum()))
    hit = ok & (ids >= 0)
    tg = got["t"].astype(np.float64)
    assert (np.abs(tg[hit] - t[hit]) <= 1e-4 * np.maximum(1.0, t[hit])).all(), what
    assert ((got["normals"][hit].astype(np.float64) * nrm[hit]).sum(1) >= 0.9999).all(), what
    miss = ok & (ids < 0)
    assert np.isposinf(got["t"][miss]).all() and (got["normals"][miss] == 0).all(), what


def _bounds(sc):
    return np.array(sc.min, float) * 0.5, np.array(sc.max, float) * 0.5


@pytest.mark.parametrize("which,n", FLAT + [("ZOO", 0)])
def test_cast_flat_and_zoo_match_oracle(g19, abi, which, n):
    rt, sc, chk, cam = _scene(g19, abi, which, n)
    lo, hi = _bounds(sc)
    for name, (o, d) in _ray_sets(chk, cam, lo, hi).items():
        ok, ids, t, nrm = robust_mask(chk, o, d)
        got = rt.cast(o, d, want_normals=True)
        _check_vs_oracle(got, ok, ids, t, nrm, "%s/%s" % (which, name))
        # any hit agrees with nearest: robust hits are free below t/2 and blocked below 1.5 t; misses stay misses
        hit = ok & (got["ids"] >= 0)
        tg = got["t"].astype(np.float64)
        assert (rt.cast(o[hit], d[hit], tmax=0.5 * tg[hit], any_hit=True)["ids"] == -1).all()
        assert (rt.cast(o[hit], d[hit], tmax=1.5 * tg[hit], any_hit=True)["ids"] >= 0).all()
        assert (rt.cast(o[got["ids"] < 0], d[got["ids"] < 0], any_hit=True)["ids"] == -1).all()


@pytest.mark.parametrize("which,n", TREE)
def test_cast_tree_walks_match_oracle_and_each_other(g19, abi, which, n):
    per_walk = {}
    sets = None
    for walk in WALKS:
        rt, sc, chk, cam = _scene(g19, abi, which, n, walk=walk)
        if sets is None:
            sets = _ray_sets(chk, cam, *_bounds(sc))
            oracle_res = {k: robust_mask(chk, o, d) for k, (o, d) in sets.items()}
        for name, (o, d) in sets.items():
            ok, ids, t, nrm = oracle_res[name]
            got = rt.cast(o, d, want_normals=True)
            _check_vs_oracle(got, ok, ids, t, nrm, "%s/%s/walk %d" % (which, name, walk))
            hit = ok & (got["ids"] >= 0)
            tg = got["t"].astype(np.float64)
            assert (rt.cast(o[hit], d[hit], tmax=0.5 * tg[hit], any_hit=True)["ids"] == -1).all()
            assert (rt.cast(o[hit], d[hit], tmax=1.5 * tg[hit], any_hit=True)["ids"] >= 0).all()
            assert (rt.cast(o[got["ids"] < 0], d[got["ids"] < 0], any_hit=True)["ids"] == -1).all()
            per_walk[(walk, name)] = got
        del rt
    for name in sets:
        ok = oracle_res[name][0]
        a = per_walk[(WALKS[0], name)]
        for walk in WALKS[1:]:
            b = per_walk[(walk, name)]
            assert np.array_equal(a["ids"][ok], b["ids"][ok]), "%s/%s: walk %d" % (which, name, walk)
            hit = ok & (a["ids"] >= 0)
            ta, tb = a["t"][hit].astype(np.float64), b["t"][hit].astype(np.float64)
            assert (np.abs(ta - tb) <= 1e-6 * np.maximum(ta, 1e-30)).all(), "%s/%s: walk %d" % (which, name, walk)


@pytest.mark.parametrize("which,n,walk", [(w, n, None) for w, n in FLAT] + [(w, n, k) for w, n in TREE for k in WALKS])
def test_cast_corner_rays_equal_render_aov(g19, abi, which, n, walk):
    rt, sc, chk, cam = _scene(g19, abi, which, n, walk=walk)
    ids_r = rt.run(W, H, mode=abi.MODE_PATH, want=("ids",), spp=1, max_depth=1)["ids"]
    o, d = corner_rays(cam, W, H)
    got = rt.cast(o, d)["ids"].reshape(H, W)
    m = _interior(ids_r)
    assert m.mean() > 0.5
    assert np.array_equal(got[m], ids_r[m])


def test_cast_invalid_rays(g19, abi):
    rt, sc, chk, cam = _scene(g19, abi, "HEIGHTFIELD_ROOM", 64)
    nan, inf = float("nan"), float("inf")
    o = np.array([[0, 0, 0]] * 4 + [[nan, 0, 0], [0, inf, 0], [0, 0, -inf]] + [[0, 0, 0]] * 3, np.float64)
    d = np.array([[0, 0, 0], [nan, 1, 0], [1, inf, 0], [0, 0, -inf]] + [[1, 0, 0]] * 6, np.float64)
    tmax = np.array([1e9] * 7 + [0.0, -1.0, nan])
    for walk in WALKS + ("flat",):
        if walk == "flat":
            rt, sc, chk, cam = _scene(g19, abi, "CORNELL", 0)
        else:
            rt.tune("walk", walk)
            rt.setScene(sc)
        got = rt.cast(o, d, tmax=tmax, want_normals=True)
        assert (got["ids"] == -1).all() and np.isposinf(got["t"]).all() and (got["normals"] == 0).all(), walk
        assert (rt.cast(o, d, tmax=tmax, any_hit=True)["ids"] == -1).all(), walk


def _room_bounce_rays(rt, cam, n, seed):
    """bounce rays off the first hits of the 1080p corner rays (the GPU's own cast finds the hits)."""
    o, d = corner_rays(cam, 1920, 1080)
    got = rt.cast(o, d, want_normals=True)
    hit = got["ids"] >= 0
    p = o[hit] + unit(d[hit]) * got["t"][hit, None].astype(np.float64)
    return as_cast(*bounce_rays(p, got["normals"][hit].astype(np.float64), n, seed=seed))


def test_cast_full_size_room(g19, abi):
    from oracle import binding
    sc, cam, _ = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD_ROOM, n=708, w=1920, h=1080)
    rt = g19.RayTracer(cam, (0.0, 0.0, 10.0))
    rt.setScene(sc)
    rt.start()
    o, d = _room_bounce_rays(rt, cam, 1 << 22, seed=7)
    a = rt.cast(o, d, want_normals=True)
    b = rt.cast(o, d, want_normals=True)
    for k in ("ids", "t", "normals"):
        assert a[k].tobytes() == b[k].tobytes(), k
    assert (a["ids"] >= 0).mean() > 0.5
    sub = np.random.default_rng(8).choice(len(o), 1 << 14, replace=False)
    chk = mirror(binding.CheckerLib("oracle"), sc)
    ok, ids, t, nrm = robust_mask(chk, o[sub], d[sub])
    _check_vs_oracle({k: v[sub] for k, v in a.items()}, ok, ids, t, nrm, "room n=708")


def test_cast_device_form_on_a_side_stream_and_stats(g19, abi):
    import torch
    for which, n in (("CORNELL", 0), ("HEIGHTFIELD_ROOM", 64)):
        rt, sc, chk, cam = _scene(g19, abi, which, n)
        o, d = box_rays(*_bounds(sc), 5000, seed=4)
        host = rt.cast(o, d, want_normals=True)
        st = rt.stats()
        assert st.extend_segments == 5000 and st.shadow_segments == 0 and st.kernel_launches == 1 and st.render_ms > 0
        rays = np.zeros((5000, 8), np.float32)
        rays[:, 0:3], rays[:, 3], rays[:, 4:7] = o, np.inf, d
        dev = torch.device("cuda", 0)
        r = torch.from_numpy(rays).to(dev)
        assert r.data_ptr() % 16 == 0
        ids = torch.empty(5000, dtype=torch.int32, device=dev)
        t = torch.empty(5000, dtype=torch.float32, device=dev)
        nrm = torch.empty(5000, 3, dtype=torch.float32, device=dev)
        s = torch.cuda.Stream(device=dev)
        s.wait_stream(torch.cuda.current_stream(dev))
        rt.cast_device(5000, r.data_ptr(), ids.data_ptr(), t.data_ptr(), nrm.data_ptr(), 0, s.cuda_stream)
        s.synchronize()
        assert np.array_equal(ids.cpu().numpy(), host["ids"])
        assert t.cpu().numpy().tobytes() == host["t"].tobytes()
        assert nrm.cpu().numpy().tobytes() == host["normals"].tobytes()
        rt.cast(o, d, any_hit=True)
        st = rt.stats()
        assert st.shadow_segments == 5000 and st.extend_segments == 0
        rt.cast(o, d, count=True)
        st = rt.stats()
        if which != "CORNELL":  # the default 4-wide walk counts its tests
            assert st.node_tests > 0 and st.prim_tests > 0


@pytest.mark.parametrize("which,n", [("CORNELL", 0), ("HEIGHTFIELD_ROOM", 64)])
def test_render_unaffected_by_cast(g19, abi, which, n):
    rt, sc, chk, cam = _scene(g19, abi, which, n)
    before = rt.run(W, H, mode=abi.MODE_PATH, want=("radiance", "ids", "rgb"), spp=4, max_depth=4, seed=3)
    o, d = box_rays(*_bounds(sc), 1 << 16, seed=5)
    rt.cast(o, d, want_normals=True)
    rt.cast(o, d, any_hit=True, count=True)
    after = rt.run(W, H, mode=abi.MODE_PATH, want=("radiance", "ids", "rgb"), spp=4, max_depth=4, seed=3)
    for k in ("radiance", "ids", "rgb"):
        assert before[k].tobytes() == after[k].tobytes(), k


def test_cast_error_codes(g19, abi):
    L = g19.lib()
    rt = g19.RayTracer(g19.Camera((-10.0, 0.0, 0.0), (1.0, 0.0, 0.0), 0.1), (0.0, 0.0, 10.0))
    buf = np.zeros(8 * 4 + 4, np.float32)
    skip = (-buf.ctypes.data % 16) // 4
    rays = buf[skip:skip + 32]
    ids = np.zeros(4, np.int32)
    t = np.zeros(4, np.float32)
    p = lambda a: C.c_void_p(a.ctypes.data)
    assert L.g19_cast_rays(rt.h, 4, p(rays), 0, p(ids), None, None) == abi.ERR_NO_SCENE
    sc, _, _ = g19.Octree.builtin(abi.SCENE_CORNELL, w=64, h=36)
    rt.setScene(sc)
    assert L.g19_cast_rays(None, 4, p(rays), 0, p(ids), None, None) == abi.ERR_INVALID
    assert L.g19_cast_rays(rt.h, -1, p(rays), 0, p(ids), None, None) == abi.ERR_INVALID
    assert L.g19_cast_rays(rt.h, 4, None, 0, p(ids), None, None) == abi.ERR_INVALID
    assert L.g19_cast_rays(rt.h, 4, p(rays), 0, None, None, None) == abi.ERR_INVALID
    assert L.g19_cast_rays(rt.h, 3, C.c_void_p(rays.ctypes.data + 4), 0, p(ids), None, None) == abi.ERR_INVALID
    assert L.g19_cast_rays(rt.h, 4, p(rays), abi.CAST_ANY_HIT, p(ids), p(t), None) == abi.ERR_INVALID
    assert L.g19_cast_rays(rt.h, 4, p(rays), abi.CAST_ANY_HIT, p(ids), None, p(t)) == abi.ERR_INVALID
    assert L.g19_cast_rays(rt.h, 4, p(rays), 4, p(ids), None, None) == abi.ERR_INVALID
    assert L.g19_cast_rays_device(rt.h, -1, None, 0, None, None, None, None) == abi.ERR_INVALID
    assert L.g19_cast_rays(rt.h, 0, None, 0, None, None, None) == abi.OK
    assert L.g19_cast_rays_device(rt.h, 0, None, 0, None, None, None, None) == abi.OK
    assert L.g19_cast_rays(rt.h, 4, p(rays), abi.CAST_ANY_HIT | abi.CAST_COUNT, p(ids), None, None) == abi.OK


CPP = r"""
#include <cmath>
#include <cstdio>
#include "entities.h"
#include "octree.h"
int main(int argc, char** argv) {
    Octree scene({-20, -20, -20}, {20, 20, 20});
    scene.push_back(new ExpQuad(glm::dvec3{0, 0, 0}, 2, 3, (90.0 * M_PI / 180.0), {1, 2, 3}));
    scene.push_back(new ImpSphere(glm::dvec3{3, 4, 4}, 2, {1, 0, 0}));
    scene.push_back(new ImpSphere(glm::dvec3{4, -4, 4}, 2, {0, 0, 1}));
    std::vector<Ray> rays;
    FILE* f = std::fopen(argv[1], "rb");
    double v[6];
    while (std::fread(v, sizeof v, 1, f) == 1) rays.emplace_back(glm::dvec3{v[0], v[1], v[2]}, glm::dvec3{v[3], v[4], v[5]});
    std::fclose(f);
    std::vector<double> t;
    const std::vector<Entity*> hit = scene.nearest(rays, &t);
    for (size_t i = 0; i < hit.size(); ++i) {
        int id = -1;
        for (size_t k = 0; k < scene.entities().size(); ++k)
            if (scene.entities()[k] == hit[i]) id = int(k);
        std::printf("%d %.9g\n", id, t[i]);
    }
    return 0;
}
"""


def test_cpp_octree_nearest_matches_python_cast(g19, abi, tmp_path):
    src = tmp_path / "nearest.cpp"
    src.write_text(CPP)
    exe = str(tmp_path / "nearest")
    libdir = os.path.join(ROOT, "2019global_b200")
    subprocess.run(["g++", "-std=c++14", "-O1", "-DG19_NO_QT", "-I", os.path.join(ROOT, "include"), str(src), "-o", exe,
                    "-L", libdir, "-l2019global_b200", "-Wl,-rpath," + libdir, "-pthread"], check=True)
    sc = g19.Octree((-20,) * 3, (20,) * 3)
    sc.push_back(g19.ExpQuad((0, 0, 0), 2, 3, 90.0 * math.pi / 180.0, (1, 2, 3)))
    sc.push_back(g19.ImpSphere((3, 4, 4), 2, (1, 0, 0)))
    sc.push_back(g19.ImpSphere((4, -4, 4), 2, (0, 0, 1)))
    cam = g19.Camera((-10.0, 0.0, 0.0), (1.0, 0.0, 0.0), 0.1)
    o, d = corner_rays(cam, 100, 100)
    d = unit(d)  # (Ray normalises in FP64: both sides then round the same unit vector to FP32)
    rayfile = tmp_path / "rays.bin"
    np.ascontiguousarray(np.concatenate([o, d], 1), np.float64).tofile(str(rayfile))
    out = subprocess.run([exe, str(rayfile)], capture_output=True, text=True, check=True, timeout=300).stdout.split("\n")
    ids_cpp = np.array([int(line.split()[0]) for line in out if line.strip()], np.int32)
    rt = g19.RayTracer(cam, (-10.0, 10.0, 10.0))
    rt.setScene(sc)
    got = rt.cast(o, d)
    assert (got["ids"] >= 0).sum() > 1000
    assert np.array_equal(ids_cpp, got["ids"])

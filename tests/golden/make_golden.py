"""Generates tests/golden/ref_golden.npz from the UNMODIFIED reference (oracle/_ref/libg19ref.so).

Run where a checkout of the reference exists, after `make -C oracle ref G19_REFERENCE=<checkout>`:
    python tests/golden/make_golden.py
The .npz travels with the repo, so the oracle stays pinned to the reference's own outputs on
machines where neither the reference sources nor the compiled oracle/_ref exist.
Contents (all produced by calling the reference's public API through oracle/ref_harness):
  c1_sha256, c1_hist        RayTracer::run(500,500) on the main.cpp:24-57 scene
  kat_*                     main.cpp:90-133 entity_test / bbox_test vectors
  zoo_<i>_{hit,pts,nrm,uv,bbox,tris}   20 000-ray Entity::intersect probes per entity kind
  zoo_ids, zoo_pts          200x200 frame of the nine-entity scene (ids, hit points)
  cornell_ids               96x54 Cornell primary-hit ids through the subdivided octree
  height_ids                96x54 heightfield (n=32) ids through a deep octree
  cand_*                    Octree::intersect candidate lists for 64 rays
"""
import hashlib
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import binding  # noqa: E402
from util import mirror, probe_rays, quiet_stdout, zoo  # noqa: E402


def main():
    g19 = importlib.import_module("2019global_b200")
    abi = g19.abi
    ref = binding.CheckerLib("ref")
    out = {}
    sc, cam, light = g19.Octree.builtin(abi.SCENE_DEFAULT)
    chk = mirror(ref, sc)
    rgb = chk.render(cam, light, 500, 500)
    out["c1_sha256"] = np.frombuffer(hashlib.sha256(rgb.tobytes()).digest(), np.uint8)
    t = chk.trace(cam, light, 500, 500, want=("ids",), threads=8)
    out["c1_hist"] = np.bincount(t["ids"].ravel() + 1, minlength=4)

    s1 = g19.Octree((-20,) * 3, (20,) * 3)
    s1.push_back(g19.ImpSphere((2, 0, 0), 10, (0, 1, 0)))
    h, p, n = mirror(ref, s1).intersect(0, [[-10, 0, 0]], [[1, .5, .5]])
    out["kat_entity_hit"], out["kat_entity_pt"], out["kat_entity_nrm"] = h, p, n

    z = zoo(g19)
    zc = mirror(ref, z)
    for i in range(len(z)):
        o, d = probe_rays(20000, seed=i)
        h, p, n = zc.intersect(i, o, d)
        m = h.astype(bool)
        out["zoo_%d_hit" % i] = np.packbits(m)
        out["zoo_%d_pts" % i] = p[m][:512]
        out["zoo_%d_nrm" % i] = n[m][:512]
        out["zoo_%d_ptsha" % i] = np.frombuffer(hashlib.sha256(p[m].tobytes() + n[m].tobytes()).digest(), np.uint8)
        with quiet_stdout():
            out["zoo_%d_uv" % i] = zc.texcoord(i, p[m][:512])
        out["zoo_%d_bbox" % i] = zc.bbox(i)
        out["zoo_%d_tris" % i] = zc.triangles(i)
    zcam = g19.Camera((-10, 0, 0), (1, 0, 0), 0.1)
    with quiet_stdout():
        t = zc.trace(zcam, (-10, 10, 10), 200, 200, want=("ids", "points", "rgb"), threads=8)
    out["zoo_ids"] = t["ids"].astype(np.int8)
    out["zoo_ptsha"] = np.frombuffer(hashlib.sha256(t["points"].tobytes()).digest(), np.uint8)
    out["zoo_rgb"] = t["rgb"]
    rng = np.random.default_rng(5)
    cands = []
    for _ in range(64):
        o, d = rng.uniform(-15, 15, 3), rng.uniform(-1, 1, 3)
        c = zc.candidates(o, d)
        cands.append(np.concatenate([[len(c)], c]))
    out["cand_flat"] = np.concatenate(cands).astype(np.int16)

    w, h = 96, 54
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    t = mirror(ref, sc).trace(cam, light, w, h, want=("ids", "rgb"), threads=8)
    out["cornell_ids"] = t["ids"].astype(np.int8)
    out["cornell_rgb"] = t["rgb"]
    sc, cam, light = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD, n=32, w=w, h=h)
    t = mirror(ref, sc).trace(cam, light, w, h, want=("ids",), threads=8)
    out["height_ids"] = t["ids"].astype(np.int16)
    path = os.path.join(HERE, "ref_golden.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

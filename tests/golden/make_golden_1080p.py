"""Generates tests/golden/ref_1080p.npz from the UNMODIFIED reference (oracle/_ref/libg19ref.so): REF-mode primary-hit
ids AT THE SIZE BASELINE.json states (1920x1080), so that the north-star's "primary hits bit-exact" is checked where
it is claimed and not only on toy frames (VERDICT r01 weak 4, SURVEY.md hard part 8).

Run where a checkout of the reference exists, after `make -C oracle ref G19_REFERENCE=<checkout>`:
    python tests/golden/make_golden_1080p.py        (about 2 minutes on 8 cores)
Contents (all from RayTracer::run's own loop, reference include/raytracer.h:41-74, through oracle/ref_harness):
  cornell_ids      (1080, 1920) int8   the walls-first Cornell box (configs[1]/[2] geometry), whole frame
  cornell_rgb_sha  sha256 of the reference's RGB888 frame (row-major, row 0 = top)
  height_rows      row indices of the bands below
  height_ids       (len(height_rows), 1920) int32  the n = 708 heightfield (1 002 528 ImpTriangle entities, the
                   reference octree ~1.5 M nodes deep) WITHOUT the light panel (tests/test_path_link.py explains why)
  room_rows / room_ids   the same bands of the heightfield ROOM scene (bench.py's C4), walls and light included
"""
import hashlib
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import binding  # noqa: E402
from util import quiet_stdout  # noqa: E402

W, H, N = 1920, 1080, 708
BANDS = [(96, 100), (322, 326), (538, 546), (760, 764), (1001, 1005)]  # 24 rows of 1080
SCENE_CORNELL, SCENE_HEIGHTFIELD, SCENE_HEIGHTFIELD_ROOM = 1, 3, 4
ROOT_BOX = ((-20.0,) * 3, (20.0,) * 3)


def bands(chk, cam, light, threads):
    rows, ids = [], []
    for y0, y1 in BANDS:
        t = chk.trace(cam, light, W, H, y0=y0, y1=y1, want=("ids",), threads=threads)
        rows.extend(range(y0, y1))
        ids.append(t["ids"][y0:y1])
    return np.array(rows, np.int32), np.concatenate(ids).astype(np.int32)


def main():
    threads = os.cpu_count() or 8
    ref = binding.CheckerLib("ref")
    out = {}
    t0 = time.time()
    descs, cam, light = binding.builtin_descs(SCENE_CORNELL, 0, W, H)
    chk = ref.scene(*ROOT_BOX, descs)
    with quiet_stdout():
        t = chk.trace(cam, light, W, H, want=("ids", "rgb"), threads=threads)
    assert t["ids"].max() < 127
    out["cornell_ids"] = t["ids"].astype(np.int8)
    out["cornell_rgb_sha"] = np.frombuffer(hashlib.sha256(t["rgb"].tobytes()).digest(), np.uint8)
    print("cornell 1080p: %.1f s, hit %.3f" % (time.time() - t0, (t["ids"] >= 0).mean()))

    t0 = time.time()
    descs, cam, light = binding.builtin_descs(SCENE_HEIGHTFIELD, N, W, H)
    chk = ref.scene(*ROOT_BOX, list(descs)[:-2])  # without the light panel behind the camera
    print("heightfield n=%d built on the reference in %.1f s" % (N, time.time() - t0))
    t0 = time.time()
    with quiet_stdout():
        out["height_rows"], out["height_ids"] = bands(chk, cam, light, threads)
    print("heightfield bands: %.1f s, hit %.3f" % (time.time() - t0, (out["height_ids"] >= 0).mean()))
    del chk

    t0 = time.time()
    descs, cam, light = binding.builtin_descs(SCENE_HEIGHTFIELD_ROOM, N, W, H)
    chk = ref.scene(*ROOT_BOX, descs)
    with quiet_stdout():
        out["room_rows"], out["room_ids"] = bands(chk, cam, light, threads)
    print("room bands: %.1f s, hit %.3f" % (time.time() - t0, (out["room_ids"] >= 0).mean()))

    path = os.path.join(HERE, "ref_1080p.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

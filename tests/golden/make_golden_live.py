"""Generates tests/golden/ref_live.npz: what the comparisons against the reference in tests/test_oracle_ref.py,
tests/test_path_link.py and tests/test_ref_fullsize_gpu.py compare with, so that they run without oracle/_ref.

    python tests/golden/make_golden_live.py

Source, recorded in the file as `source`:
  reference     the UNMODIFIED reference (oracle/_ref/libg19ref.so, built by `make -C oracle ref` from a checkout
                named by G19_REFERENCE), when it is built;
  restatement   otherwise oracle/libg19oracle.so, which those same tests hold byte-equal to the compiled reference on
                exactly these inputs. Before writing, the restatement is checked against the outputs stored from the
                reference itself (ref_golden.npz: config-1 sha256 and histogram; ref_1080p.npz: the 1080p Cornell ids
                and the sha256 of its RGB888 frame); a mismatch writes nothing.
Contents:
  zoo_<i>_{hit,ptsha,uv}, tri_derived     util.live_zoo
  frame_<scene>_{ids,points,normals,rgb,run}   util.live_frames (sha256 digests)
  material_{shade,ids,rgb}                util.live_material
  c1_ids            (500, 500) int8   config-1 primary-hit ids of the per-pixel trace
  band_rows, band_cornell_rgb   rows 700..715 of the 1080p Cornell RGB888 frame
  room96_ids        (180, 320) int16  HEIGHTFIELD_ROOM n=96 ids at 320x180
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
from util import live_frames, live_material, live_zoo, mirror, quiet_stdout, zoo  # noqa: E402

BAND = (700, 716)


def check_restatement(g19, abi, oracle, threads):
    gold = np.load(os.path.join(HERE, "ref_golden.npz"))
    g1080 = np.load(os.path.join(HERE, "ref_1080p.npz"))
    sc, cam, light = g19.Octree.builtin(abi.SCENE_DEFAULT)
    c = mirror(oracle, sc)
    assert hashlib.sha256(c.render(cam, light, 500, 500).tobytes()).digest() == bytes(gold["c1_sha256"])
    t = c.trace(cam, light, 500, 500, want=("ids",), threads=threads)
    assert np.bincount(t["ids"].ravel() + 1, minlength=4).tolist() == gold["c1_hist"].tolist()
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=1920, h=1080)
    t = mirror(oracle, sc).trace(cam, light, 1920, 1080, want=("ids", "rgb"), threads=threads)
    assert np.array_equal(t["ids"], g1080["cornell_ids"].astype(np.int32))
    assert hashlib.sha256(t["rgb"].tobytes()).digest() == bytes(g1080["cornell_rgb_sha"])


def main():
    g19 = importlib.import_module("2019global_b200")
    abi = g19.abi
    threads = os.cpu_count() or 8
    oracle = binding.CheckerLib("oracle")
    if binding.available("ref"):
        chk, source = binding.CheckerLib("ref"), "reference"
    else:
        check_restatement(g19, abi, oracle, threads)
        chk, source = oracle, "restatement"
    out = {"source": np.array(source)}
    out.update(live_zoo(chk, zoo(g19)))
    out.update(live_frames(chk, g19, abi))
    out.update(live_material(chk, g19))
    sc, cam, light = g19.Octree.builtin(abi.SCENE_DEFAULT)
    with quiet_stdout():
        t = mirror(chk, sc).trace(cam, light, 500, 500, want=("ids",), threads=threads)
    out["c1_ids"] = t["ids"].astype(np.int8)
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=1920, h=1080)
    with quiet_stdout():
        t = mirror(chk, sc).trace(cam, light, 1920, 1080, y0=BAND[0], y1=BAND[1], want=("rgb",), threads=threads)
    out["band_rows"] = np.array(BAND, np.int32)
    out["band_cornell_rgb"] = t["rgb"][BAND[0]:BAND[1]]
    sc, cam, light = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD_ROOM, n=96, w=320, h=180)
    with quiet_stdout():
        t = mirror(chk, sc).trace(cam, light, 320, 180, want=("ids",), threads=threads)
    out["room96_ids"] = t["ids"].astype(np.int16)
    path = os.path.join(HERE, "ref_live.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes, source:", source)


if __name__ == "__main__":
    main()

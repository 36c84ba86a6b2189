"""The closed-form ray-query answers of tests/walk_cases.py, checked without a GPU: the rebuilt heightfield equals the
engine's scene bit for bit, and every aimed answer equals the FP64 PATH oracle's (cast_util.path_cast). A failure of
tests/test_walk_exact_gpu.py can then only be the kernel's."""
import numpy as np
import pytest

import walk_cases as wc
from cast_util import as_cast, path_cast
from util import mirror


def _check_vs_oracle(chk, case, what):
    o, d = as_cast(case["o"], case["d"])  # the rays as a cast receives them
    ids, t, nrm = path_cast(chk, o, d)
    ok = (ids[:, None] == case["ids"]).any(1)
    assert ok.all(), "%s: %d of %d aimed rays hit another primitive (first: %s, expected %s)" % (
        what, int((~ok).sum()), len(ok), ids[~ok][:5], case["ids"][~ok][:5])
    err = np.abs(t - case["t"])
    assert (err <= case["tol"]).all(), "%s: t off by up to %.3g" % (what, err.max())
    assert ((nrm * case["normal"]).sum(1) >= 0.9999).all(), what
    hi, lo = wc.occlusion_pairs(case)
    assert (path_cast(chk, o, d, tmax=hi, any_hit=True)[0] >= 0).all(), what
    assert (path_cast(chk, o, d, tmax=lo, any_hit=True)[0] == -1).all(), what


@pytest.mark.parametrize("which,n", [("HEIGHTFIELD_ROOM", 64), ("HEIGHTFIELD", 64), ("HEIGHTFIELD_ROOM", 708),
                                     ("HEIGHTFIELD", 708)])
def test_rebuilt_heightfield_equals_the_engine_scene(g19, abi, which, n):
    sc, _, _ = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=n, w=64, h=36)
    tris, first = wc.heightfield_scene(n, which.endswith("ROOM"))
    assert len(sc) == len(tris)
    rng = np.random.default_rng(0)
    mesh = np.arange(first, first + 2 * n * n)
    check = np.union1d(np.setdiff1d(np.arange(len(tris)), mesh), rng.choice(mesh, min(len(mesh), 4096), replace=False))
    check = np.union1d(check, [first, first + 1, first + 2 * n * n - 1])
    for i in check:
        got = sc.triangles(int(i))
        assert got.shape == (1, 9), i
        assert got[0].tobytes() == tris[i].reshape(9).tobytes(), "entity %d" % i


@pytest.mark.parametrize("room", [True, False])
def test_heightfield_answers_equal_oracle_n64(g19, abi, oracle, room):
    which = "SCENE_HEIGHTFIELD_ROOM" if room else "SCENE_HEIGHTFIELD"
    sc, _, _ = g19.Octree.builtin(getattr(abi, which), n=64, w=64, h=36)
    chk = mirror(oracle, sc)
    for name, case in wc.heightfield_cases(64, room, wall_points=64).items():
        _check_vs_oracle(chk, case, "%s n=64 %s" % (which, name))
    for v in wc.axis_variants(wc.subset(wc.heightfield_cases(64, room, wall_points=1)["axis"], slice(0, 4096))):
        _check_vs_oracle(chk, v, "%s n=64 axis variant" % which)


@pytest.mark.parametrize("room", [True, False])
def test_heightfield_answers_equal_oracle_n708_sample(g19, abi, oracle, room):
    which = "SCENE_HEIGHTFIELD_ROOM" if room else "SCENE_HEIGHTFIELD"
    sc, _, _ = g19.Octree.builtin(getattr(abi, which), n=708, w=64, h=36)
    chk = mirror(oracle, sc)
    rng = np.random.default_rng(1)
    for name, case in wc.heightfield_cases(708, room).items():
        n = len(case["t"])
        idx = np.sort(rng.choice(n, min(n, 1 << 16), replace=False))
        _check_vs_oracle(chk, wc.subset(case, idx), "%s n=708 %s" % (which, name))


def test_closed_room_rays_hit_in_the_oracle(g19, abi, oracle):
    sc, _, _ = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD_ROOM, n=64, w=64, h=36)
    chk = mirror(oracle, sc)
    o, d, seam = wc.closed_room_rays(1 << 16, seed=3)
    ids, _, _ = path_cast(chk, *as_cast(o, d))
    assert (ids >= 0).all()
    assert seam.sum() < 10  # the exemption is a thin set


@pytest.mark.parametrize("name", list(wc.edge_cases()))
def test_edge_case_answers_equal_oracle(g19, oracle, name):
    case = wc.edge_cases()[name]()
    sc = wc.build_octree(g19, case)
    chk = mirror(oracle, sc)
    for cname, c in case["cases"].items():
        _check_vs_oracle(chk, c, "%s/%s" % (name, cname))
        if np.all(np.abs(c["d"]).max(1) == 1.0):
            for v in wc.axis_variants(c):
                _check_vs_oracle(chk, v, "%s/%s variant" % (name, cname))

"""The PATH oracle's batched ray queries (g19o_path_cast) and the Python side of g19_cast_rays. No GPU needed."""
import numpy as np
import pytest

from cast_util import corner_rays, path_cast, unit
from test_path_link import SCENES, _interior
from util import mirror


@pytest.mark.parametrize("which,w,h,n", SCENES)
def test_oracle_cast_of_corner_rays_equals_path_primary(g19, abi, oracle, which, w, h, n):
    from oracle import binding
    sc, cam, _ = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=n, w=w, h=h)
    chk = mirror(oracle, sc)
    ids_p, pts_p, nrm_p = binding.path_primary(chk, cam, w, h)
    o, d = corner_rays(cam, w, h)
    ids, t, nrm = path_cast(chk, o, d)
    ids, t, nrm = ids.reshape(h, w), t.reshape(h, w), nrm.reshape(h, w, 3)
    m = _interior(ids_p)
    assert m.sum() > 0.5 * w * h
    assert np.array_equal(ids[m], ids_p[m])
    hit = m & (ids_p >= 0)
    pts = o.reshape(h, w, 3) + unit(d).reshape(h, w, 3) * t[..., None]
    assert np.abs(pts[hit] - pts_p[hit]).max() <= 1e-9
    assert np.abs(nrm[hit] - nrm_p[hit]).max() <= 1e-9
    miss = m & (ids_p < 0)
    assert (t[miss] == np.finfo(np.float64).max).all() and (nrm[miss] == 0).all()


@pytest.mark.parametrize("which", ["CORNELL", "HEIGHTFIELD_ROOM"])
def test_oracle_any_hit_consistent_with_nearest(g19, abi, oracle, which):
    from cast_util import bounce_rays
    sc, cam, _ = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=32, w=64, h=36)
    chk = mirror(oracle, sc)
    o, d = corner_rays(cam, 64, 36)
    ids, t, nrm = path_cast(chk, o, d)
    hit = ids >= 0
    bo, bd = bounce_rays(o[hit] + unit(d[hit]) * t[hit, None], nrm[hit], 2000, seed=3)
    for oo, dd in ((o, d), (bo, bd)):
        ids, t, _ = path_cast(chk, oo, dd)
        hit = ids >= 0
        assert hit.sum() > 0.5 * len(ids)
        near, _, _ = path_cast(chk, oo[hit], dd[hit], tmax=0.5 * t[hit], any_hit=True)
        far, _, _ = path_cast(chk, oo[hit], dd[hit], tmax=1.5 * t[hit], any_hit=True)
        assert (near == -1).all()
        assert (far >= 0).all()
        miss, _, _ = path_cast(chk, oo[~hit], dd[~hit], any_hit=True)
        assert (miss == -1).all()


def test_oracle_cast_invalid_rays(g19, abi, oracle):
    sc, _, _ = g19.Octree.builtin(abi.SCENE_CORNELL, w=64, h=36)
    chk = mirror(oracle, sc)
    nan, inf = float("nan"), float("inf")
    o = np.array([[0, 0, 0]] * 3 + [[nan, 0, 0], [0, inf, 0]] + [[0, 0, 0]] * 3, float)
    d = np.array([[0, 0, 0], [nan, 1, 0], [1, inf, 0], [1, 0, 0], [1, 0, 0]] + [[1, 0, 0]] * 3, float)
    tmax = np.array([1e9] * 5 + [0.0, -1.0, nan])
    for any_hit in (False, True):
        ids, t, nrm = path_cast(chk, o, d, tmax=tmax, any_hit=any_hit)
        assert (ids == -1).all() and (t == np.finfo(np.float64).max).all() and (nrm == 0).all()


def test_cast_abi_constants_and_exports(g19, abi):
    assert abi.ABI_VERSION == 6
    assert (abi.CAST_ANY_HIT, abi.CAST_COUNT) == (1, 2)
    assert "g19_cast_rays" in g19.EXPORTS and "g19_cast_rays_device" in g19.EXPORTS
    L = g19.lib()
    assert L.g19_cast_rays.argtypes is not None and len(L.g19_cast_rays.argtypes) == 7
    assert L.g19_cast_rays_device.argtypes is not None and len(L.g19_cast_rays_device.argtypes) == 8

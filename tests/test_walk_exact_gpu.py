"""Every tree walk and traversal knob against exact per-primitive answers (tests/walk_cases.py): rays aimed at every
triangle of the 1 M-triangle heightfield and at the primitives of builder edge cases must return that primitive, at
the distance they were aimed from, under each walk (1, 3, 4, the counting forms) and each knob that selects other
code or another kernel instantiation. A primitive lost from a leaf or a box rounded inwards fails the rays aimed at it.
The render kernels (primary_kernel, trace_kernel) are checked under the same knobs against the default configuration."""
import numpy as np
import pytest

import walk_cases as wc
from cast_util import corner_rays
from test_path_link import _interior
from util import rel_rmse

pytestmark = pytest.mark.gpu

# upload-time knobs (walk, leaf_max, top_level, tree_build, bvh_leaf) are set before setScene; every knob of this list
# not named by a configuration is reset to its default first
KNOBS = ("walk", "coop_leaf", "walk_steps", "leaf_batch", "top_level", "leaf_max", "trace_occ", "refill", "tree_build",
         "bvh_leaf", "bvh_spec", "bvh_stack", "sort_rays")


def _configs():
    c = [("walk%d" % w, {"walk": w}, False) for w in (1, 3, 4)]
    w1 = [("coop_leaf", 0), ("walk_steps", 1), ("walk_steps", 16), ("leaf_batch", 1), ("leaf_batch", 16), ("top_level", 0),
          ("top_level", 3), ("top_level", 8), ("leaf_max", 1), ("leaf_max", 2), ("leaf_max", 64), ("trace_occ", 3),
          ("refill", 1), ("refill", 32), ("tree_build", "host")]
    c += [("walk1_%s%s" % (k, v), {"walk": 1, k: v}, False) for k, v in w1]
    bvh = [("bvh_leaf", 1), ("bvh_leaf", 2), ("bvh_leaf", 3), ("bvh_leaf", 8), ("bvh_spec", 0), ("bvh_spec", 1), ("bvh_spec", 2),
           ("bvh_spec", 3), ("bvh_stack", 4), ("bvh_stack", 64), ("walk_steps", 1), ("walk_steps", 16), ("trace_occ", 3),
           ("refill", 1), ("refill", 32)]
    c += [("walk%d_%s%s" % (w, k, v), {"walk": w, k: v}, False) for w in (3, 4) for k, v in bvh]
    c += [("walk%d_count" % w, {"walk": w}, True) for w in (1, 4)]
    return c


CONFIGS = _configs()


def _configure(rt, sc, knobs):
    for k in KNOBS:
        rt.tune(k, knobs.get(k))
    rt.setScene(sc)


@pytest.fixture(scope="module")
def tracer(g19):
    rt = g19.RayTracer(g19.Camera((-10.0, 0.0, 0.0), (1.0, 0.0, 0.0), 0.1), (0.0, 0.0, 10.0))
    rt.start()
    return rt


# ---- casts on the device: the full-size sets hold millions of rays -------------------------------------------------
def _records(o, d, tmax=None):
    import torch
    r = np.zeros((len(o), 8), np.float32)
    r[:, 0:3], r[:, 4:7] = o, d
    r[:, 3] = np.inf if tmax is None else tmax
    return torch.from_numpy(r).cuda()


def _dev_case(case):
    import torch
    hi, lo = wc.occlusion_pairs(case)
    return {"rays": _records(case["o"], case["d"]), "hi": _records(case["o"], case["d"], hi), "lo": _records(case["o"], case["d"], lo),
            "ids": torch.from_numpy(case["ids"]).cuda(), "t": torch.from_numpy(case["t"]).cuda(),
            "normal": torch.from_numpy(case["normal"]).cuda(), "tol": case["tol"]}


def _cast(rt, rays, any_hit=False, count=False):
    import torch
    n = rays.shape[0]
    ids = torch.empty(n, dtype=torch.int32, device="cuda")
    t = None if any_hit else torch.empty(n, dtype=torch.float32, device="cuda")
    nrm = None if any_hit else torch.empty(n, 3, dtype=torch.float32, device="cuda")
    flags = (1 if any_hit else 0) | (2 if count else 0)  # G19_CAST_ANY_HIT, G19_CAST_COUNT
    rt.cast_device(n, rays.data_ptr(), ids.data_ptr(), 0 if t is None else t.data_ptr(), 0 if nrm is None else nrm.data_ptr(),
                   flags, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return ids, t, nrm


def _check_dev(rt, c, count, what):
    import torch
    ids, t, nrm = _cast(rt, c["rays"], count=count)
    bad = ~(ids[:, None].long() == c["ids"].long()).any(1)
    if bad.any():
        k = torch.nonzero(bad)[:5, 0]
        pytest.fail("%s: %d of %d aimed rays answer another id (got %s, expected %s)" % (
            what, int(bad.sum()), len(bad), ids[k].tolist(), c["ids"][k, 0].tolist()))
    err = (t.double() - c["t"]).abs()
    assert bool((err <= c["tol"]).all()), "%s: |t - expected| up to %.3g" % (what, float(err.max()))
    dot = (nrm.double() * c["normal"]).sum(1)
    assert bool((dot >= 0.9999).all()), "%s: %d normals off" % (what, int((dot < 0.9999).sum()))
    hit = _cast(rt, c["hi"], any_hit=True, count=count)[0]
    assert bool((hit >= 0).all()), "%s: %d occlusion queries with tmax above t miss" % (what, int((hit < 0).sum()))
    free = _cast(rt, c["lo"], any_hit=True, count=count)[0]
    assert bool((free == -1).all()), "%s: %d occlusion queries with tmax below t hit" % (what, int((free >= 0).sum()))


_full = {}


def _full_size(g19, abi, which):
    """(scene, device sets, closed-room rays and seam mask) of a heightfield scene at n = 708, built once per module."""
    if which not in _full:
        room = which == "HEIGHTFIELD_ROOM"
        sc, _, _ = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=708, w=64, h=36)
        cases = wc.heightfield_cases(708, room)
        sets = {k: _dev_case(v) for k, v in cases.items()}
        for i, v in enumerate(wc.axis_variants(wc.subset(cases["axis"], slice(0, 1 << 16)))):
            sets["axis_variant%d" % i] = _dev_case(v)
        closed = None
        if room:
            o, d, seam = wc.closed_room_rays(1 << 22, seed=11)
            closed = (_records(o, d), seam, o, d)
        _full[which] = (sc, sets, closed)
    return _full[which]


@pytest.mark.parametrize("name,knobs,count", CONFIGS, ids=[c[0] for c in CONFIGS])
@pytest.mark.parametrize("which", ["HEIGHTFIELD_ROOM", "HEIGHTFIELD"])
def test_full_size_aimed_rays_exact(g19, abi, tracer, which, name, knobs, count):
    sc, sets, closed = _full_size(g19, abi, which)
    _configure(tracer, sc, knobs)
    for set_name, c in sets.items():
        _check_dev(tracer, c, count, "%s n=708 %s %s" % (which, name, set_name))
    if closed is not None:
        rays, seam, o, d = closed
        ids = _cast(tracer, rays, count=count)[0].cpu().numpy()
        miss = ids < 0
        assert not (miss & ~seam).any(), "%s %s: %d closed-room rays escape away from the seams (first: o %s d %s)" % (
            which, name, int((miss & ~seam).sum()), o[miss & ~seam][:2].tolist(), d[miss & ~seam][:2].tolist())


@pytest.mark.parametrize("walk", [1, 4])
def test_axis_rays_visit_no_more_nodes_than_tilted_ones(g19, abi, tracer, walk):
    """A zero direction component is replaced by +-1e-20 before a walk forms 1 / d. Without that, the slab along the
    zero axis is NaN, which fminf / fmaxf drop: the ray enters every box its other two slabs cross. The hits stay the
    same, but the walk visits a whole slice of the mesh. The counting walks' node tests for 64 K axis rays must stay
    close to those of the same rays turned by about 1e-4 rad."""
    import torch
    sc, sets, _ = _full_size(g19, abi, "HEIGHTFIELD")
    axis = sets["axis"]["rays"]
    rays = torch.cat([axis[:1 << 15], axis[-(1 << 15):]])  # both +x and -x
    tilted = rays.clone()
    tilted[:, 5], tilted[:, 6] = 1e-4, -1e-4
    _configure(tracer, sc, {"walk": walk})
    nodes = []
    for r in (rays, tilted):
        _cast(tracer, r, count=True)
        st = tracer.stats()
        nodes.append(int(st.node_tests))
    assert nodes[1] > 0
    assert nodes[0] <= 1.5 * nodes[1], "walk %d: axis rays %d node tests, tilted %d" % (walk, nodes[0], nodes[1])


# ---- builder edge cases -----------------------------------------------------------------------------------------
EDGE_CONFIGS = [("walk1", {"walk": 1}), ("walk3", {"walk": 3}), ("walk4", {"walk": 4}), ("walk3_bvh_leaf1", {"walk": 3, "bvh_leaf": 1}),
                ("walk4_bvh_leaf1", {"walk": 4, "bvh_leaf": 1}), ("walk3_bvh_leaf8", {"walk": 3, "bvh_leaf": 8}),
                ("walk4_bvh_leaf8", {"walk": 4, "bvh_leaf": 8})]
_edge = {}


@pytest.mark.parametrize("cfg,knobs", EDGE_CONFIGS, ids=[c[0] for c in EDGE_CONFIGS])
@pytest.mark.parametrize("case_name", list(wc.edge_cases()))
def test_edge_case_aimed_rays_exact(g19, tracer, case_name, cfg, knobs):
    if case_name not in _edge:
        case = wc.edge_cases()[case_name]()
        sets = dict(case["cases"])
        for k, c in case["cases"].items():
            if np.all(np.abs(c["d"]).max(1) == 1.0):
                for i, v in enumerate(wc.axis_variants(c)):
                    sets["%s_variant%d" % (k, i)] = v
        _edge[case_name] = (wc.build_octree(g19, case), {k: _dev_case(v) for k, v in sets.items()})
    sc, sets = _edge[case_name]
    _configure(tracer, sc, knobs)
    for set_name, c in sets.items():
        _check_dev(tracer, c, False, "%s %s %s" % (case_name, cfg, set_name))


# ---- the render kernels under the same knobs ------------------------------------------------------------------------
RW, RH = 96, 54
RENDER_CONFIGS = [c for c in CONFIGS if not c[2]] + [("walk%d_sort_rays%d" % (w, s), {"walk": w, "sort_rays": s}, False)
                                                      for w in (1, 4) for s in (0, 1)]
_render = {}


def _render_run(g19, abi, rt, knobs):
    sc, cam = _render["scene"]
    rt.camera = cam
    _configure(rt, sc, knobs)
    rad = rt.run(RW, RH, mode=abi.MODE_PATH, want=("radiance",), spp=4, max_depth=5, seed=23)["radiance"]
    st = rt.stats()
    ids = rt.run(RW, RH, mode=abi.MODE_PATH, want=("ids",), spp=1, max_depth=1)["ids"]
    return rad, int(st.extend_segments), int(st.shadow_segments), ids


@pytest.mark.parametrize("name,knobs,count", RENDER_CONFIGS, ids=[c[0] for c in RENDER_CONFIGS])
def test_render_under_knobs_matches_default(g19, abi, tracer, name, knobs, count):
    if "scene" not in _render:
        sc, cam, _ = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD_ROOM, n=40, w=RW, h=RH)
        _render["scene"] = (sc, cam)
        _render["default"] = _render_run(g19, abi, tracer, {})
    rad0, ext0, shd0, _ = _render["default"]
    rad, ext, shd, ids = _render_run(g19, abi, tracer, knobs)
    assert rad0.mean() > 0.005
    assert rel_rmse(rad, rad0) <= 2e-3, name
    assert abs(ext - ext0) <= 1e-3 * ext0 + 2 and abs(shd - shd0) <= 1e-3 * shd0 + 2, (name, ext, ext0, shd, shd0)
    o, d = corner_rays(_render["scene"][1], RW, RH)
    got = tracer.cast(o, d)["ids"].reshape(RH, RW)
    m = _interior(ids)
    # a mesh cell of n = 40 spans a few pixels at 96 x 54, so about 45 % of the pixels see one id in their 3 x 3
    # neighbourhood: enough to compare, and the same share under every knob
    assert m.sum() >= 2000
    assert np.array_equal(got[m], ids[m]), name

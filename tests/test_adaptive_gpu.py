"""Noise-targeted adaptive sampling (g19_render_adaptive) on the GPU.

A path's random numbers depend only on (pixel, sample, bounce) and accumulate adds a pixel's samples in sample order, so
a tile that stopped after n samples must hold exactly the bytes of a uniform render at spp = n: everything below that is
about the images is checked bit for bit. The variance output is checked against the FP64 oracle's sample moments and
against the spread of independent seeds.
"""
import threading

import numpy as np
import pytest

from adaptive_util import (TILE, allowed_counts, luminance, path_moments, per_pixel, tile_error, tile_max, variance_of_mean)
from oracle import binding
from util import mirror

pytestmark = pytest.mark.gpu

# (id, builtin scene, heightfield n, max_depth, w, h): a flat diffuse scene (C2), flat with mirror and glass (C3), and two
# tree scenes (the room at n = 40, the open heightfield); ragged frames, so that edge tiles carry padding
SCENES = [("cornell", "CORNELL", 0, 5, 100, 70), ("glass", "CORNELL_GLASS", 0, 8, 130, 75),
          ("room", "HEIGHTFIELD_ROOM", 40, 5, 100, 70), ("heightfield", "HEIGHTFIELD", 24, 4, 130, 75)]
IDS = [c[0] for c in SCENES]


def _tracer(g19, abi, which, n, w, h):
    sc, cam, light = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=n, w=w, h=h)
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()
    return rt, sc, cam


def _uniform(rt, abi, w, h, spp, depth, seed, **kw):
    out = rt.run(w, h, mode=abi.MODE_PATH, want=("rgb", "radiance"), spp=spp, max_depth=depth, seed=seed, **kw)
    return out, rt.stats()


def _tiles_of(a, h, w):
    """Per-tile count map (tiles_y, tiles_x) of a per-pixel spp map, checking that every tile is uniform."""
    t = tile_max(a.astype(np.float64))
    assert np.array_equal(per_pixel(t, h, w), a), "a tile's pixels disagree on their count"
    return t.astype(np.int64)


def _pick_tau(rt, w, h, depth, seed, min_spp):
    """A target that half of the tiles meet by 4 min_spp samples (E is a tile's worst pixel: it falls slowly)."""
    r = rt.run_adaptive(w, h, 1e-30, min_spp, 4 * min_spp, depth, seed)
    return float(np.median(tile_error(r["radiance"], r["variance"])))


@pytest.mark.parametrize("case", SCENES, ids=IDS)
def test_degenerate_targets_bit_identical(g19, abi, case):
    _, which, n, depth, w, h = case
    rt, _, _ = _tracer(g19, abi, which, n, w, h)
    spp, min_spp, seed = 16, 4, 3
    full, st_full = _uniform(rt, abi, w, h, spp, depth, seed)
    low, st_low = _uniform(rt, abi, w, h, min_spp, depth, seed)
    # unreachable target: every tile takes spp -- except a tile with no noise at all (E = 0 <= tau: the open
    # heightfield's sky), which stops at min_spp
    a = rt.run_adaptive(w, h, 1e-30, min_spp, spp, depth, seed)
    st = rt.stats()
    quiet = a["spp"] != spp
    assert (a["spp"][quiet] == min_spp).all() and (a["variance"][quiet] == 0).all()
    if which != "HEIGHTFIELD":
        assert not quiet.any()
    for mask, u in ((~quiet, full), (quiet, low)):
        assert np.array_equal(a["radiance"][mask].view(np.uint32), u["radiance"][mask].view(np.uint32))
        assert np.array_equal(a["rgb"][mask], u["rgb"][mask])
    assert st.samples == int(a["spp"].astype(np.int64).sum())
    if not quiet.any():
        assert st.samples == st_full.samples == w * h * spp
    # target met at once: every tile stops at min_spp
    b = rt.run_adaptive(w, h, 1e30, min_spp, spp, depth, seed)
    assert (b["spp"] == min_spp).all()
    assert b["radiance"].tobytes() == low["radiance"].tobytes()
    assert b["rgb"].tobytes() == low["rgb"].tobytes()
    assert rt.stats().samples == st_low.samples


@pytest.mark.parametrize("case", SCENES, ids=IDS)
def test_tiles_exact_and_stopping_rule(g19, abi, case):
    _, which, n, depth, w, h = case
    rt, _, _ = _tracer(g19, abi, which, n, w, h)
    spp, min_spp, seed = 32, 4, 5
    tau = _pick_tau(rt, w, h, depth, seed, min_spp)
    a = rt.run_adaptive(w, h, tau, min_spp, spp, depth, seed)
    samples = rt.stats().samples
    counts = _tiles_of(a["spp"], h, w)
    seen = sorted(set(counts.ravel().tolist()))
    print("%s: tau %.4g, tile counts %s" % (which, tau, {c: int((counts == c).sum()) for c in seen}))
    assert set(seen) <= set(allowed_counts(min_spp, spp))
    assert len(seen) >= 2, "the target should split the tiles"
    assert samples == int(a["spp"].astype(np.int64).sum())
    # every tile holds the bytes of a uniform render at its count
    for c in seen:
        u, _ = _uniform(rt, abi, w, h, c, depth, seed)
        mask = a["spp"] == c
        assert np.array_equal(a["radiance"][mask].view(np.uint32), u["radiance"][mask].view(np.uint32)), c
        assert np.array_equal(a["rgb"][mask], u["rgb"][mask]), c
    # the rule: a tile below spp met the target; a tile above min_spp missed it at its previous count
    E = tile_error(a["radiance"], a["variance"])
    band = 1e-4 * tau
    stopped = counts < spp
    assert (E[stopped] <= tau + band).all(), E[stopped].max()
    for c in seen:
        if c == min_spp:
            continue
        prev = max(k for k in allowed_counts(min_spp, spp) if k < c)
        p = rt.run_adaptive(w, h, 1e-30, min_spp, prev, depth, seed)
        E_prev = tile_error(p["radiance"], p["variance"])
        assert (E_prev[counts == c] > tau - band).all(), (c, E_prev[counts == c].min())


def test_variance_matches_oracle(g19, abi, oracle):
    """The GPU's v against v from the oracle's FP64 moments of the same samples (same seed) on a window."""
    w, h, depth, n, seed = 96, 54, 5, 16, 7
    rt, sc, cam = _tracer(g19, abi, "CORNELL", 0, w, h)
    r = rt.run_adaptive(w, h, 1e-30, 2, n, depth, seed)
    win = (16, 8, 80, 40)
    mom = path_moments(mirror(oracle, sc), cam, w, h, 0, n, depth, seed, win)
    v_ref, m_ref = variance_of_mean(mom, n)
    v = r["variance"][win[1]:win[3], win[0]:win[2]].astype(np.float64)
    err = float(np.sqrt(np.mean((v - v_ref) ** 2)) / v_ref.mean())
    m_err = float(np.sqrt(np.mean((luminance(r["radiance"][win[1]:win[3], win[0]:win[2]]) - m_ref) ** 2)) / m_ref.mean())
    print("variance relRMSE vs oracle %.3e (mean luminance %.3e), mean v %.4g" % (err, m_err, v_ref.mean()))
    assert v_ref.mean() > 0
    assert m_err <= 1e-2
    # measured on a B200: 4.3e-6 (FP32 sums of the same samples); a path that parts ways with the oracle's at a
    # discontinuity would show far above the bar
    assert err <= 1e-3


def test_variance_matches_seed_spread(g19, abi):
    """Over 8 seeds at fixed n: the mean over pixels of the variance of the per-seed means against the mean reported v."""
    w, h, depth, n = 64, 64, 5, 16
    rt, _, _ = _tracer(g19, abi, "CORNELL", 0, w, h)
    means, vs = [], []
    for seed in range(8):
        r = rt.run_adaptive(w, h, 1e-30, 2, n, depth, 100 + seed)
        means.append(luminance(r["radiance"]))
        vs.append(r["variance"].astype(np.float64))
    spread = np.var(np.stack(means), axis=0, ddof=1).mean()
    reported = np.stack(vs).mean()
    ratio = spread / reported
    print("seed spread %.5g, reported v %.5g, ratio %.3f" % (spread, reported, ratio))
    # the per-pixel sample variance over 8 seeds has a relative spread of sqrt(2/7); 4096 pixels average most of it out,
    # what is left is the heavy tail of the few pixels that see the light through a rare path
    assert 0.85 <= ratio <= 1.15


def test_pass_and_lane_invariance(g19, abi):
    w, h, depth = 100, 70, 8
    rt, _, _ = _tracer(g19, abi, "CORNELL_GLASS", 0, w, h)
    spp, min_spp, seed = 24, 3, 11
    tau = _pick_tau(rt, w, h, depth, seed, min_spp)
    ref = rt.run_adaptive(w, h, tau, min_spp, spp, depth, seed)
    samples = rt.stats().samples
    assert len(set(ref["spp"].ravel().tolist())) >= 2
    variants = [dict(spp_per_pass=1), dict(spp_per_pass=5), dict(spp_per_pass=0), dict(pixels_per_pass=1024),
                dict(pixels_per_pass=3000, spp_per_pass=5)]
    for lanes in (1, 4):
        rt.tune("lanes", lanes)
        for kw in variants:
            r = rt.run_adaptive(w, h, tau, min_spp, spp, depth, seed, **kw)
            for k in ("rgb", "radiance", "variance", "spp"):
                assert r[k].tobytes() == ref[k].tobytes(), (lanes, kw, k)
            assert rt.stats().samples == samples
    rt.tune("lanes")


@pytest.mark.parametrize("which,n", [("CORNELL", 0), ("HEIGHTFIELD_ROOM", 40)], ids=["cornell", "room"])
def test_tile_sharding_bit_identical(g19, abi, which, n):
    w, h, depth = 130, 75, 5
    rt, _, _ = _tracer(g19, abi, which, n, w, h)
    spp, min_spp, seed = 16, 2, 9
    tau = _pick_tau(rt, w, h, depth, seed, min_spp)
    one = rt.run_adaptive(w, h, tau, min_spp, spp, depth, seed)
    samples = rt.stats().samples
    out = {"rgb": np.zeros((h, w, 3), np.uint8), "radiance": np.zeros((h, w, 3), np.float32),
           "variance": np.zeros((h, w), np.float32), "spp": np.zeros((h, w), np.int32)}
    total = 0
    for rank in range(4):
        rt.run_adaptive(w, h, tau, min_spp, spp, depth, seed, out=out, rank=rank, world=4)
        total += rt.stats().samples
    assert total == samples
    for k in out:
        assert out[k].tobytes() == one[k].tobytes(), k


def test_isolation_from_uniform_renders(g19, abi):
    """A uniform render just before and just after an adaptive one are byte-equal (frames in a row overlap on the side
    lanes, tune overlap_frames), with a flat and a tree scene alternating on one context."""
    w, h = 100, 70
    sc_f, cam_f, light_f = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    sc_t, cam_t, light_t = g19.Octree.builtin(abi.SCENE_HEIGHTFIELD_ROOM, n=40, w=w, h=h)
    rt = g19.RayTracer(cam_f, light_f)
    rt.tune("overlap_frames", 1)
    rt.start()
    for _ in range(2):
        for sc, cam, light in ((sc_f, cam_f, light_f), (sc_t, cam_t, light_t)):
            rt.camera, rt.light = cam, light
            rt.setScene(sc)
            before, _ = _uniform(rt, abi, w, h, 8, 5, 1)
            again, _ = _uniform(rt, abi, w, h, 8, 5, 1)
            a = rt.run_adaptive(w, h, 0.05, 2, 16, 5, 1)
            after, _ = _uniform(rt, abi, w, h, 8, 5, 1)
            assert before["radiance"].tobytes() == again["radiance"].tobytes() == after["radiance"].tobytes()
            assert before["rgb"].tobytes() == after["rgb"].tobytes()
            assert a["spp"].min() >= 2


def test_errors(g19, abi):
    import ctypes as C
    L = g19.lib()
    w, h = 64, 48
    sc, cam, light = g19.Octree.builtin(abi.SCENE_CORNELL, w=w, h=h)
    rt = g19.RayTracer(cam, light)
    rt.start()

    def call(p, ad, ctx=None):
        return L.g19_render_adaptive(rt.h if ctx is None else ctx, C.byref(cam), abi.d3(light),
                                     None if p is None else C.byref(p), None if ad is None else C.byref(ad), None, None, None, None)

    good = rt.params(w, h, abi.MODE_PATH, spp=8, max_depth=3)
    ad = abi.Adaptive(0.1, 2)
    assert call(good, ad) == abi.ERR_NO_SCENE
    rt.setScene(sc)
    assert call(good, ad) == abi.OK
    assert call(good, ad, ctx=C.c_void_p(0)) == abi.ERR_INVALID
    assert call(None, ad) == abi.ERR_INVALID
    assert call(good, None) == abi.ERR_INVALID
    assert call(rt.params(w, h, abi.MODE_REF, spp=8, max_depth=3), ad) == abi.ERR_INVALID
    for tau in (0.0, -1.0, float("inf"), float("nan")):
        assert call(good, abi.Adaptive(tau, 2)) == abi.ERR_INVALID, tau
    for m in (1, 0, 9):
        assert call(good, abi.Adaptive(0.1, m)) == abi.ERR_INVALID, m
    assert call(rt.params(w, h, abi.MODE_PATH, spp=8, max_depth=0), ad) == abi.ERR_INVALID
    assert call(rt.params(w, h, abi.MODE_PATH, spp=8, max_depth=65), ad) == abi.ERR_INVALID
    assert call(rt.params(w, h, abi.MODE_PATH, spp=8, max_depth=3, rank=1, world=1), ad) == abi.ERR_INVALID
    # the device form validates the same way
    assert L.g19_render_adaptive_device(rt.h, C.byref(cam), abi.d3(light), C.byref(good), C.byref(abi.Adaptive(0.0, 2)),
                                        None, None, None, None, None) == abi.ERR_INVALID
    # after every refusal the context still renders
    r = rt.run_adaptive(w, h, 0.1, 2, 8, 3, 1)
    assert (r["spp"] >= 2).all()


def test_cancel_between_passes(g19, abi):
    w, h = 512, 512
    rt, _, _ = _tracer(g19, abi, "CORNELL", 0, w, h)
    t = threading.Timer(0.05, rt.stop)
    t.start()
    p = rt.params(w, h, abi.MODE_PATH, spp=4096, max_depth=5, spp_per_pass=1)
    import ctypes as C
    rc = g19.lib().g19_render_adaptive(rt.h, C.byref(rt.camera), abi.d3(rt.light), C.byref(p),
                                       C.byref(abi.Adaptive(1e-30, 2)), None, None, None, None)
    t.join()
    assert rc == abi.ERR_CANCELLED
    assert 0.0 <= rt.progress() < 1.0
    rt.start()
    r = rt.run_adaptive(64, 64, 1e30, 2, 4, 3, 1)  # the context renders again
    assert (r["spp"] == 2).all()


def test_device_form_on_side_stream(g19, abi):
    torch = pytest.importorskip("torch")
    w, h, depth = 100, 70, 5
    rt, _, _ = _tracer(g19, abi, "CORNELL_GLASS", 0, w, h)
    spp, min_spp, seed, tau = 16, 2, 4, 0.05
    host = rt.run_adaptive(w, h, tau, min_spp, spp, depth, seed)
    dev = torch.device("cuda")
    rgb = torch.zeros((h, w, 3), dtype=torch.uint8, device=dev)
    rad = torch.zeros((h, w, 3), dtype=torch.float32, device=dev)
    var = torch.zeros((h, w), dtype=torch.float32, device=dev)
    cnt = torch.zeros((h, w), dtype=torch.int32, device=dev)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        p = rt.params(w, h, abi.MODE_PATH, spp=spp, max_depth=depth, seed=seed)
        rt.run_adaptive_device(p, abi.Adaptive(tau, min_spp), rgb.data_ptr(), rad.data_ptr(), var.data_ptr(), cnt.data_ptr(),
                               side.cuda_stream)
    side.synchronize()
    assert np.array_equal(rgb.cpu().numpy(), host["rgb"])
    assert rad.cpu().numpy().tobytes() == host["radiance"].tobytes()
    assert var.cpu().numpy().tobytes() == host["variance"].tobytes()
    assert np.array_equal(cnt.cpu().numpy(), host["spp"])
    assert rt.stats().samples == int(host["spp"].astype(np.int64).sum())

"""The adaptive-sampling helpers (tests/adaptive_util.py, tests/path_moments_oracle.c) on the FP64 PATH oracle: no GPU.

What test_adaptive_gpu.py takes from them has to be right on its own: the oracle's per-pixel sample moments are the
samples g19o_path_render averages, and the numpy round rule stops a tile exactly when its error meets the target.
"""
import numpy as np

from adaptive_util import TILE, allowed_counts, path_moments, pixel_error, round_counts, tile_max, variance_of_mean
from oracle import binding
from util import mirror


def test_moment_means_equal_path_render(g19, abi, oracle):
    w, h, spp, depth, seed = 48, 40, 6, 4, 3
    sc, cam, _ = g19.Octree.builtin(abi.SCENE_CORNELL_GLASS, w=w, h=h)
    chk = mirror(oracle, sc)
    win = (5, 7, 37, 29)
    mom = path_moments(chk, cam, w, h, 0, spp, depth, seed, win)
    ref, _ = binding.path_render(chk, cam, w, h, spp, depth, seed=seed, window=win, threads=2)
    got = (mom[..., :3] / spp).astype(np.float32)
    assert np.array_equal(got, ref[win[1]:win[3], win[0]:win[2]])
    # moments are additive over sample ranges, and S2 is at least n m^2
    a = path_moments(chk, cam, w, h, 0, 2, depth, seed, win)
    b = path_moments(chk, cam, w, h, 2, spp, depth, seed, win)
    assert np.allclose(a + b, mom, rtol=1e-12, atol=1e-12)
    v, m = variance_of_mean(mom, spp)
    assert (v >= 0).all() and (mom[..., 3] >= spp * m * m * (1 - 1e-12) - 1e-12).all()


def test_round_rule_on_oracle_moments(g19, abi, oracle):
    w, h, depth, seed, min_spp, spp = 128, 72, 5, 2, 2, 16
    sc, cam, _ = g19.Octree.builtin(abi.SCENE_CORNELL_GLASS, w=w, h=h)
    chk = mirror(oracle, sc)
    cache = {0: np.zeros((h, w, 4))}

    def moments_at(n):
        if n not in cache:
            k = max(c for c in cache if c < n)
            cache[n] = moments_at(k) + path_moments(chk, cam, w, h, k, n, depth, seed)
        return cache[n]

    def E(n):
        v, m = variance_of_mean(moments_at(n), n)
        return tile_max(pixel_error(m, v))

    tau = float(np.median(E(8)))  # a target that half of the tiles meet by 8 samples
    counts = round_counts(moments_at, h, w, tau, min_spp, spp)
    print("tau %.4g, tile counts %s" % (tau, np.unique(counts, return_counts=True)))
    assert counts.shape == (-(-h // TILE), -(-w // TILE))
    assert set(np.unique(counts).tolist()) <= set(allowed_counts(min_spp, spp))
    assert len(np.unique(counts)) >= 2
    for c in np.unique(counts):
        sel = counts == c
        if c < spp:
            assert (E(c)[sel] <= tau).all()
        if c > min_spp:
            prev = max(k for k in allowed_counts(min_spp, spp) if k < c)
            assert (E(prev)[sel] > tau).all()
    # the degenerate targets
    assert (round_counts(moments_at, h, w, 1e30, min_spp, spp) == min_spp).all()
    assert (round_counts(moments_at, h, w, 1e-30, min_spp, spp) == spp).all()

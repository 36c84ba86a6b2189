"""Adaptive sampling (g19_render_adaptive) for the tests: the PATH oracle's per-pixel sample moments
(tests/path_moments_oracle.c) and the contract's error and round rule in numpy."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
TILE = 32
W_R, W_G, W_B = 0.2126, 0.7152, 0.0722
_lib = None


def _moments_lib():
    """tests/path_moments_oracle.c (oracle/path_oracle.c plus g19o_path_moments), compiled once per process into a
    temporary directory with the flags of oracle/Makefile."""
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="g19_moments_oracle_"), "libg19momentsoracle.so")
        subprocess.run(["/usr/bin/gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-pthread",
                        "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "oracle"), "-Wall", "-Wno-unused-function",
                        os.path.join(HERE, "path_moments_oracle.c"), "-o", out, "-lm"], check=True)
        lib = C.CDLL(out)
        lib.g19o_path_moments.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int] * 5 + [C.c_uint32] + [C.c_int] * 4 + [C.c_void_p]
        _lib = lib
    return _lib


def path_moments(scene, cam, w, h, s0, s1, max_depth, seed, window=None):
    """FP64 sums over samples [s0, s1) per pixel of window (x0, y0, x1, y1) (default: the frame) on an oracle
    CheckerScene -> (y1 - y0, x1 - x0, 4): sum R, sum G, sum B, sum Y^2."""
    assert scene.lib.which == "oracle"
    x0, y0, x1, y1 = window or (0, 0, w, h)
    out = np.zeros((y1 - y0, x1 - x0, 4))
    _moments_lib().g19o_path_moments(scene.h, C.byref(cam), w, h, s0, s1, max_depth, seed, x0, y0, x1, y1,
                                     out.ctypes.data_as(C.c_void_p))
    return out


def luminance(rgb):
    rgb = np.asarray(rgb, np.float64)
    return W_R * rgb[..., 0] + W_G * rgb[..., 1] + W_B * rgb[..., 2]


def variance_of_mean(mom, n):
    """v = max(S2 - n m^2, 0) / (n (n - 1)) from sums (..., 4) over n samples, in FP64."""
    m = luminance(mom[..., :3] / n)
    return np.maximum(mom[..., 3] - n * m * m, 0.0) / (n * (n - 1.0)), m


def pixel_error(m, v):
    """e = sqrt(v) / max(m, 0.05)."""
    return np.sqrt(np.asarray(v, np.float64)) / np.maximum(np.asarray(m, np.float64), 0.05)


def tile_max(a):
    """Largest value of each 32x32 tile of an (h, w) array (in-frame pixels only) -> (tiles_y, tiles_x)."""
    h, w = a.shape
    ty, tx = -(-h // TILE), -(-w // TILE)
    pad = np.full((ty * TILE, tx * TILE), -np.inf)
    pad[:h, :w] = a
    return pad.reshape(ty, TILE, tx, TILE).max(axis=(1, 3))


def tile_error(radiance, variance):
    """The tile error E of the contract recomputed from a render's radiance (m) and variance (v) outputs."""
    return tile_max(pixel_error(luminance(radiance), variance))


def per_pixel(tiles, h, w):
    """Broadcast a (tiles_y, tiles_x) array to the pixels of an (h, w) frame."""
    return np.repeat(np.repeat(tiles, TILE, axis=0), TILE, axis=1)[:h, :w]


def round_counts(moments_at, h, w, tau, min_spp, spp):
    """The round rule of the contract: round 0 gives every tile [0, min_spp); a tile whose E <= tau stops, any other with
    n samples takes [n, min(2n, spp)) next. moments_at(n) -> (h, w, 4) sums over samples [0, n). Returns the count of
    each tile (tiles_y, tiles_x)."""
    ty, tx = -(-h // TILE), -(-w // TILE)
    counts = np.zeros((ty, tx), np.int64)
    active = np.ones((ty, tx), bool)
    n = min_spp
    while active.any():
        v, m = variance_of_mean(moments_at(n), n)
        E = tile_max(pixel_error(m, v))
        counts[active] = n
        active &= (E > tau) & (n < spp)
        n = min(2 * n, spp)
    return counts


def allowed_counts(min_spp, spp):
    out, n = [], min_spp
    while n < spp:
        out.append(n)
        n *= 2
    return out + [spp]

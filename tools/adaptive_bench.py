"""Noise-targeted adaptive sampling (g19_render_adaptive) on one GPU: what it costs and what it buys.

    python tools/adaptive_bench.py [--reps 3] [--only overhead|benefit]

overhead  an adaptive render whose target no tile can meet (every tile takes spp) against g19_render at the same spp,
          alternating, on C2 (Cornell 1080p x 64 spp, depth 5), C3 (glass Cornell, depth 12) and C4 (the 1 M-triangle
          room, 256 spp): the price of the fourth accum plane, the rounds' host round trips and the tile tests. Both
          frames are byte-compared as well.
benefit   C3 at 1080p (min_spp 16, spp 1024) and C4 (min_spp 16, spp 512) at noise targets 0.05 / 0.02 / 0.01. For each:
          time, total samples, mean spp, and the 95th percentile and maximum over tiles of the tile error against a
          uniform reference at 4 x spp (per pixel |Y - Y_ref| / max(Y_ref, 0.05), the largest in the tile); the same for
          a uniform render with the same total samples (spp = the rounded mean), and the time of the uniform render that
          meets the target everywhere (spp = the largest tile count).
Times are host wall clock around the blocking call (the adaptive render synchronises once per round anyway). The card's
name and power limit are printed first, from the same process.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
g19 = importlib.import_module("2019global_b200")
abi = g19.abi

W, H = 1920, 1080
SCENES = {"c2": ("CORNELL", 0, 5), "c3": ("CORNELL_GLASS", 0, 12), "c4": ("HEIGHTFIELD_ROOM", 708, 5)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def tracer(cfg):
    which, n, depth = SCENES[cfg]
    sc, cam, light = g19.Octree.builtin(getattr(abi, "SCENE_" + which), n=n, w=W, h=H)
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()
    rt._keep = sc
    return rt, depth


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, 1e3 * (time.perf_counter() - t0)


def luminance(rgb):
    rgb = np.asarray(rgb, np.float64)
    return 0.2126 * rgb[..., 0] + 0.7152 * rgb[..., 1] + 0.0722 * rgb[..., 2]


def tile_errors(rad, ref):
    y, yr = luminance(rad), luminance(ref)
    e = np.abs(y - yr) / np.maximum(yr, 0.05)
    ty, tx = -(-H // 32), -(-W // 32)
    pad = np.full((ty * 32, tx * 32), -np.inf)
    pad[:H, :W] = e
    E = pad.reshape(ty, 32, tx, 32).max(axis=(1, 3)).ravel()
    return float(np.percentile(E, 95)), float(E.max())


def overhead(reps):
    rows = []
    for cfg, spp in (("c2", 64), ("c3", 64), ("c4", 256)):
        rt, depth = tracer(cfg)
        kw = dict(spp=spp, max_depth=depth, seed=1)
        rt.run(W, H, mode=abi.MODE_PATH, want=("radiance",), **kw)  # warm-up: modules, buffers
        rt.run_adaptive(W, H, 1e-30, 16, spp, depth, 1, want=("radiance",))
        tu, ta = [], []
        same = True
        for _ in range(reps):
            u, t = timed(lambda: rt.run(W, H, mode=abi.MODE_PATH, want=("rgb", "radiance"), **kw))
            tu.append(t)
            a, t = timed(lambda: rt.run_adaptive(W, H, 1e-30, 16, spp, depth, 1, want=("rgb", "radiance", "spp")))
            ta.append(t)
            same &= a["radiance"].tobytes() == u["radiance"].tobytes() and a["rgb"].tobytes() == u["rgb"].tobytes()
        mu, ma = statistics.median(tu), statistics.median(ta)
        row = dict(kind="overhead", config=cfg, spp=spp, uniform_ms=[round(x, 2) for x in tu], adaptive_ms=[round(x, 2) for x in ta],
                   uniform_median_ms=round(mu, 2), adaptive_median_ms=round(ma, 2), overhead_pct=round(100 * (ma / mu - 1), 2),
                   byte_equal=bool(same))
        print(json.dumps(row), flush=True)
        rows.append(row)
        del rt
    return rows


def benefit():
    rows = []
    for cfg, spp in (("c3", 1024), ("c4", 512)):
        rt, depth = tracer(cfg)
        ref, t_ref = timed(lambda: rt.run(W, H, mode=abi.MODE_PATH, want=("radiance",), spp=4 * spp, max_depth=depth, seed=99))
        ref = ref["radiance"].copy()
        print(json.dumps(dict(kind="reference", config=cfg, spp=4 * spp, ms=round(t_ref, 1))), flush=True)
        for tau in (0.05, 0.02, 0.01):
            a, ta = timed(lambda: rt.run_adaptive(W, H, tau, 16, spp, depth, 1, want=("radiance", "spp")))
            total = int(a["spp"].astype(np.int64).sum())
            mean = total / (W * H)
            u_spp = max(1, int(round(mean)))
            u, tu = timed(lambda: rt.run(W, H, mode=abi.MODE_PATH, want=("radiance",), spp=u_spp, max_depth=depth, seed=1))
            top = int(a["spp"].max())
            _, t_top = timed(lambda: rt.run(W, H, mode=abi.MODE_PATH, want=("radiance",), spp=top, max_depth=depth, seed=1))
            pa, ma = tile_errors(a["radiance"], ref)
            pu, mu = tile_errors(u["radiance"], ref)
            row = dict(kind="benefit", config=cfg, tau=tau, spp_max=spp, adaptive_ms=round(ta, 1), samples=total,
                       mean_spp=round(mean, 1), adaptive_E95=round(pa, 4), adaptive_Emax=round(ma, 4), uniform_spp=u_spp,
                       uniform_ms=round(tu, 1), uniform_E95=round(pu, 4), uniform_Emax=round(mu, 4), largest_count=top,
                       uniform_at_largest_count_ms=round(t_top, 1))
            print(json.dumps(row), flush=True)
            rows.append(row)
        del rt
    return rows


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", choices=("overhead", "benefit"), default=None)
    args = ap.parse_args()
    print("card: %s" % card(), flush=True)
    if args.only in (None, "overhead"):
        overhead(args.reps)
    if args.only in (None, "benefit"):
        benefit()


if __name__ == "__main__":
    main()

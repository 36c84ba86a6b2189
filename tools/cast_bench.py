"""Throughput of the batched ray queries (g19_cast_rays_device) on their own, outside a render.

    python tools/cast_bench.py [--min-seconds 1.0] [--out FILE]

Prints one JSON line per (scene, ray set, walk): n rays, ms per cast, Mrays/s, and node / primitive tests per ray
(from a separate G19_CAST_COUNT cast; timed casts never count). Scenes: C2, the Cornell box (flat: the staged pair
loops), and C4, HEIGHTFIELD_ROOM n = 708 with 1 002 528 triangles (tree: walks 1, 3 and 4). Ray sets, seeded on the
host: camera = the 1920x1080 corner rays; bounce = 2^24 rays leaving first-hit points (offset 1e-3 along the normal),
cosine-distributed around the normal; shadow = any-hit rays from those origins to points on the ceiling light. Each
line times at least --min-seconds of casts with CUDA events after a warm-up; rays and outputs stay on the device.
A last line gives the trace rate of one C4 render in the same process ((extend + shadow segments) / render_ms) and
the card's name and power limit (nvidia-smi, read only).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def corner_rays(cam, w, h):
    """The un-jittered rays through the pixel corners (raytracer.h:41-43), FP64."""
    cpos = np.array(cam.pos[:])
    fwd = np.array(cam.look_at[:]) - cpos
    fwd /= np.linalg.norm(fwd)
    up = np.array([0.0, 0.0, 1.0])
    left = np.cross(up, fwd)
    left /= np.linalg.norm(left)
    top_left = cam.focal * fwd + (left + up) * float(w) * 0.5 * 0.0002
    ys, xs = np.mgrid[0:h, 0:w]
    d = top_left[None, :] - left[None, :] * (xs.reshape(-1, 1) * 0.0002) - up[None, :] * (ys.reshape(-1, 1) * 0.0002)
    return np.repeat(cpos[None, :], h * w, 0), d / np.linalg.norm(d, axis=1, keepdims=True)


def bounce_rays(p, nn, n, rng):
    k = rng.integers(0, len(p), n)
    p, nn = p[k], nn[k] / np.linalg.norm(nn[k], axis=1, keepdims=True)
    a = np.where(np.abs(nn[:, :1]) > 0.9, np.array([[0.0, 1.0, 0.0]]), np.array([[1.0, 0.0, 0.0]]))
    tx = np.cross(nn, a)
    tx /= np.linalg.norm(tx, axis=1, keepdims=True)
    ty = np.cross(nn, tx)
    u1, phi = rng.random(n), 2 * np.pi * rng.random(n)
    r = np.sqrt(u1)
    d = tx * (r * np.cos(phi))[:, None] + ty * (r * np.sin(phi))[:, None] + nn * np.sqrt(1 - u1)[:, None]
    return p + 1e-3 * nn, d


def light_points(sc, g19, abi, n, rng):
    """n points on the scene's emitters (uniform over their triangles by area)."""
    tris = []
    for i in range(len(sc)):
        if sc.entity(i).bsdf == abi.BSDF_EMITTER:
            tris.append(sc.triangles(i))
    t = np.concatenate(tris).reshape(-1, 3, 3)
    area = np.linalg.norm(np.cross(t[:, 1] - t[:, 0], t[:, 2] - t[:, 0]), axis=1)
    k = rng.choice(len(t), n, p=area / area.sum())
    u, v = rng.random(n), rng.random(n)
    flip = u + v > 1
    u[flip], v[flip] = 1 - u[flip], 1 - v[flip]
    return t[k, 0] + (t[k, 1] - t[k, 0]) * u[:, None] + (t[k, 2] - t[k, 0]) * v[:, None]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--bounce", type=int, default=1 << 24)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("cast_bench.py needs a CUDA device")
    g19 = importlib.import_module("2019global_b200")
    abi = g19.abi
    dev = torch.device("cuda", 0)
    lines = []

    def emit(rec):
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    def to_dev(o, d, tmax):
        rays = np.zeros((len(o), 8), np.float32)
        rays[:, 0:3], rays[:, 3], rays[:, 4:7] = o, tmax, d
        return torch.from_numpy(rays).to(dev)

    def timed(rt, name, ray_set, rays, any_hit, walk):
        n = rays.shape[0]
        ids = torch.empty(n, dtype=torch.int32, device=dev)
        t = None if any_hit else torch.empty(n, dtype=torch.float32, device=dev)
        flags = abi.CAST_ANY_HIT if any_hit else 0
        s = torch.cuda.current_stream(dev).cuda_stream
        call = lambda f: rt.cast_device(n, rays.data_ptr(), ids.data_ptr(), 0 if t is None else t.data_ptr(), 0, f, s)
        call(flags | abi.CAST_COUNT)  # the tallies (and the warm-up of the counting kernel)
        torch.cuda.synchronize()
        st = rt.stats()
        for _ in range(2):
            call(flags)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 1
        while True:
            e0.record()
            for _ in range(reps):
                call(flags)
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            if ms >= 1000.0 * args.min_seconds:
                break
            reps = max(reps * 2, int(reps * 1000.0 * args.min_seconds / max(ms, 1e-3) * 1.1) + 1)
        hits = int((ids >= 0).sum().item())
        emit({"scene": name, "rays": ray_set, "walk": walk, "n": n, "ms": ms / reps, "Mrays_per_s": n * reps / ms / 1e3,
              "hit_fraction": hits / n, "node_tests_per_ray": st.node_tests / n, "prim_tests_per_ray": st.prim_tests / n,
              "casts_timed": reps})

    for name, which, nn, walks in (("c2", abi.SCENE_CORNELL, 0, (None,)), ("c4", abi.SCENE_HEIGHTFIELD_ROOM, 708, (1, 3, 4))):
        sc, cam, light = g19.Octree.builtin(which, n=nn, w=1920, h=1080)
        rt = g19.RayTracer(cam, light, device=0)
        rt.start()
        rng = np.random.default_rng(19)
        sets = None
        for walk in walks:
            if walk is not None:
                rt.tune("walk", walk)
            rt.setScene(sc)
            if sets is None:  # the ray sets, from this scene's first hits
                co, cd = corner_rays(cam, 1920, 1080)
                first = rt.cast(co, cd, want_normals=True)
                hit = first["ids"] >= 0
                p = co[hit] + cd[hit] * first["t"][hit, None].astype(np.float64)
                bo, bd = bounce_rays(p, first["normals"][hit].astype(np.float64), args.bounce, rng)
                lp = light_points(sc, g19, abi, args.bounce, rng)
                sd = lp - bo
                dist = np.linalg.norm(sd, axis=1)
                sets = [("camera", to_dev(co, cd, np.inf), False), ("bounce", to_dev(bo, bd, np.inf), False),
                        ("shadow", to_dev(bo, sd / dist[:, None], dist - 2e-3), True)]
            for ray_set, rays, any_hit in sets:
                timed(rt, name, ray_set, rays, any_hit, walk)
        del sets
        torch.cuda.empty_cache()
        if name == "c4":  # the render's own trace rate, same process, default walk
            rt.tune("walk", None)
            rt.setScene(sc)
            p = rt.params(1920, 1080, mode=abi.MODE_PATH, spp=256, max_depth=5, seed=1)
            rt.run_device(p)  # warm-up
            torch.cuda.synchronize()
            rt.run_device(p)
            torch.cuda.synchronize()
            st = rt.stats()
            emit({"scene": "c4", "render": "1920x1080 x 256 spp, depth 5", "extend_segments": st.extend_segments,
                  "shadow_segments": st.shadow_segments, "render_ms": st.render_ms,
                  "Msegments_per_s": (st.extend_segments + st.shadow_segments) / st.render_ms / 1e3})
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    emit({"gpu": q.stdout.strip()})
    if args.out:
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()

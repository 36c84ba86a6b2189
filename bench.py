#!/usr/bin/env python
"""bench.py -- Msamples/s of the per-pixel radiance loop (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Timed workload (config.workload), default c2 = BASELINE.json configs[1]: procedural Cornell box (diffuse walls +
2 spheres, one area light), 1920x1080, 64 spp, max depth 5, G19_MODE_PATH. One "step" = one whole frame =
132 710 400 camera paths. Strong scaling: the frame's 32x32 tiles are interleaved over the ranks (no data-path
collective); every rank's resolve kernel stores its pixels straight into rank 0's frame over NVLink, and that
gather is inside every timed step.

  value    whole-job Msamples/s, outputs resident in HBM on rank 0 (device timed, CUDA events, max over ranks)
  e2e      same metric through the host-buffer C-ABI call g19_render (N=1) / render + gather + D2H into pinned
           host memory (N>1): the reference-facing RayTracer::run equivalent
  parity   correctness of THE TIMED PATH, checked after the timed region at every N: four windows of the frame
           against the FP64 CPU oracle at the same seed (relRMSE <= 1e-2 each), and at N > 1 the sha256 of the
           N-rank radiance frame against a 1-rank render of the same frame on rank 0. A failure exits non-zero.
  roofline dominant kernel class, algorithmic bytes (DESIGN.md section 5) / CUDA-event time
  other_configs  BASELINE.json configs[2..4] AT THEIR STATED SIZE, measured after the timed region (one warm-up at
           reduced spp, then whole frames timed with CUDA events): C3 glass Cornell 1080p x 64 spp depth 12, C4 the
           1 002 528-triangle heightfield room 1080p x 256 spp, C5 Cornell 3840x2160 x 1024 spp depth 8 -- each with
           ms/frame, Msamples/s, segments/sample, roofline fraction and window parity. At N > 1: C5 (the 4K curve).
  cpu_baseline   this repo's FP64 path oracle (same work per sample) on all host cores, on a bounded crop of the
           same frame; `literal_reference` = the unmodified reference (oracle/_ref) on the depth-0, 1-spp slice
           it is able to execute
  config   the WORKLOAD only (same keys and values in both arms + the L2 statement); `engine` = how this arm runs it
  clocks   nvidia-smi on rank 0's GPU, sampled from the warm-up on; a timed region shorter than 1 s (8 GPUs: 40 ms)
           is followed by 1 s of the same steps so that the sampler sees the load, and `window` says which samples count

--impl reference times the CPU implementation (see reference_arm()); it never loads the product library.

--dump-outputs DIR writes the frame the last timed step delivered to rank 0 -- DIR/radiance.npy (h,w,3) and DIR/rgb.npy
(h,w,3, the RGB888 bytes), both float32 -- so that two builds can be compared output for output: the inputs depend
only on the arguments (builtin scene, SEED). A frame larger than DUMP_MAX_BYTES (C5) is cut to DUMP_PIXELS pixels
drawn with a fixed seed, whose row-major indices go to DIR/pixel_index.npy (float64). The copy into host buffers
allocated before the warm-up (under 1 ms for C2) and a barrier sit between the timed steps and the 1 s of the same
steps a short timed region is followed by, so `clocks` may differ slightly from a run without the flag; the timed
value does not include them.
"""
import argparse
import hashlib
import importlib
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 0
METRIC, UNIT = "Msamples/s", "Msamples/s"
# enum g19_builtin_scene (include/g19.h)
SCENE_CORNELL, SCENE_CORNELL_GLASS, SCENE_HEIGHTFIELD_ROOM = 1, 2, 4
CONFIGS = {
    "c2": dict(scene=SCENE_CORNELL, n=0, w=1920, h=1080, spp=64, depth=5,
               workload="cornell_box_1920x1080_64spp_depth5 (BASELINE.json configs[1])"),
    "c3": dict(scene=SCENE_CORNELL_GLASS, n=0, w=1920, h=1080, spp=64, depth=12,
               workload="cornell_box_mirror_glass_1920x1080_64spp_depth12 (BASELINE.json configs[2])"),
    "c4": dict(scene=SCENE_HEIGHTFIELD_ROOM, n=708, w=1920, h=1080, spp=256, depth=5,
               workload="heightfield_room_1002528_triangles_1920x1080_256spp_depth5 (BASELINE.json configs[3])"),
    "c5": dict(scene=SCENE_CORNELL, n=0, w=3840, h=2160, spp=1024, depth=8,
               workload="cornell_box_3840x2160_1024spp_depth8 (BASELINE.json configs[4])"),
}
PARITY_TOL = 1e-2       # same-seed relRMSE per window (SURVEY.md 8(c))
WINDOW = (64, 36)       # parity window size in pixels
WINDOW_AT = ((0.5, 0.5), (0.3, 0.74), (0.68, 0.74), (0.08, 0.1))  # centres (fraction of w, h): middle, both spheres, a corner
DUMP_MAX_BYTES = 64 * 10 ** 6  # --dump-outputs: a 1080p frame (49.8 MB as float32) is written whole
DUMP_PIXELS = 1 << 20          # pixels kept of a larger frame (33.6 MB with their indices)
DUMP_SEED = 0


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")] + [time.time()])
        except Exception:
            pass

    def stop(self, t0=None, t1=None, label="timed"):
        """Summary of the samples taken in [t0, t1] (wall clock: the timed region). The sampler starts before the warm-up
        steps -- nvidia-smi needs ~0.1 s to come up and an 8-GPU timed region is 40 ms -- so when no sample falls inside
        the region the ones taken under the same load around it are used, and `window` says so."""
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        rows, window = self.rows, "warmup+timed"
        if t0 is not None:
            inside = [r for r in self.rows if t0 <= r[-1] <= t1]
            if inside:
                rows, window = inside, label
            else:
                near = [r for r in self.rows if t0 - 1.0 <= r[-1] <= t1 + 0.25]
                if near:
                    rows = near
        sm = sorted(float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        self.window = window
        for r in rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ---- CPU side: the oracle as checker / CPU baseline (never the product library) -----------------------------
_checker_cache = {}


def checker_scene(cfg):
    """(oracle scene, camera, light) of a config, generated by oracle/oracle_scenes.c."""
    key = (cfg["scene"], cfg["n"], cfg["w"], cfg["h"])
    if key not in _checker_cache:
        from oracle import binding
        _checker_cache.clear()  # one big scene at a time
        _checker_cache[key] = binding.CheckerLib("oracle").builtin(cfg["scene"], cfg["n"], cfg["w"], cfg["h"])
    return _checker_cache[key]


def cpu_path_oracle(cfg, threads, budget_s=12.0):
    """The like-for-like CPU path tracer (oracle/path_oracle.c, FP64) on a centred crop of the SAME frame at the
    SAME spp/depth; the crop grows until the run takes a few seconds. Returns (Msamples/s, description)."""
    from oracle import binding
    chk, cam, _ = checker_scene(cfg)
    W, H, spp, depth = cfg["w"], cfg["h"], cfg["spp"], cfg["depth"]
    cw, ch = max(16, W // 20), max(9, H // 20)
    scale = max(1, spp // 64)  # heavier configs start from a smaller crop
    cw, ch = max(16, cw // scale), max(9, ch // scale)
    while True:
        x0, y0 = (W - cw) // 2, (H - ch) // 2
        t = time.perf_counter()
        binding.path_render(chk, cam, W, H, spp, depth, seed=SEED, window=(x0, y0, x0 + cw, y0 + ch), threads=threads)
        dt = time.perf_counter() - t
        if dt >= budget_s / 4 or (cw, ch) == (W, H):
            break
        cw, ch = (cw * 2, ch * 2) if cw * 2 <= W * 4 // 5 else (W, H)
    n = cw * ch * spp
    return n / dt / 1e6, "centred %dx%d crop of the %dx%d frame, %d spp, depth %d (%d paths, %.1f s)" % (
        cw, ch, W, H, spp, depth, n, dt)


def cpu_literal_reference(cfg, threads):
    """The UNMODIFIED reference (oracle/_ref) on what it can execute: 1 primary ray per pixel, direct shading, on
    rows of the same scene. Returns dict or None."""
    from oracle import binding
    if not binding.available("ref") or cfg["n"] > 100:
        return None
    ref = binding.CheckerLib("ref")
    descs, cam, light = binding.builtin_descs(cfg["scene"], cfg["n"], cfg["w"], cfg["h"])
    chk = ref.scene((-20.0,) * 3, (20.0,) * 3, descs)
    W, H = cfg["w"], cfg["h"]
    rows = 8 * max(1, threads)
    y0 = (H - rows) // 2
    t = time.perf_counter()
    chk.trace(cam, light, W, H, y0=y0, y1=y0 + rows, want=("ids",), threads=threads)
    dt = time.perf_counter() - t
    return {"value": rows * W / dt / 1e6, "unit": UNIT, "cores": threads,
            "sample": "%d rows of the frame, depth-0 samples (1 primary ray + direct shade): all the reference can "
                      "execute" % rows}


def reference_arm(args):
    """bench.py --impl reference. The reference's CPU implementation of the path on the box's host cores. The
    compiled reference (oracle/_ref) cannot run this workload -- it has no spp, bounces or area light
    (raytracer.h:32-86) -- so the arm times this repo's CPU port of the SAME path-traced workload (kind "port", all
    host threads) and reports the literal reference's depth-0 rate beside it. The scene comes from
    oracle/oracle_scenes.c: the product library is never loaded."""
    if env_int("RANK", 0) != 0:
        return 0
    cfg = CONFIGS[args.config]
    threads = os.cpu_count() or 1
    vals, sample = [], ""
    for i in range(args.warmup + args.steps):
        v, sample = cpu_path_oracle(cfg, threads, budget_s=8.0 if args.steps > 1 else 16.0)
        if i >= args.warmup:
            vals.append(v)
    value = sum(vals) / len(vals)
    samples_per_step = cfg["w"] * cfg["h"] * cfg["spp"]
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * samples_per_step / (value * 1e6),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "width": cfg["w"], "height": cfg["h"], "spp": cfg["spp"],
                       "max_depth": cfg["depth"], "seed": SEED, "mode": "PATH"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "literal_reference": cpu_literal_reference(cfg, threads),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "ms_per_step is extrapolated from the bounded crop to the full frame"}
    print(json.dumps(line))
    return 0


def rel_rmse(a, b):
    import numpy as np
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return math.sqrt(float(np.mean((a - b) ** 2))) / max(float(np.mean(b)), 1e-12)


def window_parity(cfg, frame_rad, threads):
    """relRMSE of WINDOW-sized windows of the rendered frame (h,w,3 float32, host) against the oracle, same seed."""
    from oracle import binding
    chk, cam, _ = checker_scene(cfg)
    W, H = cfg["w"], cfg["h"]
    out = []
    for fx, fy in WINDOW_AT:
        x0 = min(max(0, int(fx * W) - WINDOW[0] // 2), W - WINDOW[0])
        y0 = min(max(0, int(fy * H) - WINDOW[1] // 2), H - WINDOW[1])
        x1, y1 = x0 + WINDOW[0], y0 + WINDOW[1]
        exp, _ = binding.path_render(chk, cam, W, H, cfg["spp"], cfg["depth"], seed=SEED, window=(x0, y0, x1, y1), threads=threads)
        out.append({"window": [x0, y0, x1, y1], "relrmse": rel_rmse(frame_rad[y0:y1, x0:x1], exp[y0:y1, x0:x1]),
                    "oracle_mean": float(exp[y0:y1, x0:x1].mean())})
    worst = max(o["relrmse"] for o in out)
    return {"windows": out, "windows_relrmse_max": worst, "tolerance": PARITY_TOL, "seed": SEED,
            "oracle": "oracle/path_oracle.c (FP64, same Philox stream), %d windows of %dx%d px at full spp/depth" % (
                len(out), WINDOW[0], WINDOW[1]), "ok": bool(worst <= PARITY_TOL and all(o["oracle_mean"] > 0 for o in out))}


def dump_outputs(out_dir, rad, rgb):
    """--dump-outputs: the frame (radiance (h,w,3) float32, rgb (h,w,3) uint8) as DIR/<name>.npy in float32, cut to a
    seeded sample of DUMP_PIXELS pixels (plus their indices) when the whole frame would exceed DUMP_MAX_BYTES."""
    import numpy as np
    h, w, _ = rad.shape
    arrays = {"radiance": rad, "rgb": rgb}
    if 2 * rad.size * 4 > DUMP_MAX_BYTES:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(h * w, DUMP_PIXELS, replace=False))
        arrays = {k: a.reshape(h * w, 3)[idx] for k, a in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


# ---------------------------------------------------------------------------------------------
class Job:
    """One config on this rank's GPU: scene upload, shared frame (or NCCL gather buffers), the step."""

    def __init__(self, mods, cfg, rank, world, local, gather, spp_per_pass, rt=None):
        g19, torch, dist, g19dist = mods
        self.mods, self.cfg, self.rank, self.world, self.local = mods, cfg, rank, world, local
        self.abi = g19.abi
        W, H = cfg["w"], cfg["h"]
        sc, cam, light = g19.Octree.builtin(cfg["scene"], n=cfg["n"], w=W, h=H)
        if rt is None:
            rt = g19.RayTracer(cam, light, device=local)
        rt.camera, rt.light = cam, tuple(light)
        t0 = time.perf_counter()
        rt.setScene(sc)
        self.upload_s = time.perf_counter() - t0
        rt.start()
        self.rt, self.scene = rt, sc
        self.spp_per_pass = spp_per_pass
        self.stream = torch.cuda.current_stream().cuda_stream
        dev = torch.device("cuda", local)
        self.dev = dev
        self.host_rgb = torch.empty(H * W * 3, dtype=torch.uint8).pin_memory() if rank == 0 else None
        self.host_rad = None
        self.shared = g19dist.shared_frame(rt, W, H) if gather == "frame" else None
        if self.shared is None:
            # one payload per rank = its compact tile arrays [float radiance | RGB888], padded to rank 0's length
            pad = g19dist.padded_len(W, H, world)
            self.rad_bytes = pad * 3 * 4
            self.payload = torch.zeros(self.rad_bytes + pad * 3, dtype=torch.uint8, device=dev)
            self.f_rad = torch.zeros(H * W * 3, dtype=torch.float32, device=dev) if rank == 0 else None
            self.f_rgb = torch.zeros(H * W * 3, dtype=torch.uint8, device=dev) if rank == 0 else None

    def params(self, profile=0, spp=None, rank=None, world=None):
        c = self.cfg
        return self.rt.params(c["w"], c["h"], mode=self.abi.MODE_PATH, spp=spp or c["spp"], max_depth=c["depth"], seed=SEED,
                              rank=self.rank if rank is None else rank, world=self.world if world is None else world,
                              spp_per_pass=self.spp_per_pass, profile=profile)

    def step(self, profile=0, read_host=False, read_rad=False, spp=None):
        g19, torch, dist, g19dist = self.mods
        c, rt, stream = self.cfg, self.rt, self.stream
        if read_rad and self.rank == 0 and self.host_rad is None:
            self.host_rad = torch.empty(c["h"] * c["w"] * 3, dtype=torch.float32).pin_memory()
        if self.shared is not None:
            # fused: resolve stores into rank 0's frame (peer mapping), then a system-scope signal; rank 0 enqueues a
            # wait -- no collective, no staging copy, no host round trip
            self.shared.render(self.params(profile, spp), stream=stream)
            if self.rank == 0:
                self.shared.wait(self.world, stream=stream)
                if read_host or read_rad:
                    self.shared.read(rgb=self.host_rgb.data_ptr() if read_host else 0,
                                     rad=self.host_rad.data_ptr() if read_rad else 0, stream=stream)
                self.shared.release(stream=stream)
            return
        rt.render_tiles(self.params(profile, spp), t_rad=self.payload.data_ptr(), t_rgb=self.payload.data_ptr() + self.rad_bytes,
                        stream=stream)

        def untile_both(r, buf, _frame):
            rt.untile(c["w"], c["h"], r, self.world, t_rad=buf.data_ptr(), t_rgb=buf.data_ptr() + self.rad_bytes,
                      d_rad=self.f_rad.data_ptr(), d_rgb=self.f_rgb.data_ptr(), stream=stream)
        g19dist.gather_frame(self.payload, c["w"], c["h"], 3, self.f_rgb, untile_both)
        if self.rank == 0:
            if read_host:
                self.host_rgb.copy_(self.f_rgb, non_blocking=True)
            if read_rad:
                self.host_rad.copy_(self.f_rad, non_blocking=True)

    def frame_buffers(self):
        """Pinned host buffers for read_frame."""
        torch = self.mods[1]
        c = self.cfg
        return (torch.empty(c["h"] * c["w"] * 3, dtype=torch.float32).pin_memory(),
                torch.empty(c["h"] * c["w"] * 3, dtype=torch.uint8).pin_memory())

    def read_frame(self, rad, rgb):
        """Rank 0, after the last step has completed: (radiance (h,w,3) float32, rgb (h,w,3) uint8) copied into the
        frame_buffers() rad, rgb."""
        torch = self.mods[1]
        c = self.cfg
        if self.shared is not None:
            self.shared.read(rgb=rgb.data_ptr(), rad=rad.data_ptr(), stream=self.stream)
        else:
            rad.copy_(self.f_rad, non_blocking=True)
            rgb.copy_(self.f_rgb, non_blocking=True)
        torch.cuda.synchronize()
        return rad.numpy().reshape(c["h"], c["w"], 3), rgb.numpy().reshape(c["h"], c["w"], 3)

    def check_frame(self):
        """Raises if a device-side wait of the shared frame gave up (G19_ERR_TIMEOUT)."""
        if self.shared is not None:
            self.shared.check(stream=self.stream)

    def close(self):
        if self.shared is not None:
            self.shared.close()
            self.shared = None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="the timed workload (default c2 = BASELINE.json configs[1])")
    ap.add_argument("--spp-per-pass", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-others", action="store_true", help="skip the other_configs block")
    ap.add_argument("--gather", default="frame", choices=["frame", "nccl"],
                    help="frame: every rank's resolve kernel stores its pixels straight into rank 0's frame over "
                         "NVLink (fused gather, no collective); nccl: compact tile arrays + torch.distributed.gather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the frames of --impl ours")
    if args.impl == "reference":
        return reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    g19 = importlib.import_module("2019global_b200")
    g19dist = importlib.import_module("2019global_b200.dist")
    abi = g19.abi
    world, rank, local = env_int("WORLD_SIZE", 1), env_int("RANK", 0), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: lib2019global_b200 has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    mods = (g19, torch, dist, g19dist)
    threads = os.cpu_count() or 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def all_ok(flag):
        return sum_over_ranks(0.0 if flag else 1.0) == 0.0

    def parity_of(job):
        """Window parity of the frame the timed path produces (all ranks render, rank 0 checks) and, at N > 1,
        bit-identity of the N-rank radiance frame with a 1-rank render on rank 0."""
        cfg = job.cfg
        job.step(read_rad=True)
        barrier()
        job.check_frame()
        out = None
        if rank == 0:
            frame = job.host_rad.numpy().reshape(cfg["h"], cfg["w"], 3)
            out = window_parity(cfg, frame, threads)
            if world > 1:
                alone = job.rt.run(cfg["w"], cfg["h"], mode=abi.MODE_PATH, want=("radiance",), spp=cfg["spp"],
                                   max_depth=cfg["depth"], seed=SEED, spp_per_pass=job.spp_per_pass)["radiance"]
                same = hashlib.sha256(alone.tobytes()).hexdigest() == hashlib.sha256(frame.tobytes()).hexdigest()
                out["nrank_bit_identical"] = bool(same)
                out["ok"] = bool(out["ok"] and same)
            else:
                out["nrank_bit_identical"] = None
        barrier()
        return out

    def class_profile(job, steps):
        """Per-kernel-class CUDA-event times and counters (event brackets on, one pass in flight)."""
        cls_ms = [0.0] * 8
        agg = {"extend": 0, "shadow": 0, "shade": 0, "shade_first": 0, "shade_folded": 0, "lit": 0, "rad_stores": 0, "samples": 0,
               "node_tests": 0, "prim_tests": 0, "launch": [0] * 8}
        for _ in range(steps):
            job.step(profile=1)
            torch.cuda.synchronize()
            s = job.rt.stats()
            for k in range(8):
                cls_ms[k] += s.class_ms[k]
                agg["launch"][k] += s.class_launches[k]
            agg["extend"] += s.extend_segments
            agg["shadow"] += s.shadow_segments
            agg["shade"] += s.shade_calls
            agg["shade_first"] += s.shade_calls_first
            agg["shade_folded"] += s.shade_calls_folded
            agg["lit"] += s.lit_samples
            agg["rad_stores"] += s.radiance_stores
            agg["samples"] += s.samples
            agg["node_tests"] += s.node_tests
            agg["prim_tests"] += s.prim_tests
        return cls_ms, agg

    def roofline_of(job, cls_ms, agg, steps, ms_step, clocks):
        """HBM roofline of the dominant kernel class from the algorithmic byte model (DESIGN.md section 5) for flat
        scenes; issue roofline (SURVEY.md 8(d) T_issue) for tree scenes."""
        cfg = job.cfg
        E, S0, C, C0, ST = agg["extend"], agg["samples"], agg["shade"], agg["shade_first"], agg["rad_stores"]
        npix_local = g19.engine.tile_pixels(cfg["w"], cfg["h"], rank, world)
        flat = cfg["n"] == 0
        if flat:
            # diffuse-only scenes trace the camera segment inside the first bounce's launch (no raygen kernel): the 48-byte
            # camera records are neither written nor read
            cam_rec = 0 if agg["launch"][abi.K_EXTEND] == 0 else 48 * C0
            CR = C - C0 - agg["shade_folded"]  # vertices that travel as records (a path's last vertex is shaded where it is found)
            bytes_cls = {
                "raygen_extend": cam_rec,                       # record written per shaded camera hit
                "bounce": (cam_rec + 64 * CR                    # record read per shaded vertex
                           + 64 * CR                            # record written per continuation hit (= vertices shaded later)
                           + 16 * ST),                          # radiance delivered once per path that ends in this kernel
                "accumulate": 16 * S0 + 24 * npix_local * max(1, agg["launch"][abi.K_ACCUM]),
            }
        else:
            # tree scenes: slot-indexed state (hp/dw/tp 16 B each), ray records 48 B written + read, radiance planes
            bytes_cls = {
                "raygen_extend": 32 * C0 + 4 * C0,
                "bounce": 48 * C + 32 * (E - S0) + 96 * (E - S0 + agg["shadow"]) + 24 * agg["lit"] + 20 * (E - S0),
                "accumulate": 12 * S0 + 24 * npix_local * max(1, agg["launch"][abi.K_ACCUM]),
            }
        ms_cls = {"raygen_extend": cls_ms[abi.K_EXTEND], "bounce": cls_ms[abi.K_SHADE], "accumulate": cls_ms[abi.K_ACCUM]}
        top = max(ms_cls, key=lambda k: ms_cls[k])
        peak, peak_src = measured_peak()
        n_launch = {"raygen_extend": agg["launch"][abi.K_EXTEND], "bounce": agg["launch"][abi.K_SHADE],
                    "accumulate": agg["launch"][abi.K_ACCUM]}
        achieved = bytes_cls[top] / (ms_cls[top] * 1e-3) / 1e9 if ms_cls[top] > 0 else 0.0
        props = torch.cuda.get_device_properties(local)
        sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        traffic, issue_pct, issue = None, None, None
        if flat and cfg is CONFIGS["c2"]:
            try:
                with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                    tj = json.load(f)
                    traffic = tj.get(top)
                    issue_pct = tj.get("issue_active_pct", {}).get(top)
                    # warp instructions per launch (ncu, same pass size as this run's) over the live launch time,
                    # against SMs x 4 schedulers x SM clock
                    winst = tj.get("warp_inst_per_launch", {}).get(top)
                    if winst and ms_cls[top] > 0:
                        peak_i = props.multi_processor_count * 4 * sm_hz
                        ach_i = winst / (ms_cls[top] / max(1, n_launch[top]) * 1e-3)
                        issue = {"warp_inst_per_launch": winst, "achieved_Ginst_s": ach_i / 1e9, "peak_Ginst_s": peak_i / 1e9,
                                 "frac": ach_i / peak_i, "source": "profiles/roofline_traffic.json (ncu smsp__inst_executed.sum)"}
            except Exception:
                pass
        total_bytes = sum(bytes_cls.values())
        roof = {
            "bound": "hbm", "kernel": top + "_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
            "bytes_per_launch": bytes_cls[top] / max(1, n_launch[top]),
            "avg_launch_ms": ms_cls[top] / max(1, n_launch[top]),
            "share_of_step": ms_cls[top] / max(1e-9, sum(cls_ms)),
            "issue": issue,
            "note": "per-class times and shares are CUDA-event brackets taken with ONE pass in flight (params.profile); the "
                    "timed steps behind `value` keep up to four passes in flight on four streams, so ms_per_step < the sum "
                    "of the classes",
            "per_class": {k: {"ms_per_step": ms_cls[k] / steps, "launches_per_step": n_launch[k] / steps,
                              "algorithmic_GB_per_step": bytes_cls[k] / steps / 1e9,
                              "GBps": (bytes_cls[k] / (ms_cls[k] * 1e-3) / 1e9) if ms_cls[k] > 0 else None}
                          for k in ms_cls},
            "whole_step": {"algorithmic_GB": total_bytes / steps / 1e9, "bytes_per_segment": total_bytes / max(1, E + agg["shadow"]),
                           "segments_per_sample": (E + agg["shadow"]) / max(1, S0),
                           "GBps_over_step": world * total_bytes / steps / (ms_step * 1e-3) / 1e9,
                           "frac_of_peak_per_gpu": total_bytes / steps / (ms_step * 1e-3) / 1e9 / peak},
        }
        if flat:
            roof["binding_resource"] = "issue slots (ncu: smsp__issue_active %s%% of peak) -- see DESIGN.md section 5" % issue_pct
            if agg["launch"][abi.K_EXTEND] == 0:
                roof["note_fused"] = ("the camera segment is traced inside the first bounce's launch and a path's last vertex is shaded "
                                      "by the launch that finds it: their vertex records are no longer written and read back, so the "
                                      "algorithmic bytes per frame fell by 40 % while the frame got 11 % faster -- the HBM fraction of "
                                      "this issue-bound kernel fell with them (0.57 -> ~0.4), the issue fraction did not")
        if not flat and agg["node_tests"] > 0:
            # SURVEY.md 8(d): T_issue = (N_node*20 + N_tri*50 + S*150) thread instructions / (SMs * 128 lanes * f_sm);
            # N_node / N_tri counted by the walk itself (params.profile builds of the tree kernels), S = all segments
            S = E + agg["shadow"]
            inst = (agg["node_tests"] * 20 + agg["prim_tests"] * 50 + S * 150) / steps
            t_issue_ms = inst / (props.multi_processor_count * 128 * sm_hz) * 1e3
            roof.update({"bound": "issue", "kernel": "trace_kernel + raygen_extend_kernel (tree walk)", "unit": "Gthread-inst/s",
                         "achieved": inst / (ms_step * 1e-3) / 1e9, "peak": props.multi_processor_count * 128 * sm_hz / 1e9,
                         "frac": t_issue_ms / ms_step, "t_issue_ms": t_issue_ms,
                         "node_tests_per_step": agg["node_tests"] / steps, "prim_tests_per_step": agg["prim_tests"] / steps,
                         "model": "SURVEY.md 8(d): 20 thread instructions per node test, 50 per primitive test, 150 per segment",
                         "hbm_view": {"achieved": achieved, "peak": peak, "frac": achieved / peak, "kernel": top + "_kernel"}})
        return roof

    # ================= the timed workload =======================================================
    cfg = CONFIGS[args.config]
    W, H, SPP, DEPTH = cfg["w"], cfg["h"], cfg["spp"], cfg["depth"]
    samples_per_step = W * H * SPP
    job = Job(mods, cfg, rank, world, local, args.gather, args.spp_per_pass)
    rt = job.rt
    dump_bufs = job.frame_buffers() if args.dump_outputs and rank == 0 else None
    sampler = ClockSampler(local)
    if rank == 0:  # rank 0's GPU is the one reported (eight nvidia-smi processes starting at once take seconds to come up)
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        job.step()
    # ---- timed region: K steps, device clock, barrier + synchronize on both sides -------------
    barrier()
    wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        job.step()
    e1.record()
    barrier()
    wall1 = time.time()
    ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    frame_out = None
    if args.dump_outputs:
        if rank == 0:
            frame_out = job.read_frame(*dump_bufs)
        barrier()  # no rank renders the next frame into rank 0's until its copy has landed
    short = ms * args.steps < 1000.0
    if short:  # a short timed region (N = 8: 40 ms): keep the same load up until the sampler has seen it
        for _ in range(int(math.ceil(1000.0 / max(ms, 1e-3)))):  # the same count on every rank (ms is the max over ranks)
            job.step()
        barrier()
    clocks = (sampler.stop(wall0, wall1 + (1.0 if short else 0.0), "timed + 1 s of the same steps after it" if short else "timed")
              if rank == 0 else {})
    job.check_frame()
    st = rt.stats()
    # this library's kernels inside the timed region: every rank's render + rank 0's wait/release (frame) or its
    # untile per payload (nccl)
    launches = (sum_over_ranks(float(st.kernel_launches)) + (2 if job.shared is not None else world)) * args.steps
    value = samples_per_step / (ms * 1e-3) / 1e6

    barrier()
    cls_ms, agg = class_profile(job, args.steps)
    barrier()
    roofline = roofline_of(job, cls_ms, agg, args.steps, ms, clocks)
    total_bytes_step = roofline["whole_step"]["algorithmic_GB"]

    # ---- e2e: the reference-facing call with HOST buffers ---------------------------------------
    cam_bytes = 7 * 8 + 3 * 8 + 11 * 4  # g19_camera + light + g19_params
    if world == 1:
        host_np = job.host_rgb.numpy().reshape(H, W, 3)

        def e2e_step():
            rt.run(W, H, mode=abi.MODE_PATH, want=("rgb",), out={"rgb": host_np}, spp=SPP, max_depth=DEPTH, seed=SEED,
                   spp_per_pass=args.spp_per_pass)
    else:
        def e2e_step():
            job.step(read_host=True)
            torch.cuda.synchronize()
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / args.steps
    job.check_frame()
    e2e = {"value": samples_per_step / (e2e_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": cam_bytes, "d2h_bytes_per_step": W * H * 3,
           "api": "g19_render (host RGB888 out)" if world == 1 else (
               "g19_render_to_frame on every rank (peer stores into rank 0's frame over NVLink) + g19_frame_wait + "
               "g19_frame_read into pinned host memory on rank 0" if job.shared is not None else
               "g19_render_tiles_device + NCCL gather + D2H on rank 0")}

    # ---- parity of the timed path ------------------------------------------------------------------
    parity = parity_of(job)
    gather_desc = ("shared frame: resolve kernels store into rank 0's HBM over NVLink, no collective"
                   if job.shared is not None else "nccl gather of compact tile arrays")
    timeouts = job.shared.timeouts() if (job.shared is not None and rank == 0) else 0
    job.close()

    # ---- BASELINE configs 3..5 at their stated size --------------------------------------------------
    others = []
    if not args.no_others and args.config == "c2":
        names = ["c3", "c4", "c5"] if world == 1 else ["c5"]
        for name in names:
            oc = CONFIGS[name]
            oj = Job(mods, oc, rank, world, local, args.gather, args.spp_per_pass, rt=rt)
            oj.step(spp=min(oc["spp"], 32))  # warm-up: every lane allocates its full-size pass buffers (a pass is <= 8 spp), kernel attributes
            barrier()
            n_frames = 3 if name == "c3" else 1
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(n_frames):
                oj.step()
            a1.record()
            barrier()
            oms = max_over_ranks(a0.elapsed_time(a1)) / n_frames
            oj.check_frame()
            ocls, oagg = class_profile(oj, 1)
            barrier()
            oroof = roofline_of(oj, ocls, oagg, 1, oms, clocks)
            opar = parity_of(oj)
            segs = sum_over_ranks(float(oagg["extend"] + oagg["shadow"]))
            if rank == 0:
                n_samp = oc["w"] * oc["h"] * oc["spp"]
                others.append({"config": name, "workload": oc["workload"], "width": oc["w"], "height": oc["h"], "spp": oc["spp"],
                               "max_depth": oc["depth"], "frames_timed": n_frames, "ms_per_frame": oms,
                               "value": n_samp / (oms * 1e-3) / 1e6, "unit": UNIT, "segments_per_sample": segs / n_samp,
                               "scene_upload_s": oj.upload_s,
                               "roofline": {k: oroof.get(k) for k in ("bound", "kernel", "achieved", "peak", "unit", "frac",
                                                                        "t_issue_ms", "hbm_view")},
                               "roofline_frac": oroof["frac"], "parity": opar})
            oj.close()

    rc = 0
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            v, sample = cpu_path_oracle(cfg, threads)
            cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                   "literal_reference": cpu_literal_reference(cfg, threads)}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            # the WORKLOAD (the same keys and values as the reference arm's line, plus the L2 statement the timing rules ask for)
            "config": {"workload": cfg["workload"], "width": W, "height": H, "spp": SPP, "max_depth": DEPTH, "seed": SEED,
                       "mode": "PATH",
                       "l2": "per-step wavefront state streams (%.1f GB algorithmic) far exceed the 126 MB L2; "
                             "no flush needed" % (world * total_bytes_step)},
            # how THIS arm runs it
            "engine": {"tiles": "32x32 interleaved, rank = tile % world", "gather": gather_desc, "frame_time_ms": ms},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "parity": parity, "roofline": roofline,
            "cpu_baseline": cpu, "other_configs": others,
        }
        if frame_out is not None:
            dump_outputs(args.dump_outputs, *frame_out)
        print(json.dumps(line))
        bad = [("timed config " + args.config, parity)] + [(o["config"], o["parity"]) for o in others]
        for name, p in bad:
            if not p or not p.get("ok"):
                sys.stderr.write("bench.py: PARITY FAILURE on %s: %s\n" % (name, json.dumps(p)))
                rc = 1
        if timeouts:
            sys.stderr.write("bench.py: %d device-side frame spins timed out\n" % timeouts)
            rc = 1
    if world > 1:
        rc = 0 if all_ok(rc == 0) else 1
        dist.barrier()
        dist.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main())

"""bench.py --impl reference (the CPU arm) prints ONE JSON line with the contract's keys. Runs the CPU
path oracle on a bounded crop, no GPU needed. The GPU arm's line is checked on the GPU box (-m gpu)."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMMON = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
          "dtype", "data", "config", "e2e", "cpu_baseline")


def _line(args, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _line(["--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert d["impl"] == "reference"
    for k in COMMON:
        assert k in d, k
    assert d["metric"] == "Msamples/s" and d["unit"] == "Msamples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_never_loads_the_product_library():
    """The arm's scene comes from oracle/oracle_scenes.c; the timed call is the oracle's. The product .so must not
    even be mapped into the process (the driver records which .so files each arm loaded)."""
    code = ("import sys, runpy; sys.argv = ['bench.py', '--impl', 'reference', '--steps', '1', '--warmup', '0']\n"
            "try:\n    runpy.run_path(%r, run_name='__main__')\nexcept SystemExit:\n    pass\n"
            "maps = open('/proc/self/maps').read()\n"
            "assert 'libg19oracle.so' in maps\n"
            "assert 'lib2019global_b200.so' not in maps, 'product library loaded by the reference arm'\n"
            "print('CLEAN')\n") % os.path.join(ROOT, "bench.py")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "CLEAN" in r.stdout, r.stdout[-500:] + r.stderr[-2000:]


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_outputs_whole_frame_and_seeded_sample(tmp_path):
    """A 1080p frame is written whole; a 4K one (C5) as the same seeded pixel sample on every run, under 64 MB."""
    bench = _bench_module()
    rng = np.random.default_rng(3)
    rad = rng.random((1080, 1920, 3), dtype=np.float32)
    rgb = rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    bench.dump_outputs(str(tmp_path / "hd"), rad, rgb)
    assert sorted(os.listdir(tmp_path / "hd")) == ["radiance.npy", "rgb.npy"]
    got_rad, got_rgb = np.load(tmp_path / "hd" / "radiance.npy"), np.load(tmp_path / "hd" / "rgb.npy")
    assert got_rad.dtype == got_rgb.dtype == np.float32
    assert np.array_equal(got_rad, rad) and np.array_equal(got_rgb, rgb.astype(np.float32))
    rad = rng.random((2160, 3840, 3), dtype=np.float32)
    rgb = rng.integers(0, 256, (2160, 3840, 3), dtype=np.uint8)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), rad, rgb)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["pixel_index.npy", "radiance.npy", "rgb.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    idx = np.load(tmp_path / "a" / "pixel_index.npy")
    assert idx.dtype == np.float64 and len(np.unique(idx)) == idx.size == bench.DUMP_PIXELS
    px = idx.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "radiance.npy"), rad.reshape(-1, 3)[px])
    assert np.array_equal(np.load(tmp_path / "a" / "rgb.npy"), rgb.reshape(-1, 3)[px].astype(np.float32))


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_rejected_arguments(args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and r.stdout == "", r.stderr


def test_reference_arm_other_ranks_print_nothing():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                       text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1"))
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_gpu_arm_line(tmp_path):
    d = _line(["--steps", "2", "--warmup", "3", "--no-cpu", "--no-others", "--dump-outputs", str(tmp_path)])
    for k in COMMON + ("gpu_launches", "clocks", "roofline", "parity", "other_configs"):
        assert k in d, k
    # the timed path's own correctness, checked inside bench.py after the timed region
    par = d["parity"]
    assert par["ok"] is True and par["windows_relrmse_max"] <= par["tolerance"] == 1e-2 and len(par["windows"]) >= 4
    assert d["metric"] == "Msamples/s" and d["n_gpus"] == 1 and d["gpu_launches"] > 0 and d["value"] > 100
    assert d["e2e"]["d2h_bytes_per_step"] == 1920 * 1080 * 3 and d["e2e"]["value"] > 100
    ro = d["roofline"]
    assert ro["bound"] in ("hbm", "tensor") and 0 < ro["frac"] < 1.5 and ro["unit"] == "GB/s" and ro["peak"] > 1000
    # --dump-outputs: the timed path's last frame, whole at 1080p, within the parity tolerance of the CPU oracle
    assert sorted(os.listdir(tmp_path)) == ["radiance.npy", "rgb.npy"]
    rad, rgb = np.load(tmp_path / "radiance.npy"), np.load(tmp_path / "rgb.npy")
    assert rad.dtype == rgb.dtype == np.float32 and rad.shape == rgb.shape == (1080, 1920, 3)
    assert np.isfinite(rad).all() and rad.mean() > 0
    assert np.array_equal(rgb, np.round(rgb)) and rgb.min() >= 0 and rgb.max() <= 255 and rgb.max() > 0
    bench = _bench_module()
    assert bench.window_parity(bench.CONFIGS["c2"], rad, os.cpu_count() or 1)["ok"]

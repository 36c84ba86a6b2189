"""The interface-compatible C++ headers (include/*.h) driven the way main.cpp + viewer.h drive the
reference: tools/g19_headless.cpp builds the default scene with the reference's own constructor
calls, copies the RayTracer by value, start(), run(500,500) on a worker thread, writes a PPM."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tools", "bin", "g19_headless")
# a checkout of preon7/2019global, optional: the same variable and default oracle/Makefile builds oracle/_ref from
REFERENCE = os.environ.get("G19_REFERENCE") or os.path.join(os.path.dirname(ROOT), "2019global")
C1_SHA = "9ab0129419a4c328d4ea865adf74b66e3c91d10c6190cc34373fa2b0187bba85"


def _ppm(path):
    raw = open(path, "rb").read()
    parts = raw.split(b"\n", 3)
    assert parts[0] == b"P6"
    w, h = map(int, parts[1].split())
    return np.frombuffer(parts[3], np.uint8).reshape(h, w, 3)


def test_headers_compile_against_shim_and_glm():
    """No GPU needed: the headers build with the built-in vector shim and, when the reference is
    named by G19_REFERENCE, against its vendored GLM (what a real drop-in build uses)."""
    if not os.path.exists(os.path.join(ROOT, "2019global_b200", "lib2019global_b200.so")):
        pytest.skip("library not built")
    base = ["g++", "-std=c++14", "-fsyntax-only", "-DG19_NO_QT", "-I", os.path.join(ROOT, "include"),
            os.path.join(ROOT, "tools", "g19_headless.cpp")]
    subprocess.run(base, check=True)
    glm = os.path.join(REFERENCE, "3rd_party")
    if os.path.isdir(glm):
        subprocess.run(base + ["-I", glm], check=True)


@pytest.mark.gpu
def test_headless_driver_reproduces_config1(tmp_path):
    if not os.path.exists(BIN):
        pytest.skip("tools/bin/g19_headless not built (run __graft_entry__.build())")
    out = str(tmp_path / "c1.ppm")
    r = subprocess.run([BIN, out], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    img = _ppm(out)
    assert img.shape == (500, 500, 3)
    # config-1 golden (SURVEY.md section 4): the contract allows <= 1 LSB with <= 0.1 % of shaded pixels exempt
    # (SURVEY 8(c)); on B200 with this toolchain the image is byte-exact, and that is what is asserted
    assert hashlib.sha256(img.tobytes()).hexdigest() == C1_SHA, r.stdout
    # every pixel the reference shades is non-black here (ambient term 0.1 * texture > 0), every miss is black
    assert int((img.reshape(-1, 3).max(1) > 0).sum()) == 14702 + 20806 + 17674
    assert "ImpSphere::intersect -> 1" in r.stdout and "candidates 3" in r.stdout
    import importlib
    g19 = importlib.import_module("2019global_b200")
    sc, cam, light = g19.Octree.builtin(g19.abi.SCENE_DEFAULT)
    rt = g19.RayTracer(cam, light)
    rt.setScene(sc)
    rt.start()
    assert np.array_equal(rt.run(500, 500)["rgb"], img)  # same bytes as the Python front end
    # ... and the same bytes as the CPU oracle (itself byte-equal to the compiled reference, test_oracle_ref.py)
    from oracle import binding
    from util import mirror
    exp = mirror(binding.CheckerLib("oracle"), sc).trace(cam, light, 500, 500, want=("rgb",), threads=8)["rgb"]
    assert np.array_equal(exp, img)


@pytest.mark.gpu
def test_headless_driver_path_mode(tmp_path):
    if not os.path.exists(BIN):
        pytest.skip("tools/bin/g19_headless not built")
    out = str(tmp_path / "p.ppm")
    r = subprocess.run([BIN, out, "96", "64", "--path", "4", "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert _ppm(out).shape == (64, 96, 3)
    # progressive refreshes into the live Image (viewer.h:18-21) + "Save as... PNG" (gui.h:39-45)
    png = str(tmp_path / "p.png")
    r = subprocess.run([BIN, png, "640", "360", "--path", "256", "4", "--refresh", "0"], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    n = int(r.stdout.split(" progressive refreshes")[0].split()[-1])
    assert n >= 3, r.stdout
    assert open(png, "rb").read(8) == b"\x89PNG\r\n\x1a\n"


def test_reference_main_cpp_helpers_compile_against_these_headers(tmp_path):
    """Drop-in check without Qt: the four helper functions of the reference's own main.cpp (insert_tris,
    entity_test, matrix_test, bbox_test -- reference main.cpp:63-133, everything below main()) are compiled, text
    unchanged, against include/*.h + the reference's vendored GLM; the scene literal (main.cpp:24-57) is compiled
    the same way with the Gui lines dropped. A signature or public member that drifted away from the reference's
    classes fails here. Only runs where G19_REFERENCE names a checkout of the reference."""
    main_cpp = os.path.join(REFERENCE, "main.cpp")
    if not os.path.exists(main_cpp):
        pytest.skip("no checkout of the reference (G19_REFERENCE, default ../2019global)")
    lines = open(main_cpp).read().split("\n")
    helpers = "\n".join(lines[62:133])                       # main.cpp:63-133
    literal = "\n".join(l for l in lines[23:57] if "Gui" not in l and "window" not in l)  # main.cpp:24-57
    src = tmp_path / "ref_main_helpers.cpp"
    src.write_text('#include <iostream>\n#include <vector>\n#include "camera.h"\n#include "raytracer.h"\n#include "ray.h"\n'
                   '#include "entities.h"\n#include "octree.h"\n#include "glm/ext.hpp"\n'
                   "void entity_test();\nvoid bbox_test();\nvoid matrix_test();\nvoid insert_tris(Octree& scene);\n"
                   "void scene_literal() {\n" + literal + "\n}\n" + helpers + "\n")
    cmd = ["g++", "-std=c++14", "-fsyntax-only", "-DG19_NO_QT", "-I", os.path.join(ROOT, "include"), "-I",
           os.path.join(REFERENCE, "3rd_party"), str(src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]

"""The C++ drop-in layer (TileRenderer / RayTracer / intersect* over the C ABI):
compiles against the re-authored headers and — when a checkout of the reference is found
(oracle.harness.reference_dir) — against the reference's own headers (CPU); on a GPU the reference's TileRenderer tests,
re-expressed in tests/cpp/dropin_test.cpp, run through it and its frame is compared with the oracle."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
CORE = ROOT / "minecraftskin_raytracer_b200" / "csrc" / "core"
LIBDIR = ROOT / "minecraftskin_raytracer_b200" / "_lib"


def _compile(sources, out, include_dirs, link=True):
    cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-Werror"] + [f"-I{d}" for d in include_dirs]
    if link:
        cmd += [str(s) for s in sources] + ["-o", str(out), f"-L{LIBDIR}", "-lmcskin_cuda", f"-Wl,-rpath,{LIBDIR}"]
    else:
        cmd += ["-fsyntax-only"] + [str(s) for s in sources]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return out


def test_dropin_layer_compiles_against_own_headers(mclib, tmp_path):
    _compile([CORE / "tile_renderer.cpp", CORE / "raytracer_api.cpp", ROOT / "tools" / "mcskin_bench.cpp"],
             tmp_path / "mcskin_bench", [ROOT / "include", ROOT / "include" / "mcskin"])
    r = subprocess.run([str(tmp_path / "mcskin_bench"), "--width", "32", "--height", "32", "--frames", "1"],
                       capture_output=True, text=True)
    if mclib.device_count() == 0:   # no CPU fallback: the CLI reports the missing device and fails
        assert r.returncode == 1 and "no CUDA device" in r.stderr
    else:
        assert r.returncode == 0, r.stderr


def test_dropin_layer_compiles_against_reference_headers():
    from oracle.harness import reference_dir
    ref = reference_dir()
    if ref is None:
        pytest.skip("no checkout of the reference (MCSKIN_REFERENCE_DIR, or `reference` beside this repository)")
    _compile([CORE / "tile_renderer.cpp", CORE / "raytracer_api.cpp"], None, [ROOT / "include", ref / "src"], link=False)


@pytest.mark.gpu
def test_reference_tile_renderer_tests_through_dropin(gpu, oracle, tmp_path):
    exe = _compile([ROOT / "tests" / "cpp" / "dropin_test.cpp", CORE / "tile_renderer.cpp", CORE / "raytracer_api.cpp"],
                   tmp_path / "dropin_test", [ROOT / "include", ROOT / "include" / "mcskin"])
    dump = tmp_path / "frame.bin"
    r = subprocess.run([str(exe), str(dump)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = dump.read_bytes()
    atlas = np.frombuffer(raw[:64 * 64 * 4], dtype=np.uint8).reshape(64, 64, 4)
    frame = np.frombuffer(raw[64 * 64 * 4:], dtype=np.float32).reshape(64, 80, 4)
    from tests.conftest import pixel_report
    from tests.scenes import make_config
    scene = gpu.build_skin_scene(atlas, "walking")
    want = oracle.render(scene, make_config(width=80, height=64, samples_per_pixel=2, max_bounces=2))
    rep = pixel_report(frame, want, oracle.quantize)
    assert rep["within1"] >= 0.999, rep
    same_as_python_api, _, _ = gpu.render(scene, make_config(width=80, height=64, samples_per_pixel=2, max_bounces=2))
    assert np.array_equal(frame.view(np.uint32), same_as_python_api.view(np.uint32))

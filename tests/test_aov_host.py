"""AOV planes on the CPU side (no GPU): the oracle's planes are pinned, agree with the unmodified reference where the
reference has a view of them (one sample per pixel, no lens), and the C header's McAovTargets matches its Python mirror."""
import ctypes as C
import json
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from minecraftskin_raytracer_b200 import _abi
from tests.aov_oracle import render_aovs
from tests.golden.make_aov_pins import PATH as PINS, PLANES
from tests.golden.make_oracle_pins import digest
from tests.scenes import RENDER_CASES, make_config, synth_skin

ROOT = Path(__file__).resolve().parent.parent


def _case_scene(case):
    from minecraftskin_raytracer_b200.lib import build_skin_scene
    _, seed, kind, pose, _ = case
    return build_skin_scene(synth_skin(seed, kind), pose)


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("case", RENDER_CASES, ids=[c[0] for c in RENDER_CASES])
def test_oracle_aov_planes_equal_pins(oracle, case, rng_mode):
    name, *_, over = case
    scene = _case_scene(case)
    cfg = make_config(**over, rng_mode=rng_mode)
    planes = render_aovs(scene, cfg)
    want = json.loads(PINS.read_text())[f"{name}/rng{rng_mode}"]
    assert {p: digest(planes[p]) for p in PLANES} == want
    # an uncovered pixel (no sample hits) is, in the colour oracle's frame, the pure gradient: the empty scene's pixel
    img = oracle.render(scene, cfg)
    empty = scene.__class__(light_pos=scene.light_pos, cam_pos=scene.cam_pos, cam_target=scene.cam_target,
                            cam_up=scene.cam_up, cam_fov_deg=scene.cam_fov_deg, background=scene.background)
    background = (img.view(np.uint32) == oracle.render(empty, cfg).view(np.uint32)).all(axis=-1)
    assert (background | (planes["tri_id"] >= 0)).all()
    # the three planes agree on which pixels are covered
    covered = planes["tri_id"] >= 0
    assert np.array_equal(covered, planes["coverage"] > 0) and np.array_equal(covered, planes["depth"] > 0)


SPP1_PINHOLE = [c for c in RENDER_CASES if c[4].get("samples_per_pixel", 1) == 1 and not c[4].get("dof_enabled")]


@pytest.mark.parametrize("case", SPP1_PINHOLE, ids=[c[0] for c in SPP1_PINHOLE])
def test_oracle_aov_planes_equal_reference_at_one_sample(oracle, reference, case):
    """At one sample per pixel without a lens the sample ray is the pixel-centre pinhole ray: tri_id is the reference's
    own hit id (Reference.aov) and depth the t of its intersectScene on that ray."""
    scene = _case_scene(case)
    cfg = make_config(**case[4])
    planes = render_aovs(scene, cfg)
    assert np.array_equal(planes["tri_id"], reference.aov(scene, cfg))
    assert np.array_equal(planes["tri_id"], oracle.aov(scene, cfg))
    h, w = cfg.height, cfg.width
    py, px = np.mgrid[0:h, 0:w]
    uv = np.stack([(px.astype(np.float32) + np.float32(0.5)) / np.float32(w),
                   (py.astype(np.float32) + np.float32(0.5)) / np.float32(h)], axis=-1).reshape(-1, 2)
    rays = reference.generate_rays(scene, np.float32(w) / np.float32(h), uv)
    hits = reference.intersect(scene, rays)
    t = np.where(hits["hit"] == 1, hits["t"], np.float32(0.0)).astype(np.float32).reshape(h, w)
    assert np.array_equal(planes["depth"].view(np.uint32), t.view(np.uint32))
    assert np.array_equal(planes["coverage"], (hits["hit"] == 1).reshape(h, w).astype(np.float32))


def test_aov_targets_struct_matches_header(tmp_path):
    """sizeof and member offsets of McAovTargets as a C compiler lays out include/mcskin_cuda.h."""
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "sizes.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "mcskin_cuda.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu\\n", sizeof(McAovTargets), offsetof(McAovTargets, coverage),'
                   ' offsetof(McAovTargets, depth), offsetof(McAovTargets, tri_id)); return 0; }\n')
    exe = tmp_path / "sizes"
    subprocess.run([cc, "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    M = _abi.McAovTargets
    assert got == [C.sizeof(M), M.coverage.offset, M.depth.offset, M.tri_id.offset]

"""The guide planes (normal, albedo; McAovTargets in include/mcskin_cuda.h) on the CPU side (no GPU): the oracle's
planes are pinned, agree with the unmodified reference at one sample per pixel without a lens, agree with the other
planes on which pixels are covered, and the header's grown McAovTargets matches its Python mirror."""
import ctypes as C
import json
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from minecraftskin_raytracer_b200 import _abi
from tests.aov_oracle import render_aovs as render_three_planes
from tests.guide_oracle import render_aovs
from tests.golden.make_guide_pins import PATH as PINS, PLANES
from tests.golden.make_oracle_pins import digest
from tests.scenes import RENDER_CASES, make_config, synth_skin

ROOT = Path(__file__).resolve().parent.parent


def _case_scene(case):
    from minecraftskin_raytracer_b200.lib import build_skin_scene
    _, seed, kind, pose, _ = case
    return build_skin_scene(synth_skin(seed, kind), pose)


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("case", RENDER_CASES, ids=[c[0] for c in RENDER_CASES])
def test_oracle_guide_planes_equal_pins(case, rng_mode):
    name, *_, over = case
    scene = _case_scene(case)
    cfg = make_config(**over, rng_mode=rng_mode)
    planes = render_aovs(scene, cfg, guides=True)
    want = json.loads(PINS.read_text())[f"{name}/rng{rng_mode}"]
    assert {p: digest(planes[p]) for p in PLANES} == want
    # the other three planes are the AOV oracle's, with or without the guides
    plain = render_three_planes(scene, cfg)
    assert set(render_aovs(scene, cfg)) == {"coverage", "depth", "tri_id"}
    for p in ("coverage", "depth", "tri_id"):
        assert np.array_equal(planes[p], plain[p]), p
    # skins have no negative alpha, and a hit never has alpha 0: albedo's alpha is > 0 exactly where a sample hit
    covered = planes["tri_id"] >= 0
    assert np.array_equal(covered, planes["albedo"][..., 3] > 0)
    assert (planes["normal"][~covered] == 0).all() and (planes["albedo"][~covered] == 0).all()
    assert (np.abs(planes["normal"][covered]).sum(axis=-1) > 0).all()


SPP1_PINHOLE = [c for c in RENDER_CASES if c[4].get("samples_per_pixel", 1) == 1 and not c[4].get("dof_enabled")]


@pytest.mark.parametrize("case", SPP1_PINHOLE, ids=[c[0] for c in SPP1_PINHOLE])
def test_oracle_guide_planes_equal_reference_at_one_sample(oracle, reference, case):
    """At one sample per pixel without a lens the sample ray is the pixel-centre pinhole ray: normal and albedo are
    McHit.normal and McHit.tex_color of intersectScene on that ray, in the reference and in the oracle, folded as the
    planes fold one hit: 0.0f + value (a -0 component reads +0), divided by 1."""
    scene = _case_scene(case)
    cfg = make_config(**case[4])
    planes = render_aovs(scene, cfg, guides=True)
    h, w = cfg.height, cfg.width
    py, px = np.mgrid[0:h, 0:w]
    uv = np.stack([(px.astype(np.float32) + np.float32(0.5)) / np.float32(w),
                   (py.astype(np.float32) + np.float32(0.5)) / np.float32(h)], axis=-1).reshape(-1, 2)
    rays = reference.generate_rays(scene, np.float32(w) / np.float32(h), uv)
    for checker in (reference, oracle):
        hits = checker.intersect(scene, rays)
        hit = (hits["hit"] == 1)[:, None]
        fold = lambda v: np.where(hit, (np.float32(0.0) + v) / np.float32(1.0), np.float32(0.0)).astype(np.float32)  # noqa: E731
        normal = fold(hits["normal"]).reshape(h, w, 3)
        albedo = fold(hits["tex_color"]).reshape(h, w, 4)
        assert np.array_equal(planes["normal"].view(np.uint32), normal.view(np.uint32))
        assert np.array_equal(planes["albedo"].view(np.uint32), albedo.view(np.uint32))


def test_aov_targets_grown_struct_matches_header(tmp_path):
    """sizeof and every member offset of McAovTargets, guide planes included, as a C compiler lays out the header."""
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    members = ("coverage", "depth", "tri_id", "normal", "albedo")
    src = tmp_path / "sizes.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "mcskin_cuda.h"\n'
                   'int main(void) { printf("%zu %d' + ' %zu' * len(members) + '\\n", sizeof(McAovTargets), MCSKIN_ABI_VERSION'
                   + "".join(f", offsetof(McAovTargets, {m})" for m in members) + '); return 0; }\n')
    exe = tmp_path / "sizes"
    subprocess.run([cc, "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    M = _abi.McAovTargets
    assert got == [C.sizeof(M), _abi.ABI_VERSION] + [getattr(M, m).offset for m in members]

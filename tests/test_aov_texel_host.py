"""The texel plane (McAovTargets::texel in include/mcskin_cuda.h) on the CPU side (no GPU): the oracle's plane is pinned,
its other five planes are the guide oracle's, every texel lies in the window of the face tri_id names and has that hit's
colour, the reference agrees at one sample per pixel, lib.skin_texel_atlas maps every pool texel of a skin to its atlas
pixel, and the grown McAovTargets matches its Python mirror."""
import ctypes as C
import json
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

from minecraftskin_raytracer_b200 import _abi
from minecraftskin_raytracer_b200.scene import synth_skin
from tests.golden.make_oracle_pins import digest
from tests.golden.make_texel_pins import PATH as PINS, free_texel_scenes
from tests.guide_oracle import render_aovs as render_five_planes
from tests.scenes import RENDER_CASES, make_config
from tests.texel_oracle import render_aovs

ROOT = Path(__file__).resolve().parent.parent
FIVE = ("coverage", "depth", "tri_id", "normal", "albedo")
FREE = free_texel_scenes()


def _case_scene(case):
    from minecraftskin_raytracer_b200.lib import build_skin_scene
    _, seed, kind, pose, _ = case
    return build_skin_scene(synth_skin(seed, kind), pose)


def _bits(a):
    return a.view(np.uint32) if a.dtype == np.float32 else a


def _check_texels_in_face_windows(scene, planes):
    """texel >= 0 exactly where tri_id >= 0, and each texel lies in the window of face (tri_id % 12) / 2 of box
    tri_id // 12, or is the sentinel of that face's texture kind.  Returns the sentinels seen."""
    tri, tex = planes["tri_id"], planes["texel"]
    assert np.array_equal(tex >= 0, tri >= 0)
    assert (tex[tri < 0] == -1).all()
    n = len(scene.texels)
    t, k = tri[tri >= 0], tex[tri >= 0]
    off, w, h = np.moveaxis(scene.boxes["face"][t // 12, (t % 12) // 2], -1, 0)
    magenta, blank = off < 0, (off >= 0) & ((w <= 0) | (h <= 0))
    window = ~magenta & ~blank
    assert (k[magenta] == n).all() and (k[blank] == n + 1).all()
    assert ((off[window] <= k[window]) & (k[window] < off[window] + w[window] * h[window])).all()
    seen = {"magenta"} if magenta.any() else set()
    if blank.any():
        seen.add("blank")
    return seen


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("case", RENDER_CASES, ids=[c[0] for c in RENDER_CASES])
def test_oracle_texel_plane_equals_pins(case, rng_mode):
    name, *_, over = case
    scene = _case_scene(case)
    cfg = make_config(**over, rng_mode=rng_mode)
    planes = render_aovs(scene, cfg)
    assert digest(planes["texel"]) == json.loads(PINS.read_text())[f"{name}/rng{rng_mode}"]
    five = render_five_planes(scene, cfg, guides=True)
    for p in FIVE:
        assert np.array_equal(_bits(planes[p]), _bits(five[p])), p
    _check_texels_in_face_windows(scene, planes)


def test_oracle_texel_plane_free_scenes():
    """Scenes with magenta and blank faces, posed boxes, nested and outer boxes and up to 212 boxes: pinned, the other
    five planes are the guide oracle's, and between them the scenes show both sentinels."""
    pins = json.loads(PINS.read_text())
    seen = set()
    for name, scene, cfg in FREE:
        planes = render_aovs(scene, cfg)
        assert digest(planes["texel"]) == pins[f"free/{name}"], name
        five = render_five_planes(scene, cfg, guides=True)
        for p in FIVE:
            assert np.array_equal(_bits(planes[p]), _bits(five[p])), (name, p)
        seen |= _check_texels_in_face_windows(scene, planes)
    assert seen == {"magenta", "blank"}


def test_pins_cover_every_case_and_nothing_else():
    want = {f"{c[0]}/rng{m}" for c in RENDER_CASES for m in (0, 1)} | {f"free/{n}" for n, _, _ in FREE}
    assert set(json.loads(PINS.read_text())) == want


def _pool(scene):
    """The scene's texels with the two synthetic texels the product appends (magenta, then (0, 0, 0, 1))."""
    return np.concatenate([scene.texels.astype(np.float32), np.float32([[1, 0, 1, 1], [0, 0, 0, 1]])])


SPP1_PINHOLE = [c for c in RENDER_CASES if c[4].get("samples_per_pixel", 1) == 1 and not c[4].get("dof_enabled")]


@pytest.mark.parametrize("case", SPP1_PINHOLE, ids=[c[0] for c in SPP1_PINHOLE])
def test_texel_colour_is_albedo_at_one_sample(case):
    """At one sample per pixel the albedo plane is (0.0f + tex_color) / 1.0f of the one hit: the texel's colour."""
    scene = _case_scene(case)
    planes = render_aovs(scene, make_config(**case[4]))
    hit = planes["texel"] >= 0
    colour = _pool(scene)[planes["texel"][hit]]
    assert np.array_equal(((np.float32(0) + colour) / np.float32(1)).view(np.uint32), planes["albedo"][hit].view(np.uint32))


@pytest.mark.parametrize("case", SPP1_PINHOLE, ids=[c[0] for c in SPP1_PINHOLE])
def test_texel_colour_equals_reference_at_one_sample(oracle, reference, case):
    """At one sample per pixel without a lens the sample ray is the pixel-centre pinhole ray: the texel's colour is
    McHit.tex_color of intersectScene on that ray, in the reference and in the oracle."""
    scene = _case_scene(case)
    cfg = make_config(**case[4])
    planes = render_aovs(scene, cfg)
    h, w = cfg.height, cfg.width
    py, px = np.mgrid[0:h, 0:w]
    uv = np.stack([(px.astype(np.float32) + np.float32(0.5)) / np.float32(w),
                   (py.astype(np.float32) + np.float32(0.5)) / np.float32(h)], axis=-1).reshape(-1, 2)
    rays = reference.generate_rays(scene, np.float32(w) / np.float32(h), uv)
    texel = planes["texel"].reshape(-1)
    for checker in (reference, oracle):
        hits = checker.intersect(scene, rays)
        hit = hits["hit"] == 1
        assert np.array_equal(hit, texel >= 0)
        assert np.array_equal(_pool(scene)[texel[hit]].view(np.uint32), hits["tex_color"][hit].view(np.uint32))


def _hollow_outer_skin(seed):
    """A 64x64 skin whose body overlay is fully transparent: that outer box is not built, and the pool after it moves."""
    atlas = synth_skin(seed)
    atlas[32:48, 16:40, 3] = 0
    return atlas


SKINS = [(kind, seed) for kind in ("64x64", "legacy", "slim") for seed in (0, 1, 2, 3)] + [("hollow_body_overlay", 5)]


@pytest.mark.parametrize("kind,seed", SKINS, ids=[f"{k}-{s}" for k, s in SKINS])
def test_skin_texel_atlas_maps_every_pool_texel(kind, seed):
    from minecraftskin_raytracer_b200 import lib
    atlas = _hollow_outer_skin(seed) if kind == "hollow_body_overlay" else synth_skin(seed, kind)
    table = lib.skin_texel_atlas(atlas)
    assert table.dtype == np.int32
    for pose in (None, "walking", "dab", "sitting"):
        scene = lib.build_skin_scene(atlas, pose)
        n = len(scene.texels)
        assert table.shape == (n + 2, 2)
        assert (table[n:] == -1).all() and (table[:n] >= 0).all()
        want = atlas[table[:n, 1], table[:n, 0]].astype(np.float32) / np.float32(255.0)
        assert np.array_equal(scene.texels.astype(np.float32).view(np.uint32), want.view(np.uint32)), pose
        # skin_layout describes the same face windows as the built scene, posed or not
        boxes, faces, _, n_texels = lib.skin_layout(atlas, pose)
        assert n_texels == n and len(boxes) == len(scene.boxes)
        windows = faces[:, [0, 3, 4]].reshape(len(boxes), 6, 3)  # (dst, w, h) = (texel_offset, width, height)
        assert np.array_equal(windows, scene.boxes["face"])
        assert np.array_equal(boxes["face"], scene.boxes["face"])
    # the table reads the -1 of an uncovered pixel as the last row: (-1, -1)
    assert (table[np.int32([-1, n, n + 1])] == -1).all()


def test_skin_texel_atlas_mirrors_legacy_limbs():
    """Legacy skins take the left limbs from the right ones, flipped: some texels come from the same atlas pixel twice,
    once mirrored."""
    from minecraftskin_raytracer_b200 import lib
    atlas = synth_skin(2, "legacy")
    _, faces, _, _ = lib.skin_layout(atlas)
    assert faces[:, 5].any() and not faces[:, 5].all()
    table = lib.skin_texel_atlas(atlas)
    mirrored = faces[faces[:, 5] == 1][0]
    dst, x, y, w = (int(v) for v in mirrored[:4])
    assert tuple(table[dst]) == (x + w - 1, y)


def test_aov_targets_six_plane_struct_matches_header(tmp_path):
    """sizeof and every member offset of McAovTargets, the texel plane included, and the ABI version, as a C compiler
    lays out the header."""
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    members = ("coverage", "depth", "tri_id", "normal", "albedo", "texel")
    src = tmp_path / "sizes.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "mcskin_cuda.h"\n'
                   'int main(void) { printf("%zu %d' + ' %zu' * len(members) + '\\n", sizeof(McAovTargets), MCSKIN_ABI_VERSION'
                   + "".join(f", offsetof(McAovTargets, {m})" for m in members) + '); return 0; }\n')
    exe = tmp_path / "sizes"
    subprocess.run([cc, "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    M = _abi.McAovTargets
    assert got == [C.sizeof(M), 4, *(getattr(M, m).offset for m in members)]
    assert _abi.ABI_VERSION == 4 and C.sizeof(M) == 6 * C.sizeof(C.c_void_p)

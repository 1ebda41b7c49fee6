"""Free scenes (tests/free_scenes.py) on the CPU: the generator is deterministic, the oracle's outputs for them equal the
pins in tests/golden/free_scene_pins.json, and each builder reaches the gate its name claims — shown from its inputs in
numpy or from the oracle's own results.  With a checkout of the reference, the oracle equals it on a subset."""
import json
from pathlib import Path

import numpy as np
import pytest

from oracle.harness import rays_array
from tests import free_scenes as fs
from tests.golden.make_free_scene_pins import scene_config_digest
from tests.golden.make_oracle_pins import digest

PINS = Path(__file__).parent / "golden" / "free_scene_pins.json"


@pytest.fixture(scope="module")
def scenes(mclib):
    return {name: (scene, cfg) for name, scene, cfg in fs.free_scenes()}


@pytest.fixture(scope="module")
def pins():
    return json.loads(PINS.read_text())


def test_generator_is_deterministic_and_pinned(scenes, pins):
    assert sorted(scenes) == sorted(pins)
    again = {name: scene_config_digest(s, c) for name, s, c in fs.free_scenes()}
    for name, (scene, cfg) in scenes.items():
        assert scene_config_digest(scene, cfg) == again[name] == pins[name]["input"], name


@pytest.mark.parametrize("name", sorted(json.loads(PINS.read_text())))
def test_oracle_frames_equal_pins(oracle, scenes, pins, name):
    scene, cfg = scenes[name]
    img, cnt = oracle.render(scene, cfg, counters=True)
    assert digest(img) == pins[name]["image"]
    assert cnt["n_intersect_scene"] == pins[name]["calls"]
    assert digest(oracle.aov(scene, cfg)) == pins[name]["tri_id"]


# ---------------------------------------------------------------- camera geometry, as prepare_frame computes it
def _basis(scene):
    pos, tgt, up = (np.float64(np.float32(v)) for v in (scene.cam_pos, scene.cam_target, scene.cam_up))
    fwd = (tgt - pos) / np.linalg.norm(tgt - pos)
    right = np.cross(fwd, up)
    return pos, fwd, right


def _corners(lo, hi):
    return np.array([[hi[0] if c & 1 else lo[0], hi[1] if c & 2 else lo[1], hi[2] if c & 4 else lo[2]] for c in range(8)],
                    dtype=np.float64)


def _depths(scene):
    pos, fwd, _ = _basis(scene)
    return np.concatenate([(_corners(b["bounds_min"], b["bounds_max"]) - pos) @ fwd for b in scene.boxes])


def test_camera_builders_reach_their_gates(scenes):
    # a box corner behind the camera (the figure's rectangle is given up)
    assert (_depths(scenes["cam_inside_figure_bounds"][0]) <= 1e-3).any()
    assert (_depths(scenes["cam_inside_outer_layer"][0]) <= 1e-3).any()
    s = scenes["cam_inside_outer_layer"][0]
    outer = [b for b in s.boxes if b["is_outer_layer"] and np.all(b["bounds_min"] < s.cam_pos) and np.all(s.cam_pos < b["bounds_max"])]
    inner = [b for b in s.boxes if not b["is_outer_layer"] and np.all(b["bounds_min"] < s.cam_pos) and np.all(s.cam_pos < b["bounds_max"])]
    assert len(outer) == 1 and not inner
    # up parallel to the view direction: no right vector
    _, _, right = _basis(scenes["cam_up_parallel"][0])
    assert np.linalg.norm(right) == 0.0
    # the close-up's figure runs past every edge of the frame
    scene, cfg = scenes["cam_closeup_clipped"]
    pos, fwd, right = _basis(scene)
    right /= np.linalg.norm(right)
    true_up = np.cross(right, fwd)
    half_h = np.tan(np.radians(scene.cam_fov_deg) / 2)
    half_w = half_h * cfg.width / cfg.height
    pts = np.concatenate([_corners(b["bounds_min"], b["bounds_max"]) for b in scene.boxes]) - pos
    assert ((pts @ fwd) > 1e-3).all()
    px = ((pts @ right) / (pts @ fwd) / half_w + 1) * 0.5 * cfg.width
    py = (1 - ((pts @ true_up) / (pts @ fwd) / half_h + 1) * 0.5) * cfg.height
    assert px.min() < 0 and px.max() > cfg.width and py.min() < 0 and py.max() > cfg.height
    assert scenes["cam_fov1"][0].cam_fov_deg == 1.0 and scenes["cam_fov170"][0].cam_fov_deg == 170.0
    assert {(scenes[n][1].width, scenes[n][1].height) for n in ("frame_300x20", "frame_20x300")} == {(300, 20), (20, 300)}


def test_light_builders(scenes):
    radii = {n: np.float32(scenes[n][0].light_radius) for n in scenes if n.startswith("light_r")}
    assert radii["light_r0"] == 0 and radii["light_r5e-5"] < np.float32(1e-4) <= radii["light_r1e-3"]
    assert radii["light_r40"] == 40.0
    boxes = scenes["light_in_inner_box"][0].boxes

    def holders(p):
        return [bool(b["is_outer_layer"]) for b in boxes if np.all(b["bounds_min"] < p) and np.all(p < b["bounds_max"])]

    assert sorted(holders(np.float32(scenes["light_in_inner_box"][0].light_pos))) == [False, True]
    assert holders(np.float32(scenes["light_between_layers"][0].light_pos)) == [True]
    lp = np.float32(scenes["light_near_face"][0].light_pos)
    assert any(abs(lp[2] - b["bounds_max"][2]) <= 0.0500001 for b in boxes)
    lp = np.float32(scenes["light_on_box_bound"][0].light_pos)
    assert any((lp == b["bounds_max"]).sum() >= 2 for b in boxes)
    assert scenes["light_below"][0].light_pos[1] < boxes["bounds_min"][:, 1].min()
    s = scenes["light_behind_camera"][0]
    _, fwd, _ = _basis(s)
    assert (np.float64(s.light_pos) - np.float64(s.cam_pos)) @ fwd < 0


def _inside(lo_i, hi_i, lo_j, hi_j):
    """host_prep.cpp's inside(i, j) in float32."""
    eps = np.float32(1e-3)
    return bool(np.all(lo_i >= lo_j + eps) and np.all(hi_i <= hi_j - eps))


def test_nesting_spares_in_float32(scenes):
    for name, want_all in (("nest_chains_exact_spare", True), ("nest_spare_minus_one_step", False)):
        b = scenes[name][0].boxes
        pairs = [(b[i + 1], b[i]) for i in range(9, 15, 2)]  # (child, parent) at exactly the spare
        got = [_inside(c["bounds_min"], c["bounds_max"], p["bounds_min"], p["bounds_max"]) for c, p in pairs]
        assert got == [want_all] * 3, name
        for c, p in pairs:  # the spare is exactly 1e-3f on the sides that pass
            assert (c["bounds_min"] == p["bounds_min"] + np.float32(1e-3)).sum() >= 2
        # three-deep chains in both scenes
        for k in range(3):
            assert _inside(b[3 * k + 2]["bounds_min"], b[3 * k + 2]["bounds_max"], b[3 * k + 1]["bounds_min"], b[3 * k + 1]["bounds_max"])
            assert _inside(b[3 * k + 1]["bounds_min"], b[3 * k + 1]["bounds_max"], b[3 * k]["bounds_min"], b[3 * k]["bounds_max"])


def test_box_builders(scenes):
    b = scenes["boxes_zero_thickness_all_ones_size"][0].boxes
    size = (b["bounds_max"] - b["bounds_min"]).astype(np.float32)
    assert (size == 0).any()
    bits = size.view(np.uint32) & 0x7FFFFF
    assert (bits == 0x7FFFFF).any() and (bits == 0).any()   # kBoxRecip off for one box, on for another
    p = scenes["posed_rotation_thresholds"][0].boxes
    rot = np.abs(np.concatenate([p["rot_x_deg"], p["rot_z_deg"]]))
    assert (rot == np.float32(0.01)).any() and (rot == np.nextafter(np.float32(0.01), np.float32(1))).any()
    assert (rot == np.float32(0.005)).any() and {90.0, 180.0} <= set(rot.tolist())
    assert (p["rot_x_deg"] == -180).any() and p["has_rotation"].all()
    for k in range(3):
        r = scenes[f"boxes_random_{k}"][0]
        sizes = (r.boxes["bounds_max"] - r.boxes["bounds_min"]).ravel()
        assert sizes.min() >= 0.0099 and sizes.max() <= 40.0 and (sizes != np.round(sizes)).all()
    pooled = [scenes[f"boxes_random_{k}"][0] for k in range(3)]
    faces = np.concatenate([s.boxes["face"].reshape(-1, 3) for s in pooled])
    assert (faces[:, 0] < 0).any() and (faces[:, 1] <= 0).any()
    assert any((s.texels[:, 3] == 0).any() for s in pooled) and any((s.boxes["n_triangles"] == 0).any() for s in pooled)
    for name, n in (("boxes_33", 33), ("boxes_64", 64)):
        boxes = scenes[name][0].boxes
        assert len(boxes) == n and (boxes["n_triangles"][32:] == 0).any() and (boxes["n_triangles"][:32] > 0).all()


def test_largest_staged_scene_fits_and_one_more_does_not():
    def blob(n):  # SceneBlobLayout(n).bytes(): lo, hi and rectangle rows padded to 4 boxes, then 144-byte DevBox records
        return 48 * ((n + 3) & ~3) + 144 * n

    assert blob(fs.MAX_STAGED_BOXES) <= 40 * 1024 < blob(fs.MAX_STAGED_BOXES + 1)
    assert len(fs.largest_scene().boxes) == fs.MAX_STAGED_BOXES and len(fs.largest_scene(1).boxes) == fs.MAX_STAGED_BOXES + 1


def _camera_hits(oracle, scene, cfg, n=64):
    u, v = np.meshgrid((np.arange(n) + 0.5) / n, (np.arange(n) + 0.5) / n)
    rays = oracle.generate_rays(scene, cfg.width / cfg.height, np.stack([u.ravel(), v.ravel()], axis=1))
    hits = oracle.intersect(scene, rays)
    return hits[hits["hit"] == 1]


def test_memo_scenes_straddle_the_window_edges(oracle, scenes):
    """traceRay's shadow seeds of the memo scenes' hits, through the seed formula and the oracle's seed_cast, fall on both
    sides of each edge of the window [-2^20, 2^23 - 2^20); the 1e5 shift wraps the cast through int64."""
    lo_edge, hi_edge = -(1 << 20), (1 << 23) - (1 << 20)
    for name, edge in (("memo_window_top", hi_edge), ("memo_window_bottom", lo_edge), ("memo_int64_wrap", None)):
        scene, cfg = scenes[name]
        p = _camera_hits(oracle, scene, cfg)["point"].astype(np.float32)
        assert len(p) > 100, name
        for depth in (0, 1):
            v = (p[:, 0] * np.float32(12345.0) + p[:, 1] * np.float32(67890.0) + p[:, 2] * np.float32(11111.0)
                 + np.float32(depth) * np.float32(99999.0)).astype(np.float32)
            seeds = np.array([oracle.seed_cast(float(x)) for x in v], dtype=np.int64)
            assert np.array_equal(seeds, v.astype(np.int64) & 0xFFFFFFFF), name
            signed = np.where(seeds >= 1 << 31, seeds - (1 << 32), seeds)
            if edge is not None:
                assert (signed < edge).any() and (signed >= edge).any(), (name, depth)
            else:
                assert (v.astype(np.float64) >= 2.0**32).all(), name    # every seed wrapped


def test_counters_show_each_route(oracle, scenes):
    def counts(name):
        return oracle.render(*scenes[name], counters=True)[1]

    assert counts("posed_rotation_thresholds")["n_rotated_hits"] > 100
    for name in ("light_r0", "light_r40", "light_in_inner_box", "boxes_64"):
        c = counts(name)
        assert c["n_soft_shadow"] > 0 and c["n_reflect_rays"] > 0, name
    for name in ("mirrors_70", "mirrors_200"):
        c = counts(name)
        hitting = c["n_primary_rays"] - c["n_background_primary"]
        assert hitting == c["n_primary_rays"] and c["n_reflect_rays"] > 64 * hitting, (name, c)   # paths deeper than 64
    assert counts("mirrors_200")["n_soft_shadow"] == 0 and counts("mirrors_70")["n_soft_shadow"] > 0


def test_hits_on_boxes_past_31(oracle, scenes):
    from tests.scenes import random_rays
    for name in ("boxes_64", "boxes_212_largest_staged"):
        scene, cfg = scenes[name]
        hits = oracle.intersect(scene, random_rays(np.random.default_rng(5), 20000))
        hit_boxes = hits["box"][hits["hit"] == 1]
        assert (hit_boxes >= 32).any(), name
        assert not np.isin(hit_boxes, np.nonzero(scene.boxes["n_triangles"] == 0)[0]).any(), name
        cam = _camera_hits(oracle, scene, cfg)
        assert (cam["box"] >= 32).any(), name


def test_frames_are_not_background_only(oracle, scenes):
    from minecraftskin_raytracer_b200.scene import FlatScene
    for name, (scene, cfg) in scenes.items():
        img = oracle.render(scene, cfg)
        empty = FlatScene(light_pos=scene.light_pos, cam_pos=scene.cam_pos, cam_target=scene.cam_target,
                          cam_up=scene.cam_up, cam_fov_deg=scene.cam_fov_deg, background=scene.background)
        differs = not np.array_equal(img.view(np.uint32), oracle.render(empty, cfg).view(np.uint32))
        assert differs, name


REFERENCE_SUBSET = ["cam_orbit_0", "cam_closeup_clipped", "cam_inside_outer_layer", "cam_up_parallel", "light_r0",
                    "light_between_layers", "boxes_random_1", "nest_spare_minus_one_step",
                    "boxes_zero_thickness_all_ones_size", "posed_rotation_thresholds", "boxes_64", "memo_int64_wrap",
                    "mirrors_70", "frame_tile1"]


@pytest.mark.parametrize("name", REFERENCE_SUBSET)
def test_oracle_equals_live_reference_on_free_scenes(oracle, reference, scenes, name):
    scene, cfg = scenes[name]
    a, calls = reference.render(scene, cfg, counters=True)
    b, cnt = oracle.render(scene, cfg, counters=True)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert calls == cnt["n_intersect_scene"]
    assert np.array_equal(reference.aov(scene, cfg), oracle.aov(scene, cfg))
    rays = rays_array(np.float32(scene.cam_pos) + np.zeros((1, 3), np.float32), np.float32([[0, 0, -1]]))
    assert np.array_equal(reference.intersect(scene, rays)["hit"], oracle.intersect(scene, rays)["hit"])

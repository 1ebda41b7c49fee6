"""The reference's own hot-path unit tests, re-expressed once and run against every
implementation of the path: the CPU oracle, the unmodified reference (oracle/_ref) and
the CUDA library.  Each case cites the gtest it restates (the reference's tests/...).

A backend offers: intersect(scene, rays, box=-1), shade(scene, cfg, hits, view_dirs, sf),
in_shadow(scene, p, n, l), trace(scene, cfg, rays, depth, use_config),
generate_rays(scene, aspect, uv), background(scene, cfg, uv, use_config),
render(scene, cfg) -> float image, generate_tiles(w, h, ts).
"""
from __future__ import annotations

import numpy as np

from minecraftskin_raytracer_b200 import _abi
from minecraftskin_raytracer_b200.scene import FlatScene, make_box
from oracle.harness import rays_array

F = np.float32


def solid_box(color, center=(0, 0, 0), size=(2, 2, 2), offset=0.0, tex=(4, 4), texel_base=0):
    w, h = tex
    texels = np.tile(np.asarray(color, dtype=F), (w * h, 1))
    half = F(size) / F(2.0) + F(offset)
    box = make_box(F(center) - half, F(center) + half, [(texel_base, w, h)] * 6, outer=offset > 0)
    return box, texels


def scene_of(*parts, **kw) -> FlatScene:
    boxes, pools, base = [], [], 0
    for color, center, size, offset in parts:
        b, t = solid_box(color, center, size, offset, texel_base=base)
        boxes.append(b)
        pools.append(t)
        base += len(t)
    return FlatScene(boxes=np.array(boxes, dtype=_abi.BOX_DTYPE) if boxes else np.zeros(0, _abi.BOX_DTYPE),
                     texels=np.concatenate(pools) if pools else np.zeros((0, 4), F), **kw)


def untextured_box_scene(center, half, **kw) -> FlatScene:
    """tests/test_shading.cpp makeBoxMesh: a box whose triangles carry texture == nullptr."""
    c = F(center)
    box = make_box(c - F(half), c + F(half), [(-1, 0, 0)] * 6)
    return FlatScene(boxes=np.array([box]), **kw)


def one_ray(o, d):
    return rays_array([o], [d])


# ------------------------------------------------------------------ test_intersection.cpp
def case_ray_hits_box_front(B):  # :20-37
    sc = scene_of(((1, 0, 0, 1), (0, 0, 0), (2, 2, 2), 0.0))
    h = B.intersect(sc, one_ray((0, 0, 5), (0, 0, -1)), box=0)[0]
    assert h["hit"] == 1
    assert abs(h["t"] - 4.0) < 1e-4 and abs(h["point"][2] - 1.0) < 1e-4 and abs(h["normal"][2] - 1.0) < 1e-4
    assert h["tex_color"][0] == 1.0 and h["tex_color"][3] == 1.0 and h["is_outer_layer"] == 0


def case_ray_misses_box(B):  # :40-50
    sc = scene_of(((0, 0, 1, 1), (0, 0, 0), (2, 2, 2), 0.0))
    assert B.intersect(sc, one_ray((0, 5, 5), (0, 0, -1)), box=0)[0]["hit"] == 0


def case_ray_hits_box_side(B):  # :53-66
    sc = scene_of(((0, 1, 0, 1), (0, 0, 0), (2, 2, 2), 0.0))
    h = B.intersect(sc, one_ray((5, 0, 0), (-1, 0, 0)), box=0)[0]
    assert h["hit"] == 1 and abs(h["t"] - 4.0) < 1e-4 and abs(h["point"][0] - 1.0) < 1e-4 and abs(h["normal"][0] - 1.0) < 1e-4


def case_transparent_pixel_is_miss(B):  # :69-79
    sc = scene_of(((0, 0, 0, 0), (0, 0, 0), (2, 2, 2), 0.0))
    assert B.intersect(sc, one_ray((0, 0, 5), (0, 0, -1)), box=0)[0]["hit"] == 0


def case_outer_flag_propagated(B):  # :81-92
    sc = scene_of(((1, 1, 1, 1), (0, 0, 0), (2, 2, 2), 0.5))
    h = B.intersect(sc, one_ray((0, 0, 5), (0, 0, -1)), box=0)[0]
    assert h["hit"] == 1 and h["is_outer_layer"] == 1


def case_ray_behind_box(B):  # :95-105
    sc = scene_of(((1, 0, 0, 1), (0, 0, 0), (2, 2, 2), 0.0))
    assert B.intersect(sc, one_ray((0, 0, 5), (0, 0, 1)), box=0)[0]["hit"] == 0


def case_scene_finds_closest(B):  # :108-129
    sc = scene_of(((1, 0, 0, 1), (0, 0, 2), (2, 2, 2), 0.0), ((0, 0, 1, 1), (0, 0, -5), (2, 2, 2), 0.0), background=(0, 0, 0, 1))
    h = B.intersect(sc, one_ray((0, 0, 10), (0, 0, -1)))[0]
    assert h["hit"] == 1 and h["tex_color"][0] == 1.0 and h["tex_color"][2] == 0.0


def case_transparent_outer_hits_inner(B):  # :132-154
    sc = scene_of(((1, 0, 0, 1), (0, 0, 0), (2, 2, 2), 0.0), ((0, 0, 0, 0), (0, 0, 0), (2, 2, 2), 0.5), background=(0, 0, 0, 1))
    h = B.intersect(sc, one_ray((0, 0, 10), (0, 0, -1)))[0]
    assert h["hit"] == 1 and h["tex_color"][0] == 1.0 and h["tex_color"][3] == 1.0 and h["is_outer_layer"] == 0


def case_empty_scene_no_hit(B):  # :157-165
    assert B.intersect(FlatScene(background=(0, 0, 0, 1)), one_ray((0, 0, 10), (0, 0, -1)))[0]["hit"] == 0


# ------------------------------------------------------------------ test_shading.cpp
def _hit(point, normal, tex):
    h = np.zeros(1, dtype=_abi.HIT_DTYPE)
    h["hit"], h["t"], h["point"], h["normal"], h["tex_color"] = 1, 1.0, point, normal, tex
    return h


def _params(**kw):
    return _abi.default_config(**kw)


def _light_scene(light, **kw):
    return FlatScene(light_pos=light, light_color=(1, 1, 1, 1), background=(0, 0, 0, 1), **kw)


PHONG = dict(kd=0.7, ks=0.3, ambient=0.1, shininess=32.0)


def case_ambient_only_light_behind(B):  # :71-86
    c = B.shade(_light_scene((0, 0, -10)), _params(**PHONG), _hit((0, 0, 0), (0, 0, 1), (1, 1, 1, 1)), [(0, 0, 1)])[0]
    assert np.allclose(c[:3], 0.1, atol=1e-4)


def case_diffuse_and_specular(B):  # :90-113
    c = B.shade(_light_scene((0, 10, 0)), _params(**PHONG), _hit((0, 0, 0), (0, 1, 0), (0.8, 0.6, 0.4, 1)), [(0, 1, 0)])[0]
    want = [min(0.1 * t + 0.7 * t + 0.3, 1.0) for t in (0.8, 0.6, 0.4)]
    assert np.allclose(c[:3], want, atol=1e-3)


def case_grazing_angle(B):  # :115-131
    c = B.shade(_light_scene((10, 0, 0)), _params(**PHONG), _hit((0, 0, 0), (0, 1, 0), (1, 1, 1, 1)), [(0, 1, 0)])[0]
    assert abs(c[0] - 0.1) < 0.05


def case_in_shadow_ambient_only(B):  # :134-150
    sc = untextured_box_scene((0, 5, 0), 2.0, light_pos=(0, 10, 0), background=(0, 0, 0, 1))
    c = B.shade(sc, _params(**PHONG), _hit((0, 0, 0), (0, 1, 0), (1, 1, 1, 1)), [(0, 1, 0)])[0]
    assert np.allclose(c[:3], 0.1, atol=1e-4)


def case_is_in_shadow_variants(B):  # :152-186
    assert B.in_shadow(_light_scene((0, 10, 0)), [(0, 0, 0)], [(0, 1, 0)], [(0, 10, 0)])[0] == 0
    blocked = untextured_box_scene((0, 5, 0), 1.0, light_pos=(0, 10, 0))
    assert B.in_shadow(blocked, [(0, 0, 0)], [(0, 1, 0)], [(0, 10, 0)])[0] == 1
    behind = untextured_box_scene((0, 20, 0), 1.0, light_pos=(0, 10, 0))
    assert B.in_shadow(behind, [(0, 0, 0)], [(0, 1, 0)], [(0, 10, 0)])[0] == 0


def case_texture_colour_and_zero_coefficients(B):  # :189-222
    sc = _light_scene((0, 10, 0))
    red = B.shade(sc, _params(), _hit((0, 0, 0), (0, 1, 0), (1, 0, 0, 1)), [(0, 1, 0)])[0]
    blue = B.shade(sc, _params(), _hit((0, 0, 0), (0, 1, 0), (0, 0, 1, 1)), [(0, 1, 0)])[0]
    assert red[0] > red[2] and blue[2] > blue[0]
    flat = B.shade(sc, _params(kd=0.0, ks=0.0, ambient=0.5), _hit((0, 0, 0), (0, 1, 0), (1, 1, 1, 1)), [(0, 1, 0)])[0]
    assert np.allclose(flat[:3], 0.5, atol=1e-4)


def case_shade_matches_formula(B):  # test_shading_props.cpp:72-146, seeded instead of RapidCheck
    rng = np.random.default_rng(5)
    sc = _light_scene((3.0, 7.0, -2.0))
    for _ in range(40):
        n = rng.normal(size=3); n /= np.linalg.norm(n)
        v = rng.normal(size=3); v /= np.linalg.norm(v)
        tex = np.append(rng.random(3), 1.0)
        p = rng.uniform(-2, 2, size=3)
        cfg = _params(kd=0.7, ks=0.3, ambient=0.1, shininess=float(rng.integers(1, 64)))
        got = B.shade(sc, cfg, _hit(p, n, tex), [v])[0]
        L = np.array(sc.light_pos) - p; L /= np.linalg.norm(L)
        ndl = max(0.0, float(n @ L))
        H = L + v
        H = H / np.linalg.norm(H) if np.linalg.norm(H) > 1e-8 else H * 0
        spec = max(0.0, float(n @ H)) ** cfg.shininess
        want = np.clip(0.1 * tex[:3] + 0.7 * ndl * tex[:3] + 0.3 * spec, 0, 1)
        assert np.allclose(got[:3], want, atol=1e-3)


# ------------------------------------------------------------------ test_raytracer.cpp
def _simple_scene(with_box=True) -> FlatScene:
    """makeSimpleScene + makeTestBox (:84-146): a 2x2x2 box at the origin sharing ONE external 2x2 texture."""
    kw = dict(background=(0.2, 0.3, 0.5, 1.0), light_pos=(10, 10, -10), light_color=(1, 1, 1, 1),
              cam_pos=(0, 0, -10), cam_target=(0, 0, 0), cam_up=(0, 1, 0), cam_fov_deg=60.0)
    if not with_box:
        return FlatScene(**kw)
    texels = np.array([(1, 0, 0, 1), (0, 1, 0, 1), (0, 0, 1, 1), (1, 1, 0, 1)], dtype=F)
    box = make_box((-1, -1, -1), (1, 1, 1), [(0, 2, 2)] * 6)
    return FlatScene(boxes=np.array([box]), texels=texels, **kw)


def case_camera_rays(B):  # :16-81
    sc = _simple_scene(False)
    r = B.generate_rays(sc, 1.0, [(0.5, 0.5), (0.1, 0.9), (0.0, 0.5), (0.5, 0.0)])
    assert np.allclose(r["dir"][0], (0, 0, 1), atol=1e-5) and np.allclose(r["origin"][0], (0, 0, -10))
    assert np.allclose(np.linalg.norm(r["dir"], axis=1), 1.0, atol=1e-5)
    wide = B.generate_rays(sc, 2.0, [(0.0, 0.5)])
    assert abs(wide["dir"][0][0]) > abs(r["dir"][2][0])     # wider aspect spreads rays in x
    assert r["dir"][3][1] > 0                                  # v = 0 is the top of the image


def case_trace_miss_and_depth(B):  # :148-172, :212-224
    cfg = _params(max_bounces=3)
    empty = _simple_scene(False)
    bg = np.array(empty.background, dtype=F)
    assert np.array_equal(B.trace(empty, cfg, one_ray((0, 0, -10), (0, 0, 1)), use_config=False)[0], bg)
    boxed = _simple_scene(True)
    assert np.array_equal(B.trace(boxed, cfg, one_ray((0, 0, -10), (0, 0, 1)), depth=5, use_config=False)[0], bg)
    assert np.array_equal(B.trace(boxed, cfg, one_ray((0, 0, -10), (0, 1, 0)), use_config=False)[0], bg)


def case_trace_hit_not_background(B):  # :174-210
    boxed = _simple_scene(True)
    bg = np.array(boxed.background[:3], dtype=F)
    for bounces in (3, 0, 5):
        c = B.trace(boxed, _params(max_bounces=bounces), one_ray((0, 0, -10), (0, 0, 1)), use_config=False)[0]
        assert np.abs(c[:3] - bg).max() > 1e-5
        assert np.all(c >= 0) and np.all(c <= 1)


def case_zero_bounce_trace_is_clamped_shade(B):  # test_raytracer_props.cpp:141-170
    boxed = _simple_scene(True)
    rng = np.random.default_rng(9)
    origins = rng.uniform(-6, 6, size=(64, 3)).astype(F)
    origins[:, 2] = -10
    targets = rng.uniform(-0.9, 0.9, size=(64, 3)).astype(F)
    d = targets - origins
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = rays_array(origins, d)
    hits = B.intersect(boxed, rays)
    keep = hits["hit"] == 1
    assert keep.sum() > 10
    cfg = _params(max_bounces=0)
    traced = B.trace(boxed, cfg, rays[keep], use_config=False)
    view = origins[keep] - hits["point"][keep]
    shaded = B.shade(boxed, cfg, hits[keep], view)
    assert np.abs(traced - np.clip(shaded, 0, 1)).max() <= 1e-4


def case_transparent_outer_never_changes_inner(B):  # test_raytracer_props.cpp:315-372
    rng = np.random.default_rng(13)
    inner_only = scene_of(((0.3, 0.7, 0.2, 1), (0, 0, 0), (2, 2, 2), 0.0))
    both = scene_of(((0.3, 0.7, 0.2, 1), (0, 0, 0), (2, 2, 2), 0.0), ((0, 0, 0, 0), (0, 0, 0), (2, 2, 2), 0.5))
    o = rng.normal(size=(200, 3)); o = (o / np.linalg.norm(o, axis=1, keepdims=True) * 8).astype(F)
    t = rng.uniform(-0.8, 0.8, size=(200, 3)).astype(F)
    d = t - o; d /= np.linalg.norm(d, axis=1, keepdims=True)
    rays = rays_array(o, d)
    a, b = B.intersect(inner_only, rays), B.intersect(both, rays)
    assert np.array_equal(a["hit"], b["hit"]) and np.array_equal(a["t"], b["t"]) and np.array_equal(a["tex_color"], b["tex_color"])


# ------------------------------------------------------------------ test_tile_renderer*.cpp
def case_generate_tiles(B):  # :9-57 and props :30-80
    t = B.generate_tiles(64, 64, 32)
    assert len(t) == 4 and all(x["width"] == 32 and x["height"] == 32 for x in t)
    t = B.generate_tiles(100, 70, 32)
    assert len(t) == 12 and tuple(t[3]) == (96, 0, 4, 32) and tuple(t[11]) == (96, 64, 4, 6)
    assert len(B.generate_tiles(10, 10, 32)) == 1 and tuple(B.generate_tiles(10, 10, 32)[0]) == (0, 0, 10, 10)
    for bad in ((0, 10, 8), (10, 0, 8), (10, 10, 0), (-1, 10, 8)):
        assert len(B.generate_tiles(*bad)) == 0
    rng = np.random.default_rng(21)
    for _ in range(25):
        w, h, ts = int(rng.integers(1, 2049)), int(rng.integers(1, 2049)), int(rng.integers(1, 257))
        tiles = B.generate_tiles(w, h, ts)
        assert int((tiles["width"].astype(np.int64) * tiles["height"]).sum()) == w * h
        assert tiles["x"].min() == 0 and tiles["y"].min() == 0
        assert (tiles["x"] + tiles["width"]).max() == w and (tiles["y"] + tiles["height"]).max() == h
        assert np.all(tiles["width"] <= ts) and np.all(tiles["height"] <= ts)


def case_render_sizes_and_empty_scene(B):  # test_tile_renderer.cpp:60-83, :106-120, :147-159
    sc = _simple_scene(False)
    for (w, h, ts) in ((32, 32, 16), (16, 16, 8), (8, 8, 8), (33, 17, 16)):
        img = B.render(sc, _params(width=w, height=h, tile_size=ts, max_bounces=0))
        assert img.shape == (h, w, 4)
        assert np.all(img[..., 3] == 1.0)


CASES = [v for k, v in sorted(globals().items()) if k.startswith("case_")]

"""GPU parity on the free scenes (tests/free_scenes.py): cameras, lights and box layouts the render cases never reach,
whole frames through the library's code paths, single queries, the seed memo, batches whose scenes differ in camera and
light, and a check under the profiler that each primary-kernel form and shading route named here really runs."""
import re

import numpy as np
import pytest

from tests import free_scenes as fs
from tests.conftest import pixel_report
from tests.scenes import make_config, random_rays, synth_skin
from tests.test_parity_gpu import RENDER_MODES, _background_pixels, _flip_budget, _render_with_options

pytestmark = pytest.mark.gpu

FRAME_MODES = ["default", "all_active", "megakernel", "megakernel_warp", "tiny_queue", "split_tiles"]


def _names():
    """The free scenes' names, from their pins (collecting the tests needs no library)."""
    import json
    from pathlib import Path
    return sorted(json.loads((Path(__file__).parent / "golden" / "free_scene_pins.json").read_text()))


SCENE_NAMES = _names()
BOX_AND_LIGHT = [n for n in SCENE_NAMES if n.startswith(("boxes_", "nest_", "posed_", "light_"))]
SUBSET = ["cam_orbit_0", "cam_closeup_clipped", "cam_inside_figure_bounds", "cam_up_parallel", "light_r0", "light_r40",
          "light_in_inner_box", "boxes_random_1", "nest_spare_minus_one_step", "posed_rotation_thresholds", "boxes_64",
          "boxes_212_largest_staged", "memo_window_top", "mirrors_70", "frame_tile1"]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def scenes(gpu):
    return {name: (scene, cfg) for name, scene, cfg in fs.free_scenes()}


_ORACLE_FRAMES = {}


def _oracle_frame(oracle, name, scene, cfg):
    key = (name, cfg.rng_mode)
    if key not in _ORACLE_FRAMES:
        _ORACLE_FRAMES[key] = oracle.render(scene, cfg)
    return _ORACLE_FRAMES[key]


def _assert_frame(oracle, scene, cfg, got, want, what):
    rep = pixel_report(got, want, oracle.quantize)
    assert rep["within1"] >= 0.999, (what, rep)
    if _flip_budget() == 0.0:
        assert np.array_equal(_bits(got), _bits(want)), (what, rep)
    bg = _background_pixels(oracle, scene, cfg, want)
    assert np.array_equal(_bits(got[bg]), _bits(want[bg])), what


@pytest.mark.parametrize("mode", FRAME_MODES)
@pytest.mark.parametrize("name", SCENE_NAMES)
def test_free_scene_frame(gpu, oracle, scenes, name, mode):
    scene, cfg = scenes[name]
    want = _oracle_frame(oracle, name, scene, cfg)
    got = _render_with_options(gpu, scene, cfg, RENDER_MODES[mode])
    _assert_frame(oracle, scene, cfg, got, want, (name, mode))
    if mode == "default":
        assert np.array_equal(gpu.aov(scene, cfg), oracle.aov(scene, cfg)), name


@pytest.mark.parametrize("mode", ["default", "megakernel", "split_tiles"])
@pytest.mark.parametrize("name", SUBSET)
def test_free_scene_counter_rng(gpu, oracle, scenes, name, mode):
    scene, base = scenes[name]
    cfg = type(base).from_buffer_copy(base)
    cfg.rng_mode = 1
    want = _oracle_frame(oracle, name, scene, cfg)
    got = _render_with_options(gpu, scene, cfg, RENDER_MODES[mode])
    _assert_frame(oracle, scene, cfg, got, want, (name, mode, "rng1"))


@pytest.mark.parametrize("name", SUBSET)
def test_free_scene_tile_sets(gpu, oracle, scenes, name):
    """mcskin_partition_tiles' cost-balanced sets of 3 (their weights come from the box rectangles, or the figure's, or
    the tile area when there are none), each rendered by its own context into one frame: the oracle's frame."""
    import torch
    scene, cfg = scenes[name]
    want = _oracle_frame(oracle, name, scene, cfg)
    n_tiles = len(gpu.generate_tiles(cfg.width, cfg.height, cfg.tile_size))
    parts = [gpu.partition_tiles(scene, cfg, 3, r) for r in range(3)]
    assert sorted(np.concatenate(parts).tolist()) == list(range(n_tiles))
    frame = torch.full((cfg.height, cfg.width, 4), -1.0, dtype=torch.float32, device="cuda:0")
    torch.cuda.synchronize()
    for r in range(3):
        ctx = gpu.Context(0)
        try:
            ctx.set_scene(scene, cfg)
            ctx.render_tiles_into_frame(parts[r], frame.data_ptr(), 0, 0)
            ctx.sync()
        finally:
            ctx.close()
    _assert_frame(oracle, scene, cfg, frame.cpu().numpy(), want, name)


# ---------------------------------------------------------------- single queries
@pytest.mark.parametrize("name", BOX_AND_LIGHT)
def test_free_scene_queries(gpu, oracle, scenes, name):
    scene, _ = scenes[name]
    rays = random_rays(np.random.default_rng(17), 50_000)
    want, got = oracle.intersect(scene, rays), gpu.intersect(scene, rays)
    assert want["hit"].mean() > 0.01, name
    for f in ("hit", "box", "face", "is_outer_layer"):
        assert np.array_equal(got[f], want[f]), (name, f)
    for f in ("t", "point", "normal", "tex_color"):
        assert np.array_equal(_bits(got[f]), _bits(want[f])), (name, f)
    hits = want[want["hit"] == 1][:6000]
    lights = np.tile(np.float32(scene.light_pos), (len(hits), 1))
    a = oracle.in_shadow(scene, hits["point"], hits["normal"], lights)
    assert np.array_equal(gpu.in_shadow(scene, hits["point"], hits["normal"], lights), a), name
    seeds = np.random.default_rng(3).integers(0, 2**32, size=len(hits), dtype=np.uint32)
    for samples in (8, 13):
        w = oracle.soft_shadow(scene, hits["point"], hits["normal"], seeds, samples)
        g = gpu.soft_shadow(scene, hits["point"], hits["normal"], seeds, samples)
        assert (g != w).mean() <= _flip_budget(), (name, samples, (g != w).mean())


def test_one_box_more_than_the_staging_area_is_refused(gpu):
    from minecraftskin_raytracer_b200 import _abi
    scene = fs.largest_scene(1)
    cfg = make_config(width=32, height=32, samples_per_pixel=1, max_bounces=1)
    with pytest.raises(gpu.McSkinError) as err:
        gpu.render(scene, cfg)
    assert err.value.code == _abi.MC_ERR_LIMIT
    ctx = gpu.Context(0)
    try:
        with pytest.raises(gpu.McSkinError) as err:
            ctx.set_scene(scene, cfg)
        assert err.value.code == _abi.MC_ERR_LIMIT
    finally:
        ctx.close()


# ---------------------------------------------------------------- the seed memo window
@pytest.mark.parametrize("memo", [1, 0])
def test_memo_scenes_after_the_standard_figure(gpu, oracle, scenes, memo):
    """One context renders the standard figure (its seeds fill the memo) and then the scenes whose shadow seeds straddle
    the window's edges or wrap through int64: every frame is the oracle's, with and without the memo."""
    import torch
    ctx = gpu.Context(0)
    try:
        ctx.set_option("shadow_seed_memo", memo)
        std = fs.skin("walking")
        std_cfg = make_config(width=64, height=64, samples_per_pixel=2, max_bounces=2)
        for name, scene, cfg in [("standard", std, std_cfg)] + [(n, *scenes[n]) for n in fs.MEMO_OFFSETS] + [("standard", std, std_cfg)]:
            out = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
            torch.cuda.synchronize()
            ctx.set_scene(scene, cfg)
            ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
            ctx.sync()
            _assert_frame(oracle, scene, cfg, out.cpu().numpy(), _oracle_frame(oracle, name, scene, cfg), (name, memo))
    finally:
        ctx.close()


# ---------------------------------------------------------------- batches
BATCH_CONFIGS = {
    "flat16": dict(samples_per_pixel=16, gradient_bg=0),
    "flat4": dict(samples_per_pixel=4, gradient_bg=0),
    "grad16": dict(samples_per_pixel=16),
    "spp3": dict(samples_per_pixel=3),
    "spp2_dof": dict(samples_per_pixel=2, dof_enabled=1, aperture=0.3),
    "hard": dict(samples_per_pixel=4, soft_shadows=0),
    "ao": dict(samples_per_pixel=4, ao_enabled=1, ao_samples=16),
}


@pytest.mark.parametrize("which", list(BATCH_CONFIGS))
def test_batches_at_every_form(gpu, oracle, which):
    import torch
    n = 6
    cfg = make_config(width=48, height=48, max_bounces=2, **BATCH_CONFIGS[which])
    atlases = np.stack([synth_skin(500 + i, "64x64") for i in range(n)])
    scenes = [gpu.build_skin_scene(atlases[i], "walking") for i in range(n)]
    ctx = gpu.Context(0)
    try:
        a = torch.zeros((n, cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
        b = torch.zeros_like(a)
        torch.cuda.synchronize()
        ctx.render_batch(scenes, cfg, a.data_ptr(), 0, 0)
        ctx.sync()
        ctx.render_skin_batch(atlases, cfg, "walking", b.data_ptr(), 0, 0)
        ctx.sync()
        got, got_skin = a.cpu().numpy(), b.cpu().numpy()
    finally:
        ctx.close()
    for i in range(n):
        single, _, _ = gpu.render(scenes[i], cfg)
        assert np.array_equal(_bits(got[i]), _bits(single)), (which, i)
        assert np.array_equal(_bits(got_skin[i]), _bits(single)), (which, i)
    for i in (0, n - 1):
        _assert_frame(oracle, scenes[i], cfg, got[i], oracle.render(scenes[i], cfg), (which, i))


def test_batch_of_cameras_and_lights(gpu, oracle):
    """One render_batch of the same figure from three cameras under two lights, interleaved: several groups of equal
    frame descriptions in one chunk; every image is the oracle's."""
    import dataclasses
    import torch
    base = fs.skin("dab")
    cams = [((0.0, 18.0, 50.0), (0.0, 18.0, 0.0)), ((30.0, 25.0, 35.0), (0.0, 16.0, 0.0)), ((-8.0, 10.0, 20.0), (0.0, 20.0, 0.0))]
    lights = [((0.0, 40.0, 30.0), 3.0), ((-20.0, 10.0, 15.0), 0.5)]
    scenes = [dataclasses.replace(base, cam_pos=cams[i % 3][0], cam_target=cams[i % 3][1], light_pos=lights[i % 2][0],
                                  light_radius=lights[i % 2][1]) for i in range(6)]
    cfg = make_config(width=48, height=48, samples_per_pixel=4, max_bounces=2)
    ctx = gpu.Context(0)
    try:
        out = torch.zeros((6, 48, 48, 4), dtype=torch.float32, device="cuda:0")
        torch.cuda.synchronize()
        for _ in range(2):
            ctx.render_batch(scenes, cfg, out.data_ptr(), 0, 0)
            ctx.sync()
        got = out.cpu().numpy()
    finally:
        ctx.close()
    for i, s in enumerate(scenes):
        _assert_frame(oracle, s, cfg, got[i], oracle.render(s, cfg), i)


# ---------------------------------------------------------------- which kernel forms run
def _kernels_run(gpu, fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {re.sub(r"\s+", "", e.name) for e in prof.events()}


ROUTES = [
    # (frame config, batch?, options, kernel the frame must launch)
    (dict(samples_per_pixel=16), False, {}, "k_primary_pix_fixed<16,true,false>"),
    (dict(samples_per_pixel=16, gradient_bg=0), False, {}, "k_primary_pix_fixed<16,false,false>"),
    (dict(samples_per_pixel=4), False, {}, "k_primary_pix_fixed<4,true,false>"),
    (dict(samples_per_pixel=4, gradient_bg=0), False, {}, "k_primary_pix_fixed<4,false,false>"),
    (dict(samples_per_pixel=8), False, {}, "k_primary_pix<false>"),
    (dict(samples_per_pixel=16), True, {}, "k_primary_pix_fixed<16,true,true>"),
    (dict(samples_per_pixel=16, gradient_bg=0), True, {}, "k_primary_pix_fixed<16,false,true>"),
    (dict(samples_per_pixel=4), True, {}, "k_primary_pix_fixed<4,true,true>"),
    (dict(samples_per_pixel=4, gradient_bg=0), True, {}, "k_primary_pix_fixed<4,false,true>"),
    (dict(samples_per_pixel=8), True, {}, "k_primary_pix<true>"),
    (dict(samples_per_pixel=16, dof_enabled=1, aperture=0.3), False, {}, "k_primary_warp"),
    (dict(samples_per_pixel=4), False, {"force_all_active": 1}, "k_primary_cta"),
    (dict(samples_per_pixel=4, shadow_samples=114), False, {}, "k_wf_shade<false,false>"),
    (dict(samples_per_pixel=4, shadow_samples=8), False, {}, "k_wf_shade<true,false>"),
    (dict(samples_per_pixel=4, soft_shadows=0), True, {}, "k_wf_hardshadow<true>"),
]


def test_each_route_launches_its_kernel(gpu):
    """Under torch.profiler (CUDA activities, graphs off) each frame launches the kernel instantiation named for it."""
    import torch
    scene = fs.skin("walking")
    launched = []
    for over, batch, opts, kernel in ROUTES:
        cfg = make_config(width=48, height=48, max_bounces=1, **over)
        ctx = gpu.Context(0)
        try:
            ctx.set_option("use_graphs", 0)
            for k, v in opts.items():
                ctx.set_option(k, v)
            if batch:
                out = torch.zeros((4, 48, 48, 4), dtype=torch.float32, device="cuda:0")
                scenes = [gpu.build_skin_scene(synth_skin(600 + i), "walking") for i in range(4)]
                names = _kernels_run(gpu, lambda: (ctx.render_batch(scenes, cfg, out.data_ptr(), 0, 0), ctx.sync()))
            else:
                out = torch.zeros((48, 48, 4), dtype=torch.float32, device="cuda:0")
                ctx.set_scene(scene, cfg)
                names = _kernels_run(gpu, lambda: (ctx.render_bands(0, 1, out.data_ptr(), 0, 0), ctx.sync()))
        finally:
            ctx.close()
        launched.append((kernel, [n for n in names if "k_primary" in n or "k_wf_" in n]))
    if not any(ours for _, ours in launched):
        pytest.skip("the profiler reported none of this library's kernels")
    for kernel, ours in launched:  # once it reports them, every route must show its own
        pattern = re.escape(kernel) + (r"(\(|$)" if "<" in kernel else r"(<|\(|$)")
        assert any(re.search(pattern, n) for n in ours), (kernel, sorted(ours))

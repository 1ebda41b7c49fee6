"""GPU parity on the free configurations (tests/free_configs.py): shading weights, light colour, background, AO, lens and
sampling fields away from the reference defaults — whole frames through the library's code paths in float bits and 8-bit
bytes, counter-based streams, tile sets and tile rows, batches whose scenes differ only in light colour or background,
single queries, and the AOV planes, which no shading field may change."""
import json
from pathlib import Path

import numpy as np
import pytest

from minecraftskin_raytracer_b200 import _abi
from tests import free_configs as fc
from tests.conftest import pixel_report
from tests.scenes import random_rays, synth_skin
from tests.test_parity_gpu import RENDER_MODES, _flip_budget, _render_with_options

pytestmark = pytest.mark.gpu

FRAME_MODES = ["default", "all_active", "megakernel", "megakernel_warp", "tiny_queue", "split_tiles"]
# the names, from the pins (collecting the tests needs no library)
NAMES = sorted(json.loads((Path(__file__).parent / "golden" / "free_config_pins.json").read_text()))
SUBSET = ["phong_shininess_negative_hard", "phong_ks_bright_clamp", "light_color_distinct", "bg_flat_alpha_out_of_range",
          "bg_gradient_spp16_fixed_form", "bg_gradient_spp4_fixed_form", "ao_samples_0_nan", "ao_radius_1e6",
          "soft_shadow_samples_2", "lens_aperture_above_gate", "lens_focus_1e4", "spp_negative", "tile_33", "mixed_1",
          "mixed_5", "mixed_8"]
QUERY_NAMES = [n for n in NAMES if n.startswith(("phong_", "light_color_", "bg_", "ao_"))]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def cases(gpu):
    return {c.name: c for c in fc.free_configs()}


_ORACLE_FRAMES = {}


def _oracle_frame(oracle, name, scene, cfg):
    key = (name, cfg.rng_mode)
    if key not in _ORACLE_FRAMES:
        _ORACLE_FRAMES[key] = oracle.render(scene, cfg)
    return _ORACLE_FRAMES[key]


def _differences(got, want):
    """How many channels differ in bits, and the first few as (pixel, channel, got bits, oracle bits)."""
    g, w = _bits(got), _bits(want)
    idx = np.argwhere(g != w)
    return len(idx), [(tuple(int(v) for v in i[:-1]), int(i[-1]), hex(int(g[tuple(i)])), hex(int(w[tuple(i)]))) for i in idx[:4]]


def _assert_frame(oracle, got, want, what, got_u8=None):
    exact = _flip_budget() == 0.0
    if exact:
        assert np.array_equal(_bits(got), _bits(want)), (what, _differences(got, want))
    else:
        assert pixel_report(got, want, oracle.quantize)["within1"] >= 0.999, what
    if got_u8 is not None:
        assert np.array_equal(got_u8, oracle.quantize(want if exact else got)), what


def _frame(gpu, scene, cfg, opts):
    """The float and 8-bit frames: mcskin_cuda_render without options, else a context's render_bands with them (direct
    launches, the call that captures the graph, a replay: all three the same)."""
    if not opts:
        f32, u8, _ = gpu.render(scene, cfg, want_u8=True)
        return f32, u8
    import torch
    ctx = gpu.Context(0)
    try:
        for k, v in opts.items():
            ctx.set_option(k, v)
        ctx.set_scene(scene, cfg)
        out = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
        out8 = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.uint8, device="cuda:0")
        frames = []
        for _ in range(3):
            out.fill_(-1.0)
            out8.fill_(7)
            torch.cuda.synchronize()
            ctx.render_bands(0, 1, out.data_ptr(), out8.data_ptr(), 0)
            ctx.sync()
            frames.append((out.cpu().numpy(), out8.cpu().numpy()))
        for f32, u8 in frames[:2]:
            assert np.array_equal(_bits(f32), _bits(frames[2][0])) and np.array_equal(u8, frames[2][1])
        return frames[2]
    finally:
        ctx.close()


@pytest.mark.parametrize("mode", FRAME_MODES)
@pytest.mark.parametrize("name", NAMES)
def test_free_config_frame(gpu, oracle, cases, name, mode):
    c = cases[name]
    want = _oracle_frame(oracle, name, c.scene, c.cfg)
    got, got_u8 = _frame(gpu, c.scene, c.cfg, RENDER_MODES[mode])
    _assert_frame(oracle, got, want, (name, mode), got_u8)


@pytest.mark.parametrize("mode", ["default", "megakernel", "split_tiles"])
@pytest.mark.parametrize("name", SUBSET)
def test_free_config_counter_rng(gpu, oracle, cases, name, mode):
    c = cases[name]
    cfg = _abi.copy_config(c.cfg, rng_mode=1)
    want = _oracle_frame(oracle, name, c.scene, cfg)
    _assert_frame(oracle, _render_with_options(gpu, c.scene, cfg, RENDER_MODES[mode]), want, (name, mode, "rng1"))


@pytest.mark.parametrize("name", SUBSET)
def test_free_config_tile_sets_and_rows(gpu, oracle, cases, name):
    """Three cost-balanced tile sets of partition_tiles, each rendered by its own context into one frame, and the tile
    rows of render_bands at stride 2, reassembled: the oracle's frame."""
    import torch
    from minecraftskin_raytracer_b200 import bands
    c = cases[name]
    scene, cfg = c.scene, c.cfg
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
    _assert_frame(oracle, frame.cpu().numpy(), want, (name, "tile sets"))
    ctx = gpu.Context(0)
    try:
        ctx.set_scene(scene, cfg)
        rows = []
        for r in range(2):
            band = torch.full((bands.padded_band_rows(cfg.height, cfg.tile_size, 2), cfg.width, 4), -1.0, device="cuda:0")
            ctx.render_bands(r, 2, band.data_ptr(), 0, 0)
            ctx.sync()
            rows.append(band)
        whole = bands.deinterleave(rows, torch.zeros((cfg.height, cfg.width, 4), device="cuda:0"), cfg.tile_size)
        _assert_frame(oracle, whole.cpu().numpy(), want, (name, "bands stride 2"))
    finally:
        ctx.close()


# ---------------------------------------------------------------- batches
LIGHT_COLOURS = [(1.0, 1.0, 1.0, 1.0), (1.0, 0.55, 0.2, 1.0), (0.9, 0.0, 0.7, 0.5)]
BACKGROUNDS = [(0.2, 0.3, 0.5, 1.0), (0.9, 0.1, 0.35, 0.6)]


@pytest.mark.parametrize("gradient_bg", [1, 0])
def test_batch_of_light_colours_and_backgrounds(gpu, oracle, gradient_bg):
    """One render_batch of the same figure under three light colours and two backgrounds, interleaved: scenes whose frame
    descriptions differ in these fields alone must not share a group, and every image is its own scene's oracle frame."""
    import dataclasses
    import torch
    base = fc.skin("dab")
    scenes = [dataclasses.replace(base, light_color=LIGHT_COLOURS[i % 3], background=BACKGROUNDS[(i // 3) % 2])
              for i in range(6)]
    cfg = _abi.default_config(width=48, height=48, samples_per_pixel=4, max_bounces=2, gradient_bg=gradient_bg)
    ctx = gpu.Context(0)
    try:
        out = torch.zeros((6, 48, 48, 4), dtype=torch.float32, device="cuda:0")
        out8 = torch.zeros((6, 48, 48, 4), dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        for _ in range(2):
            ctx.render_batch(scenes, cfg, out.data_ptr(), out8.data_ptr(), 0)
            ctx.sync()
        got, got8 = out.cpu().numpy(), out8.cpu().numpy()
    finally:
        ctx.close()
    wants = [oracle.render(s, cfg) for s in scenes]
    assert len({_bits(w).tobytes() for w in wants}) == 6     # six different frames
    for i, s in enumerate(scenes):
        _assert_frame(oracle, got[i], wants[i], i, got8[i])


@pytest.mark.parametrize("name", ["mixed_0", "mixed_5"])
def test_skin_batch_with_a_mixed_config(gpu, oracle, cases, name):
    """render_skin_batch (atlases sliced on the device) under a mixed configuration: every image is the oracle's frame
    of the host-built scene."""
    import torch
    cfg = cases[name].cfg
    atlases = np.stack([synth_skin(800 + i, "64x64") for i in range(4)])
    scenes = [gpu.build_skin_scene(a, "walking") for a in atlases]
    ctx = gpu.Context(0)
    try:
        out = torch.zeros((4, cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
        out8 = torch.zeros((4, cfg.height, cfg.width, 4), dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        ctx.render_skin_batch(atlases, cfg, "walking", out.data_ptr(), out8.data_ptr(), 0)
        ctx.sync()
        got, got8 = out.cpu().numpy(), out8.cpu().numpy()
    finally:
        ctx.close()
    for i, s in enumerate(scenes):
        _assert_frame(oracle, got[i], oracle.render(s, cfg), (name, i), got8[i])


# ---------------------------------------------------------------- single queries
def _assert_query(got, want, what):
    if _flip_budget() == 0.0:
        assert np.array_equal(_bits(got), _bits(want)), (what, _differences(got, want))
    else:
        close = np.isclose(got, want, rtol=0, atol=1e-5, equal_nan=True).reshape(len(got), -1).all(axis=1)
        assert close.mean() >= 0.99, what


@pytest.mark.parametrize("name", QUERY_NAMES)
def test_free_config_queries(gpu, oracle, cases, name):
    """shade (hard shadow test inside, and given shadow factors), trace (with and without the config, from depth 0 and
    2), background and ambient_occlusion (the configuration's sample count and radius) against the oracle in bits."""
    c = cases[name]
    scene, cfg = c.scene, c.cfg
    rays = random_rays(np.random.default_rng(17), 200_000 if name == "phong_shininess_4000_underflow" else 30_000)
    hits = oracle.intersect(scene, rays)
    keep = hits["hit"] == 1
    hits, view = hits[keep], -rays["dir"][keep]
    for sf in (None, np.random.default_rng(0).random(len(hits)).astype(np.float32), np.ones(len(hits), np.float32)):
        _assert_query(gpu.shade(scene, cfg, hits, view, sf), oracle.shade(scene, cfg, hits, view, sf), (name, "shade"))
    sub = rays[:4000]
    for use_config, depth in ((True, 0), (False, 0), (True, 2)):
        _assert_query(gpu.trace(scene, cfg, sub, depth, use_config), oracle.trace(scene, cfg, sub, depth, use_config),
                      (name, "trace", use_config, depth))
    uv = np.random.default_rng(3).uniform(-0.2, 1.2, (5000, 2)).astype(np.float32)
    for use_config in (True, False):
        _assert_query(gpu.background(scene, cfg, uv, use_config), oracle.background(scene, cfg, uv, use_config),
                      (name, "background", use_config))
    pts = hits[:3000]
    seeds = np.random.default_rng(4).integers(0, 2**32, size=len(pts), dtype=np.uint32)
    ao_args = (pts["point"], pts["normal"], seeds, cfg.ao_samples, cfg.ao_radius)
    _assert_query(gpu.ambient_occlusion(scene, *ao_args), oracle.ambient_occlusion(scene, *ao_args), (name, "ao"))


# ---------------------------------------------------------------- AOV planes
SHADING_FIELDS = ("max_bounces", "thread_count", "kd", "ks", "ambient", "shininess", "ao_enabled", "ao_samples",
                  "ao_radius", "ao_intensity", "soft_shadows", "shadow_samples", "gradient_bg", "gradient_scale",
                  "bg_center", "bg_edge")


@pytest.mark.parametrize("name", NAMES)
def test_free_config_aov_planes(gpu, oracle, cases, name):
    """render_aovs(guides=True): all five planes equal the guide oracle's, and equal the device's planes of the same
    frame at default shading, light colour and background (the planes depend on the camera rays alone); the colour is
    render's."""
    import dataclasses
    from tests.guide_oracle import render_aovs
    c = cases[name]
    d = _abi.default_config()
    plain_cfg = _abi.copy_config(c.cfg, **{f: tuple(getattr(d, f)) if f.startswith("bg_") else getattr(d, f)
                                          for f in SHADING_FIELDS})
    plain_scene = dataclasses.replace(c.scene, light_color=(1.0, 1.0, 1.0, 1.0), background=(0.2, 0.3, 0.5, 1.0))
    f32, _, planes, _ = gpu.render_aovs(c.scene, c.cfg, guides=True)
    _, _, plain, _ = gpu.render_aovs(plain_scene, plain_cfg, guides=True)
    want = render_aovs(c.scene, c.cfg, guides=True)
    exact = _flip_budget() == 0.0
    for p in want:
        assert np.array_equal(planes[p].view(np.uint32), plain[p].view(np.uint32)), (name, p)
        if exact:
            assert np.array_equal(planes[p].view(np.uint32), want[p].view(np.uint32)), (name, p)
        else:
            assert (planes[p].view(np.uint32) == want[p].view(np.uint32)).mean() >= 0.999, (name, p)
    assert np.array_equal(_bits(f32), _bits(gpu.render(c.scene, c.cfg)[0])), name

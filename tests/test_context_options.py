"""Context options (mcskin_cuda_context_set_option, INTEGRATION.md §6): every documented name is accepted, an environment
override renders exactly what the same value given through set_option renders, and a captured frame graph is not
replayed once a launch option changed."""
import os
import re
from pathlib import Path

import numpy as np
import pytest

from minecraftskin_raytracer_b200.lib import McSkinError
from tests.scenes import make_config, synth_skin

pytestmark = pytest.mark.gpu

INTEGRATION = Path(__file__).resolve().parents[1] / "INTEGRATION.md"

# environment variable -> (option, a value other than the default)
ENV_OPTIONS = {
    "MCSKIN_FORCE_ALL_ACTIVE": ("force_all_active", 1),
    "MCSKIN_HEAVY_TILES": ("heavy_tiles_per_sm", 0),
    "MCSKIN_PRIMARY_BLOCKS": ("primary_blocks_per_sm", 100000),
    "MCSKIN_WAVE_QUEUE_PCT": ("wave_queue_pct", 150),
    "MCSKIN_BATCH_GROUP": ("batch_group", 7),
    "MCSKIN_BATCH_MODE": ("batch_mode", 0),
    "MCSKIN_GRAPHS": ("use_graphs", 0),
    "MCSKIN_STAGED_COPY": ("staged_copy_out", 0),
    "MCSKIN_SEED_MEMO": ("shadow_seed_memo", 0),
    "MCSKIN_OVERLAP_COPY": ("overlap_copy_out", 1),
    "MCSKIN_FRAME_LANES": ("frame_lanes", 1),
    "MCSKIN_CACHE_TILE_SEEDS": ("cache_tile_seeds", 0),
    "MCSKIN_SHADE_BLOCKS": ("shade_blocks_per_sm", 2),
    "MCSKIN_SOFT_BLOCKS": ("soft_blocks_per_sm", 1),
    "MCSKIN_SHADE_MODE": ("shade_mode", 1),
}


def _documented_options():
    text = INTEGRATION.read_text()
    section = text[text.index("## 6."):]
    names = set()
    for line in section.splitlines():
        if line.startswith("| `"):
            first_cell = line.split("|")[1]
            names.update(n for n in re.findall(r"`([a-z_0-9]+)`", first_cell))
    return names


def test_documented_options_are_accepted(gpu):
    names = _documented_options()
    assert {opt for opt, _ in ENV_OPTIONS.values()} <= names
    assert "debug_primary_timing" in names and "record_budget_bytes" in names
    section = INTEGRATION.read_text().split("## 6.")[1]
    for env in ENV_OPTIONS:
        assert f"`{env}`" in section, env
    ctx = gpu.Context(0)
    try:
        for name in sorted(names):
            ctx.set_option(name, 1)
        with pytest.raises(McSkinError):
            ctx.set_option("no_such_option", 1)
    finally:
        ctx.close()


def _frame():
    """A frame of 6 tile rows (soft shadows on: the seed memo is in play)."""
    from minecraftskin_raytracer_b200 import lib
    scene = lib.build_skin_scene(synth_skin(3, "64x64"), "walking")
    cfg = make_config(width=96, height=96, tile_size=16, samples_per_pixel=4, max_bounces=2)
    return scene, cfg


def _render(ctx, scene, cfg, times=1):
    import torch
    out = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
    for _ in range(times):
        ctx.set_scene(scene, cfg)
        ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
        stats = ctx.sync()
    return out.cpu().numpy().view(np.uint32).copy(), stats


def _context_with_env(gpu, env, value):
    old = os.environ.get(env)
    os.environ[env] = str(value)
    try:
        return gpu.Context(0)
    finally:
        if old is None:
            del os.environ[env]
        else:
            os.environ[env] = old


@pytest.mark.parametrize("env", sorted(ENV_OPTIONS))
def test_environment_override_equals_set_option(gpu, env):
    option, value = ENV_OPTIONS[env]
    scene, cfg = _frame()
    by_env = _context_with_env(gpu, env, value)
    by_option = gpu.Context(0)
    try:
        by_option.set_option(option, value)
        img_env, st_env = _render(by_env, scene, cfg, times=3)
        img_opt, st_opt = _render(by_option, scene, cfg, times=3)
        assert np.array_equal(img_env, img_opt)
        assert st_env["n_kernel_launches"] == st_opt["n_kernel_launches"]
        assert st_env["n_tiles"] == st_opt["n_tiles"] == 36
    finally:
        by_env.close()
        by_option.close()


def test_frame_lanes_from_environment_is_read(gpu):
    """One lane renders the 6 tile rows with half the launches of the default two lanes."""
    scene, cfg = _frame()
    one = _context_with_env(gpu, "MCSKIN_FRAME_LANES", 1)
    two = gpu.Context(0)
    try:
        img_one, st_one = _render(one, scene, cfg)
        img_two, st_two = _render(two, scene, cfg)
        assert np.array_equal(img_one, img_two)
        assert st_two["n_kernel_launches"] == 2 * st_one["n_kernel_launches"]
    finally:
        one.close()
        two.close()


def test_debug_primary_timing_after_graph_capture(gpu):
    """Switching a launch option on after a frame's graph was captured renders anew instead of replaying the graph."""
    scene, cfg = _frame()
    ctx = gpu.Context(0)
    try:
        ctx.set_option("frame_lanes", 1)
        first, _ = _render(ctx, scene, cfg, times=3)  # rendered, captured, replayed
        assert len(ctx.debug_block_times()) == 0
        ctx.set_option("debug_primary_timing", 1)
        again, _ = _render(ctx, scene, cfg)
        assert np.array_equal(first, again)
        assert len(ctx.debug_block_times()) > 0
    finally:
        ctx.close()

"""Shared scene / config fixtures for the tests (pure data, no oracle or GPU use)."""
from __future__ import annotations

import numpy as np

from minecraftskin_raytracer_b200 import _abi
from minecraftskin_raytracer_b200.scene import FlatScene, make_box, solid_box_scene, synth_skin  # noqa: F401

# (name, skin seed, skin kind, pose, config overrides) — small enough for the CPU oracle in seconds
RENDER_CASES = [
    ("c1_small", 1, "64x64", None, dict(width=160, height=160, samples_per_pixel=1, max_bounces=2)),
    ("jitter4", 1, "64x64", None, dict(width=128, height=96, samples_per_pixel=4, max_bounces=4)),
    ("legacy_walk", 2, "legacy", "walking", dict(width=160, height=90, samples_per_pixel=3, max_bounces=4, tile_size=16)),
    ("slim_dab_hard", 3, "slim", "dab", dict(width=100, height=100, samples_per_pixel=2, max_bounces=2, soft_shadows=0)),
    ("waving_ao", 4, "64x64", "waving", dict(width=96, height=96, samples_per_pixel=2, max_bounces=3, ao_enabled=1, ao_samples=16)),
    ("fighting_dof", 5, "64x64", "fighting", dict(width=96, height=96, samples_per_pixel=2, max_bounces=3, dof_enabled=1, aperture=0.3)),
    ("sitting_flatbg", 6, "64x64", "sitting", dict(width=96, height=64, samples_per_pixel=1, max_bounces=8, gradient_bg=0, shadow_samples=3)),
    ("running_neg_bounce", 7, "64x64", "running", dict(width=70, height=50, samples_per_pixel=5, max_bounces=-1)),
    ("dof_spp1", 8, "64x64", None, dict(width=64, height=64, samples_per_pixel=1, max_bounces=0, dof_enabled=1, aperture=0.5, focus_distance=40.0, ao_enabled=1)),
    ("headline_small", 0, "64x64", None, dict(width=192, height=108, samples_per_pixel=16, max_bounces=4)),
    ("tile7_spp3", 9, "64x64", "walking", dict(width=53, height=41, samples_per_pixel=3, max_bounces=2, tile_size=7)),
    ("tile7_spp4", 9, "64x64", "walking", dict(width=53, height=41, samples_per_pixel=4, max_bounces=2, tile_size=7)),
    ("spp32", 11, "64x64", "dab", dict(width=64, height=48, samples_per_pixel=32, max_bounces=2)),
    ("spp2_dof", 12, "64x64", None, dict(width=80, height=60, samples_per_pixel=2, max_bounces=3, dof_enabled=1, aperture=0.4)),
    ("spp8_tile24", 13, "legacy", "running", dict(width=100, height=60, samples_per_pixel=8, max_bounces=3, tile_size=24)),
    ("spp64", 14, "64x64", None, dict(width=40, height=40, samples_per_pixel=64, max_bounces=2)),
    ("spp300", 15, "64x64", None, dict(width=24, height=24, samples_per_pixel=300, max_bounces=1)),
    ("many_shadow_samples", 10, "64x64", None, dict(width=48, height=48, samples_per_pixel=1, max_bounces=1, shadow_samples=64)),
    # route cases: kernel forms and shading routes the cases above never select (kernels.cu launch_primary_pix,
    # wavefront.cu shadow_mode_of, dev_shade.cuh ambient_occlusion)
    # flat 16-spp pixel-per-lane form; 13 shadow samples = one full round of 8 and a partial one; the largest AO that
    # still draws from a FreshStream (2 * 113 <= 227)
    ("flat16_sh13_ao113", 16, "64x64", "walking", dict(width=48, height=48, samples_per_pixel=16, max_bounces=2,
                                                        gradient_bg=0, shadow_samples=13, ao_enabled=1, ao_samples=113)),
    # flat 4-spp form; 114 shadow samples shade in-thread from a LocalEngine, 114 AO samples take ambient_occlusion_large
    ("flat4_sh114_ao114", 17, "64x64", "dab", dict(width=48, height=48, samples_per_pixel=4, max_bounces=1, gradient_bg=0,
                                                   tile_size=16, shadow_samples=114, ao_enabled=1, ao_samples=114)),
    # generic pixel-per-lane form at spp x draws = 60, the largest ring that fits; one shadow sample: hard shadows
    ("spp30_sh1", 18, "legacy", "running", dict(width=48, height=48, samples_per_pixel=30, max_bounces=2, shadow_samples=1)),
    # generic form with lens draws at spp x draws = 60
    ("dof_spp15", 19, "64x64", "fighting", dict(width=48, height=48, samples_per_pixel=15, max_bounces=1, dof_enabled=1,
                                                aperture=0.4, shadow_samples=113)),
    # lens draws at spp x draws = 64 > 61: the warp-per-pixel form
    ("dof_spp16", 20, "64x64", None, dict(width=48, height=48, samples_per_pixel=16, max_bounces=2, dof_enabled=1,
                                          aperture=0.3)),
]


def make_config(**kw):
    return _abi.default_config(**kw)


def random_rays(rng: np.random.Generator, n: int, scene: FlatScene | None = None) -> np.ndarray:
    """Rays aimed at (and around) the figure from points on a shell, plus axis-parallel and interior origins."""
    rays = np.zeros(n, dtype=_abi.RAY_DTYPE)
    centre = np.array([0.0, 16.0, 0.0], dtype=np.float32)
    origins = rng.normal(size=(n, 3)).astype(np.float32)
    origins /= np.linalg.norm(origins, axis=1, keepdims=True) + 1e-9
    origins = centre + origins * rng.uniform(1.0, 60.0, size=(n, 1)).astype(np.float32)
    targets = centre + rng.uniform(-10, 10, size=(n, 3)).astype(np.float32) * np.array([1.0, 1.8, 0.6], dtype=np.float32)
    dirs = targets - origins
    # a share of exactly axis-parallel directions (the 1e-8 branch of the slab test)
    k = n // 8
    axes = rng.integers(0, 3, size=k)
    dirs[:k] = 0
    dirs[np.arange(k), axes] = rng.choice([-1.0, 1.0], size=k)
    origins[:k] = np.round(origins[:k])
    norm = np.linalg.norm(dirs, axis=1, keepdims=True)
    dirs = (dirs / np.maximum(norm, 1e-9)).astype(np.float32)
    rays["origin"] = origins
    rays["dir"] = dirs
    return rays

"""Generates tests/golden/reference_vectors.npz from the UNMODIFIED reference
(oracle/_ref/libmcskin_ref.so, built by oracle/build_ref.sh from the checkout that
MCSKIN_REFERENCE_DIR names, else `reference` beside this repository).

The reference ships no golden images (SURVEY.md §4), so these vectors are outputs of the
reference itself: small full-scene renders (float RGBA + the intersectScene call count),
pixel-centre triangle ids, single-ray intersections, Blinn-Phong values, traced colours,
soft-shadow / AO factors and the libstdc++ RNG streams behind them.  They are committed
so that the tests need no copy of the reference.

    [MCSKIN_REFERENCE_DIR=<reference checkout>] python tests/golden/make_golden.py
"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from minecraftskin_raytracer_b200 import _abi  # noqa: E402
from minecraftskin_raytracer_b200.scene import synth_skin  # noqa: E402
from oracle.harness import Reference, build_reference  # noqa: E402
from tests.scenes import make_config, random_rays  # noqa: E402

# (name, seed, kind, pose, config)
GOLDEN_RENDERS = [
    ("g_standing_1spp", 1, "64x64", None, dict(width=64, height=64, samples_per_pixel=1, max_bounces=2)),
    ("g_walking_4spp", 2, "64x64", "walking", dict(width=64, height=48, samples_per_pixel=4, max_bounces=3)),
    ("g_legacy_hard", 3, "legacy", "running", dict(width=48, height=48, samples_per_pixel=2, max_bounces=2, soft_shadows=0)),
    ("g_dab_ao_dof", 4, "64x64", "dab", dict(width=48, height=40, samples_per_pixel=2, max_bounces=2, ao_enabled=1, dof_enabled=1, aperture=0.3)),
    ("g_headline_tiny", 0, "64x64", None, dict(width=96, height=54, samples_per_pixel=16, max_bounces=4)),
    ("g_tile5_spp3_flat", 5, "slim", "waving", dict(width=37, height=29, samples_per_pixel=3, max_bounces=1, tile_size=5, gradient_bg=0)),
]


def main():
    build_reference()
    ref = Reference.load()
    if ref is None:
        raise SystemExit("oracle/_ref/libmcskin_ref.so is missing and no checkout of the reference was found (set MCSKIN_REFERENCE_DIR)")
    out = {}
    for name, seed, kind, pose, over in GOLDEN_RENDERS:
        atlas = synth_skin(seed, kind)
        scene = ref.scene_from_atlas(atlas, pose)
        cfg = make_config(**over)
        img, calls = ref.render(scene, cfg, counters=True)
        out[f"{name}/image"] = img
        out[f"{name}/calls"] = np.int64(calls)
        out[f"{name}/tri_id"] = ref.aov(scene, cfg)
        out[f"{name}/boxes"] = scene.boxes           # the reference's own Scene, flattened
        out[f"{name}/texels"] = scene.texels
    # single-ray vectors on a posed 12-box scene
    scene = ref.scene_from_atlas(synth_skin(6, "64x64"), "fighting")
    rays = random_rays(np.random.default_rng(101), 4000)
    hits = ref.intersect(scene, rays)
    out["rays/rays"] = rays
    out["rays/hits"] = hits
    keep = hits["hit"] == 1
    cfg = make_config(max_bounces=3)
    out["rays/shade_hard"] = ref.shade(scene, cfg, hits[keep], -rays["dir"][keep], None)
    sf = np.random.default_rng(7).random(int(keep.sum())).astype(np.float32)
    out["rays/shade_sf"] = sf
    out["rays/shade_soft"] = ref.shade(scene, cfg, hits[keep], -rays["dir"][keep], sf)
    out["rays/trace_cfg"] = ref.trace(scene, cfg, rays[:1500], depth=0, use_config=True)
    out["rays/trace_nocfg"] = ref.trace(scene, cfg, rays[:1500], depth=0, use_config=False)
    seeds = np.random.default_rng(8).integers(0, 2**32, size=int(keep.sum()), dtype=np.uint32)
    out["rays/seeds"] = seeds
    out["rays/soft8"] = ref.soft_shadow(scene, hits["point"][keep], hits["normal"][keep], seeds, 8)
    out["rays/ao16"] = ref.ambient_occlusion(scene, hits["point"][keep], hits["normal"][keep], seeds, 16, 3.0)
    uv = np.random.default_rng(9).random((512, 2)).astype(np.float32)
    out["rays/uv"] = uv
    out["rays/camera"] = ref.generate_rays(scene, 16.0 / 9.0, uv)
    out["rays/background"] = ref.background(scene, cfg, uv)
    # libstdc++ std::mt19937 + uniform_real_distribution<float>(0,1)
    for seed in (0, 1, 5489, 1920 * 32 + 64, 0xFFFFFFFF):
        u, f = ref.mt19937(seed, 2000)
        out[f"rng/{seed}/u32"] = u
        out[f"rng/{seed}/canonical"] = f
    casts = np.array([0.0, 1.5, -5.7, 5e9, -3e9, 4294967296.0, 1e19, -1e19, 123456.789], dtype=np.float32)
    out["rng/seed_cast_in"] = casts
    out["rng/seed_cast_out"] = np.array([ref.seed_cast(float(c)) for c in casts], dtype=np.uint32)
    path = Path(__file__).with_name("reference_vectors.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, f"{path.stat().st_size / 1024:.0f} KiB", len(out), "arrays")


if __name__ == "__main__":
    main()

"""Generates tests/golden/oracle_pins.json: SHA-256 digests of what the CPU oracle and the host scene builder
compute for the inputs the live-reference tests use (tests.scenes.RENDER_CASES, the single-ray set, every
built-in pose of three skins).

These are NOT outputs of the unmodified reference: that is tests/golden/reference_vectors.npz, which covers
fewer inputs.  They pin the oracle and the builder as they stand, so that a change to either that alters
one bit of these outputs fails without a copy of the reference; such a change is then checked against the
reference itself (MCSKIN_REFERENCE_DIR, tests test_oracle_equals_live_reference*,
test_skin_scene_builder_equals_live_reference) and the pins regenerated.

    python tests/golden/make_oracle_pins.py
"""
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from minecraftskin_raytracer_b200.scene import BUILTIN_POSE_ORDER, synth_skin  # noqa: E402
from tests.scenes import RENDER_CASES, make_config, random_rays  # noqa: E402

PATH = Path(__file__).with_name("oracle_pins.json")
SCENE_SKINS = ((0, "64x64"), (2, "legacy"), (3, "slim"))


def digest(*arrays) -> str:
    """Digest of array values, field by field for structured arrays (padding bytes are not part of it)."""
    h = hashlib.sha256()

    def add(a):
        a = np.asarray(a)
        if a.dtype.names:
            for name in a.dtype.names:
                add(a[name])
        else:
            h.update(str(a.dtype).encode() + str(a.shape).encode())
            h.update(np.ascontiguousarray(a).tobytes())

    for a in arrays:
        add(a)
    return h.hexdigest()


def scene_digest(scene) -> str:
    return digest(scene.boxes, scene.texels)


def overlay_atlas():
    """Skin 5 with a fully transparent head overlay (dropped by the builder, mesh_builder.cpp:176-186)."""
    atlas = synth_skin(5)
    atlas[:16, 32:, 3] = 0
    return atlas


def single_ray_inputs(scene_builder):
    scene = scene_builder(synth_skin(21, "64x64"), "dab")
    return scene, random_rays(np.random.default_rng(3), 6000), make_config(max_bounces=4, ao_enabled=1)


def compute(oracle, build_skin_scene) -> dict:
    out = {"renders": {}, "scenes": {}}
    for name, seed, kind, pose, over in RENDER_CASES:
        scene = build_skin_scene(synth_skin(seed, kind), pose)
        cfg = make_config(**over)
        img, cnt = oracle.render(scene, cfg, counters=True)
        out["renders"][name] = {"image": digest(img), "calls": cnt["n_intersect_scene"], "tri_id": digest(oracle.aov(scene, cfg))}
    scene, rays, cfg = single_ray_inputs(build_skin_scene)
    out["rays"] = {"hits": digest(oracle.intersect(scene, rays)), "trace": digest(oracle.trace(scene, cfg, rays[:800])),
                   "mt19937_77": digest(oracle.mt19937(77, 500)[0])}
    for seed, kind in SCENE_SKINS:
        for pose in [None] + BUILTIN_POSE_ORDER:
            out["scenes"][f"{seed}/{kind}/{pose}"] = scene_digest(build_skin_scene(synth_skin(seed, kind), pose))
    out["scenes"]["overlay_dropped"] = scene_digest(build_skin_scene(overlay_atlas(), None))
    return out


def main():
    from minecraftskin_raytracer_b200 import lib
    from oracle.harness import Oracle
    PATH.write_text(json.dumps(compute(Oracle(), lib.build_skin_scene), indent=1, sort_keys=True) + "\n")
    print("wrote", PATH)


if __name__ == "__main__":
    main()

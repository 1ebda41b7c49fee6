"""Generates tests/golden/texel_pins.json: SHA-256 digests of the texel plane the CPU oracle of all six AOV planes
(tests/texel_oracle.c) computes for tests.scenes.RENDER_CASES, with the std::mt19937 streams (rng_mode 0) and the
counter-based ones (rng_mode 1), and for the free scenes of TEXEL_FREE_SCENES (magenta and blank faces, posed boxes at the
rotation thresholds, an outer layer seen from inside, nested boxes, and the 33- and 212-box scenes).  They pin that oracle
as it stands; the oracle checks every texel it restates against its own intersection, and the GPU is checked against it.

    python tests/golden/make_texel_pins.py
"""
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from minecraftskin_raytracer_b200.scene import synth_skin  # noqa: E402
from tests.golden.make_oracle_pins import digest  # noqa: E402
from tests.scenes import RENDER_CASES, make_config  # noqa: E402

PATH = Path(__file__).with_name("texel_pins.json")
TEXEL_FREE_SCENES = ("boxes_random_0", "boxes_random_1", "posed_rotation_thresholds", "boxes_212_largest_staged",
                     "nest_chains_exact_spare", "cam_inside_outer_layer", "boxes_33")


def free_texel_scenes():
    """(name, scene, config) of TEXEL_FREE_SCENES, in that order."""
    from tests.free_scenes import free_scenes
    by_name = {name: (name, scene, cfg) for name, scene, cfg in free_scenes()}
    return [by_name[n] for n in TEXEL_FREE_SCENES]


def compute(render_aovs, build_skin_scene) -> dict:
    out = {}
    for name, seed, kind, pose, over in RENDER_CASES:
        scene = build_skin_scene(synth_skin(seed, kind), pose)
        for rng_mode in (0, 1):
            out[f"{name}/rng{rng_mode}"] = digest(render_aovs(scene, make_config(**over, rng_mode=rng_mode))["texel"])
    for name, scene, cfg in free_texel_scenes():
        out[f"free/{name}"] = digest(render_aovs(scene, cfg)["texel"])
    return out


def main():
    from minecraftskin_raytracer_b200 import lib
    from tests.texel_oracle import render_aovs
    PATH.write_text(json.dumps(compute(render_aovs, lib.build_skin_scene), indent=1, sort_keys=True) + "\n")
    print("wrote", PATH)


if __name__ == "__main__":
    main()

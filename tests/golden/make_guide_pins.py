"""Generates tests/golden/guide_pins.json: SHA-256 digests of the guide planes (normal, albedo) the CPU oracle of the
AOV planes (tests/guide_oracle.c) computes for tests.scenes.RENDER_CASES, with the std::mt19937 streams (rng_mode 0) and
the counter-based ones (rng_mode 1).  They pin that oracle as it stands; the planes themselves are checked against the
unmodified reference at one sample per pixel (tests/test_aov_guides_host.py) and the GPU against the oracle.

    python tests/golden/make_guide_pins.py
"""
import json
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from minecraftskin_raytracer_b200.scene import synth_skin  # noqa: E402
from tests.golden.make_oracle_pins import digest  # noqa: E402
from tests.scenes import RENDER_CASES, make_config  # noqa: E402

PATH = Path(__file__).with_name("guide_pins.json")
PLANES = ("normal", "albedo")


def compute(render_aovs, build_skin_scene) -> dict:
    out = {}
    for name, seed, kind, pose, over in RENDER_CASES:
        scene = build_skin_scene(synth_skin(seed, kind), pose)
        for rng_mode in (0, 1):
            planes = render_aovs(scene, make_config(**over, rng_mode=rng_mode), guides=True)
            out[f"{name}/rng{rng_mode}"] = {p: digest(planes[p]) for p in PLANES}
    return out


def main():
    from minecraftskin_raytracer_b200 import lib
    from tests.guide_oracle import render_aovs
    PATH.write_text(json.dumps(compute(render_aovs, lib.build_skin_scene), indent=1, sort_keys=True) + "\n")
    print("wrote", PATH)


if __name__ == "__main__":
    main()

"""Generates tests/golden/free_scene_pins.json: SHA-256 digests of every free scene (tests/free_scenes.py) — the scene's
bytes and config, so the generator stays deterministic — and of what the CPU oracle computes for it: the frame, its
intersectScene count and the hit ids at pixel centres.  Like oracle_pins.json they pin the oracle as it stands.

    python tests/golden/make_free_scene_pins.py
"""
import ctypes as C
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from tests.golden.make_oracle_pins import digest  # noqa: E402

PATH = Path(__file__).with_name("free_scene_pins.json")


def scene_config_digest(scene, cfg) -> str:
    scalars = np.array(list(scene.light_pos) + list(scene.light_color) + [scene.light_radius] + list(scene.cam_pos) +
                       list(scene.cam_target) + list(scene.cam_up) + [scene.cam_fov_deg] + list(scene.background),
                       dtype=np.float32)
    return digest(scene.boxes, scene.texels, scalars, np.frombuffer(C.string_at(C.addressof(cfg), C.sizeof(cfg)), dtype=np.uint8))


def compute(oracle, scenes) -> dict:
    out = {}
    for name, scene, cfg in scenes:
        img, cnt = oracle.render(scene, cfg, counters=True)
        out[name] = {"input": scene_config_digest(scene, cfg), "image": digest(img), "calls": cnt["n_intersect_scene"],
                     "tri_id": digest(oracle.aov(scene, cfg))}
    return out


def main():
    from oracle.harness import Oracle
    from tests.free_scenes import free_scenes
    PATH.write_text(json.dumps(compute(Oracle(), free_scenes()), indent=1, sort_keys=True) + "\n")
    print("wrote", PATH)


if __name__ == "__main__":
    main()

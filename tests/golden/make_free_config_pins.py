"""Generates tests/golden/free_config_pins.json: SHA-256 digests of every free configuration (tests/free_configs.py) — the
scene's bytes and config, so the generator stays deterministic — and of what the CPU oracle computes for it: the frame's
float bits, its 8-bit bytes (kept apart: a NaN channel changes the first and not the second), its intersectScene count,
and whether the frame equals its twin's ("equal" / "differs"; absent for a configuration without a twin).  Like
oracle_pins.json they pin the oracle as it stands.

    python tests/golden/make_free_config_pins.py
"""
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from tests.golden.make_free_scene_pins import scene_config_digest  # noqa: E402
from tests.golden.make_oracle_pins import digest  # noqa: E402

PATH = Path(__file__).with_name("free_config_pins.json")


def same_bits(a, b) -> bool:
    return np.array_equal(a.view(np.uint32), b.view(np.uint32))


def compute(oracle, cases) -> dict:
    out = {}
    for c in cases:
        img, cnt = oracle.render(c.scene, c.cfg, counters=True)
        pin = {"input": scene_config_digest(c.scene, c.cfg), "image": digest(img), "u8": digest(oracle.quantize(img)),
               "calls": cnt["n_intersect_scene"]}
        if c.twin is not None:
            pin["twin"] = "equal" if same_bits(img, oracle.render(*c.twin)) else "differs"
        out[c.name] = pin
    return out


def main():
    from oracle.harness import Oracle
    from tests.free_configs import free_configs
    PATH.write_text(json.dumps(compute(Oracle(), free_configs()), indent=1, sort_keys=True) + "\n")
    print("wrote", PATH)


if __name__ == "__main__":
    main()

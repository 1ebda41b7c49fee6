"""The CPU oracle of all six AOV planes, texel plane included (tests/texel_oracle.c, built around the unmodified
oracle/mcskin_oracle.c), and its ctypes front-end.  The library is compiled on first use into a temporary directory with
the oracle's own flags."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile
from functools import lru_cache
from pathlib import Path

import numpy as np

from minecraftskin_raytracer_b200 import _abi

ROOT = Path(__file__).resolve().parent.parent
SOURCES = [ROOT / "tests" / "texel_oracle.c", ROOT / "oracle" / "mcskin_oracle.c", ROOT / "oracle" / "mcskin_oracle.h",
           ROOT / "include" / "mcskin_cuda.h"]
# oracle/Makefile's CFLAGS: x86-64 baseline, no FMA contraction, no fast-math
CFLAGS = ["-O2", "-std=gnu99", "-fPIC", "-fno-fast-math", "-ffp-contract=off", "-shared"]
PLANES = ("coverage", "depth", "tri_id", "normal", "albedo", "texel")


@lru_cache(maxsize=None)
def _lib() -> C.CDLL:
    h = hashlib.sha1(" ".join(CFLAGS).encode())
    for p in SOURCES:
        h.update(p.read_bytes())
    out = Path(tempfile.gettempdir()) / f"mcskin_texel_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so"
    if not out.exists():
        cc = os.environ.get("CC") or shutil.which("cc") or shutil.which("gcc")
        if cc is None:
            raise RuntimeError("no C compiler for the texel oracle")
        tmp = out.with_name(out.name + f".{os.getpid()}")
        subprocess.run([cc, *CFLAGS, "-I", str(ROOT / "include"), "-I", str(ROOT / "oracle"), "-o", str(tmp),
                        str(SOURCES[0]), "-lm", "-lpthread"], check=True)
        os.replace(tmp, out)
    lib = C.CDLL(str(out))
    lib.texelorc_render_aovs.restype = C.c_int32
    return lib


def render_aovs(scene, cfg) -> dict:
    """All six planes of the frame `cfg` describes: "coverage", "depth" float32 [H, W], "tri_id" int32 [H, W], "normal"
    float32 [H, W, 3], "albedo" float32 [H, W, 4] and "texel" int32 [H, W].  Raises if the restated texel of any hit
    disagrees with the oracle's own intersection (its colour or its face)."""
    h, w = max(cfg.height, 0), max(cfg.width, 0)
    planes = {"coverage": np.zeros((h, w), dtype=np.float32), "depth": np.zeros((h, w), dtype=np.float32),
              "tri_id": np.zeros((h, w), dtype=np.int32), "normal": np.zeros((h, w, 3), dtype=np.float32),
              "albedo": np.zeros((h, w, 4), dtype=np.float32), "texel": np.zeros((h, w), dtype=np.int32)}
    targets = _abi.McAovTargets(**{p: planes[p].ctypes.data for p in PLANES})
    cs = scene.as_c()
    rc = _lib().texelorc_render_aovs(C.byref(cs), C.byref(cfg), C.byref(targets))
    if rc != 0:
        raise RuntimeError(f"texel oracle failed: {rc} (a restated texel disagrees with the oracle's hit; see stderr)")
    return planes

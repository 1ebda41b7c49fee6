"""The CPU oracle of the AOV planes (tests/aov_oracle.c, built around the unmodified oracle/mcskin_oracle.c) and its
ctypes front-end.  The library is compiled on first use into a temporary directory with the oracle's own flags."""
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
SOURCES = [ROOT / "tests" / "aov_oracle.c", ROOT / "oracle" / "mcskin_oracle.c", ROOT / "oracle" / "mcskin_oracle.h",
           ROOT / "include" / "mcskin_cuda.h"]
# oracle/Makefile's CFLAGS: x86-64 baseline, no FMA contraction, no fast-math
CFLAGS = ["-O2", "-std=gnu99", "-fPIC", "-fno-fast-math", "-ffp-contract=off", "-shared"]


@lru_cache(maxsize=None)
def _lib() -> C.CDLL:
    h = hashlib.sha1(" ".join(CFLAGS).encode())
    for p in SOURCES:
        h.update(p.read_bytes())
    out = Path(tempfile.gettempdir()) / f"mcskin_aov_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so"
    if not out.exists():
        cc = os.environ.get("CC") or shutil.which("cc") or shutil.which("gcc")
        if cc is None:
            raise RuntimeError("no C compiler for the AOV oracle")
        tmp = out.with_name(out.name + f".{os.getpid()}")
        subprocess.run([cc, *CFLAGS, "-I", str(ROOT / "include"), "-I", str(ROOT / "oracle"), "-o", str(tmp),
                        str(SOURCES[0]), "-lm", "-lpthread"], check=True)
        os.replace(tmp, out)
    lib = C.CDLL(str(out))
    lib.aovorc_render_aovs.restype = C.c_int32
    return lib


def render_aovs(scene, cfg) -> dict:
    """{"coverage": float32 [H, W], "depth": float32 [H, W], "tri_id": int32 [H, W]} of the frame `cfg` describes."""
    h, w = max(cfg.height, 0), max(cfg.width, 0)
    planes = {"coverage": np.zeros((h, w), dtype=np.float32), "depth": np.zeros((h, w), dtype=np.float32),
              "tri_id": np.zeros((h, w), dtype=np.int32)}
    targets = _abi.McAovTargets(planes["coverage"].ctypes.data, planes["depth"].ctypes.data, planes["tri_id"].ctypes.data)
    cs = scene.as_c()
    rc = _lib().aovorc_render_aovs(C.byref(cs), C.byref(cfg), C.byref(targets))
    if rc != 0:
        raise RuntimeError(f"AOV oracle failed: {rc}")
    return planes

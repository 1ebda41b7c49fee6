"""TEST INFRASTRUCTURE ONLY — ctypes front-ends of the two CPU checkers.

* `Oracle`    : oracle/libmcskin_oracle.so, the plain-C restatement (mcskin_oracle.c).
                Built on demand with gcc (present on the GPU box too).
* `Reference` : oracle/_ref/libmcskin_ref.so, the UNMODIFIED reference core behind
                ref_shim.cpp.  Built by oracle/build_ref.sh from a checkout of the
                reference (not part of this repository): the one MCSKIN_REFERENCE_DIR
                names, else `reference` beside this repository.  None when absent.

Both expose the same operations on the flat PODs of include/mcskin_cuda.h.
"""
from __future__ import annotations

import ctypes as C
import fcntl
import hashlib
import os
import subprocess
from pathlib import Path

import numpy as np

from minecraftskin_raytracer_b200 import _abi
from minecraftskin_raytracer_b200.scene import FlatScene, pose_array

HERE = Path(__file__).resolve().parent
ORACLE_SO = HERE / "libmcskin_oracle.so"
REF_SO = HERE / "_ref" / "libmcskin_ref.so"
# where the reference is looked for when MCSKIN_REFERENCE_DIR is not set: a checkout named `reference` beside this repository
DEFAULT_REFERENCE_DIR = HERE.parent.parent / "reference"

COUNTER_FIELDS = [
    "n_intersect_scene", "n_primary_rays", "n_retests", "n_shadow_rays", "n_ao_rays", "n_reflect_rays",
    "n_box_tests_plain", "n_box_tests_rotated", "n_slab_pass", "n_backface_eval", "n_rotated_hits",
    "n_background_primary", "n_shade", "n_soft_shadow", "n_hard_shadow",
]


class McOracleCounters(C.Structure):
    _fields_ = [(name, C.c_int64) for name in COUNTER_FIELDS]

    def as_dict(self) -> dict:
        return {name: int(getattr(self, name)) for name in COUNTER_FIELDS}


def _oracle_digest() -> str:
    h = hashlib.sha1()
    for path in (HERE / "mcskin_oracle.c", HERE / "mcskin_oracle.h", HERE / "Makefile", HERE.parent / "include" / "mcskin_cuda.h"):
        h.update(path.read_bytes())
    return h.hexdigest()


def build_oracle(force: bool = False) -> Path:
    """gcc build of the C restatement; content-hashed and locked so parallel test workers and
    torchrun ranks do not rebuild it on top of each other."""
    stamp = HERE / ".oracle.hash"

    def stale():
        return not ORACLE_SO.exists() or not stamp.exists() or stamp.read_text().strip() != _oracle_digest()

    if not force and not stale():
        return ORACLE_SO
    with open(HERE / ".oracle.lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if force or stale():
                tmp = HERE / f".libmcskin_oracle.{os.getpid()}.so"
                subprocess.run(["make", "-C", str(HERE), "-B", "libmcskin_oracle.so", f"OUT={tmp.name}"], check=True,
                               capture_output=True)
                os.replace(tmp, ORACLE_SO)
                stamp.write_text(_oracle_digest())
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return ORACLE_SO


def reference_dir() -> Path | None:
    """The checkout of the reference to build the checker from: MCSKIN_REFERENCE_DIR when set (an error when it names
    no checkout), else DEFAULT_REFERENCE_DIR when it holds one, else None."""
    env = os.environ.get("MCSKIN_REFERENCE_DIR")
    if env:
        if not (Path(env) / "src").is_dir():
            raise RuntimeError(f"MCSKIN_REFERENCE_DIR={env} is not a checkout of the reference (no src/)")
        return Path(env)
    try:
        return DEFAULT_REFERENCE_DIR if (DEFAULT_REFERENCE_DIR / "src").is_dir() else None
    except OSError:  # e.g. a parent directory this user may not enter: not present
        return None


def build_reference() -> Path | None:
    """Compiles oracle/_ref when a checkout of the reference is found (reference_dir); returns the .so path or None."""
    ref = reference_dir()
    if ref is not None:
        subprocess.run(["bash", str(HERE / "build_ref.sh")], check=True, capture_output=True,
                       env={**os.environ, "MCSKIN_REFERENCE_DIR": str(ref)})
    return REF_SO if REF_SO.exists() else None


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a.reshape(shape) if shape is not None else a


def _ptr(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


def rays_array(origins, dirs) -> np.ndarray:
    origins = _f32(origins).reshape(-1, 3)
    dirs = _f32(dirs).reshape(-1, 3)
    r = np.zeros(len(origins), dtype=_abi.RAY_DTYPE)
    r["origin"] = origins
    r["dir"] = dirs
    return r


class _Common:
    """Operations shared by both checkers; subclasses bind `_call(name, scene, *args)`."""

    def intersect(self, scene, rays: np.ndarray, box: int = -1) -> np.ndarray:
        rays = np.ascontiguousarray(rays, dtype=_abi.RAY_DTYPE)
        out = np.zeros(len(rays), dtype=_abi.HIT_DTYPE)
        self._call("intersect", scene, C.c_int32(box), _ptr(rays, _abi.McRay), C.c_int32(len(rays)),
                   _ptr(out, _abi.McHit))
        return out

    def trace(self, scene, cfg, rays, depth=0, use_config=True) -> np.ndarray:
        rays = np.ascontiguousarray(rays, dtype=_abi.RAY_DTYPE)
        out = np.zeros((len(rays), 4), dtype=np.float32)
        self._call("trace", scene, C.byref(cfg), C.c_int32(int(use_config)), C.c_int32(depth),
                   _ptr(rays, _abi.McRay), C.c_int32(len(rays)), _ptr(out, C.c_float))
        return out

    def shade(self, scene, cfg, hits, view_dirs, shadow_factors=None) -> np.ndarray:
        hits = np.ascontiguousarray(hits, dtype=_abi.HIT_DTYPE)
        view_dirs = _f32(view_dirs, (-1, 3))
        sf = None if shadow_factors is None else _f32(shadow_factors)
        out = np.zeros((len(hits), 4), dtype=np.float32)
        self._call("shade", scene, C.byref(cfg), _ptr(hits, _abi.McHit), _ptr(view_dirs, C.c_float),
                   None if sf is None else _ptr(sf, C.c_float), C.c_int32(len(hits)), _ptr(out, C.c_float))
        return out

    def in_shadow(self, scene, points, normals, lights) -> np.ndarray:
        p, n, l = _f32(points, (-1, 3)), _f32(normals, (-1, 3)), _f32(lights, (-1, 3))
        out = np.zeros(len(p), dtype=np.int32)
        self._call("in_shadow", scene, _ptr(p, C.c_float), _ptr(n, C.c_float), _ptr(l, C.c_float),
                   C.c_int32(len(p)), _ptr(out, C.c_int32))
        return out

    def soft_shadow(self, scene, points, normals, seeds, samples) -> np.ndarray:
        p, n = _f32(points, (-1, 3)), _f32(normals, (-1, 3))
        s = np.ascontiguousarray(seeds, dtype=np.uint32)
        out = np.zeros(len(p), dtype=np.float32)
        self._call("soft_shadow", scene, _ptr(p, C.c_float), _ptr(n, C.c_float), _ptr(s, C.c_uint32),
                   C.c_int32(samples), C.c_int32(len(p)), _ptr(out, C.c_float))
        return out

    def ambient_occlusion(self, scene, points, normals, seeds, samples, radius) -> np.ndarray:
        p, n = _f32(points, (-1, 3)), _f32(normals, (-1, 3))
        s = np.ascontiguousarray(seeds, dtype=np.uint32)
        out = np.zeros(len(p), dtype=np.float32)
        self._call("ambient_occlusion", scene, _ptr(p, C.c_float), _ptr(n, C.c_float), _ptr(s, C.c_uint32),
                   C.c_int32(samples), C.c_float(radius), C.c_int32(len(p)), _ptr(out, C.c_float))
        return out

    def generate_rays(self, scene, aspect, uv) -> np.ndarray:
        uv = _f32(uv, (-1, 2))
        out = np.zeros(len(uv), dtype=_abi.RAY_DTYPE)
        self._call("generate_rays", scene, C.c_float(aspect), _ptr(uv, C.c_float), C.c_int32(len(uv)),
                   _ptr(out, _abi.McRay))
        return out

    def background(self, scene, cfg, uv, use_config=True) -> np.ndarray:
        uv = _f32(uv, (-1, 2))
        out = np.zeros((len(uv), 4), dtype=np.float32)
        self._call("background", scene, C.byref(cfg), C.c_int32(int(use_config)), _ptr(uv, C.c_float),
                   C.c_int32(len(uv)), _ptr(out, C.c_float))
        return out

    def aov(self, scene, cfg) -> np.ndarray:
        out = np.zeros((cfg.height, cfg.width), dtype=np.int32)
        self._call("aov", scene, C.byref(cfg), _ptr(out, C.c_int32))
        return out

    def generate_tiles(self, w, h, tile_size) -> np.ndarray:
        fn = getattr(self.lib, self.prefix + "generate_tiles")
        fn.restype = C.c_int32
        n = fn(C.c_int32(w), C.c_int32(h), C.c_int32(tile_size), None, C.c_int32(0))
        out = np.zeros(n, dtype=_abi.TILE_DTYPE)
        if n:
            fn(C.c_int32(w), C.c_int32(h), C.c_int32(tile_size), _ptr(out, _abi.McTile), C.c_int32(n))
        return out


class Oracle(_Common):
    prefix = "mcorc_"

    def __init__(self):
        self.lib = C.CDLL(str(build_oracle()))
        self.lib.mcorc_seed_cast.restype = C.c_uint32
        self.lib.mcorc_seed_cast.argtypes = [C.c_float]

    def _call(self, name, scene: FlatScene, *args):
        fn = getattr(self.lib, self.prefix + name)
        fn.restype = C.c_int32
        cs = scene.as_c()
        rc = fn(C.byref(cs), *args)
        if rc != 0:
            raise RuntimeError(f"oracle {name} failed: {rc}")

    def render(self, scene: FlatScene, cfg, threads: int = 0, counters: bool = False):
        out = np.zeros((max(cfg.height, 0), max(cfg.width, 0), 4), dtype=np.float32)
        cnt = McOracleCounters()
        cs = scene.as_c()
        self.lib.mcorc_render.restype = C.c_int32
        rc = self.lib.mcorc_render(C.byref(cs), C.byref(cfg), C.c_int32(threads), _ptr(out, C.c_float), C.byref(cnt))
        if rc != 0:
            raise RuntimeError(f"oracle render failed: {rc}")
        return (out, cnt.as_dict()) if counters else out

    def render_tile(self, scene, cfg, tile, image: np.ndarray) -> np.ndarray:
        image = np.ascontiguousarray(image, dtype=np.float32)
        t = _abi.McTile(*[int(v) for v in tile])
        cs = scene.as_c()
        self.lib.mcorc_render_tile(C.byref(cs), C.byref(cfg), C.byref(t), _ptr(image, C.c_float))
        return image

    def quantize(self, rgba: np.ndarray) -> np.ndarray:
        rgba = np.ascontiguousarray(rgba, dtype=np.float32)
        out = np.zeros(rgba.shape, dtype=np.uint8)
        self.lib.mcorc_quantize(_ptr(rgba, C.c_float), C.c_int64(rgba.size), _ptr(out, C.c_uint8))
        return out

    def mt19937(self, seed: int, n: int):
        u = np.zeros(n, dtype=np.uint32)
        f = np.zeros(n, dtype=np.float32)
        self.lib.mcorc_mt19937(C.c_uint32(seed), C.c_int32(n), _ptr(u, C.c_uint32), _ptr(f, C.c_float))
        return u, f

    def seed_cast(self, f: float) -> int:
        return int(self.lib.mcorc_seed_cast(C.c_float(f)))

    def hardware_threads(self) -> int:
        return int(self.lib.mcorc_hardware_threads())


class Reference(_Common):
    """The unmodified reference (oracle/_ref).  Scenes are rebuilt as real `Scene` objects."""
    prefix = "mcref_"

    def __init__(self, path: Path = REF_SO):
        self.lib = C.CDLL(str(path))
        for name in ("mcref_scene_from_flat", "mcref_scene_from_atlas", "mcref_default_scene"):
            getattr(self.lib, name).restype = C.c_void_p
        self.lib.mcref_scene_free.argtypes = [C.c_void_p]
        self._cache: dict[int, tuple[FlatScene, int]] = {}

    @classmethod
    def load(cls) -> "Reference | None":
        return cls() if REF_SO.exists() else None

    # -- scene handles -------------------------------------------------------
    def _handle(self, scene: FlatScene) -> int:
        key = id(scene)
        hit = self._cache.get(key)
        if hit is not None and hit[0] is scene:
            return hit[1]
        cs = scene.as_c()
        h = self.lib.mcref_scene_from_flat(C.byref(cs))
        if not h:
            raise RuntimeError("mcref_scene_from_flat failed")
        if len(self._cache) > 64:
            for _, (_, old) in self._cache.items():
                self.lib.mcref_scene_free(C.c_void_p(old))
            self._cache.clear()
        self._cache[key] = (scene, h)
        return h

    def _flatten_handle(self, h) -> FlatScene:
        boxes = np.zeros(64, dtype=_abi.BOX_DTYPE)
        texels = np.zeros((8192, 4), dtype=np.float32)
        cs = _abi.McScene()
        self.lib.mcref_scene_flatten.restype = C.c_int32
        rc = self.lib.mcref_scene_flatten(C.c_void_p(h), _ptr(boxes, _abi.McBox), C.c_int32(len(boxes)),
                                          _ptr(texels, C.c_float), C.c_int32(len(texels)), C.byref(cs))
        if rc != 0:
            raise RuntimeError("mcref_scene_flatten: capacity")
        return FlatScene.from_c(cs)

    def scene_from_atlas(self, atlas: np.ndarray, pose=None) -> FlatScene:
        """SkinParser::parse + MeshBuilder::buildScene by the reference itself, flattened."""
        atlas = np.ascontiguousarray(atlas, dtype=np.uint8)
        p = pose_array(pose)
        h = self.lib.mcref_scene_from_atlas(_ptr(atlas, C.c_uint8), C.c_int32(atlas.shape[1]),
                                            C.c_int32(atlas.shape[0]), None if p is None else _ptr(p, C.c_float))
        if not h:
            raise RuntimeError("reference SkinParser::parse rejected the atlas")
        try:
            return self._flatten_handle(h)
        finally:
            self.lib.mcref_scene_free(C.c_void_p(h))

    def default_scene(self, pose=None) -> FlatScene:
        p = pose_array(pose)
        h = self.lib.mcref_default_scene(None if p is None else _ptr(p, C.c_float))
        try:
            return self._flatten_handle(h)
        finally:
            self.lib.mcref_scene_free(C.c_void_p(h))

    def builtin_poses(self) -> np.ndarray:
        n = self.lib.mcref_builtin_pose_count()
        out = np.zeros((n, 12), dtype=np.float32)
        for i in range(n):
            self.lib.mcref_builtin_pose(C.c_int32(i), _ptr(out[i], C.c_float))
        return out

    def _call(self, name, scene: FlatScene, *args):
        fn = getattr(self.lib, self.prefix + name)
        fn.restype = C.c_int32
        rc = fn(C.c_void_p(self._handle(scene)), *args)
        if rc != 0:
            raise RuntimeError(f"reference {name} failed: {rc}")

    def render(self, scene: FlatScene, cfg, counters: bool = False):
        out = np.zeros((max(cfg.height, 0), max(cfg.width, 0), 4), dtype=np.float32)
        out[..., 3] = 1.0
        calls = C.c_longlong(0)
        self.lib.mcref_render.restype = C.c_int32
        errs = self.lib.mcref_render(C.c_void_p(self._handle(scene)), C.byref(cfg), _ptr(out, C.c_float),
                                     C.byref(calls) if counters else None)
        if errs != 0:
            raise RuntimeError(f"reference render recorded {errs} tile errors")
        return (out, int(calls.value)) if counters else out

    def render_tile(self, scene, cfg, tile, image: np.ndarray) -> np.ndarray:
        image = np.ascontiguousarray(image, dtype=np.float32)
        t = _abi.McTile(*[int(v) for v in tile])
        self.lib.mcref_render_tile(C.c_void_p(self._handle(scene)), C.byref(cfg), C.byref(t), _ptr(image, C.c_float))
        return image

    def mt19937(self, seed: int, n: int):
        u = np.zeros(n, dtype=np.uint32)
        f = np.zeros(n, dtype=np.float32)
        self.lib.mcref_mt19937(C.c_uint32(seed), C.c_int32(n), _ptr(u, C.c_uint32), _ptr(f, C.c_float))
        return u, f

    def seed_cast(self, f: float) -> int:
        self.lib.mcref_seed_cast.restype = C.c_uint32
        self.lib.mcref_seed_cast.argtypes = [C.c_float]
        return int(self.lib.mcref_seed_cast(C.c_float(f)))

    def write_png(self, rgba: np.ndarray, path: str) -> bool:
        rgba = np.ascontiguousarray(rgba, dtype=np.float32)
        h, w = rgba.shape[:2]
        return bool(self.lib.mcref_write_png(_ptr(rgba, C.c_float), C.c_int32(w), C.c_int32(h), path.encode()))

    def hardware_threads(self) -> int:
        return int(self.lib.mcref_hardware_threads())

"""Loader and typed front-end of libmcskin_cuda.so (the C ABI of include/mcskin_cuda.h).

The CUDA extension is the product: there is no CPU fallback here.  If the shared
library is missing the import of this module raises; if no CUDA device is present,
every compute call raises McSkinError(MC_ERR_NO_DEVICE).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from . import _abi
from ._abi import McConfig, McContext_p, McHit, McRay, McRenderStats, McScene, McTile  # noqa: F401
from .scene import FlatScene, pose_array

import os

# MCSKIN_LIB selects an alternative build of the same library (kernel tuning experiments)
LIB_PATH = Path(os.environ.get("MCSKIN_LIB") or (Path(__file__).resolve().parent / "_lib" / "libmcskin_cuda.so"))

# streams a frame's tile rows are dealt to by default (McOptions::frameLanes in csrc/capi_internal.hpp)
DEFAULT_FRAME_LANES = 2

# every symbol include/mcskin_cuda.h declares
EXPORTS = [
    "mcskin_config_defaults", "mcskin_counter_word", "mcskin_host_copy_rows", "mcskin_generate_tiles", "mcskin_cuda_device_count", "mcskin_cuda_last_error",
    "mcskin_cuda_abi_version", "mcskin_cuda_abi_sizes", "mcskin_cuda_render", "mcskin_cuda_render_tile",
    "mcskin_cuda_render_multi", "mcskin_cuda_context_create", "mcskin_cuda_context_destroy",
    "mcskin_cuda_context_set_scene", "mcskin_cuda_context_render_bands", "mcskin_cuda_band_rows",
    "mcskin_cuda_context_sync", "mcskin_cuda_context_set_option", "mcskin_cuda_context_render_batch",
    "mcskin_cuda_intersect", "mcskin_cuda_trace", "mcskin_cuda_shade", "mcskin_cuda_in_shadow",
    "mcskin_cuda_soft_shadow", "mcskin_cuda_ambient_occlusion", "mcskin_cuda_generate_rays",
    "mcskin_cuda_background", "mcskin_cuda_aov", "mcskin_build_skin_scene", "mcskin_cuda_sincos",
    "mcskin_sincos_model", "mcskin_cuda_powf", "mcskin_powf_model", "mcskin_cuda_context_render_rows_into_frame",
    "mcskin_cuda_device_alloc", "mcskin_cuda_device_free", "mcskin_cuda_ipc_export", "mcskin_cuda_ipc_open",
    "mcskin_cuda_ipc_close", "mcskin_cuda_fp32_issue_peak", "mcskin_cuda_peer_signal", "mcskin_cuda_peer_wait",
    "mcskin_primary_launch_order", "mcskin_cuda_context_render_tiles_into_frame", "mcskin_partition_tiles",
    "mcskin_cuda_host_register", "mcskin_cuda_host_unregister", "mcskin_cuda_render_batch_multi",
    "mcskin_cuda_enable_peer_access", "mcskin_cuda_context_render_scene_tiles",
    "mcskin_cuda_context_debug_block_times", "mcskin_cuda_context_render_skin_batch",
    "mcskin_skin_layout", "mcskin_cuda_render_aovs", "mcskin_cuda_context_set_aov_targets",
]


class McSkinError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"mcskin_cuda error {code}: {message}")
        self.code = code
        self.message = message


def _load() -> C.CDLL:
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA extension first "
            "(python -c 'import __graft_entry__ as g; g.build()').  There is no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    lib.mcskin_cuda_last_error.restype = C.c_char_p
    for name in EXPORTS:
        fn = getattr(lib, name)  # raises AttributeError if a declared symbol is not exported
        if name not in ("mcskin_cuda_last_error", "mcskin_config_defaults", "mcskin_cuda_context_destroy",
                        "mcskin_cuda_abi_sizes"):
            fn.restype = C.c_int32
    lib.mcskin_config_defaults.restype = None
    lib.mcskin_cuda_context_destroy.restype = None
    lib.mcskin_cuda_abi_sizes.restype = None
    lib.mcskin_counter_word.restype = C.c_uint32
    lib.mcskin_counter_word.argtypes = [C.c_uint32, C.c_uint32]
    return lib


_lib = _load()


def raw() -> C.CDLL:
    return _lib


def last_error() -> str:
    return (_lib.mcskin_cuda_last_error() or b"").decode("utf-8", "replace")


def _check(rc: int):
    if rc != 0:
        raise McSkinError(rc, last_error())


def _ptr(a: np.ndarray, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a.reshape(shape) if shape is not None else a


def device_count() -> int:
    return int(_lib.mcskin_cuda_device_count())


def abi_sizes() -> list[int]:
    out = (C.c_int32 * 8)()
    _lib.mcskin_cuda_abi_sizes(out)
    return list(out)


def config_defaults() -> McConfig:
    cfg = McConfig()
    _lib.mcskin_config_defaults(C.byref(cfg))
    return cfg


def counter_word(seed: int, k: int) -> int:
    """Word k of the counter-based stream seeded `seed` (McConfig.rng_mode 1; mc_rng_counter_word in mcskin_cuda.h)."""
    return int(_lib.mcskin_counter_word(seed & 0xFFFFFFFF, k & 0xFFFFFFFF))


def host_copy_rows(dst: np.ndarray, src: np.ndarray, row_bytes: int, rows: int, pieces: int = 8,
                   dst_pitch: int | None = None, src_pitch: int | None = None):
    """mcskin_host_copy_rows over two byte arrays (the library's host copy threads; no device needed)."""
    _check(_lib.mcskin_host_copy_rows(C.c_void_p(dst.ctypes.data), C.c_void_p(src.ctypes.data),
                                      C.c_uint64(row_bytes if dst_pitch is None else dst_pitch),
                                      C.c_uint64(row_bytes if src_pitch is None else src_pitch),
                                      C.c_uint64(row_bytes), C.c_uint64(rows), C.c_int32(pieces)))


def generate_tiles(width: int, height: int, tile_size: int) -> np.ndarray:
    """TileRenderer::generateTiles (tile_renderer.cpp:18-39) as a structured array."""
    n = _lib.mcskin_generate_tiles(C.c_int32(width), C.c_int32(height), C.c_int32(tile_size), None, C.c_int32(0))
    out = np.zeros(n, dtype=_abi.TILE_DTYPE)
    if n:
        _lib.mcskin_generate_tiles(C.c_int32(width), C.c_int32(height), C.c_int32(tile_size),
                                   _ptr(out, McTile), C.c_int32(n))
    return out


def build_skin_scene(atlas: np.ndarray, pose=None) -> FlatScene:
    """SkinParser::parse + MeshBuilder::buildScene for an RGBA8 atlas [H,64,4] (host-side C++)."""
    atlas = np.ascontiguousarray(atlas, dtype=np.uint8)
    if atlas.ndim != 3 or atlas.shape[2] != 4:
        raise ValueError("atlas must be uint8 [H, W, 4]")
    p = pose_array(pose)
    boxes = np.zeros(12, dtype=_abi.BOX_DTYPE)
    texels = np.zeros((4096, 4), dtype=np.float32)
    cs = McScene()
    _check(_lib.mcskin_build_skin_scene(_ptr(atlas, C.c_uint8), C.c_int32(atlas.shape[1]), C.c_int32(atlas.shape[0]),
                                        None if p is None else _ptr(p, C.c_float), _ptr(boxes, _abi.McBox),
                                        _ptr(texels, C.c_float), C.byref(cs)))
    return FlatScene.from_c(cs)


def skin_layout(atlas: np.ndarray, pose=None):
    """mcskin_skin_layout: (boxes, faces [n, 6] = (dst, x, y, w, h, mirror), box_opaque, n_texels) of a skin — its flat
    scene without the float texels (host code)."""
    atlas = np.ascontiguousarray(atlas, dtype=np.uint8)
    p = pose_array(pose)
    boxes = np.zeros(12, dtype=_abi.BOX_DTYPE)
    faces = np.zeros((72, 6), dtype=np.int32)
    opaque = np.zeros(12, dtype=np.uint8)
    n_faces = C.c_int32(0)
    cs = McScene()
    _check(_lib.mcskin_skin_layout(_ptr(atlas, C.c_uint8), C.c_int32(atlas.shape[1]), C.c_int32(atlas.shape[0]),
                                   None if p is None else _ptr(p, C.c_float), _ptr(boxes, _abi.McBox), _ptr(faces, C.c_int32),
                                   C.byref(n_faces), _ptr(opaque, C.c_uint8), C.byref(cs)))
    return boxes[:cs.n_boxes].copy(), faces[:n_faces.value].copy(), opaque[:cs.n_boxes].copy(), int(cs.n_texels)


# ---------------------------------------------------------------- whole-frame calls
def render(scene, cfg: McConfig, device: int = 0, want_f32: bool = True, want_u8: bool = False,
           progress=None, multi_devices: int = 0, out_f32: np.ndarray | None = None, out_u8: np.ndarray | None = None):
    """mcskin_cuda_render: host scene in, host image(s) out.  Returns (f32|None, u8|None, stats dict).

    scene: a FlatScene, or its C view (FlatScene.as_c(), for callers that render the same scene object again and again).
    out_f32 / out_u8: caller-owned [H, W, 4] arrays to render into (reused across frames; page-locked
    arrays, e.g. numpy views of torch pin_memory tensors, are filled by DMA without a staging copy)."""
    h, w = max(cfg.height, 0), max(cfg.width, 0)

    def _buffer(given, want, dtype, one):
        if given is not None:
            if given.shape != (h, w, 4) or given.dtype != dtype or not given.flags.c_contiguous:
                raise ValueError(f"output buffer must be C-contiguous {dtype} [{h}, {w}, 4]")
            return given
        if not want:
            return None
        buf = np.empty((h, w, 4), dtype=dtype)
        n_tiles = len(generate_tiles(cfg.width, cfg.height, cfg.tile_size)) if (w and h) else 0
        if n_tiles == 0 and buf.size:  # nothing is rendered: Image(w,h) pixels stay (0,0,0,1) (image.h:15, color.h:8)
            buf[...] = 0
            buf[..., 3] = one
        return buf

    f32 = _buffer(out_f32, want_f32, np.float32, 1.0)
    u8 = _buffer(out_u8, want_u8, np.uint8, 255)
    stats = McRenderStats()
    cs = scene.as_c() if isinstance(scene, FlatScene) else scene
    if multi_devices and multi_devices > 0:
        _check(_lib.mcskin_cuda_render_multi(C.byref(cs), C.byref(cfg), C.c_int32(multi_devices),
                                             None if f32 is None else _ptr(f32, C.c_float),
                                             None if u8 is None else _ptr(u8, C.c_uint8), C.byref(stats)))
    else:
        cb = _abi.McProgressFn(lambda d, t, _u: progress(d, t)) if progress else C.cast(None, _abi.McProgressFn)
        _check(_lib.mcskin_cuda_render(C.byref(cs), C.byref(cfg), C.c_int32(device),
                                       None if f32 is None else _ptr(f32, C.c_float),
                                       None if u8 is None else _ptr(u8, C.c_uint8), cb, None, C.byref(stats)))
    return f32, u8, {k: getattr(stats, k) for k, _ in McRenderStats._fields_}


def render_aovs(scene, cfg: McConfig, device: int = 0, want_u8: bool = False, guides: bool = False):
    """mcskin_cuda_render_aovs: the frame of `render` plus its AOV planes.  Returns (f32 [H, W, 4], u8 [H, W, 4] | None,
    {"coverage": float32 [H, W], "depth": float32 [H, W], "tri_id": int32 [H, W]}, stats dict).  guides: the planes also
    hold "normal" float32 [H, W, 3] and "albedo" float32 [H, W, 4]."""
    h, w = max(cfg.height, 0), max(cfg.width, 0)
    f32 = np.empty((h, w, 4), dtype=np.float32)
    u8 = np.empty((h, w, 4), dtype=np.uint8) if want_u8 else None
    n_tiles = len(generate_tiles(cfg.width, cfg.height, cfg.tile_size)) if (w and h) else 0
    if n_tiles == 0 and f32.size:  # nothing is rendered: Image(w,h) pixels stay (0,0,0,1) (image.h:15, color.h:8)
        f32[...] = 0
        f32[..., 3] = 1
        if u8 is not None:
            u8[...] = 0
            u8[..., 3] = 255
    planes = {"coverage": np.empty((h, w), dtype=np.float32), "depth": np.empty((h, w), dtype=np.float32),
              "tri_id": np.empty((h, w), dtype=np.int32)}
    if guides:
        planes["normal"] = np.empty((h, w, 3), dtype=np.float32)
        planes["albedo"] = np.empty((h, w, 4), dtype=np.float32)
    targets = _abi.McAovTargets(*(planes[p].ctypes.data for p in planes))
    stats = McRenderStats()
    cs = scene.as_c() if isinstance(scene, FlatScene) else scene
    _check(_lib.mcskin_cuda_render_aovs(C.byref(cs), C.byref(cfg), C.c_int32(device), _ptr(f32, C.c_float),
                                        None if u8 is None else _ptr(u8, C.c_uint8), C.byref(targets), C.byref(stats)))
    return f32, u8, planes, {k: getattr(stats, k) for k, _ in McRenderStats._fields_}


def render_batch_multi(scenes: list[FlatScene], cfg: McConfig, n_devices: int, want_f32: bool = True, want_u8: bool = False):
    """mcskin_cuda_render_batch_multi: a batch of skins, host scenes in, host images out, skin i on device i % n_devices.
    Returns (f32 [n, H, W, 4] | None, u8 [n, H, W, 4] | None)."""
    n, h, w = len(scenes), max(cfg.height, 0), max(cfg.width, 0)
    f32 = np.zeros((n, h, w, 4), dtype=np.float32) if want_f32 else None
    u8 = np.zeros((n, h, w, 4), dtype=np.uint8) if want_u8 else None
    arr = (McScene * n)(*[s.as_c() for s in scenes])
    _check(_lib.mcskin_cuda_render_batch_multi(arr, C.c_int32(n), C.byref(cfg), C.c_int32(n_devices),
                                               None if f32 is None else _ptr(f32, C.c_float),
                                               None if u8 is None else _ptr(u8, C.c_uint8)))
    return f32, u8


def render_tile(scene: FlatScene, cfg: McConfig, tile, image_f32: np.ndarray, device: int = 0) -> np.ndarray:
    image_f32 = np.ascontiguousarray(image_f32, dtype=np.float32)
    t = McTile(*[int(v) for v in tile])
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_render_tile(C.byref(cs), C.byref(cfg), C.c_int32(device), C.byref(t),
                                        _ptr(image_f32, C.c_float), None))
    return image_f32


class DeviceBuffer:
    """A plain cudaMalloc allocation owned by this process, shareable with the other processes of the box
    (one per GPU) through a 64-byte IPC handle.  Exposes __cuda_array_interface__ so torch can view it."""

    def __init__(self, device: int, shape, dtype=np.float32):
        self.device, self.shape, self.dtype = device, tuple(int(v) for v in shape), np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        p = C.c_void_p()
        _check(_lib.mcskin_cuda_device_alloc(C.c_int32(device), C.c_uint64(self.nbytes), C.byref(p)))
        self.ptr = int(p.value)

    @property
    def __cuda_array_interface__(self):
        return {"shape": self.shape, "typestr": self.dtype.str, "data": (self.ptr, False), "version": 2}

    def ipc_handle(self) -> bytes:
        h = (C.c_uint8 * 64)()
        _check(_lib.mcskin_cuda_ipc_export(C.c_int32(self.device), C.c_void_p(self.ptr), h))
        return bytes(h)

    def free(self):
        if self.ptr:
            _check(_lib.mcskin_cuda_device_free(C.c_int32(self.device), C.c_void_p(self.ptr)))
            self.ptr = 0


def ipc_open(device: int, handle: bytes) -> int:
    """Maps a peer process's DeviceBuffer into this process; returns the device address valid here."""
    h = (C.c_uint8 * 64)(*handle)
    p = C.c_void_p()
    _check(_lib.mcskin_cuda_ipc_open(C.c_int32(device), h, C.byref(p)))
    return int(p.value)


def enable_peer_access(device: int, peer: int):
    """Kernels on `device` may address memory allocated on `peer` afterwards (one process, several devices)."""
    _check(_lib.mcskin_cuda_enable_peer_access(C.c_int32(device), C.c_int32(peer)))


def peer_signal(device: int, d_flag: int, value: int, stream: int = 0):
    """Stream-ordered release of a 32-bit flag in (peer-mapped) device memory."""
    _check(_lib.mcskin_cuda_peer_signal(C.c_int32(device), C.c_void_p(d_flag), C.c_uint32(value & 0xffffffff), C.c_void_p(stream or None)))


def peer_wait(device: int, d_flags: int, n: int, value: int, d_timeout: int = 0, stream: int = 0):
    """Holds `stream` until the n flags at d_flags have all reached `value` (or ~2 s have passed)."""
    _check(_lib.mcskin_cuda_peer_wait(C.c_int32(device), C.c_void_p(d_flags), C.c_int32(n), C.c_uint32(value & 0xffffffff),
                                      C.c_void_p(d_timeout or None), C.c_void_p(stream or None)))


def partition_tiles(scene: FlatScene, cfg: McConfig, n_parts: int, part: int, root_part: int = -1) -> np.ndarray:
    """Frame tile indices (ty * tiles_x + tx, ascending) of `part` in the cost-balanced deal of the frame's tiles
    to n_parts renderers (host code, needs no GPU).  The parts are disjoint and cover the frame.  root_part: the part
    whose device holds the frame the others store into over NVLink (-1: none)."""
    cs = scene.as_c()
    n = _lib.mcskin_partition_tiles(C.byref(cs), C.byref(cfg), C.c_int32(n_parts), C.c_int32(part), C.c_int32(root_part), None, C.c_int32(0))
    _check(min(n, 0))
    out = np.zeros(n, dtype=np.int32)
    if n:
        _check(min(_lib.mcskin_partition_tiles(C.byref(cs), C.byref(cfg), C.c_int32(n_parts), C.c_int32(part), C.c_int32(root_part),
                                               _ptr(out, C.c_int32), C.c_int32(n)), 0))
    return out


def host_register(array: np.ndarray) -> int:
    """Page-locks a host array (e.g. a view of a shared-memory segment) and maps it into the device address
    space; returns the device address kernels can store to."""
    p = C.c_void_p()
    _check(_lib.mcskin_cuda_host_register(C.c_void_p(array.ctypes.data), C.c_uint64(array.nbytes), C.byref(p)))
    return int(p.value)


def host_unregister(array: np.ndarray):
    _check(_lib.mcskin_cuda_host_unregister(C.c_void_p(array.ctypes.data)))


def ipc_close(device: int, ptr: int):
    _check(_lib.mcskin_cuda_ipc_close(C.c_int32(device), C.c_void_p(ptr)))


class Context:
    """Device-resident renderer (McContext): scene uploaded once, output in caller-owned device memory."""

    def __init__(self, device: int = 0):
        self._h = McContext_p()
        _check(_lib.mcskin_cuda_context_create(C.c_int32(device), C.byref(self._h)))
        self.device = device
        self.cfg: McConfig | None = None

    def close(self):
        if self._h:
            _lib.mcskin_cuda_context_destroy(self._h)
            self._h = McContext_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def set_option(self, name: str, value: int):
        _check(_lib.mcskin_cuda_context_set_option(self._h, name.encode(), C.c_int64(value)))

    def set_aov_targets(self, coverage: int = 0, depth: int = 0, tri_id: int = 0, normal: int = 0, albedo: int = 0):
        """AOV planes for the following render calls: raw device addresses of float32 / float32 / int32 planes laid out
        like the colour image of each call, and of float32 planes of 3 (normal) and 4 (albedo) values per pixel
        (0: that plane is not written; all 0 switches them off)."""
        t = _abi.McAovTargets(coverage or None, depth or None, tri_id or None, normal or None, albedo or None)
        _check(_lib.mcskin_cuda_context_set_aov_targets(self._h, C.byref(t)))

    def set_scene(self, scene: FlatScene, cfg: McConfig):
        cs = scene.as_c()
        _check(_lib.mcskin_cuda_context_set_scene(self._h, C.byref(cs), C.byref(cfg)))
        self.cfg = _abi.copy_config(cfg)

    def band_rows(self, first_tile_row: int = 0, stride: int = 1) -> int:
        return int(_lib.mcskin_cuda_band_rows(C.byref(self.cfg), C.c_int32(first_tile_row), C.c_int32(stride)))

    def render_bands(self, first_tile_row: int, stride: int, d_out_f32: int = 0, d_out_u8: int = 0, stream: int = 0):
        """Asynchronous. d_out_* are raw device addresses (e.g. torch.Tensor.data_ptr())."""
        _check(_lib.mcskin_cuda_context_render_bands(self._h, C.c_int32(first_tile_row), C.c_int32(stride),
                                                     C.c_void_p(d_out_f32 or None), C.c_void_p(d_out_u8 or None),
                                                     C.c_void_p(stream or None)))

    def render_rows_into_frame(self, first_tile_row: int, stride: int, d_frame_f32: int = 0, d_frame_u8: int = 0, stream: int = 0):
        """Asynchronous: the same rows written at their own place in a full [H, W, 4] frame (possibly a peer's)."""
        _check(_lib.mcskin_cuda_context_render_rows_into_frame(self._h, C.c_int32(first_tile_row), C.c_int32(stride),
                                                               C.c_void_p(d_frame_f32 or None), C.c_void_p(d_frame_u8 or None),
                                                               C.c_void_p(stream or None)))

    def render_tiles_into_frame(self, tiles: np.ndarray, d_frame_f32: int = 0, d_frame_u8: int = 0, stream: int = 0):
        """Asynchronous: any set of whole tiles (frame tile indices) written at their own place in a full frame."""
        tiles = np.ascontiguousarray(tiles, dtype=np.int32)
        _check(_lib.mcskin_cuda_context_render_tiles_into_frame(self._h, _ptr(tiles, C.c_int32), C.c_int32(len(tiles)),
                                                                C.c_void_p(d_frame_f32 or None), C.c_void_p(d_frame_u8 or None),
                                                                C.c_void_p(stream or None)))

    def render_scene_tiles(self, scene, cfg: McConfig, tiles: np.ndarray, host_f32: np.ndarray | None = None,
                           host_u8: np.ndarray | None = None) -> float:
        """Blocking: upload the scene, render these tiles into the page-locked, mapped HOST image(s) (full frames,
        e.g. bands.HostFrame.frame or a registered array), wait.  Returns the kernels' milliseconds.
        `scene` may be a FlatScene or its cached C view (FlatScene.as_c())."""
        cs = scene.as_c() if isinstance(scene, FlatScene) else scene
        ms = C.c_float(0.0)
        _check(_lib.mcskin_cuda_context_render_scene_tiles(
            self._h, C.byref(cs), C.byref(cfg), _ptr(tiles, C.c_int32), C.c_int32(len(tiles)),
            None if host_f32 is None else C.cast(C.c_void_p(host_f32.ctypes.data), C.POINTER(C.c_float)),
            None if host_u8 is None else C.cast(C.c_void_p(host_u8.ctypes.data), C.POINTER(C.c_uint8)), C.byref(ms)))
        self.cfg = cfg
        return float(ms.value)

    def render_batch(self, scenes: list[FlatScene], cfg: McConfig, d_out_f32: int = 0, d_out_u8: int = 0, stream: int = 0):
        """Asynchronous: scene i -> image i of the [n, H, W, 4] device buffer(s) (one skin per scene, same config)."""
        arr = (McScene * len(scenes))(*[s.as_c() for s in scenes])
        self._keep = (arr, scenes)
        _check(_lib.mcskin_cuda_context_render_batch(self._h, arr, C.c_int32(len(scenes)), C.byref(cfg),
                                                     C.c_void_p(d_out_f32 or None), C.c_void_p(d_out_u8 or None),
                                                     C.c_void_p(stream or None)))
        self.cfg = _abi.copy_config(cfg)

    def render_skin_batch(self, atlases: np.ndarray, cfg: McConfig, poses=None, d_out_f32: int = 0, d_out_u8: int = 0, stream: int = 0):
        """Asynchronous: skins straight from their RGBA8 atlases, uint8 [n, H, 64, 4] (H = 64 or 32) -> image i of the
        [n, H, W, 4] device buffer(s).  poses: None (standing), one pose (name / index / 12 numbers) for all, or [n, 12]."""
        atlases = np.ascontiguousarray(atlases, dtype=np.uint8)
        if atlases.ndim != 4 or atlases.shape[3] != 4:
            raise ValueError("atlases must be uint8 [n, H, W, 4]")
        n, h, w = atlases.shape[:3]
        p, stride = None, 0
        if poses is not None:
            arr = np.asarray(poses, dtype=np.float32) if not isinstance(poses, (str, int)) else None
            if arr is not None and arr.ndim == 2:
                p, stride = np.ascontiguousarray(arr.reshape(n, 12)), 12
            else:
                p = pose_array(poses)
        self._keep = (atlases, p)
        _check(_lib.mcskin_cuda_context_render_skin_batch(self._h, _ptr(atlases, C.c_uint8), C.c_int32(w), C.c_int32(h), C.c_int32(n),
                                                          None if p is None else _ptr(p, C.c_float), C.c_int32(stride), C.byref(cfg),
                                                          C.c_void_p(d_out_f32 or None), C.c_void_p(d_out_u8 or None),
                                                          C.c_void_p(stream or None)))
        self.cfg = _abi.copy_config(cfg)

    def debug_block_times(self) -> np.ndarray:
        """[n, 4] uint64 (entry ns, exit ns, frame tile, part | parts << 16) of the last primary launch
        (option "debug_primary_timing")."""
        n = _lib.mcskin_cuda_context_debug_block_times(self._h, None, C.c_int32(0))
        _check(min(n, 0))
        out = np.zeros((n, 4), dtype=np.uint64)
        if n:
            _check(min(_lib.mcskin_cuda_context_debug_block_times(self._h, _ptr(out, C.c_uint64), C.c_int32(n)), 0))
        return out

    def sync(self) -> dict:
        stats = McRenderStats()
        _check(_lib.mcskin_cuda_context_sync(self._h, C.byref(stats)))
        return {k: getattr(stats, k) for k, _ in McRenderStats._fields_}


# ---------------------------------------------------------------- single-ray views
def intersect(scene: FlatScene, rays: np.ndarray, box: int = -1, device: int = 0) -> np.ndarray:
    rays = np.ascontiguousarray(rays, dtype=_abi.RAY_DTYPE)
    out = np.zeros(len(rays), dtype=_abi.HIT_DTYPE)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_intersect(C.byref(cs), C.c_int32(device), C.c_int32(box), _ptr(rays, McRay),
                                      C.c_int32(len(rays)), _ptr(out, McHit)))
    return out


def trace(scene: FlatScene, cfg: McConfig, rays: np.ndarray, depth: int = 0, use_config: bool = True,
          device: int = 0) -> np.ndarray:
    rays = np.ascontiguousarray(rays, dtype=_abi.RAY_DTYPE)
    out = np.zeros((len(rays), 4), dtype=np.float32)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_trace(C.byref(cs), C.byref(cfg), C.c_int32(device), C.c_int32(int(use_config)),
                                  C.c_int32(depth), _ptr(rays, McRay), C.c_int32(len(rays)), _ptr(out, C.c_float)))
    return out


def shade(scene: FlatScene, cfg: McConfig, hits: np.ndarray, view_dirs, shadow_factors=None,
          device: int = 0) -> np.ndarray:
    hits = np.ascontiguousarray(hits, dtype=_abi.HIT_DTYPE)
    vd = _f32(view_dirs, (-1, 3))
    sf = None if shadow_factors is None else _f32(shadow_factors)
    out = np.zeros((len(hits), 4), dtype=np.float32)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_shade(C.byref(cs), C.byref(cfg), C.c_int32(device), _ptr(hits, McHit), _ptr(vd, C.c_float),
                                  None if sf is None else _ptr(sf, C.c_float), C.c_int32(len(hits)),
                                  _ptr(out, C.c_float)))
    return out


def in_shadow(scene: FlatScene, points, normals, lights, device: int = 0) -> np.ndarray:
    p, n, l = _f32(points, (-1, 3)), _f32(normals, (-1, 3)), _f32(lights, (-1, 3))
    out = np.zeros(len(p), dtype=np.int32)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_in_shadow(C.byref(cs), C.c_int32(device), _ptr(p, C.c_float), _ptr(n, C.c_float),
                                      _ptr(l, C.c_float), C.c_int32(len(p)), _ptr(out, C.c_int32)))
    return out


def soft_shadow(scene: FlatScene, points, normals, seeds, samples: int, device: int = 0) -> np.ndarray:
    p, n = _f32(points, (-1, 3)), _f32(normals, (-1, 3))
    s = np.ascontiguousarray(seeds, dtype=np.uint32)
    out = np.zeros(len(p), dtype=np.float32)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_soft_shadow(C.byref(cs), C.c_int32(device), _ptr(p, C.c_float), _ptr(n, C.c_float),
                                        _ptr(s, C.c_uint32), C.c_int32(samples), C.c_int32(len(p)),
                                        _ptr(out, C.c_float)))
    return out


def ambient_occlusion(scene: FlatScene, points, normals, seeds, samples: int, radius: float,
                      device: int = 0) -> np.ndarray:
    p, n = _f32(points, (-1, 3)), _f32(normals, (-1, 3))
    s = np.ascontiguousarray(seeds, dtype=np.uint32)
    out = np.zeros(len(p), dtype=np.float32)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_ambient_occlusion(C.byref(cs), C.c_int32(device), _ptr(p, C.c_float), _ptr(n, C.c_float),
                                              _ptr(s, C.c_uint32), C.c_int32(samples), C.c_float(radius),
                                              C.c_int32(len(p)), _ptr(out, C.c_float)))
    return out


def generate_rays(scene: FlatScene, aspect: float, uv, device: int = 0) -> np.ndarray:
    uv = _f32(uv, (-1, 2))
    out = np.zeros(len(uv), dtype=_abi.RAY_DTYPE)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_generate_rays(C.byref(cs), C.c_int32(device), C.c_float(aspect), _ptr(uv, C.c_float),
                                          C.c_int32(len(uv)), _ptr(out, McRay)))
    return out


def background(scene: FlatScene, cfg: McConfig, uv, use_config: bool = True, device: int = 0) -> np.ndarray:
    uv = _f32(uv, (-1, 2))
    out = np.zeros((len(uv), 4), dtype=np.float32)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_background(C.byref(cs), C.byref(cfg), C.c_int32(device), C.c_int32(int(use_config)),
                                       _ptr(uv, C.c_float), C.c_int32(len(uv)), _ptr(out, C.c_float)))
    return out


def sincos(angles, device: int = 0):
    """(sin, cos) of float32 angles as the kernels evaluate them (glibc-exact for |angle| < 120)."""
    a = _f32(angles, (-1,))
    sn = np.zeros(len(a), dtype=np.float32)
    cs = np.zeros(len(a), dtype=np.float32)
    _check(_lib.mcskin_cuda_sincos(C.c_int32(device), _ptr(a, C.c_float), C.c_int32(len(a)), _ptr(sn, C.c_float),
                                   _ptr(cs, C.c_float)))
    return sn, cs


def powf(x, y, device: int = 0) -> np.ndarray:
    """std::pow(x, y) for float32 arrays as the shading kernels evaluate it."""
    x, y = _f32(x, (-1,)), _f32(y, (-1,))
    out = np.zeros(len(x), dtype=np.float32)
    _check(_lib.mcskin_cuda_powf(C.c_int32(device), _ptr(x, C.c_float), _ptr(y, C.c_float), C.c_int32(len(x)), _ptr(out, C.c_float)))
    return out


def powf_model(x, y) -> np.ndarray:
    """The device's powf arithmetic evaluated on the host (needs no GPU)."""
    x, y = _f32(x, (-1,)), _f32(y, (-1,))
    out = np.zeros(len(x), dtype=np.float32)
    _lib.mcskin_powf_model(_ptr(x, C.c_float), _ptr(y, C.c_float), C.c_int32(len(x)), _ptr(out, C.c_float))
    return out


def primary_launch_order(scene: FlatScene, cfg: McConfig, first_tile_row: int = 0, stride: int = 1, parts_heavy: int = 1,
                         parts_light: int = 1):
    """(tile, part, parts) per block of the primary pass for a band, as the kernels map them (no GPU needed)."""
    cs = scene.as_c()
    n = _lib.mcskin_primary_launch_order(C.byref(cs), C.byref(cfg), C.c_int32(first_tile_row), C.c_int32(stride),
                                         C.c_int32(parts_heavy), C.c_int32(parts_light), None, None, None, C.c_int32(0))
    _check(min(n, 0))
    tile, part, parts = (np.zeros(n, dtype=np.int32) for _ in range(3))
    if n:
        _lib.mcskin_primary_launch_order(C.byref(cs), C.byref(cfg), C.c_int32(first_tile_row), C.c_int32(stride),
                                         C.c_int32(parts_heavy), C.c_int32(parts_light), _ptr(tile, C.c_int32),
                                         _ptr(part, C.c_int32), _ptr(parts, C.c_int32), C.c_int32(n))
    return tile, part, parts


def fp32_issue_peak(device: int = 0) -> float:
    """Measured non-FMA FP32 issue rate of the device in lane-ops per second (FADD/FMUL microbenchmark)."""
    out = C.c_double(0.0)
    _check(_lib.mcskin_cuda_fp32_issue_peak(C.c_int32(device), C.byref(out)))
    return float(out.value)


def sincos_model(angles):
    """The device's sin/cos arithmetic evaluated on the host (needs no GPU)."""
    a = _f32(angles, (-1,))
    sn = np.zeros(len(a), dtype=np.float32)
    cs = np.zeros(len(a), dtype=np.float32)
    _lib.mcskin_sincos_model(_ptr(a, C.c_float), C.c_int32(len(a)), _ptr(sn, C.c_float), _ptr(cs, C.c_float))
    return sn, cs


def aov(scene: FlatScene, cfg: McConfig, device: int = 0) -> np.ndarray:
    out = np.full((max(cfg.height, 0), max(cfg.width, 0)), -1, dtype=np.int32)
    cs = scene.as_c()
    _check(_lib.mcskin_cuda_aov(C.byref(cs), C.byref(cfg), C.c_int32(device), _ptr(out, C.c_int32)))
    return out

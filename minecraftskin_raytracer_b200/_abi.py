"""ctypes mirror of include/mcskin_cuda.h (the C ABI of the render hot path).

Field order and widths follow the header exactly; tests/test_abi.py checks the
struct sizes against the compiled library (mcskin_cuda_abi_sizes).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

ABI_VERSION = 3

MC_OK = 0
MC_ERR_INVALID = -1
MC_ERR_NO_DEVICE = -2
MC_ERR_CUDA = -3
MC_ERR_LIMIT = -4


class McFaceTex(C.Structure):
    _fields_ = [("texel_offset", C.c_int32), ("width", C.c_int32), ("height", C.c_int32)]


class McBox(C.Structure):
    _fields_ = [
        ("bounds_min", C.c_float * 3),
        ("bounds_max", C.c_float * 3),
        ("pivot", C.c_float * 3),
        ("rot_x_deg", C.c_float),
        ("rot_z_deg", C.c_float),
        ("has_rotation", C.c_int32),
        ("is_outer_layer", C.c_int32),
        ("n_triangles", C.c_int32),
        ("face", McFaceTex * 6),
    ]


class McScene(C.Structure):
    _fields_ = [
        ("n_boxes", C.c_int32),
        ("boxes", C.POINTER(McBox)),
        ("n_texels", C.c_int32),
        ("texels_rgba", C.POINTER(C.c_float)),
        ("light_pos", C.c_float * 3),
        ("light_color", C.c_float * 4),
        ("light_radius", C.c_float),
        ("cam_pos", C.c_float * 3),
        ("cam_target", C.c_float * 3),
        ("cam_up", C.c_float * 3),
        ("cam_fov_deg", C.c_float),
        ("background", C.c_float * 4),
    ]


class McConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32),
        ("height", C.c_int32),
        ("max_bounces", C.c_int32),
        ("samples_per_pixel", C.c_int32),
        ("tile_size", C.c_int32),
        ("thread_count", C.c_int32),
        ("soft_shadows", C.c_int32),
        ("shadow_samples", C.c_int32),
        ("ao_enabled", C.c_int32),
        ("ao_samples", C.c_int32),
        ("ao_radius", C.c_float),
        ("ao_intensity", C.c_float),
        ("dof_enabled", C.c_int32),
        ("aperture", C.c_float),
        ("focus_distance", C.c_float),
        ("gradient_bg", C.c_int32),
        ("gradient_scale", C.c_float),
        ("bg_center", C.c_float * 4),
        ("bg_edge", C.c_float * 4),
        ("kd", C.c_float),
        ("ks", C.c_float),
        ("ambient", C.c_float),
        ("shininess", C.c_float),
        ("rng_mode", C.c_int32),
    ]


class McTile(C.Structure):
    _fields_ = [("x", C.c_int32), ("y", C.c_int32), ("width", C.c_int32), ("height", C.c_int32)]


class McRenderStats(C.Structure):
    _fields_ = [
        ("n_tiles", C.c_int32),
        ("n_active_pixels", C.c_int32),
        ("n_samples", C.c_int64),
        ("ms_device", C.c_float),
        ("n_kernel_launches", C.c_int32),
        ("ms_primary", C.c_float),
        ("ms_shade", C.c_float),
    ]


class McAovTargets(C.Structure):
    """Per-pixel planes rendered next to the colour (include/mcskin_cuda.h); null members are not written."""
    _fields_ = [("coverage", C.c_void_p), ("depth", C.c_void_p), ("tri_id", C.c_void_p), ("normal", C.c_void_p),
                ("albedo", C.c_void_p)]


class McRay(C.Structure):
    _fields_ = [("origin", C.c_float * 3), ("dir", C.c_float * 3)]


class McHit(C.Structure):
    _fields_ = [
        ("hit", C.c_int32),
        ("t", C.c_float),
        ("point", C.c_float * 3),
        ("normal", C.c_float * 3),
        ("tex_color", C.c_float * 4),
        ("is_outer_layer", C.c_int32),
        ("box", C.c_int32),
        ("face", C.c_int32),
    ]


McProgressFn = C.CFUNCTYPE(None, C.c_int32, C.c_int32, C.c_void_p)
McContext_p = C.c_void_p  # opaque McContext*

# numpy views of the same layouts (arrays of rays / hits cross the ABI as raw buffers)
RAY_DTYPE = np.dtype([("origin", np.float32, 3), ("dir", np.float32, 3)])
HIT_DTYPE = np.dtype(
    [
        ("hit", np.int32),
        ("t", np.float32),
        ("point", np.float32, 3),
        ("normal", np.float32, 3),
        ("tex_color", np.float32, 4),
        ("is_outer_layer", np.int32),
        ("box", np.int32),
        ("face", np.int32),
    ]
)
BOX_DTYPE = np.dtype(
    [
        ("bounds_min", np.float32, 3),
        ("bounds_max", np.float32, 3),
        ("pivot", np.float32, 3),
        ("rot_x_deg", np.float32),
        ("rot_z_deg", np.float32),
        ("has_rotation", np.int32),
        ("is_outer_layer", np.int32),
        ("n_triangles", np.int32),
        ("face", np.int32, (6, 3)),  # (texel_offset, width, height)
    ]
)
TILE_DTYPE = np.dtype([("x", np.int32), ("y", np.int32), ("width", np.int32), ("height", np.int32)])

assert RAY_DTYPE.itemsize == C.sizeof(McRay)
assert HIT_DTYPE.itemsize == C.sizeof(McHit)
assert BOX_DTYPE.itemsize == C.sizeof(McBox)
assert TILE_DTYPE.itemsize == C.sizeof(McTile)


def default_config(**overrides) -> McConfig:
    """RayTracer::Config{} + ShadingParams{} defaults (raytracer.h:10-38, shading.h:9-14)."""
    cfg = McConfig()
    cfg.width, cfg.height = 256, 256
    cfg.max_bounces = 3
    cfg.samples_per_pixel = 1
    cfg.tile_size = 32
    cfg.thread_count = 0
    cfg.soft_shadows = 1
    cfg.shadow_samples = 8
    cfg.ao_enabled = 0
    cfg.ao_samples = 8
    cfg.ao_radius = 3.0
    cfg.ao_intensity = 0.5
    cfg.dof_enabled = 0
    cfg.aperture = 0.5
    cfg.focus_distance = 0.0
    cfg.gradient_bg = 1
    cfg.gradient_scale = 1.0
    cfg.bg_center[:] = [0.91, 0.89, 0.86, 1.0]
    cfg.bg_edge[:] = [0.56, 0.63, 0.71, 1.0]
    cfg.kd, cfg.ks, cfg.ambient, cfg.shininess = 0.75, 0.15, 0.20, 16.0
    cfg.rng_mode = 0
    for k, v in overrides.items():
        if k in ("bg_center", "bg_edge"):
            getattr(cfg, k)[:] = list(v)
        else:
            if not hasattr(cfg, k):
                raise AttributeError(f"McConfig has no field {k!r}")
            setattr(cfg, k, v)
    return cfg


def copy_config(cfg: McConfig, **overrides) -> McConfig:
    out = McConfig()
    C.memmove(C.byref(out), C.byref(cfg), C.sizeof(McConfig))
    for k, v in overrides.items():
        if k in ("bg_center", "bg_edge"):
            getattr(out, k)[:] = list(v)
        else:
            setattr(out, k, v)
    return out

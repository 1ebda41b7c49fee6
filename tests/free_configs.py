"""Free render configurations: the scalar fields of McConfig and the scene's light colour and background away from the
reference defaults the render cases and free scenes use (pure data).

Every builder is deterministic (fixed values, or seeded numpy generators) and returns FreeConfig records whose name says
which field or gate it aims at:
  * Blinn-Phong: kd, ks, ambient at 0, bright enough to drive the clamp, negative; shininess from 0 to ~4000 (where
    powf's result underflows to 2^-149 and to 0) and negative (powf(0, y < 0) is inf: ks * inf * 0 is NaN);
  * light colour: distinct channels, a channel at 0 or above 1, alpha != 1 (never read);
  * background: the scene's flat colour (alpha != 1, channels outside [0, 1]; with the gradient on it still colours
    reflection rays that miss), the gradient's per-channel colours and its scale, also through the fixed 4- and 16-spp
    pixel-per-lane forms of the primary pass;
  * ambient occlusion: radius, intensity and sample count (0 samples: 0 / 0 in computeAO, a NaN in every hit pixel);
  * soft shadows with 2 samples and with the counts <= 1 that mean hard shadows;
  * the lens gate aperture > 1e-6f and the focus distance (<= 0: the camera's distance to its target);
  * samples_per_pixel <= 0 (one sample), thread_count (never changes a pixel), tiles larger than the frame or of 33;
  * mixed: every field above drawn at once.
Most records carry a twin: the same scene and config with the aimed-at field at its default (the frame must differ), or
at a setting the reference treats alike (`same`: the frame must equal the twin's bit for bit).
"""
from __future__ import annotations

import dataclasses

import numpy as np

from minecraftskin_raytracer_b200 import _abi
from minecraftskin_raytracer_b200.scene import FlatScene
from tests import free_scenes as fs

SKIN_SEED = 43
SCENE_FIELDS = ("light_color", "background")
F32_1E6 = float(np.float32(1e-6))                                   # the lens gate, exactly: the lens stays off
F32_1E6_UP = float(np.nextafter(np.float32(1e-6), np.float32(1)))  # the next float up: the lens is on


@dataclasses.dataclass
class FreeConfig:
    name: str
    scene: FlatScene
    cfg: _abi.McConfig
    twin: tuple | None = None   # (scene, cfg) that differs from this one only in the field(s) the name aims at
    same: bool = False          # True: the twin's frame equals this one's bit for bit; False: it differs


def _cfg(**kw) -> _abi.McConfig:
    base = dict(width=48, height=48, samples_per_pixel=2, max_bounces=2)
    base.update(kw)
    return _abi.default_config(**base)


def _split(fields: dict):
    return ({k: v for k, v in fields.items() if k in SCENE_FIELDS},
            {k: v for k, v in fields.items() if k not in SCENE_FIELDS})


def _default_of(scene: FlatScene, field: str):
    if field in SCENE_FIELDS:
        return getattr(scene, field)
    v = getattr(_abi.default_config(), field)
    return tuple(v) if field in ("bg_center", "bg_edge") else v


def _case(name, scene, base: dict, vary: dict, twin: dict | None = None, same: bool = False) -> FreeConfig:
    """`scene` and a config of `base` with the fields of `vary` set (scene or config fields).  The twin sets `twin`'s
    fields instead of `vary`'s, or, without one, `vary`'s fields at their defaults (the scene's own for scene fields)."""
    if twin is None:
        twin = {k: _default_of(scene, k) for k in vary}
    sv, cv = _split(vary)
    st, ct = _split(twin)
    return FreeConfig(name, dataclasses.replace(scene, **sv), _cfg(**{**base, **cv}),
                      (dataclasses.replace(scene, **st), _cfg(**{**base, **ct})), same)


def skin(pose):
    return fs.skin(pose, SKIN_SEED)


# ---------------------------------------------------------------------------------------------------- Blinn-Phong
def blinn_phong_configs():
    s, boxes = skin("walking"), fs.random_box_scene(200, 10)
    spec_only = dict(kd=0.0, ambient=0.0, ks=1.0)   # the specular term alone: powf's result reaches the frame unmixed
    out = [
        _case("phong_kd0", s, {}, dict(kd=0.0)),
        _case("phong_ks0", s, {}, dict(ks=0.0)),
        _case("phong_ambient0", s, {}, dict(ambient=0.0)),
        _case("phong_kd_bright_clamp", s, {}, dict(kd=4.0)),
        _case("phong_ks_bright_clamp", boxes, {}, dict(ks=6.5)),
        _case("phong_ambient_bright_clamp", s, {}, dict(ambient=1.7)),
        _case("phong_kd_negative", boxes, {}, dict(kd=-0.6)),
    ]
    for tag, y in (("0", 0.0), ("0.5", 0.5), ("1", 1.0), ("7.3", 7.3), ("128", 128.0)):
        out.append(_case(f"phong_shininess_{tag}", s if tag != "7.3" else boxes, {}, dict(shininess=y)))
    out.append(_case("phong_shininess_4000_underflow", s, spec_only, dict(shininess=4000.0)))
    out.append(_case("phong_shininess_negative_soft", s, {}, dict(shininess=-2.5)))
    out.append(_case("phong_shininess_negative_hard", s, dict(soft_shadows=0), dict(shininess=-2.5)))
    return out


# ---------------------------------------------------------------------------------------------------- light colour
def light_color_configs():
    s, touching = skin("dab"), fs.touching_scene()
    return [
        _case("light_color_distinct", s, {}, dict(light_color=(1.0, 0.55, 0.2, 1.0))),
        _case("light_color_green_zero", s, {}, dict(light_color=(0.9, 0.0, 0.7, 1.0))),
        _case("light_color_red_above_one", touching, {}, dict(light_color=(2.5, 1.0, 0.4, 1.0))),
        _case("light_color_alpha", s, {}, dict(light_color=(1.0, 1.0, 1.0, 0.3)), same=True),
    ]


# ---------------------------------------------------------------------------------------------------- background
def background_configs():
    s, boxes = skin("fighting"), fs.random_box_scene(201, 12)
    center, edge = (0.95, 0.3, 0.1, 0.4), (0.05, 0.6, 1.3, 0.2)
    out = [
        _case("bg_flat_alpha_out_of_range", s, dict(gradient_bg=0), dict(background=(1.4, -0.25, 0.6, 0.35))),
        # with the gradient on, the flat colour is what reflection rays that miss return (raytracer.cpp:94-102)
        _case("bg_flat_in_reflections", s, {}, dict(background=(0.9, 0.1, 0.35, 0.6))),
        _case("bg_gradient_channels", boxes, {}, dict(bg_center=center, bg_edge=edge)),
        # the gradient's alpha is always 1 (raytracer.cpp:31)
        _case("bg_gradient_alpha", s, {}, dict(bg_center=(0.91, 0.89, 0.86, 0.25), bg_edge=(0.56, 0.63, 0.71, 3.0)),
              same=True),
    ]
    for tag, g in (("0", 0.0), ("0.3", 0.3), ("4", 4.0), ("-1", -1.0)):
        out.append(_case(f"bg_gradient_scale_{tag}", s, {}, dict(gradient_scale=g)))
    # the fixed pixel-per-lane forms of the primary pass with the gradient inlined (k_primary_pix_fixed<SPP, true, B>)
    out.append(_case("bg_gradient_spp16_fixed_form", s, dict(samples_per_pixel=16, max_bounces=1),
                     dict(bg_center=center, bg_edge=edge, gradient_scale=0.3)))
    out.append(_case("bg_gradient_spp4_fixed_form", boxes, dict(samples_per_pixel=4),
                     dict(bg_center=edge, bg_edge=center, gradient_scale=1.7)))
    return out


# ---------------------------------------------------------------------------------------------------- ambient occlusion
def ao_configs():
    s = skin("waving")
    ao = dict(ao_enabled=1)
    out = []
    for tag, r in (("0", 0.0), ("1e-3", 1e-3), ("0.5", 0.5), ("1e6", 1e6), ("-1", -1.0)):
        out.append(_case(f"ao_radius_{tag}", s, ao, dict(ao_radius=r)))
    for tag, k in (("0", 0.0), ("1", 1.0), ("2.5", 2.5), ("-0.5", -0.5)):
        out.append(_case(f"ao_intensity_{tag}", s, ao, dict(ao_intensity=k)))
    # no samples: computeAO returns 1 - 0.0f / 0.0f, a NaN in every pixel with a hitting sample
    out.append(_case("ao_samples_0_nan", s, ao, dict(ao_samples=0)))
    out.append(_case("ao_samples_1", s, ao, dict(ao_samples=1)))
    out.append(_case("ao_samples_2", s, ao, dict(ao_samples=2)))
    # a negative count draws nothing: 0 / -3 = -0, so AO = 1 and the factor 1 - intensity * 0 = 1
    out.append(_case("ao_samples_negative", s, ao, dict(ao_samples=-3), twin=dict(ao_enabled=0), same=True))
    return out


# ---------------------------------------------------------------------------------------------------- shadows
def shadow_configs():
    s = skin("running")
    hard = dict(soft_shadows=0)
    return [
        # soft shadows need shadow_samples > 1 (raytracer.cpp:109): fewer is the hard test
        _case("soft_shadow_samples_0", s, {}, dict(shadow_samples=0), twin=hard, same=True),
        _case("soft_shadow_samples_1", s, {}, dict(shadow_samples=1), twin=hard, same=True),
        _case("soft_shadow_samples_negative", s, {}, dict(shadow_samples=-5), twin=hard, same=True),
        _case("soft_shadow_samples_2", s, {}, dict(shadow_samples=2)),
    ]


# ---------------------------------------------------------------------------------------------------- lens
def lens_configs():
    s = skin("walking")
    dof = dict(dof_enabled=1, aperture=0.3)
    off = dict(dof_enabled=0)
    return [
        _case("lens_aperture_at_gate", s, dict(dof_enabled=1), dict(aperture=F32_1E6), twin=off, same=True),
        _case("lens_aperture_above_gate", s, dict(dof_enabled=1), dict(aperture=F32_1E6_UP), twin=off),
        # focus_distance <= 0: the lens focuses at the camera's distance to its target (tile_renderer.cpp:82-85)
        _case("lens_focus_0", s, dict(aperture=0.3), dict(dof_enabled=1), twin=off),
        _case("lens_focus_negative", s, dof, dict(focus_distance=-5.0), twin=dict(focus_distance=0.0), same=True),
        _case("lens_focus_1e4", s, dof, dict(focus_distance=1e4)),
    ]


# ---------------------------------------------------------------------------------------------------- sampling and tiles
def sampling_configs():
    s = skin("dab")
    frame = dict(width=56, height=40)
    one = dict(samples_per_pixel=1)
    return [
        _case("spp_0", s, frame, dict(samples_per_pixel=0), twin=one, same=True),
        _case("spp_negative", s, frame, dict(samples_per_pixel=-4), twin=one, same=True),
        # thread_count 0 is the default of every other configuration
        _case("thread_count_negative", s, frame, dict(thread_count=-1), same=True),
        _case("thread_count_64", s, frame, dict(thread_count=64), same=True),
        # one tile seeds one stream for the whole frame
        _case("tile_larger_than_frame", s, frame, dict(tile_size=100)),
        _case("tile_33", s, frame, dict(tile_size=33, samples_per_pixel=3)),
    ]


# ---------------------------------------------------------------------------------------------------- mixed
def _pick(rng, values):
    return values[int(rng.integers(len(values)))]


def mixed_configs(n: int = 10):
    scenes = [lambda: skin("walking"), lambda: skin("dab"), lambda: skin(None), lambda: fs.random_box_scene(202, 9),
              fs.touching_scene, fs.posed_thresholds_scene]
    out = []
    for k in range(n):
        rng = np.random.default_rng(700 + k)
        scene = scenes[k % len(scenes)]()
        f3 = lambda lo, hi: tuple(float(np.float32(x)) for x in rng.uniform(lo, hi, 3))  # noqa: E731
        scene = dataclasses.replace(scene, light_color=f3(0.0, 2.0) + (float(np.float32(rng.uniform(0, 2))),),
                                    background=f3(-0.3, 1.5) + (float(np.float32(rng.uniform(0, 1.5))),))
        cfg = _cfg(
            width=int(_pick(rng, [32, 40, 48, 64])), height=int(_pick(rng, [24, 40, 48, 64])),
            samples_per_pixel=_pick(rng, [-2, 0, 1, 2, 3, 4, 5, 16]), max_bounces=_pick(rng, [0, 1, 2, 3]),
            tile_size=_pick(rng, [8, 16, 32, 33, 100]), thread_count=_pick(rng, [-1, 0, 3, 64]),
            kd=_pick(rng, [0.0, 0.75, 1.9, -0.4, float(rng.uniform(0, 1))]),
            ks=_pick(rng, [0.0, 0.15, 3.0, float(rng.uniform(0, 1))]),
            ambient=_pick(rng, [0.0, 0.2, 1.3, float(rng.uniform(0, 0.5))]),
            shininess=_pick(rng, [0.0, 0.5, 1.0, 7.3, 16.0, 128.0, 4000.0, -2.5]),
            gradient_bg=_pick(rng, [0, 1, 1]), gradient_scale=_pick(rng, [0.0, 0.3, 1.0, 4.0, -1.0]),
            bg_center=f3(-0.2, 1.4) + (float(rng.uniform(0, 2)),), bg_edge=f3(-0.2, 1.4) + (float(rng.uniform(0, 2)),),
            ao_enabled=_pick(rng, [0, 1]), ao_samples=_pick(rng, [0, 1, 2, 5, 16]),
            ao_radius=_pick(rng, [0.0, 0.5, 3.0, 1e6, -1.0]), ao_intensity=_pick(rng, [0.0, 0.5, 1.0, 2.5, -0.5]),
            soft_shadows=_pick(rng, [0, 1, 1]), shadow_samples=_pick(rng, [-1, 0, 1, 2, 3, 8, 13]),
            dof_enabled=_pick(rng, [0, 1]), aperture=_pick(rng, [F32_1E6, F32_1E6_UP, 0.2, 0.6]),
            focus_distance=_pick(rng, [0.0, -5.0, 30.0, 1e4]))
        out.append(FreeConfig(f"mixed_{k}", scene, cfg))
    return out


def free_configs():
    """Every free configuration, in a fixed order."""
    return (blinn_phong_configs() + light_color_configs() + background_configs() + ao_configs() + shadow_configs() +
            lens_configs() + sampling_configs() + mixed_configs())

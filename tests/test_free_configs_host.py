"""Free configurations (tests/free_configs.py) on the CPU: the generator is deterministic, the oracle's frames for them
equal the pins in tests/golden/free_config_pins.json, every field a configuration aims at changes the frame where the
reference reads it and changes no bit where it does not, and the edge values reach the arithmetic their names claim."""
import json
from pathlib import Path

import numpy as np
import pytest

from tests import free_configs as fc
from tests.golden.make_free_config_pins import same_bits
from tests.golden.make_free_scene_pins import scene_config_digest
from tests.golden.make_oracle_pins import digest

PINS = Path(__file__).parent / "golden" / "free_config_pins.json"
_PINNED = json.loads(PINS.read_text())
DIFFERS = sorted(n for n, p in _PINNED.items() if p.get("twin") == "differs")
EQUAL = sorted(n for n, p in _PINNED.items() if p.get("twin") == "equal")


@pytest.fixture(scope="module")
def cases(mclib):
    return {c.name: c for c in fc.free_configs()}


@pytest.fixture(scope="module")
def pins():
    return json.loads(PINS.read_text())


def test_generator_is_deterministic_and_pinned(cases, pins):
    assert sorted(cases) == sorted(pins)
    again = {c.name: c for c in fc.free_configs()}
    for name, c in cases.items():
        assert scene_config_digest(c.scene, c.cfg) == scene_config_digest(again[name].scene, again[name].cfg) == pins[name]["input"], name
        if c.twin is not None:
            assert scene_config_digest(*c.twin) == scene_config_digest(*again[name].twin), name
    assert {n for n, c in cases.items() if c.twin is not None and c.same} == set(EQUAL)
    assert {n for n, c in cases.items() if c.twin is not None and not c.same} == set(DIFFERS)


@pytest.mark.parametrize("name", sorted(_PINNED))
def test_oracle_frames_equal_pins(oracle, cases, pins, name):
    c = cases[name]
    img, cnt = oracle.render(c.scene, c.cfg, counters=True)
    assert digest(img) == pins[name]["image"]
    assert digest(oracle.quantize(img)) == pins[name]["u8"]
    assert cnt["n_intersect_scene"] == pins[name]["calls"]


def _changed_fields(c):
    """The scene and config fields in which a configuration and its twin differ."""
    import ctypes as C
    (ts, tc) = c.twin
    fields = [f for f in fc.SCENE_FIELDS if not np.array_equal(np.float32(getattr(c.scene, f)), np.float32(getattr(ts, f)))]
    for f, _ in type(c.cfg)._fields_:
        a, b = getattr(c.cfg, f), getattr(tc, f)
        if isinstance(a, C.Array):
            a, b = list(a), list(b)
        if a != b:
            fields.append(f)
    return fields


@pytest.mark.parametrize("name", DIFFERS)
def test_field_changes_the_frame(oracle, cases, name):
    """The configuration and its twin differ in the aimed-at field(s) alone, and the oracle's frames differ in bits: a
    kernel that ignored the field, or read another in its place, would not give the oracle's frame for both."""
    c = cases[name]
    assert 1 <= len(_changed_fields(c)) <= 3, _changed_fields(c)
    assert not same_bits(oracle.render(c.scene, c.cfg), oracle.render(*c.twin)), name


@pytest.mark.parametrize("name", EQUAL)
def test_field_is_inert(oracle, cases, name):
    """Light alpha, the gradient's alpha, thread_count, samples_per_pixel <= 0 against 1, aperture == 1e-6f against no
    lens, a negative AO sample count against no AO, shadow_samples <= 1 against hard shadows, a negative focus distance
    against 0: the frames are equal bit for bit."""
    c = cases[name]
    assert 1 <= len(_changed_fields(c)) <= 2, _changed_fields(c)
    assert same_bits(oracle.render(c.scene, c.cfg), oracle.render(*c.twin)), name


def test_edge_values_are_the_floats_named(cases):
    assert np.float32(cases["lens_aperture_at_gate"].cfg.aperture) == np.float32(1e-6)
    above = np.float32(cases["lens_aperture_above_gate"].cfg.aperture)
    assert above > np.float32(1e-6) and np.nextafter(above, np.float32(0)) == np.float32(1e-6)
    for name, spp in (("bg_gradient_spp16_fixed_form", 16), ("bg_gradient_spp4_fixed_form", 4)):
        cfg = cases[name].cfg   # the fixed pixel-per-lane forms: jitter draws only, the gradient on
        assert cfg.samples_per_pixel == spp and cfg.gradient_bg == 1 and cfg.dof_enabled == 0
    for name in ("tile_larger_than_frame",):
        cfg = cases[name].cfg
        assert cfg.tile_size > max(cfg.width, cfg.height)


def test_mixed_configs_draw_every_field(cases):
    """Across the mixed configurations every field takes more than one value, and the edge values appear."""
    import ctypes as C
    mixed = [c for n, c in cases.items() if n.startswith("mixed_")]
    assert len(mixed) == 10
    for f, _ in type(mixed[0].cfg)._fields_:
        if f == "rng_mode":
            continue
        vals = {tuple(getattr(c.cfg, f)) if isinstance(getattr(c.cfg, f), C.Array) else getattr(c.cfg, f) for c in mixed}
        assert len(vals) > 1, f
    for f in fc.SCENE_FIELDS:
        assert len({tuple(getattr(c.scene, f)) for c in mixed}) == len(mixed), f
    seen = lambda f: {getattr(c.cfg, f) for c in mixed}  # noqa: E731
    assert seen("samples_per_pixel") & {0, -2} and seen("shininess") & {4000.0, -2.5} and seen("tile_size") & {33, 100}


def _hits(oracle, scene, n=200_000, seed=17):
    from tests.scenes import random_rays
    rays = random_rays(np.random.default_rng(seed), n)
    hits = oracle.intersect(scene, rays)
    keep = hits["hit"] == 1
    return hits[keep], -rays["dir"][keep]


def test_shininess_4000_reaches_powf_underflow(oracle, cases):
    """With only the specular term (kd = ambient = 0, ks = 1) and full visibility, shade() returns powf(NdotH, 4000)
    itself: the hits of the query set reach powf's underflow returns 2^-149 and 0 and its subnormal results."""
    c = cases["phong_shininess_4000_underflow"]
    hits, view = _hits(oracle, c.scene)
    rgb = oracle.shade(c.scene, c.cfg, hits, view, np.ones(len(hits), np.float32))[:, :3].view(np.uint32)
    assert (rgb == 1).sum() >= 30 and ((rgb > 1) & (rgb < 0x00800000)).sum() >= 300 and (rgb == 0).any()


def test_nan_frames_carry_the_x86_default_nan(oracle, cases):
    """ao_samples = 0 (1 - 0 / 0 in computeAO) and a negative shininess (ks * inf * 0 where NdotH <= 0 in shadow) make
    NaN channels; every one is x86's default NaN 0xffc00000, and quantises to 0."""
    for name, least in (("ao_samples_0_nan", 300), ("phong_shininess_negative_soft", 10), ("phong_shininess_negative_hard", 10)):
        c = cases[name]
        img = oracle.render(c.scene, c.cfg)
        nan = np.isnan(img)
        assert nan.any(axis=-1).sum() >= least, name
        assert (img.view(np.uint32)[nan] == 0xFFC00000).all() and not nan[..., 3].any(), name
        assert (oracle.quantize(img)[nan] == 0).all(), name

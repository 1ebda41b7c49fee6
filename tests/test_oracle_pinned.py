"""Pins the CPU oracle (oracle/mcskin_oracle.c) to the reference:
  * against committed outputs of the UNMODIFIED reference (tests/golden/reference_vectors.npz) —
    always, with no copy of the reference at hand;
  * against the unmodified reference itself (oracle/_ref) when it was built (oracle.harness.reference_dir).
Everything is required to match bit for bit: both are CPU code using the same glibc/libstdc++
arithmetic, so any difference is a restatement error.
"""
import numpy as np
import pytest

from minecraftskin_raytracer_b200 import _abi
from tests.golden.make_oracle_pins import digest, single_ray_inputs
from tests.golden_data import golden_render_cases, golden_scene, pins, ray_scene, vectors
from tests.scenes import RENDER_CASES, make_config, random_rays, synth_skin


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _same_struct(a, b, fields):
    return all(np.array_equal(a[f].view(np.uint32) if a[f].dtype == np.float32 else a[f],
                              b[f].view(np.uint32) if b[f].dtype == np.float32 else b[f]) for f in fields)


@pytest.mark.parametrize("name,cfg", golden_render_cases(), ids=[c[0] for c in golden_render_cases()])
def test_oracle_renders_equal_golden(oracle, name, cfg):
    v = vectors()
    scene = golden_scene(name)
    img, cnt = oracle.render(scene, cfg, counters=True)
    assert np.array_equal(_bits(img), _bits(v[f"{name}/image"]))
    assert cnt["n_intersect_scene"] == int(v[f"{name}/calls"])       # same number of intersectScene calls
    assert np.array_equal(oracle.aov(scene, cfg), v[f"{name}/tri_id"])


def test_oracle_single_ray_vectors_equal_golden(oracle, mclib):
    v = vectors()
    scene = ray_scene(mclib.build_skin_scene)
    rays, want = v["rays/rays"], v["rays/hits"]
    got = oracle.intersect(scene, rays)
    assert np.array_equal(got["hit"], want["hit"]) and np.array_equal(got["box"], want["box"])
    assert np.array_equal(got["face"], want["face"]) and np.array_equal(got["is_outer_layer"], want["is_outer_layer"])
    for f in ("t", "point", "normal", "tex_color"):
        assert np.array_equal(_bits(got[f]), _bits(want[f])), f
    keep = want["hit"] == 1
    cfg = make_config(max_bounces=3)
    assert np.array_equal(_bits(oracle.shade(scene, cfg, want[keep], -rays["dir"][keep], None)), _bits(v["rays/shade_hard"]))
    assert np.array_equal(_bits(oracle.shade(scene, cfg, want[keep], -rays["dir"][keep], v["rays/shade_sf"])), _bits(v["rays/shade_soft"]))
    assert np.array_equal(_bits(oracle.trace(scene, cfg, rays[:1500], 0, True)), _bits(v["rays/trace_cfg"]))
    assert np.array_equal(_bits(oracle.trace(scene, cfg, rays[:1500], 0, False)), _bits(v["rays/trace_nocfg"]))
    seeds = v["rays/seeds"]
    assert np.array_equal(_bits(oracle.soft_shadow(scene, want["point"][keep], want["normal"][keep], seeds, 8)), _bits(v["rays/soft8"]))
    assert np.array_equal(_bits(oracle.ambient_occlusion(scene, want["point"][keep], want["normal"][keep], seeds, 16, 3.0)), _bits(v["rays/ao16"]))
    cam = oracle.generate_rays(scene, 16.0 / 9.0, v["rays/uv"])
    assert np.array_equal(_bits(cam["dir"]), _bits(v["rays/camera"]["dir"]))
    assert np.array_equal(_bits(oracle.background(scene, cfg, v["rays/uv"])), _bits(v["rays/background"]))


def test_oracle_rng_equals_libstdcxx(oracle):
    """std::mt19937 and uniform_real_distribution<float>(0,1) of libstdc++ 13 (SURVEY.md §8c, §9.15-16)."""
    v = vectors()
    for seed in (0, 1, 5489, 1920 * 32 + 64, 0xFFFFFFFF):
        u, f = oracle.mt19937(seed, 2000)
        assert np.array_equal(u, v[f"rng/{seed}/u32"])
        assert np.array_equal(_bits(f), _bits(v[f"rng/{seed}/canonical"]))
    # the 10000th output of mt19937() seeded with 5489 is 4123659995 (ISO C++ [rand.predef])
    assert oracle.mt19937(5489, 10000)[0][-1] == 4123659995
    for x, want in zip(v["rng/seed_cast_in"], v["rng/seed_cast_out"]):
        assert oracle.seed_cast(float(x)) == int(want), x


@pytest.mark.parametrize("case", RENDER_CASES, ids=[c[0] for c in RENDER_CASES])
def test_oracle_equals_live_reference(oracle, reference, case):
    name, seed, kind, pose, over = case
    scene = reference.scene_from_atlas(synth_skin(seed, kind), pose)
    cfg = make_config(**over)
    a, calls = reference.render(scene, cfg, counters=True)
    b, cnt = oracle.render(scene, cfg, counters=True)
    assert np.array_equal(_bits(a), _bits(b))
    assert calls == cnt["n_intersect_scene"]
    assert np.array_equal(reference.aov(scene, cfg), oracle.aov(scene, cfg))


def test_oracle_equals_live_reference_single_rays(oracle, reference):
    scene = reference.scene_from_atlas(synth_skin(21, "64x64"), "dab")
    rays = random_rays(np.random.default_rng(3), 6000)
    a, b = reference.intersect(scene, rays), oracle.intersect(scene, rays)
    assert _same_struct(a, b, ("hit", "t", "point", "normal", "tex_color", "is_outer_layer", "box", "face"))
    cfg = make_config(max_bounces=4, ao_enabled=1)
    assert np.array_equal(_bits(reference.trace(scene, cfg, rays[:800])), _bits(oracle.trace(scene, cfg, rays[:800])))
    assert reference.mt19937(77, 500)[0].tolist() == oracle.mt19937(77, 500)[0].tolist()


@pytest.mark.parametrize("case", RENDER_CASES, ids=[c[0] for c in RENDER_CASES])
def test_oracle_renders_equal_pins(oracle, mclib, case):
    """The inputs of test_oracle_equals_live_reference without the reference: frame, intersectScene count and hit ids
    equal the digests in tests/golden/oracle_pins.json (the oracle's outputs, not the reference's)."""
    name, seed, kind, pose, over = case
    want = pins()["renders"][name]
    scene = mclib.build_skin_scene(synth_skin(seed, kind), pose)
    cfg = make_config(**over)
    img, cnt = oracle.render(scene, cfg, counters=True)
    assert digest(img) == want["image"]
    assert cnt["n_intersect_scene"] == want["calls"]
    assert digest(oracle.aov(scene, cfg)) == want["tri_id"]


def test_oracle_single_rays_equal_pins(oracle, mclib):
    """The inputs of test_oracle_equals_live_reference_single_rays (4 bounces, AO on) without the reference."""
    want = pins()["rays"]
    scene, rays, cfg = single_ray_inputs(mclib.build_skin_scene)
    assert digest(oracle.intersect(scene, rays)) == want["hits"]
    assert digest(oracle.trace(scene, cfg, rays[:800])) == want["trace"]
    assert digest(oracle.mt19937(77, 500)[0]) == want["mt19937_77"]


def test_render_tile_equals_render(oracle, mclib):
    """renderTile over generateTiles == render (tile_renderer.cpp:71-189)."""
    scene = mclib.build_skin_scene(synth_skin(4), "walking")
    cfg = make_config(width=70, height=45, samples_per_pixel=2, tile_size=16)
    full = oracle.render(scene, cfg)
    img = np.zeros_like(full)
    img[..., 3] = 1
    for t in oracle.generate_tiles(70, 45, 16):
        img = oracle.render_tile(scene, cfg, tuple(t), img)
    assert np.array_equal(_bits(img), _bits(full))
    for threads in (1, 3):
        assert np.array_equal(_bits(oracle.render(scene, cfg, threads=threads)), _bits(full))  # test_tile_renderer.cpp:122-145


# ---- McConfig.rng_mode 1 (an extension, not the reference's streams): the switch the oracle shares with the product ----

def _lowbias32(x):
    x &= 0xFFFFFFFF
    x ^= x >> 16
    x = (x * 0x7FEB352D) & 0xFFFFFFFF
    x ^= x >> 15
    x = (x * 0x846CA68B) & 0xFFFFFFFF
    x ^= x >> 16
    return x


def test_counter_stream_words_and_statistics(mclib):
    from minecraftskin_raytracer_b200 import lib
    for seed in (0, 1, 12345, 0xFFFFFFFF, 0x9E3779B9):
        for k in (0, 1, 2, 411, 0xFFFFFFFF):
            assert lib.counter_word(seed, k) == _lowbias32(_lowbias32(seed ^ 0x9E3779B9) + k)
    # uniform and uncorrelated enough for a Monte-Carlo estimator: bucket counts of one stream and of the first
    # word of consecutive seeds (how the renderer seeds neighbouring hits and tiles)
    n = 1 << 14
    for words in ([lib.counter_word(7, k) for k in range(n)], [lib.counter_word(s, 0) for s in range(n)]):
        u = np.array(words, dtype=np.float64) / 2.0**32
        counts = np.bincount((u * 16).astype(int), minlength=16)
        chi2 = ((counts - n / 16) ** 2 / (n / 16)).sum()
        assert chi2 < 45.0, chi2                      # 15 degrees of freedom: p(chi2 > 45) < 1e-4
        assert abs(u.mean() - 0.5) < 0.01
        assert abs(np.corrcoef(u[:-1], u[1:])[0, 1]) < 0.03


def test_oracle_counter_mode_changes_the_noise_only(oracle, mclib):
    from minecraftskin_raytracer_b200 import lib
    scene = lib.build_skin_scene(synth_skin(1, "64x64"), None)
    base = dict(width=96, height=96, max_bounces=3)
    # no stream is drawn from: the two modes are the same frame
    still = dict(samples_per_pixel=1, soft_shadows=0, **base)
    a, b = oracle.render(scene, make_config(**still)), oracle.render(scene, make_config(rng_mode=1, **still))
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    # streams in use: other noise, same picture
    noisy = dict(samples_per_pixel=16, **base)
    a, b = oracle.render(scene, make_config(**noisy)), oracle.render(scene, make_config(rng_mode=1, **noisy))
    assert not np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert abs(float(a[..., :3].mean()) - float(b[..., :3].mean())) < 2e-3
    assert float(np.abs(a - b).mean()) < 0.02
    # the unmodified reference has no such switch: its wrapper ignores the field


def test_shadow_seeds_of_a_figure_fall_into_the_memo_window(oracle, mclib):
    """The premise of the product's seed memo (FreshStream::seed_memo, csrc/dev_mt19937.cuh): traceRay's shadow seed,
    unsigned(x*12345 + y*67890 + z*11111 + depth*99999) (raytracer.cpp:110-112), is a small integer for every point of a
    skin figure in every built-in pose and at every bounce depth, inside the table's window [-2^20, 2^23 - 2^20) — and
    many hits share one seed, which is what makes keeping its seeding worth while."""
    from minecraftskin_raytracer_b200 import lib
    from minecraftskin_raytracer_b200.scene import BUILTIN_POSE_ORDER
    offset, entries = 1 << 20, 1 << 23
    for pose in BUILTIN_POSE_ORDER:
        scene = lib.build_skin_scene(synth_skin(3, "64x64"), None if pose == "standing" else pose)
        rays = random_rays(np.random.default_rng(11), 6000)
        hits = oracle.intersect(scene, rays)
        p = hits["point"][hits["hit"] == 1].astype(np.float32)
        assert len(p) > 500
        for depth in (0, 4, 8):
            v = (p[:, 0] * np.float32(12345.0) + p[:, 1] * np.float32(67890.0) + p[:, 2] * np.float32(11111.0)
                 + np.float32(depth) * np.float32(99999.0)).astype(np.float32)
            seeds = v.astype(np.int64).astype(np.uint32)          # cvttss2si to 64 bits, low half (x86-64 semantics)
            index = (seeds + np.uint32(offset)).astype(np.uint32)  # wraps like the device's
            assert (index < entries).all(), (pose, depth, int((index >= entries).sum()))
    # the headline frame: 2.8 M shaded hits (tests/golden/work_counts.json) over a window of 8.4 M seeds of which a
    # figure reaches a third at most
    assert 32 * 67890 + 8 * 12345 + 5 * 11111 + 8 * 99999 < entries - offset

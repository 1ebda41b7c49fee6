"""CPU-only checks of the product's host side: the C-ABI library loads and exports every
declared symbol, struct layouts agree, the skin -> scene builder equals the reference's
SkinParser + MeshBuilder, tile generation, defaults, and loud failure without a GPU."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

from minecraftskin_raytracer_b200 import _abi
from minecraftskin_raytracer_b200.scene import BUILTIN_POSE_ORDER, BUILTIN_POSES, FlatScene, pose_array, synth_skin
from tests.golden_data import golden_scene, pins, vectors
from tests.golden.make_golden import GOLDEN_RENDERS
from tests.golden.make_oracle_pins import SCENE_SKINS, overlay_atlas, scene_digest
from tests.scenes import make_config

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol(mclib):
    header = (ROOT / "include" / "mcskin_cuda.h").read_text()
    declared = set(re.findall(r"\b(mcskin_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations found"
    raw = mclib.raw()
    for name in sorted(declared):
        assert hasattr(raw, name), f"{name} is declared in include/mcskin_cuda.h but not exported"
    assert declared == set(mclib.EXPORTS), declared ^ set(mclib.EXPORTS)
    assert raw.mcskin_cuda_abi_version() == _abi.ABI_VERSION


def test_struct_layouts_match(mclib):
    mirror = [C.sizeof(t) for t in (_abi.McFaceTex, _abi.McBox, _abi.McScene, _abi.McConfig, _abi.McTile,
                                    _abi.McRenderStats, _abi.McRay, _abi.McHit)]
    assert mclib.abi_sizes() == mirror


def test_config_defaults_are_the_reference_defaults(mclib):
    d = mclib.config_defaults()
    # raytracer.h:10-38, shading.h:9-14
    assert (d.width, d.height, d.max_bounces, d.samples_per_pixel, d.tile_size, d.thread_count) == (256, 256, 3, 1, 32, 0)
    assert (d.soft_shadows, d.shadow_samples, d.ao_enabled, d.ao_samples, d.dof_enabled, d.gradient_bg) == (1, 8, 0, 8, 0, 1)
    assert np.allclose([d.ao_radius, d.ao_intensity, d.aperture, d.focus_distance, d.gradient_scale], [3.0, 0.5, 0.5, 0.0, 1.0])
    assert np.allclose(list(d.bg_center), [0.91, 0.89, 0.86, 1.0]) and np.allclose(list(d.bg_edge), [0.56, 0.63, 0.71, 1.0])
    assert np.allclose([d.kd, d.ks, d.ambient, d.shininess], [0.75, 0.15, 0.20, 16.0])
    assert bytes(d) == bytes(_abi.default_config())


@pytest.mark.parametrize("name,seed,kind,pose,_over", GOLDEN_RENDERS, ids=[g[0] for g in GOLDEN_RENDERS])
def test_skin_scene_builder_equals_golden_reference_scene(mclib, name, seed, kind, pose, _over):
    """mcskin_build_skin_scene == SkinParser::parse + MeshBuilder::buildScene (flattened), byte for byte."""
    built = mclib.build_skin_scene(synth_skin(seed, kind), pose)
    assert built.same_as(golden_scene(name))


def test_skin_scene_builder_equals_live_reference(mclib, reference):
    for seed, kind in ((0, "64x64"), (2, "legacy"), (3, "slim")):
        for pose in [None] + BUILTIN_POSE_ORDER:
            assert mclib.build_skin_scene(synth_skin(seed, kind), pose).same_as(
                reference.scene_from_atlas(synth_skin(seed, kind), pose)), (seed, kind, pose)
    # a fully transparent outer layer is dropped (mesh_builder.cpp:176-186); legacy skins keep 7 boxes
    atlas = synth_skin(5)
    atlas[:16, 32:, 3] = 0
    a, b = mclib.build_skin_scene(atlas), reference.scene_from_atlas(atlas)
    assert a.same_as(b) and len(a.boxes) == 11
    assert len(mclib.build_skin_scene(synth_skin(2, "legacy")).boxes) == 7
    poses = reference.builtin_poses()
    for i, name in enumerate(BUILTIN_POSE_ORDER):          # src/scene/pose.h:25-92
        assert np.array_equal(poses[i], pose_array(name)), name


@pytest.mark.parametrize("seed,kind,pose", [(s, k, p) for s, k in SCENE_SKINS for p in [None] + BUILTIN_POSE_ORDER],
                         ids=[f"{s}-{k}-{p}" for s, k in SCENE_SKINS for p in [None] + BUILTIN_POSE_ORDER])
def test_skin_scene_builder_equals_pins(mclib, seed, kind, pose):
    """The scenes of test_skin_scene_builder_equals_live_reference without the reference: equal to the digests in
    tests/golden/oracle_pins.json (the builder's output, not the reference's)."""
    assert scene_digest(mclib.build_skin_scene(synth_skin(seed, kind), pose)) == pins()["scenes"][f"{seed}/{kind}/{pose}"]


def test_skin_scene_builder_drops_transparent_overlay(mclib):
    """A fully transparent outer layer is dropped (mesh_builder.cpp:176-186); legacy skins keep 7 boxes."""
    scene = mclib.build_skin_scene(overlay_atlas())
    assert len(scene.boxes) == 11 and scene_digest(scene) == pins()["scenes"]["overlay_dropped"]
    assert len(mclib.build_skin_scene(synth_skin(2, "legacy")).boxes) == 7


def test_skin_layout_equals_the_scene_builder(mclib):
    """mcskin_skin_layout (what render_skin_batch runs per skin before the device cuts the texel pool): the same boxes
    and face windows as mcskin_build_skin_scene, and face sources that reproduce its texel pool from the atlas bytes."""
    cases = [(synth_skin(0), None), (synth_skin(2, "legacy"), "walking"), (synth_skin(3, "slim"), "dab")]
    a = synth_skin(5)
    a[:16, 32:, 3] = 0          # head overlay fully transparent: dropped
    a[16:32, 16:40, 3] = 255    # (body inner stays opaque)
    cases.append((a, "running"))
    b = synth_skin(6)
    b[..., 3] = 255             # no holes at all
    cases.append((b, None))
    for atlas, pose in cases:
        scene = mclib.build_skin_scene(atlas, pose)
        boxes, faces, opaque, n_texels = mclib.skin_layout(atlas, pose)
        assert boxes.tobytes() == np.ascontiguousarray(scene.boxes).tobytes()
        assert n_texels == len(scene.texels) and len(faces) == 6 * len(boxes)
        pool = np.zeros((n_texels, 4), dtype=np.float32)
        for dst, x, y, w, h, mirror in faces:
            win = atlas[y:y + h, x:x + w].astype(np.float32) / np.float32(255.0)
            if mirror:
                win = win[:, ::-1]
            pool[dst:dst + w * h] = win.reshape(-1, 4)
        assert np.array_equal(pool.view(np.uint32), np.ascontiguousarray(scene.texels, dtype=np.float32).view(np.uint32))
        for i, bx in enumerate(boxes):
            alphas = np.concatenate([pool[o:o + w * h, 3] for o, w, h in bx["face"]])
            assert bool(opaque[i]) == bool((alphas != 0).all()), i
    with pytest.raises(mclib.McSkinError):
        mclib.skin_layout(np.zeros((48, 64, 4), dtype=np.uint8))


def test_skin_scene_builder_rejects_bad_sizes(mclib):
    with pytest.raises(mclib.McSkinError) as e:
        mclib.build_skin_scene(np.zeros((48, 64, 4), dtype=np.uint8))
    assert "expected 64x64 or 64x32" in str(e.value)       # skin_parser.cpp:127-131


def test_generate_tiles_matches_oracle(mclib, oracle):
    for args in ((1920, 1080, 32), (100, 70, 32), (7, 5, 3), (64, 64, 64), (0, 5, 5), (5, 5, -1)):
        assert np.array_equal(mclib.generate_tiles(*args), oracle.generate_tiles(*args)), args


def test_band_rows(mclib):
    cfg = make_config(width=1920, height=1080, tile_size=32)
    raw = mclib.raw()
    total = sum(raw.mcskin_cuda_band_rows(C.byref(cfg), C.c_int32(r), C.c_int32(8)) for r in range(8))
    assert total == 1080
    assert raw.mcskin_cuda_band_rows(C.byref(cfg), C.c_int32(1), C.c_int32(8)) == 5 * 32 - (34 * 32 - 1080)  # rows 1,9,17,25,33 (33 clipped)
    assert raw.mcskin_cuda_band_rows(C.byref(cfg), C.c_int32(40), C.c_int32(8)) == 0


def test_no_cpu_fallback(mclib):
    """Without a CUDA device every compute entry point fails loudly with MC_ERR_NO_DEVICE."""
    if mclib.device_count() > 0:
        pytest.skip("a CUDA device is present")
    scene = mclib.build_skin_scene(synth_skin(0))
    cfg = make_config(width=32, height=32)
    for call in (lambda: mclib.render(scene, cfg), lambda: mclib.aov(scene, cfg), lambda: mclib.Context(0),
                 lambda: mclib.intersect(scene, np.zeros(1, dtype=_abi.RAY_DTYPE))):
        with pytest.raises(mclib.McSkinError) as e:
            call()
        assert e.value.code == _abi.MC_ERR_NO_DEVICE


def test_argument_errors_do_not_need_a_device(mclib):
    raw = mclib.raw()
    assert raw.mcskin_cuda_render(None, None, 0, None, None, C.cast(None, _abi.McProgressFn), None, None) == _abi.MC_ERR_INVALID
    assert b"null" in raw.mcskin_cuda_last_error()
    # a zero-tile frame is an empty success (tile_renderer.cpp:144-146), with or without a GPU
    f32, _, stats = mclib.render(FlatScene(), make_config(width=0, height=16))
    assert f32.shape == (16, 0, 4) and stats["n_tiles"] == 0


def test_synth_skin_is_deterministic():
    a, b = synth_skin(3), synth_skin(3)
    assert np.array_equal(a, b) and a.shape == (64, 64, 4) and synth_skin(3, "legacy").shape == (32, 64, 4)
    assert not np.array_equal(a, synth_skin(4))
    holes = a[..., 3] == 0
    assert 0.1 < holes[:16, 32:].mean() < 0.9 and not holes[:16, :32].any()   # only outer-layer blocks have holes


def _libm_sincos(angles):
    """sinf / cosf of the host's libm (what the reference calls per soft-shadow / lens / AO sample)."""
    import ctypes.util
    libm = C.CDLL(ctypes.util.find_library("m") or "libm.so.6")
    libm.sinf.restype = libm.cosf.restype = C.c_float
    libm.sinf.argtypes = libm.cosf.argtypes = [C.c_float]
    sn = np.array([libm.sinf(float(a)) for a in angles], dtype=np.float32)
    cs = np.array([libm.cosf(float(a)) for a in angles], dtype=np.float32)
    return sn, cs


def _host_has_fma():
    try:
        return " fma " in Path("/proc/cpuinfo").read_text()
    except OSError:
        return False


def sincos_test_angles(n=200_000, seed=7):
    """Angles the path produces (2*pi*u for canonical draws u) plus the branch boundaries of the algorithm."""
    rng = np.random.default_rng(seed)
    u = (rng.integers(0, 2**32, size=n, dtype=np.uint64).astype(np.float32) * np.float32(2.0**-32))
    u = np.minimum(u, np.float32(0.99999994))
    two_pi = np.float32(2.0) * np.float32(np.pi)
    angles = [two_pi * u, rng.uniform(-119.9, 119.9, size=n // 4).astype(np.float32)]
    edges = np.array([0.0, 2.0**-13, 2.0**-12, np.pi / 4, np.pi / 2, np.pi, 3 * np.pi / 2, 2 * np.pi, 119.99], dtype=np.float32)
    for e in edges:  # every float within 64 ulps of each boundary
        bits = np.float32(e).view(np.uint32).astype(np.int64) + np.arange(-64, 65)
        angles.append(bits[bits >= 0].astype(np.uint32).view(np.float32))
    return np.concatenate(angles).astype(np.float32)


@pytest.mark.skipif(not _host_has_fma(), reason="glibc selects its non-FMA sinf/cosf on this CPU")
def test_sincos_model_equals_libm(mclib):
    """The restated glibc sincosf (host model of the device function) is bit-identical to libm's sinf/cosf."""
    a = sincos_test_angles(60_000)
    want_s, want_c = _libm_sincos(a)
    got_s, got_c = mclib.sincos_model(a)
    assert np.array_equal(got_s.view(np.uint32), want_s.view(np.uint32))
    assert np.array_equal(got_c.view(np.uint32), want_c.view(np.uint32))


def _libm_powf(x, y):
    import ctypes.util
    libm = C.CDLL(ctypes.util.find_library("m") or "libm.so.6")
    libm.powf.restype = C.c_float
    libm.powf.argtypes = [C.c_float, C.c_float]
    return np.array([libm.powf(float(a), float(b)) for a, b in zip(x, y)], dtype=np.float32)


def powf_test_values(n=100_000, seed=11):
    """(x, y) pairs: N.H values in [0, 1] raised to shininess-like exponents, plus the ranges where the
    result underflows, subnormal x, x slightly above 1, and special values that take the fallback."""
    rng = np.random.default_rng(seed)
    x = [rng.random(n).astype(np.float32), (1.0 - rng.random(n // 4) ** 4).astype(np.float32),
         rng.integers(1, 0x40000000, size=n // 2, dtype=np.uint32).view(np.float32),      # any positive float <= 2
         np.array([0.0, 1.0, 1.0000001, 0.99999994, 1e-39, 5e-45, 0.5, 2.0], dtype=np.float32)]
    x = np.concatenate(x)
    y = rng.choice(np.array([16.0, 32.0, 8.0, 64.0, 1.0, 2.0, 0.5, 100.5, 3.7, 12.25], dtype=np.float32), size=len(x))
    return x.astype(np.float32), y.astype(np.float32)


@pytest.mark.skipif(not _host_has_fma(), reason="glibc selects its non-FMA powf on this CPU")
def test_powf_model_equals_libm(mclib):
    x, y = powf_test_values(40_000)
    got = mclib.powf_model(x, y)
    assert np.array_equal(got.view(np.uint32), _libm_powf(x, y).view(np.uint32))


@pytest.mark.parametrize("width,height,tile,first,stride", [(1920, 1080, 32, 0, 1), (1920, 1080, 32, 1, 3), (300, 200, 16, 0, 1),
                                                             (300, 200, 16, 2, 4), (97, 131, 32, 0, 2), (64, 64, 32, 1, 2)])
@pytest.mark.parametrize("parts", [(1, 1), (3, 1), (4, 2)])
def test_primary_launch_order_covers_every_tile_part_once(mclib, width, height, tile, first, stride, parts):
    """The primary pass launches the figure's tiles first and may split them over several blocks: every
    (tile, part) of the band must be rendered by exactly one block, heavy tiles ahead of the rest."""
    scene = mclib.build_skin_scene(synth_skin(0), "walking")
    cfg = make_config(width=width, height=height, tile_size=tile, samples_per_pixel=4)
    t, p, n = mclib.primary_launch_order(scene, cfg, first, stride, parts_heavy=parts[0], parts_light=parts[1])
    tiles_x, tiles_y = -(-width // tile), -(-height // tile)
    rows = len(range(first, tiles_y, stride))
    n_tiles = rows * tiles_x
    assert t.min() >= 0 and t.max() < n_tiles and set(t.tolist()) == set(range(n_tiles))
    seen = set(zip(t.tolist(), p.tolist()))
    assert len(seen) == len(t)                                     # no (tile, part) twice
    per_tile = {}
    for ti, ni in zip(t.tolist(), n.tolist()):
        assert per_tile.setdefault(ti, ni) == ni                   # one split factor per tile
    assert all((ti, k) in seen for ti, ni in per_tile.items() for k in range(ni))
    assert set(per_tile.values()) <= {max(parts), parts[1]}
    heavy = [ti for ti, ni in per_tile.items() if ni == max(parts)] if parts[0] > parts[1] else []
    if heavy:                                                      # split tiles come first, and form a rectangle of tiles
        first_light = next((i for i, ni in enumerate(n.tolist()) if ni == parts[1]), len(n))
        assert set(t[:first_light].tolist()) == set(heavy)
        cols, rws = sorted({h % tiles_x for h in heavy}), sorted({h // tiles_x for h in heavy})
        assert len(heavy) == len(cols) * len(rws) and cols == list(range(cols[0], cols[-1] + 1))


def libm_golden():
    return np.load(ROOT / "tests" / "golden" / "libm_vectors.npz")


def test_sincos_and_powf_models_equal_golden_libm_vectors(mclib):
    """Host models of the device's sinf/cosf/powf against committed outputs of glibc 2.39 (FMA variants),
    whatever libm variant this host would pick (tests/golden/make_libm_golden.py)."""
    g = libm_golden()
    sn, cs = mclib.sincos_model(g["angles"])
    assert np.array_equal(sn.view(np.uint32), g["sin"].view(np.uint32))
    assert np.array_equal(cs.view(np.uint32), g["cos"].view(np.uint32))
    pw = mclib.powf_model(g["pow_x"], g["pow_y"])
    assert np.array_equal(pw.view(np.uint32), g["pow"].view(np.uint32))


def test_partition_tiles_covers_the_frame_and_balances(mclib):
    """mcskin_partition_tiles (host code): disjoint parts that cover every tile once, deterministic, and balanced
    by the cost model — checked against the oracle's hit mask: the parts' shares of the pixels that hit the
    figure differ by a few percent where interleaved tile rows differ by 14 % at 8 parts."""
    from minecraftskin_raytracer_b200 import _abi
    from minecraftskin_raytracer_b200.scene import synth_skin
    from oracle.harness import Oracle
    scene = mclib.build_skin_scene(synth_skin(0), None)
    cfg = _abi.default_config(width=1920, height=1080, samples_per_pixel=16, max_bounces=4)
    ts = cfg.tile_size
    tx, ty = (cfg.width + ts - 1) // ts, (cfg.height + ts - 1) // ts
    hit = Oracle().aov(scene, cfg) >= 0
    per_tile = np.array([[hit[r * ts:(r + 1) * ts, c * ts:(c + 1) * ts].sum() for c in range(tx)] for r in range(ty)]).reshape(-1)
    for n in (1, 2, 3, 8):
        parts = [mclib.partition_tiles(scene, cfg, n, p) for p in range(n)]
        again = [mclib.partition_tiles(scene, cfg, n, p) for p in range(n)]
        assert all(np.array_equal(a, b) for a, b in zip(parts, again))
        assert sorted(np.concatenate(parts).tolist()) == list(range(tx * ty))
        # (tile COUNTS may differ by what one figure tile weighs in background tiles: the deal balances cost)
        assert max(len(p) for p in parts) - min(len(p) for p in parts) <= max(2, 51 if n > 1 else 0)
        # the background tiles of a part are a contiguous run in frame order: few rectangles on the way to a host frame
        hot_cols = [c for c in range(tx) if per_tile.reshape(ty, tx)[:, c].any()]
        hot_rows = [r for r in range(ty) if per_tile.reshape(ty, tx)[r].any()]
        for p in parts:
            light = [t for t in p.tolist() if not (min(hot_rows) - 1 <= t // tx <= max(hot_rows) + 1 and min(hot_cols) - 1 <= t % tx <= max(hot_cols) + 1)]
            if light:
                inside = [t for t in range(min(light), max(light) + 1)
                          if not (min(hot_rows) - 1 <= t // tx <= max(hot_rows) + 1 and min(hot_cols) - 1 <= t % tx <= max(hot_cols) + 1)]
                assert len(inside) - len(light) <= 4 * (max(hot_cols) - min(hot_cols) + 3), (n, len(inside), len(light))
        share = np.array([per_tile[p].sum() for p in parts], dtype=np.float64)
        assert share.max() / share.mean() < 1.05, (n, share)
    rows = np.array([per_tile.reshape(ty, tx)[r::8].sum() for r in range(8)], dtype=np.float64)
    assert rows.max() / rows.mean() > 1.10  # what the interleaved tile rows of round 1 gave
    # degenerate inputs
    empty = _abi.default_config(width=0, height=10)
    assert len(mclib.partition_tiles(scene, empty, 4, 0)) == 0
    small = _abi.default_config(width=40, height=40)   # 4 tiles over 8 parts: some parts get none
    parts = [mclib.partition_tiles(scene, small, 8, p) for p in range(8)]
    assert sorted(np.concatenate(parts).tolist()) == [0, 1, 2, 3]
    with pytest.raises(mclib.McSkinError):
        mclib.partition_tiles(scene, cfg, 4, 4)


def test_host_copy_threads(mclib):
    """The host threads that carry finished pieces of a frame into pageable images (csrc/host_copy.cpp): pitched rows,
    aligned (streaming stores) and unaligned (memcpy) ends, more pieces than rows, several callers at once."""
    import threading
    rng = np.random.default_rng(3)
    for row_bytes, rows, dst_off, src_off, pieces in ((30720, 97, 0, 0, 8), (30720, 97, 4, 0, 5), (1000, 13, 0, 16, 64),
                                                       (64, 1, 0, 0, 3), (4096, 700, 16, 32, 37), (17, 5, 1, 3, 2)):
        src_pitch, dst_pitch = row_bytes + 48, row_bytes + 80
        src = rng.integers(0, 256, size=src_off + src_pitch * rows + 64, dtype=np.uint8)
        dst = np.full(dst_off + dst_pitch * rows + 64, 0xEE, dtype=np.uint8)
        mclib.host_copy_rows(dst[dst_off:], src[src_off:], row_bytes, rows, pieces, dst_pitch=dst_pitch, src_pitch=src_pitch)
        want = np.full_like(dst, 0xEE)
        for r in range(rows):
            want[dst_off + r * dst_pitch: dst_off + r * dst_pitch + row_bytes] = src[src_off + r * src_pitch: src_off + r * src_pitch + row_bytes]
        assert np.array_equal(dst, want), (row_bytes, rows, dst_off, src_off, pieces)
    # concurrent callers share the pool one call at a time
    src = rng.integers(0, 256, size=(6, 1 << 20), dtype=np.uint8)
    dst = np.zeros_like(src)
    threads = [threading.Thread(target=lambda i=i: [mclib.host_copy_rows(dst[i], src[i], 4096, 256, 16) for _ in range(5)]) for i in range(6)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert np.array_equal(dst, src)
    with pytest.raises(mclib.McSkinError):
        mclib.host_copy_rows(dst[0], src[0], 4096, 4, 2, dst_pitch=100)

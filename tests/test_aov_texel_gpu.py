"""The texel plane (include/mcskin_cuda.h McAovTargets::texel) on the GPU: all six planes bit for bit the CPU oracle of
the planes (tests/texel_oracle.c) through every path that renders a pixel, without changing a bit of the colour; any
subset of the planes may be asked for; and for a skin, lib.skin_texel_atlas turns the plane into atlas pixels."""
import numpy as np
import pytest

from tests.golden.make_texel_pins import free_texel_scenes
from tests.scenes import RENDER_CASES, make_config, synth_skin
from tests.test_aov_guides_gpu import GUIDE_MODES, MODE_CASES, _assert_planes_equal, _bits, _context_frames
from tests.test_parity_gpu import _flip_budget

pytestmark = pytest.mark.gpu

PLANES = ("coverage", "depth", "tri_id", "normal", "albedo", "texel")
CASES = {c[0]: c for c in RENDER_CASES}
FREE = {name: (scene, cfg) for name, scene, cfg in free_texel_scenes()}

_ORACLE = {}


def _oracle_case(name, rng_mode):
    if (name, rng_mode) not in _ORACLE:
        from oracle.harness import Oracle
        from minecraftskin_raytracer_b200 import lib
        from tests.texel_oracle import render_aovs
        if name in FREE:
            scene, cfg = FREE[name]
        else:
            _, seed, kind, pose, over = CASES[name]
            scene = lib.build_skin_scene(synth_skin(seed, kind), pose)
            cfg = make_config(**over, rng_mode=rng_mode)
        _ORACLE[(name, rng_mode)] = (scene, cfg, Oracle().render(scene, cfg), render_aovs(scene, cfg))
    return _ORACLE[(name, rng_mode)]


class Planes:
    """Device planes for n images of h x w pixels, filled with sentinels the renderer never writes; `only` picks a subset."""

    def __init__(self, n, h, w, only=PLANES):
        import torch
        shapes = {"coverage": (), "depth": (), "tri_id": (), "normal": (3,), "albedo": (4,), "texel": ()}
        self.only = tuple(only)
        self.t = {p: torch.empty((n, h, w) + shapes[p], dtype=torch.int32 if p in ("tri_id", "texel") else torch.float32,
                                 device="cuda:0") for p in self.only}
        self.fill()

    def fill(self):
        import torch
        for p in self.only:
            self.t[p].fill_(-7)
        torch.cuda.synchronize()

    def set_on(self, ctx):
        ctx.set_aov_targets(**{p: self.t[p].data_ptr() for p in self.only})

    def host(self, i=0):
        return {p: self.t[p][i].cpu().numpy() for p in self.only}


def _check_frame(gpu, name, rng_mode, opts, only=PLANES):
    from tests.conftest import pixel_report
    scene, cfg, want_img, want = _oracle_case(name, rng_mode)
    planes = Planes(1, cfg.height, cfg.width, only)
    with_aov, without_aov, got = _context_frames(gpu, scene, cfg, opts, planes)
    assert np.array_equal(_bits(with_aov), _bits(without_aov))   # the planes change no bit of the colour
    exact = _flip_budget() == 0.0
    if exact:
        assert np.array_equal(_bits(with_aov), _bits(want_img))
    else:
        assert pixel_report(with_aov, want_img, lambda a: np.clip(a * 255 + 0.5, 0, 255).astype(np.uint8))["within1"] >= 0.999
    _assert_planes_equal(got, want, exact)
    return got


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("case", list(CASES), ids=list(CASES))
def test_texel_plane_parity_every_case(gpu, case, rng_mode):
    _check_frame(gpu, case, rng_mode, {})


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("case", MODE_CASES)
@pytest.mark.parametrize("mode", [m for m in GUIDE_MODES if m != "default"])
def test_texel_plane_parity_modes(gpu, case, mode, rng_mode):
    _check_frame(gpu, case, rng_mode, GUIDE_MODES[mode])


@pytest.mark.parametrize("only", [("texel",), ("tri_id", "texel"), ("albedo", "texel"), PLANES], ids=lambda o: "+".join(o))
@pytest.mark.parametrize("mode", ["default", "megakernel", "tiny_queue"])
def test_texel_plane_subsets(gpu, only, mode):
    _check_frame(gpu, "jitter4", 0, GUIDE_MODES[mode], only)


@pytest.mark.parametrize("mode", ["default", "megakernel"])
@pytest.mark.parametrize("name", list(FREE))
def test_texel_plane_free_scenes(gpu, name, mode):
    """Magenta and blank faces, posed boxes at the rotation thresholds, an outer layer seen from inside, nested boxes
    and the 33- and 212-box scenes."""
    _check_frame(gpu, name, 0, GUIDE_MODES[mode])


def test_texel_plane_follows_the_target_into_a_captured_graph(gpu):
    """On one context, after the frame's graph has been captured and replayed, pointing texel at a second buffer makes
    the same frame write the plane there (the graph key holds the texel pointer)."""
    import torch
    scene, cfg, _, want = _oracle_case("jitter4", 0)
    exact = _flip_budget() == 0.0
    ctx = gpu.Context(0)
    try:
        ctx.set_scene(scene, cfg)
        out = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
        first, second = Planes(1, cfg.height, cfg.width), Planes(1, cfg.height, cfg.width, ("texel",))
        first.set_on(ctx)
        for _ in range(3):  # direct, capture, replay
            ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
            ctx.sync()
        _assert_planes_equal(first.host(), want, exact)
        first.fill()
        ctx.set_aov_targets(**{p: first.t[p].data_ptr() for p in PLANES if p != "texel"},
                            texel=second.t["texel"].data_ptr())
        for _ in range(2):
            ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
            ctx.sync()
        _assert_planes_equal(second.host(), want, exact)
        assert (first.host()["texel"] == -7).all()
    finally:
        ctx.close()


def test_render_aovs_texel(gpu):
    """mcskin_cuda_render_aovs with texel=True: the oracle's texel plane next to the other planes and mcskin_cuda_render's
    colour; without it, the planes of before; a frame without tiles gives -1."""
    scene, cfg, _, want = _oracle_case("headline_small", 1)
    exact = _flip_budget() == 0.0
    f32, _, planes, stats = gpu.render_aovs(scene, cfg, guides=True, texel=True)
    assert set(planes) == set(PLANES)
    assert planes["texel"].shape == (cfg.height, cfg.width) and planes["texel"].dtype == np.int32
    _assert_planes_equal(planes, want, exact)
    assert np.array_equal(_bits(f32), _bits(gpu.render(scene, cfg)[0]))
    f32_t, _, only_texel, _ = gpu.render_aovs(scene, cfg, texel=True)
    assert set(only_texel) == {"coverage", "depth", "tri_id", "texel"}
    assert np.array_equal(only_texel["texel"], planes["texel"])
    _, _, plain, _ = gpu.render_aovs(scene, cfg)
    assert set(plain) == {"coverage", "depth", "tri_id"}
    _, _, guides, _ = gpu.render_aovs(scene, cfg, guides=True)
    assert set(guides) == set(PLANES) - {"texel"}
    assert np.array_equal(_bits(f32_t), _bits(f32))
    assert int((planes["texel"] >= 0).sum()) == stats["n_active_pixels"]
    empty_cfg = make_config(width=50, height=40, tile_size=0, samples_per_pixel=2)
    _, _, empty, _ = gpu.render_aovs(scene, empty_cfg, texel=True)
    assert (empty["texel"] == -1).all()


def test_texel_plane_split_renders(gpu):
    """Three tile sets of partition_tiles (one context each) and tile rows of stride 2 write the whole frame's planes."""
    import torch
    scene, cfg, _, want = _oracle_case("legacy_walk", 0)
    exact = _flip_budget() == 0.0
    frame = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
    planes = Planes(1, cfg.height, cfg.width)
    ctxs = [gpu.Context(0) for _ in range(3)]
    try:
        for c in ctxs:
            c.set_scene(scene, cfg)
            planes.set_on(c)
        parts = [gpu.partition_tiles(scene, cfg, 3, r) for r in range(3)]
        for _ in range(3):  # direct, capture, replay
            planes.fill()
            for r in range(3):
                ctxs[r].render_tiles_into_frame(parts[r], frame.data_ptr(), 0, 0)
                ctxs[r].sync()
            _assert_planes_equal(planes.host(), want, exact)
        for _ in range(3):
            planes.fill()
            for r in range(2):
                ctxs[0].render_rows_into_frame(r, 2, frame.data_ptr(), 0, 0)
                ctxs[0].sync()
            _assert_planes_equal(planes.host(), want, exact)
    finally:
        for c in ctxs:
            c.close()


def _batch(gpu, mode, n=7):
    """(colour, per-image planes, scenes, cfg) of a batch of n skins rendered with all six planes, and checks that the
    colour is the same without planes."""
    import torch
    from minecraftskin_raytracer_b200.scene import BUILTIN_POSE_ORDER, pose_array
    cfg = make_config(width=48, height=40, samples_per_pixel=4, max_bounces=2)
    atlases = np.stack([synth_skin(300 + i, "slim" if i % 3 == 2 else "64x64") for i in range(n)])
    p12 = np.stack([pose_array(BUILTIN_POSE_ORDER[i % len(BUILTIN_POSE_ORDER)]) for i in range(n)])
    scenes = [gpu.build_skin_scene(atlases[i], p12[i]) for i in range(n)]
    ctx = gpu.Context(0)
    try:
        if mode == "frame_by_frame":
            ctx.set_option("batch_mode", 0)
        if mode == "grouped_small_groups":
            ctx.set_option("batch_group", 3)
        outs = {}
        planes = Planes(n, cfg.height, cfg.width)
        for with_planes in (True, False):
            out = torch.zeros((n, cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
            if with_planes:
                planes.set_on(ctx)
            else:
                ctx.set_aov_targets()
            for _ in range(2):  # buffers and staging are reused
                planes.fill()
                if mode == "skin_batch":
                    ctx.render_skin_batch(atlases, cfg, p12, out.data_ptr(), 0, 0)
                else:
                    ctx.render_batch(scenes, cfg, out.data_ptr(), 0, 0)
                ctx.sync()
                if with_planes:
                    got = [planes.host(i) for i in range(n)]
            outs[with_planes] = out.cpu().numpy()
        assert np.array_equal(_bits(outs[True]), _bits(outs[False]))
        return outs[True], got, scenes, cfg
    finally:
        ctx.close()


@pytest.mark.parametrize("mode", ["grouped", "grouped_small_groups", "frame_by_frame", "skin_batch"])
def test_texel_plane_batches(gpu, mode):
    """Image i's six planes of render_batch / render_skin_batch equal the oracle's for scene i: its texel indexes scene
    i's own pool."""
    from tests.texel_oracle import render_aovs
    _, got, scenes, cfg = _batch(gpu, mode)
    exact = _flip_budget() == 0.0
    for i, scene in enumerate(scenes):
        _assert_planes_equal(got[i], render_aovs(scene, cfg), exact)


def test_skin_batch_planes_equal_render_batch(gpu):
    """render_skin_batch (scenes built on the device) gives the colour and planes render_batch gives for
    build_skin_scene's scenes of the same atlases and poses."""
    img_skin, got_skin, _, _ = _batch(gpu, "skin_batch")
    img, got, _, _ = _batch(gpu, "grouped")
    assert np.array_equal(_bits(img_skin), _bits(img))
    for a, b in zip(got_skin, got):
        for p in PLANES:
            assert np.array_equal(_bits(a[p]), _bits(b[p])), p


@pytest.mark.parametrize("kind,seed,pose", [("64x64", 40, "walking"), ("legacy", 41, "running"), ("slim", 42, None)])
def test_skin_texel_atlas_end_to_end(gpu, kind, seed, pose):
    """A skin at one sample per pixel: the atlas pixel skin_texel_atlas gives for each covered pixel's texel, / 255, is
    the albedo plane there; uncovered pixels map to (-1, -1)."""
    atlas = synth_skin(seed, kind)
    scene = gpu.build_skin_scene(atlas, pose)
    cfg = make_config(width=96, height=128, samples_per_pixel=1, max_bounces=1)
    _, _, planes, _ = gpu.render_aovs(scene, cfg, guides=True, texel=True)
    xy = gpu.skin_texel_atlas(atlas)[planes["texel"]]
    covered = planes["texel"] >= 0
    assert covered.any() and (xy[~covered] == -1).all()
    rgba = atlas[xy[covered][:, 1], xy[covered][:, 0]].astype(np.float32) / np.float32(255.0)
    assert np.array_equal(_bits(rgba), _bits(planes["albedo"][covered]))

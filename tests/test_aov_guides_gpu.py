"""The guide planes (normal, albedo; include/mcskin_cuda.h McAovTargets) on the GPU: all five planes bit for bit the CPU
oracle of the planes (tests/guide_oracle.c) through every path that renders a pixel, without changing a bit of the colour;
and any subset of the planes may be asked for."""
import numpy as np
import pytest

from tests.conftest import pixel_report
from tests.scenes import RENDER_CASES, make_config, synth_skin
from tests.test_parity_gpu import _flip_budget

pytestmark = pytest.mark.gpu

PLANES = ("coverage", "depth", "tri_id", "normal", "albedo")
CASES = {c[0]: c for c in RENDER_CASES}
# the context options of the render paths: the wavefront (shade_mode 0, its chunked form, its overflowing hit queue and
# the megakernel it hands pixels beyond its paths to), the two megakernels, tiles split over blocks, frame lanes
GUIDE_MODES = {
    "default": {},
    "megakernel": {"shade_mode": 1},
    "megakernel_warp": {"shade_mode": 2},
    "chunked": {"record_budget_bytes": 4096},
    "tiny_queue": {"wave_queue_pct": 1},
    "tiny_wave_budget": {"wave_budget_bytes": 1 << 20},
    "split_tiles": {"primary_blocks_per_sm": 100000},
    "one_lane_no_graph": {"frame_lanes": 1, "use_graphs": 0, "cache_tile_seeds": 0},
    "five_lanes": {"frame_lanes": 5},
}
# the cases every mode runs (every case runs in the default mode): posed and unposed, 1..300 samples, lens, warp and
# pixel resolve, tiles of 7
MODE_CASES = ["headline_small", "jitter4", "legacy_walk", "fighting_dof", "tile7_spp3", "spp300"]


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


_ORACLE = {}


def _oracle_case(name, rng_mode):
    if (name, rng_mode) not in _ORACLE:
        from oracle.harness import Oracle
        from minecraftskin_raytracer_b200 import lib
        from tests.guide_oracle import render_aovs
        _, seed, kind, pose, over = CASES[name]
        scene = lib.build_skin_scene(synth_skin(seed, kind), pose)
        cfg = make_config(**over, rng_mode=rng_mode)
        _ORACLE[(name, rng_mode)] = (scene, cfg, Oracle().render(scene, cfg), render_aovs(scene, cfg, guides=True))
    return _ORACLE[(name, rng_mode)]


class Planes:
    """Device planes for n images of h x w pixels, filled with sentinels the renderer never writes; `only` picks a subset."""

    def __init__(self, n, h, w, only=PLANES):
        import torch
        shapes = {"coverage": (), "depth": (), "tri_id": (), "normal": (3,), "albedo": (4,)}
        self.only = tuple(only)
        self.t = {p: torch.empty((n, h, w) + shapes[p], dtype=torch.int32 if p == "tri_id" else torch.float32,
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


def _assert_planes_equal(got, want, exact=True):
    for p in got:
        if exact:
            assert np.array_equal(_bits(got[p]), _bits(want[p])), p
        else:  # (non-FMA glibc host: a thin-lens ray may differ in the last ulp; see _flip_budget)
            assert (_bits(got[p]) == _bits(want[p])).mean() >= 0.999, p


def _context_frames(gpu, scene, cfg, opts, planes):
    """Three renders through a context (direct launches, the call that captures the graph, a replay) with the planes
    set, then one without: returns the colour with, the colour without, and the planes."""
    import torch
    ctx = gpu.Context(0)
    try:
        for k, v in opts.items():
            ctx.set_option(k, v)
        ctx.set_scene(scene, cfg)
        out = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
        planes.set_on(ctx)
        colours, got = [], []
        for _ in range(3):
            out.zero_()
            planes.fill()
            ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
            ctx.sync()
            colours.append(out.cpu().numpy())
            got.append(planes.host())
        for k in (1, 2):
            assert np.array_equal(_bits(colours[k]), _bits(colours[0]))
            for p in got[0]:
                assert np.array_equal(_bits(got[k][p]), _bits(got[0][p])), (k, p)
        ctx.set_aov_targets()
        out.zero_()
        torch.cuda.synchronize()
        ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
        ctx.sync()
        return colours[0], out.cpu().numpy(), got[0]
    finally:
        ctx.close()


def _check_frame(gpu, name, rng_mode, opts, only=PLANES):
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


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("case", list(CASES), ids=list(CASES))
def test_guide_planes_parity_every_case(gpu, case, rng_mode):
    _check_frame(gpu, case, rng_mode, {})


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("case", MODE_CASES)
@pytest.mark.parametrize("mode", [m for m in GUIDE_MODES if m != "default"])
def test_guide_planes_parity_modes(gpu, case, mode, rng_mode):
    _check_frame(gpu, case, rng_mode, GUIDE_MODES[mode])


@pytest.mark.parametrize("only", [("normal",), ("albedo",), ("depth", "albedo"), ("normal", "albedo")],
                         ids=lambda o: "+".join(o))
@pytest.mark.parametrize("mode", ["default", "megakernel", "tiny_queue"])
def test_guide_plane_subsets(gpu, only, mode):
    _check_frame(gpu, "jitter4", 0, GUIDE_MODES[mode], only)


def test_render_aovs_guides(gpu):
    """mcskin_cuda_render_aovs with guides=True: the oracle's five planes and mcskin_cuda_render's colour; without, the
    three planes of before; a frame without tiles gives zeros."""
    scene, cfg, _, want = _oracle_case("headline_small", 1)
    exact = _flip_budget() == 0.0
    f32, _, planes, stats = gpu.render_aovs(scene, cfg, guides=True)
    assert set(planes) == set(PLANES)
    assert planes["normal"].shape == (cfg.height, cfg.width, 3) and planes["albedo"].shape == (cfg.height, cfg.width, 4)
    _assert_planes_equal(planes, want, exact)
    assert np.array_equal(_bits(f32), _bits(gpu.render(scene, cfg)[0]))
    f32_plain, _, plain, _ = gpu.render_aovs(scene, cfg)
    assert set(plain) == {"coverage", "depth", "tri_id"}
    assert np.array_equal(_bits(f32_plain), _bits(f32))
    covered = planes["tri_id"] >= 0
    assert np.array_equal(covered, planes["albedo"][..., 3] > 0)
    assert int(covered.sum()) == stats["n_active_pixels"]
    empty_cfg = make_config(width=50, height=40, tile_size=0, samples_per_pixel=2)
    _, _, empty, _ = gpu.render_aovs(scene, empty_cfg, guides=True)
    assert (empty["normal"] == 0).all() and (empty["albedo"] == 0).all()


def test_guide_planes_split_renders(gpu):
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


@pytest.mark.parametrize("mode", ["grouped", "grouped_small_groups", "frame_by_frame", "skin_batch"])
def test_guide_planes_batches(gpu, mode):
    """Image i's five planes of render_batch / render_skin_batch equal the oracle's for skin i, and the colour is the
    same with and without planes."""
    import torch
    from minecraftskin_raytracer_b200.scene import BUILTIN_POSE_ORDER, pose_array
    from tests.guide_oracle import render_aovs
    n = 7
    cfg = make_config(width=48, height=40, samples_per_pixel=4, max_bounces=2)
    atlases = np.stack([synth_skin(300 + i, "64x64") for i in range(n)])
    p12 = np.stack([pose_array(BUILTIN_POSE_ORDER[i % len(BUILTIN_POSE_ORDER)]) for i in range(n)])
    poses = list(p12) if mode == "skin_batch" else [BUILTIN_POSE_ORDER[i % len(BUILTIN_POSE_ORDER)] if i % 3 else None
                                                    for i in range(n)]
    scenes = [gpu.build_skin_scene(atlases[i], poses[i]) for i in range(n)]
    exact = _flip_budget() == 0.0
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
        for i in range(n):
            _assert_planes_equal(got[i], render_aovs(scenes[i], cfg, guides=True), exact)
    finally:
        ctx.close()

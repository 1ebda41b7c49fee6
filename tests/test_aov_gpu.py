"""AOV planes on the GPU (coverage, depth, tri_id; include/mcskin_cuda.h McAovTargets): bit for bit the CPU oracle of the
planes (tests/aov_oracle.c) through every path that renders a pixel, without changing a bit of the colour (the CPU
oracle's, oracle/mcskin_oracle.c)."""
import ctypes as C
from functools import lru_cache

import numpy as np
import pytest

from minecraftskin_raytracer_b200 import _abi
from tests.conftest import pixel_report
from tests.scenes import RENDER_CASES, make_config, synth_skin
from tests.test_parity_gpu import _flip_budget

pytestmark = pytest.mark.gpu

PLANES = ("coverage", "depth", "tri_id")
CASES = {c[0]: c for c in RENDER_CASES}
# the context options of the render paths (a subset of tests/test_parity_gpu.py's RENDER_MODES)
AOV_MODES = {
    "default": {},
    "all_active": {"force_all_active": 1},
    "megakernel": {"shade_mode": 1},
    "megakernel_warp": {"shade_mode": 2},
    "tiny_wave_budget": {"wave_budget_bytes": 1 << 20},
    "tiny_queue": {"wave_queue_pct": 1},
    "split_tiles": {"primary_blocks_per_sm": 100000},
    "one_lane_no_graph": {"frame_lanes": 1, "use_graphs": 0, "cache_tile_seeds": 0},
    "five_lanes": {"frame_lanes": 5},
}


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _scene(lib, seed, kind="64x64", pose=None):
    return lib.build_skin_scene(synth_skin(seed, kind), pose)


@lru_cache(maxsize=None)
def _oracle_case(name, rng_mode):
    from oracle.harness import Oracle
    from minecraftskin_raytracer_b200 import lib
    from tests.aov_oracle import render_aovs
    _, seed, kind, pose, over = CASES[name]
    scene = _scene(lib, seed, kind, pose)
    cfg = make_config(**over, rng_mode=rng_mode)
    return scene, cfg, Oracle().render(scene, cfg), render_aovs(scene, cfg)


class Planes:
    """Device planes for n images of h x w pixels, filled with sentinels the renderer never writes."""

    def __init__(self, n, h, w):
        import torch
        self.t = {"coverage": torch.empty((n, h, w), dtype=torch.float32, device="cuda:0"),
                  "depth": torch.empty((n, h, w), dtype=torch.float32, device="cuda:0"),
                  "tri_id": torch.empty((n, h, w), dtype=torch.int32, device="cuda:0")}
        self.fill()

    def fill(self):
        import torch
        self.t["coverage"].fill_(-7.0)
        self.t["depth"].fill_(-7.0)
        self.t["tri_id"].fill_(-7)
        torch.cuda.synchronize()

    def set_on(self, ctx):
        ctx.set_aov_targets(*(self.t[p].data_ptr() for p in PLANES))

    def host(self, i=0):
        return {p: self.t[p][i].cpu().numpy() for p in PLANES}


def _assert_planes_equal(got, want, exact=True):
    for p in PLANES:
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
            for p in PLANES:
                assert np.array_equal(_bits(got[k][p]), _bits(got[0][p])), (k, p)
        ctx.set_aov_targets()
        out.zero_()
        torch.cuda.synchronize()
        ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
        ctx.sync()
        return colours[0], out.cpu().numpy(), got[0]
    finally:
        ctx.close()


@pytest.mark.parametrize("rng_mode", [0, 1])
@pytest.mark.parametrize("case", list(CASES), ids=list(CASES))
@pytest.mark.parametrize("mode", list(AOV_MODES), ids=list(AOV_MODES))
def test_aov_planes_parity(gpu, case, mode, rng_mode):
    scene, cfg, want_img, want = _oracle_case(case, rng_mode)
    planes = Planes(1, cfg.height, cfg.width)
    with_aov, without_aov, got = _context_frames(gpu, scene, cfg, AOV_MODES[mode], planes)
    assert np.array_equal(_bits(with_aov), _bits(without_aov))   # the planes change no bit of the colour
    exact = _flip_budget() == 0.0
    if exact:
        assert np.array_equal(_bits(with_aov), _bits(want_img))
    else:
        assert pixel_report(with_aov, want_img, lambda a: np.clip(a * 255 + 0.5, 0, 255).astype(np.uint8))["within1"] >= 0.999
    _assert_planes_equal(got, want, exact)


def _render_aovs_into(gpu, scene, cfg, f32, cov, dep, tri):
    targets = _abi.McAovTargets(cov.ctypes.data, dep.ctypes.data, tri.ctypes.data)
    stats = _abi.McRenderStats()
    cs = scene.as_c()
    rc = gpu.raw().mcskin_cuda_render_aovs(C.byref(cs), C.byref(cfg), C.c_int32(0), C.c_void_p(f32.ctypes.data), None,
                                          C.byref(targets), C.byref(stats))
    assert rc == 0, gpu.last_error()


def test_render_aovs_host_forms(gpu):
    """mcskin_cuda_render_aovs into pageable and page-locked destinations equals the context form, also when the
    context renders the frame in chunks; the colour is mcskin_cuda_render's."""
    import torch
    scene, cfg, _, want = _oracle_case("headline_small", 0)
    f32, u8, planes, stats = gpu.render_aovs(scene, cfg, want_u8=True)
    plain, plain_u8, _ = gpu.render(scene, cfg, want_u8=True)
    assert np.array_equal(_bits(f32), _bits(plain)) and np.array_equal(u8, plain_u8)
    _assert_planes_equal(planes, want, _flip_budget() == 0.0)
    assert stats["n_active_pixels"] == int((planes["tri_id"] >= 0).sum())
    h, w = cfg.height, cfg.width
    pinned = {"f32": torch.zeros((h, w, 4), dtype=torch.float32).pin_memory(),
              "coverage": torch.zeros((h, w), dtype=torch.float32).pin_memory(),
              "depth": torch.zeros((h, w), dtype=torch.float32).pin_memory(),
              "tri_id": torch.zeros((h, w), dtype=torch.int32).pin_memory()}
    arrs = {k: v.numpy() for k, v in pinned.items()}
    _render_aovs_into(gpu, scene, cfg, arrs["f32"], arrs["coverage"], arrs["depth"], arrs["tri_id"])
    assert np.array_equal(_bits(arrs["f32"]), _bits(f32))
    for p in PLANES:
        assert np.array_equal(_bits(arrs[p]), _bits(planes[p])), p
    dev = Planes(1, h, w)
    _, _, chunked = _context_frames(gpu, scene, cfg, {"record_budget_bytes": 4096}, dev)
    for p in PLANES:
        assert np.array_equal(_bits(chunked[p]), _bits(planes[p])), p


@pytest.mark.parametrize("w,h,ts", [(1, 1, 32), (3, 200, 32), (200, 3, 7), (50, 40, 0)])
def test_render_aovs_degenerate_sizes(gpu, oracle, w, h, ts):
    scene = _scene(gpu, 1)
    cfg = make_config(width=w, height=h, tile_size=ts, samples_per_pixel=2, max_bounces=1)
    f32, _, planes, _ = gpu.render_aovs(scene, cfg)
    from tests.aov_oracle import render_aovs
    want = render_aovs(scene, cfg)
    if ts <= 0:  # no tiles: nothing is rendered, every plane keeps its defaults
        assert (planes["coverage"] == 0).all() and (planes["depth"] == 0).all() and (planes["tri_id"] == -1).all()
    _assert_planes_equal(planes, want, _flip_budget() == 0.0)
    assert np.array_equal(_bits(f32), _bits(gpu.render(scene, cfg)[0]))


def test_aov_at_one_sample_equals_pixel_centre_ids(gpu):
    """At 1 spp without a lens the sample ray is the pixel-centre ray of mcskin_cuda_aov."""
    for name in ("c1_small", "sitting_flatbg", "many_shadow_samples"):
        scene, cfg, _, _ = _oracle_case(name, 0)
        _, _, planes, _ = gpu.render_aovs(scene, cfg)
        assert np.array_equal(planes["tri_id"], gpu.aov(scene, cfg)), name
        assert np.array_equal(planes["coverage"], (planes["tri_id"] >= 0).astype(np.float32)), name


def test_aov_split_renders_give_whole_frame_planes(gpu):
    """Three tile sets of partition_tiles (one context each) and tile rows of stride 2 write the whole frame's planes."""
    import torch
    scene = _scene(gpu, 8, "64x64", "running")
    cfg = make_config(width=200, height=330, samples_per_pixel=4, max_bounces=3)
    _, _, want, _ = gpu.render_aovs(scene, cfg)
    frame = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
    planes = Planes(1, cfg.height, cfg.width)
    ctxs = [gpu.Context(0) for _ in range(3)]
    try:
        for c in ctxs:
            c.set_scene(scene, cfg)
            planes.set_on(c)
        parts = [gpu.partition_tiles(scene, cfg, 3, r) for r in range(3)]
        for rep in range(3):  # direct, capture, replay
            planes.fill()
            for r in range(3):
                ctxs[r].render_tiles_into_frame(parts[r], frame.data_ptr(), 0, 0)
                ctxs[r].sync()
            _assert_planes_equal(planes.host(), want)
        for rep in range(3):
            planes.fill()
            for r in range(2):
                ctxs[0].render_rows_into_frame(r, 2, frame.data_ptr(), 0, 0)
                ctxs[0].sync()
            _assert_planes_equal(planes.host(), want)
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("mode", ["grouped", "grouped_small_groups", "frame_by_frame", "skin_batch"])
def test_aov_batches(gpu, mode):
    """Image i's planes of render_batch / render_skin_batch equal a single render of skin i."""
    import torch
    from minecraftskin_raytracer_b200.scene import BUILTIN_POSE_ORDER, pose_array
    n = 13
    cfg = make_config(width=64, height=64, samples_per_pixel=4, max_bounces=2)
    atlases = np.stack([synth_skin(200 + i, "64x64") for i in range(n)])
    poses = [BUILTIN_POSE_ORDER[i % len(BUILTIN_POSE_ORDER)] if i % 4 else None for i in range(n)]
    p12 = np.stack([pose_array(p) if p is not None else pose_array(BUILTIN_POSE_ORDER[0]) for p in poses])
    if mode == "skin_batch":  # per-skin poses, as 12 numbers each
        poses = list(p12)
    scenes = [gpu.build_skin_scene(atlases[i], poses[i]) for i in range(n)]
    ctx = gpu.Context(0)
    try:
        if mode == "frame_by_frame":
            ctx.set_option("batch_mode", 0)
        if mode == "grouped_small_groups":
            ctx.set_option("batch_group", 5)
        out = torch.zeros((n, 64, 64, 4), dtype=torch.float32, device="cuda:0")
        planes = Planes(n, 64, 64)
        planes.set_on(ctx)
        for _ in range(2):  # buffers and staging are reused
            planes.fill()
            if mode == "skin_batch":
                ctx.render_skin_batch(atlases, cfg, p12, out.data_ptr(), 0, 0)
            else:
                ctx.render_batch(scenes, cfg, out.data_ptr(), 0, 0)
            ctx.sync()
        for i in range(n):
            f32, _, want, _ = gpu.render_aovs(scenes[i], cfg)
            assert np.array_equal(_bits(out[i].cpu().numpy()), _bits(f32)), i
            _assert_planes_equal(planes.host(i), want)
    finally:
        ctx.close()


def test_aov_targets_off_leaves_old_planes_untouched(gpu):
    """Targets switched off: the next frames (direct, graph capture, replay) write no plane, also after a graph was
    captured with targets set; render_scene_tiles refuses to run while targets are set."""
    import torch
    scene, cfg, _, want = _oracle_case("jitter4", 0)
    out = torch.zeros((cfg.height, cfg.width, 4), dtype=torch.float32, device="cuda:0")
    planes = Planes(1, cfg.height, cfg.width)
    ctx = gpu.Context(0)
    try:
        ctx.set_scene(scene, cfg)
        planes.set_on(ctx)
        for _ in range(3):  # the graph of this frame is captured with the targets set
            ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
            ctx.sync()
        _assert_planes_equal(planes.host(), want, _flip_budget() == 0.0)
        with pytest.raises(gpu.McSkinError):
            ctx.render_scene_tiles(scene, cfg, np.arange(4, dtype=np.int32))
        ctx.set_aov_targets()
        planes.fill()
        for _ in range(4):
            ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
            ctx.sync()
        got = planes.host()
        assert (got["coverage"] == -7.0).all() and (got["depth"] == -7.0).all() and (got["tri_id"] == -7).all()
        planes.set_on(ctx)  # and on again: the planes come back
        ctx.render_bands(0, 1, out.data_ptr(), 0, 0)
        ctx.sync()
        _assert_planes_equal(planes.host(), want, _flip_budget() == 0.0)
    finally:
        ctx.close()


def test_aov_invariants_headline_small(gpu):
    scene, cfg, _, _ = _oracle_case("headline_small", 0)
    _, _, planes, stats = gpu.render_aovs(scene, cfg)
    miss = planes["tri_id"] == -1
    assert np.array_equal(miss, planes["coverage"] == 0) and np.array_equal(miss, planes["depth"] == 0)
    assert int((~miss).sum()) == stats["n_active_pixels"]
    assert 0 < (~miss).mean() < 1

"""Free scenes: cameras, lights and box layouts away from the one skin setup the render cases use (pure data).

Every builder is deterministic (seeded numpy generators only) and returns (name, FlatScene, McConfig); its name says
which conservative gate of the product it aims at:
  * screen rectangles (host_prep.cpp prepare_frame: the figure's and every box's projected rectangle, given up when a
    corner is not in front of the camera or the camera basis is degenerate);
  * the two-level reject pass (a box "enclosed" by another with 1e-3 to spare) and the per-chunk masks of scenes with
    more than 32 boxes;
  * the shadow bundles (bundle_box_mask grows a box by radius * 1.01 + 0.01), the opaque shortcut and posed boxes;
  * face-texel quotients (kBoxRecip off for a size whose significand is all ones);
  * the seed memo window [-2^20, 2^23 - 2^20) of FreshStream::seed_memo;
  * paths deeper than the 64 bounce levels the device keeps, and frame shapes at the edges of the tile arithmetic.
Frames are small so that the CPU oracle renders all of them in seconds.
"""
from __future__ import annotations

import dataclasses

import numpy as np

from minecraftskin_raytracer_b200 import _abi
from minecraftskin_raytracer_b200.scene import FlatScene, make_box, synth_skin

SKIN_SEED = 31


def _cfg(**kw):
    base = dict(width=64, height=64, samples_per_pixel=2, max_bounces=2)
    base.update(kw)
    return _abi.default_config(**base)


def _f3(v):
    return tuple(float(x) for x in np.asarray(v, dtype=np.float32))


def skin(pose="walking", seed=SKIN_SEED, kind="64x64") -> FlatScene:
    from minecraftskin_raytracer_b200 import lib
    return lib.build_skin_scene(synth_skin(seed, kind), pose)


def translated(scene: FlatScene, offset) -> FlatScene:
    """The whole scene (boxes, pivots, camera, light) moved by `offset` (float32 adds)."""
    off = np.asarray(offset, dtype=np.float32)
    boxes = scene.boxes.copy()
    for f in ("bounds_min", "bounds_max", "pivot"):
        boxes[f] = boxes[f] + off
    return dataclasses.replace(scene, boxes=boxes, cam_pos=_f3(np.float32(scene.cam_pos) + off),
                               cam_target=_f3(np.float32(scene.cam_target) + off),
                               light_pos=_f3(np.float32(scene.light_pos) + off))


def texel_pool(rng: np.random.Generator, n: int = 4096) -> np.ndarray:
    """Random opaque RGBA texels with holes (alpha 0) in about one in six."""
    t = rng.random((n, 4), dtype=np.float32)
    t[:, 3] = 1.0
    t[rng.random(n) < 1 / 6, 3] = 0.0
    return t


def random_faces(rng: np.random.Generator, n_texels: int):
    """Six face windows into the pool: mostly real windows, some magenta (offset < 0), some blank (width <= 0)."""
    faces = []
    for _ in range(6):
        r = rng.random()
        if r < 0.1:
            faces.append((-1, 4, 4))
        elif r < 0.2:
            faces.append((0, 0 if rng.random() < 0.5 else -3, 4))
        else:
            w, h = int(rng.integers(1, 9)), int(rng.integers(1, 9))
            faces.append((int(rng.integers(0, n_texels - w * h + 1)), w, h))
    return faces


def opaque_faces(rng, pool_opaque_from: int, n_texels: int):
    """Windows into the opaque tail of a pool (see _scene_with_opaque_tail)."""
    faces = []
    for _ in range(6):
        w, h = int(rng.integers(1, 9)), int(rng.integers(1, 9))
        faces.append((int(rng.integers(pool_opaque_from, n_texels - w * h + 1)), w, h))
    return faces


def _pool_with_opaque_tail(rng, n=4096, opaque=1024):
    t = texel_pool(rng, n)
    t[n - opaque:, 3] = 1.0
    return t, n - opaque


def _box_scene(boxes, texels, **kw) -> FlatScene:
    return FlatScene(boxes=np.array(boxes, dtype=_abi.BOX_DTYPE), texels=texels, **kw)


# ---------------------------------------------------------------------------------------------------- cameras
def _look(scene, pos, target, up=(0.0, 1.0, 0.0), fov=60.0):
    return dataclasses.replace(scene, cam_pos=_f3(pos), cam_target=_f3(target), cam_up=_f3(up), cam_fov_deg=float(fov))


def camera_scenes():
    out = []
    rng = np.random.default_rng(101)
    centre = np.array([0.0, 16.0, 0.0])
    for k in range(4):
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        dist = rng.uniform(8.0, 120.0)
        up = rng.normal(size=3)
        fov = rng.uniform(10.0, 120.0)
        pose = ["walking", "dab", None, "fighting"][k]
        out.append((f"cam_orbit_{k}", _look(skin(pose), centre + d * dist, centre + rng.uniform(-3, 3, 3), up, fov),
                    _cfg(width=64, height=56)))
    # the figure runs past every edge of the frame: rectangles reach beyond the frame and below 0
    out.append(("cam_closeup_clipped", _look(skin("running"), (3.0, 20.0, 9.0), (0.0, 18.0, 0.0), fov=70.0), _cfg()))
    # inside the figure's bounds but in no box: the head's corners are behind the camera (no rectangles at all)
    out.append(("cam_inside_figure_bounds", _look(skin(None), (0.0, 10.0, 3.5), (0.0, 4.0, -10.0), fov=90.0),
                _cfg(max_bounces=1)))
    # inside the head's outer layer (between it and the head), looking out through its holes
    out.append(("cam_inside_outer_layer", _look(skin(None), (0.0, 28.0, 4.25), (2.0, 26.0, 40.0), fov=100.0),
                _cfg(max_bounces=1)))
    # up parallel to the view direction: a degenerate camera basis (no projection possible; every ray goes straight ahead)
    out.append(("cam_up_parallel", _look(skin("walking"), (0.0, 18.0, 50.0), (0.0, 18.0, 0.0), up=(0.0, 0.0, -1.0)),
                _cfg(width=48, height=48)))
    out.append(("cam_fov1", _look(skin("dab"), (0.0, 18.0, 600.0), (0.0, 26.0, 0.0), fov=1.0), _cfg(width=48, height=48)))
    out.append(("cam_fov170", _look(skin("waving"), (0.0, 18.0, 20.0), (0.0, 18.0, 0.0), fov=170.0), _cfg()))
    out.append(("frame_300x20", skin("walking"), _cfg(width=300, height=20, samples_per_pixel=4, max_bounces=1)))
    out.append(("frame_20x300", skin("dab"), _cfg(width=20, height=300, samples_per_pixel=4, max_bounces=1)))
    return out


# ---------------------------------------------------------------------------------------------------- lights
def light_scenes():
    out = []
    base_cfg = dict(width=64, height=64, samples_per_pixel=2, max_bounces=1, shadow_samples=8)
    for tag, r in (("r0", 0.0), ("r5e-5", 5e-5), ("r1e-3", 1e-3), ("r0.5", 0.5), ("r15", 15.0), ("r40", 40.0)):
        out.append((f"light_{tag}", dataclasses.replace(skin("walking"), light_radius=float(np.float32(r))), _cfg(**base_cfg)))
    lights = [
        ("light_in_inner_box", (0.0, 28.0, 0.0), 1.0),              # inside the head
        ("light_between_layers", (0.0, 28.0, 4.25), 0.2),           # between the head and its outer layer
        ("light_near_face", (0.0, 18.0, 2.55), 0.5),                # 0.05 in front of the body's outer layer
        ("light_on_box_bound", (4.5, 32.5, 30.0), 3.0),             # two coordinates equal to the head overlay's bounds
        ("light_below", (0.0, -30.0, 10.0), 3.0),
        ("light_behind_camera", (5.0, 20.0, 80.0), 3.0),
    ]
    for name, pos, radius in lights:
        out.append((name, dataclasses.replace(skin("fighting"), light_pos=_f3(pos), light_radius=radius), _cfg(**base_cfg)))
    return out


# ---------------------------------------------------------------------------------------------------- boxes
def random_box_scene(seed: int, n: int) -> FlatScene:
    """Boxes of non-integer sizes 0.01-40 around the default camera's view, windows into a pool with holes, magenta and
    blank faces, some boxes with no triangles, some posed."""
    rng = np.random.default_rng(seed)
    texels = texel_pool(rng)
    boxes = []
    for i in range(n):
        size = np.exp(rng.uniform(np.log(0.01), np.log(40.0), 3)).astype(np.float32)
        centre = np.array([rng.uniform(-18, 18), rng.uniform(0, 36), rng.uniform(-12, 10)], dtype=np.float32)
        lo, hi = centre - size / np.float32(2), centre + size / np.float32(2)
        posed = rng.random() < 0.3
        boxes.append(make_box(lo, hi, random_faces(rng, len(texels)), outer=bool(rng.random() < 0.3),
                              pivot=centre + rng.uniform(-6, 6, 3).astype(np.float32), rot_x=float(rng.uniform(-180, 180)) if posed else 0.0,
                              rot_z=float(rng.uniform(-180, 180)) if posed else 0.0, has_rotation=posed,
                              n_triangles=0 if rng.random() < 0.1 else 12))
    return _box_scene(boxes, texels, light_pos=(3.0, 45.0, 28.0), light_radius=2.0)


def nested_scene(spare_minus_step: bool) -> FlatScene:
    """Chains of three nested boxes and children inside their parent by exactly the reject pass's 1e-3 (float32: child
    lo = parent lo + 1e-3f, hi = parent hi - 1e-3f), or by one float step less on one side of each child."""
    rng = np.random.default_rng(7 if spare_minus_step else 8)
    texels = texel_pool(rng)
    eps = np.float32(1e-3)
    boxes = []
    for cx in (-9.0, 0.0, 9.0):
        lo = np.array([cx - 4.3, 6.7, -4.1], dtype=np.float32)
        hi = np.array([cx + 4.1, 30.3, 3.9], dtype=np.float32)
        chain = [(lo, hi)]
        for _ in range(2):  # three deep, 0.6 to spare
            lo, hi = lo + np.float32(0.6), hi - np.float32(0.6)
            chain.append((lo, hi))
        for j, (l, h) in enumerate(chain):
            boxes.append(make_box(l, h, random_faces(rng, len(texels)), outer=j == 0))
    for px in (-9.0, 0.0, 9.0):  # exact-spare children of the outer box at the same x as a chain
        plo = np.array([px - 3.0, 33.0, -2.0], dtype=np.float32)
        phi = np.array([px + 3.0, 38.5, 2.0], dtype=np.float32)
        clo, chi = plo + eps, phi - eps
        if spare_minus_step:
            axis = int(px > 0) + int(px > -1)
            clo[axis] = np.nextafter(clo[axis], np.float32(-np.inf))  # one float step beyond the spare
        boxes.append(make_box(plo, phi, random_faces(rng, len(texels)), outer=True))
        boxes.append(make_box(clo, chi, random_faces(rng, len(texels))))
    return _box_scene(boxes, texels, light_pos=(-4.0, 44.0, 30.0), light_radius=2.5)


def touching_scene() -> FlatScene:
    rng = np.random.default_rng(9)
    texels, opaque_from = _pool_with_opaque_tail(rng)
    f = lambda: opaque_faces(rng, opaque_from, len(texels))  # noqa: E731
    g = lambda: random_faces(rng, len(texels))  # noqa: E731
    boxes = [
        make_box((-8, 4, -3), (0, 14, 3), f()), make_box((0, 4, -3), (8, 14, 3), g()),          # touch at x = 0
        make_box((-8, 14, -3), (8, 20, 3), f()),                                                  # on top of both
        make_box((-6, 20, -2), (-1, 26, 2), g()), make_box((-6, 20, -2), (-1, 26, 2), f()),      # coincident boxes
        make_box((2, 20, -2), (6, 26, 2), g()), make_box((2.0, 22.5, -2.0), (6.0, 30.0, 1.0), f()),  # coincident faces
    ]
    return _box_scene(boxes, texels, light_pos=(6.0, 40.0, 25.0), light_radius=3.0)


def degenerate_sizes_scene() -> FlatScene:
    """Zero-thickness boxes (the size a face-texel quotient divides by becomes 1.0), and a size whose significand is
    all ones (no host reciprocal: kBoxRecip cleared) beside sizes with one."""
    rng = np.random.default_rng(10)
    texels = texel_pool(rng)
    all_ones = np.uint32(0x40FFFFFF).view(np.float32)   # 7.9999995: significand all ones
    boxes = [
        make_box((-10, 8, 0), (-4, 20, 0), random_faces(rng, len(texels))),                 # zero depth
        make_box((-3, 10, -2), (3, 10, 2), random_faces(rng, len(texels))),                 # zero height
        make_box((-2.5, 22, -1), (np.float32(-2.5) + all_ones, 30, 2), [(0, 8, 8)] * 6),
        make_box((6, 22, -1), (14, 30, 2), [(0, 8, 8)] * 6),                                # size 8: reciprocal kept
        make_box((4, 8, -1), (np.float32(4) + all_ones, np.float32(8) + all_ones, np.float32(-1) + all_ones),
                 random_faces(rng, len(texels))),
    ]
    return _box_scene(boxes, texels, light_pos=(0.0, 40.0, 30.0), light_radius=1.5)


def posed_thresholds_scene() -> FlatScene:
    """Posed boxes at the |rot| > 0.01 thresholds of kBoxRotX / kBoxRotZ (0.01 exactly and one float above), 0.005
    with has_rotation set, 90, 180, -180 and arbitrary angles, pivots away from the box, opaque and holed boxes."""
    rng = np.random.default_rng(11)
    texels, opaque_from = _pool_with_opaque_tail(rng)
    above = float(np.nextafter(np.float32(0.01), np.float32(1)))
    poses = [(0.01, 0.0), (above, 0.0), (0.0, 0.01), (0.0, above), (0.005, 0.005), (90.0, 0.0), (0.0, 180.0),
             (-180.0, 0.0), (37.3, -71.9), (-123.4, 15.5), (180.0, -180.0), (63.0, 90.0)]
    boxes = []
    for i, (rx, rz) in enumerate(poses):
        col, row = i % 4, i // 4
        lo = np.array([-15 + 8 * col, 4 + 10 * row, -2], dtype=np.float32)
        hi = lo + np.array([4.3, 6.1, 3.7], dtype=np.float32)
        far = i % 3 == 2
        pivot = (lo + hi) / np.float32(2) + (np.float32([0.0, 7.5, -3.0]) if far else np.float32([0.2, 1.0, 0.0]))
        faces = opaque_faces(rng, opaque_from, len(texels)) if i % 2 == 0 else random_faces(rng, len(texels))
        boxes.append(make_box(lo, hi, faces, pivot=pivot, rot_x=rx, rot_z=rz, has_rotation=True, outer=i % 4 == 3))
    return _box_scene(boxes, texels, light_pos=(2.0, 42.0, 28.0), light_radius=3.0)


def many_boxes_scene(n: int, seed: int) -> FlatScene:
    """n > 32 boxes: the masks are derived per chunk of 32 and there are no screen rectangles.  Boxes 32, 35, 38, ... are
    empty (no triangles) and sit right in view, in front of the others."""
    rng = np.random.default_rng(seed)
    texels = texel_pool(rng)
    boxes = []
    for i in range(n):
        col, row = i % 8, (i // 8) % 8
        lo = np.array([-16 + 4 * col, 2 + 4.5 * row, -2 - 0.5 * (i // 64)], dtype=np.float32)
        lo += rng.uniform(0, 0.4, 3).astype(np.float32)
        hi = lo + rng.uniform(1.5, 3.5, 3).astype(np.float32)
        empty = i >= 32 and i % 3 == 2
        if empty:  # an empty box in front of the others: any hit on it is wrong
            lo[2], hi[2] = np.float32(4.0), np.float32(6.0)
        boxes.append(make_box(lo, hi, random_faces(rng, len(texels)), n_triangles=0 if empty else 12,
                              has_rotation=i % 11 == 5, rot_x=25.0 if i % 11 == 5 else 0.0, pivot=(lo + hi) / np.float32(2)))
    return _box_scene(boxes, texels, light_pos=(0.0, 45.0, 30.0), light_radius=2.0)


def largest_scene(extra: int = 0) -> FlatScene:
    """The most boxes whose blob fits the 40 KB shared-memory staging area (SceneBlobLayout: 48 B a box padded to 4 plus
    the 144-byte box records), or `extra` more."""
    n = MAX_STAGED_BOXES + extra
    rng = np.random.default_rng(12)
    texels = texel_pool(rng, 1024)
    boxes = []
    for i in range(n):
        col, row = i % 16, i // 16
        lo = np.array([-16 + 2 * col, 2 + 2.2 * row, -1 + 0.1 * (i % 5)], dtype=np.float32)
        boxes.append(make_box(lo, lo + np.float32([1.6, 1.7, 1.3]), random_faces(rng, len(texels)), n_triangles=0 if i % 17 == 16 else 12))
    return _box_scene(boxes, texels, light_pos=(0.0, 45.0, 30.0), light_radius=2.0)


MAX_STAGED_BOXES = 212  # 48 * 212 + 144 * 212 = 40 704 <= 40 960 bytes; 213 boxes need 48 * 216 + 144 * 213 = 41 040


def box_scenes():
    out = []
    for k, n in enumerate((10, 12, 9)):
        out.append((f"boxes_random_{k}", random_box_scene(200 + k, n), _cfg(samples_per_pixel=2, max_bounces=2)))
    out.append(("nest_chains_exact_spare", nested_scene(False), _cfg(max_bounces=2)))
    out.append(("nest_spare_minus_one_step", nested_scene(True), _cfg(max_bounces=2)))
    out.append(("boxes_touching_coincident", touching_scene(), _cfg(max_bounces=2)))
    out.append(("boxes_zero_thickness_all_ones_size", degenerate_sizes_scene(), _cfg(max_bounces=2)))
    out.append(("posed_rotation_thresholds", posed_thresholds_scene(), _cfg(max_bounces=2, shadow_samples=13)))
    out.append(("boxes_33", many_boxes_scene(33, 301), _cfg(max_bounces=2)))
    out.append(("boxes_64", many_boxes_scene(64, 302), _cfg(max_bounces=1)))
    out.append(("boxes_212_largest_staged", largest_scene(), _cfg(width=48, height=48, samples_per_pixel=1, max_bounces=1)))
    # the same scene through the warp form of the primary pass (lens draws at 16 spp), whose static shared memory plus
    # the blob passes 48 KB
    out.append(("boxes_212_warp_form", largest_scene(), _cfg(width=48, height=48, samples_per_pixel=16, max_bounces=1,
                                                             dof_enabled=1, aperture=0.3)))
    return out


# ---------------------------------------------------------------------------------------------------- seed memo window
MEMO_OFFSETS = {"memo_window_top": (0.0, 90.0, 0.0), "memo_window_bottom": (0.0, -30.0, 0.0),
                "memo_int64_wrap": (0.0, 1e5, 0.0)}


def memo_scenes():
    return [(name, translated(skin("walking"), off), _cfg(width=64, height=64, samples_per_pixel=2, max_bounces=2))
            for name, off in MEMO_OFFSETS.items()]


# ---------------------------------------------------------------------------------------------------- mirrors, frame edges
def mirror_scene() -> FlatScene:
    """Two large opaque boxes facing each other 12 apart, the camera between them looking at one: every camera ray
    bounces between them far beyond the 64 levels the device keeps."""
    texels = np.tile(np.float32([0.8, 0.7, 0.6, 1.0]), (16, 1))
    faces = [(0, 4, 4)] * 6
    boxes = [make_box((-400, -400, -12), (400, 400, -6), faces), make_box((-400, -400, 6), (400, 400, 12), faces)]
    return FlatScene(boxes=np.array(boxes, dtype=_abi.BOX_DTYPE), texels=texels, light_pos=(0.0, 3.0, 0.0),
                     light_radius=1.0, cam_pos=(0.0, 0.0, 4.0), cam_target=(0.3, 0.2, -6.0), cam_fov_deg=20.0)


def edge_scenes():
    return [
        ("mirrors_70", mirror_scene(), _cfg(width=16, height=16, samples_per_pixel=1, max_bounces=70, shadow_samples=2)),
        ("mirrors_200", mirror_scene(), _cfg(width=12, height=12, samples_per_pixel=1, max_bounces=200, soft_shadows=0)),
        ("frame_65535x2", skin("walking"), _cfg(width=65535, height=2, samples_per_pixel=4, max_bounces=1)),
        ("frame_tile1", skin("dab"), _cfg(width=24, height=20, samples_per_pixel=2, max_bounces=1, tile_size=1)),
        ("frame_1x1", _look(skin(None), (0.0, 18.0, 50.0), (0.0, 18.0, 0.0), fov=5.0), _cfg(width=1, height=1, samples_per_pixel=4)),
    ]


def free_scenes():
    """Every free scene, in a fixed order."""
    return camera_scenes() + light_scenes() + box_scenes() + memo_scenes() + edge_scenes()

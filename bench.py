#!/usr/bin/env python
"""bench.py — headline benchmark of the render hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl own|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one frame of the headline workload of BASELINE.json
("1080p 16spp 4-bounce": synthetic 64x64 skin seed 0, standing pose, 1920x1080,
16 spp, 4 bounces, reference defaults otherwise: soft shadows x8, gradient
background, 32x32 tiles).  Metric: M unique rays/s, where the unique-ray count of the
frame is the fixed integer the reference algorithm performs (intersectScene calls
minus the redundant re-test, counted by the CPU oracle: tests/golden/work_counts.json).

value    : frame time measured with CUDA events, scene resident on the device, output
           left in device memory (N>1: every rank stores its tiles into rank 0's frame over
           NVLink peer memory; the barrier that completes the frame is inside the step).
e2e      : the same frame through the public host API (host scene in, host image out,
           host<->device copies inside the timed region).  N>1: every rank uploads the scene
           and its kernels store its tiles into ONE page-locked host frame (shared memory).
roofline : FP32 issue roofline (SURVEY.md §8d): algorithmic lane-ops of the frame /
           event time / (SMs x 128 lanes x max SM clock).
Outside the timed region the line also carries: `sustained` (>= 2 s of back-to-back frames),
`cold_first_frame_ms`, `ms_per_step_with_tile_seed`, `extra_workloads` (BASELINE configs C2, C3, C5
and the C4 batch at this N) and `cpu_baseline` (the reference's CPU renderer on this box's cores).

--dump-outputs DIR writes the frame the last timed step computed (float32 RGBA, height x width x 4) as
DIR/frame.npy; the inputs are fixed, so two builds can be compared output for output.  (Under the
MCSKIN_BENCH_SPLIT tuning aid the step renders one part of the frame, and only that part is filled.)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it (it may be read-only)

WORKLOAD = "headline_1080p_16spp_4b"
# ncu counters of one frame of the committed code (tools/ncu_frame_counters.py): warp instructions and DRAM bytes
FRAME_COUNTERS = ROOT / "profiles" / "r02" / "frame_counters.json"

# BASELINE.json configs other than the headline (SURVEY.md §8d "Configs restated"), timed outside the headline's
# timed region: (name, skin seed, skin kind, pose, config overrides)
EXTRA_FRAMES = [
    ("c2_legacy_1080p_4spp_4b", 2, "legacy", None, dict(width=1920, height=1080, samples_per_pixel=4, max_bounces=4)),
    ("c3_slim_4k_16spp_4b", 3, "slim", None, dict(width=3840, height=2160, samples_per_pixel=16, max_bounces=4)),
    ("c5_8k_64spp_8b", 5, "64x64", None, dict(width=7680, height=4320, samples_per_pixel=64, max_bounces=8)),
    # SURVEY §8d secondary rows of the headline: pose 1 ("walking", 8 rotated boxes) and hard shadows
    ("headline_walking_1080p_16spp_4b", 0, "64x64", "walking", dict(width=1920, height=1080, samples_per_pixel=16, max_bounces=4)),
    ("headline_hard_shadows_1080p_16spp_4b", 0, "64x64", None, dict(width=1920, height=1080, samples_per_pixel=16, max_bounces=4, soft_shadows=0)),
    # not the reference's frame: the headline with McConfig.rng_mode 1 (counter-based streams, DESIGN.md §3) — equal to
    # the oracle with the same switch, reported beside the mt19937 number, never in its place
    ("headline_counter_rng_1080p_16spp_4b", 0, "64x64", None, dict(width=1920, height=1080, samples_per_pixel=16, max_bounces=4, rng_mode=1)),
]
C4_SKINS_PER_GPU = 512
C4_CONFIG = dict(width=256, height=256, samples_per_pixel=4, max_bounces=2)


def load_counts():
    return json.loads((ROOT / "tests" / "golden" / "work_counts.json").read_text())


def alg_ops(entry: dict) -> dict:
    """Algorithmic FP32 lane-ops of one frame (SURVEY.md §8d work model, DESIGN.md "Work model")."""
    c = entry["counters"]
    cfg = entry["config"]
    P, R = entry["n_boxes_plain"], entry["n_boxes_rotated"]
    S = c["n_primary_rays"]
    rays = entry["unique_rays"]
    n_shadow_samples = 8  # reference default (raytracer.h:19); the workloads do not override it
    per_ray = 6 + 28 * P + 74 * R
    primary = 35 * S + S * per_ray + 21 * c["n_background_primary"] + (4 * cfg["samples_per_pixel"] + 5) * cfg["width"] * cfg["height"]
    secondary = ((rays - S) * per_ray + 26 * (c["n_slab_pass"] + c["n_backface_eval"]) + 48 * c["n_rotated_hits"]
                 + 118 * c["n_shade"] + (60 + 42 * n_shadow_samples) * c["n_soft_shadow"] + 20 * c["n_hard_shadow"]
                 + 68 * c["n_reflect_rays"])
    return {"total": primary + secondary, "primary_pass": primary, "shade_pass": secondary}


def measured_peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text())
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "_fallback": True}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the benchmark runs; every sample is time-stamped so
    that the samples of a given window (the timed region, the sustained leg) can be picked out afterwards."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index: int, period_ms: int = 20):
        self.gpu_index = gpu_index
        self.period_ms = period_ms
        self.proc = None
        self.samples: list[tuple[float, float, float, list[str]]] = []  # (time, sm MHz, max MHz, reasons)
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.period_ms), "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm, smax = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            reasons = [n for n, v in zip(self.NAMES, parts[5:9]) if v.lower().startswith("active")]
            self.samples.append((time.time(), sm, smax, reasons))

    def wait_for_samples(self, n: int = 1, timeout_s: float = 5.0):
        """nvidia-smi takes a moment to produce its first line: block until it has (or give up)."""
        t0 = time.time()
        while self.proc is not None and len(self.samples) < n and time.time() - t0 < timeout_s:
            time.sleep(0.01)

    def window(self, t0: float, t1: float, pad_s: float = 0.0) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        rows = [s for s in list(self.samples) if t0 - pad_s <= s[0] <= t1 + pad_s]
        reasons = sorted({r for s in rows for r in s[3]})
        return {"sm_mhz": statistics.median(s[1] for s in rows) if rows else None,
                "sm_max_mhz": max(s[2] for s in rows) if rows else None, "reasons": reasons, "samples": len(rows)}

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def dump_frame(out_dir: str, frame: np.ndarray):
    """DIR/frame.npy: the float32 RGBA frame of the last timed step (1080p: 33 MB)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "frame.npy"), np.ascontiguousarray(frame, dtype=np.float32))


# ------------------------------------------------------------------------- reference arm
def cpu_reference_run(entry_name: str, steps: int, warmup: int):
    """Times the reference's own CPU renderer (oracle/_ref when it was built, else the C port)."""
    from minecraftskin_raytracer_b200 import _abi
    from minecraftskin_raytracer_b200.scene import synth_skin
    from oracle.harness import Oracle, Reference
    counts = load_counts()
    entry = counts[entry_name]
    ref = Reference.load()
    kind = "reference" if ref is not None else "port"
    runner = ref if ref is not None else Oracle()
    cores = runner.hardware_threads()
    cfg = _abi.default_config(**entry["config"])
    # scene through the checker's own builder when it has one (reference), else the product's host builder
    if ref is not None:
        scene = ref.scene_from_atlas(synth_skin(entry["skin_seed"], entry["skin_kind"]), entry["pose"])
    else:
        from minecraftskin_raytracer_b200 import lib
        scene = lib.build_skin_scene(synth_skin(entry["skin_seed"], entry["skin_kind"]), entry["pose"])
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        image = runner.render(scene, cfg)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return {"value": entry["unique_rays"] / sec / 1e6, "unit": "Mrays/s", "cores": cores, "kind": kind, "image": image,
            "sample": f"{entry_name}: the full {entry['config']['width']}x{entry['config']['height']} frame at "
                      f"{entry['config']['samples_per_pixel']} spp ({entry['unique_rays']} unique rays) through "
                      f"TileRenderer::render, threadCount=0, mean of {len(times)} run(s) after {warmup} warm-up run(s)",
            "ms_per_sample": sec * 1e3}


def run_reference_arm(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    # every step is the whole headline frame (16 spp): the same config as the own arm's step
    res = cpu_reference_run(WORKLOAD, args.steps, args.warmup)
    if args.dump_outputs:
        dump_frame(args.dump_outputs, res["image"])
    counts = load_counts()
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": res["value"], "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_sample"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "step_sample": WORKLOAD, "width": 1920, "height": 1080, "spp": 16, "max_bounces": 4,
                   "unique_rays_per_frame": counts[WORKLOAD]["unique_rays"]},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- own arm
class FrameJob:
    """One frame workload on this rank: a context with the scene resident, this rank's share of the frame
    (the whole frame at N=1, its cost-balanced tile set at N>1) and where the pixels go."""

    def __init__(self, torch, dist, lib, bands, scene, cfg, rank, world, local_rank, stream, emulate=0, exchange="p2p"):
        self.torch, self.dist, self.lib, self.bands = torch, dist, lib, bands
        self.scene, self.cfg, self.rank, self.world, self.local_rank, self.stream = scene, cfg, rank, world, local_rank, stream
        self.dev = torch.device("cuda", local_rank)
        self.H, self.W, self.ts = cfg.height, cfg.width, cfg.tile_size
        self.ctx = lib.Context(local_rank)
        self.ctx.set_scene(scene, cfg)
        self.split = emulate if emulate > 1 else world
        self.exchange = exchange if world > 1 else "none"
        self.peer = None
        self.tiles = None
        self.diag = os.environ.get("MCSKIN_BENCH_DIAG", "")  # "local" / "nofence": see step()
        if self.diag == "local":
            self.local_frame = torch.zeros((self.H, self.W, 4), dtype=torch.float32, device=self.dev)
        if self.split > 1 and self.exchange != "gather":
            part = int(os.environ.get("MCSKIN_BENCH_PART", "0")) if emulate > 1 else rank
            # value: rank 0 holds the frame, the others store into it over NVLink (their background tiles count a little more)
            self.tiles = lib.partition_tiles(scene, cfg, self.split, part, 0 if (self.exchange == "p2p" and not emulate) else -1)
            self.tiles_host = lib.partition_tiles(scene, cfg, self.split, part, -1)  # e2e: every rank writes to the host frame
        if self.exchange == "p2p":
            self.peer = bands.PeerFrame(lib, self.H, self.W, local_rank)
            self.frame_ptr = self.peer.ptr
            self.frame = self.peer.frame
        elif self.exchange == "gather":
            self.max_rows = bands.padded_band_rows(self.H, self.ts, world)
            self.band = torch.zeros((self.max_rows, self.W, 4), dtype=torch.float32, device=self.dev)
            self.gathered = torch.empty((world * self.max_rows, self.W, 4), dtype=torch.float32, device=self.dev) if rank == 0 else None
            self.row_index = bands.frame_row_index(self.H, self.ts, world, self.max_rows, self.dev) if rank == 0 else None
            self.frame = torch.zeros((self.H, self.W, 4), dtype=torch.float32, device=self.dev) if rank == 0 else None
        else:
            self.frame = torch.zeros((self.H, self.W, 4), dtype=torch.float32, device=self.dev)
            self.frame_ptr = self.frame.data_ptr()

    def render_into(self, frame_ptr: int):
        """This rank's share of the frame into a full-frame image at `frame_ptr` (asynchronous)."""
        s = self.stream.cuda_stream
        if self.tiles is not None:
            self.ctx.render_tiles_into_frame(self.tiles, frame_ptr, 0, s)
        else:
            self.ctx.render_rows_into_frame(0, 1, frame_ptr, 0, s)

    def render_local(self):
        """This rank's share without the exchange step."""
        if self.exchange == "gather":
            self.ctx.render_bands(self.rank, self.world, self.band.data_ptr(), 0, self.stream.cuda_stream)
        else:
            self.render_into(self.frame_ptr)

    def step(self):
        if self.exchange == "gather":
            self.ctx.render_bands(self.rank, self.world, self.band.data_ptr(), 0, self.stream.cuda_stream)
            self.bands.gather_frame(self.band, self.frame, self.ts, self.gathered, self.row_index)
        elif self.diag == "local":      # diagnosis only: every rank into a frame of its own, no exchange at all
            self.render_into(self.local_frame.data_ptr())
        elif self.diag == "nofence":    # diagnosis only: peer stores without the barrier
            self.render_into(self.frame_ptr)
        else:
            self.render_into(self.frame_ptr)
            if self.peer is not None:
                self.peer.fence(self.stream.cuda_stream)  # ranks release a flag in the root's memory; the root's stream acquires them

    def release(self):
        """After step(): the root has the frame; the peers may overwrite it (PeerFrame.release)."""
        if self.peer is not None and not self.diag:
            self.peer.release(self.stream.cuda_stream)

    def close(self):
        self.ctx.close()
        if self.peer is not None:
            self.peer.close()


def time_steps(torch, dist, job, flush, steps, warmup, world, dev):
    """W warm-up + K timed steps: CUDA events on the job's stream around every step, an L2 flush before each,
    barrier + synchronize on both sides, max over ranks.  Returns (ms per step, library stats of the last frame,
    ms of this rank's launches per frame — the timed events themselves on one GPU, without the exchange step at
    N>1 —, wall-clock window of the timed loop)."""
    for i in range(warmup):
        flush.fill_(1)
        job.step()
        job.release()
    torch.cuda.synchronize(dev)
    job.ctx.sync()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    w0 = time.time()
    # Every step is queued without a host round trip in between (a rank that synchronised with its host after each frame
    # would start the next one late, and the root, whose queue is already full, would count that as exchange time).
    for i in range(steps):
        flush.fill_(i & 0xff)  # L2 flush between timed iterations (outside the timed events)
        starts[i].record(job.stream)
        job.step()
        ends[i].record(job.stream)
        job.release()  # (untimed) the root is done with the frame: the peers may store the next one
    torch.cuda.synchronize(dev)
    w1 = time.time()
    st = job.ctx.sync()
    if world > 1:
        dist.barrier()
    total_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    if world > 1:
        # this rank's launches without the exchange step: one more frame on its own, the library's events around it
        flush.fill_(1)
        job.render_local()
        device_ms = job.ctx.sync()["ms_device"] * steps
    else:
        device_ms = total_ms  # one GPU: the step IS the frame's launches
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        if os.environ.get("MCSKIN_BENCH_VERBOSE"):  # per-rank view: event time of the step, the library's own kernel time
            mine = torch.tensor([total_ms / steps, device_ms / steps], dtype=torch.float64, device=dev)
            every = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(every, mine)
            if dist.get_rank() == 0:
                print("per-rank ms (step, kernels): " + "  ".join(f"{float(e[0]):.4f}/{float(e[1]):.4f}" for e in every), file=sys.stderr)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps, st, device_ms / steps, (w0, w1)


def run_own_arm(args):
    import torch
    import torch.distributed as dist

    from minecraftskin_raytracer_b200 import _abi, build
    build.build()
    from minecraftskin_raytracer_b200 import bands, lib
    from minecraftskin_raytracer_b200.scene import synth_skin

    rank, local_rank, world = dist_env()
    # tuning aid: time ONE rank's share of an N-way split on a single GPU (no exchange): MCSKIN_BENCH_SPLIT=N
    emulate = int(os.environ.get("MCSKIN_BENCH_SPLIT", "0")) if world == 1 else 0
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    counts = load_counts()
    entry = counts[WORKLOAD]
    cfg = _abi.default_config(**entry["config"])
    W, H, ts = cfg.width, cfg.height, cfg.tile_size
    scene = lib.build_skin_scene(synth_skin(entry["skin_seed"], entry["skin_kind"]), entry["pose"])
    ops = alg_ops(entry)
    unique_rays = entry["unique_rays"]
    lanes_default = int(os.environ.get("MCSKIN_FRAME_LANES", "0")) or lib.DEFAULT_FRAME_LANES
    # a dedicated (non-default) stream: handle 0 would mean "the context's own stream" to the C ABI,
    # and torch.cuda.Event only sees the stream it is recorded on
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # N>1: every rank stores its tiles straight into rank 0's frame over NVLink peer memory and the exchange step is
    # a barrier ("p2p", default); or rank 0 gathers compact bands of interleaved tile rows with NCCL ("gather").
    exchange = os.environ.get("MCSKIN_EXCHANGE", "p2p") if world > 1 else "none"

    # ---- cold first frame: fresh context, buffers not allocated yet, no cached tile seeds, no graph
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    job = FrameJob(torch, dist, lib, bands, scene, cfg, rank, world, local_rank, stream, emulate, exchange)
    job.step()
    job.ctx.sync()
    torch.cuda.synchronize(dev)
    cold_ms = (time.perf_counter() - t0) * 1e3

    # ---- parity of the split (N>1): the frame assembled from every rank's tiles must equal, bit for bit, the frame one GPU
    # renders on its own; and the NCCL gather of interleaved tile rows must give the same bits again
    split_checked = None
    if world > 1:
        job.step()
        torch.cuda.synchronize(dev)
        dist.barrier()
        if job.peer is not None:
            job.peer.check_timeout()
        if rank == 0:
            solo = lib.Context(local_rank)
            solo.set_scene(scene, cfg)
            whole = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
            solo.render_rows_into_frame(0, 1, whole.data_ptr(), 0, stream.cuda_stream)
            solo.sync()
            torch.cuda.synchronize(dev)
            if not torch.equal(job.frame.view(torch.int32), whole.view(torch.int32)):
                raise SystemExit(f"bench.py: the frame assembled from {world} GPUs differs from the single-GPU frame")
            solo.close()
        other = FrameJob(torch, dist, lib, bands, scene, cfg, rank, world, local_rank, stream, 0, "gather" if exchange == "p2p" else "p2p")
        other.step()
        torch.cuda.synchronize(dev)
        dist.barrier()
        if rank == 0 and not torch.equal(other.frame.view(torch.int32), job.frame.view(torch.int32)):
            raise SystemExit("bench.py: peer-written frame differs from the gathered frame")
        other.close()
        split_checked = f"{world}-GPU frame == single-GPU frame == the other exchange's frame, bit for bit"

    # ---- headline: W warm-up + K timed frames
    if rank == 0:
        sampler.wait_for_samples(1)
    ms_per_step, st, device_ms, timed_window = time_steps(torch, dist, job, flush, args.steps, args.warmup, world, dev)
    launches_per_step = st["n_kernel_launches"]
    n_active = st["n_active_pixels"]
    if job.peer is not None:
        job.peer.check_timeout()
    if args.dump_outputs:  # before the legs below render into the same frame again
        if world > 1:
            dist.barrier()  # the peers' stores into the root's frame (time_steps ends with one more) are complete
        if rank == 0:
            dump_frame(args.dump_outputs, job.frame.cpu().numpy())

    # ---- pass breakdown, outside the timed region: the same frame on ONE stream with direct launches
    # (the timed frames interleave several lanes inside a CUDA graph, where pass times overlap)
    pass_ms = {"primary": 0.0, "shade": 0.0}
    job.ctx.set_option("use_graphs", 0)
    job.ctx.set_option("frame_lanes", 1)
    n_serial = max(1, min(args.steps, 5))
    for i in range(1 + n_serial):
        flush.fill_(i & 0xff)
        job.render_local()
        s2 = job.ctx.sync()
        if i > 0:
            pass_ms["primary"] += s2["ms_primary"] / n_serial
            pass_ms["shade"] += s2["ms_shade"] / n_serial
    job.ctx.set_option("use_graphs", 1)
    job.ctx.set_option("frame_lanes", lanes_default)
    if world > 1:
        dist.barrier()

    extras = {}
    nomemo_ms = None
    if not args.kernel_only:
        # ---- sustained: >= 2 s of back-to-back frames (no flush: a frame's queue traffic alone exceeds the L2)
        for _ in range(3):
            job.step()
            job.release()
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        n_sus = max(50, int(2200.0 / max(ms_per_step, 0.05)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0 = time.time()
        e0.record(stream)
        for _ in range(n_sus):
            job.step()
            job.release()  # (the handshake is part of a sustained pipeline: inside this figure)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        s1 = time.time()
        if world > 1:
            dist.barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        sus_ms = float(tt.item()) / n_sus
        extras["sustained"] = {"frames": n_sus, "seconds": float(tt.item()) / 1e3, "ms_per_frame": sus_ms,
                               "value": unique_rays / (sus_ms * 1e-3) / 1e6, "unit": "Mrays/s",
                               "what": "back-to-back frames (CUDA graph replay, no L2 flush between frames), CUDA events around the whole run, max over ranks",
                               "clocks": sampler.window(s0, s1) if rank == 0 else None}
        # ---- the frame with the per-tile engine seeding inside (k_tile_seed; cached across frames of equal geometry otherwise)
        # (and without the memo of the shadow engines' seeding recurrence, shadow_seed_memo: the frame with nothing kept
        # from earlier frames but its buffers and the captured graph)
        job.ctx.set_option("cache_tile_seeds", 0)
        job.ctx.set_option("shadow_seed_memo", 0)
        seed_ms, _, _, _ = time_steps(torch, dist, job, flush, max(3, min(args.steps, 10)), 3, world, dev)
        job.ctx.set_option("cache_tile_seeds", 1)
        job.ctx.set_option("shadow_seed_memo", 1)
        extras["ms_per_step_with_tile_seed"] = seed_ms
        extras["ms_per_step_with_tile_seed_what"] = ("the frame with k_tile_seed inside (cache_tile_seeds 0) and every shaded hit's "
                                                     "engine seeded by the 396-step recurrence (shadow_seed_memo 0)")
        # ---- the configuration the committed ncu capture was taken in (tile seeds kept, no seed memo): the frame
        #      time its instruction count is set against (roofline.frac_executed)
        job.ctx.set_option("shadow_seed_memo", 0)
        nomemo_ms, _, _, _ = time_steps(torch, dist, job, flush, max(3, min(args.steps, 10)), 3, world, dev)
        job.ctx.set_option("shadow_seed_memo", 1)
        extras["ms_per_step_without_seed_memo"] = nomemo_ms

    # ---- e2e: host scene in, host image out, copies inside the timed region
    h2d_bytes = scene.boxes.nbytes + scene.texels.nbytes + C.sizeof(_abi.McScene) + C.sizeof(_abi.McConfig)
    d2h_bytes = H * W * 16
    e2e_ms, e2e_how = None, None
    if args.kernel_only:
        pass
    elif world == 1:
        # the public host call: host scene in (re-flattened, re-uploaded every step), host float image
        # out, into a page-locked result buffer the caller reuses from frame to frame
        host_img = torch.empty((H, W, 4), dtype=torch.float32, pin_memory=True).numpy()
        c_scene = scene.as_c()  # the C view of the host scene (McScene: pointers to the host arrays), built once
        for _ in range(max(1, min(args.warmup, 3))):
            lib.render(c_scene, cfg, device=local_rank, out_f32=host_img)
        e2e_dev = [0.0, 0]
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_dev[0] += lib.render(c_scene, cfg, device=local_rank, out_f32=host_img)[2]["ms_device"]
            e2e_dev[1] += 1
        e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        e2e_how = ("mcskin_cuda_render: host scene in, float image out to a page-locked host buffer (the tiles the figure touches are "
                   "stored by the kernels straight into it, the background tiles leave the device image by DMA after the primary pass, "
                   f"next to the shading kernels); the kernels take {e2e_dev[0] / max(1, e2e_dev[1]):.3f} ms of it")
    else:
        # every rank: host scene -> device, its tiles rendered straight into ONE page-locked host frame (shared memory,
        # mapped into every GPU: N PCIe links carry the image); the step ends when the root has seen every rank publish
        host = bands.HostFrame(lib, H, W)

        e2e_dev = [0.0, 0]
        my_tiles = np.ascontiguousarray(job.tiles_host, dtype=np.int32)
        c_scene = scene.as_c()  # the C view of the host scene, built once

        def e2e_step():
            # one C call: scene upload (re-flattened on the host every step), this rank's tiles into the host frame, wait
            e2e_dev[0] += job.ctx.render_scene_tiles(c_scene, cfg, my_tiles, host.frame)
            e2e_dev[1] += 1
            host.publish()
            if rank == 0:
                host.wait_all()
                host.release()
            else:
                host.wait_released()

        for _ in range(3):
            e2e_step()
        if rank == 0:  # the host frame holds the single-GPU frame's bits
            got = torch.from_numpy(host.frame).view(torch.int32)
            if not torch.equal(got, job.frame.cpu().view(torch.int32)):
                raise SystemExit("bench.py: the host frame written by all ranks differs from the device frame")
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        tt = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_ms = float(tt.item())
        h2d_bytes *= world
        e2e_how = (f"every rank: one call = scene upload + its tiles into ONE page-locked host frame in shared memory ({world} PCIe "
                   f"links): the tiles the figure touches are stored by the kernels straight into it, the background tiles leave "
                   f"a device image by DMA after the primary pass, next to the shading kernels; the step ends when rank 0 has seen "
                   f"every rank's flag; rank 0's kernels take {e2e_dev[0] / max(1, e2e_dev[1]):.3f} ms of it")
        dist.barrier()
        host.close()

    # ---- the other BASELINE configs at this N (outside the headline's timed region)
    if not args.kernel_only and not args.no_extra:
        extras["extra_workloads"] = run_extra_workloads(torch, dist, lib, bands, _abi, synth_skin, rank, world, local_rank, stream, flush, dev, exchange)

    if rank != 0:
        job.close()
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = measured_peaks()
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    fp32_peak = sm_count * 128 * peaks["sm_max_mhz"] * 1e6 / 1e12  # T lane-ops/s, non-FMA issue rate
    try:
        fp32_peak_measured = lib.fp32_issue_peak(local_rank) / 1e12  # FADD/FMUL microbenchmark on this device
    except Exception:  # noqa: BLE001
        fp32_peak_measured = None
    clocks = sampler.window(timed_window[0], timed_window[1], pad_s=0.05)
    sampler.stop()
    # The frame is one pipeline of 5 kernels per lane, two lanes in flight at once, so the roofline entry is that
    # of the whole step: the frame's algorithmic lane-ops over the event time of a frame's launches.  At N>1 each
    # rank does ~1/N of the frame.
    step_ops = ops["total"] / max(world, emulate, 1)
    achieved = step_ops / (device_ms * 1e-3) / 1e12 if device_ms > 0 else 0.0
    fb_bytes = W * H * (16 + 4)
    counters = json.loads(FRAME_COUNTERS.read_text()) if FRAME_COUNTERS.exists() else None
    sm_hz = (clocks["sm_mhz"] or peaks["sm_max_mhz"]) * 1e6
    frac_executed = None
    if counters and world == 1 and not emulate and device_ms > 0:
        # issue slots used by the frame's warp instructions (ncu smsp__inst_executed.sum over the frame's kernels)
        # / issue slots the chip has in the measured frame time (4 schedulers per SM, one instruction per clock each)
        # (a capture taken without the seed memo is set against the time of such a frame)
        counted_ms = nomemo_ms if (counters.get("captured_without_seed_memo") and nomemo_ms) else device_ms
        frac_executed = counters["warp_instructions_per_frame"] / (sm_count * 4 * sm_hz * counted_ms * 1e-3)
    partition = "whole frame"
    if world > 1:
        partition = (f"cost-balanced tile sets over {world} GPUs (mcskin_partition_tiles), stored into rank 0's frame over NVLink peer memory + flag barrier"
                     if exchange == "p2p" else f"interleaved tile rows over {world} GPUs + NCCL gather")
    elif emulate:
        partition = f"one part of a {emulate}-way tile split on one GPU (tuning aid)"
    line = {
        "metric": "Mrays/s", "value": unique_rays / (ms_per_step * 1e-3) / 1e6, "unit": "Mrays/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "width": W, "height": H, "spp": cfg.samples_per_pixel,
                   "max_bounces": cfg.max_bounces, "shadow_samples": cfg.shadow_samples, "tile_size": ts,
                   "skin": "synthetic 64x64 seed 0", "unique_rays_per_frame": unique_rays, "partition": partition,
                   "split_check": split_checked,
                   "l2": "flushed between timed iterations (256 MiB fill outside the timed events)",
                   "frame_lanes": lanes_default, "launch": "CUDA graph replay of the frame's kernels"},
        "clocks": clocks,
        "e2e": {"value": unique_rays / (e2e_ms * 1e-3) / 1e6 if e2e_ms else None, "unit": "Mrays/s", "ms_per_frame": e2e_ms,
                "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes), "how": e2e_how},
        "gpu_launches": int(launches_per_step * args.steps),
        "cold_first_frame_ms": cold_ms,
        "roofline": {
            "bound": "fp32", "kernel": f"frame pipeline ({launches_per_step} kernel launches: primary pass + wavefront shading)",
            "achieved": achieved, "peak": fp32_peak, "unit": "Tlane-op/s",
            "frac": achieved / fp32_peak,
            # DRAM bytes of one frame's kernels (dram__bytes_read.sum + dram__bytes_write.sum over the launches of a serial
            # frame, one ncu --set full capture of the committed code: profiles/r02/frame_counters.json), else null
            "traffic": counters["dram_bytes_per_frame"] if (counters and world == 1 and not emulate) else None,
            "traffic_source": str(FRAME_COUNTERS.relative_to(ROOT)) if counters else None,
            "frac_executed": frac_executed,
            "frac_executed_source": ("warp instructions of one frame (ncu smsp__inst_executed.sum, same capture) / (SMs x 4 schedulers x sampled SM clock x "
                                     + ("ms_per_step_without_seed_memo: the capture was taken without the seed memo, whose frame executes fewer instructions)"
                                        if (counters and counters.get("captured_without_seed_memo") and nomemo_ms) else "ms_per_launch)")) if frac_executed else None,
            "peak_source": f"{sm_count} SMs x 128 FP32 lanes x {peaks['sm_max_mhz']:.0f} MHz (sm_max_mhz of MEASURED_PEAKS.json"
                           + (", fallback" if peaks.get("_fallback") else "") + "); non-FMA issue rate, SURVEY.md §8d",
            "peak_measured": fp32_peak_measured,
            "frac_of_measured_peak": (achieved / fp32_peak_measured) if fp32_peak_measured else None,
            "peak_measured_source": "mcskin_cuda_fp32_issue_peak: 8 independent unfused FMUL+FADD chains per thread, best of 6 launches",
            "alg_ops_per_launch": step_ops, "ms_per_launch": device_ms,
            "serial_breakdown": {
                "what": "one stream, direct launches, same frame (outside the timed region); the algorithmic credit of the primary "
                        "pass counts the slab tests screen-rectangle culling never executes, so only the shade-pass fraction is a pipe figure",
                "ms_primary_pass": pass_ms["primary"], "ms_shade_pass": pass_ms["shade"],
                "frac_shade_pass": (ops["shade_pass"] / max(world, emulate, 1) / (pass_ms["shade"] * 1e-3) / 1e12 / fp32_peak) if pass_ms["shade"] > 0 else None},
            "hbm_framebuffer": {"bytes_per_frame": fb_bytes, "achieved_gbs": fb_bytes / (ms_per_step * 1e-3) / 1e9,
                                "peak_gbs": peaks["hbm_gbs"], "frac": fb_bytes / (ms_per_step * 1e-3) / 1e9 / peaks["hbm_gbs"]},
        },
        "active_pixels": int(n_active),
    }
    line.update(extras)
    if world == 1 and not args.no_cpu_baseline and not args.kernel_only:
        try:
            res = cpu_reference_run(WORKLOAD, 2, 1)  # the whole 16-spp frame: ~3.5 s per run on 16 cores
            line["cpu_baseline"] = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
        except Exception as exc:  # noqa: BLE001
            line["cpu_baseline"] = {"value": None, "unit": "Mrays/s", "cores": None, "kind": "unavailable", "sample": str(exc)}
    print(json.dumps(line), flush=True)
    job.close()
    if world > 1:
        dist.destroy_process_group()


def run_extra_workloads(torch, dist, lib, bands, _abi, synth_skin, rank, world, local_rank, stream, flush, dev, exchange):
    """BASELINE.json configs C2, C3, C5 (one frame split over the ranks like the headline) and C4 (a batch of skins
    sharded by skin, no exchange), device-timed, max over ranks."""
    out = {}
    for name, seed, kind, pose, over in EXTRA_FRAMES:
        cfg = _abi.default_config(**over)
        scene = lib.build_skin_scene(synth_skin(seed, kind), pose)
        job = FrameJob(torch, dist, lib, bands, scene, cfg, rank, world, local_rank, stream, 0, exchange)
        big = over["width"] * over["height"] * over["samples_per_pixel"] > 2e8
        ms, st, _, _ = time_steps(torch, dist, job, flush, 3 if big else 10, 3, world, dev)
        if job.peer is not None:
            job.peer.check_timeout()
        samples = over["width"] * over["height"] * over["samples_per_pixel"]
        out[name] = {"ms_per_frame": ms, "Msamples_per_s": samples / ms / 1e3, "n_gpus": world,
                     "width": over["width"], "height": over["height"], "spp": over["samples_per_pixel"],
                     "max_bounces": over["max_bounces"], "skin": f"synthetic {kind} seed {seed}"}
        job.close()
        if world > 1:
            dist.barrier()
    # C4: 512 skins per GPU at 256x256 / 4 spp / 2 bounces, skin i -> rank i mod N (weak scaling: 4096 skins at N=8)
    n_total = C4_SKINS_PER_GPU * world
    mine = bands.shard_batch(n_total, rank, world)
    cfg = _abi.default_config(**C4_CONFIG)
    atlases = np.stack([synth_skin(i) for i in mine])  # raw RGBA8 atlases: sliced into texel pools on the device
    ctx = lib.Context(local_rank)
    imgs = torch.empty((len(mine), cfg.height, cfg.width, 4), dtype=torch.uint8, device=dev)
    ctx.render_skin_batch(atlases[:128], cfg, None, 0, imgs.data_ptr(), stream.cuda_stream)  # warm-up at the steady-state chunk size
    ctx.sync()
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    ctx.render_skin_batch(atlases, cfg, None, 0, imgs.data_ptr(), stream.cuda_stream)
    ctx.sync()
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dt = float(tt.item())
    out["c4_batch_256_4spp_2b"] = {"skins": n_total, "skins_per_gpu": C4_SKINS_PER_GPU, "n_gpus": world, "seconds": dt,
                                   "skins_per_s": n_total / dt, "ms_per_skin_per_gpu": dt * 1e3 / C4_SKINS_PER_GPU,
                                   "what": "host RGBA8 atlases in (box layout on the host, atlas uploaded and sliced into the texel pool on the "
                                           "device inside the call), 8-bit images left on the device; wall clock around render_skin_batch + sync, "
                                           "max over ranks; sharded by skin, no exchange"}
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["own", "reference"], default="own")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_workloads leg")
    ap.add_argument("--kernel-only", action="store_true", help="tuning runs: only the timed frames and the pass breakdown")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step to DIR/frame.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_own_arm(args)


if __name__ == "__main__":
    main()

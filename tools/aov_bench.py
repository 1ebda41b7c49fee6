"""What the AOV planes (coverage, depth, tri_id; McAovTargets) cost on the GPU.

  * the headline frame (bench.py's workload: 1920x1080, 16 spp, 4 bounces, one context, render_rows_into_frame into a
    device frame) with and without all three planes, alternating in rounds: CUDA events around every frame, the
    bench's L2 flush (a 256 MiB fill outside the timed events) before each, graph replay as in the bench;
  * the C4 batch (512 skins, 256x256, 4 spp, 2 bounces, render_skin_batch, 8-bit images) with and without planes,
    wall clock around the call + sync.

Prints one JSON object (and writes it to --out): the card, its power limit, and the numbers.

    python tools/aov_bench.py --steps 50 --warmup 10 --rounds 5 --out profiles/aov/aov_bench.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as exc:  # noqa: BLE001
        return {"error": str(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from minecraftskin_raytracer_b200 import _abi, build
    build.build()
    from minecraftskin_raytracer_b200 import lib
    from minecraftskin_raytracer_b200.scene import synth_skin

    if not torch.cuda.is_available():
        raise SystemExit("aov_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    cfg = _abi.default_config(width=1920, height=1080, samples_per_pixel=16, max_bounces=4)
    scene = lib.build_skin_scene(synth_skin(0, "64x64"), None)
    H, W = cfg.height, cfg.width
    frame = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    cov = torch.zeros((H, W), dtype=torch.float32, device=dev)
    dep = torch.zeros((H, W), dtype=torch.float32, device=dev)
    tri = torch.zeros((H, W), dtype=torch.int32, device=dev)
    ctx = {False: lib.Context(0), True: lib.Context(0)}  # one context per form: each keeps its own captured graph
    for aov, c in ctx.items():
        c.set_scene(scene, cfg)
        if aov:
            c.set_aov_targets(cov.data_ptr(), dep.data_ptr(), tri.data_ptr())

    def frames(aov, n, timed):
        c = ctx[aov]
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)] if timed else []
        for i in range(n):
            flush.fill_(i & 0xff)
            if timed:
                ev[i][0].record(stream)
            c.render_rows_into_frame(0, 1, frame.data_ptr(), 0, stream.cuda_stream)
            if timed:
                ev[i][1].record(stream)
        torch.cuda.synchronize(dev)
        st = c.sync()
        return ([a.elapsed_time(b) for a, b in ev], st)

    for aov in (False, True):
        frames(aov, args.warmup, False)
    per = {False: [], True: []}
    for r in range(args.rounds):
        for aov in ((False, True) if r % 2 == 0 else (True, False)):
            ms, st = frames(aov, args.steps, True)
            per[aov].append(statistics.mean(ms))
    launches = {aov: ctx[aov].sync()["n_kernel_launches"] for aov in (False, True)}
    for c in ctx.values():
        c.close()

    # C4 batch, 512 skins
    c4cfg = _abi.default_config(width=256, height=256, samples_per_pixel=4, max_bounces=2)
    n = 512
    atlases = __import__("numpy").stack([synth_skin(i) for i in range(n)])
    imgs = torch.empty((n, 256, 256, 4), dtype=torch.uint8, device=dev)
    planes = [torch.empty((n, 256, 256), dtype=dt, device=dev) for dt in (torch.float32, torch.float32, torch.int32)]
    c4 = {}
    for aov in (False, True, False, True):
        c = lib.Context(0)
        if aov:
            c.set_aov_targets(*(p.data_ptr() for p in planes))
        c.render_skin_batch(atlases[:128], c4cfg, None, 0, imgs.data_ptr(), stream.cuda_stream)  # warm-up
        c.sync()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        c.render_skin_batch(atlases, c4cfg, None, 0, imgs.data_ptr(), stream.cuda_stream)
        c.sync()
        torch.cuda.synchronize(dev)
        c4.setdefault(aov, []).append(time.perf_counter() - t0)
        c.close()

    base, with_aov = statistics.median(per[False]), statistics.median(per[True])
    out = {
        "card": card(),
        "headline_1080p_16spp_4b": {
            "ms_per_frame_without_aov": base, "ms_per_frame_with_aov": with_aov,
            "overhead_pct": 100.0 * (with_aov - base) / base,
            "round_means_without": per[False], "round_means_with": per[True],
            "kernel_launches_per_frame": {"without": launches[False], "with": launches[True]},
            "extra_bytes_stored_per_frame": H * W * 12,
            "what": f"{args.rounds} alternating rounds of {args.steps} frames after {args.warmup} warm-up frames per form; CUDA events "
                    "around each render_rows_into_frame (graph replay), 256 MiB L2 flush before each frame outside the events; "
                    "median of the round means",
        },
        "c4_batch_512_skins_256_4spp_2b": {
            "seconds_without_aov": min(c4[False]), "seconds_with_aov": min(c4[True]),
            "skins_per_s_without_aov": n / min(c4[False]), "skins_per_s_with_aov": n / min(c4[True]),
            "what": "render_skin_batch of 512 host atlases into 8-bit device images (+ three device planes per skin), wall clock "
                    "around the call + sync, best of 2 per form (fresh context each, 128-skin warm-up)",
        },
    }
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()

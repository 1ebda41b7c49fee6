"""What the guide planes (normal, albedo; McAovTargets) cost on the GPU, next to the three planes before them.

The headline frame (bench.py's workload: 1920x1080, 16 spp, 4 bounces, one context, render_rows_into_frame into a
device frame) with no planes, with coverage + depth + tri_id, and with all five planes, alternating in rounds: CUDA
events around every frame, a 256 MiB fill before each (outside the events) so that no frame finds the last one in L2,
graph replay as in the bench.  Prints one JSON object (and writes it to --out): the card, its power limit, the numbers.

    python tools/guide_bench.py --steps 50 --warmup 10 --rounds 6 --out profiles/aov/guide_bench.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

from tools.aov_bench import card  # noqa: E402

FORMS = ("none", "three", "five")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    from minecraftskin_raytracer_b200 import _abi, build
    build.build()
    from minecraftskin_raytracer_b200 import lib
    from minecraftskin_raytracer_b200.scene import synth_skin

    if not torch.cuda.is_available():
        raise SystemExit("guide_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    cfg = _abi.default_config(width=1920, height=1080, samples_per_pixel=16, max_bounces=4)
    scene = lib.build_skin_scene(synth_skin(0, "64x64"), None)
    H, W = cfg.height, cfg.width
    frame = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    planes = {"coverage": torch.zeros((H, W), dtype=torch.float32, device=dev),
              "depth": torch.zeros((H, W), dtype=torch.float32, device=dev),
              "tri_id": torch.zeros((H, W), dtype=torch.int32, device=dev),
              "normal": torch.zeros((H, W, 3), dtype=torch.float32, device=dev),
              "albedo": torch.zeros((H, W, 4), dtype=torch.float32, device=dev)}
    ctx = {f: lib.Context(0) for f in FORMS}  # one context per form: each keeps its own captured graph
    for form, c in ctx.items():
        c.set_scene(scene, cfg)
        names = {"none": (), "three": ("coverage", "depth", "tri_id"), "five": tuple(planes)}[form]
        if names:
            c.set_aov_targets(**{p: planes[p].data_ptr() for p in names})

    def frames(form, n, timed):
        c = ctx[form]
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)] if timed else []
        for i in range(n):
            flush.fill_(i & 0xff)
            if timed:
                ev[i][0].record(stream)
            c.render_rows_into_frame(0, 1, frame.data_ptr(), 0, stream.cuda_stream)
            if timed:
                ev[i][1].record(stream)
        torch.cuda.synchronize(dev)
        c.sync()
        return [a.elapsed_time(b) for a, b in ev]

    for form in FORMS:
        frames(form, args.warmup, False)
    per = {f: [] for f in FORMS}
    for r in range(args.rounds):
        order = FORMS[r % 3:] + FORMS[:r % 3]  # every form leads a round in turn
        for form in order:
            per[form].append(statistics.mean(frames(form, args.steps, True)))
    launches = {f: ctx[f].sync()["n_kernel_launches"] for f in FORMS}
    for c in ctx.values():
        c.close()

    med = {f: statistics.median(per[f]) for f in FORMS}
    out = {
        "card": card(),
        "headline_1080p_16spp_4b": {
            "ms_per_frame": med,
            "overhead_pct_vs_none": {f: 100.0 * (med[f] - med["none"]) / med["none"] for f in ("three", "five")},
            "overhead_pct_five_vs_three": 100.0 * (med["five"] - med["three"]) / med["three"],
            "round_means": per,
            "kernel_launches_per_frame": launches,
            "plane_bytes_stored_per_frame": {"three": H * W * 12, "five": H * W * 40},
            "what": f"{args.rounds} rounds of {args.steps} frames per form, the forms in rotating order, after {args.warmup} "
                    "warm-up frames each; CUDA events around each render_rows_into_frame (graph replay), 256 MiB L2 flush "
                    "before each frame outside the events; median of the round means",
        },
    }
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()

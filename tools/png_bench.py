"""What PNG files made on the device cost (mcskin_cuda_context_encode_png), next to what they save.

  * the C4 batch (512 skins, 256x256, 4 spp, 2 bounces, render_skin_batch into 8-bit device images): the render alone,
    and the render followed by encode_png, in alternating rounds;
  * encode_png alone on the C4 batch and on the headline 1080p frame (1920x1080, 16 spp, 4 bounces);
  * bytes per image, and the device-to-host copy of the raw 8-bit images against that of the files, into pinned memory;
  * host zlib at levels 1 and 6 on the same filtered rows, per image, on one core of this machine.

Device times are CUDA events around each call with the L2 flushed (a 256 MiB fill outside the events) before it;
medians over the rounds.  Prints one JSON object (and writes it to --out) with the card and its power limit.

    python tools/png_bench.py --rounds 10 --out profiles/png/png_bench.json
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
import zlib
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
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--skins", type=int, default=512)
    ap.add_argument("--zlib-images", type=int, default=16)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import numpy as np
    import torch
    from minecraftskin_raytracer_b200 import _abi, build
    build.build()
    from minecraftskin_raytracer_b200 import lib
    from minecraftskin_raytracer_b200.scene import synth_skin
    from tests import png_oracle as po

    if not torch.cuda.is_available():
        raise SystemExit("png_bench.py: no CUDA device")
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(stream)
    s = stream.cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def timed(fn, rounds):
        ms = []
        for r in range(rounds):
            flush.fill_(r & 0xff)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            torch.cuda.synchronize(dev)
            ms.append(a.elapsed_time(b))
        return ms

    # C4 batch
    n = args.skins
    c4 = _abi.default_config(width=256, height=256, samples_per_pixel=4, max_bounces=2)
    atlases = np.stack([synth_skin(i) for i in range(n)])
    imgs = torch.empty((n, 256, 256, 4), dtype=torch.uint8, device=dev)
    bound = lib.png_bound(256, 256)
    files = torch.empty(n * bound, dtype=torch.uint8, device=dev)
    offsets = torch.empty(n + 1, dtype=torch.int64, device=dev)
    ctx = lib.Context(0)

    def render():
        ctx.render_skin_batch(atlases, c4, None, 0, imgs.data_ptr(), s)

    def encode():
        ctx.encode_png(imgs.data_ptr(), 256, 256, n, files.data_ptr(), files.numel(), offsets.data_ptr(), s)

    def both():
        render()
        encode()

    for f in (render, encode, both):
        timed(f, 2)  # warm-up: module loads, scratch growth
    per = {"render": [], "render_encode": [], "encode": []}
    for r in range(args.rounds):
        forms = [("render", render), ("render_encode", both), ("encode", encode)]
        for name, f in (forms if r % 2 == 0 else forms[::-1]):
            per[name] += timed(f, 1)
    offs = offsets.cpu().tolist()
    c4_bytes = offs[n]
    host_files = torch.empty(c4_bytes, dtype=torch.uint8, pin_memory=True)
    host_raw = torch.empty(imgs.numel(), dtype=torch.uint8, pin_memory=True)
    d2h_raw = timed(lambda: host_raw.copy_(imgs.view(-1), non_blocking=True), args.rounds)
    d2h_png = timed(lambda: host_files.copy_(files[:c4_bytes], non_blocking=True), args.rounds)

    # host zlib on the same filtered rows (one core of this machine)
    images = imgs[:args.zlib_images].cpu().numpy()
    streams = [po.filter_image(im)[0] for im in images]
    zl = {}
    for level in (1, 6):
        t0 = time.perf_counter()
        sizes = [len(zlib.compress(st, level)) for st in streams]
        zl[level] = {"ms_per_image": 1e3 * (time.perf_counter() - t0) / len(streams),
                     "bytes_per_image": statistics.mean(sizes)}
    ours_first = statistics.mean(offs[i + 1] - offs[i] for i in range(args.zlib_images))

    # headline frame, encode alone
    hcfg = _abi.default_config(width=1920, height=1080, samples_per_pixel=16, max_bounces=4)
    scene = lib.build_skin_scene(synth_skin(0, "64x64"), None)
    _, u8, _ = lib.render(scene, hcfg, device=0, want_f32=False, want_u8=True)
    frame = torch.from_numpy(u8).to(dev)
    fbound = lib.png_bound(1920, 1080)
    ffile = torch.empty(fbound, dtype=torch.uint8, device=dev)
    foffs = torch.empty(2, dtype=torch.int64, device=dev)

    def encode_frame():
        ctx.encode_png(frame.data_ptr(), 1920, 1080, 1, ffile.data_ptr(), fbound, foffs.data_ptr(), s)

    timed(encode_frame, 2)
    frame_ms = timed(encode_frame, args.rounds)
    frame_bytes = foffs.cpu().tolist()[1]
    ctx.close()

    med = {k: statistics.median(v) for k, v in per.items()}
    out = {
        "card": card(),
        "c4_batch_512_skins_256_4spp_2b": {
            "ms_render": med["render"], "ms_render_and_encode": med["render_encode"], "ms_encode": med["encode"],
            "round_ms": per,
            "skins_per_s_render": n / med["render"] * 1e3, "skins_per_s_render_and_encode": n / med["render_encode"] * 1e3,
            "png_bytes_per_image": c4_bytes / n, "raw_bytes_per_image": 256 * 256 * 4,
            "ratio_to_raw": c4_bytes / imgs.numel(),
            "ms_d2h_raw_u8": statistics.median(d2h_raw), "ms_d2h_png": statistics.median(d2h_png),
            "what": f"{args.rounds} alternating rounds; CUDA events around each call on one stream, 256 MiB L2 flush before "
                    "each outside the events; render_skin_batch from host atlases (its host staging included); D2H into "
                    "pinned host memory; medians",
        },
        "host_zlib_first_images": {
            "images": args.zlib_images, "png_bytes_per_image_device": ours_first,
            "level1": zl[1], "level6": zl[6],
            "what": "zlib.compress of the filtered stream (filter bytes included) per image, one core of the benchmark host",
        },
        "headline_1080p_encode": {"ms_encode": statistics.median(frame_ms), "round_ms": frame_ms, "png_bytes": frame_bytes,
                                  "ratio_to_raw": frame_bytes / (1920 * 1080 * 4)},
    }
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()

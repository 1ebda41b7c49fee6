"""PNG files made on the device (mcskin_cuda_context_encode_png): every file decodes to its image with PIL and with
zlib + the numpy unfilter, takes the oracle's filter on every row, carries correct CRCs, fits png_bound, and has the
same bytes on a second run, alone, and at any place in a batch."""
from __future__ import annotations

import io
import struct
import zlib

import numpy as np
import pytest

from tests import png_oracle as po

pytestmark = pytest.mark.gpu


def _encode(lib, ctx, images: np.ndarray) -> list[bytes]:
    import torch
    n, h, w = images.shape[:3]
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(dev)  # (a stream of its own: handle 0 would mean the context's stream)
    with torch.cuda.stream(stream):
        d_img = torch.from_numpy(np.ascontiguousarray(images)).to(dev)
        cap = max(1, n * lib.png_bound(w, h))
        files = torch.full((cap,), 0xA5, dtype=torch.uint8, device=dev)
        offsets = torch.full((n + 1,), -1, dtype=torch.int64, device=dev)
        ctx.encode_png(d_img.data_ptr(), w, h, n, files.data_ptr(), cap, offsets.data_ptr(), stream.cuda_stream)
        offs = offsets.cpu().tolist()
        data = files[:offs[n]].cpu().numpy().tobytes()
    assert offs[0] == 0 and all(a < b for a, b in zip(offs, offs[1:]))
    return [data[offs[i]:offs[i + 1]] for i in range(n)]


def _check_file(lib, data: bytes, img: np.ndarray):
    from PIL import Image
    h, w = img.shape[:2]
    assert len(data) <= lib.png_bound(w, h)
    chunks = po.chunks(data)
    kinds = [c[0] for c in chunks]
    assert kinds[0] == b"IHDR" and kinds[-1] == b"IEND" and set(kinds[1:-1]) == {b"IDAT"}
    for kind, payload, crc in chunks:
        assert zlib.crc32(kind + payload) == crc, kind
    assert chunks[0][1] == struct.pack(">IIBBBBB", w, h, 8, 6, 0, 0, 0)
    # one IDAT per 32 KiB segment; each segment inflates on its own (no match reaches before it) and ends with the
    # empty stored block
    stream_len = h * (4 * w + 1)
    idats = [c[1] for c in chunks[1:-1]]
    assert len(idats) == -(-stream_len // po.SEGMENT_BYTES)
    zs = b"".join(idats)
    assert zs[:2] == b"\x78\x01"
    for k, payload in enumerate(idats):
        seg = payload[2 if k == 0 else 0:len(payload) - (4 if k == len(idats) - 1 else 0)]
        assert seg[-4:] == b"\x00\x00\xff\xff"
        d = zlib.decompressobj(-15)
        part = d.decompress(seg)
        assert len(part) == min(po.SEGMENT_BYTES, stream_len - k * po.SEGMENT_BYTES)
        assert d.eof == (k == len(idats) - 1)
    stream = zlib.decompress(zs)
    assert len(stream) == stream_len
    back, types = po.unfilter(stream, w, h)
    assert np.array_equal(back, img)
    want_stream, want_types = po.filter_image(img)
    assert types == want_types
    assert stream == want_stream
    assert np.array_equal(np.asarray(Image.open(io.BytesIO(data)).convert("RGBA")), img)
    return stream


def _skins(lib, n, cfg=None):
    import torch
    from minecraftskin_raytracer_b200 import _abi
    from minecraftskin_raytracer_b200.scene import synth_skin
    cfg = cfg or _abi.default_config(width=256, height=256, samples_per_pixel=4, max_bounces=2)
    atlases = np.stack([synth_skin(i) for i in range(n)])
    out = torch.empty((n, cfg.height, cfg.width, 4), dtype=torch.uint8, device="cuda:0")
    ctx = lib.Context(0)
    ctx.render_skin_batch(atlases, cfg, None, 0, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ctx.close()
    return atlases, cfg, out.cpu().numpy()


def test_c4_skins_decode_and_meet_the_compression_bar(gpu):
    _, cfg, images = _skins(gpu, 16)
    ctx = gpu.Context(0)
    files = _encode(gpu, ctx, images)
    ours = ref = raw = 0
    for data, img in zip(files, images):
        stream = _check_file(gpu, data, img)
        ours += len(data)
        ref += len(po.reference_png(img, 1))
        raw += img.nbytes
        assert len(zlib.compress(stream, 1)) <= len(po.reference_png(img, 1))
    print(f"C4 skins: {ours} B, zlib-1 {ref} B ({ours / ref:.3f}x), raw {raw} B ({ours / raw:.3f})")
    assert ours <= 1.25 * ref
    assert ours <= 0.35 * raw
    # the same bytes on a second run, alone, and at other places in other batches
    assert _encode(gpu, ctx, images) == files
    for i in (0, 5, 15):
        assert _encode(gpu, ctx, images[i:i + 1]) == [files[i]]
    order = [3, 15, 0, 7]
    assert _encode(gpu, ctx, images[order]) == [files[i] for i in order]
    assert _encode(gpu, ctx, images[::-1]) == files[::-1]
    ctx.close()


def test_render_skin_batch_png(gpu):
    atlases, cfg, images = _skins(gpu, 5)
    ctx = gpu.Context(0)
    files = ctx.render_skin_batch_png(atlases, cfg)
    ctx.close()
    assert len(files) == 5
    for data, img in zip(files, images):
        _check_file(gpu, data, img)
    assert files == _encode(gpu, gpu.Context(0), images)


def _render(lib, w, h, spp):
    from minecraftskin_raytracer_b200 import _abi
    from minecraftskin_raytracer_b200.scene import synth_skin
    scene = lib.build_skin_scene(synth_skin(0, "64x64"), None)
    cfg = _abi.default_config(width=w, height=h, samples_per_pixel=spp, max_bounces=4 if spp == 16 else 2)
    _, u8, _ = lib.render(scene, cfg, device=0, want_f32=False, want_u8=True)
    return u8


@pytest.mark.parametrize("w,h,spp", [(1920, 1080, 16), (7680, 4320, 1)])
def test_rendered_frames(gpu, w, h, spp):
    img = _render(gpu, w, h, spp)
    ctx = gpu.Context(0)
    files = _encode(gpu, ctx, img[None])
    _check_file(gpu, files[0], img)
    assert _encode(gpu, ctx, img[None]) == files
    ctx.close()


def _idat_segments(data):
    idats = [c[1] for c in po.chunks(data)[1:-1]]
    return [p[2 if k == 0 else 0:] for k, p in enumerate(idats)]


def test_constant_and_noise_images(gpu):
    rng = np.random.default_rng(11)
    const = np.full((300, 500, 4), (12, 200, 77, 255), np.uint8)
    noise = rng.integers(0, 256, (300, 500, 4), dtype=np.uint8)
    ctx = gpu.Context(0)
    files = _encode(gpu, ctx, np.stack([const, noise, const]))
    for data, img in zip(files, (const, noise, const)):
        _check_file(gpu, data, img)
    assert files[0] == files[2]
    assert len(files[0]) < 0.02 * const.nbytes  # (at least one token per thread's 128 bytes: about 1/80 of raw)
    # noise: every segment is stored (BTYPE 00), and the file is the bound
    assert all(seg[0] & 0x7 == 0 for seg in _idat_segments(files[1]))
    assert len(files[1]) == gpu.png_bound(500, 300)
    ctx.close()


@pytest.mark.parametrize("w,h", [(1, 1), (1, 2), (2, 1), (1, 777), (777, 1), (1, 9000), (65535, 1), (1, 65535), (3, 5)])
def test_small_and_thin_images(gpu, w, h):
    rng = np.random.default_rng(w * 7 + h)
    imgs = rng.integers(0, 256, (3, h, w, 4), dtype=np.uint8)
    imgs[1] //= 64
    imgs[2] = imgs[2, :1, :1]
    ctx = gpu.Context(0)
    files = _encode(gpu, ctx, imgs)
    for data, img in zip(files, imgs):
        _check_file(gpu, data, img)
    assert _encode(gpu, ctx, imgs[1:2]) == files[1:2]
    ctx.close()


@pytest.mark.parametrize("w", [1, 3])
def test_stream_an_exact_multiple_of_the_segment(gpu, w):
    h = 32768  # h * (4w + 1) bytes: exactly 4w + 1 segments
    yy, xx = np.mgrid[0:h, 0:w]
    img = np.stack([(yy % 251), (yy // 7 % 256), (xx * 50 + yy % 3), np.full_like(yy, 255)], -1).astype(np.uint8)
    ctx = gpu.Context(0)
    files = _encode(gpu, ctx, np.stack([img, img[::-1].copy()]))
    for data, im in zip(files, (img, img[::-1])):
        _check_file(gpu, data, im)
        assert len(_idat_segments(data)) == 4 * w + 1
    ctx.close()


def test_bad_arguments(gpu):
    import torch
    ctx = gpu.Context(0)
    img = torch.zeros((2, 8, 8, 4), dtype=torch.uint8, device="cuda:0")
    offsets = torch.full((3,), -1, dtype=torch.int64, device="cuda:0")
    bound = gpu.png_bound(8, 8)
    files = torch.empty(2 * bound, dtype=torch.uint8, device="cuda:0")
    with pytest.raises(gpu.McSkinError) as e:
        ctx.encode_png(img.data_ptr(), 8, 8, 2, files.data_ptr(), 2 * bound - 1, offsets.data_ptr())
    assert e.value.code == -1
    for args in [(0, 8, 8, 2, files.data_ptr(), 2 * bound, offsets.data_ptr()),
                 (img.data_ptr(), 0, 8, 2, files.data_ptr(), 2 * bound, offsets.data_ptr()),
                 (img.data_ptr(), 8, 65536, 2, files.data_ptr(), 2 * bound, offsets.data_ptr()),
                 (img.data_ptr(), 8, 8, -1, files.data_ptr(), 2 * bound, offsets.data_ptr()),
                 (img.data_ptr(), 8, 8, 2, 0, 2 * bound, offsets.data_ptr()),
                 (img.data_ptr(), 8, 8, 2, files.data_ptr(), 2 * bound, 0)]:
        with pytest.raises(gpu.McSkinError) as e:
            ctx.encode_png(*args)
        assert e.value.code == -1
    torch.cuda.synchronize()
    assert offsets.cpu().tolist() == [-1, -1, -1]  # nothing was written
    ctx.encode_png(img.data_ptr(), 8, 8, 0, files.data_ptr(), 0, offsets.data_ptr())
    torch.cuda.synchronize()
    assert offsets.cpu().tolist()[0] == 0
    ctx.close()

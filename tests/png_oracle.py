"""numpy restatement of the PNG rules in include/mcskin_cuda.h: libpng's filter choice, unfiltering, a chunk parser,
and a reference encoder (the same filters, then zlib) for the size comparisons."""
from __future__ import annotations

import struct
import zlib

import numpy as np

SIGNATURE = b"\x89PNG\r\n\x1a\n"
SEGMENT_BYTES = 32768


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(row: np.ndarray, up: np.ndarray | None) -> np.ndarray:
    """The five filtered forms (0 None .. 4 Paeth) of one RGBA8 row ([4w] uint8, previous row or None): [5, 4w] uint8."""
    x = row.astype(np.int32)
    b = up.astype(np.int32) if up is not None else np.zeros_like(x)
    a = np.concatenate([np.zeros(4, np.int32), x[:-4]])
    c = np.concatenate([np.zeros(4, np.int32), b[:-4]])
    preds = [np.zeros_like(x), a, b, (a + b) >> 1, _paeth(a, b, c)]
    return np.stack([(x - p) & 0xFF for p in preds]).astype(np.uint8)


def choose_filter(forms: np.ndarray) -> int:
    """libpng's heuristic: the smallest sum of |filtered byte| read as int8; the lower type on a tie."""
    sums = np.abs(forms.view(np.int8).astype(np.int64)).sum(axis=1)
    return int(np.argmin(sums))  # argmin returns the first of equal minima


def filter_image(img: np.ndarray) -> tuple[bytes, list[int]]:
    """The filtered stream of an [h, w, 4] uint8 image and every row's filter type."""
    h, w = img.shape[:2]
    rows = img.reshape(h, 4 * w)
    out, types = bytearray(), []
    for y in range(h):
        forms = filter_rows(rows[y], rows[y - 1] if y else None)
        t = choose_filter(forms)
        types.append(t)
        out.append(t)
        out += forms[t].tobytes()
    return bytes(out), types


def unfilter(stream: bytes, w: int, h: int) -> tuple[np.ndarray, list[int]]:
    """The [h, w, 4] uint8 image of a filtered stream, and the filter types it names."""
    n = 4 * w + 1
    assert len(stream) == h * n, (len(stream), h * n)
    raw = np.frombuffer(stream, np.uint8).reshape(h, n)
    types = raw[:, 0].astype(np.int32)
    if types.max(initial=0) > 4:
        raise ValueError(f"row {int(np.argmax(types > 4))}: filter type {int(types.max())}")
    f = raw[:, 1:].reshape(h, w, 4).astype(np.int32)
    # pixel (y, x) needs (y, x-1), (y-1, x) and (y-1, x-1): one anti-diagonal at a time; out has a zero border
    out = np.zeros((h + 1, w + 1, 4), np.int32)
    for d in range(h + w - 1):
        y = np.arange(max(0, d - w + 1), min(h, d + 1))
        x = d - y
        a, b, c = out[y + 1, x], out[y, x + 1], out[y, x]
        t = types[y][:, None]
        pred = np.select([t == 1, t == 2, t == 3, t == 4], [a, b, (a + b) >> 1, _paeth(a, b, c)], 0)
        out[y + 1, x + 1] = (f[y, x] + pred) & 0xFF
    return out[1:, 1:].astype(np.uint8), [int(v) for v in types]


def chunks(data: bytes) -> list[tuple[bytes, bytes, int]]:
    """(type, payload, stored CRC) of every chunk of a PNG file; the signature and the framing are checked."""
    assert data[:8] == SIGNATURE
    out, at = [], 8
    while at < len(data):
        (n,) = struct.unpack(">I", data[at:at + 4])
        kind = data[at + 4:at + 8]
        payload = data[at + 8:at + 8 + n]
        (crc,) = struct.unpack(">I", data[at + 8 + n:at + 12 + n])
        out.append((kind, payload, crc))
        at += 12 + n
    assert at == len(data), "trailing bytes after the last chunk"
    return out


def reference_png(img: np.ndarray, level: int = 1) -> bytes:
    """A PNG of the same filtered stream, deflated by zlib at `level` (one IDAT)."""
    h, w = img.shape[:2]
    stream, _ = filter_image(img)

    def chunk(kind: bytes, payload: bytes) -> bytes:
        return struct.pack(">I", len(payload)) + kind + payload + struct.pack(">I", zlib.crc32(kind + payload))

    ihdr = struct.pack(">IIBBBBB", w, h, 8, 6, 0, 0, 0)
    return SIGNATURE + chunk(b"IHDR", ihdr) + chunk(b"IDAT", zlib.compress(stream, level)) + chunk(b"IEND", b"")


def png_bound(w: int, h: int) -> int:
    """mcskin_png_bound restated: every segment one stored block plus the empty stored block, in its own IDAT."""
    if not (1 <= w <= 65535 and 1 <= h <= 65535):
        return 0
    n = h * (4 * w + 1)
    segments = -(-n // SEGMENT_BYTES)
    return 8 + 25 + 2 + 4 + 12 + n + 22 * segments

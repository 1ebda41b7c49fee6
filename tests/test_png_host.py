"""PNG encoding, host side: mcskin_png_bound, the oracle's filter choice on rows built to tie, and the declarations."""
from __future__ import annotations

import io
import re
from pathlib import Path

import numpy as np
import pytest

from tests import png_oracle as po

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("w,h", [(1, 1), (1, 2), (2, 1), (3, 5), (5, 3), (7, 7), (13, 1), (1, 65535), (65535, 1), (256, 256),
                                 (1920, 1080), (1921, 1081), (7680, 4320), (1, 32768), (3, 32768), (65535, 65535)])
def test_png_bound_is_the_all_stored_file(mclib, w, h):
    n = h * (4 * w + 1)
    segments = -(-n // po.SEGMENT_BYTES)
    # signature, IHDR, zlib header and Adler-32, IEND; per segment an IDAT chunk, a stored block and the empty one
    assert mclib.png_bound(w, h) == 8 + 25 + 2 + 4 + 12 + n + segments * (12 + 5 + 5) == po.png_bound(w, h)


@pytest.mark.parametrize("w,h", [(0, 1), (1, 0), (-1, 5), (5, -1), (65536, 1), (1, 65536), (0, 0)])
def test_png_bound_refuses_bad_sizes(mclib, w, h):
    assert mclib.png_bound(w, h) == 0


def test_png_bound_covers_zlib_on_incompressible_rows(mclib):
    rng = np.random.default_rng(3)
    for w, h in [(1, 1), (3, 7), (64, 64)]:
        img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        assert len(po.reference_png(img, 9)) <= mclib.png_bound(w, h)


def _row(values):
    return np.asarray(values, dtype=np.uint8)


def test_filter_choice_takes_the_lower_type_on_a_tie():
    # a zero row with no row above: every filter gives zeros
    assert po.choose_filter(po.filter_rows(_row([0] * 8), None)) == 0
    # constant row, no row above: None sums 8*10, Sub 4*10, Up = None, Avg 4*10 + 4*5, Paeth = Sub (a is the predictor)
    forms = po.filter_rows(_row([10] * 8), None)
    sums = np.abs(forms.view(np.int8).astype(int)).sum(axis=1).tolist()
    assert sums == [80, 40, 80, 60, 40]
    assert po.choose_filter(forms) == 1
    # equal to the row above: Up and Paeth (b predicts) give zeros; Avg does not; Up wins the tie
    up = _row([7, 9, 11, 13, 7, 9, 11, 13])
    forms = po.filter_rows(up, up)
    sums = np.abs(forms.view(np.int8).astype(int)).sum(axis=1).tolist()
    assert sums[2] == sums[4] == 0 and po.choose_filter(forms) == 2


def test_filter_choice_reads_bytes_as_signed():
    # two pixels of 200 under two of 100.  Read as int8, 200 is -56: None 8*56, Sub 4*56 (200, then 0), Up 8*100,
    # Avg 4*106 + 4*50, Paeth 4*100 (b, then a) -> Sub.  Read unsigned, Paeth's 400 would beat Sub's 800.
    forms = po.filter_rows(_row([200] * 8), _row([100] * 8))
    assert np.abs(forms.view(np.int8).astype(int)).sum(axis=1).tolist() == [448, 224, 800, 624, 400]
    assert forms.astype(int).sum(axis=1).tolist() == [1600, 800, 800, 800, 400]
    assert po.choose_filter(forms) == 1
    # 255 is -1: None and Up (no row above) both cost 12, Sub and Paeth 14 -> None, the lower of the tie
    forms = po.filter_rows(_row([255, 0, 255, 0, 1, 2, 3, 4]), None)
    sums = np.abs(forms.view(np.int8).astype(int)).sum(axis=1).tolist()
    assert sums[0] == sums[2] == 12 and sums[1] == sums[4] == 14
    assert po.choose_filter(forms) == 0


def test_oracle_round_trips_through_pil():
    from PIL import Image
    rng = np.random.default_rng(5)
    for h, w in [(1, 1), (1, 9), (9, 1), (23, 17)]:
        img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
        img[h // 2:] //= 32  # some rows worth filtering
        data = po.reference_png(img)
        assert [c[0] for c in po.chunks(data)] == [b"IHDR", b"IDAT", b"IEND"]
        assert np.array_equal(np.asarray(Image.open(io.BytesIO(data)).convert("RGBA")), img)
        stream, types = po.filter_image(img)
        back, got = po.unfilter(stream, w, h)
        assert np.array_equal(back, img) and got == types


def test_header_declares_the_png_entry_points(mclib):
    header = (ROOT / "include" / "mcskin_cuda.h").read_text()
    assert re.search(r"uint64_t mcskin_png_bound\(int32_t width, int32_t height\);", header)
    assert re.search(r"int32_t mcskin_cuda_context_encode_png\(McContext\* ctx, const void\* d_rgba8, int32_t width, int32_t height, "
                     r"int32_t n_images,\s+void\* d_png, uint64_t capacity, uint64_t\* d_offsets, void\* stream\);", header)
    assert "#define MCSKIN_ABI_VERSION 4" in header
    for name in ("mcskin_png_bound", "mcskin_cuda_context_encode_png"):
        assert name in mclib.EXPORTS and hasattr(mclib.raw(), name)

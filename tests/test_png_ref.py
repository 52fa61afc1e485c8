"""The CPU restatement of the device PNG encoder (tests/png_ref.py): its streams decode with zlib and PIL to the
input pixels, its combined checksums equal zlib's, its Huffman codes are complete and within the length limits, and
every rule (filters, runs, blocks, stored fallback) is exercised."""
import io
import struct
import zlib

import numpy as np
import pytest
from PIL import Image

from tests import png_ref


def particle_crop(rng, h, w, sigma=3.0):
    """Seeded particle-like RGB crop: smooth background, a dark elliptical blob, Gaussian noise of `sigma`."""
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    bg = 180 + 30 * np.sin(xx / max(w, 1) * 3 + rng.uniform(0, 6)) * np.cos(yy / max(h, 1) * 2)
    cy, cx = h * rng.uniform(0.3, 0.7), w * rng.uniform(0.3, 0.7)
    blob = ((yy - cy) / max(h * 0.3, 1)) ** 2 + ((xx - cx) / max(w * 0.3, 1)) ** 2 < 1
    img = np.stack([bg, bg * 0.95, bg * 0.9], axis=2)
    img[blob] *= np.array([0.35, 0.3, 0.25], np.float32)
    img += rng.normal(0, sigma, img.shape)
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


def _ramp(h, w, kind):
    y, x = np.mgrid[0:h, 0:w]
    if kind == 1:          # sub: constant step along x
        return ((x * 7) % 256).astype(np.uint8)
    if kind == 2:          # up: rows repeat a noisy row
        row = np.random.default_rng(0).integers(0, 256, w, dtype=np.uint8)
        return np.tile(row, (h, 1))
    if kind == 3:          # average
        return ((x * 3 + y * 5) // 2 % 256).astype(np.uint8)
    if kind == 4:          # paeth: a plane with a noisy column offset per row and column
        rng = np.random.default_rng(1)
        return ((rng.integers(0, 256, h)[:, None] + rng.integers(0, 256, w)[None, :]) % 256).astype(np.uint8)
    return np.random.default_rng(2).integers(0, 4, (h, w)).astype(np.uint8) * 60


def hand_cases():
    """(name, uint8 crop) of the encoder's edge cases; shared with the device test."""
    rng = np.random.default_rng(0)
    B = png_ref.BLOCK
    cases = [("1x1", np.array([[7]], np.uint8)),
             ("1xN", rng.integers(0, 256, (1, 37, 3), dtype=np.uint8)),
             ("Nx1", rng.integers(0, 256, (41, 1, 2), dtype=np.uint8)),
             ("single colour", np.full((120, 333, 4), 9, np.uint8)),
             ("uniform random", rng.integers(0, 256, (90, 110, 3), dtype=np.uint8)),
             ("mask", (((np.mgrid[0:80, 0:60][0] - 40) / 30) ** 2 + ((np.mgrid[0:80, 0:60][1] - 30) / 20) ** 2 < 1)
              .astype(np.uint8) * 255)]
    for k in range(5):
        cases.append((f"ramp {k}", _ramp(40, 64, k)))
    # filtered sizes B - 1, B, B + 1 and several blocks: h * (1 + w) with one channel
    for name, (h, w) in (("B-1", (1, B - 2)), ("B", (1, B - 1)), ("B+1", (3, 10922)), ("4 blocks", (257, 511))):
        cases.append((name, particle_crop(rng, h, w, 3)[..., 1].copy()))
    cases.append(("photo", particle_crop(rng, 150, 170, 3)))
    return cases


@pytest.mark.parametrize("name,a", hand_cases(), ids=[n for n, _ in hand_cases()])
def test_stream_decodes_and_checksums(name, a):
    info = {}
    s = png_ref.encode(a, info)
    assert s[:8] == png_ref.SIGNATURE
    n = struct.unpack(">I", s[33:37])[0]
    assert s[37:41] == b"IDAT"
    idat = s[41:41 + n]
    raw = zlib.decompress(idat)
    assert raw == info["filtered"]
    assert info["adler"] == zlib.adler32(raw)
    assert info["crc"] == zlib.crc32(b"IDAT" + idat) == struct.unpack(">I", s[41 + n:45 + n])[0]
    assert np.array_equal(np.array(Image.open(io.BytesIO(s))), a)
    assert len(s) <= png_ref.png_bound(a.shape[0], a.shape[1], 1 if a.ndim == 2 else a.shape[2])
    for blk in info["blocks"]:
        for lens, limit in ((blk["ll"], 15), (blk["bl"], 7)):
            assert max(lens) <= limit
            assert sum(2.0 ** -l for l in lens if l) == 1.0          # Kraft equality: every code is complete


def test_block_sizes_and_kinds():
    B = png_ref.BLOCK
    cases = dict(hand_cases())
    for name, blocks in (("B-1", 1), ("B", 1), ("B+1", 2), ("4 blocks", 5)):
        info = {}
        png_ref.encode(cases[name], info)
        assert len(info["blocks"]) == blocks, name
    assert len(png_ref.filtered_stream(cases["B-1"])) == B - 1
    assert len(png_ref.filtered_stream(cases["B"])) == B
    assert len(png_ref.filtered_stream(cases["B+1"])) == B + 1
    info = {}
    png_ref.encode(cases["uniform random"], info)
    assert {b["kind"] for b in info["blocks"]} == {"stored"}
    info = {}
    png_ref.encode(cases["single colour"], info)
    assert {b["kind"] for b in info["blocks"]} == {"dynamic"}


def test_each_filter_wins():
    seen = set()
    for k in range(5):
        a = _ramp(40, 64, k)
        ftype, _ = png_ref.filter_rows(a, 1)
        seen |= set(ftype[1:].tolist())
    assert seen == {0, 1, 2, 3, 4}


def test_run_tokens():
    d = np.array([5] * 600 + [6, 6, 6] + [7], np.uint8)
    is_match, value = png_ref.block_tokens(d)
    # 5: literal, 599 repeats = 258 + 258 + 83; 6: literal + 2 literals; 7: literal
    assert list(zip(is_match.tolist(), value.tolist())) == [(False, 5), (True, 258), (True, 258), (True, 83),
                                                           (False, 6), (False, 6), (False, 6), (False, 7)]


def test_checksum_combine():
    rng = np.random.default_rng(4)
    a, b = rng.integers(0, 256, 1000, dtype=np.uint8).tobytes(), rng.integers(0, 256, 777, dtype=np.uint8).tobytes()
    assert png_ref.crc32_combine(zlib.crc32(a), zlib.crc32(b), len(b)) == zlib.crc32(a + b)
    pa = (len(a),) + png_ref.adler_partial(np.frombuffer(a, np.uint8))
    pb = (len(b),) + png_ref.adler_partial(np.frombuffer(b, np.uint8))
    assert png_ref.adler_combine([pa, pb]) == zlib.adler32(a + b)


def test_zero_area_and_channels():
    assert png_ref.encode(np.zeros((0, 5, 3), np.uint8)) == b""
    with pytest.raises(ValueError):
        png_ref.encode(np.zeros((2, 2, 5), np.uint8))

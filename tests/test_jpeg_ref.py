"""tests/jpeg_ref.py (the CPU restatement of mb_jpeg_encode) against PIL's own JPEG writer: the whole file, byte for byte,
on a seeded sweep of sizes (every h, w remainder mod 16) and contents; and mb_jpeg_bound_bytes' formula against the
worst cases."""
import io

import numpy as np
import pytest
from PIL import Image

from tests import jpeg_ref


def pil_jpeg(a):
    b = io.BytesIO()
    Image.fromarray(a).save(b, format="JPEG")
    return b.getvalue()


def content(rng, kind, h, w, channels):
    """noise (long codes, many 0xFF bytes), flat (EOB only), a smooth ramp, and 0 / 255 at the edges."""
    shape = (h, w) if channels == 1 else (h, w, 3)
    if kind == "noise":
        return rng.integers(0, 256, shape, dtype=np.uint8)
    if kind == "flat":
        return np.full(shape, int(rng.integers(0, 256)), np.uint8)
    if kind == "ramp":
        r = np.add.outer(np.arange(h) * 5, np.arange(w) * 3)
        r = r if channels == 1 else np.stack([r, r[::-1, ::-1] if r.size else r, r * 2], -1)
        return (r % 256).astype(np.uint8)
    a = np.full(shape, 128, np.uint8)                   # edges: 0 / 255 columns and rows at the borders
    a[0], a[-1], a[:, 0], a[:, -1] = 0, 255, 255, 0
    return a


KINDS = ("noise", "flat", "ramp", "edges")


def sweep_cases(channels, seed=0):
    """Every (h mod 16, w mod 16) with each kind, 1 x N and N x 1 strips, and a few larger sizes."""
    rng = np.random.default_rng(seed + channels)
    sizes = [(h, w) for h in range(1, 17) for w in range(1, 17)]
    sizes += [(1, n) for n in (17, 31, 33, 64, 65, 100)] + [(n, 1) for n in (17, 31, 33, 64, 65, 100)]
    sizes += [(37, 53), (64, 64), (80, 23), (23, 80), (100, 3)]
    for i, (h, w) in enumerate(sizes):
        for kind in KINDS:
            yield f"{kind}_{h}x{w}", content(rng, kind, h, w, channels)


@pytest.mark.parametrize("channels", [1, 3])
def test_whole_file_equals_pil(channels):
    n = 0
    for name, a in sweep_cases(channels):
        assert jpeg_ref.encode(a) == pil_jpeg(a), name
        n += 1
    assert n == 4 * (256 + 17)


def test_header_layout():
    for channels, shape in ((1, (5, 7)), (3, (5, 7, 3))):
        f = jpeg_ref.encode(np.zeros(shape, np.uint8))
        assert f[:2] == b"\xff\xd8" and f[-2:] == b"\xff\xd9"
        assert f[:jpeg_ref.HEADER_BYTES[channels]] == jpeg_ref.header(5, 7, channels)
        sof = 20 + 69 * (1 if channels == 1 else 2)
        assert f[sof:sof + 2] == b"\xff\xc0" and f[sof + 5:sof + 9] == b"\x00\x05\x00\x07"


def test_zero_area_and_channels():
    assert jpeg_ref.encode(np.zeros((0, 5), np.uint8)) == b""
    assert jpeg_ref.encode(np.zeros((4, 0, 3), np.uint8)) == b""
    for bad in (np.zeros((4, 4, 2), np.uint8), np.zeros((4, 4, 4), np.uint8), np.zeros((4, 4), np.uint16)):
        with pytest.raises(ValueError):
            jpeg_ref.encode(bad)
    assert jpeg_ref.jpeg_bound(100, 1, 2) == -1 and jpeg_ref.jpeg_bound(100, 1, 4) == -1


@pytest.mark.parametrize("channels", [1, 3])
def test_bound_holds_for_worst_cases(channels):
    """Noise and 0 / 255 checkerboards on 1-pixel-wide and thin crops, and larger noise crops: the files of any set
    stay within mb_jpeg_bound_bytes' formula, and so does each crop alone."""
    rng = np.random.default_rng(9)
    crops = []
    for h, w in [(1, 1), (1, 2), (2, 1), (1, 17), (33, 1), (100, 1), (1, 100), (3, 5), (9, 9), (16, 16), (64, 48)]:
        crops.append(content(rng, "noise", h, w, channels))
        board = ((np.add.outer(np.arange(h), np.arange(w)) % 2) * 255).astype(np.uint8)
        crops.append(board if channels == 1 else np.repeat(board[..., None], 3, -1))
    total = 0
    for a in crops:
        n = len(jpeg_ref.encode(a))
        total += n
        assert n <= jpeg_ref.jpeg_bound(a.size, 1, channels)
        assert jpeg_ref.max_blocks(a.size // channels, 1, channels) >= (
            -(-a.shape[0] // 8) * -(-a.shape[1] // 8) if channels == 1 else 6 * -(-a.shape[0] // 16) * -(-a.shape[1] // 16))
    assert total <= jpeg_ref.jpeg_bound(sum(a.size for a in crops), len(crops), channels)

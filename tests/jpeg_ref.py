"""CPU restatement of mb_jpeg_encode (include/misob200.h): the file PIL.Image.fromarray(a).save(f, "JPEG") writes with
default arguments through libjpeg-turbo — baseline, quality 75, 4:2:0 for RGB, the standard Huffman tables, the islow
DCT — for uint8 [h, w] (mode L) and [h, w, 3] (RGB) arrays. The tables are Annex K's, not read back from PIL.

encode(a) returns the whole file; jpeg_bound(packed_bytes, crops, channels) is mb_jpeg_bound_bytes' formula."""
import numpy as np

# ---- ITU-T T.81 Annex K ----------------------------------------------------------------------------------------------
ZIGZAG = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,
                   7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,
                   39, 46, 53, 60, 61, 54, 47, 55, 62, 63])          # zigzag index -> natural (row-major) index
STD_LUMA = [16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22,
            29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103,
            121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99]
STD_CHROMA = ([17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99,
               99, 99, 99, 99, 99] + [99] * 32)
DC_LUMA_BITS = [0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0]
DC_CHROMA_BITS = [0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0]
DC_VALS = list(range(12))
AC_LUMA_BITS = [0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d]
AC_LUMA_VALS = [
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07,
    0x22, 0x71, 0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0,
    0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28,
    0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49,
    0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69,
    0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89,
    0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7,
    0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5,
    0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
    0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8,
    0xf9, 0xfa]
AC_CHROMA_BITS = [0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77]
AC_CHROMA_VALS = [
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71,
    0x13, 0x22, 0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0,
    0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26,
    0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
    0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68,
    0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87,
    0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5,
    0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
    0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
    0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8,
    0xf9, 0xfa]

QUALITY = 75
HEADER_BYTES = {1: 328, 3: 623}   # SOI .. SOS
MAX_BLOCK_BITS = 22 + 63 * 26     # DC code + amplitude <= 11 + 11; each AC <= 16 code + 10 amplitude bits


def quant_table(std, quality=QUALITY):
    """jcparam.c jpeg_add_quant_table with force_baseline: natural order, int64 [64]."""
    s = 5000 // quality if quality < 50 else 200 - 2 * quality
    return np.array([min(255, max(1, (v * s + 50) // 100)) for v in std], np.int64)


def huff_codes(bits, vals):
    """Canonical codes: symbol -> (code, length)."""
    code, k, tab = 0, 0, {}
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            tab[vals[k]] = (code, length)
            k += 1
            code += 1
        code <<= 1
    return tab


# ---- jfdctint.c (islow) ----------------------------------------------------------------------------------------------
CONST_BITS, PASS1_BITS = 13, 2
_F = {k: int(v * (1 << CONST_BITS) + 0.5) for k, v in dict(
    f0298=0.298631336, f0390=0.390180644, f0541=0.541196100, f0765=0.765366865, f0899=0.899976223, f1175=1.175875602,
    f1501=1.501321110, f1847=1.847759065, f1961=1.961570560, f2053=2.053119869, f2562=2.562915447,
    f3072=3.072711026).items()}


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _pass(d, first):
    d0, d1, d2, d3, d4, d5, d6, d7 = [d[..., i] for i in range(8)]
    t0, t7, t1, t6 = d0 + d7, d0 - d7, d1 + d6, d1 - d6
    t2, t5, t3, t4 = d2 + d5, d2 - d5, d3 + d4, d3 - d4
    t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    o = [None] * 8
    if first:
        o[0], o[4], sh = (t10 + t11) << PASS1_BITS, (t10 - t11) << PASS1_BITS, CONST_BITS - PASS1_BITS
    else:
        o[0], o[4], sh = _descale(t10 + t11, PASS1_BITS), _descale(t10 - t11, PASS1_BITS), CONST_BITS + PASS1_BITS
    z1 = (t12 + t13) * _F["f0541"]
    o[2] = _descale(z1 + t13 * _F["f0765"], sh)
    o[6] = _descale(z1 - t12 * _F["f1847"], sh)
    z1, z2, z3, z4 = t4 + t7, t5 + t6, t4 + t6, t5 + t7
    z5 = (z3 + z4) * _F["f1175"]
    t4, t5, t6, t7 = t4 * _F["f0298"], t5 * _F["f2053"], t6 * _F["f3072"], t7 * _F["f1501"]
    z1, z2 = -z1 * _F["f0899"], -z2 * _F["f2562"]
    z3, z4 = -z3 * _F["f1961"] + z5, -z4 * _F["f0390"] + z5
    o[7], o[5] = _descale(t4 + z1 + z3, sh), _descale(t5 + z2 + z4, sh)
    o[3], o[1] = _descale(t6 + z2 + z3, sh), _descale(t7 + z1 + z4, sh)
    return np.stack(o, -1)


def fdct(b):
    """b [..., 8, 8] int64 samples - 128 (row = y) -> coefficients [..., v, u], scaled by 8 as libjpeg leaves them."""
    r = _pass(b, True)
    return np.swapaxes(_pass(np.swapaxes(r, -1, -2), False), -1, -2)


def quantize(c, q):
    """Round half away from zero: (|c| + 4q) // 8q with the sign of c."""
    dv = q.reshape(8, 8) << 3
    v = (np.abs(c) + (dv >> 1)) // dv
    return np.where(c < 0, -v, v)


# ---- colour and sampling ---------------------------------------------------------------------------------------------
def ycc(a):
    """jccolor.c rgb_ycc_convert: int64 Y, Cb, Cr planes of an [h, w, 3] uint8 array."""
    r, g, b = [a[..., i].astype(np.int64) for i in range(3)]

    def fix(x):
        return int(x * 65536 + 0.5)
    half, cb = 1 << 15, (128 << 16) + (1 << 15) - 1
    y = (fix(0.29900) * r + fix(0.58700) * g + fix(0.11400) * b + half) >> 16
    u = (-fix(0.16874) * r - fix(0.33126) * g + fix(0.5) * b + cb) >> 16
    v = (fix(0.5) * r - fix(0.41869) * g - fix(0.08131) * b + cb) >> 16
    return y, u, v


def _pad(a, h, w):
    return np.pad(a, ((0, h - a.shape[0]), (0, w - a.shape[1])), mode="edge")


def downsample(c):
    """Chroma plane [h, w] -> [ceil(h/2) padded to 8k, 8 * ceil(ceil(w/2) / 8)]: full-resolution rows padded to an even
    count and columns to 16 * blocks by replication, h2v2 with bias 1, 2, 1, 2, ... along each output row, then the
    downsampled rows padded by replication to a whole block row."""
    h, w = c.shape
    ch, cwb = -(-h // 2), -(-(-(-w // 2)) // 8)
    p = _pad(c, 2 * ch, 16 * cwb)
    s = p.reshape(ch, 2, 8 * cwb, 2).sum((1, 3))
    bias = np.tile([1, 2], 4 * cwb)
    return _pad((s + bias) >> 2, 8 * -(-ch // 8), 8 * cwb)


def blocks(plane, q):
    """Plane [8 by, 8 bx] -> quantised coefficients [by, bx, 64] in zigzag order."""
    hb, wb = plane.shape[0] // 8, plane.shape[1] // 8
    b = plane.reshape(hb, 8, wb, 8).swapaxes(1, 2) - 128
    return quantize(fdct(b), q).reshape(hb, wb, 64)[..., ZIGZAG]


# ---- entropy coding --------------------------------------------------------------------------------------------------
class BitWriter:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def put(self, code, length):
        self.acc = (self.acc << length) | code
        self.n += length
        while self.n >= 8:
            self.n -= 8
            byte = (self.acc >> self.n) & 255
            self.out.append(byte)
            if byte == 0xFF:
                self.out.append(0)
        self.acc &= (1 << self.n) - 1

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)


def category(v):
    return int(abs(int(v))).bit_length()


def amplitude(v, n):
    return v if v >= 0 else v + (1 << n) - 1


def encode_block(bw, z, prev, dc, ac):
    d = int(z[0]) - prev
    n = category(d)
    bw.put(*dc[n])
    if n:
        bw.put(amplitude(d, n), n)
    run = 0
    for k in range(1, 64):
        v = int(z[k])
        if v == 0:
            run += 1
            continue
        while run > 15:
            bw.put(*ac[0xF0])
            run -= 16
        n = category(v)
        bw.put(*ac[(run << 4) | n])
        bw.put(amplitude(v, n), n)
        run = 0
    if run:
        bw.put(*ac[0x00])
    return int(z[0])


TABLES = [(huff_codes(DC_LUMA_BITS, DC_VALS), huff_codes(AC_LUMA_BITS, AC_LUMA_VALS)),
          (huff_codes(DC_CHROMA_BITS, DC_VALS), huff_codes(AC_CHROMA_BITS, AC_CHROMA_VALS))]


def scan(a):
    """The entropy-coded segment (stuffed, padded with 1-bits) of a uint8 [h, w] or [h, w, 3] array."""
    ql, qc = quant_table(STD_LUMA), quant_table(STD_CHROMA)
    bw = BitWriter()
    if a.ndim == 2:
        h, w = a.shape
        q = blocks(_pad(a.astype(np.int64), 8 * -(-h // 8), 8 * -(-w // 8)), ql)
        prev = 0
        for by in range(q.shape[0]):
            for bx in range(q.shape[1]):
                prev = encode_block(bw, q[by, bx], prev, *TABLES[0])
    else:
        h, w, _ = a.shape
        y, cb, cr = ycc(a)
        comps = [blocks(_pad(y, 8 * -(-h // 8), 8 * -(-w // 8)), ql), blocks(downsample(cb), qc),
                 blocks(downsample(cr), qc)]
        prev = [0, 0, 0]
        for my in range(-(-h // 16)):
            for mx in range(-(-w // 16)):
                for ci, (q, n) in enumerate(zip(comps, (2, 1, 1))):
                    last = 0
                    for yy in range(n):
                        for xx in range(n):
                            by, bx = my * n + yy, mx * n + xx
                            if by < q.shape[0] and bx < q.shape[1]:
                                z = q[by, bx]
                            else:                   # dummy block (jccoefct.c): zero AC, the DC of the block before it
                                z = np.zeros(64, np.int64)
                                z[0] = last
                            prev[ci] = encode_block(bw, z, prev[ci], *TABLES[min(ci, 1)])
                            last = int(z[0])
    bw.flush()
    return bytes(bw.out)


# ---- framing ---------------------------------------------------------------------------------------------------------
def _segment(marker, body):
    return bytes([0xFF, marker]) + (len(body) + 2).to_bytes(2, "big") + body


def header(h, w, channels):
    """SOI .. SOS of the file (HEADER_BYTES[channels] bytes)."""
    ql, qc = quant_table(STD_LUMA), quant_table(STD_CHROMA)
    out = b"\xff\xd8" + _segment(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    out += _segment(0xDB, bytes([0]) + bytes(int(v) for v in ql[ZIGZAG]))
    if channels == 3:
        out += _segment(0xDB, bytes([1]) + bytes(int(v) for v in qc[ZIGZAG]))
    comps = [(1, 0x11 if channels == 1 else 0x22, 0)] + ([(2, 0x11, 1), (3, 0x11, 1)] if channels == 3 else [])
    out += _segment(0xC0, bytes([8]) + h.to_bytes(2, "big") + w.to_bytes(2, "big") + bytes([channels])
                    + b"".join(bytes(c) for c in comps))
    dht = [(0x00, DC_LUMA_BITS, DC_VALS), (0x10, AC_LUMA_BITS, AC_LUMA_VALS)]
    if channels == 3:
        dht += [(0x01, DC_CHROMA_BITS, DC_VALS), (0x11, AC_CHROMA_BITS, AC_CHROMA_VALS)]
    for tc, bits, vals in dht:
        out += _segment(0xC4, bytes([tc] + bits + vals))
    sel = [(1, 0x00)] + ([(2, 0x11), (3, 0x11)] if channels == 3 else [])
    out += _segment(0xDA, bytes([channels]) + b"".join(bytes(s) for s in sel) + b"\x00\x3f\x00")
    assert len(out) == HEADER_BYTES[channels]
    return out


def encode(a):
    """The whole JPEG file of a uint8 [h, w] or [h, w, 3] array; b"" for zero area."""
    a = np.ascontiguousarray(a)
    if a.ndim == 3 and a.shape[2] == 1:
        a = a[..., 0]
    if a.dtype != np.uint8 or not (a.ndim == 2 or (a.ndim == 3 and a.shape[2] == 3)):
        raise ValueError("jpeg_ref.encode: uint8 [h, w] or [h, w, 3]")
    if a.size == 0:
        return b""
    channels = 1 if a.ndim == 2 else 3
    return header(a.shape[0], a.shape[1], channels) + scan(a) + b"\xff\xd9"


def max_blocks(pixels, crops, channels):
    """Most blocks (dummy blocks included) any crops of `pixels` pixels in total can have: a crop of h x w pixels
    (h, w >= 1, so h + w <= h w + 1) has ceil(h/8) ceil(w/8) <= (h w) / 8 + 7/8 blocks in grey and
    6 ceil(h/16) ceil(w/16) <= 6 ((h w) / 16 + 15/16) in colour; 1-pixel-wide crops come closest."""
    return pixels // 8 + crops if channels == 1 else 6 * (pixels // 16 + crops)


def jpeg_bound(packed_bytes, crops, channels):
    """mb_jpeg_bound_bytes: header and EOI per crop plus every block at MAX_BLOCK_BITS, each byte 0xFF-stuffed."""
    if channels not in (1, 3) or packed_bytes < 0 or crops < 0:
        return -1
    return crops * (HEADER_BYTES[channels] + 2) + 2 * ((MAX_BLOCK_BITS + 7) // 8) * max_blocks(packed_bytes // channels, crops, channels)

"""CPU restatement of mb_png_encode (include/misob200.h): the PNG stream of one uint8 crop, byte for byte.

  framing   signature, IHDR (bit depth 8, colour type 0 / 4 / 2 / 6 for 1..4 channels, no interlace), one IDAT, IEND
  filter    per row, libpng's heuristic: the type 0..4 with the least sum of |(int8) filtered byte| (ties: lower type);
            the previous row is the source's, so a row's choice does not depend on where blocks are cut
  blocks    the filtered stream (h * (1 + w * c) bytes) cut every BLOCK bytes; each block is one non-final deflate
            block followed by an empty stored block (a sync flush), the stream ends with an empty final fixed block
  tokens    per maximal run of n equal bytes inside a block: one literal, then the n - 1 repeats as length-258
            matches at distance 1, then the m = (n - 1) % 258 left over: one match of length m if m >= 3, else m
            literals
  codes     dynamic; lengths by package-merge (limit 15, 7 for the code-length code; symbols sorted by (frequency,
            index), leaves before packages of equal weight); fewer than two used symbols: the lowest unused indices
            are added with length 1 (so the distance code is always lengths [1, 1]); the code-length sequence is run-
            length coded per tree with zlib's scan_tree / send_tree rule
  stored    a block whose dynamic form (plus its sync flush) is not shorter than its stored form is stored
  zlib      header 78 01; Adler-32 of the filtered bytes; the IDAT CRC-32 is combined from per-block CRCs
"""
from __future__ import annotations

import struct
import zlib

import numpy as np

BLOCK = 32768
SIGNATURE = b"\x89PNG\r\n\x1a\n"
COLOR_TYPE = {1: 0, 2: 4, 3: 2, 4: 6}
ZLIB_HEADER = b"\x78\x01"
FINAL_BLOCK = b"\x03\x00"          # BFINAL = 1, fixed Huffman, end-of-block
SYNC_FLUSH = b"\x00\x00\xff\xff"   # LEN / NLEN of the empty stored block (its 3 header bits precede it)
BL_ORDER = (16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15)
MOD_ADLER = 65521

# length 3..258 -> (symbol, extra bits, base)
_LEN_BASE = [3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195,
             227, 258]
_LEN_EXTRA = [0] * 8 + [1] * 4 + [2] * 4 + [3] * 4 + [4] * 4 + [5] * 4 + [0]
LEN_SYM = np.zeros(259, np.int64)
LEN_XB = np.zeros(259, np.int64)
LEN_XV = np.zeros(259, np.int64)
for _i, (_b, _e) in enumerate(zip(_LEN_BASE, _LEN_EXTRA)):
    for _l in range(_b, (_LEN_BASE[_i + 1] if _i + 1 < len(_LEN_BASE) else 259)):
        if _l == 258 and _b != 258:
            continue
        LEN_SYM[_l], LEN_XB[_l], LEN_XV[_l] = 257 + _i, _e, _l - _b


def png_bound(h: int, w: int, c: int) -> int:
    """Largest stream of an h x w x c crop: 65 bytes of framing plus every block stored (10 bytes each)."""
    f = h * (1 + w * c) if h * w else 0
    return 65 + f + 10 * (-(-f // BLOCK)) if f else 0


# ------------------------------------------------------------------------------------------------------------------
# filters
# ------------------------------------------------------------------------------------------------------------------
def filter_rows(a: np.ndarray, c: int):
    """a: uint8 [h, w * c] -> (filter type per row, filtered rows [h, w * c]) with libpng's heuristic."""
    a = a.astype(np.int16)
    h, n = a.shape
    up = np.vstack([np.zeros((1, n), np.int16), a[:-1]])
    left = np.hstack([np.zeros((h, c), np.int16), a[:, :-c]]) if n > c else np.zeros_like(a)
    ul = np.hstack([np.zeros((h, c), np.int16), up[:, :-c]]) if n > c else np.zeros_like(a)
    p = left + up - ul
    pa, pb, pc = np.abs(p - left), np.abs(p - up), np.abs(p - ul)
    paeth = np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, up, ul))
    cand = np.stack([a, a - left, a - up, a - ((left + up) >> 1), a - paeth]) & 255
    cost = np.where(cand < 128, cand, 256 - cand).sum(axis=2)        # [5, h]
    ftype = np.argmin(cost, axis=0)                                  # first minimum: the lower type wins ties
    return ftype, cand[ftype, np.arange(h)].astype(np.uint8)


def filtered_stream(crop: np.ndarray) -> bytes:
    h, w = crop.shape[:2]
    c = 1 if crop.ndim == 2 else crop.shape[2]
    ftype, rows = filter_rows(np.ascontiguousarray(crop).reshape(h, w * c), c)
    return np.hstack([ftype.astype(np.uint8)[:, None], rows]).tobytes()


# ------------------------------------------------------------------------------------------------------------------
# Huffman code lengths
# ------------------------------------------------------------------------------------------------------------------
def package_merge(freqs, limit: int):
    """Code lengths of the used symbols (freq > 0): package-merge over the symbols sorted by (freq, index); equal
    weights merge leaves first. Fewer than two used symbols: the lowest unused indices join with length 1."""
    freqs = list(freqs)
    used = [s for s, f in enumerate(freqs) if f > 0]
    lengths = [0] * len(freqs)
    if len(used) < 2:
        extra = [s for s in range(len(freqs)) if s not in used][:2 - len(used)]
        for s in used + extra:
            lengths[s] = 1
        return lengths
    order = sorted(used, key=lambda s: (freqs[s], s))
    leaves = [freqs[s] for s in order]
    n = len(leaves)
    cur = list(leaves)
    leafpos = {limit: list(range(n))}
    for d in range(limit - 1, 0, -1):
        pk = [cur[2 * k] + cur[2 * k + 1] for k in range(len(cur) // 2)]
        merged, pos, i, j = [], [], 0, 0
        while i < n or j < len(pk):
            if j >= len(pk) or (i < n and leaves[i] <= pk[j]):
                pos.append(len(merged)); merged.append(leaves[i]); i += 1
            else:
                merged.append(pk[j]); j += 1
        leafpos[d] = pos
        cur = merged
    k = 2 * n - 2
    for d in range(1, limit + 1):
        nl = sum(1 for p in leafpos[d] if p < k)
        for i in range(nl):
            lengths[order[i]] += 1
        k = 2 * (k - nl)
    return lengths


def canonical_codes(lengths):
    """Deflate's canonical codes, bit-reversed for the LSB-first stream."""
    maxl = max(lengths) if lengths else 0
    bl_count = [0] * (maxl + 2)
    for l in lengths:
        if l:
            bl_count[l] += 1
    code, next_code = 0, [0] * (maxl + 2)
    for b in range(1, maxl + 1):
        code = (code + bl_count[b - 1]) << 1 if b > 1 else 0
        next_code[b] = code
    out = [0] * len(lengths)
    for s, l in enumerate(lengths):
        if l:
            c = next_code[l]; next_code[l] += 1
            out[s] = int(format(c, f"0{l}b")[::-1], 2)
    return out


def _tree_runs(lens):
    """zlib's scan_tree / send_tree over one tree's lengths (max_code = len(lens) - 1): [(symbol, extra, nbits)]."""
    out = []
    prevlen, nextlen, count = -1, lens[0], 0
    max_count, min_count = (138, 3) if nextlen == 0 else (7, 4)
    for n in range(len(lens)):
        curlen = nextlen
        nextlen = lens[n + 1] if n + 1 < len(lens) else 0xffff
        count += 1
        if count < max_count and curlen == nextlen:
            continue
        if count < min_count:
            out += [(curlen, 0, 0)] * count
        elif curlen != 0:
            if curlen != prevlen:
                out.append((curlen, 0, 0)); count -= 1
            out.append((16, count - 3, 2))
        elif count <= 10:
            out.append((17, count - 3, 3))
        else:
            out.append((18, count - 11, 7))
        count, prevlen = 0, curlen
        if nextlen == 0:
            max_count, min_count = 138, 3
        elif curlen == nextlen:
            max_count, min_count = 6, 3
        else:
            max_count, min_count = 7, 4
    return out


# ------------------------------------------------------------------------------------------------------------------
# one block
# ------------------------------------------------------------------------------------------------------------------
def block_tokens(d: np.ndarray):
    """Tokens of one block: (is_match, byte or length) per emitting position, in stream order."""
    L = d.size
    idx = np.arange(L)
    start = np.ones(L, bool)
    start[1:] = d[1:] != d[:-1]
    s = np.maximum.accumulate(np.where(start, idx, 0))
    nxt = np.where(start, idx, L)
    e = np.minimum.accumulate(np.append(nxt[1:], L)[::-1])[::-1]        # first run start after each position
    k, m = idx - s, e - s - 1
    q = k - 1
    full = m // 258
    r = m - 258 * full
    in_full = (k >= 1) & (q < 258 * full)
    qt = q - 258 * full
    emit_lit = (k == 0) | ((k >= 1) & ~in_full & (r < 3))
    emit_m258 = in_full & (q % 258 == 0)
    emit_mr = (k >= 1) & ~in_full & (r >= 3) & (qt == 0)
    emit = emit_lit | emit_m258 | emit_mr
    is_match = (emit_m258 | emit_mr)[emit]
    value = np.where(emit_m258, 258, np.where(emit_mr, r, d.astype(np.int64)))[emit]
    return is_match, value


def _pack_bits(vals, nbits):
    vals = np.asarray(vals, np.uint64)
    nbits = np.asarray(nbits, np.int64)
    pos = np.concatenate([[0], np.cumsum(nbits)])
    total = int(pos[-1])
    bits = np.zeros(total + (-total) % 8, np.uint8)
    for j in range(int(nbits.max()) if nbits.size else 0):
        sel = nbits > j
        bits[pos[:-1][sel] + j] = ((vals[sel] >> np.uint64(j)) & np.uint64(1)).astype(np.uint8)
    return total, bits


def encode_block(d: np.ndarray):
    """One block -> (segment bytes: the block and its sync flush, kind 'dynamic' / 'stored', litlen lengths, bl lengths)."""
    L = d.size
    is_match, value = block_tokens(d)
    sym = np.where(is_match, LEN_SYM[np.where(is_match, value, 3)], value)
    freq = np.bincount(sym, minlength=286)
    freq[256] += 1
    ll = package_merge(freq, 15)
    hlit = max(s for s in range(286) if ll[s]) + 1
    dl = [1, 1]                                      # distance code: only code 0 (distance 1) is ever used
    runs = _tree_runs(ll[:hlit]) + _tree_runs(dl)
    blf = [0] * 19
    for s, _, _ in runs:
        blf[s] += 1
    bl = package_merge(blf, 7)
    hclen = 4
    for i in range(18, 3, -1):
        if bl[BL_ORDER[i]]:
            hclen = i + 1
            break
    llc, blc = canonical_codes(ll), canonical_codes(bl)
    head = [(0, 1), (2, 2), (hlit - 257, 5), (1, 5), (hclen - 4, 4)] + [(bl[BL_ORDER[i]], 3) for i in range(hclen)]
    for s, x, xb in runs:
        head.append((blc[s], bl[s]))
        if xb:
            head.append((x, xb))
    llen = np.array(ll, np.int64)
    lcode = np.array(llc, np.uint64)
    xb = np.where(is_match, LEN_XB[np.where(is_match, value, 3)], 0)
    xv = np.where(is_match, LEN_XV[np.where(is_match, value, 3)], 0).astype(np.uint64)
    ln = llen[sym]
    tv = lcode[sym] | (xv << ln.astype(np.uint64))                  # + distance code 0: one 0 bit
    tn = ln + xb + is_match.astype(np.int64)
    vals = [v for v, _ in head] + list(tv) + [llc[256]]
    nbits = [n for _, n in head] + list(tn) + [ll[256]]
    total, bits = _pack_bits(vals, nbits)
    dyn_bytes = (total + 3 + 7) // 8 + 4
    if dyn_bytes < L + 10:
        body = np.packbits(np.append(bits, np.zeros((total + 3 + 7) // 8 * 8 - bits.size, np.uint8)), bitorder="little")
        return body.tobytes() + SYNC_FLUSH, "dynamic", ll, bl
    return (b"\x00" + struct.pack("<HH", L, L ^ 0xffff) + d.tobytes() + b"\x00" + SYNC_FLUSH), "stored", ll, bl


# ------------------------------------------------------------------------------------------------------------------
# checksums from per-block partials
# ------------------------------------------------------------------------------------------------------------------
_POLY = 0xedb88320


def multmodp(a: int, b: int) -> int:
    m, p = 1 << 31, 0
    while True:
        if a & m:
            p ^= b
            if (a & (m - 1)) == 0:
                return p
        m >>= 1
        b = (b >> 1) ^ _POLY if b & 1 else b >> 1


def x8nmodp(n: int) -> int:
    """x^(8 n) mod the CRC-32 polynomial (reflected)."""
    p, sq = 1 << 31, 1 << 23            # x^0, x^8
    while n:
        if n & 1:
            p = multmodp(sq, p)
        sq = multmodp(sq, sq)
        n >>= 1
    return p


def crc32_combine(crc1: int, crc2: int, len2: int) -> int:
    return multmodp(x8nmodp(len2), crc1) ^ crc2


def adler_partial(d: np.ndarray):
    """(sum of bytes, sum of (L - i) * byte) mod 65521 of one block."""
    v = d.astype(np.int64)
    return int(v.sum() % MOD_ADLER), int(((d.size - np.arange(d.size)) * v).sum() % MOD_ADLER)


def adler_combine(parts):
    """Adler-32 of the concatenation from [(len, A, Bw)] partials."""
    A = B = n = 0
    for L, a, b in parts:
        B = (B + (L % MOD_ADLER) * A + b) % MOD_ADLER
        A = (A + a) % MOD_ADLER
        n += L
    return (((n + B) % MOD_ADLER) << 16) | ((1 + A) % MOD_ADLER)


def _chunk(kind: bytes, data: bytes) -> bytes:
    return struct.pack(">I", len(data)) + kind + data + struct.pack(">I", zlib.crc32(kind + data))


def encode(crop: np.ndarray, info: dict | None = None) -> bytes:
    """PNG stream of one uint8 crop ([h, w] or [h, w, c], c in 1..4); b"" when h * w == 0."""
    h, w = crop.shape[:2]
    c = 1 if crop.ndim == 2 else crop.shape[2]
    if not 1 <= c <= 4:
        raise ValueError("1..4 channels")
    if h * w == 0:
        return b""
    f = np.frombuffer(filtered_stream(crop), np.uint8)
    segs, crcs, adl = [], [], []
    for b0 in range(0, f.size, BLOCK):
        d = f[b0:b0 + BLOCK]
        seg, kind, ll, bl = encode_block(d)
        segs.append(seg)
        crcs.append((zlib.crc32(seg), len(seg)))
        adl.append((d.size,) + adler_partial(d))
        if info is not None:
            info.setdefault("blocks", []).append({"kind": kind, "ll": ll, "bl": bl})
    adler = adler_combine(adl)
    tail = FINAL_BLOCK + struct.pack(">I", adler)
    crc = zlib.crc32(b"IDAT" + ZLIB_HEADER)
    for cb, n in crcs:
        crc = crc32_combine(crc, cb, n)
    crc = zlib.crc32(tail, crc)
    idat = ZLIB_HEADER + b"".join(segs) + tail
    if info is not None:
        info.update(adler=adler, crc=crc, filtered=f.tobytes())
    ihdr = struct.pack(">IIBBBBB", w, h, 8, COLOR_TYPE[c], 0, 0, 0)
    return (SIGNATURE + _chunk(b"IHDR", ihdr) + struct.pack(">I", len(idat)) + b"IDAT" + idat + struct.pack(">I", crc)
            + _chunk(b"IEND", b""))


def encode_packed(packed: np.ndarray, rects, offsets, channels: int, src_channels: int):
    """Streams of packed crops as mb_png_encode reads them: crop j at offsets[j] // src_channels * channels."""
    out = []
    for j, (_, _, w, h) in enumerate(rects):
        o = int(offsets[j]) // src_channels * channels
        a = packed[o:o + h * w * channels].reshape((h, w, channels) if channels > 1 else (h, w))
        out.append(encode(a))
    return out

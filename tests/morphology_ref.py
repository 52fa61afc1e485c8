"""CPU restatement of a crop's morphology record (mb_mask_morphology, include/misob200.h): the definitions in Python
integers, then fp64 in the order the ABI states them. Shared by tests/test_morphology_ref.py (which checks it against
an independent scipy / eigvalsh restatement) and tests/test_gpu_morphology.py (which checks the kernel against it)."""
import math

import numpy as np

FIELDS = 13
SQRT2 = math.sqrt(2.0)
DIAG = (1.0 + SQRT2) / 2.0
N1_CODES, N2_CODES, N3_CODES = (5, 7, 15, 17, 25, 27), (21, 33), (13, 23)


def perimeter_codes(m: np.ndarray) -> np.ndarray:
    """Code image of the border pixels B (0 elsewhere): 1 + 2 * (4-neighbours in B) + 10 * (diagonal neighbours in B)."""
    p = np.pad(m, 1)
    eroded = m & p[:-2, 1:-1] & p[2:, 1:-1] & p[1:-1, :-2] & p[1:-1, 2:]
    b = m & ~eroded
    q = np.pad(b, 1).astype(np.int64)
    n4 = q[1:-1, :-2] + q[1:-1, 2:] + q[:-2, 1:-1] + q[2:, 1:-1]
    nd = q[:-2, :-2] + q[:-2, 2:] + q[2:, :-2] + q[2:, 2:]
    return np.where(b, 1 + 2 * n4 + 10 * nd, 0)


def sums(mask: np.ndarray, pixels: np.ndarray):
    """Exact integer sums (A, S_r, S_c, S_rr, S_cc, S_rc, [P_k], n1, n2, n3) as Python ints. pixels: [h, w, ch] or [h, w]."""
    m = np.asarray(mask) != 0
    rr, cc = np.nonzero(m)
    rr, cc = rr.astype(np.int64), cc.astype(np.int64)
    px = np.asarray(pixels)
    px = px[..., None] if px.ndim == 2 else px
    p = [int(px[..., k][m].astype(np.int64).sum()) for k in range(px.shape[2])]
    codes = perimeter_codes(m)
    n = [int(np.isin(codes, c).sum()) for c in (N1_CODES, N2_CODES, N3_CODES)]
    return (int(m.sum()), int(rr.sum()), int(cc.sum()), int((rr * rr).sum()), int((cc * cc).sum()), int((rr * cc).sum()),
            p, n)


def record(mask: np.ndarray, pixels: np.ndarray, x: int, y: int) -> np.ndarray:
    """The 13 fp64 fields of one crop with rect origin (x, y)."""
    A, Sr, Sc, Srr, Scc, Src, P, (n1, n2, n3) = sums(mask, pixels)
    out = np.zeros(FIELDS, np.float64)
    if A == 0:
        return out
    fa = float(A)
    a2 = fa * fa
    urr = float(A * Srr - Sr * Sr) / a2
    ucc = float(A * Scc - Sc * Sc) / a2
    urc = float(A * Src - Sr * Sc) / a2
    a, b, c = ucc, -urc, urr
    root = math.sqrt((a - c) * (a - c) + 4.0 * (b * b))
    l1, l2 = ((a + c) + root) / 2.0, ((a + c) - root) / 2.0
    l1, l2 = (l1 if l1 > 0.0 else 0.0), (l2 if l2 > 0.0 else 0.0)
    out[0] = fa
    out[1] = (n1 + SQRT2 * n2) + DIAG * n3
    out[2] = x + Sc / A
    out[3] = y + Sr / A
    out[4] = 4.0 * math.sqrt(l1)
    out[5] = 4.0 * math.sqrt(l2)
    out[6] = ((-math.pi / 4 if b < 0.0 else math.pi / 4) if a == c else 0.5 * math.atan2(-2.0 * b, c - a))
    out[7] = 0.0 if l1 == 0.0 else math.sqrt(1.0 - l2 / l1)
    out[8] = math.sqrt(4 * A / math.pi)
    for k, pk in enumerate(P[:4]):
        out[9 + k] = pk / A
    return out


EXACT = [0, 1, 2, 3, 8, 9, 10, 11, 12]      # fields computed by exactly rounded operations from exact sums
APPROX = [4, 5, 6, 7]                       # 128-bit -> fp64 conversions, atan2: agree within 1e-12


def assert_records_match(got: np.ndarray, want: np.ndarray, what="") -> None:
    got, want = np.atleast_2d(got), np.atleast_2d(want)
    assert got.shape == want.shape, (got.shape, want.shape)
    bad = np.nonzero(np.any(got[:, EXACT] != want[:, EXACT], axis=1))[0]
    assert len(bad) == 0, f"{what}: exact fields differ at rows {bad[:10]}: {got[bad[0]]} vs {want[bad[0]]}"
    np.testing.assert_allclose(got[:, APPROX], want[:, APPROX], rtol=1e-12, atol=1e-12, err_msg=what)

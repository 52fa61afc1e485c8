"""The sparse greedy NMS reference (tests/nms_ref.py) against the dense C oracle, on the CPU.

The GPU route tests compare their largest cases with the sparse reference only, so it has to make exactly the
oracle's decisions: every shared NMS case, every input family of the route tests, random sets up to 20k boxes with
ties, NaN scores and zero-area duplicates, negative thresholds, per-group (vanilla) mode and the keep cap."""
import numpy as np
import pytest

from oracle import detection as D
from oracle import native
from tests import cases
from tests import nms_ref as R


def test_score_order_is_the_oracles():
    s = np.array([0.5, np.nan, -0.0, 0.0, 0.5, -1.0, np.inf, np.nan, -np.inf, 0.25], np.float32)
    assert np.array_equal(R.score_order(s), native.argsort_desc_stable(s))
    rng = np.random.default_rng(5)
    s = (np.floor(rng.uniform(-1, 1, 5000) * 16) / 16).astype(np.float32)
    s[::37] = np.nan
    s[::41] = -0.0
    assert np.array_equal(R.score_order(s), native.argsort_desc_stable(s))


def test_shared_nms_cases():
    for name, b, s, thr in cases.nms_cases():
        assert np.array_equal(R.nms(b, s, thr), native.nms(b, s, thr)), name


def test_shared_batched_nms_cases():
    for name, b, s, idx, thr in cases.batched_nms_cases():
        assert np.array_equal(R.batched_nms_vanilla(b, s, idx, thr), D.batched_nms_vanilla(b, s, idx, thr)), name
        assert np.array_equal(R.batched_nms_coordinate_trick(b, s, idx, thr),
                              D.batched_nms_coordinate_trick(b, s, idx, thr)), name


@pytest.mark.parametrize("family", cases.NMS_FAMILIES)
@pytest.mark.parametrize("n", [1, 2, 65, 1025, 4097])
def test_route_families(family, n):
    for thr in (0.0, 0.5, 0.7, 1.0, -0.25, 0.33333334):
        b, s = cases.nms_family(family, n, thr)
        want = native.nms(b, s, thr)
        assert np.array_equal(R.nms(b, s, thr), want), (family, n, thr)
        assert np.array_equal(R.nms(b, s, thr, max_keep=64), want[:64]), (family, n, thr)


def test_chain_family_alternates():
    """The chain family is what it claims: keep / remove alternate along the 1024-link chain."""
    b, s = cases.nms_family("chain", 1024, 0.5)
    keep = native.nms(b, s, 0.5)
    order = native.argsort_desc_stable(s)
    assert np.array_equal(keep, order[::2])


@pytest.mark.parametrize("n", [3000, 20000])
def test_random_sets(n):
    rng = np.random.default_rng(n)
    c = rng.uniform(0, 24.0 * np.sqrt(n), (n, 2))
    wh = np.exp(rng.uniform(np.log(4), np.log(160), (n, 2)))
    b = np.concatenate([c - wh / 2, c + wh / 2], 1).astype(np.float32)
    b[rng.integers(0, n, n // 20)] = b[rng.integers(0, n, n // 20)]           # duplicates
    z = rng.integers(0, n, n // 40)
    b[z, 2:] = b[z, :2]                                                       # zero area
    s = (np.floor(rng.uniform(0, 1, n) * 512) / 512).astype(np.float32)    # ties
    s[rng.integers(0, n, n // 100)] = np.nan
    for thr in (0.0, 0.3, 0.7, 0.33333334):
        assert np.array_equal(R.nms(b, s, thr), native.nms(b, s, thr)), (n, thr)
    g = rng.integers(0, 13, n).astype(np.int64)
    g[g == 5] = 7                                                             # a gap in the group indices
    want = D.batched_nms_vanilla(b, s, g, 0.5)
    assert np.array_equal(R.batched_nms_vanilla(b, s, g, 0.5), want)
    # keep cap per group: the first max_keep boxes each group's own NMS keeps
    capped = R.nms(b, s, 0.5, groups=g, max_keep=40)
    per_group = {}
    expect = [i for i in want if per_group.setdefault(g[i], []).append(i) or len(per_group[g[i]]) <= 40]
    assert np.array_equal(capped, np.asarray(expect, np.int64))


def test_non_finite_coordinates_and_negative_thresholds():
    rng = np.random.default_rng(3)
    b = cases.random_boxes(rng, 300, extent=100.0)
    s = cases.distinct_scores(rng, 300)
    b[5, 0] = np.nan
    b[9, 3] = np.inf
    for thr in (0.5, -1e-9, -0.5):
        assert np.array_equal(R.nms(b, s, thr), native.nms(b, s, thr)), thr
    g = rng.integers(0, 4, 300)
    assert np.array_equal(R.batched_nms_vanilla(b, s, g, -0.1), D.batched_nms_vanilla(b, s, g, -0.1))

"""Sparse, exact greedy NMS on the CPU (numpy): the decisions of oracle.native.nms at any size.

The C oracle visits every (kept, later) pair, O(N * kept): fine up to ~25k boxes, far too slow for a 140k-box segment.
For a threshold >= 0 a box can only suppress another if their intersection is positive (IoU 0 is never > thr, and 0/0
is NaN, which never suppresses), so only pairs whose x and y intervals overlap with positive extent matter. Those are
found from a uniform grid: each box is listed in every cell it touches, and a pair is examined only in the cell that
holds the lower-left corner of its intersection, so it is examined once. The IoU of a candidate pair is computed in
fp32 in the oracle's operation order (areas, max / min, clamp at 0, product, (a1 + a2) - inter, division; no FMA) and
suppresses iff (double)iou > thr. The greedy pass then walks the boxes in the oracle's order (stable descending score,
NaN first, -0 == +0, then ascending index) over adjacency lists.

Thresholds below 0 (every disjoint pair suppresses) and non-finite coordinates fall back to the dense oracle.
"""
from __future__ import annotations

import numpy as np

from oracle import native

F = np.float32


def score_order(scores) -> np.ndarray:
    """Indices in the oracle's visiting order: score descending with NaN first and -0 == +0, ties by ascending index."""
    s = np.asarray(scores, F).reshape(-1)
    nan = np.isnan(s)
    neg = np.where(nan, 0.0, -s.astype(np.float64)) + 0.0          # + 0.0 folds -0 into +0
    return np.lexsort((np.arange(s.shape[0]), neg, ~nan)).astype(np.int64)


def _candidate_pairs(b: np.ndarray, live: np.ndarray):
    """All pairs (i, j), i < j, of live boxes whose intersection has positive width and height."""
    idx = np.nonzero(live)[0]
    if idx.shape[0] < 2:
        return np.empty(0, np.int64), np.empty(0, np.int64)
    x1, y1, x2, y2 = (b[idx, k].astype(np.float64) for k in range(4))
    side = np.maximum(x2 - x1, y2 - y1)
    cell = max(float(np.percentile(side, 75)), 1e-30)
    while True:
        cx0, cx1 = np.floor(x1 / cell).astype(np.int64), np.floor(x2 / cell).astype(np.int64)
        cy0, cy1 = np.floor(y1 / cell).astype(np.int64), np.floor(y2 / cell).astype(np.int64)
        nx, ny = cx1 - cx0 + 1, cy1 - cy0 + 1
        if int((nx * ny).sum()) <= 8 * idx.shape[0] + 1_000_000:
            break
        cell *= 2.0
    # one entry per (box, cell touched)
    per = nx * ny
    box = np.repeat(np.arange(idx.shape[0]), per)
    k = np.arange(box.shape[0]) - np.repeat(np.cumsum(per) - per, per)
    ex = cx0[box] + k % nx[box]
    ey = cy0[box] + k // nx[box]
    ex0, ey0 = ex.min(), ey.min()
    key = (ex - ex0) * (int(ey.max() - ey0) + 1) + (ey - ey0)
    o = np.argsort(key, kind="stable")
    key, box, ex, ey = key[o], box[o], ex[o], ey[o]
    # pairs inside each cell: entry p with every later entry of the same cell
    end = np.searchsorted(key, key, side="right")
    cnt = end - np.arange(key.shape[0]) - 1
    first = np.repeat(np.arange(key.shape[0]), cnt)
    second = first + 1 + (np.arange(first.shape[0]) - np.repeat(np.cumsum(cnt) - cnt, cnt))
    a, c = box[first], box[second]
    ix1, iy1 = np.maximum(x1[a], x1[c]), np.maximum(y1[a], y1[c])
    ok = (ix1 < np.minimum(x2[a], x2[c])) & (iy1 < np.minimum(y2[a], y2[c]))
    # the pair is counted in the cell of its intersection's lower-left corner only
    ok &= (np.floor(ix1 / cell).astype(np.int64) == ex[first]) & (np.floor(iy1 / cell).astype(np.int64) == ey[first])
    a, c = idx[a[ok]], idx[c[ok]]
    return np.minimum(a, c), np.maximum(a, c)


def _suppresses(b: np.ndarray, i: np.ndarray, j: np.ndarray, thr: float) -> np.ndarray:
    """(double)iou(i, j) > thr, fp32 arithmetic in the oracle's operation order."""
    area = ((b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])).astype(F)
    with np.errstate(all="ignore"):
        xx1 = np.maximum(b[i, 0], b[j, 0]); yy1 = np.maximum(b[i, 1], b[j, 1])
        xx2 = np.minimum(b[i, 2], b[j, 2]); yy2 = np.minimum(b[i, 3], b[j, 3])
        w = np.maximum(xx2 - xx1, F(0)); h = np.maximum(yy2 - yy1, F(0))
        inter = (w * h).astype(F)
        uni = ((area[i] + area[j]).astype(F) - inter).astype(F)
        ovr = (inter / uni).astype(F)
    return ovr.astype(np.float64) > thr


def _greedy(n: int, order: np.ndarray, i: np.ndarray, j: np.ndarray, groups, max_keep: int) -> np.ndarray:
    """Greedy pass in `order` over the suppression edges (i, j); per-group keep cap when max_keep > 0."""
    rank = np.empty(n, np.int64)
    rank[order] = np.arange(n)
    src = np.where(rank[i] < rank[j], i, j)          # the earlier box of each pair suppresses the later one
    dst = np.where(rank[i] < rank[j], j, i)
    o = np.argsort(src, kind="stable")
    src, dst = src[o], dst[o]
    start = np.searchsorted(src, np.arange(n + 1))
    removed = np.zeros(n, bool)
    kept_in = {}
    keep = []
    for p in order.tolist():
        if removed[p]:
            continue
        if max_keep > 0:
            g = 0 if groups is None else int(groups[p])
            if kept_in.get(g, 0) >= max_keep:
                continue                              # this group is full: later boxes of it are not kept either
            kept_in[g] = kept_in.get(g, 0) + 1
        keep.append(p)
        removed[dst[start[p]:start[p + 1]]] = True
    return np.asarray(keep, np.int64)


def _dense(boxes, scores, groups, thr, max_keep):
    if groups is None:
        k = native.nms(boxes, scores, thr)
        return k[:max_keep] if max_keep > 0 else k
    keep_mask = np.zeros(scores.shape[0], bool)
    for g in np.unique(groups):
        cur = np.nonzero(groups == g)[0]
        k = native.nms(boxes[cur], scores[cur], thr)
        keep_mask[cur[k[:max_keep] if max_keep > 0 else k]] = True
    kept = np.nonzero(keep_mask)[0]
    return kept[native.argsort_desc_stable(scores[kept])].astype(np.int64)


def nms(boxes, scores, iou_threshold: float, groups=None, max_keep: int = 0) -> np.ndarray:
    """Kept indices in visiting order. groups: per-box group (vanilla batched NMS: independent NMS per group, union
    in (score desc, index asc) order); max_keep > 0 keeps at most that many boxes per group (the first ones visited)."""
    b = np.ascontiguousarray(boxes, F).reshape(-1, 4)
    s = np.ascontiguousarray(scores, F).reshape(-1)
    g = None if groups is None else np.asarray(groups).reshape(-1)
    n = b.shape[0]
    if n == 0:
        return np.empty(0, np.int64)
    thr = float(iou_threshold)
    if not thr >= 0.0 or not np.isfinite(b).all():
        return _dense(b, s, g, thr, max_keep)
    live = (b[:, 2] > b[:, 0]) & (b[:, 3] > b[:, 1])   # a box without positive extent intersects nothing
    i, j = _candidate_pairs(b, live)
    if g is not None:
        same = g[i] == g[j]
        i, j = i[same], j[same]
    sup = _suppresses(b, i, j, thr)
    return _greedy(n, score_order(s), i[sup], j[sup], g, max_keep)


def batched_nms_vanilla(boxes, scores, idxs, iou_threshold: float) -> np.ndarray:
    """oracle.detection.batched_nms_vanilla at any size."""
    return nms(boxes, scores, iou_threshold, groups=np.asarray(idxs))


def batched_nms_coordinate_trick(boxes, scores, idxs, iou_threshold: float) -> np.ndarray:
    """oracle.detection.batched_nms_coordinate_trick at any size: the same fp32 offsets, then one NMS."""
    b = np.asarray(boxes, F).reshape(-1, 4)
    if b.size == 0:
        return np.empty((0,), dtype=np.int64)
    offsets = (np.asarray(idxs).astype(F) * F(b.max() + F(1))).astype(F)
    return nms((b + offsets[:, None]).astype(F), scores, iou_threshold)


def batched_nms(boxes, scores, idxs, iou_threshold: float, device_rule: str = "cpu") -> np.ndarray:
    """oracle.detection.batched_nms (the same strategy rule) at any size."""
    b = np.asarray(boxes, F).reshape(-1, 4)
    if b.size > (4000 if device_rule == "cpu" else 100_000):
        return batched_nms_vanilla(b, scores, idxs, iou_threshold)
    return batched_nms_coordinate_trick(b, scores, idxs, iou_threshold)


"""Seeded inputs shared by the golden-vector generator, the oracle pin tests and the GPU parity
tests. Everything is numpy; sizes are kept small enough for the CPU oracle to finish in seconds."""
from __future__ import annotations

import numpy as np

F = np.float32


def random_boxes(rng, n, extent=512.0, wh=(8.0, 128.0)):
    c = rng.uniform(0, extent, (n, 2)).astype(F)
    s = np.exp(rng.uniform(np.log(wh[0]), np.log(wh[1]), (n, 2))).astype(F)
    return np.concatenate([c - s / 2, c + s / 2], axis=1).astype(F)


def distinct_scores(rng, n):
    return rng.permutation(np.linspace(0, 1, n, dtype=np.float64)).astype(F) if n > 1 else np.array([0.5], F)[:n]


def nms_cases():
    """(name, boxes, scores, iou_threshold) — SURVEY.md §8c list."""
    rng = np.random.default_rng(1234)
    out = []
    for n in (1, 2, 63, 64, 65, 129, 1000, 4507):
        for thr in (0.3, 0.5, 0.7):
            out.append((f"rand_n{n}_t{thr}", random_boxes(rng, n), distinct_scores(rng, n), thr))
    # integer coordinates: IoU lands exactly on thresholds (strict '>' keeps at equality)
    ib = np.array([[0, 0, 10, 10], [0, 0, 10, 10], [5, 0, 15, 10], [0, 5, 10, 15], [0, 0, 20, 10], [0, 0, 10, 30]], F)
    isc = np.array([0.9, 0.8, 0.7, 0.6, 0.5, 0.4], F)
    for thr in (0.3, 1.0 / 3.0, 0.33333334, 0.5, 0.7, 1.0, 0.0):
        out.append((f"integer_t{thr!r}", ib, isc, thr))
    # all-equal scores: stable order, lower index wins
    b = random_boxes(rng, 500, extent=128.0)
    out.append(("equal_scores", b, np.full(500, 0.5, F), 0.5))
    # tie-heavy: scores quantised to 1/256
    b = random_boxes(rng, 3000, extent=256.0)
    out.append(("tie_heavy", b, (np.floor(rng.uniform(0, 1, 3000) * 256) / 256).astype(F), 0.5))
    # zero-area duplicates: 0/0 -> NaN IoU -> kept
    z = np.array([[5, 5, 5, 5]] * 4 + [[1, 1, 9, 9], [1, 1, 9, 9]], F)
    out.append(("zero_area", z, np.array([0.9, 0.8, 0.7, 0.6, 0.5, 0.4], F), 0.5))
    # NaN score sorts first; negative and signed-zero scores
    b = random_boxes(rng, 64, extent=64.0)
    s = distinct_scores(rng, 64) - F(0.5)
    s[7] = np.nan; s[20] = np.nan; s[3] = 0.0; s[4] = -0.0
    out.append(("nan_scores", b, s.astype(F), 0.4))
    # dense cluster: heavy suppression chains across 64-box blocks
    b = random_boxes(rng, 2000, extent=96.0, wh=(32.0, 64.0))
    out.append(("dense_cluster", b, distinct_scores(rng, 2000), 0.5))
    return out


def batched_nms_cases():
    """(name, boxes, scores, idxs, iou_threshold)."""
    rng = np.random.default_rng(4321)
    out = []
    for ncls in (1, 5, 80):
        n = 2500
        out.append((f"c{ncls}", random_boxes(rng, n, extent=300.0), distinct_scores(rng, n),
                    rng.integers(0, ncls, n).astype(np.int64), 0.5))
    n = 1200
    out.append(("levels_t0.7", random_boxes(rng, n, extent=200.0), distinct_scores(rng, n),
                np.sort(rng.integers(0, 5, n)).astype(np.int64), 0.7))
    out.append(("tiny", random_boxes(rng, 3, extent=20.0), distinct_scores(rng, 3), np.array([2, 0, 2], np.int64), 0.3))
    return out


NMS_FAMILIES = ("random", "chain", "cluster", "ties", "zero_area")


def nms_family(family, n, thr, seed=0):
    """(boxes [n, 4], scores [n]) of one NMS input family, seeded by (family, n, seed):
    random     boxes spread so that most are disjoint, distinct scores;
    chain      suppression chains: link k overlaps k - 1 above thr and k - 2 at most at thr, scores falling along the
               chain, so keep / remove alternate. The first chain runs through min(n, 1024) consecutive score ranks (the
               fixed-point sweep's worst case, n rounds); the others are interleaved in score order, so that every link
               crosses 64-box blocks of the sorted order;
    cluster    a dense cluster in which every box overlaps dozens of others;
    ties       scores quantised to 1/64 around 0, with NaN, +0 and -0 among them;
    zero_area  random boxes with exact duplicates, zero-area boxes and zero-area duplicates (0/0 IoU)."""
    rng = np.random.default_rng([NMS_FAMILIES.index(family), n, seed])
    if family == "random":
        return random_boxes(rng, n, extent=16.0 * np.sqrt(n) + 64.0), distinct_scores(rng, n)
    if family == "cluster":
        return random_boxes(rng, n, extent=10.0 * np.sqrt(n) + 48.0, wh=(24.0, 48.0)), distinct_scores(rng, n)
    if family == "ties":
        b = random_boxes(rng, n, extent=8.0 * np.sqrt(n) + 64.0)
        s = (np.floor(rng.uniform(-1, 1, n) * 64) / 64).astype(F)
        s[rng.integers(0, n, max(1, n // 50))] = np.nan
        s[rng.integers(0, n, max(1, n // 50))] = 0.0
        s[rng.integers(0, n, max(1, n // 50))] = -0.0
        return b, s
    if family == "zero_area":
        b = random_boxes(rng, n, extent=12.0 * np.sqrt(n) + 64.0)
        q = rng.permutation(n)
        k = n // 6
        b[q[:k]] = b[q[k:2 * k]]                                            # exact duplicates: IoU 1
        b[q[2 * k:3 * k], 2] = b[q[2 * k:3 * k], 0]                         # zero width
        z = q[3 * k:3 * k + k // 2]
        b[z] = np.repeat(np.array([[7.0, 7.0, 7.0, 7.0]], F), len(z), axis=0)   # zero-area duplicates: NaN IoU
        return b.astype(F), distinct_scores(rng, n)
    assert family == "chain", family
    # link step d: IoU(d) = (w - d) / (w + d) > t >= IoU(2 d) for d = 3/4 of the step at which IoU == t
    w = 16.0
    t = min(max(float(thr), 0.0), 0.9)
    d = 0.75 * w * (1.0 - t) / (1.0 + t)
    first = min(n, 1024)
    rest = n - first
    nchains = max(1, min(64, rest // 16)) if rest else 0
    b = np.zeros((n, 4), F)
    rank = np.zeros(n, np.int64)
    b[:first, 0] = np.arange(first) * d
    b[:first, 1] = 0.0
    rank[:first] = np.arange(first)
    if rest:
        c = np.arange(rest) % nchains                                       # chain of box first + i
        k = np.arange(rest) // nchains                                      # position along it
        b[first:, 0] = k * d
        b[first:, 1] = 2.0 * w * (c + 1)
        rank[first:] = first + np.arange(rest)                              # chains interleaved in score order
    b[:, 2] = b[:, 0] + w
    b[:, 3] = b[:, 1] + w
    perm = rng.permutation(n)                                               # storage order unrelated to score order
    scores = (1.0 - (rank.astype(np.float64) + 1.0) / (n + 1.0)).astype(F)
    return b[perm], scores[perm]


ROI_GOLDEN_CHANNELS = [0, 13, 39]


def roi_align_cases():
    """(name, input[N,C,H,W], rois[K,5], spatial_scale, P, sampling_ratio, aligned)."""
    rng = np.random.default_rng(99)
    x = rng.standard_normal((2, 40, 50, 38)).astype(F)
    special = np.array([
        [0, 1.3, 2.2, 30.7, 44.1],     # ordinary
        [1, -5, -5, 3, 3],             # partially outside (negative)
        [0, 30, 40, 60, 70],           # partially outside (beyond the map)
        [1, 10, 10, 10.2, 10.3],       # tiny (<1 px -> clamped to 1 when not aligned)
        [0, -20, -20, -10, -10],       # fully outside -> zeros
        [1, 0, 0, 38, 50],             # whole map
        [0, 37, 49, 38, 50],           # exactly on the last row / column
        [1, 5, 5, 5, 5],               # zero size
        [0, 0, 0, 152, 200],           # larger than the map (scale 0.25 case covers the map exactly)
        [1, 12.5, 7.25, 13.0, 48.75],  # extreme aspect
    ], F)
    rand = np.concatenate([rng.integers(0, 2, (30, 1)).astype(F), random_boxes(rng, 30, extent=45.0, wh=(2.0, 40.0))], axis=1)
    rois = np.concatenate([special, rand], axis=0).astype(F)
    out = []
    for P in (7, 14):
        for sr in (2, 0, 3):
            for aligned in (False, True):
                for scale in (1.0, 0.25):
                    out.append((f"P{P}_sr{sr}_al{int(aligned)}_s{scale}", x, rois, scale, P, sr, aligned))
    return out


def pyramid(rng, n_img, channels, image_hw):
    """FPN-like pyramid for an image padded to a multiple of 32: strides 4, 8, 16, 32."""
    h, w = image_hw
    return [rng.standard_normal((n_img, channels, h // s, w // s)).astype(F) for s in (4, 8, 16, 32)]


def stress_rois(rng, n, image_hw, side=(16.0, 512.0), aspect=0.7):
    """BASELINE stress distribution: sqrt(area) log-uniform, aspect exp(U[-a,a]), uniform position."""
    h, w = image_hw
    s = np.exp(rng.uniform(np.log(side[0]), np.log(side[1]), n))
    a = np.exp(rng.uniform(-aspect, aspect, n))
    bw, bh = s * np.sqrt(a), s / np.sqrt(a)
    cx, cy = rng.uniform(0, w, n), rng.uniform(0, h, n)
    b = np.stack([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2], axis=1)
    b[:, 0::2] = np.clip(b[:, 0::2], 0, w)
    b[:, 1::2] = np.clip(b[:, 1::2], 0, h)
    return b.astype(F)


def multiscale_case(n_img=2, channels=24, image_hw=(512, 640), rois_per_img=150, seed=7):
    rng = np.random.default_rng(seed)
    feats = pyramid(rng, n_img, channels, image_hw)
    boxes = [stress_rois(rng, rois_per_img, image_hw, side=(8.0, 1000.0)) for _ in range(n_img)]
    return feats, boxes, [image_hw] * n_img


RPN_SIZES = ((32,), (64,), (128,), (256,), (512,))
RPN_RATIOS = ((0.5, 1.0, 2.0),) * 5


def rpn_case(n_img=2, image_hw=(224, 288), padded_hw=(224, 288), seed=11, logit_scale=2.0):
    """RPN head outputs for a small pyramid: objectness [N,3,H,W], deltas [N,12,H,W] per level."""
    rng = np.random.default_rng(seed)
    ph, pw = padded_hw
    grids = [(ph // s, pw // s) for s in (4, 8, 16, 32)] + [(-(-ph // 64), -(-pw // 64))]
    obj = [(rng.standard_normal((n_img, 3, gh, gw)) * logit_scale).astype(F) for gh, gw in grids]
    dlt = [(rng.standard_normal((n_img, 12, gh, gw)) * 0.5).astype(F) for gh, gw in grids]
    for d in dlt:  # a few deltas beyond the exp clip
        d.reshape(-1)[:: 97] *= 12
    image_sizes = [(image_hw[0], image_hw[1])] + [(image_hw[0] - 17, image_hw[1] - 40)] * (n_img - 1)
    return obj, dlt, grids, image_sizes, padded_hw


def det_case(n_img=2, props=300, num_classes=3, image_hw=(224, 288), seed=21):
    rng = np.random.default_rng(seed)
    proposals = [stress_rois(rng, props - 13 * i, image_hw, side=(8.0, 200.0)) for i in range(n_img)]
    total = sum(len(p) for p in proposals)
    logits = (rng.standard_normal((total, num_classes)) * 2.0).astype(F)
    reg = (rng.standard_normal((total, 4 * num_classes)) * 1.5).astype(F)
    reg.reshape(-1)[:: 53] *= 20
    return logits, reg, proposals, [image_hw] * n_img


def crop_case(seed=31, hw=(200, 260), channels=3, n=60):
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 256, (hw[0], hw[1], channels), dtype=np.uint8)
    if channels == 1:
        img = img[..., 0]
    b = stress_rois(rng, n, hw, side=(4.0, 150.0))
    # .5 fractions (half-to-even), boxes past the edge, zero-width after rounding, negative starts
    b[0] = [10.5, 11.5, 20.5, 31.5]
    b[1] = [12.5, 0.5, 13.49, 40.5]
    b[2] = [250.2, 190.7, 300.0, 260.0]
    b[3] = [30.4, 30.4, 30.45, 80.0]
    b[4] = [-3.2, -0.4, 25.0, 18.6]
    b[5] = [0.49999997, 2.5, 100.50001, 3.5]
    scores = rng.uniform(0, 1, n).astype(F)
    scores[6] = 0.5  # not > 0.5
    labels = rng.integers(1, 3, n).astype(np.int64)
    return img, b.astype(F), scores, labels


def box_rel_err(a, b):
    """max |a-b| relative to each box's own coordinate scale (floor 1 px): x1 = ctr - w/2 cancels,
    so a 1-ulp exp() difference in w shows up relative to the box extent, not to x1 itself."""
    a = np.asarray(a, np.float64).reshape(-1, 4)
    b = np.asarray(b, np.float64).reshape(-1, 4)
    if a.size == 0:
        return 0.0
    denom = np.maximum(np.abs(b).max(axis=1, keepdims=True), 1.0)
    return float(np.max(np.abs(a - b) / denom))


def paste_case(seed=41, r=14, image_hw=(120, 150), side=28):
    """Mask probabilities + detection boxes for paste_masks_in_image: ordinary, tiny, sub-pixel, whole
    image, past the right/bottom edge, negative start (all intersect the image, as detections do after
    clipping — the reference itself fails on a box entirely outside the image)."""
    rng = np.random.default_rng(seed)
    h, w = image_hw
    masks = rng.random((r, 1, side, side)).astype(F)
    c = rng.uniform(0, [w, h], (r, 2)); wh = np.exp(rng.uniform(np.log(2), np.log(110), (r, 2)))
    b = np.concatenate([c - wh / 2, c + wh / 2], 1).astype(F)
    b[0] = [5, 5, 5, 5]
    b[1] = [0, 0, w, h]
    b[2] = [w - 3, h - 3, w + 40, h + 50]
    b[3] = [10.6, 20.4, 10.9, 20.7]
    b[4] = [-30, -12, 40, 33]
    b[5] = [20.5, 30.5, 90.49, 100.51]
    return masks, b, image_hw


def transform_case(seed=51):
    """uint8 HWC images of different sizes for the input transform (min_size 96, max_size 150: the
    second image is limited by max_size)."""
    rng = np.random.default_rng(seed)
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in ((60, 84), (131, 58), (77, 77))]
    return imgs, 96, 150, [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]

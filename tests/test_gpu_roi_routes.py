"""Every kernel route of mb_multiscale_roi_align (miso_b200/csrc/roi_align.cu, roi_align_tma.cu) and the RoIAlign
backward (train.cu) against references, with the route each case takes asserted by kernel name.

The host picks one of seven forward kernels from the memory format, sampling_ratio, pooled size, channel count, map
pointer alignment, the workspace and a footprint-versus-pyramid heuristic. Each case below forces one route and checks
from a torch.profiler trace that the intended kernel ran, so a change of the dispatch cannot move a case elsewhere.

* exact mode must equal the CPU oracle (oracle/c/oracle_kernels.c) bit for bit;
* fast mode is compared per element with an fp64-accumulating reference that takes its sample positions, taps and
  weights in fp32 exactly as the oracle does: |got - ref| <= 32 * 2^-24 * A, where A is the same reference over |x|.
  A wrong tap, weight or sample count errs by O(A);
* a sample outside [-1, size] is skipped, not multiplied by a zero weight, so Inf / NaN features at the pixels a
  kernel might address for such a sample must not reach a bin the oracle computes as finite;
* the backward is a scatter of grad * w / count; it is compared with an fp64 scatter of the same fp32 weights,
  within (n + 3) * 2^-24 * B per element (n contributions, B the scatter of |grad|).
"""
import fnmatch
import re

import numpy as np
import pytest
import torch

from oracle import detection as D
from oracle import native
from tests import cases
from tests.test_gpu_roi_tma import mixed_rois

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F = np.float32
ULP = 2.0 ** -24


@pytest.fixture(scope="module")
def ops():
    from miso_b200 import ops as o
    o._lib.load()
    return o


def cu(a, dev=DEV):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def nhwc(x, dev=DEV, offset=0):
    """Channels-last device copy of x [N, C, H, W]; its data pointer sits `offset` floats past a 256-byte boundary."""
    n, c, h, w = x.shape
    buf = torch.empty(n * h * w * c + offset, dtype=torch.float32, device=dev)
    t = buf[offset:].view(n, h, w, c).permute(0, 3, 1, 2)
    t.copy_(cu(x, dev))
    assert t.is_contiguous(memory_format=torch.channels_last) and t.data_ptr() % 16 == 4 * offset
    return t


def device_maps(xs, layout, dev=DEV):
    """layout: "nchw", "nhwc", or "nhwc+4" (channels-last, data pointer 4 bytes off a 16-byte boundary)."""
    if layout == "nchw":
        return [cu(x, dev) for x in xs]
    return [nhwc(x, dev, offset=1 if layout == "nhwc+4" else 0) for x in xs]


# ---------------------------------------------------------------------------------------------------------------------
# route probe
# ---------------------------------------------------------------------------------------------------------------------
_KERNEL = re.compile(r"mb::(k_\w+(?:<[^>]*>)?)")


def launched(fn):
    """Runs fn() under torch.profiler; returns (its result, sorted names of the library's kernels it launched)."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names, "torch.profiler recorded no CUDA kernel for a call that launches one: the route cannot be checked"
    ours = sorted({m.group(1).replace(" ", "") for m in map(_KERNEL.search, names) if m})
    return res, ours


def assert_route(got, patterns, exact):
    want = [p.format(e="true" if exact else "false") for p in patterns]
    assert len(got) == len(want) and all(any(fnmatch.fnmatchcase(g, w) for g in got) for w in want), (got, want)


def _offset_workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 256) + 16, dtype=torch.uint8, device=device)[4:]


def pool(ops, monkeypatch, feats, rois, scales, thresholds, P, sr, aligned, exact, how, box_counts=None):
    """ops._roi_align_launch under the route options `how`: force ("tma" / "gather"), use_workspace (False: none),
    ws_offset (a workspace 4 bytes off a 16-byte boundary). Returns (out, levels, kernels, TMA launches)."""
    lib = ops._lib.load()
    with monkeypatch.context() as m:
        if how.get("ws_offset"):
            m.setattr(ops, "_workspace", _offset_workspace)
        n0 = lib.mb_roi_align_tma_launches()
        (out, levels), kernels = launched(lambda: ops._roi_align_launch(
            feats, rois, scales, thresholds, P, sr, aligned, exact, return_levels=True,
            use_workspace=how.get("use_workspace", True), force_gather=how.get("force", False), box_counts=box_counts))
        return out, levels, kernels, lib.mb_roi_align_tma_launches() - n0


# ---------------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------------
def _geometry(r, scale, P, sr, aligned):
    """roi_align's per-RoI quantities in fp32, one rounding per operation (oracle_roi_align)."""
    off = F(0.5) if aligned else F(0.0)
    s = F(scale)
    sw, sh, ew, eh = (F(r[i]) * s - off for i in (1, 2, 3, 4))
    rw, rh = ew - sw, eh - sh
    if not aligned:
        rw, rh = max(rw, F(1)), max(rh, F(1))
    bh, bw = rh / F(P[0]), rw / F(P[1])
    gh = sr if sr > 0 else int(np.ceil(rh / F(P[0])))
    gw = sr if sr > 0 else int(np.ceil(rw / F(P[1])))
    return sh, sw, bh, bw, gh, gw, max(gh * gw, 1)


def _taps(start, bin_size, P, grid, size):
    """Sample taps along one axis, [P, grid] each: (lo, hi, l, h, valid), fp32 as in bilinear_interpolate."""
    p = np.arange(P, dtype=F)[:, None]
    i = np.arange(max(grid, 0), dtype=F)[None, :]
    v = (start + p * bin_size) + ((i + F(0.5)) * bin_size) / F(max(grid, 1))
    valid = ~((v < F(-1)) | (v > F(size)))
    v = np.where(v <= F(0), F(0), v).astype(F)
    lo = np.minimum(v, F(size)).astype(np.int64)
    edge = lo >= size - 1
    lo = np.where(edge, size - 1, lo)
    v = np.where(edge, lo.astype(F), v).astype(F)
    hi = np.where(edge, lo, lo + 1)
    l = (v - lo.astype(F)).astype(F)
    return lo, hi, l, (F(1) - l).astype(F), valid


def _bilinear_terms(r, scale, P, sr, aligned, H, W):
    """The four (weight [PH, gh, PW, gw] fp32, row index, column index) corner terms, the valid-sample mask, count."""
    sh, sw, bh, bw, gh, gw, count = _geometry(r, scale, P, sr, aligned)
    ylo, yhi, ly, hy, vy = _taps(sh, bh, P[0], gh, H)
    xlo, xhi, lx, hx, vx = _taps(sw, bw, P[1], gw, W)
    Y, X = (lambda a: a[:, :, None, None]), (lambda a: a[None, None, :, :])
    terms = [(Y(hy) * X(hx), Y(ylo), X(xlo)), (Y(hy) * X(lx), Y(ylo), X(xhi)),
             (Y(ly) * X(hx), Y(yhi), X(xlo)), (Y(ly) * X(lx), Y(yhi), X(xhi))]
    return terms, Y(vy) & X(vx), count


def roi_align_fp64(x, rois, scale, P, sr, aligned):
    """(reference, magnitude) [K, C, PH, PW] in fp64: the oracle's fp32 taps and weights, products and sums in fp64;
    the magnitude is the same sum over |x|."""
    n, c, h, w = x.shape
    xs = (x.astype(np.float64), np.abs(x.astype(np.float64)))
    out = np.zeros((2, len(rois), c, P[0], P[1]))
    for k, r in enumerate(rois):
        b = int(r[0])
        if not 0 <= b < n:
            continue
        terms, mask, count = _bilinear_terms(r, scale, P, sr, aligned, h, w)
        for j, plane in enumerate(xs):
            acc = sum(np.where(mask, wt.astype(np.float64) * plane[b][:, yi, xi], 0.0) for wt, yi, xi in terms)
            out[j, k] = acc.sum(axis=(2, 4)) / count
    return out[0], out[1]


def references(xs, rois, levels, scales, P, sr, aligned, fp64=True):
    """Oracle output and (if fp64) the fp64 reference and magnitude for [K, 5] RoIs assigned to `levels`."""
    c = xs[0].shape[1]
    ora = np.zeros((len(rois), c) + tuple(P), F)
    ref, mag = np.zeros(ora.shape), np.zeros(ora.shape)
    for lvl, (x, s) in enumerate(zip(xs, scales)):
        idx = np.nonzero(levels == lvl)[0]
        if len(idx):
            ora[idx] = native.roi_align(x, rois[idx], s, P[0], P[1], sr, aligned)
            if fp64:
                ref[idx], mag[idx] = roi_align_fp64(x, rois[idx], s, P, sr, aligned)
    return ora, ref, mag


def assert_within(got, ref, mag, ulps=32):
    err = np.abs(got.astype(np.float64) - ref)
    bad = ~(err <= ulps * ULP * mag)
    assert not bad.any(), (f"{int(bad.sum())} of {bad.size} elements beyond {ulps} ulp of the summed magnitude; worst "
                           f"error {err[bad].max():.3e} where the bound is {(ulps * ULP * mag)[bad].min():.3e}")


# ---------------------------------------------------------------------------------------------------------------------
# forward route matrix, one level
# ---------------------------------------------------------------------------------------------------------------------
NHWC4D = ["k_roi_align_nhwc4d<{e},*>"]
TRANSPOSE = ["k_nchw_to_nhwc", "k_roi_align_nhwc4d<{e},*>"]
TMA = ["k_roi_geom", "k_roi_align_tma<{e}>"]
TMA_NCHW = ["k_nchw_to_nhwc", "k_roi_geom", "k_roi_align_tma<{e}>"]
SR2 = ["k_roi_align_sr2<{e}>"]
GATHER = ["k_roi_align_nhwc<{e}>"]
STAGED_SR2 = ["k_roi_align_staged<{e},true>"]
STAGED = ["k_roi_align_staged<{e},false>"]
DIRECT = ["k_roi_align_direct"]
NO_WS = {"use_workspace": False}

# (layout, channels, map width, pooled size, sampling_ratio, aligned, route options, kernels)
ROUTES = {
    "nhwc4d-256": ("nhwc", 256, 76, (7, 7), 2, False, {}, NHWC4D),
    "nhwc4d-136-aligned": ("nhwc", 136, 76, (14, 14), 2, True, {}, NHWC4D),
    "nhwc4d-36-5x9": ("nhwc", 36, 75, (5, 9), 2, False, {}, NHWC4D),
    "transpose-256": ("nchw", 256, 76, (7, 7), 2, False, {}, TRANSPOSE),
    "transpose-40-16x11-aligned": ("nchw", 40, 75, (16, 11), 2, True, {}, TRANSPOSE),
    "tma-256": ("nhwc", 256, 76, (7, 7), 2, False, {"force": "tma"}, TMA),
    "tma-36-16x9": ("nhwc", 36, 75, (16, 9), 2, False, {"force": "tma"}, TMA),
    "tma-from-nchw-128": ("nchw", 128, 76, (7, 7), 2, False, {"force": "tma"}, TMA_NCHW),
    "sr2-vec4-256": ("nchw", 256, 76, (7, 7), 2, False, NO_WS, SR2),
    "sr2-scalar-33-aligned": ("nchw", 33, 75, (14, 14), 2, True, NO_WS, SR2),
    "sr2-ws-offset-64-5x9": ("nchw", 64, 76, (5, 9), 2, False, {"ws_offset": True}, SR2),
    "gather-c3": ("nhwc", 3, 76, (7, 7), 2, False, {}, GATHER),
    "gather-c5-aligned": ("nhwc", 5, 75, (14, 14), 2, True, {}, GATHER),
    "gather-c33-5x9": ("nhwc", 33, 76, (5, 9), 2, False, {}, GATHER),
    "gather-c255": ("nhwc", 255, 76, (7, 7), 2, False, {}, GATHER),
    "gather-misaligned-64": ("nhwc+4", 64, 76, (7, 7), 2, False, {}, GATHER),
    "gather-misaligned-tma-36": ("nhwc+4", 36, 76, (7, 7), 2, False, {"force": "tma"}, GATHER),
    "staged-sr2-17x9": ("nchw", 40, 76, (17, 9), 2, False, {}, STAGED_SR2),
    "staged-sr2-from-nhwc-20x20": ("nhwc", 36, 75, (20, 20), 2, True, {}, STAGED_SR2),
    "staged-sr2-512-bins": ("nchw", 33, 76, (32, 16), 2, False, {}, STAGED_SR2),
    "direct-sr2-544-bins": ("nchw", 40, 76, (32, 17), 2, False, {}, DIRECT),
    "direct-sr2-66-samples": ("nchw", 8, 75, (33, 15), 2, False, {}, DIRECT),
    "staged-sr1-64-samples-512-bins": ("nchw", 40, 76, (64, 8), 1, False, {}, STAGED),
    "direct-sr1-65-samples": ("nchw", 40, 76, (65, 7), 1, False, {}, DIRECT),
    "direct-sr1-513-bins": ("nchw", 40, 76, (19, 27), 1, False, {}, DIRECT),
    "staged-sr8-64-samples": ("nchw", 40, 76, (8, 8), 8, False, {}, STAGED),
    "direct-sr13-65-samples": ("nchw", 40, 75, (5, 5), 13, False, {}, DIRECT),
    "staged-sr3-aligned": ("nchw", 40, 76, (7, 7), 3, True, {}, STAGED),
    "direct-adaptive": ("nchw", 40, 76, (7, 7), 0, False, {}, DIRECT),
}


@pytest.mark.parametrize("name", list(ROUTES))
def test_route_matches_references(ops, monkeypatch, name):
    layout, c, w, P, sr, aligned, how, kernels = ROUTES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    n, h = 2, 60
    x = rng.standard_normal((n, c, h, w)).astype(F)
    rois = mixed_rois(rng, n, 600, (h * 4, w * 4))
    feats, tr = device_maps([x], layout), cu(rois)
    pick = np.sort(rng.choice(len(rois), 48, replace=False))
    zeros = np.zeros(len(pick), np.int64)
    ora, ref, mag = references([x], rois[pick], zeros, [0.25], P, sr, aligned, fp64=sr > 0)
    for exact in (True, False):
        out, levels, got_kernels, tma = pool(ops, monkeypatch, feats, tr, [0.25], [], P, sr, aligned, exact, how)
        assert_route(got_kernels, kernels, exact)
        assert tma == (1 if "k_roi_geom" in kernels else 0)
        assert not levels.any()
        got = out[torch.from_numpy(pick).to(DEV)].cpu().numpy()
        if exact or sr <= 0:    # k_roi_align_direct has no fast variant: adaptive sampling is exact in both modes
            assert np.array_equal(got, ora), f"{name}, exact={exact}"
        else:
            assert_within(got, ref, mag)


# ---------------------------------------------------------------------------------------------------------------------
# multi-level pyramid, [N, R, 4] + box_counts with dead rows and an empty image, levels_out
# ---------------------------------------------------------------------------------------------------------------------
# (layout, channels, pooled size, sampling_ratio, route options, kernels)
PER_IMAGE_ROUTES = {
    "nhwc4d": ("nhwc", 36, (7, 7), 2, {}, NHWC4D),
    "transpose": ("nchw", 36, (7, 7), 2, {}, TRANSPOSE),
    "tma": ("nhwc", 36, (14, 14), 2, {"force": "tma"}, TMA),
    "tma-from-nchw": ("nchw", 36, (7, 7), 2, {"force": "tma"}, TMA_NCHW),
    "sr2": ("nchw", 33, (14, 14), 2, NO_WS, SR2),
    "sr2-ws-offset": ("nchw", 36, (7, 7), 2, {"ws_offset": True}, SR2),
    "gather-c35": ("nhwc", 35, (7, 7), 2, {}, GATHER),
    "gather-misaligned": ("nhwc+4", 36, (14, 14), 2, {}, GATHER),
    "staged-sr2": ("nchw", 36, (17, 17), 2, {}, STAGED_SR2),
    "staged-sr3": ("nchw", 36, (7, 7), 3, {}, STAGED),
    "direct-adaptive": ("nchw", 36, (7, 7), 0, {}, DIRECT),
}


@pytest.mark.parametrize("name", list(PER_IMAGE_ROUTES))
def test_route_multiscale_per_image_layout(ops, monkeypatch, name):
    layout, c, P, sr, how, kernels = PER_IMAGE_ROUTES[name]
    rng = np.random.default_rng(sum(map(ord, name)) + 1)
    n, R, hw = 3, 200, (416, 544)
    xs = cases.pyramid(rng, n, c, hw)
    boxes = np.stack([mixed_rois(rng, 1, R, hw)[:R, 1:] for _ in range(n)]).astype(F)
    counts = np.array([R, 117, 0], np.int32)
    scales, k_min, k_max = D.infer_scales([x.shape[-2:] for x in xs], [hw] * n)
    thresholds = ops.level_thresholds(k_min, k_max)
    levels_ref = D.map_levels(boxes.reshape(-1, 4), k_min, k_max)
    assert set(levels_ref.tolist()) == {0, 1, 2, 3}
    live = np.concatenate([np.arange(counts[i]) + i * R for i in range(n)])
    pick = np.sort(rng.choice(live, 40, replace=False))
    rois = np.concatenate([(pick // R)[:, None].astype(F), boxes.reshape(-1, 4)[pick]], 1)
    ora, ref, mag = references(xs, rois, levels_ref[pick], scales, P, sr, False, fp64=sr > 0)
    feats, tb, tc = device_maps(xs, layout), cu(boxes), cu(counts)
    for exact in (True, False):
        out, levels, got_kernels, _ = pool(ops, monkeypatch, feats, tb, scales, thresholds, P, sr, False, exact, how,
                                           box_counts=tc)
        assert_route(got_kernels, kernels, exact)
        assert np.array_equal(levels.cpu().numpy(), levels_ref)
        o = out.cpu().numpy()
        assert not o.reshape(n, R, -1)[1, 117:].any() and not o.reshape(n, R, -1)[2].any()   # dead rows: zeros
        if exact or sr <= 0:
            assert np.array_equal(o[pick], ora), f"{name}, exact={exact}"
        else:
            assert_within(o[pick], ref, mag)


# ---------------------------------------------------------------------------------------------------------------------
# non-finite features where a kernel could address samples outside the map
# ---------------------------------------------------------------------------------------------------------------------
NONFINITE_ROUTES = {
    "nhwc4d": ("nhwc", 36, (7, 7), 2, {}, NHWC4D),
    "transpose": ("nchw", 36, (7, 7), 2, {}, TRANSPOSE),
    "tma": ("nhwc", 36, (7, 7), 2, {"force": "tma"}, TMA),
    "sr2": ("nchw", 36, (7, 7), 2, NO_WS, SR2),
    "gather-c35": ("nhwc", 35, (7, 7), 2, {}, GATHER),
    "gather-misaligned": ("nhwc+4", 36, (7, 7), 2, {}, GATHER),
    "staged-sr2": ("nchw", 36, (18, 17), 2, {}, STAGED_SR2),
    "staged-sr3": ("nchw", 36, (7, 7), 3, {}, STAGED),
    "direct": ("nchw", 36, (33, 9), 2, {}, DIRECT),
}


def _footprint_origins(rois, P, sr, H, W):
    """(row, column) of the first valid tap of every RoI, with the column also rounded down to a multiple of 4."""
    out = set()
    for r in rois:
        sh, sw, bh, bw, gh, gw, _ = _geometry(r, 1.0, P, sr, False)
        ylo, _, _, _, vy = _taps(sh, bh, P[0], gh, H)
        xlo, _, _, _, vx = _taps(sw, bw, P[1], gw, W)
        if vy.any() and vx.any():
            y0, x0 = int(ylo[vy].min()), int(xlo[vx].min())
            out |= {(y0, x0), (y0, x0 & ~3)}
    return out


@pytest.mark.parametrize("width", [44, 42])
@pytest.mark.parametrize("name", list(NONFINITE_ROUTES))
def test_route_skips_samples_outside_the_map(ops, monkeypatch, name, width):
    """Inf / NaN at map pixel (0, 0) and at the footprint origins of RoIs partly outside the map: every route must
    equal the oracle, NaN for NaN, and the bins the oracle computes as finite must be finite."""
    layout, c, P, sr, how, kernels = NONFINITE_ROUTES[name]
    rng = np.random.default_rng(width)
    H, W = 40, width
    rois = np.array([[0, -30, 10, 20, 30], [0, 8, -25, 30, 18], [0, 30, 5, W + 30, 25], [0, 5, 28, 25, H + 20],
                     [0, -20, -20, 15, 15], [0, W - 12, H - 10, W + 25, H + 30], [0, 10, 10, 30, 30],
                     [0, -9, 3, 9, 37], [0, 2, -7, 40, 7], [0, 21, 30, 39, H + 6], [0, W - 5, 1, W + 9, 39]], F)
    x = rng.standard_normal((1, c, H, W)).astype(F)
    x[0, :, 0, 0] = np.inf
    x[0, 5, 0, 0] = np.nan
    for y0, x0 in _footprint_origins(rois, P, sr, H, W):
        if (y0, x0) != (0, 0):
            x[0, :, y0, x0] = -np.inf
            x[0, 7, y0, x0] = np.nan
    ref = native.roi_align(x, rois, 1.0, P[0], P[1], sr, False)
    # the case must probe something: finite oracle bins that have a sample outside the map
    probe = np.zeros(ref.shape, bool)
    for k, r in enumerate(rois):
        _, mask, _ = _bilinear_terms(r, 1.0, P, sr, False, H, W)
        probe[k] = ~mask.all(axis=(1, 3))[None]
    probe &= np.isfinite(ref)
    assert probe.sum() >= 100
    feats = device_maps([x], layout)
    for exact in (True, False):
        out, _, got_kernels, _ = pool(ops, monkeypatch, feats, cu(rois), [1.0], [], P, sr, False, exact, how)
        assert_route(got_kernels, kernels, exact)
        got = out.cpu().numpy()
        assert np.isfinite(got[probe]).all(), f"{name}: {int((~np.isfinite(got[probe])).sum())} bins not finite"
        if exact:
            assert np.array_equal(got, ref, equal_nan=True), name
        else:
            assert np.array_equal(np.isfinite(got), np.isfinite(ref))


# ---------------------------------------------------------------------------------------------------------------------
# backward
# ---------------------------------------------------------------------------------------------------------------------
def roi_align_backward_fp64(grad, rois, scale, P, sr, aligned, shape, chans):
    """fp64 scatter of grad * w / count with the oracle's fp32 taps and weights, for the channels `chans`:
    (gradient, same scatter of |grad|, contributions per element), [N, len(chans), H, W] / [N, H, W]."""
    n, _, h, w = shape
    idx, vals = [], []
    for k, r in enumerate(rois):
        b = int(r[0])
        if not 0 <= b < n:
            continue
        terms, mask, count = _bilinear_terms(r, scale, P, sr, aligned, h, w)
        g = grad[k][chans].astype(np.float64)[:, :, None, :, None]       # [c, PH, 1, PW, 1]
        for wt, yi, xi in terms:
            flat = np.broadcast_to(b * h * w + yi * w + xi, mask.shape)[mask]
            idx.append(flat)
            vals.append((g * wt.astype(np.float64) / count)[:, mask])
    idx, vals = np.concatenate(idx), np.concatenate(vals, axis=1)
    size = n * h * w
    ref = np.stack([np.bincount(idx, vals[j], size) for j in range(len(chans))])
    mag = np.stack([np.bincount(idx, np.abs(vals[j]), size) for j in range(len(chans))])
    cnt = np.bincount(idx, minlength=size)
    unflat = lambda a: a.reshape(-1, n, h, w).swapaxes(0, 1)
    return unflat(ref), unflat(mag), cnt.reshape(n, h, w)


def check_backward(ops, grad, rois, scale, P, sr, aligned, shape, chans, dev=DEV):
    got = ops.roi_align_backward(cu(grad, dev), cu(rois, dev), scale, P[0], P[1], *shape, sr, aligned)
    got = got[:, torch.tensor(chans, device=dev)].cpu().numpy().astype(np.float64)
    ref, mag, cnt = roi_align_backward_fp64(grad, rois, scale, P, sr, aligned, shape, chans)
    bound = (cnt[:, None] + 3) * ULP * mag
    bad = ~(np.abs(got - ref) <= bound)
    assert not bad.any(), (f"{int(bad.sum())} gradient elements beyond (n + 3) ulp of the summed magnitude; "
                           f"worst error {np.abs(got - ref)[bad].max():.3e}")
    return cnt


@pytest.mark.parametrize("sr", [2, 0])
@pytest.mark.parametrize("P", [7, 14])
def test_backward_model_scale(ops, P, sr):
    """256 channels on a 200x304 map (an 800x1216 image at stride 4), 512 RoIs; the reference covers the channels at
    the 32-channel chunk boundaries."""
    rng = np.random.default_rng(100 * P + sr)
    shape = (2, 256, 200, 304)
    img = (800, 1216)
    b = np.concatenate([cases.stress_rois(rng, 480, img, side=(4.0, 700.0)),
                        np.repeat(np.array([[100.0, 120.0, 180.0, 230.0]], F), 16, 0),                 # piled up
                        mixed_rois(rng, 1, 16, img)[:16, 1:]])
    rois = np.concatenate([rng.integers(0, 2, (len(b), 1)).astype(F), b], 1).astype(F)
    grad = rng.standard_normal((len(rois), 256, P, P)).astype(F)
    check_backward(ops, grad, rois, 0.25, (P, P), sr, False, shape, [0, 31, 32, 63, 200, 255])


def test_backward_staging_boundary_and_pileups(ops):
    """Clamped RoI footprints of 448, 449 (the largest staged in shared memory) and 450 pixels, as one row, one
    column and a block; hundreds of RoIs piling onto the same pixels."""
    rng = np.random.default_rng(449)
    H = W = 460
    shape = (1, 40, H, W)
    edge = np.float32(H - 0.8)
    # footprint rows = floor(y2) - floor(y1) + 2 (clamped to the map), the same for columns
    foot = [[3.5, edge, 449.5, edge + 0.5], [3.5, edge, 450.5, edge + 0.5], [3.5, edge, 451.5, edge + 0.5],
            [edge, 3.5, edge + 0.5, 450.5], [edge, 3.5, edge + 0.5, 451.5], [50.2, 100.3, 78.9, 113.6]]
    pile = np.repeat(np.array([[200.0, 210.0, 260.0, 240.0]]), 200, 0)
    jitter = np.array([[200.0, 210.0, 260.0, 240.0]]) + rng.uniform(-2, 2, (200, 4))
    b = np.concatenate([np.repeat(np.array(foot), 3, 0), pile, jitter]).astype(F)
    rois = np.concatenate([np.zeros((len(b), 1), F), b], 1)
    for P, sr in ((7, 2), (5, 0)):
        grad = rng.standard_normal((len(rois), 40, P, P)).astype(F)
        cnt = check_backward(ops, grad, rois, 1.0, (P, P), sr, False, shape, list(range(40)))
        assert cnt.max() >= 200                                   # the 200 identical RoIs share their taps


# ---------------------------------------------------------------------------------------------------------------------
# two devices in one process
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_second_device_in_one_process(ops):
    """The library's per-device state (dynamic shared-memory opt-ins, TMA device limits): the same calls on cuda:0,
    then with cuda:1 current and its tensors on cuda:1."""
    lib = ops._lib.load()
    rng = np.random.default_rng(2)
    x = rng.standard_normal((2, 64, 60, 76)).astype(F)
    rois = mixed_rois(rng, 2, 300, (240, 304))
    ref = native.roi_align(x, rois, 0.25, 7, 7, 2, False)
    grad = rng.standard_normal((len(rois), 64, 7, 7)).astype(F)
    for dev in ("cuda:0", "cuda:1"):
        with torch.cuda.device(dev):
            xc, tr = nhwc(x, dev), cu(rois, dev)
            assert np.array_equal(ops.roi_align(xc, tr, 7, 0.25, 2, False).cpu().numpy(), ref), dev
            assert np.array_equal(ops.roi_align(cu(x, dev), tr, 7, 0.25, 2, False).cpu().numpy(), ref), dev
            n0 = lib.mb_roi_align_tma_launches()
            got = ops.roi_align(xc, tr, 7, 0.25, 2, False, force_gather="tma").cpu().numpy()
            assert lib.mb_roi_align_tma_launches() == n0 + 1, dev
            assert np.array_equal(got, ref), dev
            check_backward(ops, grad, rois, 0.25, (7, 7), 2, False, (2, 64, 60, 76), [0, 33, 63], dev=dev)

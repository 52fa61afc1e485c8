"""Every sweep route of the segmented NMS core (miso_b200/csrc/nms_core.cuh) through its three entry points — mb_nms,
mb_rpn_proposals and mb_det_postprocess — with the route each case takes asserted from a torch.profiler trace.

launch_mask_and_sweep picks the sweep from the largest segment a call can have (mb_nms: the box count K in every
mode; RPN: min(pre_nms_top_n, largest level); detection: max_props_per_image):

    largest segment   sweep kernel                     dynamic shared memory
    <= 1024           k_nms_fixpoint (full mask)       -
    1025 - 4096       k_nms_sweep_small                -
    4097 - 6336       k_nms_sweep_wide, 4 tile buffers (T + 64 * nbuf * T) * 8 <= 200 KiB, T = ceil(K / 64)
    6337 - 8448       k_nms_sweep_wide, 3 buffers
    8449 - 12672      k_nms_sweep_wide, 2 buffers
    12673 - 25152     k_nms_sweep_wide, 1 buffer
    > 25152           k_nms_sweep                      (T + 1) * 8

Kept indices are compared bit for bit with the C oracle's greedy NMS or with the sparse reference (tests/nms_ref.py,
pinned to the oracle by tests/test_nms_ref.py); the fused stages are compared with oracle/detection.py as in
test_gpu_stages.py (indices and labels exact, boxes within 1e-5 of the box scale, scores within 1e-6)."""
import dataclasses
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

from oracle import detection as D
from tests import cases
from tests import nms_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Later torch.profiler sessions in a process that ran this module's sessions recorded no kernels (the route probes of
# test_gpu_roi_routes.py, run after this file, saw none). So the module runs in a pytest process of its own: in the
# suite's process, test_module_in_own_process starts it and every other test here is skipped.
OWN_PROCESS = os.environ.get("MB_NMS_ROUTES_OWN_PROCESS") == "1"


@pytest.fixture(autouse=True)
def _in_own_process(request):
    if not OWN_PROCESS and request.node.name != "test_module_in_own_process":
        pytest.skip("runs in the module's own pytest process (test_module_in_own_process)")


def test_module_in_own_process():
    if OWN_PROCESS:
        pytest.skip("this is the module's own process")
    env = dict(os.environ, MB_NMS_ROUTES_OWN_PROCESS="1")
    res = subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "gpu", "-p", "no:cacheprovider", "-rf",
                          os.path.abspath(__file__)], cwd=ROOT, env=env, capture_output=True, text=True, timeout=3000)
    sys.stdout.write(res.stdout[-3000:])
    assert res.returncode == 0, res.stdout[-8000:] + res.stderr[-3000:]

THRESHOLDS = (0.0, 0.5, 0.7, 1.0, -0.25, 0.33333334)
SWEEPS = ("k_nms_fixpoint", "k_nms_sweep_small", "k_nms_sweep_wide", "k_nms_sweep")
BAND_EDGES = (1024, 1025, 4096, 4097, 6336, 6337, 8448, 8449, 12672, 12673, 25152, 25153)


def sweep_route(max_seg, blocks=False):
    """(kernel, tile buffers, dynamic shared-memory bytes) launch_mask_and_sweep picks for a largest segment of
    max_seg boxes; blocks: MB_NMS_SWEEP=blocks."""
    T = -(-max_seg // 64)
    if max_seg <= 1024 and not blocks:
        return "k_nms_fixpoint", 0, 0
    if T <= 64:
        return "k_nms_sweep_small", 0, 0
    for nbuf in (4, 3, 2, 1):
        if (T + 64 * nbuf * T) * 8 <= 200 * 1024:
            return "k_nms_sweep_wide", nbuf, (T + 64 * nbuf * T) * 8
    return "k_nms_sweep", 0, (T + 1) * 8


def test_band_edges_follow_the_shared_memory_budget():
    got = [sweep_route(k)[:2] for k in BAND_EDGES + (140000,)]
    assert got == [("k_nms_fixpoint", 0), ("k_nms_sweep_small", 0), ("k_nms_sweep_small", 0), ("k_nms_sweep_wide", 4),
                   ("k_nms_sweep_wide", 4), ("k_nms_sweep_wide", 3), ("k_nms_sweep_wide", 3), ("k_nms_sweep_wide", 2),
                   ("k_nms_sweep_wide", 2), ("k_nms_sweep_wide", 1), ("k_nms_sweep_wide", 1), ("k_nms_sweep", 0),
                   ("k_nms_sweep", 0)]


def cu(a, dev=DEV):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


@pytest.fixture(scope="module")
def ops():
    from miso_b200 import ops as o
    o._lib.load()
    return o


@pytest.fixture(scope="module")
def det():
    from miso_b200 import detection
    detection._lib.load()
    return detection


# ---------------------------------------------------------------------------------------------------------------------
# route probe
# ---------------------------------------------------------------------------------------------------------------------
_KERNEL = re.compile(r"mb::(k_\w+)")


class Routes:
    """One torch.profiler session around the calls of a test. Each call announces its largest segment with expect();
    on exit, the sweep launches of the exported trace, in launch order, must be the dispatch table's kernels for those
    sizes, with one mask launch per sweep, and for the two kernels with dynamic shared memory the traced shared-memory
    size must show the tile-buffer band."""

    def __init__(self):
        self.expected = []

    def expect(self, max_seg, blocks=False, launches=1):
        self.expected += [(max_seg,) + sweep_route(max_seg, blocks)] * launches

    def __enter__(self):
        torch.cuda.synchronize()
        self.prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA])
        self.prof.__enter__()
        return self

    def __exit__(self, *exc):
        torch.cuda.synchronize()
        self.prof.__exit__(*exc)
        if exc[0] is None:
            self.check()
        return False

    def _launches(self):
        """(start, kernel name, trace args) of every library kernel the session recorded."""
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "trace.json")
            self.prof.export_chrome_trace(path)
            with open(path) as fh:
                events = json.load(fh).get("traceEvents", [])
        return [(float(e.get("ts", 0.0)), m.group(1), e.get("args", {})) for e in events if e.get("cat") == "kernel"
                for m in [_KERNEL.search(e.get("name", ""))] if m]

    def check(self):
        ours = self._launches()
        assert ours, "torch.profiler recorded no library kernel for calls that launch some: the routes cannot be checked"
        ours.sort(key=lambda k: k[0])
        sweeps = [(name, args) for _, name, args in ours if name in SWEEPS]
        assert [n for n, _ in sweeps] == [e[1] for e in self.expected], ([n for n, _ in sweeps], self.expected)
        assert sum(name == "k_nms_mask" for _, name, _ in ours) == len(self.expected)
        for (name, args), (max_seg, _, nbuf, dyn) in zip(sweeps, self.expected):
            if dyn:
                smem = int(args["shared memory"])
                assert dyn <= smem <= dyn + 1024, (max_seg, name, nbuf, dyn, smem)   # dynamic + a few static bytes


# ---------------------------------------------------------------------------------------------------------------------
# mb_nms at every band edge: plain, coordinate trick, per-group (vanilla)
# ---------------------------------------------------------------------------------------------------------------------
def _groups(n, seed):
    return np.random.default_rng(seed).integers(0, 3, n).astype(np.int64)


def run_nms_case(ops, routes, mode, family, n, thr, blocks=False, dev=DEV):
    b, s = cases.nms_family(family, n, thr)
    if mode == "plain":
        fn = lambda: ops.nms(cu(b, dev), cu(s, dev), thr)
        want = R.nms(b, s, thr)
    else:
        g = _groups(n, n)
        fn = lambda: ops.batched_nms(cu(b, dev), cu(s, dev), cu(g, dev), thr, strategy=mode)
        want = (R.batched_nms_vanilla if mode == "vanilla" else R.batched_nms_coordinate_trick)(b, s, g, thr)
    routes.expect(n, blocks)
    assert np.array_equal(fn().cpu().numpy(), want), (mode, family, n, thr)


def _thresholds(mode, fi):
    """plain mode: every threshold; the other modes: two per family, rotating, so that each threshold occurs."""
    return THRESHOLDS if mode == "plain" else (THRESHOLDS[(2 * fi) % 6], THRESHOLDS[(2 * fi + 1) % 6])


@pytest.mark.parametrize("mode", ["plain", "trick", "vanilla"])
@pytest.mark.parametrize("n", (65,) + BAND_EDGES)
def test_nms_band_edges(ops, mode, n):
    with Routes() as routes:
        for fi, family in enumerate(cases.NMS_FAMILIES):
            for thr in _thresholds(mode, fi):
                run_nms_case(ops, routes, mode, family, n, thr)


# ---------------------------------------------------------------------------------------------------------------------
# keep cap on every route: mb_det_postprocess with one segment per image, mb_rpn_proposals at small post_nms_top_n
# ---------------------------------------------------------------------------------------------------------------------
def _det_inputs(max_props, n_img=2, hw=(800, 800)):
    rng = np.random.default_rng(max_props)
    counts = [max_props, max_props - 37]
    proposals = [cases.stress_rois(rng, c, hw, side=(8.0, 160.0)) for c in counts]
    rows = sum(counts)
    # class-1 logits spread evenly, so that no two scores lie within a few ulps of each other (the kernel's expf and
    # numpy's exp may differ by an ulp, which would swap such a pair), and zero regression, so that the decoded boxes
    # are the proposals on both sides: the NMS decisions and their order are then defined exactly
    logits = np.zeros((rows, 2), F)
    logits[:, 1] = rng.permutation(np.linspace(-3.0, 3.0, rows))
    reg = np.zeros((rows, 8), F)
    padded = np.zeros((n_img, max_props, 4), F)
    for i, p in enumerate(proposals):
        padded[i, :len(p)] = p
    return logits, reg, proposals, padded, counts, [hw] * n_img


@pytest.mark.parametrize("max_props", [1000, 3000, 5000, 7000, 10000, 20000, 26000])
def test_det_keep_cap_on_every_route(det, monkeypatch, max_props):
    """2 classes: one NMS segment per image, capped at detections_per_img inside the sweep; score threshold 0, so
    every candidate enters the NMS. The cap is set below, at and above the image's kept count."""
    logits, reg, proposals, padded, counts, shapes = _det_inputs(max_props)
    monkeypatch.setattr(D, "batched_nms", R.batched_nms)       # the same strategy rule, exact at any size
    full = D.postprocess_detections(logits, reg, proposals, shapes, score_thresh=0.0, detections_per_img=max_props)
    kept = len(full[0][2])
    assert kept > 300, kept
    cut = 0
    with Routes() as routes:
        for dpi in sorted({63, 64, 65, kept - 1, kept, kept + 1, 300}):
            cfg = det.DetConfig(detections_per_img=dpi, score_thresh=0.0)
            routes.expect(max_props)
            out = det.postprocess_detections(cu(logits), cu(reg), cu(padded), torch.tensor(counts, dtype=torch.int32, device=DEV),
                                             shapes, cfg, packed=True)
            boxes, scores, labels = out.as_lists()
            for i in range(len(counts)):
                rb, rs, rl = (a[:dpi] for a in full[i])
                assert np.array_equal(labels[i].cpu().numpy(), rl), (max_props, dpi, i)
                assert cases.box_rel_err(boxes[i].cpu().numpy(), rb) < 1e-5
                assert np.max(np.abs(scores[i].cpu().numpy() - rs), initial=0.0) < 1e-6
            cut += len(labels[0]) == dpi < kept
    assert cut == 5                                             # 63, 64, 65, 300 and kept - 1 were cut by the cap


def _rpn_reference(obj, dlt, image_sizes, padded, pre, post, rule):
    objectness, deltas = D.concat_rpn_head_outputs(obj, dlt)
    napl = [o.shape[1] * o.shape[2] * o.shape[3] for o in obj]
    anchors = D.grid_anchors(padded, [o.shape[-2:] for o in obj], cases.RPN_SIZES, cases.RPN_RATIOS)
    decoded = np.stack([D.decode_boxes(deltas[i], anchors)[:, 0] for i in range(objectness.shape[0])])
    device_rule = {4000: "cpu", 100000: "cuda"}.get(rule)
    orig = D.batched_nms
    if device_rule is None:   # forced vanilla
        D.batched_nms = lambda b, s, idx, thr, device_rule="cpu": D.batched_nms_vanilla(b, s, idx, thr)
    try:
        rb, rs = D.filter_proposals(decoded, objectness, image_sizes, napl, pre_nms_top_n=pre, post_nms_top_n=post,
                                    nms_thresh=0.7, device_rule=device_rule or "cpu")
    finally:
        D.batched_nms = orig
    return objectness, napl, rb, rs


def check_rpn(det, routes, obj, dlt, image_sizes, padded, cfg, blocks=False):
    out = det.rpn_proposals([cu(o) for o in obj], [cu(d) for d in dlt], image_sizes, padded, cfg, return_topk_idx=True)
    objectness, napl, rb, rs = _rpn_reference(obj, dlt, image_sizes, padded, cfg.pre_nms_top_n, cfg.post_nms_top_n,
                                              cfg.trick_numel)
    routes.expect(min(cfg.pre_nms_top_n, max(napl)), blocks)
    for i in range(objectness.shape[0]):
        assert np.array_equal(out.topk_idx[i].cpu().numpy(), D.rpn_top_n_idx(objectness[i], napl, cfg.pre_nms_top_n)), i
    boxes, scores = out.as_lists()
    for i in range(objectness.shape[0]):
        assert boxes[i].shape == rb[i].shape, (i, boxes[i].shape, rb[i].shape)
        assert cases.box_rel_err(boxes[i].cpu().numpy(), rb[i]) < 1e-5
        assert np.max(np.abs(scores[i].cpu().numpy() - rs[i]), initial=0.0) < 1e-6
    return out


@pytest.mark.parametrize("pre", [1000, 4096])
@pytest.mark.parametrize("post", [63, 64, 65])
def test_rpn_keep_cap_fixpoint_and_small_sweep(det, pre, post):
    obj, dlt, grids, image_sizes, padded = cases.rpn_case()
    cfg = det.RpnConfig(cases.RPN_SIZES, cases.RPN_RATIOS, pre_nms_top_n=pre, post_nms_top_n=post, nms_thresh=0.7)
    with Routes() as routes:
        out = check_rpn(det, routes, obj, dlt, image_sizes, padded, cfg)
    assert out.counts.tolist() == [post] * len(image_sizes)


# ---------------------------------------------------------------------------------------------------------------------
# many groups (vanilla): skewed sizes, gaps in the indices, kept scores in one or in all score buckets
# ---------------------------------------------------------------------------------------------------------------------
def score_bucket(s):
    """The vanilla finalize's bucket of each score: the top 12 bits of desc_score_key (miso_b200/csrc/common.cuh)."""
    u = np.asarray(s, F).view(np.uint32).copy()
    u[u == 0x80000000] = 0
    asc = np.where(u >> 31 == 1, ~u, u | np.uint32(0x80000000)).astype(np.uint32)
    return np.where(np.isnan(s), 0, (~asc).astype(np.uint32) >> 20)


def _group_case(G, spread, seed=0):
    rng = np.random.default_rng([G, spread, seed])
    big = 2000
    present = np.unique(np.concatenate([rng.choice(G, max(1, (7 * G) // 8), replace=False), [G - 1, G // 2]]))
    gid = np.concatenate([np.full(big, G // 2), present, rng.choice(present, 300)]).astype(np.int64)
    n = len(gid)
    b = cases.random_boxes(rng, n, extent=24.0 * np.sqrt(n), wh=(16.0, 96.0))
    b[:big] = cases.random_boxes(rng, big, extent=600.0, wh=(16.0, 96.0))       # the large group is dense
    if spread:
        # random finite bit patterns: scores of every sign and exponent, over all 4096 buckets of the vanilla finalize
        u = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
        u = np.where((u & 0x7F800000) == 0x7F800000, u & 0xBFFFFFFF, u)
        s = u.view(F)
    else:
        s = (0.5 + rng.permutation(n).astype(np.float64) * 2.0 ** -24).astype(F)   # all in [0.5, 0.5625): one bucket
    p = rng.permutation(n)
    return b[p], s[p], gid[p]


@pytest.mark.parametrize("spread", [False, True])
@pytest.mark.parametrize("G", [32, 33, 256, 257, 1024, 1025, 5000])
def test_vanilla_many_groups(ops, G, spread):
    b, s, g = _group_case(G, spread)
    assert int(g.max()) == G - 1 and len(np.unique(g)) < G
    with Routes() as routes:
        routes.expect(len(b))
        keep = ops.batched_nms(cu(b), cu(s), cu(g), 0.5, strategy="vanilla")
    want = R.batched_nms_vanilla(b, s, g, 0.5)
    assert np.array_equal(keep.cpu().numpy(), want), G
    buckets = len(np.unique(score_bucket(s[want])))
    assert buckets > 500 if spread else buckets == 1, buckets


# ---------------------------------------------------------------------------------------------------------------------
# one huge segment: T > 2048 words (double-precision tile decode in k_nms_mask) and the generic sweep
# ---------------------------------------------------------------------------------------------------------------------
def test_huge_segment(ops):
    n = 140000
    b, s = cases.nms_family("random", n, 0.5)
    with Routes() as routes:
        routes.expect(n)
        keep = ops.nms(cu(b), cu(s), 0.5)
    assert -(-n // 64) == 2188
    assert np.array_equal(keep.cpu().numpy(), R.nms(b, s, 0.5))


# ---------------------------------------------------------------------------------------------------------------------
# mask workspace retry (vanilla mode first tries a bounded mask)
# ---------------------------------------------------------------------------------------------------------------------
def test_mask_workspace_retry(ops, monkeypatch):
    lib = ops._lib.load()
    calls = []
    real = lib.mb_nms

    def counting(*args):
        calls.append(args[3])
        return real(*args)

    b, s = cases.nms_family("cluster", 3000, 0.5)
    g = _groups(3000, 1)
    monkeypatch.setattr(ops, "_MASK_FIRST_TRY_BYTES", 4096)
    monkeypatch.setattr(lib, "mb_nms", counting)
    keep = ops.batched_nms(cu(b), cu(s), cu(g), 0.5, strategy="vanilla").cpu().numpy()
    assert len(calls) == 2
    assert np.array_equal(keep, R.batched_nms_vanilla(b, s, g, 0.5))


# ---------------------------------------------------------------------------------------------------------------------
# MB_NMS_SWEEP=blocks, and the order in which the entry points first launch the wide sweep (fresh processes)
# ---------------------------------------------------------------------------------------------------------------------
def _in_fresh_process(call, env=None):
    e = dict(os.environ)
    e["PYTHONPATH"] = ROOT + os.pathsep + e.get("PYTHONPATH", "")
    e.update(env or {})
    code = f"import tests.test_gpu_nms_routes as t; t.{call}; print('routes-ok')"
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=e, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0 and "routes-ok" in res.stdout, res.stdout[-4000:] + res.stderr[-4000:]


def block_sweeps_main():
    from miso_b200 import detection, ops as o
    with Routes() as routes:
        for n in (65, 1024):
            for mode in ("plain", "trick", "vanilla"):
                for fi, family in enumerate(cases.NMS_FAMILIES):
                    for thr in _thresholds(mode, fi):
                        run_nms_case(o, routes, mode, family, n, thr, blocks=True)
        obj, dlt, grids, image_sizes, padded = cases.rpn_case()
        cfg = detection.RpnConfig(cases.RPN_SIZES, cases.RPN_RATIOS, pre_nms_top_n=1000, post_nms_top_n=64, nms_thresh=0.7)
        check_rpn(detection, routes, obj, dlt, image_sizes, padded, cfg, blocks=True)


def test_block_sweeps_for_small_segments():
    """MB_NMS_SWEEP=blocks sends segments of <= 1024 boxes through the row-major block sweep instead of the fixed
    point; the switch is read once per process."""
    _in_fresh_process("block_sweeps_main()", {"MB_NMS_SWEEP": "blocks"})


def caller_order_main(det_first):
    """The wide sweep first launched by one entry point, then by another with a smaller shared-memory need: each
    entry point must opt its own kernel in."""
    from miso_b200 import detection, ops as o

    def via_det():
        logits, reg, proposals, padded, counts, shapes = _det_inputs(5000)
        orig, D.batched_nms = D.batched_nms, R.batched_nms
        try:
            ref = D.postprocess_detections(logits, reg, proposals, shapes, score_thresh=0.0, detections_per_img=300)
        finally:
            D.batched_nms = orig
        cfg = detection.DetConfig(detections_per_img=300, score_thresh=0.0)
        assert sweep_route(5000)[:2] == ("k_nms_sweep_wide", 4)
        with Routes() as routes:
            routes.expect(5000)
            out = detection.postprocess_detections(cu(logits), cu(reg), cu(padded),
                                                   torch.tensor(counts, dtype=torch.int32, device=DEV), shapes, cfg, packed=True)
        for i, lab in enumerate(out.as_lists()[2]):
            assert np.array_equal(lab.cpu().numpy(), ref[i][2])

    def via_nms():
        b, s = cases.nms_family("random", 6400, 0.5)
        assert sweep_route(6400)[:2] == ("k_nms_sweep_wide", 3)
        with Routes() as routes:
            routes.expect(6400)
            keep = o.nms(cu(b), cu(s), 0.5)
        assert np.array_equal(keep.cpu().numpy(), R.nms(b, s, 0.5))

    for f in ((via_det, via_nms) if det_first else (via_nms, via_det)):
        f()


@pytest.mark.parametrize("det_first", [True, False])
def test_wide_sweep_caller_order(det_first):
    _in_fresh_process(f"caller_order_main({det_first})")


# ---------------------------------------------------------------------------------------------------------------------
# the bench's shapes: 8 tiles of 800^2, 159 882 anchors per image, 1000 proposals and 300 detections per image
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bench_batch():
    from miso_b200 import workload
    w = workload.faster_rcnn_batch(num_images=8, channels=4, pin=False)
    h = {k: [t.numpy() for t in v] for k, v in w.host.items()}
    return w, h


def _bench_det(det, routes, w, h, rpn_out):
    R_ = rpn_out.proposals.shape[1]
    counts = rpn_out.counts.cpu().numpy()
    routes.expect(R_)
    out = det.postprocess_detections(cu(h["class_logits"][0]), cu(h["box_regression"][0]), rpn_out.proposals,
                                     rpn_out.counts, w.shapes.image_sizes, w.det, packed=False)
    props = [rpn_out.proposals[i, :c].cpu().numpy() for i, c in enumerate(counts)]
    rows = np.concatenate([np.arange(i * R_, i * R_ + c) for i, c in enumerate(counts)])
    ref = D.postprocess_detections(h["class_logits"][0][rows], h["box_regression"][0][rows], props, w.shapes.image_sizes,
                                   detections_per_img=w.det.detections_per_img)
    boxes, scores, labels = out.as_lists()
    for i in range(len(counts)):
        assert np.array_equal(labels[i].cpu().numpy(), ref[i][2]), i
        assert cases.box_rel_err(boxes[i].cpu().numpy(), ref[i][0]) < 1e-5
        assert np.max(np.abs(scores[i].cpu().numpy() - ref[i][1]), initial=0.0) < 1e-6


@pytest.mark.parametrize("rule", [4000, -1])
def test_bench_shapes(det, bench_batch, rule):
    w, h = bench_batch
    cfg = dataclasses.replace(w.rpn, trick_numel=rule)
    assert sum(o.shape[1] * o.shape[2] * o.shape[3] for o in h["objectness"]) == 159882
    with Routes() as routes:
        out = check_rpn(det, routes, h["objectness"], h["deltas"], w.shapes.image_sizes, w.shapes.padded_image_size, cfg)
        if rule == 4000:
            _bench_det(det, routes, w, h, out)


def test_bench_shapes_crowded_threshold_bin(det, bench_batch):
    """Level-0 logits quantised so that the histogram bin holding the 1000th largest has ~12 000 candidates (more
    than the 4096 the selection stages): the unstaged candidate path behind the level's 30 linked CTAs."""
    w, h = bench_batch
    rng = np.random.default_rng(12)
    obj = [o.copy() for o in h["objectness"]]
    u = rng.uniform(0, 1, obj[0].shape)
    obj[0] = np.where(u < 0.002, 3.0, np.where(u < 0.1, 1.0, -1.0)).astype(F)
    assert ((obj[0] == 1.0).sum(axis=(1, 2, 3)) > 4096).all() and ((obj[0] == 3.0).sum(axis=(1, 2, 3)) < 1000).all()
    with Routes() as routes:
        out = check_rpn(det, routes, obj, h["deltas"], w.shapes.image_sizes, w.shapes.padded_image_size, w.rpn)
        _bench_det(det, routes, w, h, out)


# ---------------------------------------------------------------------------------------------------------------------
# a second device in one process: the per-device shared-memory opt-in of the wide sweep
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_wide_sweep_on_second_device(ops):
    for dev in ("cuda:0", "cuda:1"):
        with torch.cuda.device(dev), Routes() as routes:
            run_nms_case(ops, routes, "plain", "random", 6400, 0.5, dev=dev)

"""The prepared sync-free plan (miso_b200.pipeline.HotPath) against the oracle composition of the
same stages (oracle/pipeline.py). Each stage is also re-checked on the GPU path's own
intermediate results, so a 1-ulp exp() difference upstream cannot hide a downstream bug."""
import numpy as np
import pytest
import torch

from oracle import detection as D
from oracle import miso_path as M
from oracle import pipeline as ref_pipeline
from tests import cases

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def build(n=2, original=320, resized=256, channels=16, post=200, dpi=50, seed=0, exact=True, layout="nchw"):
    from miso_b200 import pipeline, workload
    w = workload.faster_rcnn_batch(num_images=n, original=original, resized=resized, channels=channels,
                                   post_nms_top_n=post, detections_per_img=dpi, seed=seed, pin=False, features_layout=layout)
    hp = pipeline.HotPath(w.shapes, w.rpn, w.det, threshold=w.threshold, crop_capacity_bytes=32 << 20,
                          exact_roi_align=exact, device=DEV)
    dev = workload.to_device(w, DEV)
    hp.bind(dev["objectness"], dev["deltas"], dev["features"], dev["class_logits"][0], dev["box_regression"][0], dev["images"])
    return w, hp


def oracle_run(w):
    h = {k: [t.numpy() for t in v] for k, v in w.host.items()}
    return ref_pipeline.run(h["objectness"], h["deltas"], h["features"], h["class_logits"][0], h["box_regression"][0],
                            h["images"], padded_image_size=w.shapes.padded_image_size, image_sizes=w.shapes.image_sizes,
                            original_image_sizes=w.shapes.original_image_sizes, sizes=w.rpn.sizes,
                            aspect_ratios=w.rpn.aspect_ratios, pre_nms_top_n=w.rpn.pre_nms_top_n,
                            post_nms_top_n=w.rpn.post_nms_top_n, detections_per_img=w.det.detections_per_img,
                            threshold=w.threshold), h


@pytest.mark.parametrize("seed", [0, 1])
def test_hot_path_matches_oracle_composition(seed):
    w, hp = build(seed=seed)
    check_against_oracle(w, hp)


@pytest.mark.parametrize("layout", ["channels_last", "nchw"])
def test_hot_path_full_size_config2_matches_oracle(layout):
    """BASELINE config 2 at FULL size (batch 4, 1024^2 -> 800^2, 159 882 anchors / image, 1000 proposals, 256
    channels, 300 detections) against the oracle composition on all four images, stage by stage: proposal counts and
    boxes, RoIAlign bit-exact (4000 RoIs x 256 x 7 x 7, on the TMA-staged kernel for channels-last maps), detections,
    crops byte for byte."""
    from miso_b200 import _lib
    w, hp = build(n=4, original=1024, resized=800, channels=256, post=1000, dpi=300, seed=0, layout=layout)
    check_against_oracle(w, hp)
    assert hp.features_layout == layout
    hp.roi_params.force_gather = 2                                # the TMA-staged route on the same proposals: identical features
    want = hp.box_features.clone()
    n0 = _lib.load().mb_roi_align_tma_launches()
    hp.box_features.zero_()
    hp.roi_align()
    torch.cuda.synchronize()
    assert _lib.load().mb_roi_align_tma_launches() == n0 + 1 and torch.equal(hp.box_features, want)


def check_against_oracle(w, hp):
    hp.step()
    torch.cuda.synchronize()
    ref, h = oracle_run(w)
    n, R, dpi = w.shapes.num_images, hp.R, hp.dpi
    pc = hp.prop_counts.cpu().numpy()
    dc = hp.det_counts.cpu().numpy()
    res = hp.results()
    for i in range(n):
        # stage 1: proposals
        assert pc[i] == len(ref[i]["proposals"])
        gp = hp.proposals[i, :pc[i]].cpu().numpy()
        assert cases.box_rel_err(gp, ref[i]["proposals"]) < 1e-5
        # stage 2: RoIAlign, bit-exact on the GPU path's own proposals
        gf = hp.box_features[i * R:i * R + pc[i]].cpu().numpy()
        feats = D.multiscale_roi_align(h["features"], [gp if j == i else np.zeros((0, 4), np.float32) for j in range(n)],
                                       w.shapes.image_sizes, 7, 2)
        assert np.array_equal(gf, feats)
        assert torch.count_nonzero(hp.box_features[i * R + pc[i]:(i + 1) * R]) == 0   # dead slots are zeros
        # stage 3: detections
        assert dc[i] == len(ref[i]["labels"])
        assert np.array_equal(hp.det_labels[i, :dc[i]].cpu().numpy(), ref[i]["labels"])
        assert cases.box_rel_err(hp.det_boxes[i, :dc[i]].cpu().numpy(), ref[i]["boxes"]) < 1e-5
        assert np.max(np.abs(hp.det_scores[i, :dc[i]].cpu().numpy() - ref[i]["scores"])) < 1e-6
        # stage 4: score filter + crops, bit-exact on the GPU path's own detections
        kb, ks, kl, xywh, ci, crops = M.filter_and_crop(h["images"][i], hp.det_boxes[i, :dc[i]].cpu().numpy(),
                                                        hp.det_scores[i, :dc[i]].cpu().numpy(),
                                                        hp.det_labels[i, :dc[i]].cpu().numpy(), w.threshold)
        assert len(res[i]) == len(crops)
        for got, want, lab, xy in zip(res[i], crops, kl, xywh):
            assert got["label"] == lab
            assert np.array_equal(got["xywh"], xy)
            assert got["crop"].shape == want.shape and np.array_equal(got["crop"], want)
        assert len(res[i]) == len(ref[i]["crops"])


def test_hot_path_bind_rejects_channels_last_maps_outside_the_in_place_envelope():
    """Channels-last FPN maps that mb_multiscale_roi_align cannot read in place (here: sampling ratio 0) are refused by
    bind(); HotPath allocates nothing per step, so it cannot fall back to an NCHW copy."""
    import dataclasses
    from miso_b200 import pipeline, workload
    from miso_b200._lib import MisoB200Error
    w = workload.faster_rcnn_batch(num_images=1, original=320, resized=256, channels=16, post_nms_top_n=200,
                                   detections_per_img=50, pin=False, features_layout="channels_last")
    hp = pipeline.HotPath(dataclasses.replace(w.shapes, sampling_ratio=0), w.rpn, w.det, crop_capacity_bytes=1 << 20, device=DEV)
    d = workload.to_device(w, DEV)
    with pytest.raises(MisoB200Error, match="channels-last"):
        hp.bind(d["objectness"], d["deltas"], d["features"], d["class_logits"][0], d["box_regression"][0], d["images"])
    nchw = [f.contiguous() for f in d["features"]]
    hp.bind(d["objectness"], d["deltas"], nchw, d["class_logits"][0], d["box_regression"][0], d["images"])
    hp.step()
    torch.cuda.synchronize()
    assert hp.features_layout == "nchw"


def test_hot_path_is_deterministic_and_idempotent():
    w, hp = build(seed=3)
    hp.step(); torch.cuda.synchronize()
    a = [t.clone() for t in (hp.proposals, hp.box_features, hp.det_boxes, hp.det_labels, hp.crop_totals)]
    pix = hp.crop_pixels[: int(hp.crop_totals[1])].clone()
    for _ in range(3):
        hp.step()
    torch.cuda.synchronize()
    for x, y in zip(a, (hp.proposals, hp.box_features, hp.det_boxes, hp.det_labels, hp.crop_totals)):
        assert torch.equal(x, y)
    assert torch.equal(pix, hp.crop_pixels[: int(hp.crop_totals[1])])


def test_hot_path_graph_replay_equals_step():
    w, hp = build(seed=4)
    hp.step(); torch.cuda.synchronize()
    want = [t.clone() for t in (hp.proposals, hp.box_features, hp.det_boxes, hp.det_labels, hp.crop_totals)]
    pix = hp.crop_pixels[: int(hp.crop_totals[1])].clone()
    hp.capture()
    for t in (hp.proposals, hp.box_features, hp.det_boxes, hp.crop_pixels):
        t.fill_(3)
    hp.replay(); hp.replay()
    torch.cuda.synchronize()
    for x, y in zip(want, (hp.proposals, hp.box_features, hp.det_boxes, hp.det_labels, hp.crop_totals)):
        assert torch.equal(x, y)
    assert torch.equal(pix, hp.crop_pixels[: int(hp.crop_totals[1])])


def test_hot_path_full_size_config2_properties():
    """BASELINE config 2 at full size (batch 4, 800^2, 256 ch, 1000 proposals): size-independent
    properties — proposal scores sorted, NMS idempotence (re-running NMS on the kept proposals keeps
    all of them), kept proposals inside the image, crops consistent with their rectangles."""
    from miso_b200 import ops
    w, hp = build(n=4, original=1024, resized=800, channels=256, post=1000, dpi=300, seed=0)
    hp.step(); torch.cuda.synchronize()
    pc = hp.prop_counts.cpu().numpy()
    assert (pc == 1000).all()
    for i in range(4):
        s = hp.prop_scores[i, :pc[i]]
        assert torch.all(s[:-1] >= s[1:])
        b = hp.proposals[i, :pc[i]]
        assert b.min() >= 0 and b.max() <= 800
    tot = hp.crop_totals.tolist()
    assert tot[2] == 0 and tot[0] > 0
    offs = hp.crop_offsets[: tot[0] + 1].cpu().numpy(); rects = hp.crop_rects[: tot[0]].cpu().numpy()
    assert np.array_equal(np.diff(offs), rects[:, 2].astype(np.int64) * rects[:, 3] * 3)
    # detections: NMS idempotence per image and class on the network-scale boxes
    dc = hp.det_counts.cpu().numpy()
    for i in range(4):
        keep = ops.batched_nms(hp.det_boxes_net[i, :dc[i]], hp.det_scores[i, :dc[i]], hp.det_labels[i, :dc[i]], 0.5,
                               strategy="vanilla")
        assert keep.numel() == dc[i]


def test_host_pipeline_matches_single_steps():
    """HostPipeline (pinned host in/out, three streams, two slots) on a sequence of different
    batches: every batch's read-back equals a plain bind + step + sync of the same inputs."""
    from miso_b200 import pipeline, workload
    ws = [workload.faster_rcnn_batch(num_images=2, original=320, resized=256, channels=16, post_nms_top_n=200,
                                     detections_per_img=50, seed=s, pin=True) for s in range(5)]
    w0 = ws[0]

    def make():
        return pipeline.HotPath(w0.shapes, w0.rpn, w0.det, threshold=w0.threshold, crop_capacity_bytes=8 << 20, device=DEV)

    pipe = pipeline.HostPipeline(make, w0.host)
    got = []
    for w in ws:
        r = pipe.submit(w.host)
        if r is not None:
            got.append({k: v.clone() for k, v in r["out"].items()} | {"pixels": r["pixels"].clone()})
    for r in pipe.flush():
        got.append({k: v.clone() for k, v in r["out"].items()} | {"pixels": r["pixels"].clone()})
    assert len(got) == len(ws)
    hp = make()
    for w, g in zip(ws, got):
        d = workload.to_device(w, DEV)
        hp.bind(d["objectness"], d["deltas"], d["features"], d["class_logits"][0], d["box_regression"][0], d["images"])
        hp.step(); torch.cuda.synchronize()
        tot = hp.crop_totals.tolist()
        assert g["crop_totals"].tolist() == tot and tot[0] > 0
        dc = hp.det_counts.cpu()
        assert torch.equal(g["det_counts"], dc)
        for i in range(2):
            for k in ("det_labels", "det_boxes", "det_scores"):
                assert torch.equal(g[k][i, : dc[i]], getattr(hp, k)[i, : dc[i]].cpu()), k
        for k in ("crop_rects", "crop_xywh", "crop_src"):
            assert torch.equal(g[k][: tot[0]], getattr(hp, k)[: tot[0]].cpu()), k
        assert torch.equal(g["crop_offsets"][: tot[0] + 1], hp.crop_offsets[: tot[0] + 1].cpu())
        assert torch.equal(g["pixels"], hp.crop_pixels[: tot[1]].cpu())


def test_overlapped_plan_equals_serial_steps():
    """Three batches in flight on three streams (OverlappedHotPath), each slot bound to DIFFERENT
    inputs, many rounds: every slot ends with exactly the results of a plain serial step."""
    from miso_b200 import pipeline
    built = [build(seed=s) for s in (5, 6, 7)]
    want = []
    for w, hp in built:
        hp.step(); torch.cuda.synchronize()
        want.append([t.clone() for t in (hp.proposals, hp.prop_counts, hp.box_features, hp.det_boxes, hp.det_scores,
                                         hp.det_labels, hp.det_counts, hp.crop_totals, hp.crop_rects)]
                    + [hp.crop_pixels[: int(hp.crop_totals[1])].clone()])
        for t in (hp.proposals, hp.box_features, hp.det_boxes, hp.det_scores, hp.crop_pixels):
            t.fill_(7)                      # poison: the overlapped run must rewrite everything
    plan = pipeline.OverlappedHotPath([hp for _, hp in built])
    for _ in range(12):
        plan.submit()
    plan.drain()
    torch.cuda.synchronize()
    for (w, hp), ref in zip(built, want):
        got = [hp.proposals, hp.prop_counts, hp.box_features, hp.det_boxes, hp.det_scores, hp.det_labels, hp.det_counts,
               hp.crop_totals, hp.crop_rects, hp.crop_pixels[: int(hp.crop_totals[1])]]
        pc, dc = hp.prop_counts.cpu(), hp.det_counts.cpu()
        assert torch.equal(got[1], ref[1]) and torch.equal(got[6], ref[6]) and torch.equal(got[7], ref[7])
        assert torch.equal(got[2], ref[2])                                   # RoIAlign output incl. zeroed dead slots
        for i in range(w.shapes.num_images):
            assert torch.equal(got[0][i, : pc[i]], ref[0][i, : pc[i]])
            for j in (3, 4, 5):
                assert torch.equal(got[j][i, : dc[i]], ref[j][i, : dc[i]])
        k = int(ref[7][0])
        assert torch.equal(got[8][:k], ref[8][:k]) and torch.equal(got[9], ref[9])

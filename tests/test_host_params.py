"""The host-side parameter builders (rpn_params, det_params, pooler_levels, roi_align_params, crop_params) on the
bench's shapes and configurations, checked against torchvision's own CPU modules; no device needed."""
import dataclasses

import numpy as np
import pytest
import torch

from miso_b200 import detection, ops, workload


@pytest.fixture(scope="module")
def w():
    return workload.faster_rcnn_batch(pin=False)


def f32(v) -> float:
    return float(np.float32(v))


def test_rpn_params_anchors_and_strides_match_anchor_generator(w):
    from torchvision.models.detection.anchor_utils import AnchorGenerator
    from torchvision.models.detection.image_list import ImageList
    s = w.shapes
    p = detection.rpn_params(w.rpn, s.rpn_grids, [3] * len(s.rpn_grids), s.padded_image_size, s.image_sizes)
    ag = AnchorGenerator(w.rpn.sizes, w.rpn.aspect_ratios)
    assert p.num_levels == len(s.rpn_grids) == len(ag.cell_anchors)
    ours = []
    for l, ((gh, gw), base) in enumerate(zip(s.rpn_grids, ag.cell_anchors)):
        a = base.shape[0]
        assert (p.feat_h[l], p.feat_w[l], p.anchors_per_loc[l]) == (gh, gw, a)
        assert [[p.base_anchors[l][i][c] for c in range(4)] for i in range(a)] == base.tolist()
        # grid_anchors (tv:models/detection/anchor_utils.py:76-106) from our strides and base anchors
        sy = torch.arange(gh, dtype=torch.int32) * p.stride_h[l]
        sx = torch.arange(gw, dtype=torch.int32) * p.stride_w[l]
        yy, xx = torch.meshgrid(sy, sx, indexing="ij")
        shifts = torch.stack([xx.reshape(-1), yy.reshape(-1), xx.reshape(-1), yy.reshape(-1)], dim=1)
        ours.append((shifts.view(-1, 1, 4) + base.view(1, -1, 4)).reshape(-1, 4))
    images = ImageList(torch.zeros((1, 3) + tuple(s.padded_image_size)), [s.image_sizes[0]])
    want = ag(images, [torch.zeros((1, 1, gh, gw)) for gh, gw in s.rpn_grids])[0]
    assert torch.equal(torch.cat(ours), want)
    with pytest.raises(AssertionError, match="anchors per location"):
        detection.rpn_params(w.rpn, s.rpn_grids, [9] * len(s.rpn_grids), s.padded_image_size, s.image_sizes)


def test_rpn_params_fields(w):
    cfg = dataclasses.replace(w.rpn, pre_nms_top_n=900, post_nms_top_n=700, nms_thresh=0.65, score_thresh=0.01,
                              min_size=0.002, weights=(1.5, 2.0, 2.5, 3.0), bbox_xform_clip=4.0, trick_numel=123)
    sizes = [(800, 608), (640, 800), (800, 800), (512, 800)]
    p = detection.rpn_params(cfg, w.shapes.rpn_grids, None, (800, 800), sizes)
    assert p.num_images == 4 and [(p.image_h[i], p.image_w[i]) for i in range(4)] == sizes
    assert (p.pre_nms_top_n, p.post_nms_top_n, p.trick_numel) == (900, 700, 123)
    assert p.nms_thresh == 0.65                                  # fp64 field
    assert (p.score_thresh, p.min_size, p.bbox_xform_clip) == (f32(0.01), f32(0.002), 4.0)
    assert (p.wx, p.wy, p.ww, p.wh) == (1.5, 2.0, 2.5, 3.0)
    assert [(p.stride_h[l], p.stride_w[l]) for l in range(p.num_levels)] == [(800 // gh, 800 // gw) for gh, gw in w.shapes.rpn_grids]


def test_det_params_fields(w):
    cfg = dataclasses.replace(w.det, score_thresh=0.07, nms_thresh=0.45, detections_per_img=250, weights=(9.0, 8.0, 4.0, 3.0),
                              bbox_xform_clip=3.5, min_size=0.03, trick_numel=77)
    s = w.shapes
    p = detection.det_params(cfg, s.num_images, s.num_classes, w.rpn.post_nms_top_n, s.image_sizes, s.original_image_sizes)
    assert (p.num_images, p.num_classes, p.max_props_per_image, p.detections_per_img) == (4, 3, 1000, 250)
    assert [(p.image_h[i], p.image_w[i]) for i in range(4)] == list(s.image_sizes)
    assert [(p.orig_h[i], p.orig_w[i]) for i in range(4)] == list(s.original_image_sizes)
    assert p.nms_thresh == 0.45 and (p.score_thresh, p.min_size, p.bbox_xform_clip) == (f32(0.07), f32(0.03), 3.5)
    assert (p.wx, p.wy, p.ww, p.wh, p.trick_numel) == (9.0, 8.0, 4.0, 3.0, 77)
    q = detection.det_params(cfg, 4, 3, 1000, s.image_sizes)
    assert all(q.orig_h[i] == q.orig_w[i] == 0 for i in range(4))


def test_pooler_levels_match_multiscale_roi_align(w):
    from torchvision.ops.poolers import _setup_scales
    s = w.shapes
    scales, thresholds = ops.pooler_levels(s.feature_grids, s.image_sizes)
    tv_scales, mapper = _setup_scales([torch.zeros((1, 1, gh, gw)) for gh, gw in s.feature_grids], list(s.image_sizes), 224, 4)
    assert scales == tv_scales and len(thresholds) == len(scales) - 1
    for i, t in enumerate(thresholds):
        # entry i is the smallest fp32 area the mapper sends to a level > i
        a = np.array([t, np.nextafter(np.float32(t), np.float32(0))], dtype=np.float32)
        boxes = torch.from_numpy(np.stack([np.zeros_like(a), np.zeros_like(a), a, np.ones_like(a)], 1))
        assert mapper([boxes]).tolist() == [i + 1, i]
    assert ops.pooler_levels(s.feature_grids[:1], s.image_sizes) == ([tv_scales[0]], ())
    with pytest.raises(ValueError):
        ops.pooler_levels(s.feature_grids, [])


def test_roi_align_params_fields(w):
    s = w.shapes
    scales, thresholds = ops.pooler_levels(s.feature_grids, s.image_sizes)
    p = ops.roi_align_params(s.feature_grids, s.num_images, s.channels, (s.pooled, s.pooled), s.sampling_ratio, scales,
                             thresholds, exact=False, channels_last=True, boxes_per_image=1000)
    assert (p.num_levels, p.num_images, p.channels, p.pooled_h, p.pooled_w, p.sampling_ratio) == (4, 4, 256, 7, 7, 2)
    assert (p.aligned, p.exact, p.channels_last, p.boxes_per_image, p.force_gather, p.box_counts) == (0, 0, 1, 1000, 0, None)
    assert [(p.height[l], p.width[l]) for l in range(4)] == list(s.feature_grids)
    assert [p.spatial_scale[l] for l in range(4)] == scales == [0.25, 0.125, 0.0625, 0.03125]
    assert tuple(p.level_thresholds[l] for l in range(3)) == thresholds
    q = ops.roi_align_params(s.feature_grids[:1], 1, 8, (5, 6), 0, scales[:1], (), aligned=True)
    assert (q.num_levels, q.pooled_h, q.pooled_w, q.sampling_ratio, q.aligned, q.exact, q.channels_last) == (1, 5, 6, 0, 1, 1, 0)


def test_channels_last_predicate_envelope():
    m = workload.mosaic(1024, 1024).shapes(8)                   # the bench's per-batch shapes
    bench = dict(channels=m.channels, output_size=(m.pooled, m.pooled), sampling_ratio=m.sampling_ratio)
    assert ops.roi_align_reads_channels_last(**bench)
    assert ops.roi_align_reads_channels_last(**{**bench, "output_size": (16, 16)})
    assert not ops.roi_align_reads_channels_last(**{**bench, "sampling_ratio": 0})
    assert not ops.roi_align_reads_channels_last(**{**bench, "output_size": (17, 17)})
    assert not ops.roi_align_reads_channels_last(**{**bench, "output_size": (7, 17)})
    assert not ops.roi_align_reads_channels_last(**{**bench, "channels": 1})
    assert not ops.roi_align_reads_channels_last(**bench, dtype=torch.bfloat16)
    f = torch.zeros((2, 16, 5, 6))
    assert ops.is_channels_last(f.contiguous(memory_format=torch.channels_last)) and not ops.is_channels_last(f)


def test_crop_params_fields(w):
    s = w.shapes
    p = detection.crop_params(s.original_image_sizes, s.image_channels, w.det.detections_per_img, w.threshold)
    assert (p.num_images, p.capacity, p.channels, p.boxes_are_xywh) == (4, 300, 3, 0)
    assert [(p.image_h[i], p.image_w[i]) for i in range(4)] == list(s.original_image_sizes)
    assert p.threshold == 0.5 and not any(p.images[i] for i in range(4))
    q = detection.crop_params([(16384, 12000)], 1, 5400, 0.3, boxes_are_xywh=True)
    assert (q.num_images, q.image_h[0], q.image_w[0], q.capacity, q.channels, q.threshold, q.boxes_are_xywh) == \
        (1, 16384, 12000, 5400, 1, f32(0.3), 1)

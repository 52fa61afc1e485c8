"""Fused stages of the detection hot path (host side of mb_rpn_proposals, mb_det_postprocess,
mb_crop_plan / mb_crop_gather).

Each function mirrors one reference stage (same argument meaning, hyper-parameters read from
the model object by the caller — never hard-coded here):

  rpn_proposals        AnchorGenerator.forward + concat_box_prediction_layers + BoxCoder.decode +
                       RegionProposalNetwork.filter_proposals
                       (tv:models/detection/anchor_utils.py:115-133, rpn.py:81-110, :231-297)
  postprocess_detections   RoIHeads.postprocess_detections + transform.postprocess boxes
                       (tv:models/detection/roi_heads.py:680-737, transform.py:257-277)
  filter_and_crop      miso score filter + coords_int + crop slice
                       (ref:miso/object_detection/inference.py:53-62, crop.py:28-30)

All outputs have fixed capacity with device-side counts, so a whole batch needs no host
synchronisation until the caller reads the counts.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import CropParams, DetParams, MisoB200Error, RpnParams
from .ops import _f32c, _ptr, _require_cuda, _stream, _workspace, base_anchors

BBOX_XFORM_CLIP = math.log(1000.0 / 16)
CPU_RULE_NUMEL = 4000       # tv:ops/boxes.py:80, the reference's CPU path (the parity oracle)
CUDA_RULE_NUMEL = 100_000   # same line, CUDA tensors


# ------------------------------------------------------------------------------------------
# RPN
# ------------------------------------------------------------------------------------------
@dataclass
class RpnConfig:
    """Hyper-parameters of RegionProposalNetwork + AnchorGenerator (read from the model)."""
    sizes: Sequence[Sequence[float]]
    aspect_ratios: Sequence[Sequence[float]]
    pre_nms_top_n: int = 1000
    post_nms_top_n: int = 1000
    nms_thresh: float = 0.7
    score_thresh: float = 0.0
    min_size: float = 1e-3
    weights: Sequence[float] = (1.0, 1.0, 1.0, 1.0)
    bbox_xform_clip: float = BBOX_XFORM_CLIP
    trick_numel: int = CPU_RULE_NUMEL

    @classmethod
    def from_model(cls, rpn, trick_numel: int = CPU_RULE_NUMEL) -> "RpnConfig":
        ag = rpn.anchor_generator
        return cls(sizes=ag.sizes, aspect_ratios=ag.aspect_ratios, pre_nms_top_n=rpn.pre_nms_top_n(),
                   post_nms_top_n=rpn.post_nms_top_n(), nms_thresh=rpn.nms_thresh, score_thresh=rpn.score_thresh,
                   min_size=rpn.min_size, weights=tuple(rpn.box_coder.weights),
                   bbox_xform_clip=rpn.box_coder.bbox_xform_clip, trick_numel=trick_numel)


@dataclass
class RpnOutput:
    proposals: Tensor   # [N, post_nms_top_n, 4] fp32, rows >= counts[n] are zero
    scores: Tensor      # [N, post_nms_top_n]
    counts: Tensor      # [N] int32 (device)
    topk_idx: Optional[Tensor] = None   # [N, sum_l min(pre, A_l)] int64 when requested

    def as_lists(self) -> Tuple[List[Tensor], List[Tensor]]:
        """The reference's return type (list per image). Reads the counts: one host sync."""
        cnt = self.counts.tolist()
        return ([self.proposals[i, :c] for i, c in enumerate(cnt)], [self.scores[i, :c] for i, c in enumerate(cnt)])


def rpn_proposals(objectness: Sequence[Tensor], pred_bbox_deltas: Sequence[Tensor], image_sizes: Sequence[Tuple[int, int]],
                  padded_image_size: Tuple[int, int], cfg: RpnConfig, return_topk_idx: bool = False) -> RpnOutput:
    """objectness[l]: [N, A, H_l, W_l] logits, pred_bbox_deltas[l]: [N, 4A, H_l, W_l] — the RPN head's
    outputs exactly as the reference produces them (NCHW, no permute / cat)."""
    lib = _lib.load()
    L = len(objectness)
    if L < 1 or L > _lib.MB_MAX_LEVELS or len(pred_bbox_deltas) != L:
        raise MisoB200Error("rpn_proposals: bad number of levels")
    n = objectness[0].shape[0]
    if n > _lib.MB_MAX_IMAGES:
        raise MisoB200Error(f"rpn_proposals: at most {_lib.MB_MAX_IMAGES} images per call")
    p = RpnParams()
    p.num_images, p.num_levels = n, L
    keep = []
    for l in range(L):
        o, d = objectness[l], pred_bbox_deltas[l]
        _require_cuda(o, "objectness")
        _require_cuda(d, "pred_bbox_deltas")
        o, d = _f32c(o), _f32c(d)
        keep += [o, d]
        a, gh, gw = o.shape[1], o.shape[2], o.shape[3]
        torch._assert(d.shape == (n, 4 * a, gh, gw), "deltas must be [N, 4A, H, W]")
        p.feat_h[l], p.feat_w[l], p.anchors_per_loc[l] = gh, gw, a
        p.stride_h[l], p.stride_w[l] = padded_image_size[0] // gh, padded_image_size[1] // gw
        base = base_anchors(cfg.sizes[l], cfg.aspect_ratios[l])
        torch._assert(base.shape[0] == a, "anchors per location do not match the head's output channels")
        for ai in range(a):
            for c in range(4):
                p.base_anchors[l][ai][c] = float(base[ai, c])
        p.objectness[l], p.deltas[l] = o.data_ptr(), d.data_ptr()
    for i, (h, w) in enumerate(image_sizes):
        p.image_h[i], p.image_w[i] = int(h), int(w)
    p.pre_nms_top_n, p.post_nms_top_n = int(cfg.pre_nms_top_n), int(cfg.post_nms_top_n)
    p.nms_thresh, p.score_thresh, p.min_size = float(cfg.nms_thresh), float(cfg.score_thresh), float(cfg.min_size)
    p.wx, p.wy, p.ww, p.wh = (float(v) for v in cfg.weights)
    p.bbox_xform_clip = float(cfg.bbox_xform_clip)
    p.trick_numel = int(cfg.trick_numel)
    dev = keep[0].device
    ws_bytes = lib.mb_rpn_workspace_bytes(C.byref(p))
    if ws_bytes == 0:
        raise MisoB200Error("rpn_proposals: configuration outside the implemented envelope "
                            "(pre_nms_top_n <= 4096 per level, <= 16384 per image)")
    ws = _workspace(ws_bytes, dev)
    post = p.post_nms_top_n
    props = torch.empty((n, post, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((n, post), dtype=torch.float32, device=dev)
    counts = torch.empty((n,), dtype=torch.int32, device=dev)
    topk = None
    if return_topk_idx:
        ktot = sum(min(p.pre_nms_top_n, o.shape[1] * o.shape[2] * o.shape[3]) for o in keep[0::2])
        topk = torch.empty((n, ktot), dtype=torch.int64, device=dev)
    rc = lib.mb_rpn_proposals(C.byref(p), _ptr(props), _ptr(scores), _ptr(counts), _ptr(topk), _ptr(ws), ws.numel(),
                              _stream(props))
    _lib.check(rc, "mb_rpn_proposals")
    return RpnOutput(props, scores, counts, topk)


# ------------------------------------------------------------------------------------------
# detection post-processing
# ------------------------------------------------------------------------------------------
@dataclass
class DetConfig:
    score_thresh: float = 0.05
    nms_thresh: float = 0.5
    detections_per_img: int = 100
    weights: Sequence[float] = (10.0, 10.0, 5.0, 5.0)
    bbox_xform_clip: float = BBOX_XFORM_CLIP
    min_size: float = 1e-2                       # literal in tv:models/detection/roi_heads.py:724
    trick_numel: int = CPU_RULE_NUMEL

    @classmethod
    def from_model(cls, roi_heads, trick_numel: int = CPU_RULE_NUMEL) -> "DetConfig":
        return cls(score_thresh=roi_heads.score_thresh, nms_thresh=roi_heads.nms_thresh,
                   detections_per_img=roi_heads.detections_per_img, weights=tuple(roi_heads.box_coder.weights),
                   bbox_xform_clip=roi_heads.box_coder.bbox_xform_clip, trick_numel=trick_numel)


@dataclass
class DetOutput:
    boxes: Tensor       # [N, dpi, 4] at the original image scale
    boxes_net: Tensor   # [N, dpi, 4] at the network (resized) scale
    scores: Tensor      # [N, dpi]
    labels: Tensor      # [N, dpi] int64
    counts: Tensor      # [N] int32

    def as_lists(self):
        cnt = self.counts.tolist()
        return ([self.boxes[i, :c] for i, c in enumerate(cnt)], [self.scores[i, :c] for i, c in enumerate(cnt)],
                [self.labels[i, :c] for i, c in enumerate(cnt)])


def postprocess_detections(class_logits: Tensor, box_regression: Tensor, proposals: Tensor, prop_counts: Tensor,
                           image_shapes: Sequence[Tuple[int, int]], cfg: DetConfig,
                           original_image_sizes: Optional[Sequence[Tuple[int, int]]] = None,
                           packed: bool = False) -> DetOutput:
    """proposals [N, R, 4] with prop_counts[n] live rows (RpnOutput layout). class_logits [rows, C],
    box_regression [rows, 4C]; rows of image n start at n*R (packed=False) or at the sum of the
    earlier counts (packed=True, the reference's concatenated layout)."""
    lib = _lib.load()
    for t, nm in ((class_logits, "class_logits"), (box_regression, "box_regression"), (proposals, "proposals"),
                  (prop_counts, "prop_counts")):
        _require_cuda(t, nm)
    n, r = proposals.shape[0], proposals.shape[1]
    c = class_logits.shape[-1]
    p = DetParams()
    p.num_images, p.num_classes, p.max_props_per_image = n, c, r
    p.detections_per_img = int(cfg.detections_per_img)
    for i, (h, w) in enumerate(image_shapes):
        p.image_h[i], p.image_w[i] = int(h), int(w)
        if original_image_sizes is not None:
            p.orig_h[i], p.orig_w[i] = int(original_image_sizes[i][0]), int(original_image_sizes[i][1])
    p.nms_thresh, p.score_thresh, p.min_size = float(cfg.nms_thresh), float(cfg.score_thresh), float(cfg.min_size)
    p.wx, p.wy, p.ww, p.wh = (float(v) for v in cfg.weights)
    p.bbox_xform_clip = float(cfg.bbox_xform_clip)
    p.trick_numel = int(cfg.trick_numel)
    ws_bytes = lib.mb_det_workspace_bytes(C.byref(p))
    if ws_bytes == 0:
        raise MisoB200Error("postprocess_detections: configuration outside the implemented envelope "
                            "((classes-1) * min(proposals, detections_per_img) <= 16384)")
    dev = class_logits.device
    ws = _workspace(ws_bytes, dev)
    dpi = p.detections_per_img
    lg, rg, pr = _f32c(class_logits), _f32c(box_regression), _f32c(proposals)
    pc = prop_counts.to(torch.int32).contiguous()
    boxes = torch.empty((n, dpi, 4), dtype=torch.float32, device=dev)
    boxes_net = torch.empty((n, dpi, 4), dtype=torch.float32, device=dev)
    scores = torch.empty((n, dpi), dtype=torch.float32, device=dev)
    labels = torch.empty((n, dpi), dtype=torch.int64, device=dev)
    counts = torch.empty((n,), dtype=torch.int32, device=dev)
    rc = lib.mb_det_postprocess(C.byref(p), _ptr(lg), _ptr(rg), _ptr(pr), _ptr(pc), int(packed), _ptr(boxes),
                                _ptr(boxes_net), _ptr(scores), _ptr(labels), _ptr(counts), _ptr(ws), ws.numel(),
                                _stream(lg))
    _lib.check(rc, "mb_det_postprocess")
    return DetOutput(boxes, boxes_net, scores, labels, counts)


# ------------------------------------------------------------------------------------------
# score filter + crops
# ------------------------------------------------------------------------------------------
@dataclass
class CropOutput:
    totals: Tensor     # [4] int64: number of crops, total bytes, pixel overflow flag, mask overflow flag
    rects: Tensor      # [N*cap, 4] int32 (x_begin, y_begin, width, height)
    xywh: Tensor       # [N*cap, 4] fp32 annotation bounds (x, y, w, h)
    src: Tensor        # [N*cap] int32: n*cap + detection index
    offsets: Tensor    # [N*cap+1] int64 byte offsets into `pixels`
    pixels: Tensor     # [capacity] uint8 packed crops (HWC each)
    masks: Optional[Tensor] = None     # uint8 packed h*w masks (0 / 255) of the crops at offsets // channels

    def to_host(self, channels: int):
        """One device->host transfer; returns per-crop (image index, detection index, xywh, array)."""
        tot = self.totals.tolist()
        if tot[2]:
            raise MisoB200Error(f"crop buffer too small: {tot[1]} bytes needed")
        k = tot[0]
        rects = self.rects[:k].cpu().numpy(); xywh = self.xywh[:k].cpu().numpy(); src = self.src[:k].cpu().numpy()
        offs = self.offsets[:k + 1].cpu().numpy(); pix = self.pixels[:tot[1]].cpu().numpy()
        cap = self.rects.shape[0] // max(1, self._n)
        out = []
        for j in range(k):
            _, _, w, h = rects[j]
            a = pix[offs[j]:offs[j + 1]].reshape((h, w, channels) if channels > 1 else (h, w))
            out.append((int(src[j]) // cap, int(src[j]) % cap, xywh[j], a))
        return out

    def masks_to_host(self) -> List:
        """The crops' masks as np.uint8 [h, w] arrays in crop order (one device->host transfer of the packed bytes)."""
        if self.masks is None:
            raise MisoB200Error("no masks: filter_and_crop ran without mask_probs")
        tot = self.totals.tolist()
        if tot[3]:
            raise MisoB200Error(f"mask buffer too small: {tot[1] // self._ch} bytes needed")
        k = tot[0]
        rects = self.rects[:k].cpu().numpy()
        offs = self.offsets[:k + 1].cpu().numpy() // self._ch
        buf = self.masks[:tot[1] // self._ch].cpu().numpy()
        return [buf[offs[j]:offs[j + 1]].reshape(rects[j][3], rects[j][2]) for j in range(k)]

    _n: int = 1
    _ch: int = 1


def filter_and_crop(images: Sequence[Tensor], det_boxes: Tensor, det_scores: Tensor, det_counts: Tensor,
                    threshold: float, capacity_bytes: Optional[int] = None, boxes_are_xywh: bool = False,
                    mask_probs: Optional[Tensor] = None, paste_boxes: Optional[Tensor] = None, mask_threshold: float = 0.5,
                    mask_capacity_bytes: Optional[int] = None) -> CropOutput:
    """images[n]: uint8 [H, W, C] or [H, W] on the device (the ORIGINAL image pixels, as
    skimage.io.imread returns them); det_* as produced by postprocess_detections.

    mask_probs ([N, cap, M, M] or [N*cap, 1, M, M], Mask R-CNN's per-detection probabilities) adds each crop's instance
    mask (mb_crop_masks): paste_masks_in_image of the detection's mask into its image at paste_boxes (default
    det_boxes, xyxy), cut to the crop rectangle, 255 where > mask_threshold else 0. capacity_bytes = 0 skips the pixel
    gather; mask_capacity_bytes None sizes the mask buffer exactly (one host sync)."""
    lib = _lib.load()
    n, cap = det_boxes.shape[0], det_boxes.shape[1]
    if len(images) != n:
        raise MisoB200Error("filter_and_crop: one image per detection row expected")
    p = CropParams()
    p.num_images, p.capacity = n, cap
    ch = 1 if images[0].dim() == 2 else images[0].shape[2]
    p.channels = ch
    keep = []
    for i, im in enumerate(images):
        _require_cuda(im, "image")
        if im.dtype != torch.uint8:
            raise MisoB200Error("filter_and_crop: images must be uint8 (HWC)")
        im = im.contiguous()
        keep.append(im)
        p.image_h[i], p.image_w[i] = im.shape[0], im.shape[1]
        p.images[i] = im.data_ptr()
    p.threshold = float(threshold)
    p.boxes_are_xywh = int(bool(boxes_are_xywh))
    dev = det_boxes.device
    b, s = _f32c(det_boxes), _f32c(det_scores)
    cnt = det_counts.to(torch.int32).contiguous()
    rects = torch.empty((n * cap, 4), dtype=torch.int32, device=dev)
    xywh = torch.empty((n * cap, 4), dtype=torch.float32, device=dev)
    src = torch.empty((n * cap,), dtype=torch.int32, device=dev)
    offsets = torch.empty((n * cap + 1,), dtype=torch.int64, device=dev)
    totals = torch.zeros((4,), dtype=torch.int64, device=dev)
    st = _stream(b)
    _lib.check(lib.mb_crop_plan(C.byref(p), _ptr(b), _ptr(s), _ptr(cnt), _ptr(rects), _ptr(xywh), _ptr(src),
                                _ptr(offsets), _ptr(totals), st), "mb_crop_plan")
    if capacity_bytes is None:
        capacity_bytes = int(totals[1].item())          # exact size: costs one host sync
    pixels = torch.empty((max(int(capacity_bytes), 1),), dtype=torch.uint8, device=dev)
    _lib.check(lib.mb_crop_gather(C.byref(p), _ptr(rects), _ptr(src), _ptr(offsets), _ptr(totals), _ptr(pixels),
                                  int(capacity_bytes), st), "mb_crop_gather")
    masks = None
    if mask_probs is not None:
        m = int(mask_probs.shape[-1])
        mp = _f32c(mask_probs)
        torch._assert(mp.numel() == n * cap * m * m and mp.shape[-2] == m, "mask_probs must be [N, cap, M, M] or [N*cap, 1, M, M]")
        pb = b if paste_boxes is None else _f32c(paste_boxes)
        torch._assert(pb.numel() == n * cap * 4, "paste_boxes must be [N, cap, 4]")
        if mask_capacity_bytes is None:
            mask_capacity_bytes = int(totals[1].item()) // ch
        masks = torch.empty((max(int(mask_capacity_bytes), 1),), dtype=torch.uint8, device=dev)
        _lib.check(lib.mb_crop_masks(C.byref(p), _ptr(mp), _ptr(pb), m, 1, None, cap, float(mask_threshold), _ptr(rects),
                                     _ptr(src), _ptr(offsets), _ptr(totals), _ptr(masks), int(mask_capacity_bytes), st),
                   "mb_crop_masks")
    out = CropOutput(totals, rects, xywh, src, offsets, pixels, masks)
    out._n, out._ch = n, ch
    return out

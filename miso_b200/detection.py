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
# the columns of a crop's morphology record (mb_mask_morphology, include/misob200.h): regionprops of the crop's mask,
# in pixels; centroids in image (or mosaic) coordinates; mean_intensity_k is 0 for k >= the image's channels
MORPHOLOGY_FIELDS = ("area", "perimeter", "centroid_x", "centroid_y", "major_axis_length", "minor_axis_length",
                     "orientation", "eccentricity", "equivalent_diameter",
                     "mean_intensity_0", "mean_intensity_1", "mean_intensity_2", "mean_intensity_3")


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


def rpn_params(cfg: RpnConfig, rpn_grids: Sequence[Tuple[int, int]], anchors_per_loc: Optional[Sequence[int]],
               padded_image_size: Tuple[int, int], image_sizes: Sequence[Tuple[int, int]]) -> RpnParams:
    """mb_rpn_proposals' parameters for the RPN head's output grids (H_l, W_l), without the input pointers: anchor
    strides and base anchors (AnchorGenerator), thresholds and box-coder weights. anchors_per_loc: the head's anchors
    per location and level, checked against the configuration when given."""
    p = RpnParams()
    p.num_images, p.num_levels = len(image_sizes), len(rpn_grids)
    for l, (gh, gw) in enumerate(rpn_grids):
        base = base_anchors(cfg.sizes[l], cfg.aspect_ratios[l])
        a = base.shape[0]
        if anchors_per_loc is not None:
            torch._assert(a == anchors_per_loc[l], "anchors per location do not match the head's output channels")
        p.feat_h[l], p.feat_w[l], p.anchors_per_loc[l] = int(gh), int(gw), a
        p.stride_h[l], p.stride_w[l] = padded_image_size[0] // int(gh), padded_image_size[1] // int(gw)
        for ai in range(a):
            for c in range(4):
                p.base_anchors[l][ai][c] = float(base[ai, c])
    for i, (h, w) in enumerate(image_sizes):
        p.image_h[i], p.image_w[i] = int(h), int(w)
    p.pre_nms_top_n, p.post_nms_top_n = int(cfg.pre_nms_top_n), int(cfg.post_nms_top_n)
    p.nms_thresh, p.score_thresh, p.min_size = float(cfg.nms_thresh), float(cfg.score_thresh), float(cfg.min_size)
    p.wx, p.wy, p.ww, p.wh = (float(v) for v in cfg.weights)
    p.bbox_xform_clip = float(cfg.bbox_xform_clip)
    p.trick_numel = int(cfg.trick_numel)
    return p


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
    if len(image_sizes) != n:
        raise MisoB200Error("rpn_proposals: one image size per image expected")
    keep = []
    for o, d in zip(objectness, pred_bbox_deltas):
        _require_cuda(o, "objectness")
        _require_cuda(d, "pred_bbox_deltas")
        o, d = _f32c(o), _f32c(d)
        keep += [o, d]
        torch._assert(d.shape == (n, 4 * o.shape[1], o.shape[2], o.shape[3]), "deltas must be [N, 4A, H, W]")
    p = rpn_params(cfg, [o.shape[2:] for o in keep[0::2]], [o.shape[1] for o in keep[0::2]], padded_image_size, image_sizes)
    for l in range(L):
        p.objectness[l], p.deltas[l] = keep[2 * l].data_ptr(), keep[2 * l + 1].data_ptr()
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


def det_params(cfg: DetConfig, num_images: int, num_classes: int, max_props_per_image: int,
               image_sizes: Sequence[Tuple[int, int]], original_image_sizes: Optional[Sequence[Tuple[int, int]]] = None) -> DetParams:
    """mb_det_postprocess' parameters. Without original_image_sizes the boxes are not rescaled to the original images."""
    p = DetParams()
    p.num_images, p.num_classes, p.max_props_per_image = int(num_images), int(num_classes), int(max_props_per_image)
    p.detections_per_img = int(cfg.detections_per_img)
    for i, (h, w) in enumerate(image_sizes):
        p.image_h[i], p.image_w[i] = int(h), int(w)
        if original_image_sizes is not None:
            p.orig_h[i], p.orig_w[i] = int(original_image_sizes[i][0]), int(original_image_sizes[i][1])
    p.nms_thresh, p.score_thresh, p.min_size = float(cfg.nms_thresh), float(cfg.score_thresh), float(cfg.min_size)
    p.wx, p.wy, p.ww, p.wh = (float(v) for v in cfg.weights)
    p.bbox_xform_clip = float(cfg.bbox_xform_clip)
    p.trick_numel = int(cfg.trick_numel)
    return p


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
    p = det_params(cfg, proposals.shape[0], class_logits.shape[-1], proposals.shape[1], image_shapes, original_image_sizes)
    n = p.num_images
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
def crop_params(image_hw: Sequence[Tuple[int, int]], channels: int, capacity: int, threshold: float,
                boxes_are_xywh: bool = False) -> CropParams:
    """The crop kernels' parameters for images of the given (H, W), without the image pointers. capacity: detection
    slots per image."""
    p = CropParams()
    p.num_images, p.capacity, p.channels = len(image_hw), int(capacity), int(channels)
    for i, (h, w) in enumerate(image_hw):
        p.image_h[i], p.image_w[i] = int(h), int(w)
    p.threshold = float(threshold)
    p.boxes_are_xywh = int(bool(boxes_are_xywh))
    return p


class CropStage:
    """Score filter + crops of a batch of detections, with its parameters and fixed-capacity outputs:
    mb_crop_plan (plan()), then mb_crop_gather, mb_crop_masks and mb_mask_morphology (cut()).

    Launches neither allocate nor synchronise: every buffer is allocated by the constructor, reserve() and
    bind_masks(), so a stage can be recorded into a CUDA graph. The bound images and mask inputs are held for as
    long as the stage can launch. Outputs (first totals[0] rows in crop order):

      totals      [4] int64: number of crops, total bytes, pixel overflow flag, mask overflow flag
      rects       [N*cap, 4] int32 (x_begin, y_begin, width, height)
      xywh        [N*cap, 4] fp32 annotation bounds (x, y, w, h)
      src         [N*cap] int32: n*cap + detection index
      offsets     [N*cap+1] int64 byte offsets into `pixels`
      pixels      [capacity] uint8 packed crops (HWC each)
      masks       uint8 packed h*w masks (0 / 255) of the crops at offsets // channels (bind_masks())
      morphology  [N*cap, len(MORPHOLOGY_FIELDS)] fp64 records (bind_masks(morphology=True))
      png, png_offsets, png_status          one PNG file per crop, packed in crop order (bind_png(), mb_png_encode);
      mask_png, mask_png_offsets, mask_png_status   the same for the masks (bind_png() with bind_masks())
      jpeg        one JPEG file per crop, packed in crop order, the bytes PIL writes by default (bind_jpeg(), mb_jpeg_encode)
    """

    def __init__(self, image_hw: Sequence[Tuple[int, int]], channels: int, capacity: int, threshold: float, device,
                 capacity_bytes: Optional[int] = None, boxes_are_xywh: bool = False):
        """capacity: detection slots per image; capacity_bytes: size of the pixel buffer (None: call reserve())."""
        self.lib = _lib.load()
        self.params = crop_params(image_hw, channels, capacity, threshold, boxes_are_xywh)
        self.dev = torch.device(device)
        rows = self.params.num_images * self.params.capacity
        self.rects = torch.zeros((rows, 4), dtype=torch.int32, device=self.dev)
        self.xywh = torch.zeros((rows, 4), dtype=torch.float32, device=self.dev)
        self.src = torch.zeros((rows,), dtype=torch.int32, device=self.dev)
        self.offsets = torch.zeros((rows + 1,), dtype=torch.int64, device=self.dev)
        self.totals = torch.zeros((4,), dtype=torch.int64, device=self.dev)
        self.images: List[Tensor] = []
        self.mask_args = self.masks = self.morphology = self.morph_ws = None
        self.capacity = self.mask_capacity = 0
        self.pixels = None
        self.png = self.mask_png = self.jpeg = None
        if capacity_bytes is not None:
            self.reserve(capacity_bytes)

    def reserve(self, capacity_bytes: int) -> None:
        """Allocate the pixel buffer: crops that do not fit set totals[2] and are not written."""
        self.capacity = int(capacity_bytes)
        self.pixels = torch.empty((max(self.capacity, 1),), dtype=torch.uint8, device=self.dev)

    def bind_images(self, images: Sequence[Tensor], pointers: Optional[Sequence[int]] = None) -> None:
        """Crop from images[i] (uint8 [H, W, C] or [H, W], contiguous), addressed at pointers[i] when given (a
        virtual base pointer of a band of rows)."""
        self.images = list(images)
        for i, im in enumerate(self.images):
            self.params.images[i] = im.data_ptr() if pointers is None else int(pointers[i])

    def bind_masks(self, mask_probs: Tensor, paste_boxes: Tensor, frames: Optional[Tensor], rows_per_frame: int,
                   mask_threshold: float, capacity_bytes: int, morphology: bool = False) -> None:
        """Cut every crop's instance mask after the pixels (mb_crop_masks): slot s pastes mask_probs[s] ([slots, M, M])
        at paste_boxes[s] (xyxy) into frame s // rows_per_frame, frames[f] = (x0, y0, w, h) int32, or image f when
        frames is None; > mask_threshold -> 255. morphology=True also measures every mask (mb_mask_morphology)."""
        self.mask_args = (mask_probs, paste_boxes, frames, int(mask_probs.shape[-1]), int(rows_per_frame), float(mask_threshold))
        self.mask_capacity = int(capacity_bytes)
        self.masks = torch.empty((max(self.mask_capacity, 1),), dtype=torch.uint8, device=self.dev)
        self.morphology = self.morph_ws = None
        if self.png is not None:
            self.mask_png = self._png_buffers(self.mask_capacity, 1, self._mask_png_capacity)
        if morphology:
            self.morphology = torch.empty((self.rects.shape[0], len(MORPHOLOGY_FIELDS)), dtype=torch.float64, device=self.dev)
            nbytes = int(self.lib.mb_mask_morphology_workspace_bytes(C.byref(self.params)))
            self.morph_ws = torch.empty((max(nbytes, 1),), dtype=torch.uint8, device=self.dev)

    def bind_png(self, capacity_bytes: Optional[int] = None, mask_capacity_bytes: Optional[int] = None) -> None:
        """Encode every crop as a PNG file after the cut (mb_png_encode), and every mask when bind_masks() is (or gets)
        called. Capacities default to mb_png_bound_bytes of the pixel / mask buffers, which no crop set can exceed."""
        self.png = self._png_buffers(self.capacity, self.params.channels, capacity_bytes)
        self._mask_png_capacity = mask_capacity_bytes
        if self.masks is not None:
            self.mask_png = self._png_buffers(self.mask_capacity, 1, mask_capacity_bytes)

    def bind_jpeg(self, capacity_bytes: Optional[int] = None) -> None:
        """Encode every crop as a JPEG file after the gather (mb_jpeg_encode): the bytes PIL's Image.save writes with
        default settings. 1 or 3 channels. The capacity defaults to mb_jpeg_bound_bytes of the pixel buffer, which no
        crop set can exceed (416 B per 8x8 block of 1-pixel-wide crops); pass a smaller one to save memory, an overflow
        is then reported by jpeg_to_host()."""
        self.jpeg = self._png_buffers(self.capacity, self.params.channels, capacity_bytes, "jpeg")

    def _png_buffers(self, packed_capacity: int, channels: int, capacity_bytes: Optional[int], kind: str = "png") -> dict:
        slots = self.rects.shape[0]
        if capacity_bytes is None:
            capacity_bytes = int(getattr(self.lib, f"mb_{kind}_bound_bytes")(packed_capacity, slots, channels))
        ws = int(getattr(self.lib, f"mb_{kind}_workspace_bytes")(C.byref(self.params), packed_capacity, channels))
        if capacity_bytes < 0 or ws == 0:
            raise MisoB200Error(f"mb_{kind}_encode: {channels} channels are not supported "
                                f"({'1..4' if kind == 'png' else '1 or 3'})")
        return {"kind": kind, "channels": channels, "capacity": int(capacity_bytes),
                "out": torch.empty((max(int(capacity_bytes), 1),), dtype=torch.uint8, device=self.dev),
                "offsets": torch.zeros((slots + 1,), dtype=torch.int64, device=self.dev),
                "status": torch.zeros((2,), dtype=torch.int64, device=self.dev),
                "ws": torch.empty((ws,), dtype=torch.uint8, device=self.dev)}

    def _encode(self, buf: dict, packed: Tensor, stream) -> None:
        fn = f"mb_{buf['kind']}_encode"
        _lib.check(getattr(self.lib, fn)(C.byref(self.params), _ptr(packed), buf["channels"], _ptr(self.rects),
                                         _ptr(self.offsets), _ptr(self.totals), _ptr(buf["ws"]), buf["ws"].numel(),
                                         _ptr(buf["out"]), buf["capacity"], _ptr(buf["offsets"]), _ptr(buf["status"]),
                                         stream), fn)

    def plan(self, boxes: Tensor, scores: Tensor, counts: Tensor, stream) -> None:
        """mb_crop_plan: boxes [N, cap, 4] fp32, scores [N, cap] fp32, counts [N] int32, all contiguous."""
        _lib.check(self.lib.mb_crop_plan(C.byref(self.params), _ptr(boxes), _ptr(scores), _ptr(counts), _ptr(self.rects),
                                         _ptr(self.xywh), _ptr(self.src), _ptr(self.offsets), _ptr(self.totals), stream),
                   "mb_crop_plan")

    def cut(self, stream) -> None:
        """The planned crops' pixels, then (bind_masks()) their masks and morphology."""
        cp = C.byref(self.params)
        _lib.check(self.lib.mb_crop_gather(cp, _ptr(self.rects), _ptr(self.src), _ptr(self.offsets), _ptr(self.totals),
                                           _ptr(self.pixels), self.capacity, stream), "mb_crop_gather")
        if self.jpeg is not None:
            self._encode(self.jpeg, self.pixels, stream)
        if self.mask_args is None:
            if self.png is not None:
                self._encode(self.png, self.pixels, stream)
            return
        probs, boxes, frames, m, rpf, thr = self.mask_args
        _lib.check(self.lib.mb_crop_masks(cp, _ptr(probs), _ptr(boxes), m, 1, _ptr(frames), rpf, thr, _ptr(self.rects),
                                          _ptr(self.src), _ptr(self.offsets), _ptr(self.totals), _ptr(self.masks),
                                          self.mask_capacity, stream), "mb_crop_masks")
        if self.morphology is not None:
            _lib.check(self.lib.mb_mask_morphology(cp, _ptr(self.masks), _ptr(self.rects), _ptr(self.src), _ptr(self.offsets),
                                                   _ptr(self.totals), _ptr(self.morph_ws), self.morph_ws.numel(),
                                                   _ptr(self.morphology), stream), "mb_mask_morphology")
        # after the masks: a mask overflow flag in totals means nothing is encoded
        if self.png is not None:
            self._encode(self.png, self.pixels, stream)
        if self.mask_png is not None:
            self._encode(self.mask_png, self.masks, stream)

    def checked_totals(self, totals: Optional[Tensor] = None, pixels: bool = True, masks: bool = False) -> List[int]:
        """totals (default: this stage's, one sync; or a host copy of them) as a list, raising if the pixel buffer
        (pixels=True) or the mask buffer (masks=True) was too small."""
        tot = (self.totals if totals is None else totals).tolist()
        if pixels and tot[2]:
            raise MisoB200Error(f"crop buffer too small: {tot[1]} bytes needed, {self.capacity} available")
        if masks and tot[3]:
            raise MisoB200Error(f"mask buffer too small: {tot[1] // self.params.channels} bytes needed, "
                                f"{self.mask_capacity} available")
        return tot

    @staticmethod
    def checked_png(buf: dict, what: str = "PNG") -> List[int]:
        """A PNG buffer's status (one sync) as [total bytes, flag], raising if the buffer or workspace was too small."""
        st = buf["status"].tolist()
        if st[1] == 1:
            raise MisoB200Error(f"{what} buffer too small: {st[0]} bytes needed, {buf['capacity']} available")
        if st[1]:
            raise MisoB200Error(f"{what} workspace too small for the crops")
        return st

    def _png_host(self, buf: Optional[dict], what: str) -> List[bytes]:
        if buf is None:
            bind = "bind_jpeg()" if what == "JPEG" else "bind_png()"
            raise MisoB200Error(f"no {what} streams: {bind} was not called" + (" after bind_masks()" if "mask" in what else ""))
        # the PNG encoder skips every crop on a mask overflow, the JPEG encoder only on a pixel overflow
        k = self.checked_totals(pixels=buf is not self.mask_png, masks=buf is not self.jpeg and self.masks is not None)[0]
        total = self.checked_png(buf, what)[0]
        offs = buf["offsets"][:k + 1].cpu().numpy()
        data = buf["out"][:total].cpu().numpy().tobytes()
        return [data[offs[j]:offs[j + 1]] for j in range(k)]

    def png_to_host(self) -> List[bytes]:
        """Every crop's PNG file as bytes, crop order (b"" for a crop of zero area); one copy of the packed streams."""
        return self._png_host(self.png, "PNG")

    def jpeg_to_host(self) -> List[bytes]:
        """Every crop's JPEG file as bytes, crop order (b"" for a crop of zero area); one copy of the packed streams."""
        return self._png_host(self.jpeg, "JPEG")

    def mask_png_to_host(self) -> List[bytes]:
        """Every crop's mask as a PNG file (mode L, 0 / 255), crop order; one copy of the packed streams."""
        return self._png_host(self.mask_png, "mask PNG")

    def to_host(self, channels: int):
        """One device->host transfer; returns per-crop (image index, detection index, xywh, array)."""
        tot = self.checked_totals()
        k = tot[0]
        rects = self.rects[:k].cpu().numpy(); xywh = self.xywh[:k].cpu().numpy(); src = self.src[:k].cpu().numpy()
        offs = self.offsets[:k + 1].cpu().numpy(); pix = self.pixels[:tot[1]].cpu().numpy()
        cap = self.params.capacity
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
        tot = self.checked_totals(pixels=False, masks=True)
        k, ch = tot[0], self.params.channels
        rects = self.rects[:k].cpu().numpy()
        offs = self.offsets[:k + 1].cpu().numpy() // ch
        buf = self.masks[:tot[1] // ch].cpu().numpy()
        return [buf[offs[j]:offs[j + 1]].reshape(rects[j][3], rects[j][2]) for j in range(k)]

    def morphology_to_host(self):
        """The crops' morphology records as np.float64 [count, len(MORPHOLOGY_FIELDS)], crop order."""
        if self.morphology is None:
            raise MisoB200Error("no morphology: filter_and_crop ran without morphology=True")
        tot = self.checked_totals(pixels=False, masks=True)
        return self.morphology[:tot[0]].cpu().numpy()


def filter_and_crop(images: Sequence[Tensor], det_boxes: Tensor, det_scores: Tensor, det_counts: Tensor,
                    threshold: float, capacity_bytes: Optional[int] = None, boxes_are_xywh: bool = False,
                    mask_probs: Optional[Tensor] = None, paste_boxes: Optional[Tensor] = None, mask_threshold: float = 0.5,
                    mask_capacity_bytes: Optional[int] = None, morphology: bool = False, png: bool = False,
                    jpeg: bool = False) -> CropStage:
    """images[n]: uint8 [H, W, C] or [H, W] on the device (the ORIGINAL image pixels, as
    skimage.io.imread returns them); det_* as produced by postprocess_detections.

    mask_probs ([N, cap, M, M] or [N*cap, 1, M, M], Mask R-CNN's per-detection probabilities) adds each crop's instance
    mask (mb_crop_masks): paste_masks_in_image of the detection's mask into its image at paste_boxes (default
    det_boxes, xyxy), cut to the crop rectangle, 255 where > mask_threshold else 0. capacity_bytes = 0 skips the pixel
    gather; capacity_bytes / mask_capacity_bytes None size the buffers exactly (one host sync).

    morphology=True (needs mask_probs) also measures every crop's mask on the device (mb_mask_morphology): area,
    perimeter, centroid, axes, orientation, eccentricity, equivalent diameter and the mean of each channel over the
    mask, as regionprops computes them (MORPHOLOGY_FIELDS); CropStage.morphology / morphology_to_host().

    png=True also encodes every crop (and mask) as a lossless PNG file on the device (mb_png_encode):
    CropStage.png_to_host() / mask_png_to_host(). Images of 1..4 channels.

    jpeg=True also encodes every crop as a JPEG file on the device (mb_jpeg_encode), byte for byte the file PIL's
    Image.save writes with default settings: CropStage.jpeg_to_host(). Images of 1 or 3 channels."""
    if morphology and mask_probs is None:
        raise MisoB200Error("filter_and_crop(morphology=True) measures the instance masks: mask_probs is needed")
    n, cap = det_boxes.shape[0], det_boxes.shape[1]
    if len(images) != n:
        raise MisoB200Error("filter_and_crop: one image per detection row expected")
    keep = []
    for im in images:
        _require_cuda(im, "image")
        if im.dtype != torch.uint8:
            raise MisoB200Error("filter_and_crop: images must be uint8 (HWC)")
        keep.append(im.contiguous())
    ch = 1 if images[0].dim() == 2 else images[0].shape[2]
    stage = CropStage([im.shape[:2] for im in keep], ch, cap, threshold, det_boxes.device, boxes_are_xywh=boxes_are_xywh)
    stage.bind_images(keep)
    b, s = _f32c(det_boxes), _f32c(det_scores)
    st = _stream(b)
    cnt = det_counts.to(torch.int32).contiguous()
    stage.plan(b, s, cnt, st)
    if capacity_bytes is None or (mask_probs is not None and mask_capacity_bytes is None):
        need = int(stage.totals[1].item())          # exact size: costs one host sync
    stage.reserve(need if capacity_bytes is None else capacity_bytes)
    if mask_probs is not None:
        m = int(mask_probs.shape[-1])
        mp = _f32c(mask_probs)
        torch._assert(mp.numel() == n * cap * m * m and mp.shape[-2] == m, "mask_probs must be [N, cap, M, M] or [N*cap, 1, M, M]")
        pb = b if paste_boxes is None else _f32c(paste_boxes)
        torch._assert(pb.numel() == n * cap * 4, "paste_boxes must be [N, cap, 4]")
        stage.bind_masks(mp, pb, None, cap, mask_threshold, need // ch if mask_capacity_bytes is None else mask_capacity_bytes,
                         morphology)
    if png:
        stage.bind_png()
    if jpeg:
        stage.bind_jpeg()
    stage.cut(st)
    return stage

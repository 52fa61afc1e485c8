"""Drop-in wiring of the CUDA hot path into a loaded torchvision detection model (SURVEY.md §8 b2)
and, optionally, into the torch dispatcher (b1).

    model = torch.load("model.pt", weights_only=False).cuda().eval()
    miso_b200.patch.patch_model(model)          # FasterRCNN or MaskRCNN instance
    results = model(images)                     # same call, same return structure

Patched points (inference only — `model.training` falls through to the original code, which
needs autograd, the matcher and the samplers):
    model.rpn.forward                       anchors + decode + filter_proposals      -> mb_rpn_proposals
    model.roi_heads.box_roi_pool / mask_roi_pool   MultiScaleRoIAlign                -> mb_multiscale_roi_align
    model.roi_heads.postprocess_detections  softmax/decode/clip/filters/NMS/top-k    -> mb_det_postprocess
    model.transform.postprocess             resize_boxes + paste_masks_in_image      -> mb_resize_boxes, mb_paste_masks
    torchvision...roi_heads.maskrcnn_inference   sigmoid + per-label channel select  -> mb_mask_prob (Mask R-CNN only)
Hyper-parameters are read from the model instance at call time, never hard-coded.
"""
from __future__ import annotations

import types
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from . import detection, ops
from .detection import CPU_RULE_NUMEL, CUDA_RULE_NUMEL, DetConfig, RpnConfig

_RULES = {"cpu": CPU_RULE_NUMEL, "cuda": CUDA_RULE_NUMEL, "vanilla": -1}


class LazyProposals(list):
    """The reference's `list[Tensor]` of per-image proposals, backed by the fused RPN stage's fixed-capacity output
    ([N, R, 4] + device-side counts). The patched pooler and postprocess_detections read `.padded` / `.counts`
    directly, so a forward pass never waits for the counts; anything else that indexes or iterates the list
    materialises the per-image views (one host sync), exactly the reference's structure."""

    def __init__(self, padded: Tensor, counts: Tensor, scores: Optional[Tensor] = None):
        super().__init__()
        self.padded, self.counts, self.scores = padded, counts, scores
        self.materialised = False

    def _fill(self):
        if not self.materialised:
            cnt = self.counts.tolist()
            super().extend(self.padded[i, :c] for i, c in enumerate(cnt))
            self.materialised = True

    def __len__(self):
        return int(self.padded.shape[0])

    def __iter__(self):
        self._fill()
        return super().__iter__()

    def __getitem__(self, i):
        self._fill()
        return super().__getitem__(i)


def _rpn_forward(self, images, features: Dict[str, Tensor], targets=None):
    """RegionProposalNetwork.forward (tv:models/detection/rpn.py:336-387), eval branch."""
    if self.training:
        return self._miso_b200_orig_forward(images, features, targets)
    feats = list(features.values())
    objectness, pred_bbox_deltas = self.head(feats)
    cfg = RpnConfig.from_model(self, trick_numel=self._miso_b200_rule)
    out = detection.rpn_proposals(objectness, pred_bbox_deltas, images.image_sizes, tuple(images.tensors.shape[-2:]), cfg)
    return LazyProposals(out.proposals, out.counts, out.scores), {}     # list per image like the reference, without the sync


def _postprocess_detections(self, class_logits: Tensor, box_regression: Tensor, proposals: List[Tensor],
                            image_shapes: List[Tuple[int, int]]):
    """RoIHeads.postprocess_detections (tv:models/detection/roi_heads.py:680-737)."""
    cfg = DetConfig.from_model(self, trick_numel=self._miso_b200_rule)
    if isinstance(proposals, LazyProposals) and class_logits.shape[0] == proposals.padded.shape[0] * proposals.padded.shape[1]:
        # logits / regression rows are strided by the proposal capacity: the pooler ran on the padded layout (had somebody
        # iterated the list before pooling, the pooler would have produced the reference's packed rows instead)
        out = detection.postprocess_detections(class_logits, box_regression, proposals.padded, proposals.counts,
                                               image_shapes, cfg, packed=False)
    else:
        counts = [int(p.shape[0]) for p in proposals]
        padded = torch.nn.utils.rnn.pad_sequence(list(proposals), batch_first=True)       # [N, max R, 4], one op
        if padded.shape[1] == 0:
            padded = torch.zeros((len(counts), 1, 4), dtype=torch.float32, device=class_logits.device)
        cnt = torch.tensor(counts, dtype=torch.int32, device=class_logits.device)
        out = detection.postprocess_detections(class_logits, box_regression, padded.contiguous(), cnt, image_shapes, cfg, packed=True)
    dc = out.counts.tolist()                       # the forward pass's one host sync: the results are variable-length lists
    boxes = [out.boxes_net[i, :c] for i, c in enumerate(dc)]
    scores = [out.scores[i, :c] for i, c in enumerate(dc)]
    labels = [out.labels[i, :c] for i, c in enumerate(dc)]
    return boxes, scores, labels


def _transform_postprocess(self, result, image_shapes, original_image_sizes):
    """GeneralizedRCNNTransform.postprocess (tv:models/detection/transform.py:257-277)."""
    if self.training:
        return result
    if not all(pred["boxes"].is_cuda for pred in result):     # decided before anything is resized in place
        return self._miso_b200_orig_postprocess(result, image_shapes, original_image_sizes)
    for i, (pred, im_s, o_im_s) in enumerate(zip(result, image_shapes, original_image_sizes)):
        boxes = ops.resize_boxes(pred["boxes"], im_s, o_im_s)
        result[i]["boxes"] = boxes
        if "masks" in pred:
            result[i]["masks"] = ops.paste_masks_in_image(pred["masks"], boxes, o_im_s)
        if "keypoints" in pred:
            from torchvision.models.detection.transform import resize_keypoints
            result[i]["keypoints"] = resize_keypoints(pred["keypoints"], im_s, o_im_s)
    return result


def forward_uint8(model, images_u8: List[Tensor], paste_masks: bool = True):
    """GeneralizedRCNN.forward (tv:models/detection/generalized_rcnn.py:47-119, eval branch) for uint8 HWC CUDA
    images: ToTensor + normalize + resize + batch run as one kernel (ops.transform_images) instead of the
    reference's per-image tensor operations; everything downstream is the model's own (patched) code.
    paste_masks=False (Mask R-CNN): each result carries `mask_probs` [k, 1, M, M] (maskrcnn_inference's output) instead
    of the full-image `masks`, and no [k, 1, H, W] paste runs — for callers that cut the masks to crops
    (detection.filter_and_crop, mosaic.MosaicCrops.bind_masks)."""
    from torchvision.models.detection.image_list import ImageList
    tr = model.transform
    original_image_sizes = [(int(im.shape[0]), int(im.shape[1])) for im in images_u8]
    if getattr(tr, "fixed_size", None) is not None or getattr(tr, "_skip_resize", False):
        # the fused kernel implements the min_size / max_size rule only; the other two modes of
        # GeneralizedRCNNTransform (tv:models/detection/transform.py:160-183) run through the model's own transform
        # (torch ops on the device), so the result stays the reference's
        images, _ = tr([im.permute(2, 0, 1).to(torch.float32) / 255 for im in images_u8])
    else:
        batch, sizes = ops.transform_images(images_u8, tr.min_size[-1], tr.max_size, tr.image_mean, tr.image_std, tr.size_divisible)
        images = ImageList(batch, sizes)
    features = model.backbone(images.tensors)
    if isinstance(features, Tensor):
        features = {"0": features}
    proposals, _ = model.rpn(images, features)
    detections, _ = model.roi_heads(features, proposals, images.image_sizes)
    if not paste_masks:
        for d in detections:
            if "masks" in d:
                d["mask_probs"] = d.pop("masks")         # transform.postprocess pastes only a "masks" entry
    return tr.postprocess(detections, images.image_sizes, original_image_sizes)


def patch_model(model, exact_roi_align: bool = True, strategy_rule: str = "cpu", channels_last: bool = True):
    """Swap the post-head stages of a torchvision FasterRCNN / MaskRCNN instance for the CUDA
    path. strategy_rule picks which of torchvision's batched_nms switch-over rules the fused
    stages reproduce: "cpu" (numel > 4000, the reference CPU path = the parity oracle), "cuda"
    (numel > 100000) or "vanilla" (always per-class). channels_last moves the backbone + FPN to
    torch.channels_last: cuDNN then emits the pyramid in NHWC memory, which the RoIAlign kernel gathers in place
    (an NCHW pyramid costs a transpose of the maps per call). Returns the model."""
    if getattr(model, "_miso_b200_patched", False):
        return model
    if channels_last:
        model.backbone.to(memory_format=torch.channels_last)
    model._miso_b200_channels_last = bool(channels_last)
    rule = _RULES[strategy_rule]
    rpn, heads = model.rpn, model.roi_heads
    rpn._miso_b200_orig_forward = rpn.forward
    rpn._miso_b200_rule = rule
    rpn.forward = types.MethodType(_rpn_forward, rpn)
    heads._miso_b200_rule = rule
    heads._miso_b200_orig_postprocess = heads.postprocess_detections
    heads.postprocess_detections = types.MethodType(_postprocess_detections, heads)
    heads._miso_b200_orig_box_roi_pool = heads.box_roi_pool
    heads.box_roi_pool = ops.MultiScaleRoIAlign.from_torchvision(heads.box_roi_pool, exact=exact_roi_align)
    if getattr(heads, "mask_roi_pool", None) is not None:
        heads._miso_b200_orig_mask_roi_pool = heads.mask_roi_pool
        heads.mask_roi_pool = ops.MultiScaleRoIAlign.from_torchvision(heads.mask_roi_pool, exact=exact_roi_align)
    if getattr(heads, "mask_roi_pool", None) is not None:
        # RoIHeads.forward looks maskrcnn_inference up in its module at call time: route CUDA inputs to the fused kernel
        import torchvision.models.detection.roi_heads as tv_rh
        if not hasattr(tv_rh, "_miso_b200_orig_maskrcnn_inference"):
            tv_rh._miso_b200_orig_maskrcnn_inference = tv_rh.maskrcnn_inference

            def _maskrcnn_inference(x, labels):
                if x.is_cuda and getattr(tv_rh, "_miso_b200_fused_masks", 0) > 0:
                    return ops.maskrcnn_inference(x, labels)
                return tv_rh._miso_b200_orig_maskrcnn_inference(x, labels)
            tv_rh.maskrcnn_inference = _maskrcnn_inference
        tv_rh._miso_b200_fused_masks = getattr(tv_rh, "_miso_b200_fused_masks", 0) + 1      # patched models alive
        model._miso_b200_masks = True
    tr = model.transform
    tr._miso_b200_orig_postprocess = tr.postprocess
    tr.postprocess = types.MethodType(_transform_postprocess, tr)
    model._miso_b200_patched = True
    return model


def unpatch_model(model):
    if not getattr(model, "_miso_b200_patched", False):
        return model
    model.rpn.forward = model.rpn._miso_b200_orig_forward
    h = model.roi_heads
    h.postprocess_detections = h._miso_b200_orig_postprocess
    h.box_roi_pool = h._miso_b200_orig_box_roi_pool
    if hasattr(h, "_miso_b200_orig_mask_roi_pool"):
        h.mask_roi_pool = h._miso_b200_orig_mask_roi_pool
    if hasattr(model.transform, "_miso_b200_orig_postprocess"):
        model.transform.postprocess = model.transform._miso_b200_orig_postprocess
    if getattr(model, "_miso_b200_masks", False):
        import torchvision.models.detection.roi_heads as tv_rh
        tv_rh._miso_b200_fused_masks = max(getattr(tv_rh, "_miso_b200_fused_masks", 1) - 1, 0)
        model._miso_b200_masks = False
    if getattr(model, "_miso_b200_channels_last", False):
        model.backbone.to(memory_format=torch.contiguous_format)
    model._miso_b200_patched = False
    return model


_dispatch_lib: Optional["torch.library.Library"] = None


def override_torchvision_ops() -> None:
    """Operator-level drop-in (SURVEY.md §8 b1): route torchvision::nms and torchvision::roi_align
    for CUDA tensors through libmisob200, so unmodified callers (torchvision.ops.nms, batched_nms,
    roi_align, MultiScaleRoIAlign) use it. Autograd / autocast / meta registrations are untouched;
    only the CUDA forward kernels are replaced."""
    global _dispatch_lib
    if _dispatch_lib is not None:
        return
    import torchvision  # noqa: F401  (registers the op schemas)
    lib = torch.library.Library("torchvision", "IMPL")

    def nms_cuda(dets: Tensor, scores: Tensor, iou_threshold: float) -> Tensor:
        return ops.nms(dets, scores, iou_threshold)

    def roi_align_cuda(input: Tensor, rois: Tensor, spatial_scale: float, pooled_height: int, pooled_width: int,
                       sampling_ratio: int, aligned: bool) -> Tensor:
        return ops.roi_align(input, rois, (int(pooled_height), int(pooled_width)), spatial_scale, sampling_ratio, aligned)

    def roi_align_backward_cuda(grad: Tensor, rois: Tensor, spatial_scale: float, pooled_height: int, pooled_width: int,
                                batch_size: int, channels: int, height: int, width: int, sampling_ratio: int, aligned: bool) -> Tensor:
        return ops.roi_align_backward(grad, rois, spatial_scale, int(pooled_height), int(pooled_width), int(batch_size),
                                      int(channels), int(height), int(width), sampling_ratio, aligned)

    lib.impl("nms", nms_cuda, "CUDA", allow_override=True)
    lib.impl("roi_align", roi_align_cuda, "CUDA", allow_override=True)
    lib.impl("_roi_align_backward", roi_align_backward_cuda, "CUDA", allow_override=True)   # training: torchvision's autograd node calls it
    _dispatch_lib = lib

"""torchvision-signature operators backed by libmisob200.so (sm_100a CUDA, C ABI).

Same names, argument meaning, defaults and error behaviour as the operators the reference's
pipelines call (SURVEY.md §8 b1):

    nms(boxes, scores, iou_threshold)                         tv:ops/boxes.py:20-48
    batched_nms(boxes, scores, idxs, iou_threshold)           tv:ops/boxes.py:51-83
    roi_align(input, boxes, output_size, spatial_scale=1.0,
              sampling_ratio=-1, aligned=False)               tv:ops/roi_align.py:203-260
    box_convert(boxes, in_fmt, out_fmt)                       tv:ops/boxes.py:185-270
    clip_boxes_to_image / remove_small_boxes                  tv:ops/boxes.py:149-182, :123-146
    MultiScaleRoIAlign                                        tv:ops/poolers.py:230-327

Inputs are borrowed CUDA tensors, outputs are fresh tensors on the same device, all work is
enqueued on torch's current stream. There is no CPU path: a CPU tensor raises.
"""
from __future__ import annotations

import ctypes as C
import functools
import math
from typing import Dict, List, Optional, Sequence, Tuple, Union

import torch
from torch import Tensor

from . import _lib
from ._lib import MisoB200Error, RoiAlignParams

_FMT = {"xyxy": 0, "xywh": 1, "cxcywh": 2}


# ------------------------------------------------------------------------------------------
# plumbing
# ------------------------------------------------------------------------------------------
def _stream(t: Union[Tensor, torch.device, torch.cuda.Stream]) -> C.c_void_p:
    """The handle of stream `t`, or of torch's current stream on the device of tensor / device `t`."""
    if isinstance(t, torch.cuda.Stream):
        return C.c_void_p(t.cuda_stream)
    return C.c_void_p(torch.cuda.current_stream(t if isinstance(t, torch.device) else t.device).cuda_stream)


def _ptr(t: Optional[Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None or t.numel() == 0 else t.data_ptr())


def _require_cuda(t: Tensor, what: str) -> None:
    if not isinstance(t, Tensor):
        raise TypeError(f"{what} must be a Tensor")
    if t.device.type != "cuda":
        raise MisoB200Error(f"{what} is on {t.device}; miso_b200 runs on CUDA (sm_100a) only — no CPU fallback")


def _f32c(t: Tensor) -> Tensor:
    return t.detach().to(torch.float32).contiguous()


def _workspace(nbytes: int, device) -> Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


# ------------------------------------------------------------------------------------------
# NMS
# ------------------------------------------------------------------------------------------
_MASK_FIRST_TRY_BYTES = 256 << 20


def _nms_impl(boxes: Tensor, scores: Tensor, groups: Optional[Tensor], num_groups: int, mode: int,
              iou_threshold: float) -> Tensor:
    lib = _lib.load()
    k = boxes.shape[0]
    dev = boxes.device
    if k == 0:
        return torch.empty((0,), dtype=torch.int64, device=dev)
    boxes, scores = _f32c(boxes), _f32c(scores)
    if groups is not None:
        groups = groups.detach().to(torch.int64).contiguous()
    keep = torch.empty((k,), dtype=torch.int64, device=dev)
    status = torch.empty((4,), dtype=torch.int64, device=dev)
    ws_bytes = lib.mb_nms_workspace_bytes(k, num_groups)
    ws = _workspace(ws_bytes, dev)
    exact_words = k * ((k + 63) // 64)
    mask_bytes = exact_words * 8
    if mode == 1 and mask_bytes > _MASK_FIRST_TRY_BYTES:
        mask_bytes = _MASK_FIRST_TRY_BYTES      # per-group masks are usually far below the bound
    for _ in range(2):
        mask = _workspace(mask_bytes, dev)
        rc = lib.mb_nms(_ptr(boxes), _ptr(scores), _ptr(groups), k, num_groups, mode, float(iou_threshold),
                        _ptr(keep), _ptr(status), _ptr(ws), ws.numel(), _ptr(mask), mask.numel(), _stream(boxes))
        _lib.check(rc, "mb_nms")
        st = status.tolist()                     # the one host sync: output length is data-dependent
        if st[0] >= 0:
            return keep[: st[0]]
        if st[0] == -2:
            raise MisoB200Error("batched_nms: group index outside [0, num_groups)")
        mask_bytes = st[1] * 8                   # mask workspace was too small: retry with the exact size
    raise MisoB200Error("mb_nms: mask workspace negotiation failed")


class PreparedBatchedNms:
    """Fixed-capacity, sync-free per-category NMS: workspaces and outputs are allocated once, rows
    whose category is negative are ignored (padding), the kept indices and their count stay on
    the device. Used for the cross-tile seam NMS right behind the NCCL all-gather."""

    def __init__(self, capacity: int, num_groups: int, device):
        self.lib = _lib.load()
        self.k, self.g = int(capacity), int(num_groups)
        self.keep = torch.empty((self.k,), dtype=torch.int64, device=device)
        self.status = torch.zeros((4,), dtype=torch.int64, device=device)
        self.ws = _workspace(self.lib.mb_nms_workspace_bytes(self.k, self.g), device)
        self.mask = _workspace(self.k * ((self.k + 63) // 64) * 8, device)     # exact single-segment bound

    def __call__(self, boxes: Tensor, scores: Tensor, groups: Tensor, iou_threshold: float):
        """boxes [K,4] fp32, scores [K] fp32, groups [K] int64 (negative = ignore), all contiguous.
        Returns (keep, status) device tensors: status[0] = number kept (no host sync here)."""
        rc = self.lib.mb_nms(_ptr(boxes), _ptr(scores), _ptr(groups), self.k, self.g, 1, float(iou_threshold),
                             _ptr(self.keep), _ptr(self.status), _ptr(self.ws), self.ws.numel(), _ptr(self.mask),
                             self.mask.numel(), _stream(boxes))
        _lib.check(rc, "mb_nms")
        return self.keep, self.status


def nms(boxes: Tensor, scores: Tensor, iou_threshold: float) -> Tensor:
    """Greedy NMS; int64 indices of kept boxes in descending score order (ties: lower index
    first). Semantics of the torchvision CPU kernel: fp32 IoU, `(double)iou > iou_threshold`."""
    _require_cuda(boxes, "boxes")
    _require_cuda(scores, "scores")
    torch._assert(boxes.dim() == 2 and boxes.shape[1] == 4, f"boxes should be a 2d tensor of shape [N, 4], got {boxes.shape}")
    torch._assert(scores.dim() == 1 and scores.shape[0] == boxes.shape[0], "boxes and scores should have same number of elements")
    return _nms_impl(boxes, scores, None, 1, 0, iou_threshold)


def _batched_nms_coordinate_trick(boxes: Tensor, scores: Tensor, idxs: Tensor, iou_threshold: float) -> Tensor:
    """tv:ops/boxes.py:86-103 — offsets fl(fl(idx) * fl(max + 1)) added in fp32 on the device."""
    if boxes.numel() == 0:
        return torch.empty((0,), dtype=torch.int64, device=boxes.device)
    return _nms_impl(boxes, scores, idxs, 1, 2, iou_threshold)


def _batched_nms_vanilla(boxes: Tensor, scores: Tensor, idxs: Tensor, iou_threshold: float) -> Tensor:
    """tv:ops/boxes.py:106-120 — independent NMS per category on raw coordinates; the union is
    ordered by (score desc, index asc) (the reference's final sort leaves ties unspecified)."""
    if boxes.numel() == 0:
        return torch.empty((0,), dtype=torch.int64, device=boxes.device)
    lo, hi = (int(v) for v in torch.aminmax(idxs))
    if lo < 0 or hi >= 65536:
        # arbitrary category values: densify them (rare; categories are labels or levels)
        idxs = torch.unique(idxs, return_inverse=True)[1]
        hi = int(idxs.max())
    return _nms_impl(boxes, scores, idxs, hi + 1, 1, iou_threshold)


def batched_nms(boxes: Tensor, scores: Tensor, idxs: Tensor, iou_threshold: float, strategy: str = "auto") -> Tensor:
    """Per-category NMS. `strategy="auto"` applies torchvision's own rule for CUDA tensors
    (tv:ops/boxes.py:80: vanilla iff numel > 100000), "cpu_rule" the CPU rule (> 4000);
    "vanilla" / "trick" force one strategy so that both sides of a parity test run the same one."""
    _require_cuda(boxes, "boxes")
    _require_cuda(scores, "scores")
    _require_cuda(idxs, "idxs")
    if strategy == "auto":
        strategy = "vanilla" if boxes.numel() > 100_000 else "trick"
    elif strategy == "cpu_rule":
        strategy = "vanilla" if boxes.numel() > 4000 else "trick"
    if strategy == "vanilla":
        return _batched_nms_vanilla(boxes, scores, idxs, iou_threshold)
    if strategy == "trick":
        return _batched_nms_coordinate_trick(boxes, scores, idxs, iou_threshold)
    raise ValueError(f"unknown batched_nms strategy {strategy!r}")


# ------------------------------------------------------------------------------------------
# element-wise box operators
# ------------------------------------------------------------------------------------------
def box_convert(boxes: Tensor, in_fmt: str, out_fmt: str) -> Tensor:
    allowed = ("xyxy", "xywh", "cxcywh")
    if in_fmt not in allowed or out_fmt not in allowed:
        raise ValueError("Unsupported Bounding Box Conversions for given in_fmt and out_fmt")
    _require_cuda(boxes, "boxes")
    if in_fmt == out_fmt:
        return boxes.clone()
    b = _f32c(boxes)
    out = torch.empty_like(b)
    n = b.numel() // 4
    _lib.check(_lib.load().mb_box_convert(_ptr(b), n, _FMT[in_fmt], _FMT[out_fmt], _ptr(out), _stream(b)), "mb_box_convert")
    return out.to(boxes.dtype)


def clip_boxes_to_image(boxes: Tensor, size: Tuple[int, int]) -> Tensor:
    _require_cuda(boxes, "boxes")
    b = _f32c(boxes)
    out = torch.empty_like(b)
    h, w = size
    _lib.check(_lib.load().mb_clip_boxes(_ptr(b), b.numel() // 4, float(h), float(w), _ptr(out), _stream(b)), "mb_clip_boxes")
    return out.to(boxes.dtype)


def remove_small_boxes(boxes: Tensor, min_size: float) -> Tensor:
    _require_cuda(boxes, "boxes")
    b = _f32c(boxes).reshape(-1, 4)
    n = b.shape[0]
    keep = torch.empty((n,), dtype=torch.int64, device=b.device)
    cnt = torch.zeros((1,), dtype=torch.int64, device=b.device)
    _lib.check(_lib.load().mb_remove_small(_ptr(b), n, float(min_size), _ptr(keep), _ptr(cnt), _stream(b)), "mb_remove_small")
    return keep[: int(cnt.item())]


def decode_boxes(rel_codes: Tensor, boxes: Union[Tensor, Sequence[Tensor]], weights: Sequence[float],
                 bbox_xform_clip: float = math.log(1000.0 / 16)) -> Tensor:
    """BoxCoder.decode (tv:models/detection/_utils.py:162-224): rel_codes [M, 4C] -> [M, C, 4]."""
    if isinstance(boxes, (list, tuple)):
        boxes = torch.cat(list(boxes), dim=0)
    _require_cuda(rel_codes, "rel_codes")
    _require_cuda(boxes, "boxes")
    b = _f32c(boxes)
    m = b.shape[0]
    r = _f32c(rel_codes).reshape(m, -1) if m > 0 else _f32c(rel_codes)
    c = r.shape[1] // 4 if m > 0 else 1
    out = torch.empty((m, c, 4), dtype=torch.float32, device=b.device)
    wx, wy, ww, wh = (float(v) for v in weights)
    _lib.check(_lib.load().mb_box_decode(_ptr(r), _ptr(b), m, c, wx, wy, ww, wh, float(bbox_xform_clip), _ptr(out),
                                         _stream(b)), "mb_box_decode")
    return out


def resize_boxes(boxes: Tensor, original_size: Sequence[int], new_size: Sequence[int]) -> Tensor:
    """tv:models/detection/transform.py:306-319 (ratios are fp32 quotients of fp32 sizes)."""
    _require_cuda(boxes, "boxes")
    rh = (torch.tensor(new_size[0], dtype=torch.float32) / torch.tensor(original_size[0], dtype=torch.float32)).item()
    rw = (torch.tensor(new_size[1], dtype=torch.float32) / torch.tensor(original_size[1], dtype=torch.float32)).item()
    b = _f32c(boxes)
    out = torch.empty_like(b)
    _lib.check(_lib.load().mb_resize_boxes(_ptr(b), b.numel() // 4, rh, rw, _ptr(out), _stream(b)), "mb_resize_boxes")
    return out


def paste_masks_in_image(masks: Tensor, boxes: Tensor, img_shape: Tuple[int, int], padding: int = 1) -> Tensor:
    """tv:models/detection/roi_heads.py:490-501 — [R, 1, M, M] mask probabilities + [R, 4] boxes (image
    coordinates) -> [R, 1, H, W] fp32: every mask padded, bilinearly resized to its (expanded, integer)
    box and pasted into a zero image. One launch instead of a Python loop per detection."""
    _require_cuda(masks, "masks")
    _require_cuda(boxes, "boxes")
    torch._assert(masks.dim() == 4 and masks.shape[1] == 1 and masks.shape[2] == masks.shape[3],
                  f"masks should be [R, 1, M, M], got {tuple(masks.shape)}")
    torch._assert(boxes.dim() == 2 and boxes.shape[1] == 4 and boxes.shape[0] == masks.shape[0], "boxes should be [R, 4]")
    im_h, im_w = int(img_shape[0]), int(img_shape[1])
    r, m = int(masks.shape[0]), int(masks.shape[-1])
    out = torch.empty((r, 1, im_h, im_w), dtype=torch.float32, device=masks.device)
    if r == 0:
        return out.to(masks.dtype)
    mk, bx = _f32c(masks), _f32c(boxes)
    rc = _lib.load().mb_paste_masks(_ptr(mk), _ptr(bx), r, m, int(padding), im_h, im_w, _ptr(out), _stream(masks))
    _lib.check(rc, "mb_paste_masks")
    return out.to(masks.dtype)


def resized_image_size(h: int, w: int, min_size: int, max_size: int) -> Tuple[int, int]:
    """Output size of GeneralizedRCNNTransform.resize in eval mode (tv:models/detection/transform.py:23-70):
    scale factor = min(min_size / min(h, w), max_size / max(h, w)), then F.interpolate(recompute_scale_factor=
    True): floor(size * scale_factor), all in Python floats."""
    # eager (non-scripted) torchvision 0.26 computes the factor with Python ints/floats (double precision)
    sf = min(float(min_size) / min(h, w), float(max_size) / max(h, w))
    return int(math.floor(float(h) * sf)), int(math.floor(float(w) * sf))


def transform_images(images_u8: Sequence[Tensor], min_size: int, max_size: int, image_mean: Sequence[float],
                     image_std: Sequence[float], size_divisible: int = 32) -> Tuple[Tensor, List[Tuple[int, int]]]:
    """ToTensor + GeneralizedRCNNTransform.forward (normalize, bilinear resize, zero-padded batch) for uint8
    HWC CUDA images in ONE launch. Returns (batch [N, C, H_pad, W_pad] fp32, resized image sizes) — the
    fields of the reference's ImageList."""
    torch._assert(len(images_u8) > 0, "transform_images: at least one image")
    n, c = len(images_u8), int(images_u8[0].shape[2])
    p = _lib.TransformParams()
    p.num_images, p.channels = n, c
    sizes, keep = [], []
    for i, im in enumerate(images_u8):
        _require_cuda(im, "images")
        torch._assert(im.dtype == torch.uint8 and im.dim() == 3 and im.shape[2] == c, "uint8 HWC images expected")
        imc = im.contiguous()
        keep.append(imc)
        h, w = int(im.shape[0]), int(im.shape[1])
        oh, ow = resized_image_size(h, w, min_size, max_size)
        p.images[i], p.in_h[i], p.in_w[i], p.out_h[i], p.out_w[i] = imc.data_ptr(), h, w, oh, ow
        sizes.append((oh, ow))
    for j in range(c):
        p.mean[j], p.std[j] = float(image_mean[j]), float(image_std[j])
    d = float(size_divisible)
    p.pad_h = int(math.ceil(max(s[0] for s in sizes) / d) * d)
    p.pad_w = int(math.ceil(max(s[1] for s in sizes) / d) * d)
    out = torch.empty((n, c, p.pad_h, p.pad_w), dtype=torch.float32, device=images_u8[0].device)
    _lib.check(_lib.load().mb_image_transform(C.byref(p), _ptr(out), _stream(out)), "mb_image_transform")
    return out, sizes


def base_anchors(scales: Sequence[float], aspect_ratios: Sequence[float]) -> Tensor:
    """AnchorGenerator.generate_anchors (tv:models/detection/anchor_utils.py:58-74), host side."""
    scales_t = torch.as_tensor(scales, dtype=torch.float32)
    ar = torch.as_tensor(aspect_ratios, dtype=torch.float32)
    h_ratios = torch.sqrt(ar)
    w_ratios = 1 / h_ratios
    ws = (w_ratios[:, None] * scales_t[None, :]).view(-1)
    hs = (h_ratios[:, None] * scales_t[None, :]).view(-1)
    return (torch.stack([-ws, -hs, ws, hs], dim=1) / 2).round()


def grid_anchors(base: Tensor, grid_size: Sequence[int], stride: Sequence[int], device) -> Tensor:
    """One level of AnchorGenerator.grid_anchors: [(H*W*A), 4] in (h, w, a) order."""
    gh, gw = int(grid_size[0]), int(grid_size[1])
    a = base.shape[0]
    out = torch.empty((gh * gw * a, 4), dtype=torch.float32, device=device)
    host = (C.c_float * (4 * a))(*[float(v) for v in base.reshape(-1).tolist()])
    _lib.check(_lib.load().mb_grid_anchors(host, a, gh, gw, int(stride[0]), int(stride[1]), _ptr(out), _stream(out)),
               "mb_grid_anchors")
    return out


# ------------------------------------------------------------------------------------------
# RoIAlign
# ------------------------------------------------------------------------------------------
def _pair(v) -> Tuple[int, int]:
    return (int(v), int(v)) if isinstance(v, int) else (int(v[0]), int(v[1]))


def check_roi_boxes_shape(boxes: Union[Tensor, Sequence[Tensor]]) -> None:
    """tv:ops/_utils.py:28-38."""
    if isinstance(boxes, (list, tuple)):
        for b in boxes:
            torch._assert(b.dim() == 2 and b.size(1) == 4,
                          "The shape of the tensor in the boxes list is not correct as List[Tensor[L, 4]]")
    elif isinstance(boxes, Tensor):
        torch._assert(boxes.dim() == 2 and boxes.size(1) == 5, "The boxes tensor shape is not correct as Tensor[K, 5]")
    else:
        torch._assert(False, "boxes is expected to be a Tensor[L, 5] or a List[Tensor[K, 4]]")


def convert_boxes_to_roi_format(boxes: Sequence[Tensor]) -> Tensor:
    """tv:ops/_utils.py:18-25 / tv:ops/poolers.py:87-95: [K,5] = (batch index, x1, y1, x2, y2)."""
    concat = torch.cat(list(boxes), dim=0)
    ids = torch.cat([torch.full_like(b[:, :1], i) for i, b in enumerate(boxes)], dim=0)
    return torch.cat([ids, concat], dim=1)


def is_channels_last(t: Tensor) -> bool:
    """A 4-d map stored channels-last (what a torch.channels_last backbone produces), not also NCHW-contiguous."""
    return not t.is_contiguous() and t.is_contiguous(memory_format=torch.channels_last)


def roi_align_reads_channels_last(channels: int, output_size: Tuple[int, int], sampling_ratio: int,
                                  dtype: torch.dtype = torch.float32) -> bool:
    """Whether mb_multiscale_roi_align can gather from channels-last maps in place: fp32 maps with more than one
    channel, sampling ratio 2 and pooled sides <= 16. The library rejects channels-last maps outside this envelope
    (MB_ERR_UNSUPPORTED), so they need an NCHW copy."""
    return (int(sampling_ratio) == 2 and int(output_size[0]) <= 16 and int(output_size[1]) <= 16 and int(channels) > 1
            and dtype == torch.float32)


def roi_align_params(feature_grids: Sequence[Tuple[int, int]], num_images: int, channels: int, output_size: Tuple[int, int],
                     sampling_ratio: int, scales: Sequence[float], thresholds: Sequence[float], aligned: bool = False,
                     exact: bool = True, channels_last: bool = False, boxes_per_image: int = 0) -> RoiAlignParams:
    """mb_multiscale_roi_align's parameters for maps of the given (H, W) per level, without the map and count
    pointers. scales / thresholds: pooler_levels(). boxes_per_image > 0 selects the [N, R, 4] + box_counts layout."""
    p = RoiAlignParams()
    p.num_levels, p.num_images, p.channels = len(feature_grids), int(num_images), int(channels)
    p.pooled_h, p.pooled_w, p.sampling_ratio = int(output_size[0]), int(output_size[1]), int(sampling_ratio)
    p.aligned, p.exact, p.channels_last = int(bool(aligned)), int(bool(exact)), int(bool(channels_last))
    for l, (h, w) in enumerate(feature_grids):
        p.height[l], p.width[l], p.spatial_scale[l] = int(h), int(w), float(scales[l])
    for l, t in enumerate(thresholds):
        p.level_thresholds[l] = float(t)
    p.boxes_per_image = int(boxes_per_image)
    return p


def _roi_align_launch(features: Sequence[Tensor], rois: Tensor, scales: Sequence[float], thresholds: Sequence[float],
                      output_size: Tuple[int, int], sampling_ratio: int, aligned: bool, exact: bool,
                      return_levels: bool = False, use_workspace: bool = True, force_gather: bool = False,
                      box_counts: Optional[Tensor] = None):
    """rois: [K, 5] (batch, x1, y1, x2, y2), or — with box_counts [N] int32 — the fused path's [N, R, 4] layout
    (batch index = row // R, rows beyond an image's count produce zeros; no host sync, no RoI tensor is built)."""
    lib = _lib.load()
    f0 = features[0]
    per_image = 0
    if box_counts is not None:
        torch._assert(rois.dim() == 3 and rois.shape[2] == 4 and rois.shape[0] == f0.shape[0] and
                      box_counts.dtype == torch.int32 and box_counts.is_contiguous(), "padded RoIs: [N, R, 4] + int32 counts [N]")
        per_image = int(rois.shape[1])
        rois = rois.reshape(-1, 4)
    k = rois.shape[0]
    n, c = f0.shape[0], f0.shape[1]
    ph, pw = output_size
    out = torch.empty((k, c, ph, pw), dtype=torch.float32, device=f0.device)
    levels = torch.empty((k,), dtype=torch.int32, device=f0.device) if return_levels else None
    if k > 0:
        nhwc = (all(f.dtype == f0.dtype and is_channels_last(f) for f in features) and
                roi_align_reads_channels_last(c, output_size, sampling_ratio, f0.dtype))
        keepalive = []
        for f in features:
            torch._assert(f.shape[0] == n and f.shape[1] == c, "all feature maps must share batch and channel sizes")
            keepalive.append(f.detach() if nhwc else _f32c(f))
        p = roi_align_params([fc.shape[2:] for fc in keepalive], n, c, output_size, sampling_ratio, scales, thresholds,
                             aligned, exact, nhwc, per_image)
        p.force_gather = {False: 0, True: 1, 0: 0, 1: 1, 2: 2, 'auto': 0, 'gather': 1, 'tma': 2}[force_gather]
        if per_image:
            p.box_counts = box_counts.data_ptr()
        for i, fc in enumerate(keepalive):
            p.features[i] = fc.data_ptr()
        ws_bytes = lib.mb_roi_align_workspace_bytes(C.byref(p), k) if use_workspace else 0
        ws = _workspace(ws_bytes, f0.device) if ws_bytes else None
        rc = lib.mb_multiscale_roi_align(C.byref(p), _ptr(rois), k, _ptr(out), _ptr(levels), _ptr(ws),
                                         ws.numel() if ws is not None else 0, _stream(f0))
        _lib.check(rc, "mb_multiscale_roi_align")
    return (out, levels) if return_levels else out


def roi_align(input: Tensor, boxes: Union[Tensor, Sequence[Tensor]], output_size, spatial_scale: float = 1.0,
              sampling_ratio: int = -1, aligned: bool = False, exact: bool = True, force_gather: bool = False) -> Tensor:
    """RoIAlign forward; `exact=True` reproduces the CPU kernel's fp32 operation order bit for bit.
    `force_gather`: route for channels-last maps — "auto"/False (library default = "gather"), "gather"/True (register-gather
    kernel), "tma" (TMA-staged kernel); identical results."""
    _require_cuda(input, "input")
    check_roi_boxes_shape(boxes)
    rois = boxes if isinstance(boxes, Tensor) else convert_boxes_to_roi_format(boxes)
    _require_cuda(rois, "boxes")
    out = _roi_align_launch([input], _f32c(rois), [spatial_scale], [], _pair(output_size), sampling_ratio, aligned, exact,
                            force_gather=force_gather)
    return out.to(input.dtype)


@functools.lru_cache(maxsize=None)
def level_thresholds(k_min: int, k_max: int, canonical_scale: int = 224, canonical_level: int = 4,
                     eps: float = 1e-6) -> Tuple[float, ...]:
    """LevelMapper (tv:ops/poolers.py:73-84) as area thresholds: entry i is the smallest fp32
    box area that the mapper sends to a level > i. Found by bisection over fp32 bit patterns,
    evaluating the mapper's own formula with torch CPU fp32 ops (host-side setup, once per
    pooler configuration); the mapper is monotone in the area (SURVEY.md §7)."""
    def mapped(bits: int) -> int:
        area = torch.tensor([bits] * 16, dtype=torch.int32).view(torch.float32)
        s = torch.sqrt(area)
        t = torch.floor(canonical_level + torch.log2(s / canonical_scale) + torch.tensor(eps, dtype=s.dtype))
        t = torch.clamp(t, min=k_min, max=k_max)
        return int((t.to(torch.int64) - k_min)[0])

    out = []
    for lvl in range(1, k_max - k_min + 1):
        lo, hi = 0x00800000, 0x7F7FFFFF          # smallest normal .. largest finite
        while lo < hi:                            # first bit pattern with mapped >= lvl
            mid = (lo + hi) // 2
            if mapped(mid) >= lvl:
                hi = mid
            else:
                lo = mid + 1
        out.append(torch.tensor([lo], dtype=torch.int32).view(torch.float32).item())
    return tuple(out)


def infer_scale(feature_shape: Sequence[int], original_size: Sequence[int]) -> float:
    """_infer_scale (tv:ops/poolers.py:98-106)."""
    approx_scale = float(feature_shape[-2]) / float(original_size[0])
    return 2 ** float(torch.tensor(approx_scale).log2().round())


def pooler_levels(feature_grids: Sequence[Sequence[int]], image_sizes: Sequence[Tuple[int, int]],
                  canonical_scale: int = 224, canonical_level: int = 4) -> Tuple[List[float], Tuple[float, ...]]:
    """_setup_scales (tv:ops/poolers.py:110-134): the spatial scale of each pooler level (feature_grids: its (H, W),
    or any shape ending in them) and the LevelMapper's area thresholds (none for a single level)."""
    if not image_sizes:
        raise ValueError("images list should not be empty")
    max_x = max(s[0] for s in image_sizes)
    max_y = max(s[1] for s in image_sizes)
    scales = [infer_scale(g, (max_x, max_y)) for g in feature_grids]
    k_min = int(-math.log2(scales[0]))
    k_max = int(-math.log2(scales[-1]))
    thresholds = level_thresholds(k_min, k_max, canonical_scale, canonical_level) if len(scales) > 1 else ()
    return scales, thresholds


class MultiScaleRoIAlign(torch.nn.Module):
    """Drop-in for torchvision.ops.MultiScaleRoIAlign (tv:ops/poolers.py:230-327): same
    constructor and forward(x, boxes, image_shapes); one CUDA launch for all levels."""

    def __init__(self, featmap_names: List[str], output_size, sampling_ratio: int, *, canonical_scale: int = 224,
                 canonical_level: int = 4, exact: bool = True, force_gather: bool = False):
        super().__init__()
        self.force_gather = force_gather
        self.featmap_names = list(featmap_names)
        self.output_size = _pair(output_size)
        self.sampling_ratio = int(sampling_ratio)
        self.canonical_scale = canonical_scale
        self.canonical_level = canonical_level
        self.exact = exact
        self.scales: Optional[List[float]] = None
        self.thresholds: Optional[Tuple[float, ...]] = None

    @classmethod
    def from_torchvision(cls, pooler, exact: bool = True) -> "MultiScaleRoIAlign":
        return cls(pooler.featmap_names, tuple(pooler.output_size), pooler.sampling_ratio,
                   canonical_scale=pooler.canonical_scale, canonical_level=pooler.canonical_level, exact=exact)

    def _setup(self, features: List[Tensor], image_shapes: List[Tuple[int, int]]) -> None:
        """_setup_scales (tv:ops/poolers.py:110-134); cached after the first call like the reference."""
        self.scales, self.thresholds = pooler_levels([f.shape for f in features], image_shapes, self.canonical_scale,
                                                     self.canonical_level)

    def forward(self, x: Dict[str, Tensor], boxes: List[Tensor], image_shapes: List[Tuple[int, int]],
                return_levels: bool = False):
        feats = [v for k, v in x.items() if k in self.featmap_names]
        for f in feats:
            _require_cuda(f, "feature map")
        if self.scales is None or self.thresholds is None:
            self._setup(feats, image_shapes)
        padded = getattr(boxes, "padded", None)
        if padded is not None and not getattr(boxes, "materialised", True):
            # the fused RPN stage's [N, R, 4] + counts (patch.LazyProposals): pooled in place, no host sync; the
            # output has N*R rows (rows beyond an image's count are zero and ignored downstream)
            return _roi_align_launch(feats, _f32c(padded), self.scales, self.thresholds, self.output_size, self.sampling_ratio,
                                     False, self.exact, return_levels, force_gather=self.force_gather, box_counts=boxes.counts)
        rois = _f32c(convert_boxes_to_roi_format(boxes))
        return _roi_align_launch(feats, rois, self.scales, self.thresholds, self.output_size, self.sampling_ratio,
                                 False, self.exact, return_levels, force_gather=self.force_gather)


# ------------------------------------------------------------------------------------------
# training-side siblings (SURVEY.md §8f row 4)
# ------------------------------------------------------------------------------------------
def box_iou(boxes1: Tensor, boxes2: Tensor) -> Tensor:
    """torchvision.ops.box_iou (tv:ops/boxes.py:299-330): [N,4] x [M,4] -> [N,M], the reference's operation order."""
    _require_cuda(boxes1, "boxes1")
    _require_cuda(boxes2, "boxes2")
    b1, b2 = _f32c(boxes1), _f32c(boxes2)
    out = torch.empty((b1.shape[0], b2.shape[0]), dtype=torch.float32, device=b1.device)
    _lib.check(_lib.load().mb_box_iou(_ptr(b1), b1.shape[0], _ptr(b2), b2.shape[0], _ptr(out), _stream(b1)), "mb_box_iou")
    return out


def match_and_encode(gt_boxes: Tensor, anchors: Tensor, high_threshold: float, low_threshold: float,
                     allow_low_quality_matches: bool, weights: Sequence[float], return_targets: bool = True):
    """Matcher(box_iou(gt_boxes, anchors)) + BoxCoder.encode_single(gt_boxes[matches.clamp(min=0)], anchors) in two
    launches, without the [M, N] IoU matrix (tv:models/detection/_utils.py:345-426, :85-127; call sites
    rpn.py:193-229, roi_heads.py:580-614). Returns (matches int64 [N], matched_vals [N], targets [N,4] or None)."""
    _require_cuda(gt_boxes, "gt_boxes")
    _require_cuda(anchors, "anchors")
    if gt_boxes.shape[0] == 0:
        raise ValueError("No ground-truth boxes available for one of the images during training")   # Matcher's own error
    g, a = _f32c(gt_boxes), _f32c(anchors)
    n = a.shape[0]
    lib = _lib.load()
    matches = torch.empty((n,), dtype=torch.int64, device=a.device)
    vals = torch.empty((n,), dtype=torch.float32, device=a.device)
    targets = torch.empty((n, 4), dtype=torch.float32, device=a.device) if return_targets else None
    ws = _workspace(lib.mb_match_encode_workspace_bytes(g.shape[0], n), a.device)
    wx, wy, ww, wh = (float(v) for v in weights)
    _lib.check(lib.mb_match_encode(_ptr(g), g.shape[0], _ptr(a), n, float(high_threshold), float(low_threshold),
                                   int(bool(allow_low_quality_matches)), wx, wy, ww, wh, _ptr(matches), _ptr(vals), _ptr(targets),
                                   _ptr(ws), ws.numel(), _stream(a)), "mb_match_encode")
    return matches, vals, targets


def roi_align_backward(grad: Tensor, rois: Tensor, spatial_scale: float, pooled_height: int, pooled_width: int, batch_size: int,
                       channels: int, height: int, width: int, sampling_ratio: int, aligned: bool) -> Tensor:
    """torchvision::_roi_align_backward (same argument order as the dispatcher schema): grad [K,C,PH,PW] -> [B,C,H,W]."""
    _require_cuda(grad, "grad")
    g, r = _f32c(grad), _f32c(rois)
    out = torch.empty((batch_size, channels, height, width), dtype=torch.float32, device=g.device)
    _lib.check(_lib.load().mb_roi_align_backward(_ptr(g), _ptr(r), r.shape[0], float(spatial_scale), int(channels), int(height),
                                                 int(width), int(pooled_height), int(pooled_width), int(sampling_ratio),
                                                 int(bool(aligned)), int(batch_size), _ptr(out), _stream(g)), "mb_roi_align_backward")
    return out.to(grad.dtype)


def maskrcnn_inference(x: Tensor, labels: List[Tensor]) -> List[Tensor]:
    """tv:models/detection/roi_heads.py:56-82: per image the [R_i, 1, M, M] probabilities of the predicted classes, from
    the mask head's logits [sum R, C, M, M] — one launch that touches only the selected channels."""
    _require_cuda(x, "mask logits")
    torch._assert(x.dim() == 4 and x.shape[2] == x.shape[3], "mask logits should be [R, C, M, M]")
    per_image = [int(l.shape[0]) for l in labels]
    lab = torch.cat(list(labels)).to(torch.int64).contiguous()
    r, c, m = int(x.shape[0]), int(x.shape[1]), int(x.shape[2])
    torch._assert(lab.shape[0] == r, "one label per mask expected")
    out = torch.empty((r, 1, m, m), dtype=torch.float32, device=x.device)
    if r:
        _lib.check(_lib.load().mb_mask_prob(_ptr(_f32c(x)), _ptr(lab), r, c, m, _ptr(out), _stream(x)), "mb_mask_prob")
    out = out.to(x.dtype)
    return list(out.split(per_image, dim=0))

"""HotPath — the whole post-head detection path as one prepared, sync-free plan.

One `step()` is what happens between the CNN heads and the saved particle crops for one batch
(SURVEY.md §3.2 with the cuDNN/cuBLAS parts taken as inputs):

    RPN head outputs ──► mb_rpn_proposals ──► proposals [N, R, 4] (+counts)
    FPN features + proposals ──► mb_multiscale_roi_align ──► box features [N*R, C, 7, 7]
    box-head outputs (class logits, box regression) + proposals ──► mb_det_postprocess ──► detections
    detections + original uint8 images ──► mb_crop_plan / mb_crop_gather ──► packed crops

All parameter structs, workspaces and outputs are created once; `step()` only enqueues kernels
on the current stream (6 C-ABI calls, no allocation, no host synchronisation). `OverlappedHotPath`
keeps three batches in flight on three streams, `HostPipeline` is the pinned-host-in / pinned-host-out
loop around it, `HotPath.capture()` records the step as a CUDA graph.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import MisoB200Error
from .detection import CropStage, DetConfig, RpnConfig, det_params, rpn_params
from .ops import _ptr, _stream, is_channels_last, pooler_levels, roi_align_params, roi_align_reads_channels_last


@dataclass
class HotPathShapes:
    num_images: int
    padded_image_size: Tuple[int, int]           # network input after padding (anchor strides)
    image_sizes: Sequence[Tuple[int, int]]       # per image, after resize, before padding
    original_image_sizes: Sequence[Tuple[int, int]]
    rpn_grids: Sequence[Tuple[int, int]]         # RPN head output sizes per level (incl. 'pool')
    feature_grids: Sequence[Tuple[int, int]]     # pooler levels ('0'..'3')
    channels: int = 256
    num_classes: int = 3
    pooled: int = 7
    sampling_ratio: int = 2
    image_channels: int = 3


class HotPath:
    # kernels one step() launches, per C-ABI call (checked against the ncu launch list in profiles/)
    KERNELS = {"mb_rpn_proposals": 7,         # k_rpn_hist, k_rpn_select, k_rpn_decode, k_seg_meta, k_nms_mask, k_nms_sweep_small, k_rpn_finalize
               "mb_multiscale_roi_align": 2,  # k_roi_geom + k_roi_align_tma (k_roi_align_nhwc4d alone outside the envelope)
               "mb_det_postprocess": 7,       # k_det_init, k_det_candidates, k_seg_meta, k_rank_in_segment, k_nms_mask, k_nms_sweep_small, k_det_finalize
               "mb_crop_plan": 1, "mb_crop_gather": 1}

    # the crop stage's outputs and capacity under the names HotPath has always had (HostPipeline's result keys)
    crop_rects = property(lambda self: self.crop.rects)
    crop_xywh = property(lambda self: self.crop.xywh)
    crop_src = property(lambda self: self.crop.src)
    crop_offsets = property(lambda self: self.crop.offsets)
    crop_totals = property(lambda self: self.crop.totals)
    crop_pixels = property(lambda self: self.crop.pixels)
    crop_capacity = property(lambda self: self.crop.capacity)

    def __init__(self, shapes: HotPathShapes, rpn: RpnConfig, det: DetConfig, threshold: float = 0.5,
                 crop_capacity_bytes: int = 64 << 20, exact_roi_align: bool = True, device="cuda:0"):
        self.lib = _lib.load()
        self.s, self.dev = shapes, torch.device(device)
        n, R = shapes.num_images, int(rpn.post_nms_top_n)
        self.R, self.dpi = R, int(det.detections_per_img)
        dev = self.dev
        f32, i32, i64 = torch.float32, torch.int32, torch.int64
        # ---- outputs / intermediates (fixed capacity, device-side counts) ----
        self.proposals = torch.zeros((n, R, 4), dtype=f32, device=dev)
        self.prop_scores = torch.zeros((n, R), dtype=f32, device=dev)
        self.prop_counts = torch.zeros((n,), dtype=i32, device=dev)
        self.box_features = torch.empty((n * R, shapes.channels, shapes.pooled, shapes.pooled), dtype=f32, device=dev)
        self.det_boxes = torch.zeros((n, self.dpi, 4), dtype=f32, device=dev)
        self.det_boxes_net = torch.zeros((n, self.dpi, 4), dtype=f32, device=dev)
        self.det_scores = torch.zeros((n, self.dpi), dtype=f32, device=dev)
        self.det_labels = torch.zeros((n, self.dpi), dtype=i64, device=dev)
        self.det_counts = torch.zeros((n,), dtype=i32, device=dev)
        self.crop = CropStage(shapes.original_image_sizes, shapes.image_channels, self.dpi, threshold, dev,
                              capacity_bytes=crop_capacity_bytes)

        # ---- parameter structs (the input pointers are set by bind()) ----
        self.rpn_params = rpn_params(rpn, shapes.rpn_grids, None, shapes.padded_image_size, shapes.image_sizes)
        scales, thresholds = pooler_levels(shapes.feature_grids, shapes.image_sizes)
        self.roi_params = roi_align_params(shapes.feature_grids, n, shapes.channels, (shapes.pooled, shapes.pooled),
                                           shapes.sampling_ratio, scales, thresholds, exact=exact_roi_align, boxes_per_image=R)
        self.roi_params.box_counts = self.prop_counts.data_ptr()
        self.det_params = det_params(det, n, shapes.num_classes, R, shapes.image_sizes, shapes.original_image_sizes)

        # ---- workspaces ----
        nb = self.lib.mb_rpn_workspace_bytes(C.byref(self.rpn_params))
        db = self.lib.mb_det_workspace_bytes(C.byref(self.det_params))
        if nb == 0 or db == 0:
            raise MisoB200Error("HotPath: configuration outside the implemented envelope")
        self.rpn_ws = torch.empty((nb,), dtype=torch.uint8, device=dev)
        self.det_ws = torch.empty((db,), dtype=torch.uint8, device=dev)
        self._keep: List[Tensor] = []
        self.roi_ws = None
        self.features_layout = "nchw"
        self.kernel_launches_per_step = sum(self.KERNELS.values())

    # ------------------------------------------------------------------------------
    def bind(self, objectness: Sequence[Tensor], deltas: Sequence[Tensor], features: Sequence[Tensor],
             class_logits: Tensor, box_regression: Tensor, images: Sequence[Tensor]) -> None:
        """Attach the (device-resident) inputs. objectness/deltas: RPN head outputs per level (NCHW);
        features: pooler levels (NCHW); class_logits [N*R, C] / box_regression [N*R, 4C]: box-head
        outputs for the proposal slots; images: original uint8 HWC images."""
        self._keep = [*objectness, *deltas, *features, class_logits, box_regression, *images]
        for t in self._keep:
            dense = t.is_contiguous() or (t.dim() == 4 and t.is_contiguous(memory_format=torch.channels_last))
            if t.device.type != "cuda" or not dense:
                raise MisoB200Error("HotPath.bind: inputs must be dense CUDA tensors")
        for l, (o, dl) in enumerate(zip(objectness, deltas)):
            self.rpn_params.objectness[l], self.rpn_params.deltas[l] = o.data_ptr(), dl.data_ptr()
        # FPN maps: channels-last tensors (what a torch.channels_last backbone produces) are gathered in
        # place; NCHW maps get a workspace so that the library can transpose them once per step
        nhwc = all(is_channels_last(f) for f in features)
        q = self.roi_params
        if nhwc and not roi_align_reads_channels_last(q.channels, (q.pooled_h, q.pooled_w), q.sampling_ratio, features[0].dtype):
            raise MisoB200Error("HotPath.bind: mb_multiscale_roi_align cannot read these channels-last maps in place "
                                "(fp32, channels > 1, sampling ratio 2, pooled sides <= 16); bind NCHW maps")
        self.roi_params.channels_last = int(nhwc)
        for l, f in enumerate(features):
            self.roi_params.features[l] = f.data_ptr()
        nb = self.lib.mb_roi_align_workspace_bytes(C.byref(self.roi_params), self.s.num_images * self.R)
        self.roi_ws = torch.empty((nb,), dtype=torch.uint8, device=self.dev) if nb else None
        self.features_layout = "channels_last" if nhwc else "nchw"
        self.kernel_launches_per_step = sum(self.KERNELS.values()) + (len(features) if (nb and not nhwc) else 0)   # + k_nchw_to_nhwc per level
        self.crop.bind_images(images)
        self.class_logits, self.box_regression = class_logits, box_regression
        self._graph = None                               # a captured graph refers to the previous tensors

    def rebind(self, objectness: Sequence[Tensor], deltas: Sequence[Tensor], features: Sequence[Tensor],
               class_logits, box_regression) -> None:
        """Swap the per-batch inputs (pointers only; shapes, dtypes and memory formats as in the first bind()).
        Kernel parameters are copied at launch, so this is safe while the previous batch is still running."""
        if getattr(self, "class_logits", None) is None:
            dummy = [torch.zeros((1, 1, self.s.image_channels), dtype=torch.uint8, device=self.dev)] * self.s.num_images
            cl = class_logits[0] if isinstance(class_logits, (list, tuple)) else class_logits
            br = box_regression[0] if isinstance(box_regression, (list, tuple)) else box_regression
            self.bind(objectness, deltas, features, cl, br, dummy)
            return
        for l, (o, dl) in enumerate(zip(objectness, deltas)):
            self.rpn_params.objectness[l], self.rpn_params.deltas[l] = o.data_ptr(), dl.data_ptr()
        for l, f in enumerate(features):
            self.roi_params.features[l] = f.data_ptr()
        self.class_logits = class_logits[0] if isinstance(class_logits, (list, tuple)) else class_logits
        self.box_regression = box_regression[0] if isinstance(box_regression, (list, tuple)) else box_regression
        self._graph = None

    def rpn(self, st=None):
        st = st or _stream(self.dev)
        _lib.check(self.lib.mb_rpn_proposals(C.byref(self.rpn_params), _ptr(self.proposals), _ptr(self.prop_scores),
                                             _ptr(self.prop_counts), None, _ptr(self.rpn_ws), self.rpn_ws.numel(), st),
                   "mb_rpn_proposals")

    def roi_align(self, st=None):
        st = st or _stream(self.dev)
        _lib.check(self.lib.mb_multiscale_roi_align(C.byref(self.roi_params), _ptr(self.proposals),
                                                    self.s.num_images * self.R, _ptr(self.box_features), None,
                                                    _ptr(self.roi_ws), self.roi_ws.numel() if self.roi_ws is not None else 0, st),
                   "mb_multiscale_roi_align")

    def detections(self, st=None):
        st = st or _stream(self.dev)
        _lib.check(self.lib.mb_det_postprocess(C.byref(self.det_params), _ptr(self.class_logits), _ptr(self.box_regression),
                                               _ptr(self.proposals), _ptr(self.prop_counts), 0, _ptr(self.det_boxes),
                                               _ptr(self.det_boxes_net), _ptr(self.det_scores), _ptr(self.det_labels),
                                               _ptr(self.det_counts), _ptr(self.det_ws), self.det_ws.numel(), st),
                   "mb_det_postprocess")

    def crops(self, st=None):
        st = st or _stream(self.dev)
        self.crop.plan(self.det_boxes, self.det_scores, self.det_counts, st)
        self.crop.cut(st)

    def step(self) -> None:
        st = _stream(self.dev)
        self.rpn(st)
        self.roi_align(st)
        self.detections(st)
        self.crops(st)

    def capture(self) -> "torch.cuda.CUDAGraph":
        """Record one step() (its 21 kernel launches) into a CUDA graph; `replay()` then re-issues the whole
        step with one host call and without per-launch gaps on the device (config 2: 0.40 -> 0.375 ms).
        The graph is tied to the bound tensors: call again after bind()."""
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(torch.cuda.current_stream(self.dev))
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            self.step()                                  # warm-up outside the capture (function attributes, lazy init)
            with torch.cuda.graph(graph, stream=side):
                self.step()
        torch.cuda.current_stream(self.dev).wait_stream(side)
        self._graph = graph
        return graph

    def replay(self) -> None:
        if getattr(self, "_graph", None) is None:
            raise MisoB200Error("HotPath.replay: call capture() first")
        self._graph.replay()

    # ------------------------------------------------------------------------------
    def results(self):
        """Read back one step's results (one sync): per-image detections that passed the score
        filter, their annotation bounds and crop arrays."""
        crops = self.crop.to_host(self.s.image_channels)
        labels = self.det_labels.cpu().numpy(); scores = self.det_scores.cpu().numpy()
        out = [[] for _ in range(self.s.num_images)]
        for i, d, xywh, arr in crops:
            out[i].append({"xywh": xywh, "label": int(labels[i, d]), "score": float(scores[i, d]), "crop": arr})
        return out


class HostPipeline:
    """Host-facing driver of the hot path: inputs arrive in pinned host memory, results leave in
    pinned host memory, and the three legs of a batch run on three streams so that batch i+1's
    host->device copy, batch i's kernels and batch i-1's device->host read overlap:

        copy-in stream   H2D(i+1) ───────────────►
        compute stream          HotPath.step(i) ─►
        copy-out stream                 counts/boxes(i) ─► [host reads the crop byte count] ─► pixels(i-1)

    `depth` batches are in flight over depth+1 slots (device input buffers + a HotPath with its own
    outputs + pinned result buffers). `submit()` never blocks on the batch it enqueues; it returns the
    finished results of the batch submitted `depth` calls earlier (None while the pipeline fills) —
    views of that slot's pinned buffers, valid until the next `submit()` — and `flush()` drains.
    The only host waits are on events of batches that are already behind the GPU.
    """

    SMALL = ("det_boxes", "det_scores", "det_labels", "det_counts", "crop_rects", "crop_xywh", "crop_src",
             "crop_offsets", "crop_totals")

    def __init__(self, make_hot_path, host_example, depth: int = 2, on_computed=None, on_collect=None):
        """make_hot_path() -> HotPath (called once per slot); host_example: dict name -> list of host
        tensors (objectness, deltas, features, class_logits, box_regression, images) giving shapes,
        dtypes and memory formats; on_computed(hp, slot) is called with the compute stream current right
        after a batch's kernels were enqueued (the mosaic exchange hooks in here)."""
        self.slots = []
        for _ in range(depth + 1):
            hp = make_hot_path()
            dev = hp.dev
            d = {k: [torch.empty_like(t, device=dev) for t in v] for k, v in host_example.items()}
            hp.bind(d["objectness"], d["deltas"], d["features"], d["class_logits"][0], d["box_regression"][0], d["images"])
            out = {k: torch.empty_like(getattr(hp, k), device="cpu").pin_memory() for k in self.SMALL}
            pix = torch.empty((hp.crop_capacity,), dtype=torch.uint8).pin_memory()
            ev = {k: torch.cuda.Event() for k in ("h2d", "computed", "small", "pix")}
            self.slots.append({"hp": hp, "dev": d, "out": out, "pix": pix, "ev": ev, "state": "free", "nb": 0})
        self.dev = self.slots[0]["hp"].dev
        self.s_in, self.s_cmp, self.s_out = (torch.cuda.Stream(device=self.dev) for _ in range(3))
        self.on_computed, self.on_collect = on_computed, on_collect
        self.i = 0
        self.h2d_bytes = sum(t.numel() * t.element_size() for v in host_example.values() for t in v)

    def _pixels(self, slot):
        """Second half of a batch's read-back: needs the byte count the first half brought."""
        if slot["state"] != "small":
            return
        slot["ev"]["small"].synchronize()
        nb = slot["nb"] = slot["hp"].crop.checked_totals(slot["out"]["crop_totals"])[1]
        with torch.cuda.stream(self.s_out):
            slot["pix"][:nb].copy_(slot["hp"].crop_pixels[:nb], non_blocking=True)
            slot["ev"]["pix"].record(self.s_out)
        slot["state"] = "pix"

    def _collect(self, slot):
        if slot["state"] == "free":
            return None
        self._pixels(slot)
        slot["ev"]["pix"].synchronize()
        slot["state"] = "free"
        extra = self.on_collect(slot["hp"], slot) if self.on_collect else None
        return {"out": slot["out"], "pixels": slot["pix"][:slot["nb"]], "extra": extra}

    def submit(self, host):
        n = len(self.slots)
        slot, prev, nxt = self.slots[self.i % n], self.slots[(self.i - 1) % n], self.slots[(self.i + 1) % n]
        assert slot["state"] == "free"                   # collected by the previous call (or never used)
        with torch.cuda.stream(self.s_in):
            for k, hs in host.items():
                for src, dst in zip(hs, slot["dev"][k]):
                    dst.copy_(src, non_blocking=True)
            slot["ev"]["h2d"].record(self.s_in)
        with torch.cuda.stream(self.s_cmp):
            self.s_cmp.wait_event(slot["ev"]["h2d"])
            slot["hp"].step()
            slot["ev"]["computed"].record(self.s_cmp)
            if self.on_computed:
                self.on_computed(slot["hp"], slot)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(slot["ev"]["computed"])
            for k, ht in slot["out"].items():
                ht.copy_(getattr(slot["hp"], k), non_blocking=True)
            slot["ev"]["small"].record(self.s_out)
        slot["state"] = "small"
        if prev is not slot:
            self._pixels(prev)                           # batch i-1 computed while batch i's inputs were copied
        self.i += 1
        return self._collect(nxt)                        # batch i-depth; frees the slot the next call will use

    def flush(self):
        res = []
        for j in range(1, len(self.slots) + 1):
            r = self._collect(self.slots[(self.i + j) % len(self.slots)])
            if r is not None:
                res.append(r)
        return res


class OverlappedHotPath:
    """Software-pipelined plan for a stream of batches whose inputs are already in HBM.

    The RPN stage and the detection/crop stages are chains of small latency-bound kernels (a few
    CTAs each: one per image x level or image x class segment); RoIAlign is the one kernel that
    fills the machine. Run back to back they leave most SMs idle for half of the step, so three
    batches are kept in flight on three streams:

        stream R   rpn(k+2) ────────►
        stream A        roi_align(k+1) ───────►
        stream D              detections(k), crops(k) ─►

    Inside one batch the order of the reference is kept (rpn -> roi_align -> detections -> crops,
    chained by events); `slots` HotPath instances own the per-batch intermediates (proposals,
    box features, detections, crops). `submit()` only enqueues; `drain()` makes the current stream
    wait for everything in flight.
    """

    def __init__(self, hot_paths: Sequence[HotPath]):
        self.hps = list(hot_paths)
        self.dev = self.hps[0].dev
        # the small-kernel chains get the higher stream priority: their few CTAs are placed as soon as
        # RoIAlign CTAs retire instead of waiting for its whole grid to drain
        self.sR = torch.cuda.Stream(device=self.dev, priority=-1)
        self.sA = torch.cuda.Stream(device=self.dev, priority=0)
        self.sD = torch.cuda.Stream(device=self.dev, priority=-1)
        self.ev = [{k: torch.cuda.Event() for k in ("rpn", "roi", "done")} for _ in self.hps]
        self.used = [False] * len(self.hps)
        self.k = 0
        self.hooks = {}          # "before_roi" / "after_roi" / "before_det" / "after_det": fn(slot_index, hp, stream) —
                                 # timing events, the mosaic exchange; hooks that enqueue work must use `stream` explicitly

    def submit(self) -> int:
        i = self.k % len(self.hps)
        hp, ev = self.hps[i], self.ev[i]
        if not self.used[i]:             # first use: order behind whatever prepared the inputs on the current stream
            cur = torch.cuda.current_stream(self.dev)
            for s in (self.sR, self.sA, self.sD):
                s.wait_stream(cur)
        else:
            self.sR.wait_event(ev["done"])   # the slot's proposals / detections are free again
        self.used[i] = True
        hooks = self.hooks
        # explicit stream handles everywhere (no stream context switches on the host)
        hp.rpn(_stream(self.sR))
        ev["rpn"].record(self.sR)
        self.sA.wait_event(ev["rpn"])
        if "before_roi" in hooks:
            hooks["before_roi"](i, hp, self.sA)
        hp.roi_align(_stream(self.sA))
        ev["roi"].record(self.sA)
        if "after_roi" in hooks:
            hooks["after_roi"](i, hp, self.sA)
        self.sD.wait_event(ev["roi"])
        if "before_det" in hooks:
            hooks["before_det"](i, hp, self.sD)
        hp.detections(_stream(self.sD))
        if "after_det" in hooks:
            hooks["after_det"](i, hp, self.sD)
        hp.crops(_stream(self.sD))
        ev["done"].record(self.sD)
        self.k += 1
        return i

    def drain(self) -> None:
        cur = torch.cuda.current_stream(self.dev)
        for s in (self.sR, self.sA, self.sD):
            cur.wait_stream(s)

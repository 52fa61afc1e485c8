"""Tiled mosaic path (BASELINE config 5): overlapping tiles sharded over the GPUs of one box,
one NCCL all-gather of fixed-size detection blocks, a cross-tile "seam" NMS, crops cut by the rank
that owns the tile a detection came from.

The reference has no counterpart (ref:miso/object_detection/inference.py:86-88 feeds whole
images, which the model's transform shrinks to <= 1333 px); the semantics are DEFINED as the
single-process composition of reference operations (SURVEY.md §8(e)):

    for every tile, row-major: detections of the tile (reference path) -> add the tile origin in
    fp32 -> concatenate -> torchvision.ops.boxes._batched_nms_vanilla(boxes, scores, labels, iou)
    -> miso's `score > threshold` filter (applied before the exchange; greedy NMS only lets
    higher-scored boxes suppress lower-scored ones, so this does not change the result)
    -> RectangleAnnotation.coords_int on the mosaic coordinates -> slice of the mosaic array.

Sharding: tiles in row-major order, contiguous blocks per rank, so concatenating the rank blocks
in rank order reproduces the single-GPU tile order for any world size. Results are reported in
that order (gathered row = tile * dpi + slot), which makes the concatenation of the per-rank
outputs in rank order EQUAL to the world-size-1 output; `by_score()` gives batched_nms' order.
Each rank holds only the pixel band its tiles cover; a detection lies inside the tile that
produced it, so the owner of the tile cuts the crop without any pixel exchange.
The only collective is one all_gather_into_tensor of [tiles_per_rank_max * dpi, 6] fp32 rows.

Everything here runs on the GPU through libmisob200 (no CPU branch); the CPU restatement used by
the tests lives in tests/mosaic_ref.py.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import MisoB200Error
from .detection import MORPHOLOGY_FIELDS, CropStage
from .ops import _ptr, _stream


def tile_starts(extent: int, tile: int, overlap: int) -> List[int]:
    """Starts 0, stride, 2*stride, ... plus a clamped last tile (16384/1024/128 -> 19 starts)."""
    if extent <= tile:
        return [0]
    stride = tile - overlap
    starts = list(range(0, extent - tile, stride))
    starts.append(extent - tile)
    return starts


def tile_grid(height: int, width: int, tile: int, overlap: int) -> List[Tuple[int, int]]:
    """Row-major (y, x) origins."""
    return [(y, x) for y in tile_starts(height, tile, overlap) for x in tile_starts(width, tile, overlap)]


def rank_tiles(num_tiles: int, world: int, rank: int) -> range:
    """Contiguous block of rank r: [floor(T*r/G), floor(T*(r+1)/G))."""
    return range(num_tiles * rank // world, num_tiles * (rank + 1) // world)


def tiles_per_rank_max(num_tiles: int, world: int) -> int:
    return max(len(rank_tiles(num_tiles, world, r)) for r in range(world))


def rank_band(grid: Sequence[Tuple[int, int]], tile: int, height: int, world: int, rank: int) -> Tuple[int, int]:
    """Pixel rows [y0, y1) of the mosaic that rank's tiles cover (the only pixels it has to hold)."""
    mine = rank_tiles(len(grid), world, rank)
    if len(mine) == 0:
        return 0, 0
    return min(grid[t][0] for t in mine), min(height, max(grid[t][0] for t in mine) + tile)


def gathered_row(tile_index: int, slot: int, num_tiles: int, world: int, dpi: int) -> int:
    """Row of (tile, slot) in the gathered buffer of a `world`-rank run (rank blocks of tiles_per_rank_max*dpi rows)."""
    tmax = tiles_per_rank_max(num_tiles, world)
    for r in range(world):
        rt = rank_tiles(num_tiles, world, r)
        if tile_index in rt:
            return (r * tmax + (tile_index - rt.start)) * dpi + slot
    raise IndexError(tile_index)


def pack_block(det_boxes: Tensor, det_scores: Tensor, det_labels: Tensor, det_counts: Tensor, origins: Tensor,
               threshold: float, rows: int, out: Optional[Tensor] = None) -> Tensor:
    """[T, dpi, *] detections of tiles -> [rows, 6] = (x1, y1, x2, y2, score, label) in mosaic coordinates
    (one mb_mosaic_pack launch). Rows that hold no detection, or one that fails `score > threshold`, get
    label -1. origins: [T, 2] = (y, x) as fp32 (exact). `out` may be a row slice of a larger block."""
    t, dpi = det_scores.shape
    if not det_boxes.is_cuda:
        raise MisoB200Error("pack_block: CUDA tensors expected (miso_b200 has no CPU path)")
    if out is None:
        out = torch.empty((rows, 6), dtype=torch.float32, device=det_boxes.device)
    for x in (det_boxes, det_scores, det_labels, det_counts, origins, out):
        torch._assert(x.is_contiguous(), "pack_block: contiguous tensors expected")
    torch._assert(det_labels.dtype == torch.int64 and det_counts.dtype == torch.int32 and out.shape == (rows, 6),
                  "pack_block: int64 labels, int32 counts, [rows, 6] output expected")
    _lib.check(_lib.load().mb_mosaic_pack(_ptr(det_boxes), _ptr(det_scores), _ptr(det_labels), _ptr(det_counts), _ptr(origins),
                                          int(t), int(dpi), float(threshold), int(rows), _ptr(out), _stream(det_boxes)),
               "mb_mosaic_pack")
    return out


def exchange(block: Tensor, world: int, group=None, out: Optional[Tensor] = None) -> Tensor:
    """The path's one collective: all-gather of the per-rank blocks, rank order preserved."""
    if world == 1:
        return block
    import torch.distributed as dist
    if out is None:
        out = torch.empty((world * block.shape[0], block.shape[1]), dtype=block.dtype, device=block.device)
    dist.all_gather_into_tensor(out, block, group=group)
    return out


class SeamNms:
    """Dense seam NMS (one mb_mosaic_unpack launch + the prepared per-label mb_nms over ALL gathered rows).
    Kept as the cross-check of SparseSeamNms and for negative IoU thresholds."""

    def __init__(self, rows: int, num_classes: int, device):
        from .ops import PreparedBatchedNms
        self.nms = PreparedBatchedNms(rows, num_classes, device)
        self.rows = int(rows)
        self.boxes = torch.empty((rows, 4), dtype=torch.float32, device=device)
        self.scores = torch.empty((rows,), dtype=torch.float32, device=device)
        self.labels = torch.empty((rows,), dtype=torch.int64, device=device)

    def launch(self, gathered: Tensor, iou_threshold: float):
        torch._assert(gathered.is_contiguous() and gathered.shape == (self.rows, 6), "SeamNms: [rows, 6] contiguous block expected")
        _lib.check(_lib.load().mb_mosaic_unpack(_ptr(gathered), self.rows, _ptr(self.boxes), _ptr(self.scores),
                                                _ptr(self.labels), _stream(gathered)), "mb_mosaic_unpack")
        return self.nms(self.boxes, self.scores, self.labels, iou_threshold)

    def finish(self):
        """(boxes, scores, labels, rows) of the kept detections in batched_nms order (score desc, row asc); one sync."""
        n = int(self.nms.status[0])
        if n < 0:
            raise MisoB200Error(f"seam NMS failed on the device (status {n})")
        keep = self.nms.keep[:n]
        return self.boxes[keep], self.scores[keep], self.labels[keep], keep


class SparseSeamNms:
    """Sync-free sparse seam NMS (mb_seam_nms): the same kept set as SeamNms, found on the sparse
    "may suppress" graph between tiles whose detections' bounding boxes intersect. Every buffer is
    allocated once; `state` [rows] int32 (1 kept, 2 suppressed, 3 ignored) stays on the device."""

    def __init__(self, rows: int, rows_per_tile: int, device, edges_per_row: int = 8, want_keep: bool = False):
        self.lib = _lib.load()
        self.rows, self.rpt = int(rows), int(rows_per_tile)
        self.edge_cap = max(1024, int(edges_per_row) * self.rows)
        nb = self.lib.mb_seam_nms_workspace_bytes(self.rows, self.rpt, self.edge_cap)
        if nb == 0:
            raise MisoB200Error("SparseSeamNms: invalid configuration")
        self.ws = torch.empty((nb,), dtype=torch.uint8, device=device)
        self.state = torch.zeros((self.rows,), dtype=torch.int32, device=device)
        self.keep = torch.zeros((self.rows,), dtype=torch.int64, device=device) if want_keep else None
        self.status = torch.zeros((4,), dtype=torch.int64, device=device)

    def launch(self, gathered: Tensor, iou_threshold: float) -> Tensor:
        torch._assert(gathered.is_contiguous() and gathered.shape == (self.rows, 6) and gathered.dtype == torch.float32,
                      "SparseSeamNms: [rows, 6] contiguous fp32 block expected")
        _lib.check(self.lib.mb_seam_nms(_ptr(gathered), self.rows, self.rpt, float(iou_threshold), self.edge_cap,
                                        _ptr(self.state), _ptr(self.keep), _ptr(self.status), _ptr(self.ws), self.ws.numel(),
                                        _stream(gathered)), "mb_seam_nms")
        return self.state

    def check(self) -> Tuple[int, int]:
        """Host check of the device status (one sync): raises if the edge workspace overflowed."""
        st = self.status.tolist()
        if st[0] < 0:
            raise MisoB200Error(f"mb_seam_nms: status {st[0]} (suppression edges found: {st[1]}, capacity {self.edge_cap})")
        return int(st[0]), int(st[1])


class MosaicCrops(CropStage):
    """One rank's share of the final stage: rows of its own block that survived the seam NMS -> annotation
    bounds, integer crop rectangles in MOSAIC coordinates, packed crop bytes cut from the rank's pixel band
    (mb_seam_select, then the crop stage on the mosaic as one image; no host sync)."""

    def __init__(self, rows: int, mosaic_hw: Tuple[int, int], channels: int, threshold: float, capacity_bytes: int, device):
        super().__init__([mosaic_hw], channels, rows, threshold, device, capacity_bytes=capacity_bytes)
        self.rows = int(rows)
        self.boxes = torch.zeros((self.rows, 4), dtype=torch.float32, device=self.dev)
        self.scores = torch.zeros((self.rows,), dtype=torch.float32, device=self.dev)
        self.count = torch.tensor([self.rows], dtype=torch.int32, device=self.dev)

    def bind_band(self, band_u8: Tensor, band_y0: int) -> None:
        """band_u8: uint8 [band_h, W, C] — mosaic rows [band_y0, band_y0 + band_h). The crop kernels address the
        mosaic through a virtual base pointer; only rows inside the band are ever read (a detection lies inside the
        tile that produced it, and the rank's band covers its tiles)."""
        torch._assert(band_u8.is_cuda and band_u8.dtype == torch.uint8 and band_u8.is_contiguous() and band_u8.dim() == 3,
                      "bind_band: dense uint8 [h, W, C] CUDA tensor expected")
        torch._assert(band_u8.shape[1] == self.params.image_w[0] and band_u8.shape[2] == self.params.channels,
                      "bind_band: band width / channels differ from the mosaic's")
        self.band_y0 = int(band_y0)
        self.bind_images([band_u8], [band_u8.data_ptr() - self.band_y0 * band_u8.shape[1] * band_u8.shape[2]])

    def bind_masks(self, mask_probs: Tensor, paste_boxes: Tensor, frames: Tensor, rows_per_frame: int,
                   mask_threshold: float = 0.5, morphology: bool = False) -> None:
        """Cut every crop's instance mask as well (mb_crop_masks after the gather, results()["masks"]). Row s of this
        rank's block: mask_probs [rows, M, M] (maskrcnn_inference's output), paste_boxes [rows, 4] xyxy in the
        coordinates of its frame, the tile it came from: frames[s // rows_per_frame] = (x0, y0, w, h) int32 in mosaic
        coordinates. A crop's mask is the tile-sized paste_masks_in_image of its detection, cut to the crop rectangle
        and thresholded (> mask_threshold: 255, else 0; 0 outside the tile). morphology=True also measures every
        crop's mask (mb_mask_morphology after the masks): results()["morphology"] [count, len(MORPHOLOGY_FIELDS)] fp64,
        centroids in mosaic coordinates, channel means from the band's pixels."""
        m = int(mask_probs.shape[-1])
        for t in (mask_probs, paste_boxes, frames):
            torch._assert(t.is_cuda and t.is_contiguous(), "bind_masks: contiguous CUDA tensors expected")
        torch._assert(mask_probs.dtype == torch.float32 and mask_probs.shape == (self.rows, m, m),
                      "bind_masks: mask_probs must be fp32 [rows, M, M]")
        torch._assert(paste_boxes.dtype == torch.float32 and paste_boxes.shape == (self.rows, 4), "bind_masks: paste_boxes must be fp32 [rows, 4]")
        torch._assert(frames.dtype == torch.int32 and frames.dim() == 2 and frames.shape[1] == 4
                      and frames.shape[0] * int(rows_per_frame) >= self.rows, "bind_masks: frames must be int32 [rows / rows_per_frame, 4]")
        super().bind_masks(mask_probs, paste_boxes, frames, rows_per_frame, mask_threshold,
                           self.capacity // self.params.channels, morphology)

    def launch(self, gathered: Tensor, state: Tensor, row_lo: int) -> None:
        st = _stream(gathered)
        _lib.check(self.lib.mb_seam_select(_ptr(gathered), _ptr(state), int(row_lo), self.rows, _ptr(self.boxes),
                                           _ptr(self.scores), st), "mb_seam_select")
        self.plan(self.boxes, self.scores, self.count, st)
        self.cut(st)

    def results(self) -> Dict[str, Tensor]:
        """One sync: this rank's surviving detections in row order and their crop bytes; with bind_masks() also
        "masks", the crops' h*w mask bytes packed at offsets // channels, and with bind_masks(morphology=True)
        "morphology", one record per crop in the same row order."""
        tot = self.checked_totals(masks=self.masks is not None)
        k = tot[0]
        out = {"count": k, "bytes": tot[1], "rects": self.rects[:k], "xywh": self.xywh[:k], "src": self.src[:k],
               "offsets": self.offsets[:k + 1], "pixels": self.pixels[:tot[1]]}
        if self.masks is not None:
            out["masks"] = self.masks[:tot[1] // self.params.channels]
            if self.morphology is not None:
                out["morphology"] = self.morphology[:k]
        for key, buf in (("png", self.png), ("mask_png", self.mask_png), ("jpeg", self.jpeg)):
            if buf is not None:
                total = self.checked_png(buf, key)[0]
                out[key], out[key + "_offsets"] = buf["out"][:total], buf["offsets"][:k + 1]
        return out


class MosaicPlan:
    """One rank's share of a tiled mosaic through the post-head hot path, as a prepared, sync-free plan:

        for every batch of own tiles:  mb_rpn_proposals | mb_multiscale_roi_align | mb_det_postprocess
                                       (three batches in flight on three streams) -> mb_mosaic_pack into the block
        all_gather_into_tensor (NCCL) -> mb_seam_nms -> mb_seam_select + mb_crop_plan + mb_crop_gather (own rows)

    `batches` is this rank's list of per-batch inputs (dicts objectness/deltas/features/class_logits/
    box_regression of device tensors — in a deployment the CNN heads' outputs), in tile order; batch i covers
    own tiles [sum of earlier batch sizes, +n_i). make_hot_path(n) builds a HotPath for n tiles per batch."""

    SLOTS = 3

    def __init__(self, grid: Sequence[Tuple[int, int]], tile: int, mosaic_hw: Tuple[int, int], make_hot_path,
                 batch_sizes: Sequence[int], rank: int = 0, world: int = 1, threshold: float = 0.5,
                 iou_threshold: float = 0.5, image_channels: int = 3, crop_capacity_bytes: int = 256 << 20,
                 device="cuda:0", group=None):
        self.lib = _lib.load()
        self.dev = torch.device(device)
        self.grid, self.tile, self.hw = list(grid), int(tile), (int(mosaic_hw[0]), int(mosaic_hw[1]))
        self.rank, self.world, self.group = int(rank), int(world), group
        self.mine = rank_tiles(len(self.grid), self.world, self.rank)
        self.tmax = tiles_per_rank_max(len(self.grid), self.world)
        if sum(batch_sizes) != len(self.mine):
            raise MisoB200Error("MosaicPlan: batch sizes must add up to the rank's tile count")
        self.batch_sizes = [int(b) for b in batch_sizes]
        self.threshold, self.iou = float(threshold), float(iou_threshold)
        # HotPath slots per batch size (three batches in flight)
        self.slots: Dict[int, List] = {}
        for n in sorted(set(self.batch_sizes)):
            k = min(self.SLOTS, self.batch_sizes.count(n))
            self.slots[n] = [make_hot_path(n) for _ in range(k)]
        any_hp = next(iter(self.slots.values()))[0]
        self.dpi = any_hp.dpi
        self.block_rows = self.tmax * self.dpi
        self.block = torch.zeros((self.block_rows, 6), dtype=torch.float32, device=self.dev)
        self.block[:, 5] = -1.0                                  # padding rows (ranks with fewer tiles) stay ignored
        self.gathered = (torch.empty((self.world * self.block_rows, 6), dtype=torch.float32, device=self.dev)
                         if self.world > 1 else self.block)
        self.seam = SparseSeamNms(self.world * self.block_rows, self.dpi, self.dev)
        self.crops = MosaicCrops(self.block_rows, self.hw, image_channels, threshold, crop_capacity_bytes, self.dev)
        origins = [[float(self.grid[t][0]), float(self.grid[t][1])] for t in self.mine]
        self.origins = torch.tensor(origins, dtype=torch.float32, device=self.dev).reshape(-1, 2)
        self.sR = torch.cuda.Stream(device=self.dev, priority=-1)
        self.sA = torch.cuda.Stream(device=self.dev, priority=0)
        self.sD = torch.cuda.Stream(device=self.dev, priority=-1)
        self.ev = {n: [{k: torch.cuda.Event() for k in ("rpn", "roi", "done")} for _ in hps] for n, hps in self.slots.items()}
        self.used = {n: [False] * len(hps) for n, hps in self.slots.items()}
        self.hooks = {}
        self.launches_per_run = 0
        self._tile_launches = 0
        self._use = {n: 0 for n in self.slots}

    def bind_band(self, band_u8: Tensor, band_y0: int) -> None:
        self.crops.bind_band(band_u8, band_y0)

    def capture_tiles(self, batches, serial: bool = False) -> None:
        """Record run_tiles(batches) as a CUDA graph: the ~17 launches per batch of a rank's whole tile phase then cost
        one host call (`run(graph=True)`). The graph refers to the batches' tensors: keep them alive and in place."""
        cur = torch.cuda.current_stream(self.dev)
        side = torch.cuda.Stream(device=self.dev)
        side.wait_stream(cur)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            self.run_tiles(batches, serial=serial)               # warm-up outside the capture (function attributes, lazy init)
            side.synchronize()
            for n in self.used:
                self.used[n] = [False] * len(self.used[n])       # no waits on events recorded outside the capture
            with torch.cuda.graph(graph, stream=side):
                self.run_tiles(batches, serial=serial)
        cur.wait_stream(side)
        for n in self.used:
            self.used[n] = [False] * len(self.used[n])           # (their events were last recorded inside the capture)
        self._graph, self._graph_keep = graph, batches

    def run(self, batches=None, serial: bool = False, graph: bool = False) -> None:
        """Enqueue one whole mosaic pass of this rank (no host sync). Results: self.seam.state, self.crops.*
        graph=True replays the tile phase recorded by capture_tiles()."""
        if graph:
            if getattr(self, "_graph", None) is None:
                raise MisoB200Error("MosaicPlan.run(graph=True): call capture_tiles() first")
            self._graph.replay()
        else:
            self.run_tiles(batches, serial=serial)
        if self.world > 1:
            exchange(self.block, self.world, self.group, out=self.gathered)
        self.run_tail()

    def run_tail(self, gathered: Optional[Tensor] = None) -> None:
        """Seam NMS over the gathered rows + this rank's crops (gathered: override of the exchanged buffer — the
        single-GPU tests emulate several ranks by concatenating their blocks)."""
        if gathered is not None:
            self.gathered = gathered
        self.seam.launch(self.gathered, self.iou)
        self.crops.launch(self.gathered, self.seam.state, self.rank * self.block_rows)
        self.launches_per_run = self._tile_launches + 6 + 3      # seam: prep, pairs, 3 rounds, finish; select, plan, gather

    def run_tiles(self, batches, serial: bool = False, first: int = 0, count: Optional[int] = None) -> None:
        """This rank's tiles through rpn | roi_align | detections into self.block. `batches`: sequence of per-batch
        input dicts, or a callable (batch_index, n_tiles, stream) -> dict invoked right before the batch is enqueued
        (the host-fed pipeline copies the inputs in and makes `stream` wait for them there). Three batches are in
        flight on three streams unless `serial` (everything on the current stream, one kernel at a time: the mode
        whose per-kernel timings are those of the kernel running alone). `first`/`count` select a run of batches."""
        cur = torch.cuda.current_stream(self.dev)
        sR, sA, sD = (cur, cur, cur) if serial else (self.sR, self.sA, self.sD)
        if not serial:
            for s in (sR, sA, sD):
                s.wait_stream(cur)
        last = len(self.batch_sizes) if count is None else first + count
        t0 = sum(self.batch_sizes[:first])
        if first == 0:
            self._use = {n: 0 for n in self.slots}
            self._tile_launches = 0
        hooks = self.hooks
        for bi in range(first, last):
            n = self.batch_sizes[bi]
            i = self._use[n] % len(self.slots[n])
            self._use[n] += 1
            hp, ev = self.slots[n][i], self.ev[n][i]
            if self.used[n][i] and not serial:
                sR.wait_event(ev["done"])                    # the slot's proposals / detections are free again
            self.used[n][i] = True
            inp = batches(bi, n, sR) if callable(batches) else batches[bi - first if count is not None else bi]
            hp.rebind(inp["objectness"], inp["deltas"], inp["features"], inp["class_logits"], inp["box_regression"])
            hp.rpn(_stream(sR))
            if not serial:
                ev["rpn"].record(sR)
                sA.wait_event(ev["rpn"])
            if "before_roi" in hooks:
                hooks["before_roi"](bi, hp, sA)
            hp.roi_align(_stream(sA))
            if "after_roi" in hooks:
                hooks["after_roi"](bi, hp, sA)
            if not serial:
                ev["roi"].record(sA)
                sD.wait_event(ev["roi"])
            hp.detections(_stream(sD))
            _lib.check(self.lib.mb_mosaic_pack(_ptr(hp.det_boxes), _ptr(hp.det_scores), _ptr(hp.det_labels), _ptr(hp.det_counts),
                                               C.c_void_p(self.origins.data_ptr() + t0 * 8), n, self.dpi, self.threshold,
                                               n * self.dpi, C.c_void_p(self.block.data_ptr() + t0 * self.dpi * 24),
                                               _stream(sD)), "mb_mosaic_pack")
            if not serial:
                ev["done"].record(sD)
            if "batch_done" in hooks:
                hooks["batch_done"](bi, hp, sD)
            self._tile_launches += hp.kernel_launches_per_step - 2 + 1      # no per-batch crop stage; + k_mosaic_pack
            t0 += n
        if not serial:
            cur.wait_stream(sD)

    def results(self) -> Dict[str, Tensor]:
        self.seam.check()
        return self.crops.results()


def bind_host_near_gpu(device) -> Dict[str, object]:
    """Restrict this process to the CPUs NVML reports as local to `device` (its NUMA node), so that the pinned host
    buffers allocated afterwards — and the threads that fill them — sit on the socket whose PCIe root the GPU hangs
    off. One process per GPU on a two-socket box otherwise leaves half the ranks copying across the socket link.
    Call before allocating pinned memory. Returns what was done ({"bound": False, "why": ...} when NVML or the
    affinity call is unavailable; never raises: placement is an optimisation, not part of the result)."""
    import os
    try:
        import pynvml
        dev = torch.device(device)
        p = torch.cuda.get_device_properties(dev)
        pynvml.nvmlInit()
        bus = "%08x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        ncpu = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [i for i in range(ncpu) if (mask[i // 64] >> (i % 64)) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return {"bound": False, "why": "no overlap between the GPU's CPUs and this process's allowed set"}
        os.sched_setaffinity(0, allowed)
        return {"bound": True, "pci": bus, "cpus": len(allowed), "first_cpu": allowed[0], "last_cpu": allowed[-1], "host_cpus": ncpu}
    except Exception as e:                                       # noqa: BLE001 — diagnostics only
        return {"bound": False, "why": f"{type(e).__name__}: {e}"[:160]}


class HostMosaicRunner:
    """Host-facing driver of a MosaicPlan: every batch's head outputs arrive in (pinned) host memory and are copied
    to the device on a copy-in stream while earlier batches compute; the rank's results (annotation bounds, crop
    rectangles, crop bytes) are read back into pinned host memory. `depth` device input slots per batch size."""

    def __init__(self, plan: MosaicPlan, examples: Dict[int, Dict[str, Sequence[Tensor]]], depth: int = 4):
        self.plan, self.dev, self.depth = plan, plan.dev, int(depth)
        self.s_in = torch.cuda.Stream(device=self.dev)
        self.s_out = torch.cuda.Stream(device=self.dev)
        self.slots = {n: [{k: [torch.empty_like(t, device=self.dev) for t in v] for k, v in ex.items()} for _ in range(self.depth)]
                      for n, ex in examples.items()}
        self.ev_in = {n: [torch.cuda.Event() for _ in range(self.depth)] for n in examples}
        self.ev_free = {n: [None] * self.depth for n in examples}
        c = plan.crops
        self.small = {k: torch.empty_like(getattr(c, k), device="cpu").pin_memory() for k in ("rects", "xywh", "src", "offsets", "totals")}
        self.pix = torch.empty((c.capacity,), dtype=torch.uint8).pin_memory()
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def run(self, host_batches: Sequence[Dict[str, Sequence[Tensor]]]):
        plan = self.plan
        use = {n: 0 for n in self.slots}
        cur_slot = {}
        self.h2d_bytes = 0

        def feed(bi, n, stream):
            i = use[n] % self.depth
            use[n] += 1
            cur_slot[bi] = (n, i)
            if self.ev_free[n][i] is not None:
                self.s_in.wait_event(self.ev_free[n][i])          # the batch that last used this slot has been consumed
            dst = self.slots[n][i]
            with torch.cuda.stream(self.s_in):
                for k, hs in host_batches[bi].items():
                    for src, d in zip(hs, dst[k]):
                        d.copy_(src, non_blocking=True)
                        self.h2d_bytes += src.numel() * src.element_size()
                self.ev_in[n][i].record(self.s_in)
            stream.wait_event(self.ev_in[n][i])
            return dst

        def done(bi, hp, stream):
            n, i = cur_slot[bi]
            if self.ev_free[n][i] is None:
                self.ev_free[n][i] = torch.cuda.Event()
            self.ev_free[n][i].record(stream)

        plan.hooks["batch_done"] = done
        try:
            plan.run(feed)
        finally:
            plan.hooks.pop("batch_done", None)
        cur = torch.cuda.current_stream(self.dev)
        self.s_out.wait_stream(cur)
        c = plan.crops
        with torch.cuda.stream(self.s_out):
            for k, h in self.small.items():
                h.copy_(getattr(c, k), non_blocking=True)
        self.s_out.synchronize()
        tot = c.checked_totals(self.small["totals"])
        with torch.cuda.stream(self.s_out):
            self.pix[:tot[1]].copy_(c.pixels[:tot[1]], non_blocking=True)
        self.s_out.synchronize()
        self.d2h_bytes = sum(h.numel() * h.element_size() for h in self.small.values()) + tot[1]
        k = tot[0]
        return {"count": k, "bytes": tot[1], "rects": self.small["rects"][:k], "xywh": self.small["xywh"][:k],
                "src": self.small["src"][:k], "offsets": self.small["offsets"][:k + 1], "pixels": self.pix[:tot[1]]}


def by_score(gathered: Tensor, state: Tensor) -> Tensor:
    """Kept rows in torchvision batched_nms order (score descending, row ascending): host-facing helper."""
    rows = torch.nonzero(state == 1).flatten()
    order = torch.sort(gathered[rows, 4], descending=True, stable=True).indices
    return rows[order]


def infer_mosaic(model, band_u8: Tensor, mosaic_hw: Tuple[int, int], band_y0: int = 0, tile: int = 1024,
                 overlap: int = 128, threshold: float = 0.5, batch_size: int = 4, rank: int = 0, world: int = 1,
                 group=None, crop_capacity_bytes: int = 256 << 20, masks: bool = False, mask_threshold: float = 0.5,
                 morphology: bool = False, png: bool = False, jpeg: bool = False):
    """Detect on a large slide/mosaic image (config 5) with a (patched) torchvision detection model: this rank runs
    its contiguous share of tiles, the per-rank detection blocks are exchanged with one all-gather, the sparse seam
    NMS runs on every rank (replicated, deterministic) and each rank cuts the crops of its own tiles' survivors.

    band_u8: uint8 [band_h, W, C] on the device = mosaic rows [band_y0, band_y0 + band_h) — the pixel band this
    rank's tiles cover (rank_band()); with world == 1 simply the whole mosaic. Returns a dict: gathered [rows, 6]
    (mosaic coordinates), state [rows] (1 = kept), and this rank's crops (MosaicCrops.results()).
    masks=True (Mask R-CNN): crops["masks"] holds every crop's instance mask, its detection's mask pasted into the
    tile it came from, cut to the crop rectangle, > mask_threshold -> 255 (MosaicCrops.bind_masks).
    morphology=True (Mask R-CNN): crops["morphology"] [count, len(MORPHOLOGY_FIELDS)] fp64 on the device, each crop's
    mask measured (area, perimeter, centroid in mosaic coordinates, axes, ...; the masks are cut for it even when
    masks=False, and crops["masks"] is returned only when masks=True).
    png=True: crops["png"] / crops["png_offsets"] hold every crop as a PNG file on the device (packed in crop order,
    crop j is png[png_offsets[j]:png_offsets[j + 1]]), and crops["mask_png"] / crops["mask_png_offsets"] every mask
    when masks=True (CropStage.bind_png).
    jpeg=True: crops["jpeg"] / crops["jpeg_offsets"] hold every crop as a JPEG file on the device, byte for byte what PIL
    writes with default settings (packed in crop order, CropStage.bind_jpeg); 1 or 3 channels."""
    has_mask = getattr(model.roi_heads, "mask_predictor", None) is not None
    if (masks or morphology) and not has_mask:
        what = "masks" if masks else "morphology"
        raise MisoB200Error(f"infer_mosaic({what}=True): the model has no mask head (Mask R-CNN needed)")
    want_masks = masks or morphology
    dev = band_u8.device
    h, w = int(mosaic_hw[0]), int(mosaic_hw[1])
    grid = tile_grid(h, w, tile, overlap)
    mine = list(rank_tiles(len(grid), world, rank))
    dpi = int(model.roi_heads.detections_per_img)
    tmax = tiles_per_rank_max(len(grid), world)
    boxes = torch.zeros((max(len(mine), 1), dpi, 4), dtype=torch.float32, device=dev)
    scores = torch.zeros((max(len(mine), 1), dpi), dtype=torch.float32, device=dev)
    labels = torch.zeros((max(len(mine), 1), dpi), dtype=torch.int64, device=dev)
    counts = torch.zeros((max(len(mine), 1),), dtype=torch.int32, device=dev)
    probs = None
    with torch.inference_mode():
        for i0 in range(0, len(mine), batch_size):
            idx = mine[i0:i0 + batch_size]
            tiles = [band_u8[grid[t][0] - band_y0:grid[t][0] - band_y0 + tile, grid[t][1]:grid[t][1] + tile] for t in idx]
            if getattr(model, "_miso_b200_patched", False) and band_u8.shape[2] <= 4:
                from .patch import forward_uint8
                # ToTensor + normalize + resize + batch in one kernel; no full-tile mask paste (nobody reads it)
                res = forward_uint8(model, tiles, paste_masks=False)
            else:
                res = model([t.permute(2, 0, 1).to(torch.float32) / 255 for t in tiles])
            for j, r in enumerate(res):
                k = int(r["boxes"].shape[0])
                boxes[i0 + j, :k], scores[i0 + j, :k], labels[i0 + j, :k] = r["boxes"], r["scores"], r["labels"]
                counts[i0 + j] = k
                if want_masks:
                    if "mask_probs" not in r:
                        raise MisoB200Error("infer_mosaic(masks=True / morphology=True) needs a model patched by "
                                            "miso_b200.patch.patch_model")
                    if probs is None:
                        m = int(r["mask_probs"].shape[-1])
                        probs = torch.zeros((tmax * dpi, m, m), dtype=torch.float32, device=dev)
                    probs[(i0 + j) * dpi:(i0 + j) * dpi + k] = r["mask_probs"][:, 0]
    origins = torch.tensor([[float(grid[t][0]), float(grid[t][1])] for t in mine] or [[0.0, 0.0]], dtype=torch.float32,
                           device=dev).reshape(-1, 2)
    block = torch.zeros((tmax * dpi, 6), dtype=torch.float32, device=dev)
    block[:, 5] = -1.0
    if mine:
        pack_block(boxes[:len(mine)], scores[:len(mine)], labels[:len(mine)], counts[:len(mine)], origins, threshold,
                   len(mine) * dpi, out=block[:len(mine) * dpi])
    gathered = exchange(block, world, group)
    seam = SparseSeamNms(gathered.shape[0], dpi, dev)
    state = seam.launch(gathered, float(model.roi_heads.nms_thresh))
    crops = MosaicCrops(tmax * dpi, (h, w), int(band_u8.shape[2]), threshold, crop_capacity_bytes, dev)
    crops.bind_band(band_u8, band_y0)
    if want_masks and probs is not None:
        # frame of own row s: the tile it came from (boxes are tile-local, which is what the paste wants)
        frames = torch.zeros((tmax, 4), dtype=torch.int32)
        for i, t in enumerate(mine):
            y, x = grid[t]
            frames[i] = torch.tensor([x, y, min(tile, w - x), min(tile, h - y)], dtype=torch.int32)
        paste_boxes = torch.zeros((tmax * dpi, 4), dtype=torch.float32, device=dev)
        paste_boxes[:len(mine) * dpi] = boxes[:len(mine)].reshape(-1, 4)
        crops.bind_masks(probs, paste_boxes, frames.to(dev), dpi, mask_threshold, morphology=morphology)
    if png:
        crops.bind_png()
    if jpeg:
        crops.bind_jpeg()
    crops.launch(gathered, state, rank * tmax * dpi)
    seam.check()
    res = crops.results()
    if want_masks and probs is None:               # no own tiles: no crops
        res["masks"] = torch.empty((0,), dtype=torch.uint8, device=dev)
        if png:
            res["mask_png"] = torch.empty((0,), dtype=torch.uint8, device=dev)
            res["mask_png_offsets"] = torch.zeros((1,), dtype=torch.int64, device=dev)
        if morphology:
            res["morphology"] = torch.empty((0, len(MORPHOLOGY_FIELDS)), dtype=torch.float64, device=dev)
    if not masks:
        res.pop("masks", None)
        res.pop("mask_png", None)
        res.pop("mask_png_offsets", None)
    return {"gathered": gathered, "state": state, "crops": res}

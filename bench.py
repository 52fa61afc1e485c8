#!/usr/bin/env python
"""bench.py — headline benchmark of the detection post-processing + RoIAlign hot path on the tiled mosaic.

    python bench.py --gpus N --steps K --warmup W            (our arm, one process per GPU)
    python bench.py --impl reference --gpus N --steps K ...   (reference CPU arm, rank 0 only)
    python bench.py ... --dump-outputs DIR                    (also write the last timed step's outputs as DIR/*.npy;
                                                               the inputs are seeded, so two builds compare file by file)

Workload (every N, strong scaling): BASELINE.json config 5 — ONE 16384x16384 synthetic mosaic cut into 361 tiles
of 1024 px with 128 px overlap, partitioned over the N ranks in contiguous blocks. A "step" is one pass over the
whole mosaic: every rank runs its tiles through the post-head path in batches of 8 tiles (--batch; 4 is exactly
BASELINE config 2's batch) — every tile has config 2's per-image shape (1024^2 -> 800^2, 1000 RPN proposals/image,
256-channel pyramid, RoIAlign 7x7, 300 detections/image): RPN post-head stage -> MultiScaleRoIAlign -> detection
post-processing -> pack — then ONE
NCCL all-gather of the per-rank detection blocks, the seam NMS over all 108 300 gathered rows and the crops of the
rank's own surviving detections from its pixel band. The CNN parts (backbone, RPN head, box head) are not on
this path; their outputs are seeded random tensors (a function of the tile index, so every world size sees the
same tiles). All inputs are resident in HBM (22 GB at N=1) when the timed region starts.

  value     final detections/s of the whole mosaic (detections that survive the seam NMS and are cropped, summed
            over ranks) — K steps between two CUDA events, barrier + synchronize on both sides, max over ranks.
            Batches run one at a time (per-kernel timings are those of the kernel running alone); `pipelined` is
            the same job with three batches in flight on three streams (the plan's default mode).
  parity_gate  before timing: N>1 — every rank re-runs the WHOLE mosaic alone (world size 1) and asserts that the
            gathered rows, the seam-NMS keep set and its own crops (rectangles + bytes) are identical; N=1 — the
            keep set against torchvision's CPU _batched_nms_vanilla on the same 108 300 rows and sampled crops
            against numpy slices.
  roofline  RoIAlign (k_roi_align_nhwc4d, the default route; the opt-in TMA route is timed beside it): exact
            algorithmic bytes of every launch (SURVEY.md §8d, union of touched pixels rasterised on the GPU) /
            CUDA-event duration, over all launches of the timed region.
  aggregate Σ stage bytes / step time (SURVEY.md §8d) for the rank's whole step.
  e2e       the same job through miso_b200.mosaic.HostMosaicRunner: every batch's inputs come from pinned HOST
            memory (H2D inside the timed region), results (bounds, rectangles, crop bytes) return to pinned host.
  tv_cuda   (N=1) the kernels to beat on the same B200: torchvision's CUDA roi_align / batched_nms on the same inputs.
  cpu_baseline  (N=1) the CPU oracle port on one tile; `--impl reference` is torchvision's own CPU path on one tile/step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "detections_per_sec_posthead_path"
UNIT = "detections/s"


# ----------------------------------------------------------------------------------------------
def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="tiles per batch (each tile has BASELINE config 2's per-image shape; 4 = config 2's batch)")
    ap.add_argument("--mosaic", type=int, default=16384, help="mosaic side in pixels (16384 = BASELINE config 5)")
    ap.add_argument("--fast-roi-align", action="store_true", help="FMA RoIAlign (<=1e-5) instead of the bit-exact order")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gate", action="store_true", help="skip the parity gate (development only)")
    ap.add_argument("--no-extras", action="store_true", help="skip e2e / tv_cuda / cpu_baseline legs (development only)")
    ap.add_argument("--features-layout", default="channels_last", choices=["channels_last", "nchw"],
                    help="memory format of the synthetic FPN maps: channels_last = what the channels_last backbone that "
                         "patch_model sets up produces (gathered in place); nchw = torchvision's default layout")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


_SAMPLER_SRC = r"""
import os, sys, time
import pynvml as nv
parent = int(sys.argv[2])           # the benchmark's pid, passed in: it may be gone before this line runs
nv.nvmlInit()
h = nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))
print("max", nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM), flush=True)
while os.getppid() == parent:       # ends with the benchmark, also when that one stops on an error
    print(time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), nv.nvmlDeviceGetCurrentClocksEventReasons(h), flush=True)
    time.sleep(0.001)
"""


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: a helper process polls NVML every ~1 ms
    (its own interpreter, so it neither holds this process's GIL nor delays the launch loop); only the
    samples stamped inside [t0, t1] are kept."""

    def __init__(self, index: int):
        import tempfile
        self.out = tempfile.TemporaryFile(mode="w+")
        try:
            self.proc = subprocess.Popen([sys.executable, "-c", _SAMPLER_SRC, str(index), str(os.getpid())], stdout=self.out,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def summary(self, t0: float, t1: float):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.out.seek(0)
        mx, rows, before = None, [], None
        for line in self.out.read().splitlines():
            f = line.split()
            if len(f) == 2 and f[0] == "max":
                mx = int(f[1])
            elif len(f) == 3:
                ts, mhz, mask = float(f[0]), int(f[1]), int(f[2])
                if t0 <= ts <= t1:
                    rows.append((mhz, mask))
                elif ts < t0:
                    before = (mhz, mask)
        if not rows and before is not None:
            rows = [before]
        sm = sorted(r[0] for r in rows)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
        reasons = sorted({n for _, m in rows for n, b in bits.items() if m & b})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(rows)}


def roi_align_algorithmic_bytes(proposals, counts, grids, thresholds, scales, channels, pooled, sr=2):
    """20*K + 4*C*P^2*K + 4*C*sum_levels |union of touched pixels| (SURVEY.md §8d) for one launch, on the device:
    the sample coordinates follow the reference formula (Appendix B.2) with one fp32 rounding per torch op, the
    union is rasterised exactly into one boolean map per level. proposals [n, R, 4], counts [n] (device tensors)."""
    import torch
    dev = proposals.device
    n, R = proposals.shape[0], proposals.shape[1]
    live = torch.arange(R, device=dev)[None, :] < counts[:, None].to(torch.int64)
    b = proposals
    area = (b[..., 2] - b[..., 0]) * (b[..., 3] - b[..., 1])
    lvl = torch.zeros((n, R), dtype=torch.int64, device=dev)
    for t in thresholds:
        lvl += (area >= torch.tensor(t, dtype=torch.float32, device=dev)).to(torch.int64)
    pp = torch.arange(pooled, device=dev, dtype=torch.float32).repeat_interleave(sr)[None, :]
    ii = torch.arange(sr, device=dev, dtype=torch.float32).repeat(pooled)[None, :]
    touched = 0
    for l, (gh, gw) in enumerate(grids):
        sel = live & (lvl == l)
        idx = sel.nonzero()
        if idx.shape[0] == 0:
            continue
        bb, img = b[sel], idx[:, 0]
        sc = torch.tensor(scales[l], dtype=torch.float32, device=dev)

        def axis(lo_c, hi_c, size):
            s0, e0 = lo_c * sc, hi_c * sc
            r = torch.clamp(e0 - s0, min=1.0)
            binsz = (r / float(pooled))[:, None]
            v = (s0[:, None] + pp * binsz) + ((ii + 0.5) * binsz) / float(sr)
            ok = ~((v < -1.0) | (v > float(size)))
            v = torch.clamp(v, min=0.0)
            lo = torch.clamp(v.to(torch.int64), max=size - 1)
            hi = torch.clamp(lo + 1, max=size - 1)
            return torch.cat([lo, hi], 1), torch.cat([ok, ok], 1)

        ys, yv = axis(bb[:, 1], bb[:, 3], gh)
        xs, xv = axis(bb[:, 0], bb[:, 2], gw)
        k, S = ys.shape
        V = yv[:, :, None] & xv[:, None, :]
        m = torch.zeros((n, gh, gw), dtype=torch.bool, device=dev)
        m[img[:, None, None].expand(k, S, S)[V], ys[:, :, None].expand(k, S, S)[V], xs[:, None, :].expand(k, S, S)[V]] = True
        touched += int(m.sum())
    k_live = int(live.sum())
    return 20 * k_live + 4 * channels * pooled * pooled * k_live + 4 * channels * touched, k_live, touched


def dump_outputs(out_dir, gathered, state, res, rank=0, world=1, budget=60_000_000, seed=0):
    """Writes what one mosaic pass hands its caller as out_dir/<name>.npy, in float32 where that holds the values
    exactly and float64 otherwise: the gathered detection rows [rows, 6] (box, score, label or -1), the seam NMS
    state of every row (1 kept, 2 suppressed, 3 ignored) and the rank's crops (annotation bounds, integer
    rectangles, source rows, byte offsets). The crop bytes (~2 GB per pass at the default size) do not fit the
    budget: a fixed, seeded sample of byte positions goes to crop_pixel_index and the bytes there to crop_pixels.
    With several ranks the gathered rows and the seam state are the same on every rank and rank 0 alone writes
    them; every rank writes its own crop arrays as <name>.rank<r>.npy within an equal share of what is left.
    `budget` counts the arrays of all ranks together and keeps all files, headers included, under 64 MB.
    Returns {file name without .npy: array} of what this rank wrote."""
    import numpy as np
    import torch
    shared = {"gathered_rows": gathered.float(), "seam_state": state.float()}
    own = {"crop_xywh": res["xywh"].float(), "crop_rects": res["rects"].float(), "crop_src_rows": res["src"].float(),
           "crop_offsets": res["offsets"].double()}
    shared, own = ({k: v.cpu().numpy() for k, v in d.items()} for d in (shared, own))
    left = (budget - sum(a.nbytes for a in shared.values())) // world - sum(a.nbytes for a in own.values())
    if left < 0:
        raise SystemExit(f"--dump-outputs: the detection arrays alone exceed {budget} bytes")
    pixels = res["pixels"]
    k = min(pixels.numel(), left // 12)                          # 8 B index + 4 B value per sampled byte
    idx = np.sort(np.random.default_rng(seed).choice(pixels.numel(), k, replace=False)) if k < pixels.numel() else np.arange(k)
    own["crop_pixel_index"] = idx.astype(np.float64)
    own["crop_pixels"] = pixels[torch.from_numpy(idx).to(pixels.device)].float().cpu().numpy()
    suffix = f".rank{rank}" if world > 1 else ""
    out = dict(shared) if rank == 0 else {}
    out.update({name + suffix: a for name, a in own.items()})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return out


# ----------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU implementation of the path: torchvision 0.26 CPU ops and modules
    (filter_proposals, MultiScaleRoIAlign, postprocess_detections, resize_boxes) plus miso's score
    filter / coords_int / crop slice (restated: miso.* needs lxml/skimage, absent in this image).
    Bounded sample: ONE tile of the mosaic per step (the mosaic's per-tile work; the reference never tiles, so the
    exchange + seam NMS have no reference counterpart and are not in this arm). Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import numpy as np
    import torch
    from torchvision.models.detection.anchor_utils import AnchorGenerator
    from torchvision.models.detection.image_list import ImageList
    from torchvision.models.detection.roi_heads import RoIHeads
    from torchvision.models.detection.rpn import RegionProposalNetwork, RPNHead, concat_box_prediction_layers
    from torchvision.models.detection.transform import resize_boxes
    from torchvision.ops.poolers import MultiScaleRoIAlign
    from miso_b200 import workload
    from oracle import miso_path as M

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    mw = workload.mosaic(args.mosaic, args.mosaic, features_layout="nchw")
    w = workload.faster_rcnn_batch(num_images=1, seed=0, pin=False)
    h = w.host
    ag = AnchorGenerator(w.rpn.sizes, w.rpn.aspect_ratios)
    rpn = RegionProposalNetwork(ag, RPNHead(8, 3), 0.7, 0.3, 256, 0.5, dict(training=2000, testing=w.rpn.pre_nms_top_n),
                                dict(training=2000, testing=w.rpn.post_nms_top_n), w.rpn.nms_thresh).eval()
    heads = RoIHeads(None, None, None, 0.5, 0.5, 512, 0.25, (10.0, 10.0, 5.0, 5.0), w.det.score_thresh,
                     w.det.nms_thresh, w.det.detections_per_img)
    pool = MultiScaleRoIAlign(["0", "1", "2", "3"], 7, 2)
    il = ImageList(torch.zeros(1, 3, *w.shapes.padded_image_size), list(w.shapes.image_sizes))
    img = h["images"][0].numpy()

    def step():
        with torch.inference_mode():
            anchors = ag(il, h["objectness"])
            napl = [o.shape[1] * o.shape[2] * o.shape[3] for o in h["objectness"]]
            objectness, deltas = concat_box_prediction_layers(list(h["objectness"]), list(h["deltas"]))
            proposals = rpn.box_coder.decode(deltas, anchors).view(1, -1, 4)
            boxes, _ = rpn.filter_proposals(proposals, objectness, il.image_sizes, napl)
            feats = pool({str(i): f for i, f in enumerate(h["features"])}, boxes, il.image_sizes)
            k = boxes[0].shape[0]
            db, ds, dl = heads.postprocess_detections(h["class_logits"][0][:k], h["box_regression"][0][:k], boxes, il.image_sizes)
            rb = resize_boxes(db[0], list(w.shapes.image_sizes[0]), list(w.shapes.original_image_sizes[0]))
            _, _, _, _, _, crops = M.filter_and_crop(img, rb.numpy(), ds[0].numpy(), dl[0].numpy(), w.threshold)
        return len(crops), feats.shape[0]

    for _ in range(min(args.warmup, 2)):
        step()
    t0 = time.perf_counter()
    dets = 0
    for _ in range(args.steps):
        d, _ = step()
        dets += d
    dt = time.perf_counter() - t0
    value = dets / dt
    sample = ("1 tile of the mosaic per step (torchvision CPU ops + miso filter/crop restated in numpy); per-tile work only — "
              "the reference never tiles, so it has no exchange / seam NMS")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": mw.name + " (sampled: 1 tile/step, NCHW maps)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ----------------------------------------------------------------------------------------------
def cpu_baseline_port(steps=2):
    """The CPU oracle port of the per-tile path on ONE tile (bounded sample)."""
    from oracle import native
    from oracle import pipeline as ref_pipeline
    from miso_b200 import workload
    native.lib()
    w = workload.faster_rcnn_batch(num_images=1, seed=0, pin=False)
    h = {k: [t.numpy() for t in v] for k, v in w.host.items()}
    kw = dict(padded_image_size=w.shapes.padded_image_size, image_sizes=w.shapes.image_sizes,
              original_image_sizes=w.shapes.original_image_sizes, sizes=w.rpn.sizes, aspect_ratios=w.rpn.aspect_ratios,
              pre_nms_top_n=w.rpn.pre_nms_top_n, post_nms_top_n=w.rpn.post_nms_top_n,
              detections_per_img=w.det.detections_per_img, threshold=w.threshold)
    args_ = (h["objectness"], h["deltas"], h["features"], h["class_logits"][0], h["box_regression"][0], h["images"])
    ref_pipeline.run(*args_, **kw)
    t0 = time.perf_counter()
    dets = 0
    tm = {}
    for _ in range(steps):
        out = ref_pipeline.run(*args_, timings=tm, **kw)
        dets += sum(len(o["crops"]) for o in out)
    dt = time.perf_counter() - t0
    return {"value": dets / dt, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
            "sample": f"1 tile of the mosaic, {steps} passes of the oracle (C NMS/RoIAlign with OpenMP + numpy); "
                      f"last pass: rpn {tm.get('rpn_s', 0):.3f}s roi_align {tm.get('roi_align_s', 0):.3f}s "
                      f"det+crop {tm.get('det_crop_s', 0):.3f}s"}


def tv_cuda_leg(plan, batch0, w, dev):
    """The kernels to beat: torchvision's own CUDA ops on the same B200 and the same inputs (SURVEY §2.3 K2/K3/K5)."""
    import torch
    import torchvision
    from torchvision.ops import boxes as tvb
    from torchvision.ops.poolers import MultiScaleRoIAlign as TvPool
    from miso_b200 import mosaic, ops

    def timeit(fn, iters=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for a, b in evs:
            a.record(); fn(); b.record()
        torch.cuda.synchronize()
        t = sorted(a.elapsed_time(b) for a, b in evs)
        return t[len(t) // 2]

    out = {"torchvision": torchvision.__version__}
    hp = plan.slots[plan.batch_sizes[0]][0]
    hp.rebind(batch0["objectness"], batch0["deltas"], batch0["features"], batch0["class_logits"], batch0["box_regression"])
    hp.rpn(); torch.cuda.synchronize()
    cnt = hp.prop_counts.tolist()
    props = [hp.proposals[i, :cnt[i]].clone() for i in range(len(cnt))]
    sizes = list(w.base.shapes.image_sizes) * len(cnt)
    pool = TvPool(["0", "1", "2", "3"], 7, 2)
    for name, feats in (("nchw", [f.contiguous() for f in batch0["features"]]), ("channels_last", batch0["features"])):
        x = {str(i): f for i, f in enumerate(feats)}
        out[f"multiscale_roi_align_{name}_ms"] = timeit(lambda: pool(x, props, sizes))
    out["multiscale_roi_align_ours_ms"] = timeit(lambda: hp.roi_align())
    # seam NMS: torchvision batched_nms (CUDA, its own strategy rule) on the live rows of the gathered block
    g = plan.gathered
    live = g[:, 5] >= 0
    rows = g[live]
    bx, sc, lb = rows[:, :4].contiguous(), rows[:, 4].contiguous(), rows[:, 5].to(torch.int64)
    out["seam_rows_live"] = int(rows.shape[0])
    out["seam_batched_nms_torchvision_ms"] = timeit(lambda: tvb.batched_nms(bx, sc, lb, plan.iou), iters=3, warm=1)
    out["seam_nms_ours_sparse_ms"] = timeit(lambda: plan.seam.launch(g, plan.iou))
    dense = mosaic.SeamNms(g.shape[0], w.base.shapes.num_classes, dev)
    out["seam_nms_ours_dense_ms"] = timeit(lambda: dense.launch(g, plan.iou), iters=3, warm=1)
    # config 4: 200 000 boxes x 80 classes
    gen = torch.Generator(device=dev).manual_seed(4)
    nb = 200_000
    c = torch.rand((nb, 2), generator=gen, device=dev) * 4096
    s = torch.exp(torch.rand((nb, 2), generator=gen, device=dev) * (torch.log(torch.tensor(256.0)) - torch.log(torch.tensor(8.0))) + torch.log(torch.tensor(8.0)))
    b4 = torch.cat([c - s / 2, c + s / 2], 1).contiguous()
    s4 = torch.linspace(0, 1, nb, device=dev)[torch.randperm(nb, generator=gen, device=dev)].contiguous()
    l4 = torch.randint(0, 80, (nb,), generator=gen, device=dev)
    out["config4_batched_nms_torchvision_ms"] = timeit(lambda: tvb.batched_nms(b4, s4, l4, 0.5), iters=3, warm=1)
    out["config4_batched_nms_ours_ms"] = timeit(lambda: ops.batched_nms(b4, s4, l4, 0.5), iters=3, warm=1)
    return out


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from miso_b200 import _lib, mosaic, pipeline, workload

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    host_affinity = (mosaic.bind_host_near_gpu(dev) if world > 1 and not os.environ.get("MB_BENCH_NO_BIND")
                     else {"bound": False, "why": "single process" if world == 1 else "MB_BENCH_NO_BIND"})
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None     # started early: it must be polling before the timed region
    w = workload.mosaic(args.mosaic, args.mosaic, features_layout=args.features_layout)
    grid = mosaic.tile_grid(w.height, w.width, w.tile, w.overlap)
    T = len(grid)
    exact = not args.fast_roi_align

    def make_plan(r, g, crop_cap=None):
        mine = list(mosaic.rank_tiles(T, g, r))
        sizes = [min(args.batch, len(mine) - i) for i in range(0, len(mine), args.batch)]

        def make_hp(n):
            return pipeline.HotPath(w.shapes(n), w.base.rpn, w.base.det, threshold=w.base.threshold, crop_capacity_bytes=1 << 20,
                                    exact_roi_align=exact, device=dev)

        pl = mosaic.MosaicPlan(grid, w.tile, (w.height, w.width), make_hp, sizes, rank=r, world=g, threshold=w.base.threshold,
                               iou_threshold=w.base.det.nms_thresh, crop_capacity_bytes=crop_cap, device=dev)
        return pl, mine, sizes

    def batch_tiles(mine, sizes):
        out, i0 = [], 0
        for n in sizes:
            out.append(mine[i0:i0 + n])
            i0 += n
        return out

    # ~18 KB per crop, 300 detections per tile: room for every detection of the rank's tiles plus slack
    crop_cap = int(len(mosaic.rank_tiles(T, world, rank)) * 300 * 20_000 * 1.15) + (64 << 20)
    plan, mine, sizes = make_plan(rank, world, crop_cap)
    tiles_of = batch_tiles(mine, sizes)
    batches = [w.batch_inputs(ts, dev) for ts in tiles_of]           # resident in HBM for the whole run
    y0, y1 = mosaic.rank_band(grid, w.tile, w.height, world, rank)
    band = w.band(y0, y1, dev)
    plan.bind_band(band, y0)
    dpi = plan.dpi
    torch.cuda.synchronize()

    # ---- warm-up ----
    for _ in range(max(args.warmup, 3)):
        plan.run(batches, serial=True)
    plan.run(batches)
    barrier()
    res = plan.results()
    my_dets, my_crop_bytes = res["count"], res["bytes"]

    # ---- parity gate ----
    gate = {"ran": False}
    if not args.no_gate:
        if world > 1:
            # the WHOLE mosaic on this rank alone (inputs streamed, 8 batches at a time), then compare
            p1, mine1, sizes1 = make_plan(0, 1, 1 << 20)
            tl1 = batch_tiles(mine1, sizes1)
            CH = 8
            for c0 in range(0, len(sizes1), CH):
                chunk = [w.batch_inputs(ts, dev) for ts in tl1[c0:c0 + CH]]
                p1.run_tiles(chunk, serial=True, first=c0, count=len(chunk))
                torch.cuda.synchronize()
                del chunk
            p1.seam.launch(p1.gathered, p1.iou)
            p1.seam.check()
            rows1 = torch.arange(T * dpi, device=dev)
            tile1, slot1 = rows1 // dpi, rows1 % dpi
            bounds = [mosaic.rank_tiles(T, world, r).start for r in range(world)] + [T]
            owner = torch.bucketize(tile1, torch.tensor(bounds[1:], device=dev), right=True)
            first_tile = torch.tensor(bounds[:-1], device=dev)[owner]
            to_w = (owner * plan.tmax + (tile1 - first_tile)) * dpi + slot1          # world-1 row -> row in this run's gathered buffer
            same_rows = bool(torch.equal(plan.gathered[to_w], p1.gathered))
            k1 = torch.zeros_like(plan.seam.state)
            k1[to_w] = p1.seam.state
            pad = torch.ones_like(plan.seam.state, dtype=torch.bool)
            pad[to_w] = False
            same_keep = bool(torch.equal(plan.seam.state[~pad], k1[~pad])) and bool((plan.seam.state[pad] == 3).all())
            # own crops from the world-1 keep set (rows of this rank's tiles are contiguous in world-1 order too)
            lo1 = mine[0] * dpi
            c1 = mosaic.MosaicCrops(plan.block_rows, (w.height, w.width), 3, w.base.threshold, plan.crops.capacity, dev)
            c1.bind_band(band, y0)
            blk1 = torch.zeros((plan.block_rows, 6), dtype=torch.float32, device=dev)
            blk1[:, 5] = -1.0
            st1 = torch.full((plan.block_rows,), 3, dtype=torch.int32, device=dev)
            nmine = len(mine) * dpi
            blk1[:nmine] = p1.gathered[lo1:lo1 + nmine]
            st1[:nmine] = p1.seam.state[lo1:lo1 + nmine]
            c1.launch(blk1, st1, 0)
            r1 = c1.results()
            same_crops = (r1["count"] == res["count"] and bool(torch.equal(r1["rects"], res["rects"])) and
                          bool(torch.equal(r1["xywh"], res["xywh"])) and bool(torch.equal(r1["src"], res["src"])) and
                          bool(torch.equal(r1["pixels"], res["pixels"])))
            ok = torch.tensor([int(same_rows and same_keep and same_crops)], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            gate = {"ran": True, "kind": f"world {world} == world 1 on every rank (gathered rows, seam keep set, own crop rectangles + bytes)",
                    "rank0": {"rows": same_rows, "keep": same_keep, "crops": same_crops}, "all_ranks_ok": bool(ok[0])}
            if not bool(ok[0]):
                raise SystemExit(f"parity gate failed on rank {rank}: rows {same_rows} keep {same_keep} crops {same_crops}")
            del p1, c1, blk1, st1
            torch.cuda.empty_cache()
        else:
            from torchvision.ops import boxes as tvb
            g_host = plan.gathered.cpu()
            live = g_host[:, 5] >= 0
            idx = live.nonzero().flatten()
            torch.set_num_threads(os.cpu_count() or 1)
            t0 = time.perf_counter()
            keep = tvb._batched_nms_vanilla(g_host[idx, :4].contiguous(), g_host[idx, 4].contiguous(), g_host[idx, 5].to(torch.int64), plan.iou)
            t_ref = time.perf_counter() - t0
            ref_rows = torch.sort(idx[keep]).values
            got_rows = (plan.seam.state == 1).nonzero().flatten().cpu()
            same_keep = bool(torch.equal(ref_rows, got_rows))
            # sampled crops against numpy slices of the mosaic
            from oracle import miso_path as M
            pick = np.linspace(0, res["count"] - 1, 64).astype(np.int64) if res["count"] else np.zeros(0, np.int64)
            rects, offs = res["rects"].cpu().numpy(), res["offsets"].cpu().numpy()
            src = res["src"].cpu().numpy()
            gnp = g_host.numpy()
            same_crops = True
            for j in pick:
                ci = M.coords_int(M.annotations_xywh(gnp[src[j], :4][None]))[0]
                ref = M.crop(band[max(ci[1], 0):max(ci[3], 0)].cpu().numpy(), (ci[0], 0, ci[2], max(ci[3], 0) - max(ci[1], 0)))
                got = res["pixels"][offs[j]:offs[j + 1]].cpu().numpy().reshape(rects[j][3], rects[j][2], 3)
                same_crops = same_crops and np.array_equal(ref, got)
            gate = {"ran": True, "kind": "N=1: seam keep set == torchvision CPU _batched_nms_vanilla on all gathered rows; 64 sampled crops == numpy slices",
                    "live_rows": int(idx.numel()), "kept": int(got_rows.numel()), "keep": same_keep, "crops": bool(same_crops),
                    "torchvision_cpu_seam_nms_s": t_ref}
            if not (same_keep and same_crops):
                raise SystemExit(f"parity gate failed: keep {same_keep} crops {same_crops}")

    # ---- exact algorithmic bytes of every RoIAlign launch (proposals are deterministic per batch) ----
    alg = []
    hp0 = plan.slots[sizes[0]][0]
    q = hp0.roi_params
    thr = [q.level_thresholds[i] for i in range(q.num_levels - 1)]
    scl = [q.spatial_scale[i] for i in range(q.num_levels)]
    sh = w.base.shapes
    for bi, n in enumerate(sizes):
        hp = plan.slots[n][0]
        hp.rebind(batches[bi]["objectness"], batches[bi]["deltas"], batches[bi]["features"], batches[bi]["class_logits"], batches[bi]["box_regression"])
        hp.rpn()
        alg.append(roi_align_algorithmic_bytes(hp.proposals, hp.prop_counts, sh.feature_grids, thr, scl, sh.channels, sh.pooled))
    torch.cuda.synchronize()
    tma0 = _lib.load().mb_roi_align_tma_launches()

    # ---- timed region: K mosaic passes, batches one at a time; every RoIAlign launch bracketed by events ----
    roi_ev = []
    recording = [False]

    def before_roi(bi, hp_i, st):
        if recording[0]:
            e = (bi, torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            roi_ev.append(e)
            e[1].record(st)

    def after_roi(bi, hp_i, st):
        if recording[0]:
            roi_ev[-1][2].record(st)

    plan.hooks.update(before_roi=before_roi, after_roi=after_roi)

    def timed(k, serial):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        th = time.perf_counter()
        for _ in range(k):
            plan.run(batches, serial=serial)
        host = (time.perf_counter() - th) / k
        e1.record()
        barrier()
        t_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        return float(t_ms[0]), host

    wall0 = time.time()
    recording[0] = True
    ms, host_s = timed(args.steps, True)
    recording[0] = False
    clocks = sampler.summary(wall0, time.time()) if rank == 0 else None
    tma_used = _lib.load().mb_roi_align_tma_launches() - tma0
    if args.dump_outputs:                                    # before the legs below overwrite the plan's buffers
        dump_outputs(args.dump_outputs, plan.gathered, plan.seam.state, plan.results(), rank, world)
    t = torch.tensor([float(my_dets), float(my_crop_bytes)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    total_dets, total_crop_bytes = float(t[0]), float(t[1])
    ms_per_step = ms / args.steps
    value = total_dets / (ms_per_step * 1e-3)
    roi_ms = [(bi, a.elapsed_time(b)) for bi, a, b in roi_ev]
    roi_bytes_sum = sum(alg[bi][0] for bi, _ in roi_ms)
    roi_time_sum = sum(tt for _, tt in roi_ms) * 1e-3
    full = [tt for bi, tt in roi_ms if sizes[bi] == args.batch]

    # ---- stage breakdown of one full batch (events between the stages, outside the timed region) ----
    hp = plan.slots[sizes[0]][0]
    hp.rebind(batches[0]["objectness"], batches[0]["deltas"], batches[0]["features"], batches[0]["class_logits"], batches[0]["box_regression"])
    sev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(7)]
    for es in sev:
        es[0].record(); hp.rpn(); es[1].record(); hp.roi_align(); es[2].record(); hp.detections(); es[3].record()
    tev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(5)]
    for es in tev:
        es[0].record(); plan.seam.launch(plan.gathered, plan.iou); es[1].record()
        plan.crops.launch(plan.gathered, plan.seam.state, rank * plan.block_rows); es[2].record()
    barrier()
    med = lambda xs: sorted(xs)[len(xs) // 2]
    stage_ms = {nm: med([es[j].elapsed_time(es[j + 1]) for es in sev]) for j, nm in enumerate(("rpn", "roi_align", "det_postprocess"))}
    stage_ms["seam_nms"] = med([es[0].elapsed_time(es[1]) for es in tev])
    stage_ms["select_crop"] = med([es[1].elapsed_time(es[2]) for es in tev])

    # ---- the RoIAlign launch in the other arithmetic mode and on the gather kernel (same proposals), for reference ----
    def roi_variant(exact_flag, force):
        hp.roi_params.exact, hp.roi_params.force_gather = exact_flag, force
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(7)]
        for a_, b_ in ev:
            hp.rpn(); a_.record(); hp.roi_align(); b_.record(); hp.detections()
        torch.cuda.synchronize()
        hp.roi_params.exact, hp.roi_params.force_gather = int(exact), 0
        return med([a_.elapsed_time(b_) for a_, b_ in ev])

    other_ms = roi_variant(int(not exact), 0)
    tma_ms = roi_variant(int(exact), 2)

    # ---- host cost of enqueuing a batch (a burst that fits the launch queue, so the host never waits for the device) ----
    nb_host = min(len(batches), 8)
    torch.cuda.synchronize()
    th = time.perf_counter()
    plan.run_tiles(batches[:nb_host], serial=True, first=0, count=nb_host)
    host_us_per_batch = 1e6 * (time.perf_counter() - th) / nb_host
    torch.cuda.synchronize()

    # ---- the same K passes with three batches in flight (the plan's default mode), tile phase replayed from a CUDA graph ----
    plan.hooks.clear()
    plan.capture_tiles(batches)

    def timed_passes(k, **kw):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(k):
            plan.run(**kw)
        e1.record()
        barrier()
        t_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        return float(t_ms[0])

    timed_passes(1, graph=True)
    ms_graph = timed_passes(args.steps, graph=True) / args.steps
    timed_passes(1, batches=batches)
    ms_streams = timed_passes(args.steps, batches=batches) / args.steps
    ms3 = min(ms_graph, ms_streams)
    pipelined = {"value": total_dets / (ms3 * 1e-3), "unit": UNIT, "ms_per_step": ms3, "steps": args.steps, "batches_in_flight": 3,
                 "ms_per_step_graph_replay": ms_graph, "ms_per_step_live_streams": ms_streams,
                 "note": "rpn(k+2) | roi_align(k+1) | detections(k) on three streams, per-batch stage order kept by events; measured both "
                         "enqueued live and with the rank's whole tile phase replayed from one CUDA graph (MosaicPlan.capture_tiles); "
                         "value is the faster of the two"}

    # ---- e2e: every batch's inputs from pinned HOST memory, results back to pinned host ----
    e2e = None
    if not args.no_extras:
        POOL = min(len(batches), 12)
        host_pool = [{k: [x.cpu().pin_memory() for x in v] for k, v in batches[i].items()} for i in range(POOL)]
        by_size = {}
        for i in range(POOL):
            by_size.setdefault(sizes[i], []).append(host_pool[i])
        for i, n in enumerate(sizes):                        # sizes outside the pool (the short last batch) get their own host copy
            if n not in by_size:
                by_size[n] = [{k: [x.cpu().pin_memory() for x in v] for k, v in batches[i].items()}]
        use = {n: 0 for n in by_size}
        host_batches = []
        for n in sizes:
            host_batches.append(by_size[n][use[n] % len(by_size[n])])
            use[n] += 1
        runner = mosaic.HostMosaicRunner(plan, {n: v[0] for n, v in by_size.items()})
        runner.run(host_batches)
        barrier()
        e2e_steps = max(1, min(args.steps, 3))
        t0 = time.perf_counter()
        e2e_dets = 0
        for _ in range(e2e_steps):
            e2e_dets += runner.run(host_batches)["count"]
        barrier()
        e2e_s = (time.perf_counter() - t0) / e2e_steps
        te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        td = torch.tensor([float(e2e_dets) / e2e_steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
            dist.all_reduce(td, op=dist.ReduceOp.SUM)
        hb = torch.tensor([float(runner.h2d_bytes), float(runner.d2h_bytes)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(hb, op=dist.ReduceOp.SUM)
        e2e = {"value": float(td[0]) / float(te[0]), "unit": UNIT, "h2d_bytes_per_step": int(hb[0]), "d2h_bytes_per_step": int(hb[1]), "host_affinity": host_affinity,
               "ms_per_step": 1e3 * float(te[0]), "steps": e2e_steps,
               "h2d_gbs_per_gpu": float(hb[0]) / world / float(te[0]) / 1e9,
               "api": "miso_b200.mosaic.HostMosaicRunner (pinned host in/out; copy-in stream | 3 compute streams | copy-out stream)",
               "note": f"host inputs cycle through a pinned pool of the rank's first {POOL} batches (the bytes copied per step are those of "
                       f"the whole mosaic share); detections counted from this run"}
        del runner, host_pool, host_batches, by_size

    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        extras["tv_cuda"] = tv_cuda_leg(plan, batches[0], w, dev)
        if not args.no_cpu_baseline:
            extras["cpu_baseline"] = cpu_baseline_port()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (RoIAlign) and the aggregate of the step ----
    peak, peak_src = peaks()
    achieved = roi_bytes_sum / roi_time_sum / 1e9
    roi_kernel = "k_roi_geom+k_roi_align_tma" if tma_used > 0 else ("k_roi_align_nhwc4d" if args.features_layout == "channels_last" else "k_nchw_to_nhwc+k_roi_align_nhwc4d")
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roi_align_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as fh:
            entry = json.load(fh).get(roi_kernel, {})
            # captured per launch size (tiles per batch); a size without its own capture reports null, not a scaled guess
            traffic = entry.get("dram_bytes_per_launch_by_tiles", {}).get(str(args.batch), entry.get("dram_bytes_per_launch") if args.batch == 4 else None)
    # aggregate (SURVEY §8d): RoIAlign bytes + RPN (objectness scan 2x4 B/anchor + 36 B per decoded winner) + detection
    # post-processing (4*R*5C in + 24 B/det) per tile, pack/unpack + seam rows (24 B each, read twice), crops read+write
    n_anchor = sum(3 * gh * gw for gh, gw in sh.rpn_grids)
    per_tile_small = 8 * n_anchor + 36 * (4 * 1000 + 507) + 4 * 1000 * 5 * sh.num_classes + 24 * dpi + 24 * dpi
    rank_bytes = sum(a[0] for a in alg) + len(mine) * per_tile_small + 2 * 24 * world * plan.block_rows + 2 * my_crop_bytes
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3) + 1,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": w.name, "tiles": T, "tiles_rank0": len(mine), "tiles_per_batch": args.batch,
                   "batch_shape": f"{args.batch} tiles per batch, each with BASELINE config 2's per-image shape (1024^2 -> 800^2, 1000 proposals, 256 ch, 7x7, 300 dets)",
                   "features_layout": args.features_layout,
                   "l2": f"inputs larger than L2: every batch has its own {args.batch * w.bytes_per_tile() / 1e6:.0f} MB of inputs ({len(mine) * w.bytes_per_tile() / 1e9:.1f} GB resident on rank 0) + {args.batch * 50.2:.0f} MB RoIAlign output",
                   "roi_align_mode": "fast(fma)" if args.fast_roi_align else "exact(reference op order)",
                   "multi_gpu": (f"strong scaling: contiguous tile blocks per rank, one NCCL all_gather_into_tensor of [{plan.block_rows}, 6] rows per rank, "
                                 "sparse seam NMS replicated on every rank, crops cut by the rank that owns the source tile") if world > 1 else "single GPU",
                   "detections_per_step": total_dets, "gathered_rows": world * plan.block_rows, "crop_bytes_per_step": total_crop_bytes,
                   "tiles_per_s": T / (ms_per_step * 1e-3)},
        "parity_gate": gate,
        "roofline": {"bound": "hbm", "kernel": roi_kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "algorithmic_bytes": alg[0][0], "peak_source": peak_src,
                     "launches_timed": len(roi_ms), "kernel_ms_mean": 1e3 * roi_time_sum / len(roi_ms),
                     "kernel_ms_mean_full_batches": sum(full) / max(len(full), 1), "kernel_ms_min": min(tt for _, tt in roi_ms),
                     "rois_batch0": alg[0][1], "touched_pixels_batch0": alg[0][2],
                     "kernel_share_of_step": roi_time_sum * 1e3 / ms,
                     "note": "algorithmic bytes are exact per launch (every batch has its own proposals); the event bracket contains every kernel of the RoIAlign call (one on the default route)",
                     "limiter": "L2->SM fabric: the launch moves ~1.3 GB of deduplicated taps out of L2 at ~9.5 TB/s while DRAM sees about the algorithmic bytes (RoIs overlap, L2 absorbs the re-reads); DESIGN.md section 7, profiles/r2_roi_align_ncu_full.txt",
                     "other_mode": {"mode": "fast(fma)" if exact else "exact", "kernel_ms": other_ms, "frac": alg[0][0] / (other_ms * 1e-3) / 1e9 / peak},
                     "tma_route": {"kernel": "k_roi_geom+k_roi_align_tma (opt-in, MB_ROI_TMA=1)", "kernel_ms": tma_ms, "frac": alg[0][0] / (tma_ms * 1e-3) / 1e9 / peak}},
        "aggregate": {"bytes_rank0_per_step": rank_bytes, "achieved": rank_bytes / (ms_per_step * 1e-3) / 1e9, "unit": "GB/s",
                      "frac": rank_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                      "frac_pipelined": rank_bytes / (ms3 * 1e-3) / 1e9 / peak,
                      "note": "sum of the stages' algorithmic bytes (SURVEY 8d) on rank 0 / its step time; RoIAlign is ~99 % of the bytes"},
        "stage_ms": stage_ms, "host_enqueue_ms_per_step": 1e3 * host_s, "host_enqueue_us_per_batch": host_us_per_batch,
        "pipelined": pipelined,
        "gpu_launches": plan.launches_per_run * args.steps,
        "clocks": clocks,
    }
    if e2e is not None:
        line["e2e"] = e2e
    line.update(extras)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)

"""mb_crop_masks at mosaic size: the per-crop instance masks of config 5's seam survivors, timed alone.

Input (seeded): a 16384^2 RGB mosaic cut into 361 tiles of 1024 px (128 px overlap), 300 detections per tile = 108 300
crops, every row kept. Boxes are tile-local, drawn like tests/cases.stress_rois with sqrt(area) log-uniform in
[16, 160] px (mean crop ~5 200 px, close to config 5's 2.0 GB of RGB crops over 108 300 rows, ~6 150 px), the
paste frame of a row is its tile; M = 28 probabilities uniform in [0, 1). The plan (mb_crop_plan) and the pixel
gather run once through MosaicCrops; then mb_crop_masks alone is timed with CUDA events over `reps` launches after
a warm-up. Its working set (~0.95 GB: 340 MB of probabilities, ~600 MB of masks) exceeds the 126 MB L2, so every pass reads from HBM.

Bytes counted (algorithmic): 4*M^2*K probabilities read, 16*K paste boxes read, sum(h*w) mask bytes written. The
per-crop metadata (rect, src, offset, frame: 44 B) is not counted. The share is of the 7.7 TB/s data-sheet HBM3e
figure of one B200; the card name and power limit are read in the same run.
    python tools/mask_crop_prof.py [reps]
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from miso_b200 import _lib, mosaic  # noqa: E402
from miso_b200.mosaic import _cstream, _p  # noqa: E402
from tests import cases  # noqa: E402

DEV = "cuda:0"
H = W = 16384
TILE, OVERLAP, DPI, M = 1024, 128, 300, 28
HBM_TBS = 7.7


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main(reps: int = 50) -> None:
    if not torch.cuda.is_available():
        raise SystemExit("mask_crop_prof: needs a CUDA device")
    rng = np.random.default_rng(0)
    grid = mosaic.tile_grid(H, W, TILE, OVERLAP)
    rows = len(grid) * DPI
    local = np.concatenate([cases.stress_rois(rng, DPI, (TILE, TILE), side=(16.0, 160.0)) for _ in grid])
    origin = np.repeat(np.array([[x, y, x, y] for y, x in grid], np.float32), DPI, axis=0)
    gathered = torch.zeros((rows, 6), dtype=torch.float32)
    gathered[:, :4] = torch.from_numpy(local + origin)
    gathered[:, 4], gathered[:, 5] = 1.0, 1.0
    gathered = gathered.to(DEV)
    state = torch.ones((rows,), dtype=torch.int32, device=DEV)
    frames = torch.tensor([[x, y, TILE, TILE] for y, x in grid], dtype=torch.int32, device=DEV)
    probs = torch.rand((rows, M, M), generator=torch.Generator().manual_seed(1)).to(DEV)
    boxes = torch.from_numpy(local).to(DEV)
    band = torch.zeros((H, W, 3), dtype=torch.uint8, device=DEV)

    crops = mosaic.MosaicCrops(rows, (H, W), 3, 0.5, 4 << 30, DEV)
    crops.bind_band(band, 0)
    crops.bind_masks(probs, boxes, frames, DPI, 0.5)
    crops.launch(gathered, state, 0)
    res = crops.results()
    k, mask_bytes = res["count"], res["bytes"] // 3
    assert k == rows, (k, rows)

    lib, st = crops.lib, _cstream(gathered)

    def launch():
        _lib.check(lib.mb_crop_masks(C.byref(crops.params), _p(probs), _p(boxes), M, 1, _p(frames), DPI, 0.5, _p(crops.rects),
                                     _p(crops.src), _p(crops.offsets), _p(crops.totals), _p(crops.masks),
                                     crops.masks.numel(), st), "mb_crop_masks")
    for _ in range(5):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    assert int(crops.totals[3]) == 0
    nbytes = 4 * M * M * k + 16 * k + mask_bytes
    gbs = nbytes / (ms * 1e-3) / 1e9
    print(f"mb_crop_masks: {k} crops (M = {M}), {ms:.4f} ms per launch over {reps}; bytes {4 * M * M * k / 1e6:.1f} MB probs + "
          f"{16 * k / 1e6:.2f} MB boxes + {mask_bytes / 1e6:.1f} MB masks = {nbytes / 1e6:.1f} MB, {gbs:.0f} GB/s, "
          f"{100 * gbs / (HBM_TBS * 1e3):.1f}% of {HBM_TBS} TB/s HBM; {torch.cuda.get_device_name(0)}, power limit {power_limit()}")


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 50)

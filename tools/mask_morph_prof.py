"""mb_mask_morphology at mosaic size: the morphology records of config 5's seam survivors, timed alone.

Input (seeded): the crops of tools/mask_crop_prof.py — a 16384^2 RGB mosaic cut into 361 tiles of 1024 px (128 px
overlap), 300 detections per tile = 108 300 crops, every row kept, sqrt(area) log-uniform in [16, 160] px, M = 28
probabilities uniform in [0, 1) — over a random band (uniform bytes, not zeros). The plan, the pixel gather and the
masks (mb_crop_masks) run once through MosaicCrops; then mb_mask_morphology alone (workspace clear, band kernel,
record kernel) is timed with CUDA events over `reps` calls after a warm-up. Its working set (~0.6 GB of masks, ~1.7 GB
of crop pixels in a 805 MB band) exceeds the 126 MB L2, so every pass reads from HBM.

Bytes counted (algorithmic): sum(h*w) mask bytes + sum(h*w*3) pixel bytes read, 16*K rects + 4*K src + 8*K offsets
read, 104*K record bytes written. The workspace (128 B per crop slot, cleared and read back) is not counted. The share
is of the 7.7 TB/s data-sheet HBM3e figure of one B200; the card name and power limit are read in the same run.
    python tools/mask_morph_prof.py [reps]
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
from miso_b200.ops import _ptr, _stream  # noqa: E402
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
        raise SystemExit("mask_morph_prof: needs a CUDA device")
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
    band = torch.randint(0, 256, (H, W, 3), dtype=torch.uint8, device=DEV, generator=torch.Generator(DEV).manual_seed(2))

    crops = mosaic.MosaicCrops(rows, (H, W), 3, 0.5, 4 << 30, DEV)
    crops.bind_band(band, 0)
    crops.bind_masks(probs, boxes, frames, DPI, 0.5, morphology=True)
    crops.launch(gathered, state, 0)
    res = crops.results()
    k, mask_bytes = res["count"], res["bytes"] // 3
    assert k == rows, (k, rows)
    area = res["morphology"][:, 0].clone()
    lit = float(area.sum()) / mask_bytes

    lib, st = crops.lib, _stream(gathered)

    def launch():
        _lib.check(lib.mb_mask_morphology(C.byref(crops.params), _ptr(crops.masks), _ptr(crops.rects), _ptr(crops.src),
                                          _ptr(crops.offsets), _ptr(crops.totals), _ptr(crops.morph_ws), crops.morph_ws.numel(),
                                          _ptr(crops.morphology), st), "mb_mask_morphology")
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
    assert torch.equal(crops.morphology[:k, 0], area)
    meta = (16 + 4 + 8) * k
    nbytes = mask_bytes + 3 * mask_bytes + meta + 104 * k
    gbs = nbytes / (ms * 1e-3) / 1e9
    print(f"mb_mask_morphology: {k} crops ({100 * lit:.1f}% of mask pixels set), {ms:.4f} ms per call over {reps}; bytes "
          f"{mask_bytes / 1e6:.1f} MB masks + {3 * mask_bytes / 1e6:.1f} MB pixels + {meta / 1e6:.2f} MB rects/src/offsets + "
          f"{104 * k / 1e6:.2f} MB records = {nbytes / 1e6:.1f} MB, {gbs:.0f} GB/s, {100 * gbs / (HBM_TBS * 1e3):.1f}% of "
          f"{HBM_TBS} TB/s HBM; {torch.cuda.get_device_name(0)}, power limit {power_limit()}")


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 50)

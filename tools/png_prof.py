"""mb_png_encode at mosaic size: PNG files of config 5's 108 300 crops and their masks, timed alone, against PIL.

Input (seeded): the mask_crop_prof.py workload — a 16384^2 RGB mosaic cut into 361 tiles of 1024 px (128 px overlap),
300 detections per tile = 108 300 crops, sqrt(area) log-uniform in [16, 160] px, every row kept — but the band is a
smooth synthetic image (two low-frequency waves, dark discs, Gaussian noise sigma 3), so that blocks take the dynamic
Huffman path rather than runs only. The plan, gather and masks run once through MosaicCrops; then mb_png_encode alone
is timed with CUDA events over `reps` launches after a warm-up, for the RGB crops and for the masks. The working set
(2 GB of crops, as much again of workspace and output) exceeds the 126 MB L2.

Reported: raw (uncompressed crop) bytes per second and compressed / raw; the same for a 16-thread PIL pool
(Image.save, default PNG settings, to memory) on the first `pil_crops` crops of the same set; the card and its power
limit, read in the same run.
    python tools/png_prof.py [reps] [pil_crops]
"""
import io
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from miso_b200 import mosaic  # noqa: E402
from miso_b200.ops import _stream  # noqa: E402
from tests import cases  # noqa: E402

DEV = "cuda:0"
H = W = 16384
TILE, OVERLAP, DPI, M = 1024, 128, 300, 28


def power_limit() -> str:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def smooth_band(seed: int) -> torch.Tensor:
    g = torch.Generator(device=DEV).manual_seed(seed)
    y = torch.arange(H, device=DEV, dtype=torch.float32)[:, None]
    x = torch.arange(W, device=DEV, dtype=torch.float32)[None, :]
    bg = 170 + 35 * torch.sin(x / 700.0) * torch.cos(y / 900.0) + 15 * torch.sin((x + y) / 2300.0)
    img = torch.empty((H, W, 3), device=DEV, dtype=torch.float32)
    for c, f in enumerate((1.0, 0.95, 0.9)):
        img[..., c] = bg * f
    # dark discs on a 96 px lattice, radius 10..40 px
    cy = (y // 96) * 96 + 48
    cx = (x // 96) * 96 + 48
    r = 10 + ((cy * 7 + cx * 13) % 31)
    disc = ((y - cy) ** 2 + (x - cx) ** 2) < r * r
    img[disc] *= 0.35
    img += 3.0 * torch.randn(img.shape, device=DEV, generator=g)
    return img.round_().clamp_(0, 255).to(torch.uint8)


def main(reps: int = 5, pil_crops: int = 4000) -> None:
    if not torch.cuda.is_available():
        raise SystemExit("png_prof: needs a CUDA device")
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
    band = smooth_band(2)

    crops = mosaic.MosaicCrops(rows, (H, W), 3, 0.5, 4 << 30, DEV)
    crops.bind_band(band, 0)
    crops.bind_masks(probs, boxes, frames, DPI, 0.5)
    crops.bind_png()
    crops.launch(gathered, state, 0)
    res = crops.results()
    k, raw = res["count"], res["bytes"]
    assert k == rows, (k, rows)
    st = _stream(gathered)
    print(f"{k} crops, {raw / 1e9:.3f} GB RGB, {raw / 3e9:.3f} GB masks; {torch.cuda.get_device_name(0)}, "
          f"power limit {power_limit()}")

    def timed(buf, packed, nbytes, what):
        crops._encode(buf, packed, st)                       # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            crops._encode(buf, packed, st)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        total = crops.checked_png(buf, what)[0]
        print(f"mb_png_encode {what}: {ms:.3f} ms per launch over {reps}; raw {nbytes / 1e9:.3f} GB -> {total / 1e9:.3f} GB "
              f"(ratio {total / nbytes:.3f}), {nbytes / (ms * 1e-3) / 1e9:.1f} GB/s raw")
        return total

    timed(crops.png, crops.pixels, raw, "RGB crops")
    timed(crops.mask_png, crops.masks, raw // 3, "masks")

    # PIL: a 16-thread pool on the first pil_crops crops, default PNG settings, to memory
    host = crops.to_host(3)[:pil_crops]
    masks = crops.masks_to_host()[:pil_crops]

    def enc(a):
        b = io.BytesIO()
        from PIL import Image
        Image.fromarray(a).save(b, format="PNG")
        return len(b.getvalue())

    for what, arrs in (("RGB crops", [c[3] for c in host]), ("masks", masks)):
        nbytes = sum(a.nbytes for a in arrs)
        with ThreadPoolExecutor(max_workers=16) as pool:
            t0 = time.perf_counter()
            sizes = list(pool.map(enc, arrs))
            dt = time.perf_counter() - t0
        print(f"PIL 16 threads {what}: {len(arrs)} crops, raw {nbytes / 1e6:.1f} MB in {dt:.3f} s = "
              f"{nbytes / dt / 1e6:.1f} MB/s raw, ratio {sum(sizes) / nbytes:.3f}; host CPUs {os.cpu_count()}")


if __name__ == "__main__":
    main(*(int(a) for a in sys.argv[1:3]))

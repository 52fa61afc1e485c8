"""mb_jpeg_encode at mosaic size: JPEG files of config 5's 108 300 crops, timed alone, against PIL.

Input: png_prof.py's seeded workload — a smooth synthetic 16384^2 RGB band (two low-frequency waves, dark discs, Gaussian
noise sigma 3) cut into 361 tiles of 1024 px (128 px overlap), 300 detections per tile = 108 300 crops, sqrt(area)
log-uniform in [16, 160] px, every row kept. The plan and gather run once through MosaicCrops; then mb_jpeg_encode
alone is timed with CUDA events over `reps` launches after a warm-up. The working set (1.69 GB of crops, the workspace
and the files) exceeds the 126 MB L2. The workspace is sized for this content (2 B per crop byte) rather than by
mb_jpeg_workspace_bytes' worst case.

Reported: raw (uncompressed crop) bytes per second and file / raw; the same for a 16-thread PIL pool (Image.save,
default JPEG settings, to memory) on the first `pil_crops` crops, whose files are also checked byte for byte against
the device's; the card and its power limit, read in the same run.
    python tools/jpeg_prof.py [reps] [pil_crops]
"""
import io
import os
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
from tools.png_prof import DEV, DPI, H, OVERLAP, TILE, W, power_limit, smooth_band  # noqa: E402


def main(reps: int = 5, pil_crops: int = 4000) -> None:
    if not torch.cuda.is_available():
        raise SystemExit("jpeg_prof: needs a CUDA device")
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
    band = smooth_band(2)

    crops = mosaic.MosaicCrops(rows, (H, W), 3, 0.5, 4 << 30, DEV)
    crops.bind_band(band, 0)
    crops.launch(gathered, state, 0)
    res = crops.results()
    k, raw = res["count"], res["bytes"]
    assert k == rows, (k, rows)
    crops.jpeg = {"kind": "jpeg", "channels": 3, "capacity": raw,
                  "out": torch.empty((raw,), dtype=torch.uint8, device=DEV),
                  "offsets": torch.zeros((rows + 1,), dtype=torch.int64, device=DEV),
                  "status": torch.zeros((2,), dtype=torch.int64, device=DEV),
                  "ws": torch.empty((2 * raw,), dtype=torch.uint8, device=DEV)}
    st = _stream(gathered)
    print(f"{k} crops, {raw / 1e9:.3f} GB RGB; {torch.cuda.get_device_name(0)}, power limit {power_limit()}")

    buf = crops.jpeg
    crops._encode(buf, crops.pixels, st)                     # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        crops._encode(buf, crops.pixels, st)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    total = crops.checked_png(buf, "JPEG")[0]
    print(f"mb_jpeg_encode RGB crops: {ms:.3f} ms per launch over {reps}; raw {raw / 1e9:.3f} GB -> {total / 1e9:.3f} GB "
          f"(ratio {total / raw:.3f}), {raw / (ms * 1e-3) / 1e9:.1f} GB/s raw")

    host = [c[3] for c in crops.to_host(3)[:pil_crops]]
    files = crops.jpeg_to_host()[:pil_crops]

    def enc(a):
        b = io.BytesIO()
        from PIL import Image
        Image.fromarray(a).save(b, format="JPEG")
        return b.getvalue()

    nbytes = sum(a.nbytes for a in host)
    with ThreadPoolExecutor(max_workers=16) as pool:
        t0 = time.perf_counter()
        ref = list(pool.map(enc, host))
        dt = time.perf_counter() - t0
    same = sum(r == f for r, f in zip(ref, files))
    print(f"PIL 16 threads RGB crops: {len(host)} crops, raw {nbytes / 1e6:.1f} MB in {dt:.3f} s = "
          f"{nbytes / dt / 1e6:.1f} MB/s raw, ratio {sum(map(len, ref)) / nbytes:.3f}; host CPUs {os.cpu_count()}; "
          f"{same} of {len(host)} files byte-identical to the device's")


if __name__ == "__main__":
    main(*(int(a) for a in sys.argv[1:3]))

"""crop_objects (ref:miso/object_detection/crop.py:9-33): same output tree and file names; the
pixel gather for all boxes of an image is one mb_crop_plan + mb_crop_gather on the device, one
device-to-host copy hands over all crops of the image, and the files are encoded and written by a
thread pool (the reference encodes them one by one with skimage.io.imsave)."""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import torch

from miso.object_detection.dataset.project import Project


def _imread(path: str) -> np.ndarray:
    """Pixels as skimage.io.imread returns them (its default plugin reads through PIL): palette images expanded to
    RGB / RGBA, everything else in its stored dtype and channel count."""
    from PIL import Image
    with Image.open(path) as img:
        if img.mode == "P":
            img = img.convert("RGBA" if "transparency" in img.info else "RGB")
        return np.array(img)                       # copy: PIL-backed arrays are read-only


def crop_objects(project: Project, output_dir: str, relative_to=None, mask_dir=None):
    """Crops of every annotation under output_dir/<sub-folders>/<label>/. With mask_dir, each annotation's instance mask
    (`mask`, set by inference with_masks=True) is written as well, as a PNG (mode L, 0 / 255) with the crop's relative
    path and file name under mask_dir — a separate tree, so classifiers trained on the crop folders never see it."""
    from PIL import Image
    from miso_b200 import detection
    os.makedirs(output_dir, exist_ok=True)
    output_path = Path(output_dir)
    pool = ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1))
    pending = []

    def save(arr, target):
        Image.fromarray(arr).save(target)

    for image in project.image_dict.values():
        if len(image.boxes) == 0:
            continue
        im = _imread(image.full_path)
        # The gather moves bytes: any dtype goes through as [H, W, bytes per pixel] and is viewed back afterwards
        # (16-bit TIFFs, float images: skimage.io.imread hands those to the reference's numpy slice unchanged)
        px_shape = im.shape[2:]
        bpp = int(np.prod(px_shape, dtype=np.int64)) * im.dtype.itemsize
        as_bytes = np.ascontiguousarray(im).view(np.uint8).reshape(im.shape[0], im.shape[1], bpp)
        dev = torch.from_numpy(as_bytes).cuda()
        k = len(image.boxes)
        # integer corners exactly as the reference computes them (Annotation.coords_int: Python-float sums, np.round,
        # int) — annotations parsed from XML / CVAT are float64 and x + w can round differently in fp32; integer-valued
        # corners below 2^24 pass through the device's fp32 rounding unchanged, negative ones keep numpy's slice rules
        corners = [box.coords_int for box in image.boxes]
        if any(abs(v) >= (1 << 24) for c in corners for v in c):
            raise ValueError(f"crop_objects: box corner beyond 2^24 in {image.full_path}")
        bounds = torch.tensor(corners, dtype=torch.float32, device="cuda")
        scores = torch.ones((1, k), dtype=torch.float32, device="cuda")
        counts = torch.tensor([k], dtype=torch.int32, device="cuda")
        out = detection.filter_and_crop([dev], bounds[None], scores, counts, 0.5, boxes_are_xywh=False)
        crops = [(n, i, xywh, np.ascontiguousarray(c).reshape(c.shape[0], c.shape[1], bpp).view(im.dtype).reshape(c.shape[:2] + px_shape))
                 for n, i, xywh, c in out.to_host(bpp)]
        path = Path(image.full_path)
        for (_, idx, _xywh, crop), box in zip(crops, image.boxes):
            if relative_to is not None:
                label_path = output_path / path.relative_to(relative_to).parent / box.label
            elif len(project.task_names) > 0:
                label_path = output_path / f"{image.dataset_id} - {project.task_names[image.dataset_id]}" / box.label
            else:
                label_path = output_path / box.label
            label_path.mkdir(parents=True, exist_ok=True)
            s = box.bounds
            filename = f"{path.stem}_{s[0]:.0f}_{s[1]:.0f}_{s[2]:.0f}_{s[3]:.0f}{path.suffix}"
            if crop.size:
                pending.append(pool.submit(save, crop, os.path.join(str(label_path), filename)))
                if mask_dir is not None and getattr(box, "mask", None) is not None:
                    if box.mask.shape != crop.shape[:2]:
                        raise ValueError(f"crop_objects: mask {box.mask.shape} of {filename} differs from its crop "
                                         f"{crop.shape[:2]} (annotation changed after inference?)")
                    mask_path = Path(mask_dir) / label_path.relative_to(output_path)
                    mask_path.mkdir(parents=True, exist_ok=True)
                    pending.append(pool.submit(save, box.mask, str(mask_path / Path(filename).with_suffix(".png"))))
    for f in pending:
        f.result()                      # re-raise encoder / file-system errors
    pool.shutdown()

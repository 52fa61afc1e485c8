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


def crop_objects(project: Project, output_dir: str, relative_to=None, mask_dir=None, morphology_csv=None,
                 png_on_gpu=False, jpeg_on_gpu=False):
    """Crops of every annotation under output_dir/<sub-folders>/<label>/. With mask_dir, each annotation's instance mask
    (`mask`, set by inference with_masks=True) is written as well, as a PNG (mode L, 0 / 255) with the crop's relative
    path and file name under mask_dir — a separate tree, so classifiers trained on the crop folders never see it.
    With morphology_csv, one CSV row per written crop, in the order the crops are written: `crop` (the crop file's path
    relative to output_dir, with /), label, x, y, width, height, then the annotation's `morphology` (set by inference
    with_morphology=True) in MORPHOLOGY_FIELDS order — the fields any row has; a row lacking one leaves it empty.
    Numbers are written with repr, so they read back exactly; values are in pixels.
    png_on_gpu=True encodes the crops of .png sources (any case) that are uint8 with 1..4 channels on the device
    (mb_png_encode, lossless: the same pixels as PIL's files, other bytes); the pool then only writes the files. Other
    sources and the mask files keep PIL.
    jpeg_on_gpu=True encodes the crops of .jpg / .jpeg sources (any case) that are uint8 with 1 or 3 channels on the
    device (mb_jpeg_encode): byte for byte the files PIL writes by default. Other sources (CMYK JPEGs, PNG, TIFF, 16-bit)
    keep their path; the two options are independent."""
    from PIL import Image
    from miso_b200 import detection
    os.makedirs(output_dir, exist_ok=True)
    output_path = Path(output_dir)
    pool = ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1))
    pending = []
    morph_rows = []

    def save(arr, target):
        Image.fromarray(arr).save(target)

    def write(data, target):
        with open(target, "wb") as fh:
            fh.write(data)

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
        path = Path(image.full_path)
        suffix = path.suffix.lower()
        on_gpu = png_on_gpu and suffix == ".png" and im.dtype == np.uint8 and 1 <= bpp <= 4
        jpeg_gpu = jpeg_on_gpu and suffix in (".jpg", ".jpeg") and im.dtype == np.uint8 and bpp in (1, 3)
        out = detection.filter_and_crop([dev], bounds[None], scores, counts, 0.5, boxes_are_xywh=False,
                                        **({"png": True} if on_gpu else {}), **({"jpeg": True} if jpeg_gpu else {}))
        encoded = out.png_to_host() if on_gpu else out.jpeg_to_host() if jpeg_gpu else None
        on_gpu = on_gpu or jpeg_gpu
        crops = [(n, i, xywh, np.ascontiguousarray(c).reshape(c.shape[0], c.shape[1], bpp).view(im.dtype).reshape(c.shape[:2] + px_shape))
                 for n, i, xywh, c in out.to_host(bpp)]
        for j, ((_, idx, _xywh, crop), box) in enumerate(zip(crops, image.boxes)):
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
                target = os.path.join(str(label_path), filename)
                pending.append(pool.submit(write, encoded[j], target) if on_gpu else pool.submit(save, crop, target))
                if mask_dir is not None and getattr(box, "mask", None) is not None:
                    if box.mask.shape != crop.shape[:2]:
                        raise ValueError(f"crop_objects: mask {box.mask.shape} of {filename} differs from its crop "
                                         f"{crop.shape[:2]} (annotation changed after inference?)")
                    mask_path = Path(mask_dir) / label_path.relative_to(output_path)
                    mask_path.mkdir(parents=True, exist_ok=True)
                    pending.append(pool.submit(save, box.mask, str(mask_path / Path(filename).with_suffix(".png"))))
                if morphology_csv is not None:
                    if getattr(box, "morphology", None) is None:
                        raise ValueError(f"crop_objects: {filename} has no morphology (run inference with_morphology=True)")
                    rel = (label_path / filename).relative_to(output_path).as_posix()
                    morph_rows.append((rel, box.label, box.x, box.y, box.width, box.height, box.morphology))
    for f in pending:
        f.result()                      # re-raise encoder / file-system errors
    pool.shutdown()
    if morphology_csv is not None:
        _write_morphology_csv(morphology_csv, morph_rows)


def _write_morphology_csv(path, rows):
    import csv
    from miso_b200.detection import MORPHOLOGY_FIELDS
    fields = [f for f in MORPHOLOGY_FIELDS if any(f in r[-1] for r in rows)]
    Path(path).parent.mkdir(parents=True, exist_ok=True)
    with open(path, "w", newline="") as fh:
        w = csv.writer(fh)
        w.writerow(["crop", "label", "x", "y", "width", "height"] + fields)
        for rel, label, x, y, width, height, m in rows:
            w.writerow([rel, label] + [repr(float(v)) for v in (x, y, width, height)]
                       + [repr(float(m[f])) if f in m else "" for f in fields])

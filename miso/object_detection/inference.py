"""infer / infer_directory (ref:miso/object_detection/inference.py:16-131) on the CUDA hot path.

Same signatures and results as the reference: a Project whose images carry RectangleAnnotation
(x, y, x2-x, y2-y as np.float32, label name model_labels[label-1]) for every detection with
score > threshold. The loaded model is patched with miso_b200.patch.patch_model, so everything
between the CNN heads and the returned boxes runs in libmisob200; the score filter and the
xyxy->xywh arithmetic run in mb_crop_plan on the device (one transfer per batch, not two bool-mask
indexings and two .cpu() calls per image).
"""
from __future__ import annotations

import copy
from pathlib import Path
from typing import List

import numpy as np
import torch

from miso.object_detection.dataset.annotation import RectangleAnnotation
from miso.object_detection.dataset.image import ImageMetadata
from miso.object_detection.dataset.project import Project

IMAGE_SUFFIXES = (".jpg", ".jpeg", ".png", ".bmp", ".tiff", ".tif")


def load_model(model_path: str):
    """torch.load of the whole pickled module (ref:...training.py:136 saves it that way). torch >= 2.6
    needs weights_only=False for that (SURVEY.md Appendix C)."""
    from miso_b200.patch import patch_model
    model = torch.load(model_path, weights_only=False)
    model.cuda()
    model.eval()
    return patch_model(model)


def read_image(path) -> np.ndarray:
    from PIL import Image
    return np.asarray(Image.open(path).convert("RGB"))


def _annotate(model, images_meta: List[ImageMetadata], model_labels, threshold, batch_size, project_out: Project,
              num_workers: int = 4, with_masks: bool = False):
    """One pass over the images: decode (a pool of `num_workers` threads reads and decodes the next batches while the
    GPU works — the reference uses a DataLoader with 4 workers, ref:miso/object_detection/inference.py:102-109),
    patched model, score filter + bounds on the device, annotations. with_masks (Mask R-CNN): every annotation also
    gets `mask`, its detection's instance mask over the crop rectangle (np.uint8 [h, w], 0 / 255), cut on the device
    by the same filter_and_crop call."""
    from concurrent.futures import ThreadPoolExecutor
    from miso_b200 import detection
    if with_masks and getattr(model.roi_heads, "mask_predictor", None) is None:
        raise ValueError("instance masks need a Mask R-CNN model; this model has no mask head")
    starts = list(range(0, len(images_meta), batch_size))
    with torch.inference_mode(), ThreadPoolExecutor(max_workers=max(1, num_workers)) as pool:
        window = max(2 * batch_size, num_workers)           # images being read / decoded ahead of the GPU
        futures = [pool.submit(read_image, m.full_path) for m in images_meta[:window]]
        for bi, i0 in enumerate(starts):
            arrays = [f.result() for f in futures[i0:i0 + batch_size]]
            for m in images_meta[len(futures):i0 + batch_size + window]:
                futures.append(pool.submit(read_image, m.full_path))
            futures[i0:i0 + batch_size] = [None] * len(arrays)       # release the decoded arrays
            metas = images_meta[i0:i0 + batch_size]
            dev_u8 = [torch.from_numpy(np.ascontiguousarray(a).copy() if not a.flags.writeable else a).cuda() for a in arrays]
            if getattr(model, "_miso_b200_patched", False) and all(a.dim() == 3 and a.shape[2] == 3 for a in dev_u8):
                from miso_b200.patch import forward_uint8
                # ToTensor + model.transform fused into one kernel; Mask R-CNN masks stay 28x28 probabilities (a full-image
                # paste per detection would be thrown away, or cut to the crop rectangles below)
                results = forward_uint8(model, dev_u8, paste_masks=False)
            else:
                if with_masks:
                    raise ValueError("instance masks need a model patched by miso_b200.patch.patch_model and RGB images")
                images_cuda = [a.permute(2, 0, 1).to(torch.float32) / 255 for a in dev_u8]       # ToTensor
                results = model(images_cuda)
            pad = torch.nn.utils.rnn.pad_sequence
            counts_host = [int(r["boxes"].shape[0]) for r in results]
            boxes = pad([r["boxes"] for r in results], batch_first=True)
            scores = pad([r["scores"] for r in results], batch_first=True)
            labels_d = pad([r["labels"] for r in results], batch_first=True)
            cap = int(boxes.shape[1])
            if cap == 0:
                for m in metas:
                    project_out.add_image(m)
                continue
            counts = torch.tensor(counts_host, dtype=torch.int32, device="cuda")
            probs = pad([r["mask_probs"][:, 0] for r in results], batch_first=True) if with_masks else None
            out = detection.filter_and_crop(dev_u8, boxes.contiguous(), scores.contiguous(), counts, threshold, capacity_bytes=0,
                                            mask_probs=probs)
            kept = int(out.totals[0])
            masks = out.masks_to_host() if with_masks else [None] * kept
            xywh = out.xywh[:kept].cpu().numpy()
            src = out.src[:kept].cpu().numpy()
            labels = labels_d.cpu().numpy()
            for j in range(kept):
                k, d = int(src[j]) // cap, int(src[j]) % cap
                x, y, w, h = xywh[j]
                metas[k].boxes.append(RectangleAnnotation(x, y, w, h, model_labels[int(labels[k, d]) - 1], mask=masks[j]))
            for m in metas:
                project_out.add_image(m)
    return project_out


def infer(project: Project, model_path: str, model_labels: List[str] = None, threshold: float = 0.5, batch_size=2,
          nv: bool = False, with_masks: bool = False):
    if nv:
        model_labels = [label + "_NV" for label in model_labels]
    for label in model_labels:
        project.add_label(None, label, None)
    model = load_model(model_path)
    project = copy.deepcopy(project)
    project.remove_labelled_images()
    out = Project()
    for label in model_labels:
        out.add_label(None, label, None)
    return _annotate(model, list(project.image_dict.values()), model_labels, threshold, batch_size, out, with_masks=with_masks)


def infer_directory(input_dir: str, model_path: str, model_labels: List[str] = None, threshold: float = 0.5, batch_size=2,
                    with_masks: bool = False):
    p = Path(input_dir)
    if not p.exists():
        raise ValueError(f"Directory does not exist: {input_dir}")
    filepaths = [q for q in sorted(p.rglob("*.*")) if q.suffix.lower() in IMAGE_SUFFIXES]
    metas = [ImageMetadata(fp, "/", 0, i) for i, fp in enumerate(filepaths)]
    model = load_model(model_path)
    out = Project()
    for label in model_labels:
        out.add_label(None, label, None)
    return _annotate(model, metas, model_labels, threshold, batch_size, out, with_masks=with_masks)

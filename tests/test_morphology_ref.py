"""The CPU oracle of the per-crop morphology record (tests/morphology_ref.py) against an independent skimage-style
restatement (scipy erosion + convolution + bincount for the perimeter, float moments + eigvalsh for the axes), on the
worked examples of the ABI; and crop_objects' morphology CSV."""
import csv
import math

import numpy as np
import pytest
from scipy import ndimage

from tests import morphology_ref as ref

WEIGHTS = np.zeros(50)
WEIGHTS[[5, 7, 15, 17, 25, 27]] = 1
WEIGHTS[[21, 33]] = math.sqrt(2)
WEIGHTS[[13, 23]] = (1 + math.sqrt(2)) / 2


def independent(mask, pixels, x, y):
    """skimage.measure.regionprops' formulas (perimeter, inertia tensor) restated with scipy and floats."""
    m = np.asarray(mask) != 0
    out = np.zeros(13)
    if not m.any():
        return out
    cross = ndimage.generate_binary_structure(2, 1)
    border = (m & ~ndimage.binary_erosion(m, cross, border_value=0)).astype(np.int64)
    conv = ndimage.convolve(border, np.array([[10, 2, 10], [2, 1, 2], [10, 2, 10]]), mode="constant", cval=0)
    perimeter = np.bincount(conv.ravel(), minlength=50) @ WEIGHTS
    rr, cc = np.nonzero(m)
    rr, cc = rr.astype(np.float64), cc.astype(np.float64)
    dr, dc = rr - rr.mean(), cc - cc.mean()
    urr, ucc, urc = (dr * dr).mean(), (dc * dc).mean(), (dr * dc).mean()
    lam = np.linalg.eigvalsh(np.array([[ucc, -urc], [-urc, urr]]))
    l2, l1 = np.clip(lam, 0, None)
    px = np.asarray(pixels)
    px = px[..., None] if px.ndim == 2 else px
    out[:9] = [m.sum(), perimeter, x + cc.mean(), y + rr.mean(), 4 * np.sqrt(l1), 4 * np.sqrt(l2), np.nan,
               0.0 if l1 == 0 else np.sqrt(1 - l2 / l1), np.sqrt(4 * m.sum() / np.pi)]
    for k in range(min(px.shape[2], 4)):
        out[9 + k] = px[..., k][m].mean()
    return out


def shapes():
    rng = np.random.default_rng(0)
    sq = np.zeros((12, 14), np.uint8); sq[2:9, 3:10] = 255
    ring = np.zeros((20, 20), np.uint8); ring[3:17, 3:17] = 255; ring[7:13, 7:13] = 0
    diag = np.eye(15, dtype=np.uint8) * 255
    anti = diag[:, ::-1].copy()
    checker = ((np.add.outer(np.arange(9), np.arange(11)) % 2) * 255).astype(np.uint8)
    two = np.zeros((16, 30), np.uint8); two[2:7, 2:9] = 255; two[9:15, 18:28] = 255
    edge = np.zeros((10, 13), np.uint8); edge[0:6, 0:13] = 255; edge[4:10, 9:13] = 255
    disc = (np.add.outer((np.arange(41) - 20.3) ** 2, (np.arange(37) - 17.8) ** 2 / 0.3) < 300).astype(np.uint8) * 255
    blob = (rng.uniform(size=(33, 47)) < 0.6).astype(np.uint8) * 255
    return {"square": sq, "ring": ring, "diagonal": diag, "anti_diagonal": anti, "checkerboard": checker,
            "two_components": two, "touching_the_edge": edge, "ellipse": disc, "random": blob,
            "empty": np.zeros((7, 9), np.uint8), "empty_0x5": np.zeros((0, 5), np.uint8),
            "bar_1x9": np.full((1, 9), 255, np.uint8), "bar_9x1": np.full((9, 1), 255, np.uint8),
            "pixel": np.full((1, 1), 255, np.uint8), "full": np.full((6, 8), 7, np.uint8)}


@pytest.mark.parametrize("name", sorted(shapes()))
def test_oracle_agrees_with_an_independent_restatement(name):
    mask = shapes()[name]
    rng = np.random.default_rng(1)
    pixels = rng.integers(0, 256, mask.shape + (3,), dtype=np.uint8)
    got = ref.record(mask, pixels, 17, 5)
    want = independent(mask, pixels, 17, 5)
    keep = [k for k in range(13) if k != 6]
    np.testing.assert_allclose(got[keep], want[keep], rtol=1e-9, atol=1e-9)


def test_worked_examples():
    px = np.zeros((40, 40, 1), np.uint8)
    for n in (1, 2, 3, 8, 31):
        sq = np.full((n, n), 255, np.uint8)
        r = ref.record(sq, px[:n, :n], 0, 0)
        assert r[0] == n * n and r[1] == 4 * (n - 1)
    pixel = ref.record(np.full((1, 1), 1, np.uint8), px[:1, :1], 3, 4)
    assert pixel[1] == 0 and pixel[6] == math.pi / 4 and (pixel[2], pixel[3]) == (3.0, 4.0)
    bar = ref.record(np.full((1, 9), 255, np.uint8), px[:1, :9], 0, 0)
    assert bar[6] == math.pi / 2 and bar[4] == 4 * math.sqrt(20 / 3) and bar[5] == 0 and bar[7] == 1
    assert ref.record(np.full((9, 1), 255, np.uint8), px[:9, :1], 0, 0)[6] == 0.0
    diag = np.eye(15, dtype=np.uint8)
    assert ref.record(diag, px[:15, :15], 0, 0)[6] == -math.pi / 4
    assert ref.record(diag[:, ::-1], px[:15, :15], 0, 0)[6] == math.pi / 4
    assert not ref.record(np.zeros((5, 5), np.uint8), px[:5, :5], 2, 2).any()


def test_means_cover_the_image_channels_only():
    rng = np.random.default_rng(2)
    m = (rng.uniform(size=(10, 12)) < 0.5).astype(np.uint8)
    for ch in (1, 2, 3, 4):
        px = rng.integers(0, 256, (10, 12, ch), dtype=np.uint8)
        r = ref.record(m, px, 0, 0)
        assert np.array_equal(r[9:9 + ch], [px[..., k][m != 0].astype(np.int64).sum() / int(m.sum()) for k in range(ch)])
        assert not r[9 + ch:].any()


def crop_project(tmp_path, with_morphology=True):
    from PIL import Image
    from miso.object_detection.dataset.annotation import RectangleAnnotation
    from miso.object_detection.dataset.image import ImageMetadata
    from miso.object_detection.dataset.project import Project
    idir = tmp_path / "in" / "sub"
    idir.mkdir(parents=True)
    rng = np.random.default_rng(3)
    project = Project()
    morph = {}
    for i, name in enumerate(("a.png", "b.png")):
        Image.fromarray(rng.integers(0, 256, (40, 50, 3), dtype=np.uint8)).save(idir / name)
        meta = ImageMetadata(idir / name, "/", 0, i)
        for k, (x, y, w, h, label) in enumerate([(3.25, 4.5, 10.0, 7.0, "Coccolith"), (20.0, 2.0, 5.5, 9.0, "Coccosphere"),
                                                 (45.0, 30.0, 0.2, 0.2, "Coccolith")]):       # the last one is empty
            m = {f: float(rng.normal()) / 3.0 for f in ref_fields()[:12]} if with_morphology else None
            box = RectangleAnnotation(np.float32(x + i), np.float32(y), np.float32(w), np.float32(h), label, morphology=m)
            meta.boxes.append(box)
            morph[(name, k)] = (box, m)
        project.add_image(meta)
    return project, morph


def ref_fields():
    from miso_b200.detection import MORPHOLOGY_FIELDS
    return MORPHOLOGY_FIELDS


def test_crop_objects_morphology_csv(tmp_path, monkeypatch):
    """The CSV writer on a hand-built Project: header, one row per written crop in write order, relative paths, exact
    round trip of every number. Crops are cut by the host slice here (the pixel gather itself is tested on the GPU)."""
    from miso.object_detection import crop as crop_mod
    project, morph = crop_project(tmp_path)
    on_host(monkeypatch, crop_mod)
    out, csv_path = tmp_path / "out", tmp_path / "report" / "morph.csv"
    crop_mod.crop_objects(project, str(out), relative_to=str(tmp_path / "in"), morphology_csv=str(csv_path))
    with open(csv_path, newline="") as fh:
        rows = list(csv.reader(fh))
    assert rows[0] == ["crop", "label", "x", "y", "width", "height"] + list(ref_fields()[:12])
    written = sorted(p.relative_to(out).as_posix() for p in out.rglob("*.png"))
    assert sorted(r[0] for r in rows[1:]) == written and len(rows) == 1 + 4        # the two empty crops have no file
    order = [(name, k) for name in ("a.png", "b.png") for k in range(2)]
    for r, key in zip(rows[1:], order):
        box, m = morph[key]
        s = box.bounds
        assert r[0] == f"sub/{box.label}/{key[0][:-4]}_{s[0]:.0f}_{s[1]:.0f}_{s[2]:.0f}_{s[3]:.0f}.png"
        assert r[1] == box.label
        assert [float(v) for v in r[2:6]] == [float(box.x), float(box.y), float(box.width), float(box.height)]
        assert [float(v) for v in r[6:]] == [m[f] for f in ref_fields()[:12]]


def test_crop_objects_morphology_csv_needs_morphology(tmp_path, monkeypatch):
    from miso.object_detection import crop as crop_mod
    project, _ = crop_project(tmp_path, with_morphology=False)
    on_host(monkeypatch, crop_mod)
    with pytest.raises(ValueError, match="no morphology"):
        crop_mod.crop_objects(project, str(tmp_path / "out"), relative_to=str(tmp_path / "in"),
                              morphology_csv=str(tmp_path / "m.csv"))
    assert not (tmp_path / "m.csv").exists()


def on_host(monkeypatch, crop_mod):
    """crop_objects without a GPU: tensors stay on the host and the device crop is replaced by the numpy slice."""
    import torch
    from miso_b200 import detection

    class HostTorch:
        float32, int32 = torch.float32, torch.int32
        from_numpy = staticmethod(torch.from_numpy)
        tensor = staticmethod(lambda *a, device=None, **k: torch.tensor(*a, **k))
        ones = staticmethod(lambda *a, device=None, **k: torch.ones(*a, **k))

    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)
    monkeypatch.setattr(crop_mod, "torch", HostTorch)
    monkeypatch.setattr(detection, "filter_and_crop", host_filter_and_crop)


class _HostCrops:
    def __init__(self, crops):
        self.crops = crops

    def to_host(self, bpp):
        return self.crops


def host_filter_and_crop(images, bounds, scores, counts, threshold, boxes_are_xywh=False):
    """numpy slice of the corners crop_objects hands over (the reference's crop, ref:miso/object_detection/crop.py:28-30)."""
    im = images[0].cpu().numpy()
    out = []
    for i, (x0, y0, x1, y1) in enumerate(bounds[0].cpu().numpy().astype(np.int64)):
        out.append((0, i, None, im[y0:y1, x0:x1]))
    return _HostCrops(out)

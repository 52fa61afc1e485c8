"""Per-crop morphology records (mb_mask_morphology) against the CPU oracle of tests/morphology_ref.py: hand-made masks
through the C ABI (including a 1-pixel-wide crop and one 4096x3072 crop that is split into many row bands), then every
layer: filter_and_crop(morphology=True), MosaicCrops / infer_mosaic(morphology=True) and emulated ranks,
infer_directory(with_morphology=True) and the CLI's --morphology-csv. area, perimeter, centroids, equivalent diameter
and the channel means are bit-exact; axes, orientation and eccentricity agree within 1e-12."""
import csv
import ctypes as C

import numpy as np
import pytest
import torch

from tests import cases, morphology_ref as ref
from tests.test_gpu_crop_masks import per_image_case, save_model, write_images
from tests.test_gpu_model import make_model
from tests.test_morphology_ref import shapes

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def vp(t):
    return C.c_void_p(t.data_ptr())


def run_abi(images, crops, channels, cap=None, mask_overflow=0):
    """crops: (image index, x, y, mask [h, w]) -> mb_mask_morphology's records [K, 13] (numpy)."""
    from miso_b200 import _lib
    lib = _lib.load()
    k = len(crops)
    cap = cap or k
    p = _lib.CropParams()
    p.num_images, p.capacity, p.channels = len(images), cap, channels
    dimgs = [cu(a) for a in images]
    for i, a in enumerate(dimgs):
        p.image_h[i], p.image_w[i], p.images[i] = a.shape[0], a.shape[1], a.data_ptr()
    rects = np.array([[x, y, m.shape[1], m.shape[0]] for _, x, y, m in crops], np.int32).reshape(-1, 4)
    src = np.array([n * cap + j for j, (n, *_rest) in enumerate(crops)], np.int32)
    sizes = np.array([m.size for *_rest, m in crops], np.int64)
    offsets = np.concatenate([[0], np.cumsum(sizes * channels)]).astype(np.int64)
    masks = np.concatenate([m.ravel() for *_rest, m in crops] + [np.zeros(1, np.uint8)])
    totals = np.array([k, offsets[-1], 0, int(mask_overflow)], np.int64)
    out = torch.full((len(images) * cap, ref.FIELDS), -7.0, dtype=torch.float64, device=DEV)
    ws = torch.empty((lib.mb_mask_morphology_workspace_bytes(C.byref(p)),), dtype=torch.uint8, device=DEV)
    dm, dr, ds, do, dt = cu(masks), cu(rects), cu(src), cu(offsets), cu(totals)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.mb_mask_morphology(C.byref(p), vp(dm), vp(dr), vp(ds), vp(do), vp(dt), vp(ws), ws.numel(), vp(out), st)
    torch.cuda.synchronize()
    return rc, out.cpu().numpy()


def hand_made_crops(rng, big):
    crops = []
    x = 5
    for name, m in sorted(shapes().items()):
        crops.append((1, x % 150, 7 + x % 90, (m != 0).astype(np.uint8) * 255))
        x += 23
    crops.append((1, 259, 3, (rng.uniform(size=(57, 1)) < 0.7).astype(np.uint8) * 255))     # 1 pixel wide, last column
    crops.append((1, 40, 0, (rng.uniform(size=(1, 160)) < 0.7).astype(np.uint8) * 255))     # 1 pixel high, first row
    if big:
        yy, xx = np.mgrid[0:3072, 0:4096]
        blob = ((xx - 2100.5) ** 2 / 1900.0 ** 2 + (yy - 1400.25) ** 2 / 1300.0 ** 2 + 0.3 * (xx - 2000) * (yy - 1500) / 4e6) < 1
        blob &= rng.uniform(size=blob.shape) < 0.97                                          # holes
        crops.append((0, 3, 2, blob.astype(np.uint8) * 255))
    return crops


@pytest.mark.parametrize("ch", [1, 3, 4])
def test_hand_made_masks_through_the_abi(ch):
    rng = np.random.default_rng(ch)
    images = [rng.integers(0, 256, (3080, 4104, ch), dtype=np.uint8), rng.integers(0, 256, (200, 260, ch), dtype=np.uint8)]
    crops = hand_made_crops(rng, big=ch == 3)
    rc, got = run_abi(images, crops, ch, cap=len(crops) + 3)
    assert rc == 0
    want = np.stack([ref.record(m, images[n][y:y + m.shape[0], x:x + m.shape[1]], x, y) for n, x, y, m in crops])
    ref.assert_records_match(got[:len(crops)], want, "abi")
    assert (got[len(crops):] == -7.0).all()                     # rows past the count are not written
    areas = {name: got[i, 0] for i, name in enumerate(sorted(shapes()))}
    assert areas["empty"] == 0 and not got[sorted(shapes()).index("empty")].any()
    if ch == 3:
        assert got[len(crops) - 1, 0] > 5e6                      # the image-sized crop


def test_unsupported_channels_side_and_mask_overflow():
    from miso_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (64, 64, 5), dtype=np.uint8)
    crops = [(0, 2, 3, np.full((5, 6), 255, np.uint8))]
    rc, _ = run_abi([img], crops, 5)
    assert rc == -3
    img3 = np.ascontiguousarray(img[..., :3])
    rc, got = run_abi([img3], crops, 3, mask_overflow=1)            # totals[3] set: nothing written
    assert rc == 0 and (got == -7.0).all()
    p = _lib.CropParams()
    p.num_images, p.capacity, p.channels = 1, 1, 3
    p.image_h[0], p.image_w[0], p.images[0] = 40000, 16, 1
    assert lib.mb_mask_morphology(C.byref(p), C.c_void_p(1), C.c_void_p(1), C.c_void_p(1), C.c_void_p(1), C.c_void_p(1),
                                  C.c_void_p(1), 1 << 20, C.c_void_p(1), None) == -3
    p.image_h[0] = 32768
    assert lib.mb_mask_morphology(C.byref(p), C.c_void_p(1), C.c_void_p(1), C.c_void_p(1), C.c_void_p(1), C.c_void_p(1),
                                  C.c_void_p(1), 0, C.c_void_p(1), None) == -2          # workspace too small


def oracle_of(out, images):
    """The oracle applied to filter_and_crop's own masks and the image pixels of each crop."""
    k = int(out.totals[0])
    rects, src = out.rects[:k].cpu().numpy(), out.src[:k].cpu().numpy()
    cap = out.rects.shape[0] // len(images)
    masks = out.masks_to_host()
    return np.stack([ref.record(m, images[int(s) // cap][y:y + h, x:x + w], x, y)
                     for m, s, (x, y, w, h) in zip(masks, src, rects)]) if k else np.zeros((0, ref.FIELDS))


@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("gather", [True, False])
def test_filter_and_crop_morphology(ch, gather):
    from miso_b200 import detection
    rng = np.random.default_rng(3 + ch)
    imgs, boxes, scores, counts, probs = per_image_case(rng, ch)
    out = detection.filter_and_crop([cu(a) for a in imgs], cu(boxes), cu(scores), cu(counts), 0.3,
                                    capacity_bytes=None if gather else 0, mask_probs=cu(probs), morphology=True)
    got = out.morphology_to_host()
    assert got.shape == (int(out.totals[0]), len(detection.MORPHOLOGY_FIELDS)) and len(got) > 40
    ref.assert_records_match(got, oracle_of(out, imgs), "filter_and_crop")
    assert (got[:, 0] > 0).sum() > 20 and not got[:, 9 + ch:].any()


def test_chunked_plan_morphology():
    from miso_b200 import detection
    rng = np.random.default_rng(17)
    n, cap, hw = 60, 520, (96, 128)
    imgs = [rng.integers(0, 256, (hw[0], hw[1], 3), dtype=np.uint8) for _ in range(n)]
    boxes = np.stack([cases.stress_rois(rng, cap, hw, side=(2.0, 90.0)) for _ in range(n)])
    scores = rng.uniform(0.0, 1.0, (n, cap)).astype(np.float32)
    counts = rng.integers(0, cap + 1, n).astype(np.int32)
    probs = cu(rng.uniform(0.0, 1.0, (n * cap, 1, 28, 28)).astype(np.float32))
    out = detection.filter_and_crop([cu(a) for a in imgs], cu(boxes), cu(scores), cu(counts), 0.5, capacity_bytes=0,
                                    mask_probs=probs, morphology=True)
    got = out.morphology_to_host()
    assert len(got) > 1000
    ref.assert_records_match(got, oracle_of(out, imgs), "chunked")


def test_filter_and_crop_errors():
    from miso_b200 import detection
    from miso_b200._lib import MisoB200Error
    rng = np.random.default_rng(2)
    imgs, boxes, scores, counts, probs = per_image_case(rng, 3)
    dimgs = [cu(a) for a in imgs]
    with pytest.raises(MisoB200Error, match="mask_probs"):
        detection.filter_and_crop(dimgs, cu(boxes), cu(scores), cu(counts), 0.3, morphology=True)
    five = [cu(rng.integers(0, 256, a.shape[:2] + (5,), dtype=np.uint8)) for a in imgs]
    with pytest.raises(MisoB200Error, match="unsupported"):
        detection.filter_and_crop(five, cu(boxes), cu(scores), cu(counts), 0.3, mask_probs=cu(probs), morphology=True)
    out = detection.filter_and_crop(dimgs, cu(boxes), cu(scores), cu(counts), 0.3, mask_probs=cu(probs), morphology=True,
                                    mask_capacity_bytes=10)
    with pytest.raises(MisoB200Error, match="bytes needed"):
        out.morphology_to_host()


@pytest.fixture(scope="module")
def morph_mosaic():
    from miso_b200 import mosaic
    from miso_b200.patch import forward_uint8, patch_model
    model = patch_model(make_model("mask").to(DEV))
    g = torch.Generator().manual_seed(5)
    mos = torch.randint(0, 256, (1536, 1536, 3), dtype=torch.uint8, generator=g).to(DEV)
    kw = dict(tile=1024, overlap=128, threshold=0.1, batch_size=2, mask_threshold=0.5)
    both = mosaic.infer_mosaic(model, mos, (1536, 1536), masks=True, morphology=True, **kw)
    only = mosaic.infer_mosaic(model, mos, (1536, 1536), morphology=True, **kw)
    grid = mosaic.tile_grid(1536, 1536, 1024, 128)
    per_tile = []
    with torch.inference_mode():
        for i0 in range(0, 4, 2):
            per_tile += forward_uint8(model, [mos[y:y + 1024, x:x + 1024] for y, x in grid[i0:i0 + 2]], paste_masks=False)
    return dict(model=model, mos=mos, both=both, only=only, grid=grid, per_tile=per_tile,
                dpi=int(model.roi_heads.detections_per_img))


def test_infer_mosaic_morphology_equals_the_oracle(morph_mosaic):
    mm = morph_mosaic
    c, o = mm["both"]["crops"], mm["only"]["crops"]
    assert "masks" not in o and torch.equal(c["morphology"], o["morphology"])
    k = c["count"]
    assert k > 0 and c["morphology"].shape == (k, ref.FIELDS) and c["morphology"].is_cuda
    rects, offs, buf = c["rects"].cpu().numpy(), c["offsets"].cpu().numpy() // 3, c["masks"].cpu().numpy()
    mos = mm["mos"].cpu().numpy()
    want = np.stack([ref.record(buf[offs[j]:offs[j + 1]].reshape(h, w), mos[y:y + h, x:x + w], x, y)
                     for j, (x, y, w, h) in enumerate(rects)])
    got = c["morphology"].cpu().numpy()
    ref.assert_records_match(got, want, "mosaic")
    assert (got[:, 0] > 0).sum() > 0 and (got[:, 2] > 1024).any()          # centroids in mosaic coordinates


def test_infer_mosaic_morphology_of_two_emulated_ranks_equals_world1(morph_mosaic):
    from miso_b200 import mosaic
    mm = morph_mosaic
    dpi, grid, mos = mm["dpi"], mm["grid"], mm["mos"]
    gathered, state = mm["both"]["gathered"], mm["both"]["state"]
    outs = []
    for rank in range(2):
        mine = list(mosaic.rank_tiles(4, 2, rank))
        y0, y1 = mosaic.rank_band(grid, 1024, 1536, 2, rank)
        probs = torch.zeros((2 * dpi, 28, 28), dtype=torch.float32, device=DEV)
        boxes = torch.zeros((2 * dpi, 4), dtype=torch.float32, device=DEV)
        for i, t in enumerate(mine):
            r = mm["per_tile"][t]
            k = r["boxes"].shape[0]
            probs[i * dpi:i * dpi + k], boxes[i * dpi:i * dpi + k] = r["mask_probs"][:, 0], r["boxes"]
        frames = torch.tensor([[grid[t][1], grid[t][0], 1024, 1024] for t in mine], dtype=torch.int32, device=DEV)
        crops = mosaic.MosaicCrops(2 * dpi, (1536, 1536), 3, 0.1, 256 << 20, DEV)
        crops.bind_band(mos[y0:y1].contiguous(), y0)
        crops.bind_masks(probs, boxes, frames, dpi, 0.5, morphology=True)
        crops.launch(gathered, state, rank * 2 * dpi)
        outs.append(crops.results())
    assert all(o["count"] > 0 for o in outs)
    assert torch.equal(torch.cat([o["morphology"] for o in outs]), mm["both"]["crops"]["morphology"])


def test_infer_mosaic_rank_without_tiles_and_faster_rcnn(monkeypatch):
    from miso_b200 import mosaic
    from miso_b200._lib import MisoB200Error
    from miso_b200.patch import patch_model
    model = patch_model(make_model("mask").to(DEV))
    mos = torch.zeros((1024, 1024, 3), dtype=torch.uint8, device=DEV)
    # world 2 emulated in one process: one tile, owned by rank 0; rank 1's block (all rows dead) stands for both
    monkeypatch.setattr(mosaic, "exchange", lambda block, world, group=None, out=None: torch.cat([block] * world))
    res = mosaic.infer_mosaic(model, mos, (1024, 1024), rank=1, world=2, morphology=True)
    assert res["crops"]["morphology"].shape == (0, ref.FIELDS) and "masks" not in res["crops"]
    faster = patch_model(make_model("faster").to(DEV))
    with pytest.raises(MisoB200Error, match="mask head"):
        mosaic.infer_mosaic(faster, mos, (1024, 1024), morphology=True)


def test_infer_directory_with_morphology(tmp_path):
    from miso.object_detection.inference import infer_directory, read_image
    from miso_b200.detection import MORPHOLOGY_FIELDS
    mdir = save_model(tmp_path, "mask")
    idir = write_images(tmp_path)
    project = infer_directory(str(idir), str(mdir / "model.pt"), ["Coccolith", "Coccosphere"], 0.1, 2, with_masks=True,
                              with_morphology=True)
    seen = 0
    for m in project.image_dict.values():
        im = np.asarray(read_image(m.full_path))
        for box in m.boxes:
            assert tuple(box.morphology) == MORPHOLOGY_FIELDS[:12]
            c = box.coords_int
            want = ref.record(box.mask, im[c[1]:c[3], c[0]:c[2]], c[0], c[1])
            ref.assert_records_match(np.array([box.morphology[f] for f in MORPHOLOGY_FIELDS[:12]] + [0.0]), want, "infer")
            seen += 1
    assert seen > 0
    faster = save_model(tmp_path / "f", "faster")
    with pytest.raises(ValueError, match="mask head"):
        infer_directory(str(idir), str(faster / "model.pt"), ["Coccolith", "Coccosphere"], 0.1, 2, with_morphology=True)


def test_cli_morphology_csv(tmp_path):
    from click.testing import CliRunner
    from PIL import Image
    import miso.cli as cli
    from miso_b200.detection import MORPHOLOGY_FIELDS
    idir = write_images(tmp_path)
    save_model(tmp_path, "mask")
    save_model(tmp_path, "faster")
    base = ["infer-object-detector-directory", "-i", str(idir), "--model-dir", str(tmp_path / "models"), "--threshold", "0.1",
            "--batch-size", "2"]
    odir, kdir, csv1 = tmp_path / "out", tmp_path / "masks", tmp_path / "m1.csv"
    res = CliRunner().invoke(cli.cli, base + ["-o", str(odir), "--model", "mask", "--mask-dir", str(kdir),
                                              "--morphology-csv", str(csv1)], catch_exceptions=False)
    assert res.exit_code == 0, res.output
    with open(csv1, newline="") as fh:
        rows = list(csv.reader(fh))
    assert rows[0] == ["crop", "label", "x", "y", "width", "height"] + list(MORPHOLOGY_FIELDS[:12])
    assert sorted(r[0] for r in rows[1:]) == sorted(p.relative_to(odir).as_posix() for p in odir.rglob("*.png"))
    for r in rows[1:]:
        crop = np.asarray(Image.open(odir / r[0]))
        mask = np.asarray(Image.open(kdir / r[0]))
        x0, y0 = (max(int(np.round(np.float32(float(v)))), 0) for v in r[2:4])
        want = ref.record(mask, crop, x0, y0)
        ref.assert_records_match(np.array([float(v) for v in r[6:]] + [0.0]), want, r[0])
    # without --mask-dir: the same rows, no mask files
    csv2 = tmp_path / "m2.csv"
    res = CliRunner().invoke(cli.cli, base + ["-o", str(tmp_path / "out2"), "--model", "mask", "--morphology-csv", str(csv2)],
                             catch_exceptions=False)
    assert res.exit_code == 0, res.output
    assert csv2.read_text() == csv1.read_text()
    # a Faster R-CNN model has no masks to measure
    res = CliRunner().invoke(cli.cli, base + ["-o", str(tmp_path / "out3"), "--model", "faster", "--morphology-csv",
                                              str(tmp_path / "m3.csv")])
    assert res.exit_code != 0 and "Mask R-CNN" in res.output and not (tmp_path / "m3.csv").exists()

"""PNG files encoded on the device (mb_png_encode through CropStage.bind_png / filter_and_crop(png=True)): every stream
equals tests/png_ref.py byte for byte and decodes with PIL to exactly the crop the gather cut."""
import io

import numpy as np
import pytest
import torch
from PIL import Image

from tests import png_ref
from tests.test_png_ref import hand_cases, particle_crop

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def crop_all(images, rects_per_image, **kw):
    """filter_and_crop of the given integer (x, y, w, h) boxes (annotation bounds) on the device."""
    from miso_b200 import detection
    n = len(images)
    cap = max(1, max(len(r) for r in rects_per_image))
    boxes = np.zeros((n, cap, 4), np.float32)
    scores = np.zeros((n, cap), np.float32)
    counts = np.zeros((n,), np.int32)
    for i, rs in enumerate(rects_per_image):
        if rs:
            boxes[i, :len(rs)] = rs
            scores[i, :len(rs)] = 1.0
        counts[i] = len(rs)
    return detection.filter_and_crop([cu(im) for im in images], cu(boxes), cu(scores), cu(counts), 0.5,
                                     boxes_are_xywh=True, **kw)


def check_stage(stage, channels):
    crops = stage.to_host(channels)
    pngs = stage.png_to_host()
    assert len(pngs) == len(crops)
    for (_, _, _, a), s in zip(crops, pngs):
        assert s == png_ref.encode(a)
        if a.size:
            assert np.array_equal(np.array(Image.open(io.BytesIO(s))), a)
    return crops, pngs


def test_hand_made_cases():
    for name, a in hand_cases():
        st = crop_all([a], [[(0, 0, a.shape[1], a.shape[0])]], png=True)
        crops, pngs = check_stage(st, 1 if a.ndim == 2 else a.shape[2])
        assert len(pngs) == 1, name


@pytest.mark.parametrize("channels", [1, 3])
def test_random_rect_crops(channels):
    rng = np.random.default_rng(channels)
    images, rects = [], []
    for i in range(3):
        h, w = int(rng.integers(200, 400)), int(rng.integers(200, 400))
        base = particle_crop(rng, h, w, 3)
        images.append(base[..., 0].copy() if channels == 1 else base)
        rs = []
        for _ in range(100):
            x, y = int(rng.integers(-20, w)), int(rng.integers(-20, h))
            rs.append((x, y, int(rng.integers(0, 120)), int(rng.integers(0, 120))))
        rects.append(rs)
    st = crop_all(images, rects, png=True)
    crops, pngs = check_stage(st, channels)
    assert len(crops) == 300
    assert any(len(s) == 0 for s in pngs)          # zero-area crops (slices outside the image) give empty streams


def test_masks_route():
    rng = np.random.default_rng(5)
    im = particle_crop(rng, 300, 300, 3)
    rs = [(int(rng.integers(0, 250)), int(rng.integers(0, 250)), int(rng.integers(1, 60)), int(rng.integers(1, 60)))
          for _ in range(40)]
    probs = torch.rand((1, len(rs), 28, 28), device=DEV)
    boxes = np.array([[x, y, x + w, y + h] for x, y, w, h in rs], np.float32)
    st = crop_all([im], [rs], mask_probs=probs, paste_boxes=cu(boxes[None]), png=True)
    masks = st.masks_to_host()
    mp = st.mask_png_to_host()
    check_stage(st, 3)
    for m, s in zip(masks, mp):
        assert s == png_ref.encode(m)
        assert np.array_equal(np.array(Image.open(io.BytesIO(s))), m)


def test_chunked_plan():
    """More than 8192 slots: the chunked crop plan feeds the encoder the same way."""
    rng = np.random.default_rng(7)
    images = [particle_crop(rng, 128, 128, 3) for _ in range(3)]
    rects = [[(int(rng.integers(0, 120)), int(rng.integers(0, 120)), int(rng.integers(1, 9)), int(rng.integers(1, 9)))
              for _ in range(3000)] for _ in range(3)]
    st = crop_all(images, rects, png=True)
    crops, pngs = check_stage(st, 3)
    assert len(crops) == 9000


def test_large_crop_many_blocks():
    rng = np.random.default_rng(11)
    im = particle_crop(rng, 3072, 4096, 3)
    st = crop_all([im], [[(0, 0, 4096, 3072)]], png=True)
    (_, _, _, a), = st.to_host(3)
    s, = st.png_to_host()
    assert s == png_ref.encode(a)
    assert np.array_equal(np.array(Image.open(io.BytesIO(s))), im)


def test_edges_and_errors():
    from miso_b200 import detection
    from miso_b200._lib import MisoB200Error
    rng = np.random.default_rng(3)
    im = particle_crop(rng, 64, 64, 3)
    st = crop_all([im], [[]], png=True)                          # no crops
    assert st.png_to_host() == []
    st = crop_all([im], [[(70, 70, 5, 5), (0, 0, 0, 3)]], png=True)   # zero-area crops
    assert st.png_to_host() == [b"", b""]
    assert int(st.png["status"][0]) == 0
    # too small a capacity: flag set, nothing written, Python raises
    stage = crop_all([im], [[(0, 0, 32, 32)]])
    stage.bind_png(capacity_bytes=16)
    stage.png["out"].fill_(0xAB)
    stage.cut(torch.cuda.current_stream().cuda_stream)
    st_host = stage.png["status"].tolist()
    assert st_host[1] == 1 and st_host[0] == len(png_ref.encode(im[:32, :32]))
    assert int((stage.png["out"] != 0xAB).sum()) == 0
    with pytest.raises(MisoB200Error):
        stage.png_to_host()
    # channels outside 1..4
    five = cu(rng.integers(0, 256, (16, 16, 5), dtype=np.uint8))
    with pytest.raises(MisoB200Error):
        detection.filter_and_crop([five], cu(np.array([[[0, 0, 8, 8]]], np.float32)), cu(np.ones((1, 1), np.float32)),
                                  cu(np.ones((1,), np.int32)), 0.5, boxes_are_xywh=True, png=True)
    from miso_b200 import _lib
    lib = _lib.load()
    assert lib.mb_png_bound_bytes(100, 1, 5) == -1


def test_sizes_against_pil():
    """Seeded particle-like crops (sides log-uniform 16..160, sigma 3 noise): total <= 1.10 x PIL's default encoder.
    0/255 elliptical masks of these sizes come to about 1.16 x PIL's: the per-row filter heuristic turns mask edges
    into isolated bytes that runs do not cover (PIL's long-distance matches do), and the sync flush and final block
    add 7 bytes per file; the bound below keeps that from growing."""
    rng = np.random.default_rng(2024)
    crops = [particle_crop(rng, int(np.exp(rng.uniform(np.log(16), np.log(160)))),
                           int(np.exp(rng.uniform(np.log(16), np.log(160)))), 3) for _ in range(200)]
    H = max(c.shape[0] for c in crops)
    Wsum = sum(c.shape[1] for c in crops)
    canvas = np.zeros((H, Wsum, 3), np.uint8)
    rects, x = [], 0
    for c in crops:
        canvas[:c.shape[0], x:x + c.shape[1]] = c
        rects.append((x, 0, c.shape[1], c.shape[0]))
        x += c.shape[1]
    ys, xs = np.mgrid[0:H, 0:Wsum]
    probs = torch.zeros((1, len(rects), 28, 28), device=DEV)
    yy, xx = np.mgrid[0:28, 0:28]
    ell = (((yy - 13.5) / 11) ** 2 + ((xx - 13.5) / 8) ** 2 < 1).astype(np.float32)
    probs[:] = cu(ell)
    boxes = np.array([[x, y, x + w, y + h] for x, y, w, h in rects], np.float32)
    st = crop_all([canvas], [rects], mask_probs=probs, paste_boxes=cu(boxes[None]), png=True)
    pngs, mpngs = st.png_to_host(), st.mask_png_to_host()
    masks = st.masks_to_host()

    def pil(a):
        b = io.BytesIO()
        Image.fromarray(a).save(b, format="PNG")
        return len(b.getvalue())

    ours, theirs = sum(len(s) for s in pngs), sum(pil(c) for c in crops)
    mours, mtheirs = sum(len(s) for s in mpngs), sum(pil(m) for m in masks)
    print(f"crops: {ours / theirs:.3f} x PIL, masks: {mours / mtheirs:.3f} x PIL")
    assert ours <= 1.10 * theirs
    assert mours <= 1.20 * mtheirs


def _streams(buf, offsets):
    data, offs = buf.cpu().numpy().tobytes(), offsets.cpu().numpy()
    return [data[offs[j]:offs[j + 1]] for j in range(len(offs) - 1)]


def test_infer_mosaic_png_world1_and_two_ranks():
    """infer_mosaic(png=True): every crop's and mask's stream equals the oracle's, two emulated ranks give world 1's
    streams in rank order, and a crop gives the same bytes through filter_and_crop."""
    from miso_b200 import mosaic
    from miso_b200.patch import forward_uint8, patch_model
    from tests.test_gpu_crop_masks import make_model
    model = patch_model(make_model("mask").to(DEV))
    g = torch.Generator().manual_seed(5)
    mos = torch.randint(0, 256, (1536, 1536, 3), dtype=torch.uint8, generator=g).to(DEV)
    kw = dict(tile=1024, overlap=128, threshold=0.1, batch_size=2)
    res = mosaic.infer_mosaic(model, mos, (1536, 1536), masks=True, png=True, **kw)
    c = res["crops"]
    assert c["count"] > 0
    pngs, mpngs = _streams(c["png"], c["png_offsets"]), _streams(c["mask_png"], c["mask_png_offsets"])
    rects, offs = c["rects"].cpu().numpy(), c["offsets"].cpu().numpy()
    pix, msk = c["pixels"].cpu().numpy(), c["masks"].cpu().numpy()
    for j in range(c["count"]):
        _, _, w, h = rects[j]
        a = pix[offs[j]:offs[j + 1]].reshape(h, w, 3)
        m = msk[offs[j] // 3:offs[j + 1] // 3].reshape(h, w)
        assert pngs[j] == png_ref.encode(a) and mpngs[j] == png_ref.encode(m), j
    # two emulated ranks over the same gathered rows
    grid, dpi = mosaic.tile_grid(1536, 1536, 1024, 128), int(model.roi_heads.detections_per_img)
    per_tile = []
    with torch.inference_mode():
        for i0 in range(0, 4, 2):
            per_tile += forward_uint8(model, [mos[y:y + 1024, x:x + 1024] for y, x in grid[i0:i0 + 2]], paste_masks=False)
    got, got_m = [], []
    for rank in range(2):
        mine = list(mosaic.rank_tiles(4, 2, rank))
        y0, y1 = mosaic.rank_band(grid, 1024, 1536, 2, rank)
        probs = torch.zeros((2 * dpi, 28, 28), dtype=torch.float32, device=DEV)
        boxes = torch.zeros((2 * dpi, 4), dtype=torch.float32, device=DEV)
        for i, t in enumerate(mine):
            r = per_tile[t]
            k = r["boxes"].shape[0]
            probs[i * dpi:i * dpi + k], boxes[i * dpi:i * dpi + k] = r["mask_probs"][:, 0], r["boxes"]
        frames = torch.tensor([[grid[t][1], grid[t][0], 1024, 1024] for t in mine], dtype=torch.int32, device=DEV)
        crops = mosaic.MosaicCrops(2 * dpi, (1536, 1536), 3, 0.1, 256 << 20, DEV)
        crops.bind_band(mos[y0:y1].contiguous(), y0)
        crops.bind_png()
        crops.bind_masks(probs, boxes, frames, dpi, 0.5)          # after bind_png: the mask streams follow
        crops.launch(res["gathered"], res["state"], rank * 2 * dpi)
        o = crops.results()
        got += _streams(o["png"], o["png_offsets"])
        got_m += _streams(o["mask_png"], o["mask_png_offsets"])
    assert got == pngs and got_m == mpngs
    # the same crop through filter_and_crop of the mosaic as one image
    x, y, w, h = (int(v) for v in rects[0])
    st = crop_all([mos.cpu().numpy()], [[(x, y, w, h)]], png=True)
    assert st.png_to_host() == [pngs[0]]


def test_crop_objects_and_cli_png_on_gpu(tmp_path):
    """--png-on-gpu writes the same file tree as the default run, every PNG decoding to the same pixels; a JPEG source in
    the same directory still goes through PIL (byte-identical files)."""
    from click.testing import CliRunner
    import miso.cli as cli
    from tests.test_gpu_crop_masks import save_model, write_images
    idir = write_images(tmp_path)
    rng = np.random.default_rng(1)
    Image.fromarray(particle_crop(rng, 300, 400, 3)).save(idir / "sub" / "c.jpg", quality=95)
    Image.fromarray(particle_crop(rng, 256, 320, 3)[..., 0]).save(idir / "sub" / "d.PNG")
    save_model(tmp_path, "mask")
    base = ["infer-object-detector-directory", "-i", str(idir), "--model-dir", str(tmp_path / "models"), "--threshold",
            "0.1", "--batch-size", "2", "--model", "mask"]
    a, b = tmp_path / "cpu", tmp_path / "gpu"
    for out, extra in ((a, []), (b, ["--png-on-gpu"])):
        res = CliRunner().invoke(cli.cli, base + ["-o", str(out)] + extra, catch_exceptions=False)
        assert res.exit_code == 0, res.output
    files = sorted(p.relative_to(a) for p in a.rglob("*") if p.is_file())
    assert files and files == sorted(p.relative_to(b) for p in b.rglob("*") if p.is_file())
    n_png = n_jpg = 0
    for f in files:
        fa, fb = a / f, b / f
        if f.suffix.lower() == ".png":
            assert np.array_equal(np.asarray(Image.open(fa)), np.asarray(Image.open(fb)))
            n_png += 1
            if fa.read_bytes() != fb.read_bytes():
                assert fb.read_bytes() == png_ref.encode(np.asarray(Image.open(fb)))
        else:
            assert fa.read_bytes() == fb.read_bytes()
            n_jpg += 1
    assert n_png > 0 and n_jpg > 0

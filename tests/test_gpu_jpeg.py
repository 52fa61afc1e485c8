"""JPEG files encoded on the device (mb_jpeg_encode through CropStage.bind_jpeg / filter_and_crop(jpeg=True)): every
stream equals tests/jpeg_ref.py and PIL's default JPEG writer byte for byte."""
import ctypes as C
import io

import numpy as np
import pytest
import torch
from PIL import Image

from tests import jpeg_ref
from tests.test_gpu_png import _streams, crop_all, cu
from tests.test_jpeg_ref import pil_jpeg, sweep_cases
from tests.test_png_ref import particle_crop

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def check_stage(stage, channels, ref=True):
    crops = stage.to_host(channels)
    files = stage.jpeg_to_host()
    assert len(files) == len(crops)
    for (_, _, _, a), s in zip(crops, files):
        assert s == (pil_jpeg(a) if a.size else b"")
        if ref:
            assert s == jpeg_ref.encode(a)
    return crops, files


def canvas_of(arrays, channels):
    """The arrays side by side on one image, and their (x, y, w, h) rectangles."""
    H = max(a.shape[0] for a in arrays)
    canvas = np.zeros((H, sum(a.shape[1] for a in arrays)) + ((3,) if channels == 3 else ()), np.uint8)
    rects, x = [], 0
    for a in arrays:
        canvas[:a.shape[0], x:x + a.shape[1]] = a
        rects.append((x, 0, a.shape[1], a.shape[0]))
        x += a.shape[1]
    return canvas, rects


@pytest.mark.parametrize("channels", [1, 3])
def test_size_and_content_sweep(channels):
    arrays = [a for _, a in sweep_cases(channels)]
    canvas, rects = canvas_of(arrays, channels)
    st = crop_all([canvas], [rects], jpeg=True)
    crops, files = check_stage(st, channels)
    assert len(files) == len(arrays)
    for a, (_, _, _, c) in zip(arrays, crops):
        assert np.array_equal(a, c)


@pytest.mark.parametrize("channels", [1, 3])
def test_random_rect_crops(channels):
    rng = np.random.default_rng(10 + channels)
    images, rects = [], []
    for i in range(3):
        h, w = int(rng.integers(200, 400)), int(rng.integers(200, 400))
        base = particle_crop(rng, h, w, 3)
        images.append(base[..., 0].copy() if channels == 1 else base)
        rects.append([(int(rng.integers(-20, w)), int(rng.integers(-20, h)), int(rng.integers(0, 120)),
                       int(rng.integers(0, 120))) for _ in range(100)])
    st = crop_all(images, rects, jpeg=True)
    crops, files = check_stage(st, channels)
    assert len(crops) == 300
    assert any(len(s) == 0 for s in files)          # zero-area crops give empty streams


def test_chunked_plan():
    """More than 8192 slots: the chunked crop plan feeds the encoder the same way."""
    rng = np.random.default_rng(7)
    images = [particle_crop(rng, 128, 128, 3) for _ in range(3)]
    rects = [[(int(rng.integers(0, 120)), int(rng.integers(0, 120)), int(rng.integers(1, 9)), int(rng.integers(1, 9)))
              for _ in range(3000)] for _ in range(3)]
    st = crop_all(images, rects, jpeg=True)
    crops, _ = check_stage(st, 3)
    assert len(crops) == 9000


def test_large_noise_crop():
    rng = np.random.default_rng(11)
    im = rng.integers(0, 256, (3072, 4096, 3), dtype=np.uint8)
    st = crop_all([im], [[(0, 0, 4096, 3072)]], jpeg=True)
    s, = st.jpeg_to_host()
    assert s == pil_jpeg(im)


def test_bound_bytes_formula():
    from miso_b200 import _lib
    lib = _lib.load()
    for packed, crops, ch in ((0, 0, 1), (1, 1, 1), (100, 3, 1), (3, 1, 3), (12345678, 1000, 3), (1 << 33, 5, 1)):
        assert lib.mb_jpeg_bound_bytes(packed, crops, ch) == jpeg_ref.jpeg_bound(packed, crops, ch)
    for ch in (0, 2, 4):
        assert lib.mb_jpeg_bound_bytes(100, 1, ch) == -1


def test_overflow_unsupported_and_pixel_overflow():
    from miso_b200 import _lib, detection
    from miso_b200._lib import MisoB200Error
    from miso_b200.ops import _ptr
    rng = np.random.default_rng(3)
    im = rng.integers(0, 256, (64, 64, 3), dtype=np.uint8)
    stream = torch.cuda.current_stream().cuda_stream
    st = crop_all([im], [[]], jpeg=True)                              # no crops
    assert st.jpeg_to_host() == []
    st = crop_all([im], [[(70, 70, 5, 5), (0, 0, 0, 3)]], jpeg=True)    # zero-area crops
    assert st.jpeg_to_host() == [b"", b""]
    # output too small: flag 1, nothing written
    stage = crop_all([im], [[(0, 0, 32, 32), (5, 9, 17, 3)]])
    stage.bind_jpeg(capacity_bytes=600)
    stage.jpeg["out"].fill_(0xAB)
    stage.cut(stream)
    status = stage.jpeg["status"].tolist()
    assert status[1] == 1 and status[0] == len(pil_jpeg(im[:32, :32])) + len(pil_jpeg(im[9:12, 5:22]))
    assert int((stage.jpeg["out"] != 0xAB).sum()) == 0
    with pytest.raises(MisoB200Error):
        stage.jpeg_to_host()
    # workspace too small: flag 2, nothing written
    stage = crop_all([im], [[(0, 0, 32, 32)]])
    stage.bind_jpeg()
    stage.jpeg["ws"] = torch.empty((512,), dtype=torch.uint8, device=DEV)
    stage.jpeg["out"].fill_(0xAB)
    stage.cut(stream)
    assert stage.jpeg["status"].tolist()[1] == 2
    assert int((stage.jpeg["out"] != 0xAB).sum()) == 0
    with pytest.raises(MisoB200Error):
        stage.jpeg_to_host()
    # channels 2 and 4: MB_ERR_UNSUPPORTED from the library, an error from the Python layer
    lib = _lib.load()
    buf = stage.jpeg
    for ch in (2, 4):
        rc = lib.mb_jpeg_encode(C.byref(stage.params), _ptr(stage.pixels), ch, _ptr(stage.rects), _ptr(stage.offsets),
                                _ptr(stage.totals), _ptr(buf["ws"]), buf["ws"].numel(), _ptr(buf["out"]), buf["capacity"],
                                _ptr(buf["offsets"]), _ptr(buf["status"]), stream)
        assert rc == -3
        four = cu(rng.integers(0, 256, (16, 16, ch), dtype=np.uint8))
        with pytest.raises(MisoB200Error):
            detection.filter_and_crop([four], cu(np.array([[[0, 0, 8, 8]]], np.float32)), cu(np.ones((1, 1), np.float32)),
                                      cu(np.ones((1,), np.int32)), 0.5, boxes_are_xywh=True, jpeg=True)
    # a pixel overflow flag in totals: nothing is encoded
    stage = crop_all([im], [[(0, 0, 32, 32)]], capacity_bytes=100)
    stage.bind_jpeg()
    stage.cut(stream)
    assert int(stage.totals[2]) == 1
    assert stage.jpeg["status"].tolist() == [0, 0] and int(stage.jpeg["offsets"][0]) == 0


def test_infer_mosaic_jpeg_world1_and_two_ranks():
    """infer_mosaic(jpeg=True): every crop's file equals PIL's, and two emulated ranks give world 1's files in rank
    order."""
    from miso_b200 import mosaic
    from miso_b200.patch import forward_uint8, patch_model
    from tests.test_gpu_crop_masks import make_model
    model = patch_model(make_model("mask").to(DEV))
    g = torch.Generator().manual_seed(5)
    mos = torch.randint(0, 256, (1536, 1536, 3), dtype=torch.uint8, generator=g).to(DEV)
    kw = dict(tile=1024, overlap=128, threshold=0.1, batch_size=2)
    res = mosaic.infer_mosaic(model, mos, (1536, 1536), jpeg=True, **kw)
    c = res["crops"]
    assert c["count"] > 0
    files = _streams(c["jpeg"], c["jpeg_offsets"])
    rects, offs = c["rects"].cpu().numpy(), c["offsets"].cpu().numpy()
    pix = c["pixels"].cpu().numpy()
    for j in range(c["count"]):
        _, _, w, h = rects[j]
        a = pix[offs[j]:offs[j + 1]].reshape(h, w, 3)
        assert files[j] == (pil_jpeg(a) if a.size else b""), j
    grid, dpi = mosaic.tile_grid(1536, 1536, 1024, 128), int(model.roi_heads.detections_per_img)
    got = []
    for rank in range(2):
        y0, y1 = mosaic.rank_band(grid, 1024, 1536, 2, rank)
        crops = mosaic.MosaicCrops(2 * dpi, (1536, 1536), 3, 0.1, 256 << 20, DEV)
        crops.bind_band(mos[y0:y1].contiguous(), y0)
        crops.bind_jpeg()
        crops.launch(res["gathered"], res["state"], rank * 2 * dpi)
        o = crops.results()
        got += _streams(o["jpeg"], o["jpeg_offsets"])
    assert got == files


def _tree(root):
    return sorted(p.relative_to(root) for p in root.rglob("*") if p.is_file())


def test_crop_objects_and_cli_jpeg_on_gpu(tmp_path):
    """--jpeg-on-gpu writes the same file tree as the default run, byte for byte: RGB JPEGs, a grey JPEG and a PNG;
    crop_objects(jpeg_on_gpu=True) likewise, and together with png_on_gpu."""
    from click.testing import CliRunner
    import miso.cli as cli
    from miso.object_detection.crop import crop_objects
    from miso.object_detection.inference import infer_directory
    from tests.test_gpu_crop_masks import save_model
    idir = tmp_path / "in" / "sub"
    idir.mkdir(parents=True)
    rng = np.random.default_rng(1)
    Image.fromarray(particle_crop(rng, 384, 512, 3)).save(idir / "a.jpg", quality=95)
    Image.fromarray(rng.integers(0, 256, (300, 400, 3), dtype=np.uint8)).save(idir / "b.JPEG")
    Image.fromarray(particle_crop(rng, 256, 320, 3)[..., 0]).save(idir / "c.jpeg")
    Image.fromarray(particle_crop(rng, 256, 320, 3)).save(idir / "d.png")
    mdir = save_model(tmp_path, "mask")
    base = ["infer-object-detector-directory", "-i", str(tmp_path / "in"), "--model-dir", str(tmp_path / "models"),
            "--threshold", "0.1", "--batch-size", "2", "--model", "mask"]
    a, b = tmp_path / "cpu", tmp_path / "gpu"
    for out, extra in ((a, []), (b, ["--jpeg-on-gpu"])):
        res = CliRunner().invoke(cli.cli, base + ["-o", str(out)] + extra, catch_exceptions=False)
        assert res.exit_code == 0, res.output
    files = _tree(a)
    assert files and files == _tree(b)
    suffixes = {f.suffix for f in files}
    assert {".jpg", ".JPEG", ".jpeg", ".png"} <= suffixes
    for f in files:
        assert (a / f).read_bytes() == (b / f).read_bytes(), f
    # the Python entry point, alone and with png_on_gpu
    project = infer_directory(str(tmp_path / "in"), str(mdir / "model.pt"), ["Coccolith", "Coccosphere"], 0.1, 2)
    outs = {}
    for name, kw in (("cpu", {}), ("jpeg", {"jpeg_on_gpu": True}), ("both", {"jpeg_on_gpu": True, "png_on_gpu": True})):
        crop_objects(project, str(tmp_path / f"py_{name}"), relative_to=str(tmp_path / "in"), **kw)
        outs[name] = tmp_path / f"py_{name}"
    assert _tree(outs["cpu"]) == _tree(outs["jpeg"]) == _tree(outs["both"])
    for f in _tree(outs["cpu"]):
        if f.suffix.lower() in (".jpg", ".jpeg"):
            assert (outs["cpu"] / f).read_bytes() == (outs["jpeg"] / f).read_bytes() == (outs["both"] / f).read_bytes()
        else:
            assert (outs["cpu"] / f).read_bytes() == (outs["jpeg"] / f).read_bytes()
            assert np.array_equal(np.asarray(Image.open(outs["cpu"] / f)), np.asarray(Image.open(outs["both"] / f)))

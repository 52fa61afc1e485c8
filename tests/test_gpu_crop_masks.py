"""Per-crop instance masks (mb_crop_masks): the paste of each surviving detection's 28x28 mask probabilities into its
frame (image or tile), cut to its crop rectangle and thresholded, against torchvision's CPU paste_masks_in_image
(up to the paste kernel's documented 1-ulp band) and against mb_paste_masks (bit for bit), through every layer:
filter_and_crop, forward_uint8(paste_masks=False), MosaicCrops.bind_masks / infer_mosaic(masks=True), infer_directory
(with_masks=True), crop_objects(mask_dir=...) and the CLI's --mask-dir."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import cases
from tests.test_gpu_model import make_model

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ULP_BAND = 2.4e-7       # mb_paste_masks vs torchvision's CPU loop on small outputs (tests/test_gpu_model.py)


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def cut(full, rect, frame, thr):
    """Reference semantics: (full[y + r - y0, x + c - x0] > thr) * 255, 0 outside the frame. full: [fh, fw] numpy."""
    x, y, w, h = (int(v) for v in rect)
    x0, y0 = int(frame[0]), int(frame[1])
    out = np.zeros((h, w), np.uint8)
    vals = np.zeros((h, w), np.float32)
    ys, xs = y - y0, x - x0
    r0, r1 = max(0, -ys), min(h, full.shape[0] - ys)
    c0, c1 = max(0, -xs), min(w, full.shape[1] - xs)
    if r1 > r0 and c1 > c0:
        vals[r0:r1, c0:c1] = full[ys + r0:ys + r1, xs + c0:xs + c1]
        out[r0:r1, c0:c1] = np.where(full[ys + r0:ys + r1, xs + c0:xs + c1] > np.float32(thr), 255, 0)
    return out, vals


def check_against_references(got, full_cpu, full_gpu, rect, frame, thr, stats):
    want_gpu, _ = cut(full_gpu, rect, frame, thr)
    assert np.array_equal(got, want_gpu)                          # same paste arithmetic: bit for bit
    want_cpu, vals = cut(full_cpu, rect, frame, thr)
    bad = got != want_cpu
    assert np.all(np.abs(vals[bad] - np.float32(thr)) <= ULP_BAND)
    stats[0] += int(bad.sum()); stats[1] += got.size


def special_boxes(hw):
    h, w = hw
    return np.array([[-5.0, -3.0, 40.0, 30.0],          # partly outside (top left)
                     [w - 20.3, h - 15.7, w + 12.0, h + 9.0],    # partly outside (bottom right)
                     [10.2, 11.1, 10.5, 11.3],           # sub-pixel: pasted size clamps to 1
                     [3.0, h - 1.0, 25.0, float(h)],     # last row
                     [w - 1.0, 4.0, float(w), 50.0],     # last column
                     [7.0, 8.0, 30.0, 60.0],             # odd width / height
                     [0.0, 0.0, float(w), float(h)]], np.float32)


def per_image_case(rng, ch, cap=40, sizes=((200, 300), (233, 157)), m=28):
    n = len(sizes)
    imgs = [rng.integers(0, 256, (h, w, ch) if ch > 1 else (h, w), dtype=np.uint8) for h, w in sizes]
    boxes = np.zeros((n, cap, 4), np.float32)
    for i, hw in enumerate(sizes):
        sp = special_boxes(hw)
        boxes[i, :len(sp)] = sp
        boxes[i, len(sp):] = cases.stress_rois(rng, cap - len(sp), hw, side=(2.0, 150.0))
    scores = rng.uniform(0.0, 1.0, (n, cap)).astype(np.float32)
    scores[:, :7] = 0.9
    counts = np.array([cap, cap - 7], np.int32)
    probs = rng.uniform(0.0, 1.0, (n, cap, m, m)).astype(np.float32)
    return imgs, boxes, scores, counts, probs


@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("thr", [0.5, 0.25])
def test_crop_masks_equal_the_pasted_masks_cut_to_the_crops(ch, thr):
    from torchvision.models.detection.roi_heads import paste_masks_in_image as tv_paste
    from miso_b200 import detection, ops
    rng = np.random.default_rng(3 + ch)
    imgs, boxes, scores, counts, probs = per_image_case(rng, ch)
    cap = boxes.shape[1]
    out = detection.filter_and_crop([cu(a) for a in imgs], cu(boxes), cu(scores), cu(counts), 0.3,
                                    mask_probs=cu(probs), mask_threshold=thr)
    crops = out.to_host(ch)
    masks = out.masks_to_host()
    assert len(masks) == len(crops) > 40
    rects = out.rects[:len(crops)].cpu().numpy()
    full_cpu = [tv_paste(torch.from_numpy(probs[i, :counts[i], None]), torch.from_numpy(boxes[i, :counts[i]]), a.shape[:2]).numpy()
                for i, a in enumerate(imgs)]
    full_gpu = [ops.paste_masks_in_image(cu(probs[i, :counts[i], None]), cu(boxes[i, :counts[i]]), a.shape[:2]).cpu().numpy()
                for i, a in enumerate(imgs)]
    stats = [0, 0]
    for j, ((n, d, _, crop), mk) in enumerate(zip(crops, masks)):
        assert mk.dtype == np.uint8 and mk.shape == crop.shape[:2]
        check_against_references(mk, full_cpu[n][d, 0], full_gpu[n][d, 0], rects[j], (0, 0), thr, stats)
    assert stats[1] > 10000 and stats[0] <= max(4, stats[1] // 10000)
    assert set(np.unique(np.concatenate([m.ravel() for m in masks]))) == {0, 255}


def test_probability_equal_to_the_threshold_gives_zero():
    from miso_b200 import detection, ops
    img = np.zeros((64, 80, 3), np.uint8)
    boxes = np.array([[[4.0, 6.0, 60.0, 50.0], [10.0, 10.0, 38.0, 38.0]]], np.float32)     # 28 px box: unit scale
    probs = np.full((1, 2, 28, 28), 0.5, np.float32)
    out = detection.filter_and_crop([cu(img)], cu(boxes), cu(np.ones((1, 2), np.float32)), cu(np.array([2], np.int32)), 0.5,
                                    mask_probs=cu(probs), mask_threshold=0.5)
    masks = out.masks_to_host()
    full = ops.paste_masks_in_image(cu(probs[0, :, None]), cu(boxes[0]), (64, 80)).cpu().numpy()
    rects = out.rects[:2].cpu().numpy()
    n_equal = 0
    for j, mk in enumerate(masks):
        x, y, w, h = rects[j]
        vals = full[j, 0, y:y + h, x:x + w]
        n_equal += int((vals == np.float32(0.5)).sum())
        assert not mk[vals == np.float32(0.5)].any()
        assert np.array_equal(mk, np.where(vals > np.float32(0.5), 255, 0))
    assert n_equal > 100


def test_frames_at_nonzero_origins_and_rectangles_leaving_them():
    """MosaicCrops.bind_masks: row s pastes into frame s // rows_per_frame (mosaic coordinates); crop rectangles that
    leave their frame are 0 there."""
    from torchvision.models.detection.roi_heads import paste_masks_in_image as tv_paste
    from miso_b200 import mosaic, ops
    rng = np.random.default_rng(11)
    H, W, dpi = 300, 400, 8
    frames = np.array([[0, 0, 160, 120], [150, 100, 200, 150], [230, 170, 170, 130]], np.int32)
    rows = len(frames) * dpi
    paste = np.concatenate([cases.stress_rois(rng, dpi, (f[3], f[2]), side=(6.0, 110.0)) for f in frames])
    origin = np.repeat(frames[:, [0, 1, 0, 1]].astype(np.float32), dpi, axis=0)
    block = np.zeros((rows, 6), np.float32)
    block[:, :4] = paste + origin
    block[::3, :2] -= 25.0                          # crop rectangles reaching out of the frame
    block[1::3, 2:4] += 30.0
    block[:, 4] = rng.uniform(0.0, 1.0, rows).astype(np.float32)
    block[:, 4][:rows // 2] = 0.9
    probs = rng.uniform(0.0, 1.0, (rows, 28, 28)).astype(np.float32)
    crops = mosaic.MosaicCrops(rows, (H, W), 3, 0.3, 1 << 20, DEV)
    crops.bind_band(cu(rng.integers(0, 256, (H, W, 3), dtype=np.uint8)), 0)
    crops.bind_masks(cu(probs), cu(paste), cu(frames), dpi, 0.5)
    crops.launch(cu(block), torch.ones((rows,), dtype=torch.int32, device=DEV), 0)
    res = crops.results()
    k = res["count"]
    assert k >= rows // 2
    rects, src = res["rects"].cpu().numpy(), res["src"].cpu().numpy()
    offs, buf = res["offsets"].cpu().numpy() // 3, res["masks"].cpu().numpy()
    assert len(buf) == res["bytes"] // 3
    stats, outside = [0, 0], 0
    for j in range(k):
        s = int(src[j]); f = frames[s // dpi]
        full_cpu = tv_paste(torch.from_numpy(probs[s][None, None]), torch.from_numpy(paste[s][None]), (int(f[3]), int(f[2])))[0, 0].numpy()
        full_gpu = ops.paste_masks_in_image(cu(probs[s][None, None]), cu(paste[s][None]), (int(f[3]), int(f[2])))[0, 0].cpu().numpy()
        mk = buf[offs[j]:offs[j + 1]].reshape(rects[j][3], rects[j][2])
        check_against_references(mk, full_cpu, full_gpu, rects[j], f, 0.5, stats)
        x, y, w, h = rects[j]
        outside += w * h - max(0, min(x + w, f[0] + f[2]) - max(x, f[0])) * max(0, min(y + h, f[1] + f[3]) - max(y, f[1]))
    assert outside > 100 and stats[0] <= max(4, stats[1] // 10000)


def test_chunked_plan_masks_follow_src_and_offsets():
    """60 x 520 slots: the chunked plan kernel; every crop's mask equals mb_paste_masks' paste cut to its rectangle."""
    from miso_b200 import detection, ops
    rng = np.random.default_rng(17)
    n, cap, hw = 60, 520, (96, 128)
    imgs = [rng.integers(0, 256, (hw[0], hw[1], 3), dtype=np.uint8) for _ in range(n)]
    boxes = np.stack([cases.stress_rois(rng, cap, hw, side=(2.0, 90.0)) for _ in range(n)])
    scores = rng.uniform(0.0, 1.0, (n, cap)).astype(np.float32)
    counts = rng.integers(0, cap + 1, n).astype(np.int32)
    probs = cu(rng.uniform(0.0, 1.0, (n * cap, 1, 28, 28)).astype(np.float32))
    db = cu(boxes)
    out = detection.filter_and_crop([cu(a) for a in imgs], db, cu(scores), cu(counts), 0.5, capacity_bytes=0, mask_probs=probs)
    masks = out.masks_to_host()
    k = len(masks)
    assert k > 1000 and int(out.totals[2]) == 1          # no pixel gather ran (capacity 0); the masks do not need it
    rects, src = out.rects[:k].cpu().numpy(), out.src[:k].cpu().numpy()
    full = [ops.paste_masks_in_image(probs[i * cap:i * cap + int(counts[i])], db[i, :int(counts[i])], hw).cpu().numpy() for i in range(n)]
    for j in range(k):
        i, d = divmod(int(src[j]), cap)
        want, _ = cut(full[i][d, 0], rects[j], (0, 0), 0.5)
        assert np.array_equal(masks[j], want)


def test_edge_cases_zero_crops_overflow_and_unsupported_side():
    from miso_b200 import _lib, detection
    from miso_b200._lib import MisoB200Error
    rng = np.random.default_rng(2)
    imgs, boxes, scores, counts, probs = per_image_case(rng, 3)
    dimgs = [cu(a) for a in imgs]
    # zero crops: everything below the threshold
    out = detection.filter_and_crop(dimgs, cu(boxes), cu(scores * 0), cu(counts), 0.5, mask_probs=cu(probs))
    assert out.masks_to_host() == [] and int(out.totals[3]) == 0
    # overflow: nothing written, totals[3] set, the host helper names the bytes needed
    out = detection.filter_and_crop(dimgs, cu(boxes), cu(scores), cu(counts), 0.3, mask_probs=cu(probs))
    need = int(out.totals[1]) // 3
    small = detection.filter_and_crop(dimgs, cu(boxes), cu(scores), cu(counts), 0.3, mask_probs=cu(probs), mask_capacity_bytes=need - 1)
    with pytest.raises(MisoB200Error, match=f"{need} bytes needed"):
        small.masks_to_host()
    p = _lib.CropParams()
    p.num_images, p.capacity, p.channels = 2, boxes.shape[1], 3
    for i, a in enumerate(imgs):
        p.image_h[i], p.image_w[i] = a.shape[0], a.shape[1]
    buf = torch.full((need - 1,), 77, dtype=torch.uint8, device=DEV)
    dp, db = cu(probs), cu(boxes)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = _lib.load().mb_crop_masks(C.byref(p), C.c_void_p(dp.data_ptr()), C.c_void_p(db.data_ptr()), 28, 1, None, boxes.shape[1], 0.5,
                                   C.c_void_p(out.rects.data_ptr()), C.c_void_p(out.src.data_ptr()), C.c_void_p(out.offsets.data_ptr()),
                                   C.c_void_p(out.totals.data_ptr()), C.c_void_p(buf.data_ptr()), need - 1, st)
    assert rc == 0 and int(out.totals[3]) == 1 and bool((buf == 77).all())
    # M + 2 * padding > 64
    big = cu(rng.uniform(0.0, 1.0, (2, boxes.shape[1], 63, 63)).astype(np.float32))
    with pytest.raises(MisoB200Error, match="unsupported"):
        detection.filter_and_crop(dimgs, cu(boxes), cu(scores), cu(counts), 0.3, mask_probs=big)


def test_forward_uint8_without_paste_returns_the_mask_probabilities():
    from miso_b200 import ops
    from miso_b200.patch import forward_uint8, patch_model
    model = patch_model(make_model("mask").to(DEV))
    g = torch.Generator().manual_seed(5)
    u8 = [torch.randint(0, 256, (300 + 40 * i, 420 - 30 * i, 3), dtype=torch.uint8, generator=g).to(DEV) for i in range(2)]
    with torch.inference_mode():
        a = forward_uint8(model, u8)
        b = forward_uint8(model, u8, paste_masks=False)
    for x, y, im in zip(a, b, u8):
        assert torch.equal(x["boxes"], y["boxes"]) and torch.equal(x["labels"], y["labels"]) and torch.equal(x["scores"], y["scores"])
        assert "masks" not in y and y["mask_probs"].shape[1:] == (1, 28, 28) and y["mask_probs"].shape[0] == x["boxes"].shape[0]
        assert torch.equal(ops.paste_masks_in_image(y["mask_probs"], y["boxes"], tuple(im.shape[:2])), x["masks"])
    assert sum(int(x["boxes"].shape[0]) for x in a) > 0


@pytest.fixture(scope="module")
def mask_mosaic():
    from miso_b200 import mosaic
    from miso_b200.patch import forward_uint8, patch_model
    model = patch_model(make_model("mask").to(DEV))
    g = torch.Generator().manual_seed(5)
    mos = torch.randint(0, 256, (1536, 1536, 3), dtype=torch.uint8, generator=g).to(DEV)
    thr, mthr = 0.1, 0.5
    kw = dict(tile=1024, overlap=128, threshold=thr, batch_size=2)
    res = mosaic.infer_mosaic(model, mos, (1536, 1536), masks=True, mask_threshold=mthr, **kw)
    plain = mosaic.infer_mosaic(model, mos, (1536, 1536), **kw)
    grid = mosaic.tile_grid(1536, 1536, 1024, 128)
    per_tile = []
    with torch.inference_mode():
        for i0 in range(0, 4, 2):      # the batches infer_mosaic ran
            tiles = [mos[y:y + 1024, x:x + 1024] for y, x in grid[i0:i0 + 2]]
            full = forward_uint8(model, tiles)
            probs = forward_uint8(model, tiles, paste_masks=False)
            per_tile += [(f, p) for f, p in zip(full, probs)]
    return dict(model=model, mos=mos, res=res, plain=plain, grid=grid, per_tile=per_tile, thr=thr, mthr=mthr,
                dpi=int(model.roi_heads.detections_per_img))


def test_infer_mosaic_masks_equal_the_per_tile_paste(mask_mosaic):
    mm = mask_mosaic
    res, plain, dpi = mm["res"], mm["plain"], mm["dpi"]
    assert torch.equal(res["gathered"], plain["gathered"]) and torch.equal(res["state"], plain["state"])
    c, p = res["crops"], plain["crops"]
    assert c["count"] == p["count"] > 0 and "masks" not in p
    for key in ("rects", "xywh", "src", "offsets", "pixels"):
        assert torch.equal(c[key], p[key]), key
    rects, src = c["rects"].cpu().numpy(), c["src"].cpu().numpy()
    offs, buf = c["offsets"].cpu().numpy() // 3, c["masks"].cpu().numpy()
    assert len(buf) == c["bytes"] // 3
    lit = 0
    for j in range(c["count"]):
        t, d = divmod(int(src[j]), dpi)
        y0, x0 = mm["grid"][t]
        full = mm["per_tile"][t][0]["masks"][d, 0].cpu().numpy()
        want, _ = cut(full, rects[j], (x0, y0), mm["mthr"])
        got = buf[offs[j]:offs[j + 1]].reshape(rects[j][3], rects[j][2])
        assert np.array_equal(got, want), j
        lit += int((got == 255).sum())
    assert lit > 0


def test_infer_mosaic_masks_of_two_emulated_ranks_equal_world1(mask_mosaic):
    """World size 2 over the same gathered rows (4 tiles: rank r owns tiles 2r, 2r + 1, the gathered layout is world
    1's): each rank's MosaicCrops cuts its own rows' masks; concatenated in rank order they equal world 1's."""
    from miso_b200 import mosaic
    mm = mask_mosaic
    dpi, grid, mos = mm["dpi"], mm["grid"], mm["mos"]
    gathered, state = mm["res"]["gathered"], mm["res"]["state"]
    outs = []
    for rank in range(2):
        mine = list(mosaic.rank_tiles(4, 2, rank))
        y0, y1 = mosaic.rank_band(grid, 1024, 1536, 2, rank)
        probs = torch.zeros((2 * dpi, 28, 28), dtype=torch.float32, device=DEV)
        boxes = torch.zeros((2 * dpi, 4), dtype=torch.float32, device=DEV)
        for i, t in enumerate(mine):
            r = mm["per_tile"][t][1]
            k = r["boxes"].shape[0]
            probs[i * dpi:i * dpi + k], boxes[i * dpi:i * dpi + k] = r["mask_probs"][:, 0], r["boxes"]
        frames = torch.tensor([[grid[t][1], grid[t][0], 1024, 1024] for t in mine], dtype=torch.int32, device=DEV)
        crops = mosaic.MosaicCrops(2 * dpi, (1536, 1536), 3, mm["thr"], 256 << 20, DEV)
        crops.bind_band(mos[y0:y1].contiguous(), y0)
        crops.bind_masks(probs, boxes, frames, dpi, mm["mthr"])
        crops.launch(gathered, state, rank * 2 * dpi)
        outs.append(crops.results())
    w1 = mm["res"]["crops"]
    assert all(o["count"] > 0 for o in outs) and sum(o["count"] for o in outs) == w1["count"]
    assert torch.equal(torch.cat([o["rects"] for o in outs]), w1["rects"])
    assert torch.equal(torch.cat([o["masks"] for o in outs]), w1["masks"])


def test_masks_need_a_mask_head():
    from miso_b200 import mosaic
    from miso_b200._lib import MisoB200Error
    from miso_b200.patch import patch_model
    model = patch_model(make_model("faster").to(DEV))
    mos = torch.zeros((1024, 1024, 3), dtype=torch.uint8, device=DEV)
    with pytest.raises(MisoB200Error, match="mask head"):
        mosaic.infer_mosaic(model, mos, (1024, 1024), masks=True)


def save_model(tmp_path, kind):
    mdir = tmp_path / "models" / kind
    mdir.mkdir(parents=True)
    torch.save(make_model(kind), mdir / "model.pt")
    (mdir / "labels.txt").write_text("0,Coccolith\n1,Coccosphere\n")
    return mdir


def write_images(tmp_path):
    from PIL import Image
    idir = tmp_path / "in" / "sub"
    idir.mkdir(parents=True)
    rng = np.random.default_rng(0)
    for name in ("a.png", "b.png"):
        Image.fromarray(rng.integers(0, 256, (384, 512, 3), dtype=np.uint8)).save(idir / name)
    return tmp_path / "in"


def test_infer_directory_with_masks_equals_the_full_image_paste(tmp_path):
    """Each annotation's mask is its detection's full-image mask (forward_uint8's default paste), cut to the crop."""
    from miso.object_detection.inference import infer_directory, load_model, read_image
    from miso_b200.patch import forward_uint8
    mdir = save_model(tmp_path, "mask")
    idir = write_images(tmp_path)
    thr = 0.1
    project = infer_directory(str(idir), str(mdir / "model.pt"), ["Coccolith", "Coccosphere"], thr, 2, with_masks=True)
    metas = list(project.image_dict.values())
    model = load_model(str(mdir / "model.pt"))
    with torch.inference_mode():
        ref = forward_uint8(model, [torch.from_numpy(np.array(read_image(m.full_path))).to(DEV) for m in metas])
    seen = 0
    for m, r in zip(metas, ref):
        live = (r["scores"] > thr).cpu().numpy()
        full = r["masks"][:, 0].cpu().numpy()[live]
        assert len(m.boxes) == len(full)
        for box, f in zip(m.boxes, full):
            c = box.coords_int
            assert box.mask.dtype == np.uint8 and np.array_equal(box.mask, np.where(f[c[1]:c[3], c[0]:c[2]] > np.float32(0.5), 255, 0))
            seen += 1
    assert seen > 0


def test_cli_mask_dir_writes_one_mask_per_crop(tmp_path):
    from click.testing import CliRunner
    from PIL import Image
    import miso.cli as cli
    idir = write_images(tmp_path)
    mdir = save_model(tmp_path, "mask")
    save_model(tmp_path, "faster")
    base = ["infer-object-detector-directory", "-i", str(idir), "--model-dir", str(tmp_path / "models"), "--threshold", "0.1",
            "--batch-size", "2"]
    odir, kdir = tmp_path / "out", tmp_path / "masks"
    res = CliRunner().invoke(cli.cli, base + ["-o", str(odir), "--model", "mask", "--mask-dir", str(kdir)], catch_exceptions=False)
    assert res.exit_code == 0, res.output
    crops = sorted(odir.rglob("*.png"))
    assert crops
    for f in crops:
        mf = kdir / f.relative_to(odir).with_suffix(".png")
        assert mf.exists(), mf
        with Image.open(mf) as im:
            assert im.mode == "L"
            mk = np.asarray(im)
        assert mk.shape == np.asarray(Image.open(f)).shape[:2] and set(np.unique(mk)) <= {0, 255}
    assert len(sorted(kdir.rglob("*.png"))) == len(crops)
    # without the option: the same crops, nothing else written
    res = CliRunner().invoke(cli.cli, base + ["-o", str(tmp_path / "out2"), "--model", "mask"], catch_exceptions=False)
    assert res.exit_code == 0
    assert sorted(p.relative_to(tmp_path / "out2") for p in (tmp_path / "out2").rglob("*")) == \
        sorted(p.relative_to(odir) for p in odir.rglob("*"))
    assert sorted(p.name for p in tmp_path.iterdir()) == ["in", "masks", "models", "out", "out2"]
    # a Faster R-CNN model has no masks to write
    res = CliRunner().invoke(cli.cli, base + ["-o", str(tmp_path / "out3"), "--model", "faster", "--mask-dir", str(tmp_path / "m3")])
    assert res.exit_code != 0 and "Mask R-CNN" in res.output and not (tmp_path / "m3").exists()

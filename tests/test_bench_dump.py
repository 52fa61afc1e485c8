"""bench.py --dump-outputs: dump_outputs writes the pass's outputs as float32 / float64 .npy files within the byte
budget (all ranks together), values exact, and the crop-byte sample is the same from run to run. Runs on the CPU."""
import os

import numpy as np
import torch

import bench


def fake_pass(rows=50, k=20, crop_bytes=None, seed=1):
    """gathered rows, seam state and crop results shaped like MosaicPlan's; crop_bytes=None: small random crops."""
    g = torch.Generator().manual_seed(seed)
    gathered = torch.rand((rows, 6), generator=g) * 4096
    gathered[:, 5] = torch.randint(-1, 3, (rows,), generator=g).float()
    state = torch.randint(1, 4, (rows,), generator=g, dtype=torch.int32)
    sizes = torch.randint(10, 400, (k,), generator=g) if crop_bytes is None else torch.full((k,), crop_bytes // k)
    offsets = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(sizes, 0)])
    res = {"xywh": torch.rand((k, 4), generator=g) * 1000, "rects": torch.randint(0, 16384, (k, 4), generator=g, dtype=torch.int32),
           "src": torch.randint(0, rows, (k,), generator=g, dtype=torch.int32), "offsets": offsets,
           "pixels": torch.randint(0, 256, (int(offsets[-1]),), generator=g, dtype=torch.uint8)}
    return gathered, state, res


def on_disk(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_dump_outputs_sample_within_budget(tmp_path):
    gathered, state, res = fake_pass()
    budget = 20_000
    out = bench.dump_outputs(str(tmp_path / "a"), gathered, state, res, budget=budget)
    again = bench.dump_outputs(str(tmp_path / "b"), gathered, state, res, budget=budget)
    assert sum(a.nbytes for a in out.values()) <= budget
    idx = out["crop_pixel_index"].astype(np.int64)
    assert 0 < len(idx) < res["pixels"].numel() and np.all(np.diff(idx) > 0)
    assert np.array_equal(out["crop_pixels"], res["pixels"].numpy()[idx].astype(np.float32))
    assert np.array_equal(out["gathered_rows"], gathered.numpy()) and np.array_equal(out["seam_state"], state.numpy())
    for name, key in (("crop_xywh", "xywh"), ("crop_rects", "rects"), ("crop_src_rows", "src"), ("crop_offsets", "offsets")):
        assert np.array_equal(out[name], res[key].numpy()), name
    for name, a in out.items():
        f = np.load(tmp_path / "a" / (name + ".npy"))
        assert f.dtype in (np.float32, np.float64), name
        assert np.array_equal(f, a) and np.array_equal(f, again[name]) and np.array_equal(f, np.load(tmp_path / "b" / (name + ".npy"))), name
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in out)


def test_dump_outputs_writes_every_crop_byte_when_they_fit(tmp_path):
    gathered, state, res = fake_pass()
    out = bench.dump_outputs(str(tmp_path), gathered, state, res)
    assert np.array_equal(out["crop_pixels"], res["pixels"].numpy().astype(np.float32))
    assert np.array_equal(out["crop_pixel_index"], np.arange(res["pixels"].numel()))


def test_default_budget_stays_under_64_mb_on_disk(tmp_path):
    """The default mosaic's row count and crop count, crop bytes far beyond the budget."""
    gathered, state, res = fake_pass(rows=108_300, k=107_887, crop_bytes=100_000_000)
    out = bench.dump_outputs(str(tmp_path), gathered, state, res)
    assert len(out["crop_pixels"]) > 3_000_000
    assert on_disk(tmp_path) <= 64_000_000


def test_ranks_share_the_budget_and_write_the_replicated_arrays_once(tmp_path):
    """Four ranks of one run: identical gathered rows / seam state, each rank its own crops."""
    world = 4
    outs = []
    for r in range(world):
        gathered, state, _ = fake_pass(rows=108_300, k=10, seed=0)
        _, _, res = fake_pass(rows=108_300, k=27_000, crop_bytes=30_000_000, seed=r + 1)
        outs.append(bench.dump_outputs(str(tmp_path), gathered, state, res, rank=r, world=world))
        assert np.array_equal(outs[r][f"crop_src_rows.rank{r}"], res["src"].numpy())
    assert on_disk(tmp_path) <= 64_000_000
    assert sorted(os.listdir(tmp_path)) == sorted(n + ".npy" for o in outs for n in o)
    assert "gathered_rows" in outs[0] and all("gathered_rows" not in o and "seam_state" not in o for o in outs[1:])
    assert all(f"crop_pixels.rank{r}" in outs[r] and len(outs[r][f"crop_pixels.rank{r}"]) > 1_000_000 for r in range(world))

"""Scenes with nodata on the CPU: the mask-derivation rule (data.nodata_mask), the masked restatements against the
unmasked ones (tests/masked_oracle.py), the writers' fill, and the dataset / CLI validation of the fill value."""
import math
import os

import numpy as np
import pytest
import torch

import masked_oracle as MO
import tiled_oracle as TO
import u16_reference as U
from fastdiffsr_b200.data import LRHRDataset, nodata_mask
from fastdiffsr_b200.evaluate import _save_u16, _save_u8, load_opt, parse_args


@pytest.mark.parametrize("h,w,H,W", [(5, 7, 5, 7), (4, 6, 16, 24), (13, 21, 52, 84), (10, 7, 25, 17), (9, 12, 16, 40),
                                     (20, 16, 7, 9)])
@pytest.mark.parametrize("dtype", [torch.uint8, torch.uint16])
def test_nodata_mask_rule(h, w, H, W, dtype):
    rng = np.random.default_rng(h * 100 + W)
    V = 3
    img = rng.integers(0, 6, (2, h, w, 3)).astype(np.uint16)
    img[rng.random((2, h, w)) < 0.4] = V                       # whole fill pixels, besides the random all-V ones
    img[0, :, 0, 1] = V                                        # partial fill: one band at V is still valid
    got = nodata_mask(torch.from_numpy(img.astype(np.uint8 if dtype == torch.uint8 else np.uint16)), V, H, W)
    assert got.dtype == torch.bool and tuple(got.shape) == (2, H, W)
    src_valid = ~(img == V).all(axis=3)
    ref = np.zeros((2, H, W), bool)
    for Y in range(H):
        for X in range(W):
            # the source pixel whose area [y, y + 1) x [x, x + 1) holds the HR centre ((Y + .5) h / H, (X + .5) w / W)
            y = math.floor((Y + 0.5) * h / H)
            x = math.floor((X + 0.5) * w / W)
            ref[:, Y, X] = src_valid[:, y, x]
    assert np.array_equal(got.numpy(), ref)


def test_nodata_mask_rejects_other_types():
    with pytest.raises(ValueError):
        nodata_mask(torch.zeros(1, 4, 4, 3, dtype=torch.float32), 0, 8, 8)
    with pytest.raises(ValueError):
        nodata_mask(torch.zeros(4, 4, 3, dtype=torch.uint8), 0, 8, 8)


@pytest.fixture(scope="module")
def small(oracle):
    cfg = dict(oracle.DEFAULT_UNET)
    sd = oracle.make_state_dict(cfg, seed=0, gn_jitter=0.1)
    tab = oracle.schedule_tables(oracle.make_beta_schedule(**oracle.DEFAULT_SCHEDULE))
    return cfg, sd, tab


def test_masked_oracle_all_valid_equals_tiled(small):
    cfg, sd, tab = small
    g = torch.Generator().manual_seed(4)
    cond = torch.rand(1, 3, 40, 56, generator=g) * 2 - 1
    noises = torch.randn(20, 1, 3, 40, 56, generator=g)
    valid = torch.ones(1, 40, 56, dtype=torch.bool)
    ref = TO.tiled_sample_loop(sd, cfg, tab, cond, noises, 32, 8, continous=True)
    assert torch.equal(MO.masked_tiled_sample_loop(sd, cfg, tab, cond, noises, valid, 32, 8, continous=True), ref)


def test_active_tiles():
    valid = torch.zeros(2, 100, 140, dtype=torch.bool)
    valid[0, 50, 80] = True                                    # inside the overlap of four tiles
    ys, tey, _ = TO.tile_starts(100, 64, 16)
    xs, tex, _ = TO.tile_starts(140, 64, 16)
    want = [(0, y0, x0) for y0 in ys for x0 in xs if y0 <= 50 < y0 + tey and x0 <= 80 < x0 + tex]
    assert MO.active_tiles(valid, 64, 16) == want and len(want) == 4
    assert MO.active_tiles(torch.ones(2, 100, 140, dtype=torch.bool), 64, 16) == [
        (b, y0, x0) for b in range(2) for y0 in ys for x0 in xs]


def test_masked_metrics_all_valid_equals_unmasked():
    rng = np.random.default_rng(0)
    for M in (255, 4095):
        a = rng.integers(0, M + 1, (30, 26, 3))
        b = np.clip(a + rng.integers(-M // 20, M // 20 + 1, a.shape), 0, M)
        got = MO.masked_metrics(a, b, np.ones((30, 26), bool), M)
        ref = U.metrics(a, b, M)
        assert got[0] == ref[0] and got[1] == ref[1]
        assert abs(got[2] - ref[2]) <= 1e-12 and abs(got[3] - ref[3]) <= 1e-12 * abs(ref[3])
        assert all(math.isnan(v) for v in MO.masked_metrics(a, b, np.zeros((30, 26), bool), M))
        sparse = np.zeros((30, 26), bool)
        sparse[::3, ::3] = True                                # valid pixels, but no wholly valid window
        m = MO.masked_metrics(a, b, sparse, M)
        assert math.isfinite(m[0]) and math.isnan(m[2])


def test_writers_fill_invalid_pixels(tmp_path):
    from PIL import Image
    img = torch.linspace(-1, 1, 3 * 6 * 5).reshape(3, 6, 5)
    valid = torch.ones(6, 5, dtype=torch.bool)
    valid[2:4, 1:3] = False
    p = _save_u8(img, str(tmp_path / "a.png"), fill=(valid, 7))
    u8 = np.asarray(Image.open(p))
    assert (u8[2:4, 1:3] == 7).all() and np.array_equal(u8[valid.numpy()], np.asarray(Image.open(_save_u8(
        img, str(tmp_path / "b.png"))))[valid.numpy()])
    p = _save_u16(img, str(tmp_path / "c.tif"), 4095, fill=(valid, 65535))
    u16 = np.load(p)
    assert u16.dtype == np.uint16 and (u16[2:4, 1:3] == 65535).all() and (u16[valid.numpy()] <= 4095).all()


def _folder(tmp_path):
    root = tmp_path / "ds"
    for d in ("hr_256", "lr_64"):
        os.makedirs(root / d)
    np.save(root / "hr_256" / "a.npy", np.zeros((8, 8, 1), np.uint8))
    np.save(root / "lr_64" / "a.npy", np.zeros((2, 2, 1), np.uint8))
    return str(root)


def test_dataset_nodata_range(tmp_path):
    root = _folder(tmp_path)
    assert LRHRDataset(root, channels=1).nodata is None
    assert LRHRDataset(root, channels=1, nodata=0).nodata == 0
    assert LRHRDataset(root, channels=1, nodata=255).nodata == 255
    for bad in (-1, 256, 2.5, True, 70000):
        with pytest.raises(ValueError):
            LRHRDataset(root, channels=1, nodata=bad)


def test_dataset_nodata_range_16bit(tmp_path):
    root = tmp_path / "ds"
    for d in ("hr_256", "lr_64"):
        os.makedirs(root / d)
    np.save(root / "hr_256" / "a.npy", np.zeros((8, 8, 1), np.uint16))
    np.save(root / "lr_64" / "a.npy", np.zeros((2, 2, 1), np.uint16))
    assert LRHRDataset(str(root), channels=1, max_value=4095, nodata=65535).nodata == 65535
    for bad in (-1, 65536):
        with pytest.raises(ValueError):
            LRHRDataset(str(root), channels=1, max_value=4095, nodata=bad)


def test_nodata_flag():
    args = parse_args(["-c", "sr_fastdiffsr_test_64_256", "--nodata", "0"])
    assert load_opt(args)["datasets"]["val"]["nodata"] == 0
    assert "nodata" not in load_opt(parse_args(["-c", "sr_fastdiffsr_test_64_256"]))["datasets"]["val"]
    for bad in (["--nodata", "-1"], ["--nodata", "65536"], ["--tile", "64", "--tile-split", "--nodata", "0"]):
        with pytest.raises(SystemExit):
            parse_args(bad)

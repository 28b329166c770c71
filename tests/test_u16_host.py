"""16-bit imagery on the host side (no GPU): the loader's 16-bit files and rejections, the normalisation and the
16-bit tensor2img, the 16-bit writers, the --max-value flag, and the numpy restatement of Pillow's I;16 resize
(tests/u16_reference.py) against Pillow."""
import os

import numpy as np
import pytest
import torch

import fastdiffsr_b200 as F
from fastdiffsr_b200 import data as D
from fastdiffsr_b200.evaluate import _save_u16, _save_u8, load_opt, parse_args

import u16_reference as R

M_LEVELS = (255, 1023, 2047, 4095, 10000, 16383, 65535)


def _write(root, d, name, a, kind):
    from PIL import Image
    os.makedirs(os.path.join(root, d), exist_ok=True)
    p = os.path.join(root, d, name + "." + kind)
    if kind == "npy":
        np.save(p, a)
    else:
        Image.fromarray(a).save(p)
    return p


def _pair(root, name, hr, lr, kind):
    _write(root, "hr_64", name, hr, kind)
    _write(root, "lr_16", name, lr, kind)


# ------------------------------------------------------------------------------------------ loader
@pytest.mark.parametrize("C", [1, 3, 4, 8])
def test_dataset_reads_uint16_npy(tmp_path, C):
    rng = np.random.default_rng(C)
    root = str(tmp_path / "ds")
    hr = rng.integers(0, 65536, (2, 64, 64, C), dtype=np.uint16)
    lr = rng.integers(0, 65536, (2, 16, 16, C), dtype=np.uint16)
    for i in range(2):
        _pair(root, f"img{i}", hr[i], lr[i], "npy")
    if C == 1:                                       # (H,W) is accepted for one band
        _pair(root, "img2", hr[0, ..., 0], lr[0, ..., 0], "npy")
    ds = D.LRHRDataset(root, "img", 16, 64, channels=C, max_value=65535)
    assert len(ds) == (3 if C == 1 else 2) and ds.max_value == 65535
    for i in range(2):
        it = ds.get_raw(i)
        assert it["HR"].dtype == np.uint16 and it["LR"].dtype == np.uint16
        assert np.array_equal(it["HR"], hr[i]) and np.array_equal(it["LR"], lr[i])
    if C == 1:
        assert np.array_equal(ds.get_raw(2)["HR"], hr[0])
    batch = next(iter(D.BatchLoader(ds, 2, pin=False)))
    assert batch["HR"].dtype == torch.uint16 and tuple(batch["HR"].shape) == (2, 64, 64, C)
    assert np.array_equal(batch["LR"].numpy(), lr)
    item = ds[1]                                     # __getitem__ normalises with M
    assert item["HR"].dtype == torch.float32 and item["HR"].shape == (C, 64, 64)
    assert np.array_equal(item["HR"].numpy(), R.u16_to_cond(hr[1], 65535).transpose(2, 0, 1))


@pytest.mark.parametrize("kind", ["png", "tif"])
def test_dataset_reads_single_band_i16_images_losslessly(tmp_path, kind):
    from PIL import Image
    rng = np.random.default_rng(7)
    root = str(tmp_path / kind)
    hr = rng.integers(0, 65536, (64, 48), dtype=np.uint16)
    hr[0, 0], hr[0, 1] = 0, 65535
    lr = rng.integers(0, 65536, (16, 12), dtype=np.uint16)
    _pair(root, "a", hr, lr, kind)
    with Image.open(os.path.join(root, "hr_64", "a." + kind)) as im:
        assert im.mode.startswith("I")
    ds = D.LRHRDataset(root, "img", 16, 64, channels=1, max_value=4095)
    it = ds.get_raw(0)
    assert it["HR"].dtype == np.uint16 and it["HR"].shape == (64, 48, 1)
    assert np.array_equal(it["HR"][..., 0], hr) and np.array_equal(it["LR"][..., 0], lr)


def test_dataset_reads_mode_i_within_range_and_rejects_outside(tmp_path):
    from PIL import Image
    root = str(tmp_path / "i")
    a = np.arange(64 * 64, dtype=np.int32).reshape(64, 64) * 16
    for d, arr in (("hr_64", a), ("lr_16", a[:16, :16])):
        os.makedirs(os.path.join(root, d), exist_ok=True)
        Image.fromarray(arr).save(os.path.join(root, d, "a.tif"))
    ds = D.LRHRDataset(root, "img", 16, 64, channels=1, max_value=65535)
    assert np.array_equal(ds.get_raw(0)["HR"][..., 0], a.astype(np.uint16))
    Image.fromarray(a + 70000).save(os.path.join(root, "hr_64", "a.tif"))
    with pytest.raises(ValueError, match=r"a\.tif.*0\.\.65535"):
        ds.get_raw(0)


def _rejects(tmp_path, name, C, hr, kind, match):
    root = str(tmp_path / name)
    _pair(root, "bad", hr, hr[:16, :16], kind)
    with pytest.raises(ValueError, match=match):
        D.LRHRDataset(root, "img", 16, 64, channels=C, max_value=65535).get_raw(0)


def test_dataset_rejections_name_the_file(tmp_path):
    rng = np.random.default_rng(3)
    u8 = rng.integers(0, 256, (64, 64), dtype=np.uint8)
    u16 = rng.integers(0, 65536, (64, 64, 4), dtype=np.uint16)
    _rejects(tmp_path, "u8npy", 1, u8, "npy", r"bad\.npy.*uint16.*uint8")               # 8-bit array
    _rejects(tmp_path, "u8png", 1, u8, "png", r"bad\.png.*mode L")                       # 8-bit image
    _rejects(tmp_path, "rgb", 1, rng.integers(0, 256, (64, 64, 3), dtype=np.uint8), "png", r"bad\.png.*mode RGB")
    _rejects(tmp_path, "rgb3", 3, rng.integers(0, 256, (64, 64, 3), dtype=np.uint8), "png", r"bad\.png.*\.npy")
    _rejects(tmp_path, "f32", 4, u16.astype(np.float32), "npy", r"bad\.npy.*float32")    # other dtypes
    _rejects(tmp_path, "i32", 4, u16.astype(np.int32), "npy", r"bad\.npy.*int32")
    _rejects(tmp_path, "bands", 3, u16, "npy", r"bad\.npy.*\(H,W,3\) uint16")            # wrong band count
    _rejects(tmp_path, "i16img4", 4, u16[..., 0], "png", r"bad\.png.*\.npy")             # images serve C = 1 only


def test_dataset_max_value_arguments(tmp_path):
    with pytest.raises(ValueError, match="lmdb"):
        D.LRHRDataset("unused", "lmdb", 16, 64, kv={b"length": b"1"}, channels=1, max_value=4095)
    root = str(tmp_path / "ok")
    a = np.zeros((64, 64, 1), np.uint16)
    _pair(root, "a", a, a[:16, :16], "npy")
    for bad in (0, 65536, -1, 2.5, True):
        with pytest.raises(ValueError, match="1..65535"):
            D.LRHRDataset(root, "img", 16, 64, channels=1, max_value=bad)
    ds = D.create_dataset(F.dict_to_nonedict({"dataroot": root, "datatype": "img", "l_resolution": 16,
                                              "r_resolution": 64, "mode": "LRHR", "data_len": -1,
                                              "max_value": 1023}), "val", channels=1)
    assert ds.max_value == 1023
    with pytest.raises(ValueError, match="get_raw"):
        ds.get_u8(0)


def test_without_max_value_the_8bit_path_is_unchanged(tmp_path):
    """No max_value: uint8 files as before, and a 16-bit single-band image is still read through convert('L')."""
    from PIL import Image
    rng = np.random.default_rng(4)
    root = str(tmp_path / "u8")
    hr = rng.integers(0, 256, (64, 64), dtype=np.uint8)
    _pair(root, "a", hr, hr[:16, :16], "png")
    i16 = rng.integers(0, 65536, (64, 64), dtype=np.uint16)
    _pair(root, "b", i16, i16[:16, :16], "png")
    ds = D.LRHRDataset(root, "img", 16, 64, channels=1)
    assert ds.max_value is None
    it = ds.get_u8(0)
    assert it["HR"].dtype == np.uint8 and np.array_equal(it["HR"][..., 0], hr)
    assert np.array_equal(ds.get_raw(0)["HR"], it["HR"])
    with Image.open(os.path.join(root, "hr_64", "b.png")) as im:
        assert np.array_equal(ds.get_u8(1)["HR"][..., 0], np.asarray(im.convert("L")))
    assert torch.equal(ds[0]["HR"], D.u8_to_tensor(torch.from_numpy(it["HR"])[None])[0])
    batch = next(iter(D.BatchLoader(ds, 2, pin=False)))
    assert batch["HR"].dtype == torch.uint8
    np.save(os.path.join(root, "hr_64", "c.npy"), i16[..., None])           # a uint16 array stays an error
    np.save(os.path.join(root, "lr_16", "c.npy"), i16[:16, :16, None])
    with pytest.raises(ValueError, match="uint8"):
        D.LRHRDataset(root, "img", 16, 64, channels=1).get_u8(2)


# ------------------------------------------------------------------------------------------ normalisation
@pytest.mark.parametrize("M", M_LEVELS)
def test_normalise_then_quantise_is_the_identity(M):
    v = np.arange(0, 65536, dtype=np.uint16)
    t = D.u16_to_tensor(torch.from_numpy(v).view(1, 1, -1, 1), M)
    assert t.dtype == torch.float32 and t.shape == (1, 1, 1, 65536)
    assert np.array_equal(t.numpy().ravel(), R.u16_to_cond(v, M))
    q = R.quantise(t.numpy().ravel(), M)
    assert np.array_equal(q[:M + 1], np.arange(M + 1))
    assert (q[M + 1:] == M).all() and t.max().item() == 1.0 and t.min().item() == -1.0


# ------------------------------------------------------------------------------------------ writers
def test_save_u16_formats(tmp_path):
    from PIL import Image
    g = torch.Generator().manual_seed(0)
    for C, M in ((1, 65535), (1, 4095), (3, 65535), (4, 2047), (8, 10000)):
        img = torch.rand(C, 9, 7, generator=g) * 2.2 - 1.1
        want = R.quantise(img.permute(1, 2, 0).numpy(), M)
        for ext in ("png", "tif"):
            p = _save_u16(img, str(tmp_path / f"c{C}_{M}.{ext}"), M)
            if C == 1:
                assert p.endswith("." + ext)
                with Image.open(p) as im:
                    assert im.mode == "I;16" and im.size == (7, 9)
                    got = np.asarray(im).astype(np.int64)[..., None]
            else:
                assert p.endswith(".npy")
                got = np.load(p)
                assert got.dtype == np.uint16 and got.shape == (9, 7, C)
            assert np.array_equal(got, want), (C, M, ext)
    # the 8-bit writer is unchanged
    p = _save_u8(torch.zeros(1, 4, 4), str(tmp_path / "u8.tif"))
    with Image.open(p) as im:
        assert im.mode == "L"


# ------------------------------------------------------------------------------------------ entry scripts
def test_max_value_flag_reaches_the_dataset(tmp_path):
    root = str(tmp_path / "ds")
    a = np.zeros((256, 256, 3), np.uint16)
    for d, arr in (("hr_256", a), ("lr_64", a[:64, :64])):
        os.makedirs(os.path.join(root, d))
        np.save(os.path.join(root, d, "a.npy"), arr)
    args = parse_args(["-c", "sr_fastdiffsr_test_64_256", "--max-value", "4095"])
    opt = load_opt(args)
    assert opt["datasets"]["val"]["max_value"] == 4095
    opt["datasets"]["val"]["dataroot"] = root
    ds = D.create_dataset(opt["datasets"]["val"], "val", channels=3)
    assert ds.max_value == 4095 and ds.get_raw(0)["HR"].dtype == np.uint16
    plain = load_opt(parse_args(["-c", "sr_fastdiffsr_test_64_256"]))
    assert plain["datasets"]["val"].get("max_value") is None
    with pytest.raises(SystemExit):
        parse_args(["--max-value", "0"])


# ------------------------------------------------------------------------------------------ the restatement
def _pillow_i16(band, H, W):
    from PIL import Image
    im = Image.fromarray(band)
    assert im.mode == "I;16"
    return np.asarray(im.resize((W, H), Image.BICUBIC)).astype(np.uint16)


@pytest.mark.parametrize("shapes", [((12, 12), (48, 48)), ((13, 21), (26, 42)), ((5, 7), (40, 56)),
                                    ((13, 21), (50, 77)), ((19, 10), (40, 33)), ((7, 30), (61, 30)),
                                    ((40, 36), (17, 12))])
def test_restatement_equals_pillow_i16(shapes):
    (h, w), (H, W) = shapes
    rng = np.random.default_rng(h * 100 + W)
    cases = {"random": rng.integers(0, 65536, (h, w), dtype=np.uint16),
             "checker": (rng.integers(0, 2, (h, w)) * 65535).astype(np.uint16),
             "near0": rng.integers(0, 40, (h, w), dtype=np.uint16) * (rng.integers(0, 2, (h, w)) * 1000).astype(np.uint16)}
    for name, band in cases.items():
        assert np.array_equal(R.pil_bicubic_u16(band, H, W), _pillow_i16(band, H, W)), name


def test_checkerboard_overshoot_quirk():
    """Overshoot above 65535 is stored as 65280 + v % 256 by Pillow: a clamp would differ."""
    rng = np.random.default_rng(5)
    band = (rng.integers(0, 2, (12, 12)) * 65535).astype(np.uint16)
    ref = _pillow_i16(band, 48, 48)
    assert np.array_equal(R.pil_bicubic_u16(band, 48, 48), ref)
    assert ((ref >= 65280) & (ref < 65535)).sum() > 100      # the quirk is exercised
    assert np.array_equal(R.store_i16(np.array([-5, 0, 300, 65535, 65536, 65791, 70000])),
                          [0, 0, 300, 65535, 65280, 65535, 65280 + 70000 % 256])

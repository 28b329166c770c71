"""C-band imagery on the host side (no GPU): the state_dict surface of C-band UNets, the dataset's band-aware file
discovery and decoding, and the oracle's bicubic against Pillow band by band."""
import json
import os

import numpy as np
import pytest
import torch

import fastdiffsr_b200 as F
from fastdiffsr_b200 import data as D
from fastdiffsr_b200.config import default_config


def _opt(name, C):
    opt = json.loads(json.dumps(default_config(name)))
    opt["model"]["unet"]["in_channel"], opt["model"]["unet"]["out_channel"] = 2 * C, C
    return opt


@pytest.mark.parametrize("C", [1, 4, 8])
def test_state_dict_surface_of_band_configs(oracle, C):
    netG = F.define_G(_opt("sr_fastdiffsr_test_64_256", C))
    keys = [(k, tuple(v.shape)) for k, v in netG.denoise_fn.state_dict().items()]
    cfg = dict(oracle.DEFAULT_UNET, in_channel=2 * C, out_channel=C)
    assert [("denoise_fn." + k, s) for k, s in keys] == [(k, s) for k, s, _, _ in oracle.state_dict_spec(cfg)]
    assert dict(keys)["downs.0.weight"] == (64, 2 * C, 3, 3)
    sr3 = F.define_G(_opt("sr_ddpm_test_64_256", C))
    cfg3 = dict(oracle.SR3_UNET, in_channel=2 * C, out_channel=C)
    keys3 = [(k, tuple(v.shape)) for k, v in sr3.state_dict().items()]
    assert keys3 == [(k, s) for k, s, _, _ in oracle.sr3_state_dict_spec(cfg3, 256)]


def _write_pair(root, name, hr, lr, kind):
    from PIL import Image
    for d, a in (("hr_64", hr), ("lr_16", lr)):
        os.makedirs(os.path.join(root, d), exist_ok=True)
        if kind == "npy":
            np.save(os.path.join(root, d, name + ".npy"), a)
        else:
            Image.fromarray(a).save(os.path.join(root, d, name + "." + kind))


def test_dataset_reads_single_band_images_and_npy(tmp_path):
    rng = np.random.default_rng(0)
    root = str(tmp_path / "l")
    hr = rng.integers(0, 256, (4, 64, 64), dtype=np.uint8)
    lr = rng.integers(0, 256, (4, 16, 16), dtype=np.uint8)
    _write_pair(root, "a", hr[0], lr[0], "png")
    _write_pair(root, "b", hr[1], lr[1], "npy")                        # (H,W) allowed for one band
    _write_pair(root, "c", hr[2][..., None], lr[2][..., None], "npy")  # (H,W,1)
    _write_pair(root, "d", hr[3], lr[3], "tif")
    ds = D.LRHRDataset(root, "img", 16, 64, channels=1)
    assert len(ds) == 4
    for i in range(4):
        it = ds.get_u8(i)
        assert it["HR"].shape == (64, 64, 1) and it["LR"].shape == (16, 16, 1)
        assert np.array_equal(it["HR"][..., 0], hr[i]) and np.array_equal(it["LR"][..., 0], lr[i])
    assert ds[0]["HR"].shape == (1, 64, 64)
    # an RGB file in a single-band folder is read as its 'L' conversion
    from PIL import Image
    rgb = rng.integers(0, 256, (64, 64, 3), dtype=np.uint8)
    root2 = str(tmp_path / "rgb")
    _write_pair(root2, "a", rgb, rgb[:16, :16], "png")
    got = D.LRHRDataset(root2, "img", 16, 64, channels=1).get_u8(0)["HR"][..., 0]
    assert np.array_equal(got, np.asarray(Image.fromarray(rgb).convert("L")))


def test_dataset_reads_multiband_npy_and_rejects_images(tmp_path):
    rng = np.random.default_rng(1)
    root = str(tmp_path / "ms")
    hr = rng.integers(0, 256, (2, 64, 64, 5), dtype=np.uint8)
    for i in range(2):
        _write_pair(root, f"img{i}", hr[i], hr[i, :16, :16], "npy")
    ds = D.create_dataset(F.dict_to_nonedict({"dataroot": root, "datatype": "img", "l_resolution": 16,
                                              "r_resolution": 64, "mode": "LRHR", "data_len": -1}), "val", channels=5)
    assert len(ds) == 2 and np.array_equal(ds.get_u8(1)["HR"], hr[1])
    assert ds[0]["LR"].shape == (5, 16, 16)
    with pytest.raises(ValueError, match=r"\(H,W,4\) uint8"):                        # wrong band count in the file
        D.LRHRDataset(root, "img", 16, 64, channels=4).get_u8(0)
    img_root = str(tmp_path / "png")
    _write_pair(img_root, "a", hr[0, ..., :3], hr[0, :16, :16, :3], "png")
    with pytest.raises(ValueError, match=r"\.npy"):
        D.LRHRDataset(img_root, "img", 16, 64, channels=4)
    with pytest.raises(ValueError, match="1 or 3 bands"):
        D.LRHRDataset("unused", "lmdb", 16, 64, kv={}, channels=4)
    with pytest.raises(ValueError, match="1..8"):
        D.LRHRDataset(root, "img", 16, 64, channels=9)


def test_rgb_discovery_is_unchanged(tmp_path):
    """channels=3 keeps the reference's discovery: image files only (a stray .npy is not an image)."""
    rng = np.random.default_rng(2)
    root = str(tmp_path / "rgb")
    for i in range(2):
        a = rng.integers(0, 256, (64, 64, 3), dtype=np.uint8)
        _write_pair(root, f"img{i}", a, a[:16, :16], "png")
    np.save(os.path.join(root, "hr_64", "zz.npy"), np.zeros((64, 64, 3), np.uint8))
    paths = D.get_paths_from_images(os.path.join(root, "hr_64"))
    assert [os.path.basename(p) for p in paths] == ["img0.png", "img1.png"]
    assert D.get_paths_from_images(os.path.join(root, "hr_64"), 3) == paths
    ds = D.LRHRDataset(root, "img", 16, 64)
    assert ds.channels == 3 and ds.get_u8(0)["HR"].shape == (64, 64, 3)


@pytest.mark.parametrize("C", [1, 2, 4, 5, 8])
def test_oracle_bicubic_equals_pillow_per_band(oracle, C):
    from PIL import Image
    rng = np.random.default_rng(C)
    for (h, w), (H, W) in (((13, 21), (52, 84)), ((19, 10), (152, 80)), ((16, 16), (64, 64))):
        img = rng.integers(0, 256, (h, w, C), dtype=np.uint8)
        ref = np.stack([np.asarray(Image.fromarray(img[..., c]).resize((W, H), Image.BICUBIC)) for c in range(C)], 2)
        assert np.array_equal(oracle.pil_bicubic_u8(img, H, W), ref)


def test_save_u8_band_formats(tmp_path):
    from PIL import Image
    from fastdiffsr_b200.evaluate import _save_u8
    img = torch.rand(1, 8, 8) * 2 - 1
    p = _save_u8(img, str(tmp_path / "a.tif"))
    assert Image.open(p).mode == "L"
    p = _save_u8(torch.rand(4, 8, 8) * 2 - 1, str(tmp_path / "b.tif"))
    assert p.endswith("b.npy") and np.load(p).shape == (8, 8, 4)
    p = _save_u8(torch.rand(3, 8, 8) * 2 - 1, str(tmp_path / "c.png"))
    assert Image.open(p).mode == "RGB"

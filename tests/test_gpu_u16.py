"""16-bit imagery through the kernels, the C ABI and the drop-in (DESIGN.md §4.6): fdsr_bicubic_u16 against Pillow's
I;16 BICUBIC band by band, fdsr_metrics_u16 against a float64 restatement, and evaluate() / infer.py on 16-bit folders.
Needs a B200: `pytest -m gpu`."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

import fastdiffsr_b200 as F
from fastdiffsr_b200 import data as D

import u16_reference as R

pytestmark = pytest.mark.gpu


def unet_cfg(oracle, C):
    return dict(oracle.DEFAULT_UNET, in_channel=2 * C, out_channel=C)


@pytest.fixture(scope="module")
def engines(oracle):
    """engine(C): one context per band count; the resize and the metrics need no weights."""
    from fastdiffsr_b200 import Engine
    cache = {}

    def get(C):
        if C not in cache:
            cache[C] = Engine(unet_cfg(oracle, C), "cuda:0", "fp16")
        return cache[C]
    yield get
    for e in cache.values():
        e.close()


def _pillow(lr, H, W):
    """(h,w,C) uint16 -> (H,W,C) uint16: each band resized by Pillow as an I;16 image."""
    from PIL import Image
    out = []
    for c in range(lr.shape[2]):
        im = Image.fromarray(np.ascontiguousarray(lr[..., c]))
        assert im.mode == "I;16"
        out.append(np.asarray(im.resize((W, H), Image.BICUBIC)).astype(np.uint16))
    return np.stack(out, 2)


def _lr_cases(rng, B, h, w, C):
    return {"random": rng.integers(0, 65536, (B, h, w, C), dtype=np.uint16),
            "checker": (rng.integers(0, 2, (B, h, w, C)) * 65535).astype(np.uint16),
            "near0": (rng.integers(0, 40, (B, h, w, C)) * rng.integers(0, 2, (B, h, w, C)) * 1000).astype(np.uint16)}


SHAPES = [((13, 21), (52, 84)), ((12, 12), (48, 48)), ((5, 7), (40, 56)),        # x4, x4, x8
          ((13, 21), (50, 77)), ((19, 10), (40, 33)), ((7, 30), (61, 30)),       # non-integer ratios
          ((40, 36), (17, 12))]                                                  # downscale


# ------------------------------------------------------------------------------------------ resize
@pytest.mark.parametrize("C", [1, 3, 4, 8])
def test_bicubic_u16_vs_pillow_i16(engines, C):
    e = engines(C)
    rng = np.random.default_rng(C)
    for (h, w), (H, W) in SHAPES:
        for name, lr in _lr_cases(rng, 2, h, w, C).items():
            u16, cond = e.bicubic_u16(torch.from_numpy(lr).cuda(), H, W, 65535)
            assert u16.dtype == torch.uint16 and tuple(u16.shape) == (2, H, W, C)
            u16 = u16.cpu().numpy()
            ref = np.stack([_pillow(lr[b], H, W) for b in range(2)])
            assert np.array_equal(u16, ref), (C, h, w, H, W, name, int((u16 != ref).sum()))
            assert torch.equal(cond.cpu(), D.u16_to_tensor(torch.from_numpy(ref), 65535))
            if name == "checker" and H > h:
                assert ((ref >= 65280) & (ref < 65535)).any()     # the store quirk is exercised


@pytest.mark.parametrize("M", [65535, 4095, 10000])
def test_bicubic_u16_cond_at_white_level(engines, M):
    """cond = u16_to_tensor(Pillow's result, M) bit for bit, values above M included; u16_to_tensor gives the same
    bits on the device, and the u16 output is the raw resized levels whatever M is."""
    e = engines(4)
    rng = np.random.default_rng(M)
    for (h, w), (H, W) in SHAPES[:4] + SHAPES[-1:]:
        lr = rng.integers(0, 65536, (2, h, w, 4), dtype=np.uint16)
        ref = np.stack([_pillow(lr[b], H, W) for b in range(2)])
        assert (ref > M).any() or M == 65535
        u16, cond = e.bicubic_u16(torch.from_numpy(lr).cuda(), H, W, M)
        assert np.array_equal(u16.cpu().numpy(), ref)
        want = D.u16_to_tensor(torch.from_numpy(ref), M)
        assert torch.equal(cond.cpu(), want)
        assert np.array_equal(want.numpy(), R.u16_to_cond(ref, M).transpose(0, 3, 1, 2))
        assert torch.equal(D.u16_to_tensor(torch.from_numpy(ref).cuda(), M).cpu(), want)
        _, only = e.bicubic_u16(torch.from_numpy(lr).cuda(), H, W, M, want_u16=False)
        assert torch.equal(only, cond)


# ------------------------------------------------------------------------------------------ metrics
def _pair(C, seed):
    g = torch.Generator().manual_seed(seed)
    hr = torch.nn.functional.avg_pool2d(torch.rand(3, C, 39, 53, generator=g), 3, 1) * 2.4 - 1.2
    sr = hr + 0.15 * torch.randn(hr.shape, generator=g)
    return sr, hr


@pytest.mark.parametrize("M", [255, 4095, 65535])
@pytest.mark.parametrize("C", [1, 4, 8])
def test_metrics_u16_vs_restatement(engines, C, M):
    e = engines(C)
    sr, hr = _pair(C, C * 7 + M)
    m = e.metrics_u16(sr.cuda(), hr.cuda(), M, scale=4).cpu().numpy()
    for b in range(hr.shape[0]):
        qa = R.quantise(sr[b].permute(1, 2, 0).numpy(), M)
        qb = R.quantise(hr[b].permute(1, 2, 0).numpy(), M)
        mse, psnr, ssim, ergas = R.metrics(qa, qb, M, 4)
        assert m[b, 0] == mse
        assert m[b, 1] == pytest.approx(psnr, rel=1e-13)
        assert m[b, 2] == pytest.approx(ssim, abs=1e-9)
        assert m[b, 3] == pytest.approx(ergas, rel=1e-13)


@pytest.mark.parametrize("C", [1, 3, 8])
def test_metrics_u16_at_255_is_metrics_u8(engines, C):
    e = engines(C)
    sr, hr = _pair(C, 100 + C)
    a, b = sr.cuda(), hr.cuda()
    assert torch.equal(e.metrics_u16(a, b, 255, scale=4), e.metrics_u8(a, b, scale=4))
    assert torch.equal(e.metrics_u16(a, b, 255, scale=2), e.metrics_u8(a, b, scale=2))


# ------------------------------------------------------------------------------------------ validation
def test_argument_validation(engines):
    e = engines(4)
    lr = torch.zeros((1, 8, 8, 4), dtype=torch.uint16, device="cuda")
    for M in (0, -1, 65536):
        with pytest.raises(F.FdsrError, match="max_value must be 1..65535"):
            e.bicubic_u16(lr, 32, 32, M)
    with pytest.raises(F.FdsrError, match="both outputs are null"):
        e.bicubic_u16(lr, 32, 32, 4095, want_u16=False, want_cond=False)
    with pytest.raises(F.FdsrError, match=">= 1"):
        e.bicubic_u16(lr, 0, 32, 4095)
    with pytest.raises(F.FdsrError, match=">= 1"):
        e.bicubic_u16(torch.zeros((0, 8, 8, 4), dtype=torch.uint16, device="cuda"), 32, 32, 4095)
    with pytest.raises(F.FdsrError, match="uint16"):
        e.bicubic_u16(lr.to(torch.int32), 32, 32, 4095)
    null = ctypes.c_void_p(0)
    out = torch.empty((1, 4, 32, 32), device="cuda")
    with pytest.raises(F.FdsrError, match="null argument"):
        e._call("fdsr_bicubic_u16", null, 1, 8, 8, 32, 32, 4095, null, ctypes.c_void_p(out.data_ptr()), null)
    a = torch.zeros((1, 4, 16, 16), device="cuda")
    for M in (0, 65536):
        with pytest.raises(F.FdsrError, match="max_value must be 1..65535"):
            e.metrics_u16(a, a, M)
    res = torch.empty((1, 4), dtype=torch.float64, device="cuda")
    with pytest.raises(F.FdsrError, match="null argument"):
        e._call("fdsr_metrics_u16", null, ctypes.c_void_p(a.data_ptr()), 1, 16, 16, 4095, 4.0,
                ctypes.c_void_p(res.data_ptr()), null)
    with pytest.raises(F.FdsrError, match=">= 1"):
        e._call("fdsr_metrics_u16", ctypes.c_void_p(a.data_ptr()), ctypes.c_void_p(a.data_ptr()), 1, 0, 16, 4095, 4.0,
                ctypes.c_void_p(res.data_ptr()), null)


# ------------------------------------------------------------------------------------------ evaluate and infer.py
def _opt(C, config=None):
    opt = json.loads(json.dumps(F.config.default_config(*([config] if config else []))))
    opt["model"]["unet"]["in_channel"], opt["model"]["unet"]["out_channel"] = 2 * C, C
    return opt


def _net(C):
    opt = _opt(C)
    torch.manual_seed(0)
    netG = F.define_G(opt).to("cuda")
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cuda")
    return netG.eval()


def _save(path, a, C):
    from PIL import Image
    if C == 1:
        Image.fromarray(np.ascontiguousarray(a[..., 0])).save(path + ".png")
    else:
        np.save(path + ".npy", a)


def _u16_dataset(root, C, M, n=3, l=16, r=64, with_sr=False):
    rng = np.random.default_rng(C * 11 + M)
    dirs = [f"hr_{r}", f"lr_{l}"] + ([f"sr_{l}_{r}"] if with_sr else [])
    for d in dirs:
        os.makedirs(os.path.join(root, d), exist_ok=True)
    hrs, lrs = [], []
    for i in range(n):
        hr = rng.integers(0, 65536, (r, r, C), dtype=np.uint16)
        hr = np.minimum(hr, min(M + M // 8, 65535)).astype(np.uint16)  # some levels above the white level
        lr = _pillow(hr, l, l)
        _save(os.path.join(root, f"hr_{r}", f"img{i}"), hr, C)
        _save(os.path.join(root, f"lr_{l}", f"img{i}"), lr, C)
        if with_sr:
            _save(os.path.join(root, f"sr_{l}_{r}", f"img{i}"), _pillow(lr, r, r), C)
        hrs.append(hr)
        lrs.append(lr)
    return hrs, lrs


def _read_sr(path, C):
    from PIL import Image
    if C == 1:
        with Image.open(path + ".tif") as im:
            assert im.mode == "I;16"
            return np.asarray(im).astype(np.uint16)[..., None]
    a = np.load(path + ".npy")
    assert a.dtype == np.uint16
    return a


@pytest.mark.parametrize("C,M", [(4, 4095), (1, 65535)])
def test_evaluate_u16_folders(tmp_path, C, M):
    from fastdiffsr_b200.evaluate import evaluate
    netG = _net(C)
    hrs, lrs = _u16_dataset(str(tmp_path / "ds"), C, M)
    ds = D.LRHRDataset(str(tmp_path / "ds"), "img", 16, 64, channels=C, max_value=M)
    res = evaluate(netG, ds, batch_size=2, scale=4, result_path=str(tmp_path / "res"), seed=3)
    assert res["n"] == 3
    assert set(res) == {"n", "seconds", "images_per_s"} | {p + k for p in ("bic_", "sr_")
                                                           for k in ("mse", "psnr", "ssim", "ergas")}
    # the SR is super_resolution(cond) with cond built from Pillow's I;16 resize, saved at M
    bic, srm = [], []
    for i0, idx in ((0, [0, 1]), (2, [2])):
        up = np.stack([_pillow(lrs[i], 64, 64) for i in idx])
        cond = D.u16_to_tensor(torch.from_numpy(up), M).cuda()
        sr = netG.super_resolution(cond, False, seed=3, image_offset=i0)
        for j, i in enumerate(idx):
            got = _read_sr(str(tmp_path / "res" / f"0_{i + 1}_sr"), C)
            assert np.array_equal(got, R.quantise(sr[j].permute(1, 2, 0).cpu().numpy(), M)), i
            hq = np.minimum(hrs[i], M).astype(np.int64)
            srm.append(R.metrics(got.astype(np.int64), hq, M, 4))
            bic.append(R.metrics(np.minimum(up[j], M).astype(np.int64), hq, M, 4))
    for pre, vals in (("bic_", bic), ("sr_", srm)):
        mean = np.mean(np.array(vals), axis=0)
        for k, name in enumerate(("mse", "psnr", "ssim", "ergas")):
            assert res[pre + name] == pytest.approx(mean[k], rel=1e-12, abs=1e-9), pre + name
    # an sr_ folder written by Pillow gives the result of rebuilding the conditioning from lr_
    _u16_dataset(str(tmp_path / "ds_sr"), C, M, with_sr=True)
    ds_sr = D.LRHRDataset(str(tmp_path / "ds_sr"), "img", 16, 64, channels=C, max_value=M)
    assert "SR" in ds_sr.get_raw(0)
    res_sr = evaluate(netG, ds_sr, batch_size=2, scale=4, result_path=str(tmp_path / "res_sr"), seed=3)
    for k in res:
        if k not in ("seconds", "images_per_s"):
            assert res_sr[k] == res[k], k
    for i in range(3):
        assert np.array_equal(_read_sr(str(tmp_path / "res_sr" / f"0_{i + 1}_sr"), C),
                              _read_sr(str(tmp_path / "res" / f"0_{i + 1}_sr"), C))


def test_infer_script_u16_tiled(tmp_path):
    """infer.py --tile 64 --max-value 4095 on single-band I;16 scenes whose sizes are not multiples of 8; --tile-split
    (one rank here) gives the same images."""
    from PIL import Image
    from fastdiffsr_b200.evaluate import main
    root = tmp_path / "ds"
    rng = np.random.default_rng(1)
    sizes = [(13, 21), (19, 10)]
    for d in ("hr_512", "lr_128"):
        os.makedirs(root / d)
    for i, (h, w) in enumerate(sizes):
        hr = np.minimum(rng.integers(0, 5000, (4 * h, 4 * w)), 65535).astype(np.uint16)
        Image.fromarray(hr).save(root / "hr_512" / f"img{i}.png")
        Image.fromarray(_pillow(hr[..., None], h, w)[..., 0]).save(root / "lr_128" / f"img{i}.png")
    opt = _opt(1, "sr_fastdiffsr_infer_x4")
    opt["datasets"]["val"]["dataroot"] = str(root)
    outs = {}
    for split in (False, True):
        out = tmp_path / f"results_{split}"
        opt["path"] = {"results": str(out), "log": None, "resume_state": None}
        cfg = tmp_path / "cfg.json"
        cfg.write_text(json.dumps(opt))
        argv = ["-c", str(cfg), "--tile", "64", "--tile-overlap", "16", "--tile-batch", "4", "--max-value", "4095"]
        torch.manual_seed(0)                                   # the same random-init network for both runs
        res = main(argv + (["--tile-split"] if split else []), default_config=str(cfg), prog="infer.py")
        assert res["n"] == 2 and all(np.isfinite(res[k]) for k in res if k != "n")
        imgs = []
        for i, (h, w) in enumerate(sizes):
            with Image.open(out / f"0_{i + 1}_sr.png") as im:
                assert im.mode == "I;16" and im.size == (4 * w, 4 * h)
                a = np.asarray(im).astype(np.uint16)
            assert a.max() <= 4095
            imgs.append(a)
        outs[split] = (res, imgs)
    (r0, i0), (r1, i1) = outs[False], outs[True]
    assert all(np.array_equal(a, b) for a, b in zip(i0, i1))
    assert all(r0[k] == r1[k] for k in r0 if k not in ("seconds", "images_per_s"))

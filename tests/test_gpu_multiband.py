"""Imagery of C = 1..8 bands (out_channel = C, in_channel = 2C) through the kernels, the C ABI and the drop-in, against
the oracle (whose UNet, sampler, bicubic and metrics take any channel count).  Needs a B200: `pytest -m gpu`.
Tolerances are the project's: eps relative L2 <= 1e-4 in the fp32 mode and <= 1e-2 in the 16-bit modes; a 20-step sample
within 1e-2 relative L2 and 0.05 dB PSNR of the oracle's."""
import json
import os

import numpy as np
import pytest
import torch

import fastdiffsr_b200 as F
from fastdiffsr_b200 import data as D

pytestmark = pytest.mark.gpu

B, H, W = 2, 64, 96           # non-square, B > 1
EPS_TOL = {"fp32": 1e-4, "fp16": 1e-2, "bf16": 1e-2}


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def unet_cfg(oracle, C, base=None):
    return dict(base if base is not None else oracle.DEFAULT_UNET, in_channel=2 * C, out_channel=C)


@pytest.fixture(scope="module")
def engines(oracle, schedule):
    """engine(C, dtype): one context per (C, dtype) on oracle.make_state_dict of the C-band config."""
    from fastdiffsr_b200 import Engine
    cache = {}

    def get(C, dtype="fp16"):
        if (C, dtype) not in cache:
            cfg = unet_cfg(oracle, C)
            e = Engine(cfg, "cuda:0", dtype)
            e.load_state_dict(oracle.make_state_dict(cfg, seed=C, gn_jitter=0.1))
            e.set_schedule(schedule["betas"])
            cache[(C, dtype)] = e
        return cache[(C, dtype)]
    yield get
    for e in cache.values():
        e.close()


def _inputs(C, seed):
    g = torch.Generator().manual_seed(seed)
    cond = torch.rand(B, C, H, W, generator=g) * 2 - 1
    noises = torch.randn(20, B, C, H, W, generator=g)
    return cond, noises


# ------------------------------------------------------------------------------------------ configuration rule
def test_create_rejects_unsupported_channel_configs(oracle):
    from fastdiffsr_b200 import Engine
    for cin, cout in ((5, 3), (0, 0), (18, 9), (4, 3), (8, 3)):
        with pytest.raises(F.FdsrError, match=r"in_channel must be 2 \* out_channel"):
            Engine(dict(oracle.DEFAULT_UNET, in_channel=cin, out_channel=cout), "cuda:0", "fp16")


def test_posterior_step_rejects_numel_not_multiple_of_C(engines):
    e = engines(4)
    x = torch.zeros(6, device="cuda")
    with pytest.raises(F.FdsrError, match="multiple of 4"):
        e.posterior_step(x, x, x, 5)
    with pytest.raises(F.FdsrError):
        e.unet_forward(torch.zeros(1, 3, 64, 64, device="cuda"), torch.zeros(1, 3, 64, 64, device="cuda"), 3)


# ------------------------------------------------------------------------------------------ network and sampler
@pytest.mark.parametrize("dtype", ["fp32", "fp16", "bf16"])
@pytest.mark.parametrize("C", [1, 4, 8])
def test_eps_vs_oracle(oracle, schedule, engines, C, dtype):
    cfg = unet_cfg(oracle, C)
    sd = oracle.make_state_dict(cfg, seed=C, gn_jitter=0.1)
    cond, noises = _inputs(C, 10 + C)
    t = 11
    nl = torch.full((B, 1), float(np.float32(schedule["sqrt_alphas_cumprod_prev"][t + 1])))
    ref = oracle.unet_forward(sd, cfg, torch.cat([cond, noises[0]], 1), nl)
    eps = engines(C, dtype).unet_forward(cond.cuda(), noises[0].cuda(), t).cpu()
    r = rel_l2(eps, ref)
    print(f"C={C} [{dtype}] eps rel-L2 {r:.3e}")
    assert eps.shape == (B, C, H, W) and r <= EPS_TOL[dtype]


@pytest.mark.parametrize("dtype", ["fp32", "fp16"])
def test_sr3_eps_vs_oracle_single_band(oracle, dtype):
    from fastdiffsr_b200 import Engine
    cfg = unet_cfg(oracle, 1, oracle.SR3_UNET)
    sd = oracle.make_state_dict(cfg, seed=3, gn_jitter=0.2, spec=oracle.sr3_state_dict_spec(cfg, 64))
    e = Engine(dict(cfg, model="ddpm", image_size=64), "cuda:0", dtype)
    e.load_state_dict(sd)
    e.set_schedule(oracle.make_beta_schedule(**oracle.SR3_SCHEDULE))
    cond, noises = _inputs(1, 31)
    t = 400
    ref = oracle.sr3_unet_forward(sd, cfg, torch.cat([cond, noises[0]], 1), torch.full((B,), t), image_size=64)
    eps = e.unet_forward(cond.cuda(), noises[0].cuda(), t).cpu()
    e.close()
    r = rel_l2(eps, ref)
    print(f"SR3 C=1 [{dtype}] eps rel-L2 {r:.3e}")
    assert r <= EPS_TOL[dtype]


@pytest.fixture(scope="module")
def sampled(oracle, schedule):
    """Oracle 20-step samples (continous=True) with injected noise, per C."""
    cache = {}

    def get(C):
        if C not in cache:
            cfg = unet_cfg(oracle, C)
            sd = oracle.make_state_dict(cfg, seed=C, gn_jitter=0.1)
            cond, noises = _inputs(C, 20 + C)
            seq = oracle.sample_loop(sd, cfg, schedule, cond, noises, continous=True)
            cache[C] = (cond, noises, seq)
        return cache[C]
    return get


@pytest.mark.parametrize("dtype", ["fp32", "fp16", "bf16"])
@pytest.mark.parametrize("C", [1, 4, 8])
def test_sampler_vs_oracle(oracle, engines, sampled, C, dtype):
    cond, noises, seq = sampled(C)
    e = engines(C, dtype)
    sr, tr = e.sample(cond.cuda(), noise=noises.cuda(), trace=True)
    e.check_overflow()
    sr, tr = sr.cpu(), tr.cpu()
    nfr = e.trace_frames()
    ref_tr = seq.view(B, nfr, C, H, W)
    ref = ref_tr[:, -1]
    assert tr.shape == (B, nfr, C, H, W) and torch.equal(tr[:, -1], sr)
    r, r_tr = rel_l2(sr, ref), rel_l2(tr, ref_tr)
    print(f"C={C} [{dtype}] 20-step SR rel-L2 {r:.3e}, trace {r_tr:.3e}")
    if dtype == "fp32":
        assert r <= 1e-4 and r_tr <= 1e-4
        return
    assert r <= 1e-2 and r_tr <= 1e-2
    g = torch.Generator().manual_seed(9)
    hr = (cond + 0.1 * torch.nn.functional.avg_pool2d(torch.randn(B, C, H, W, generator=g), 3, 1, 1)).clamp(-1, 1)
    for b in range(B):
        p_ours = oracle.psnr_u8(oracle.to_u8(sr[b]), oracle.to_u8(hr[b]))
        p_ref = oracle.psnr_u8(oracle.to_u8(ref[b]), oracle.to_u8(hr[b]))
        assert abs(p_ours - p_ref) <= 0.05, (b, p_ours, p_ref)


@pytest.mark.parametrize("C", [1, 4, 8])
def test_fused_tail_equals_unfused(oracle, schedule, engines, C):
    """The final conv's posterior epilogue (one 8-byte store for C <= 4, one 16-byte store for C > 4) against the
    separate pack / eps / posterior kernels, with built-in and with injected noise."""
    from fastdiffsr_b200 import Engine
    cfg = unet_cfg(oracle, C)
    os.environ["FDSR_FUSED_TAIL"] = "0"
    try:
        u = Engine(cfg, "cuda:0", "fp16")
    finally:
        os.environ.pop("FDSR_FUSED_TAIL", None)
    u.load_state_dict(oracle.make_state_dict(cfg, seed=C, gn_jitter=0.1))
    u.set_schedule(schedule["betas"])
    f = engines(C, "fp16")
    cond, noises = _inputs(C, 40 + C)
    cond, noises = cond.cuda(), noises.cuda()
    assert torch.equal(f.sample(cond, seed=5, image_offset=3), u.sample(cond, seed=5, image_offset=3))
    assert torch.equal(f.sample(cond, noise=noises), u.sample(cond, noise=noises))
    u.close()


# ------------------------------------------------------------------------------------------ built-in noise
def test_builtin_noise_bands(engines):
    """Bands 0-2 are the 3-band draws whatever C is; every band of C = 8 is N(0,1) and independent of the others."""
    from scipy import stats
    e8, e3 = engines(8), engines(3)
    a = e8.debug_noise(2, 256, 256, seed=1234, stream_id=20, image_offset=7)
    assert torch.equal(a[:, :3], e3.debug_noise(2, 256, 256, seed=1234, stream_id=20, image_offset=7))
    assert torch.equal(a[:, :4], engines(4).debug_noise(2, 256, 256, seed=1234, stream_id=20, image_offset=7))
    v = a.cpu().double().numpy()
    n = v[:, 0].size
    for c in range(8):
        f = v[:, c].ravel()
        assert abs(f.mean()) < 5.0 / np.sqrt(n), c
        assert abs(f.var() - 1.0) < 5.0 * np.sqrt(2.0 / n), c
        assert abs(stats.skew(f)) < 5.0 * np.sqrt(6.0 / n), c
        assert abs(stats.kurtosis(f)) < 5.0 * np.sqrt(24.0 / n), c
        assert stats.kstest(f[:200000], "norm").pvalue > 1e-3, c
    bound = 5.0 / np.sqrt(n)
    for i in range(8):
        for j in range(i + 1, 8):
            cc = float(np.corrcoef(v[:, i].ravel(), v[:, j].ravel())[0, 1])
            assert abs(cc) < 2 * bound, (i, j, cc)


@pytest.mark.parametrize("C", [1, 4, 8])
def test_builtin_noise_equals_injected_and_shards(engines, C):
    e = engines(C)
    cond, _ = _inputs(C, 50 + C)
    cond = cond.cuda()
    T, seed, off = 20, 77, 5
    noises = torch.stack([e.debug_noise(B, H, W, seed, T, image_offset=off)] +
                         [e.debug_noise(B, H, W, seed, t, image_offset=off) for t in range(T - 1, 0, -1)]).contiguous()
    full = e.sample(cond, seed=seed, image_offset=off)
    assert torch.equal(full, e.sample(cond, noise=noises))
    lo = e.sample(cond[:1].contiguous(), seed=seed, image_offset=off)
    hi = e.sample(cond[1:].contiguous(), seed=seed, image_offset=off + 1)
    assert torch.equal(torch.cat([lo, hi]), full)


# ------------------------------------------------------------------------------------------ bicubic and metrics
@pytest.mark.parametrize("C", [1, 2, 4, 5, 8])
def test_bicubic_u8_vs_pillow_per_band(oracle, C):
    from PIL import Image
    from fastdiffsr_b200 import Engine
    e = Engine(unet_cfg(oracle, C), "cuda:0", "fp16")     # the resize needs no weights
    rng = np.random.default_rng(C)
    for (h, w), s in (((13, 21), 4), ((19, 10), 8), ((16, 16), 4)):
        lr = rng.integers(0, 256, (2, h, w, C), dtype=np.uint8)
        u8, cond = e.bicubic_u8(torch.from_numpy(lr).cuda(), s * h, s * w)
        u8, cond = u8.cpu().numpy(), cond.cpu()
        for b in range(2):
            ref = np.stack([np.asarray(Image.fromarray(lr[b, :, :, c]).resize((s * w, s * h), Image.BICUBIC))
                            for c in range(C)], axis=2)
            assert np.array_equal(u8[b], ref), (C, h, w, s, b)
        assert torch.equal(cond, D.u8_to_tensor(torch.from_numpy(u8)))
    e.close()


@pytest.mark.parametrize("C", [1, 4, 8])
def test_metrics_u8_vs_oracle(oracle, engines, C):
    e = engines(C)
    g = torch.Generator().manual_seed(C)
    hr = torch.nn.functional.avg_pool2d(torch.rand(3, C, 39, 53, generator=g), 3, 1) * 2.4 - 1.2
    sr = hr + 0.15 * torch.randn(hr.shape, generator=g)
    m = e.metrics_u8(sr.cuda(), hr.cuda(), scale=4).cpu().numpy()
    sse = e.sse_u8(sr.cuda(), hr.cuda()).cpu().numpy()
    for b in range(hr.shape[0]):
        a8, b8 = oracle.to_u8(sr[b]), oracle.to_u8(hr[b])
        assert a8.shape[2] == C
        assert m[b, 0] == oracle.mse_u8(a8, b8)
        assert sse[b] == oracle.mse_u8(a8, b8) * a8.size
        assert m[b, 1] == pytest.approx(oracle.psnr_u8(a8, b8), rel=1e-13)
        assert m[b, 2] == pytest.approx(oracle.ssim_u8(a8, b8), abs=1e-9)
        assert m[b, 3] == pytest.approx(oracle.ergas_u8(a8, b8, 4), rel=1e-13)


# ------------------------------------------------------------------------------------------ tiled sampling
@pytest.mark.parametrize("C", [1, 8])
def test_tiled_multiband(engines, C):
    e = engines(C)
    g = torch.Generator().manual_seed(60 + C)
    one = (torch.rand(1, C, 64, 64, generator=g) * 2 - 1).cuda()
    assert torch.equal(e.sample_tiled(one, 64, overlap=16, seed=3), e.sample(one, seed=3))
    canvas = (torch.rand(1, C, 64, 128, generator=g) * 2 - 1).cuda()
    noise = torch.randn(20, 1, C, 64, 128, generator=g).cuda()
    tiled = e.sample_tiled(canvas, 64, overlap=0, noise=noise)
    for x0 in (0, 64):
        crop = e.sample(canvas[..., x0:x0 + 64].contiguous(), noise=noise[..., x0:x0 + 64].contiguous())
        assert torch.equal(tiled[..., x0:x0 + 64], crop)
    big = (torch.rand(1, C, 100, 140, generator=g) * 2 - 1).cuda()
    ref = e.sample_tiled(big, 64, overlap=16, tile_batch=16, seed=8)
    assert ref.shape == (1, C, 100, 140)
    assert torch.equal(e.sample_tiled(big, 64, overlap=16, tile_batch=2, seed=8), ref)


# ------------------------------------------------------------------------------------------ drop-in and drivers
def _opt(C, config=None):
    opt = json.loads(json.dumps(F.config.default_config(*([config] if config else []))))
    opt["model"]["unet"]["in_channel"], opt["model"]["unet"]["out_channel"] = 2 * C, C
    return opt


def test_define_G_four_bands():
    opt = _opt(4)
    torch.manual_seed(0)
    netG = F.define_G(opt).to("cuda")
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cuda")
    cond = (torch.rand(2, 4, 64, 64) * 2 - 1).cuda()
    assert netG.super_resolution(cond, False, seed=1).shape == (2, 4, 64, 64)
    seq = netG.super_resolution(cond[:1], True, seed=1)
    assert seq.shape == (netG.engine().trace_frames(), 4, 64, 64)
    eps = netG.denoise(torch.cat([cond, cond], 1), 3)
    assert torch.equal(eps, netG.engine().unet_forward(cond, cond, 3))


def _band_dataset(root, C, n=3, l=16, r=64):
    from PIL import Image
    rng = np.random.default_rng(C)
    for d in (f"hr_{r}", f"lr_{l}"):
        os.makedirs(os.path.join(root, d), exist_ok=True)
    for i in range(n):
        hr = rng.integers(0, 256, (r, r, C), dtype=np.uint8)
        lr = np.stack([np.asarray(Image.fromarray(hr[..., c]).resize((l, l), Image.BICUBIC)) for c in range(C)], 2)
        if C == 1:
            Image.fromarray(hr[..., 0]).save(os.path.join(root, f"hr_{r}", f"img{i}.png"))
            Image.fromarray(lr[..., 0]).save(os.path.join(root, f"lr_{l}", f"img{i}.png"))
        else:
            np.save(os.path.join(root, f"hr_{r}", f"img{i}.npy"), hr)
            np.save(os.path.join(root, f"lr_{l}", f"img{i}.npy"), lr)
    return root


@pytest.mark.parametrize("C", [1, 4])
def test_evaluate_band_folders(tmp_path, C):
    from PIL import Image
    from fastdiffsr_b200.evaluate import evaluate
    opt = _opt(C)
    torch.manual_seed(0)
    netG = F.define_G(opt).to("cuda")
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cuda")
    ds = D.LRHRDataset(_band_dataset(str(tmp_path / "ds"), C), "img", 16, 64, channels=C)
    out = tmp_path / "res"
    res = evaluate(netG.eval(), ds, batch_size=2, scale=4, result_path=str(out), seed=3)
    assert res["n"] == 3 and all(np.isfinite(res[k]) for k in res if k != "n")
    files = sorted(os.listdir(out))
    if C == 1:
        assert files == [f"0_{i}_sr.tif" for i in range(1, 4)]
        im = Image.open(out / files[0])
        assert im.mode == "L" and im.size == (64, 64)
    else:
        assert files == [f"0_{i}_sr.npy" for i in range(1, 4)]
        a = np.load(out / files[0])
        assert a.dtype == np.uint8 and a.shape == (64, 64, 4)


def test_infer_script_single_band_tiled(tmp_path):
    from PIL import Image
    from fastdiffsr_b200.evaluate import main
    root = tmp_path / "ds"
    rng = np.random.default_rng(1)
    sizes = [(13, 21), (19, 10)]
    for d in ("hr_512", "lr_128"):
        os.makedirs(root / d)
    for i, (h, w) in enumerate(sizes):
        hr = Image.fromarray(rng.integers(0, 256, (4 * h, 4 * w), dtype=np.uint8))
        hr.save(root / "hr_512" / f"img{i}.png")
        hr.resize((w, h), Image.BICUBIC).save(root / "lr_128" / f"img{i}.png")
    opt = _opt(1, "sr_fastdiffsr_infer_x4")
    opt["datasets"]["val"]["dataroot"] = str(root)
    opt["path"] = {"results": str(tmp_path / "results"), "log": None, "resume_state": None}
    cfg = tmp_path / "cfg.json"
    cfg.write_text(json.dumps(opt))
    res = main(["-c", str(cfg), "--tile", "64", "--tile-overlap", "16", "--tile-batch", "4"],
               default_config=str(cfg), prog="infer.py")
    assert res["n"] == 2 and all(np.isfinite(res[k]) for k in res if k != "n")
    for i, (h, w) in enumerate(sizes):
        im = Image.open(tmp_path / "results" / f"0_{i + 1}_sr.png")
        assert im.mode == "L" and im.size == (4 * w, 4 * h)

"""SR3 baseline (which_model_G = "ddpm", SURVEY 8(f) N3) on the CUDA path, through the C ABI, against the
reference's own outputs (tests/golden/sr3_*.npz, written by oracle/make_golden.py from the real reference) and
against the oracle.  Needs a B200: run with `pytest -m gpu`.

Tolerances: per-step epsilon relative L2 <= 1e-2 in the 16-bit mode, <= 1e-4 in fp32 mode; attention core
(tensor cores) vs the same engine with the CUDA-core core <= 3e-3 on the attention output."""
import json
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

DTYPE = "fp16"      # the layer / attention / sampler tests; the epsilon parity test runs both 16-bit modes in one pytest run
EPS_TOL = 1e-2      # north-star bar for fp16 AND bf16 (bf16 = bf16 storage, fp16 post-GroupNorm operands)
LAYER_TOL = 5e-3


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def make_engine(oracle, image_size, betas, dtype=DTYPE, attn_ref=False):
    from fastdiffsr_b200 import Engine
    cfg = dict(oracle.SR3_UNET)
    sd = oracle.make_state_dict(cfg, seed=3, gn_jitter=0.2, spec=oracle.sr3_state_dict_spec(cfg, image_size))
    if attn_ref:
        os.environ["FDSR_ATTN_REF"] = "1"
    try:
        eng = Engine(dict(cfg, model="ddpm", image_size=image_size), "cuda:0", dtype)
    finally:
        os.environ.pop("FDSR_ATTN_REF", None)
    eng.load_state_dict(sd)
    eng.set_schedule(betas)
    return cfg, sd, eng


@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
@pytest.mark.parametrize("image_size", [256, 64])
def test_sr3_eps_vs_reference_golden(oracle, golden, image_size, dtype):
    """UNet forward at two integer steps of the shipped T = 1000 linear schedule (the UNet sees t only); the fixture
    holds the reference's eps at the image rows `rows`."""
    g = golden(f"sr3_{image_size}")
    betas = oracle.make_beta_schedule(**oracle.SR3_SCHEDULE)
    _, _, eng = make_engine(oracle, image_size, betas, dtype=dtype)
    x6 = torch.from_numpy(g["x6"]).cuda()
    for i, t in enumerate(g["steps"]):
        eps = eng.unet_forward(x6[:, :3].contiguous(), x6[:, 3:].contiguous(), int(t)).cpu()
        r = rel_l2(eps[..., g["rows"], :], torch.from_numpy(g["eps"][i]))
        print(f"sr3[{dtype}, image_size={image_size}] t={int(t)}: eps rel-L2 vs reference = {r:.3e}")
        assert r <= EPS_TOL


def test_sr3_eps_fp32_mode(oracle, golden):
    g = golden("sr3_64")
    betas = oracle.make_beta_schedule(**oracle.SR3_SCHEDULE)
    _, _, eng = make_engine(oracle, 64, betas, dtype="fp32")
    x6 = torch.from_numpy(g["x6"]).cuda()
    for i, t in enumerate(g["steps"]):
        eps = eng.unet_forward(x6[:, :3].contiguous(), x6[:, 3:].contiguous(), int(t)).cpu()
        r = rel_l2(eps[..., g["rows"], :], torch.from_numpy(g["eps"][i]))
        print(f"sr3 fp32 mode t={int(t)}: eps rel-L2 vs reference = {r:.3e}")
        assert r <= 1e-4


def test_sr3_every_layer_vs_oracle(oracle):
    """Non-square input, 3 images, attention over 16x24 = 384 tokens (C = 128) and a 2x3 mid block."""
    image_size = 64
    betas = oracle.make_beta_schedule(schedule="linear", n_timestep=20, linear_start=1e-4, linear_end=0.2)
    cfg, sd, eng = make_engine(oracle, image_size, betas)
    gen = torch.Generator().manual_seed(5)
    B, H, W = 3, 64, 96
    cond = torch.rand(B, 3, H, W, generator=gen) * 2 - 1
    x = torch.randn(B, 3, H, W, generator=gen)
    taps = {}
    t = 13
    eps_ref = oracle.sr3_unet_forward(sd, cfg, torch.cat([cond, x], 1), torch.full((B,), t, dtype=torch.long),
                                      image_size, taps=taps)
    eps = eng.unet_forward(cond.cuda(), x.cuda(), t).cpu()
    n = 0
    for name in eng.tensor_names():
        if name in taps:
            got = eng.read_tensor(name, B, taps[name].numel()).cpu()
            assert got.shape == taps[name].shape
            r = rel_l2(got, taps[name])
            assert r <= LAYER_TOL, (name, r)
            n += 1
    assert n > 60
    assert rel_l2(eps, eps_ref) <= EPS_TOL


@pytest.mark.parametrize("image_size,H", [(64, 128), (256, 256)])
def test_sr3_tensor_core_attention_vs_cuda_core_attention(oracle, image_size, H):
    """Same engine twice: tcgen05 attention core vs the one-warp-per-query CUDA-core core.
    (64, 128): 32x32 = 1024 tokens, C = 128 (16 key blocks, two-pass softmax); (256, 256): 256 tokens, C = 256."""
    betas = oracle.make_beta_schedule(schedule="linear", n_timestep=20, linear_start=1e-4, linear_end=0.2)
    _, _, e_tc = make_engine(oracle, image_size, betas)
    _, _, e_ref = make_engine(oracle, image_size, betas, attn_ref=True)
    gen = torch.Generator().manual_seed(8)
    B = 2
    cond = (torch.rand(B, 3, H, H, generator=gen) * 2 - 1).cuda()
    x = torch.randn(B, 3, H, H, generator=gen).cuda()
    a = e_tc.unet_forward(cond, x, 5)
    b = e_ref.unet_forward(cond, x, 5)
    names = [n for n in e_tc.tensor_names() if n.endswith(".attn.o")]
    assert len(names) == 6
    for n in names:
        ta = e_tc.read_tensor(n, B, B * 256 * H * H).cpu()
        tb = e_ref.read_tensor(n, B, B * 256 * H * H).cpu()
        r = rel_l2(ta, tb)
        assert r <= 3e-3, (n, r)
    assert rel_l2(a.cpu(), b.cpu()) <= 3e-3


@pytest.mark.parametrize("image_size", [256, 64])
def test_sr3_sampler_vs_reference_golden(oracle, golden, image_size):
    g = golden(f"sr3_{image_size}")
    rows = g["rows"]                            # the image rows at which the fixture holds the reference's outputs
    sched = json.loads(str(g["sched"]))
    betas = oracle.make_beta_schedule(**sched)
    T = len(betas)
    _, _, eng = make_engine(oracle, image_size, betas)
    cond = torch.from_numpy(g["cond"]).cuda()
    H = cond.shape[-1]
    noises = torch.randn(T, 1, 3, H, H, generator=torch.Generator().manual_seed(int(g["noise_seed"])))
    assert abs(float(noises.double().sum()) - float(g["noise_sum"])) < 1e-6, "noise stream differs from the fixture's"
    ref = torch.from_numpy(g["sr"])            # (3,H,W): the reference's ret_img[-1]
    sr, tr = eng.sample(cond, noise=noises.cuda(), trace=True)
    sr, tr = sr.cpu(), tr.cpu()
    assert tuple(sr.shape) == (1, 3, H, H) and tuple(tr.shape) == (1, T + 1, 3, H, H)
    r = rel_l2(sr[0][..., rows, :], ref)
    psnr = oracle.psnr_u8(oracle.to_u8(sr[0][..., rows, :]), oracle.to_u8(ref))
    print(f"sr3 sampler[image_size={image_size}] T={T}: rel-L2 vs reference {r:.3e}, PSNR(ours, reference) {psnr:.1f} dB")
    assert r <= 1e-2
    refc = torch.from_numpy(g["sr_continous"])  # frames 0, 4, 8, 12 of the reference's continous=True output
    assert torch.equal(tr[0, 0], torch.from_numpy(g["cond"])[0])   # frame 0 is the conditioning image itself
    assert rel_l2(tr[0, ::4][..., rows, :], refc) <= 1e-2
    assert torch.equal(tr[0, -1], sr[0])
    # built-in noise: finite, reproducible per seed
    a = eng.sample(cond, seed=7).cpu()
    b = eng.sample(cond, seed=7).cpu()
    assert torch.isfinite(a).all() and torch.equal(a, b)


def test_sr3_define_G_surface(oracle):
    """define_G(which_model_G='ddpm') -> netG.super_resolution with the reference's return conventions."""
    from fastdiffsr_b200 import define_G
    from fastdiffsr_b200.config import default_config
    opt = default_config("sr_ddpm_test_64_256")
    assert opt["model"]["which_model_G"] == "ddpm"
    assert opt["model"]["beta_schedule"]["val"]["n_timestep"] == 1000
    netG = define_G(opt)
    ref_spec = oracle.sr3_state_dict_spec(oracle.SR3_UNET, 256)
    keys = [(k, tuple(v.shape)) for k, v in netG.state_dict().items()]
    assert keys == [(k, s) for k, s, _, _ in ref_spec]
    sd = oracle.make_state_dict(oracle.SR3_UNET, seed=3, spec=ref_spec)
    netG.load_state_dict(sd, strict=True)
    netG = netG.to("cuda:0")
    sched = dict(schedule="linear", n_timestep=8, linear_start=1e-4, linear_end=0.3)
    netG.set_new_noise_schedule(sched, "cuda:0")
    assert len(netG.state_dict()) == len(ref_spec) + 12
    x = torch.rand(1, 3, 64, 64, device="cuda:0") * 2 - 1
    out = netG.super_resolution(x, continous=False)
    assert tuple(out.shape) == (3, 64, 64)                     # ret_img[-1]: batch axis dropped (reference)
    outc = netG.super_resolution(x, continous=True)
    assert tuple(outc.shape) == (1 + 8, 3, 64, 64)             # sample_inter = 1 | (8 // 10) = 1
    assert torch.equal(outc[0], x[0])
    out2 = netG.super_resolution(torch.cat([x, x]), continous=False)
    assert tuple(out2.shape) == (2, 3, 64, 64)
    tabs = oracle.schedule_tables(oracle.make_beta_schedule(**sched))
    noises = torch.randn(8, 1, 3, 64, 64, generator=torch.Generator().manual_seed(1))
    ref = oracle.sr3_sample_loop(sd, oracle.SR3_UNET, tabs, x.cpu(), noises, 256)
    got = netG.super_resolution(x, noise=noises.cuda()).cpu()
    assert rel_l2(got, ref[0]) <= 1e-2

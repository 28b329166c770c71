"""Parity of the CUDA path (through the C ABI) against the oracle and the committed reference
outputs.  Needs a B200: run with `pytest -m gpu`.

Tolerances (BASELINE.json north_star): per-step epsilon relative L2 <= 1e-2 for the 16-bit modes,
final SR PSNR within 0.05 dB of the reference; integer paths (bicubic, uint8 SSE) bit-exact;
the fp32 posterior arithmetic bit-exact.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

# north-star bar: per-step eps relative L2 <= 1e-2 in BOTH 16-bit modes, checked in the same pytest run (the module's
# engine fixture is parametrized over the dtype; nothing depends on an environment variable).  fp16 measures ~1.5e-3;
# bf16 (bf16 storage, fp16 post-GroupNorm operands — fdsr.h FDSR_DTYPE_BF16) ~5e-3.  Pure bf16 operands measured
# 0.81-1.02e-2 in round 1 (SURVEY F10), which is why the operand policy changed instead of the bar.
EPS_TOL = 1e-2
LAYER_TOLS = {"fp16": 5e-3, "bf16": 1.5e-2}   # every intermediate activation (bf16 storage rounds at 2^-9 per tensor)


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


@pytest.fixture(scope="module", params=["fp16", "bf16"])
def ctx(request, oracle, schedule):
    from fastdiffsr_b200 import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no fallback exists)"
    cfg = dict(oracle.DEFAULT_UNET)
    out = {"dtype": request.param}
    for tag, jitter in (("default", 0.0), ("jitter", 0.2)):
        sd = oracle.make_state_dict(cfg, seed=0, gn_jitter=jitter)
        eng = Engine(cfg, "cuda:0", request.param)
        eng.load_state_dict(sd)
        eng.set_schedule(schedule["betas"])
        out[tag] = (sd, eng)
    out["cfg"] = cfg
    yield out
    for tag in ("default", "jitter"):
        out[tag][1].close()


def test_tables_match_reference(ctx, golden_dir):
    _, eng = ctx["default"]
    g = np.load(os.path.join(golden_dir, "schedule_T20.npz"))
    for k in g.files:
        mine = eng.table(k)
        ref = g[k]
        if ref.dtype == np.float32:
            assert np.array_equal(mine.astype(np.float32), ref), k
        else:
            assert np.array_equal(mine, ref), k


@pytest.mark.parametrize("tag", ["default", "jitter"])
def test_unet_eps_vs_reference_golden(ctx, golden, schedule, tag):
    sd, eng = ctx[tag]
    g = golden(f"unet64_{tag}")
    x6 = torch.from_numpy(g["x6"]).cuda()
    for i, t in enumerate((19, 7)):   # noise levels stored: sqrt_alphas_cumprod_prev[20], [8]
        assert abs(float(np.float32(schedule["sqrt_alphas_cumprod_prev"][t + 1])) - float(g["noise_levels"][i])) < 1e-12
        eps = eng.unet_forward(x6[:, :3].contiguous(), x6[:, 3:].contiguous(), t).cpu()
        r = rel_l2(eps, torch.from_numpy(g["eps"][i]))
        print(f"[{ctx['dtype']} {tag}] t={t}: eps rel-L2 vs reference = {r:.3e}")
        assert r <= EPS_TOL


def test_every_layer_vs_oracle(ctx, oracle, schedule):
    sd, eng = ctx["jitter"]
    cfg = ctx["cfg"]
    g = torch.Generator().manual_seed(5)
    B, H, W = 2, 64, 96      # non-square, partial tiles at every level
    cond = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    x = torch.randn(B, 3, H, W, generator=g)
    t = 11
    taps = {}
    nl = torch.full((B, 1), float(np.float32(schedule["sqrt_alphas_cumprod_prev"][t + 1])))
    eps_ref = oracle.unet_forward(sd, cfg, torch.cat([cond, x], 1), nl, taps=taps)
    eps = eng.unet_forward(cond.cuda(), x.cuda(), t).cpu()
    for name in eng.tensor_names():
        if name in taps:
            got = eng.read_tensor(name, B, taps[name].numel()).cpu()
            assert got.shape == taps[name].shape
            r = rel_l2(got, taps[name])
            assert r <= LAYER_TOLS[ctx["dtype"]], (name, r)
    assert rel_l2(eps, eps_ref) <= EPS_TOL


def test_per_step_eps_teacher_forced(ctx, oracle, schedule):
    """All 20 steps: feed the oracle's x_t into the CUDA UNet (no trajectory drift, SURVEY hard part 6)."""
    sd, eng = ctx["default"]
    cfg = ctx["cfg"]
    g = torch.Generator().manual_seed(21)
    cond = torch.rand(1, 3, 64, 64, generator=g) * 2 - 1
    noises = torch.randn(20, 1, 3, 64, 64, generator=g)
    trace = []
    oracle.sample_loop(sd, cfg, schedule, cond, noises, trace=trace)
    worst = 0.0
    for st in trace:
        eps = eng.unet_forward(cond.cuda(), st["x_t"].cuda(), st["t"]).cpu()
        r = rel_l2(eps, st["eps"])
        worst = max(worst, r)
        assert r <= EPS_TOL, (st["t"], r)
        # posterior arithmetic on the oracle's eps is exact fp32
        z = noises[20 - st["t"]].cuda() if st["t"] > 0 else None
        xp = eng.posterior_step(st["x_t"].cuda(), st["eps"].cuda(), z, st["t"]).cpu()
        assert torch.equal(xp, st["x_prev"]) or (xp - st["x_prev"]).abs().max() <= 1e-6 * st["x_prev"].abs().max()
    print(f"[{ctx['dtype']}] worst teacher-forced eps rel-L2 over 20 steps: {worst:.3e}")


@pytest.mark.parametrize("tag", ["default", "jitter"])
def test_sampler_vs_reference_golden(ctx, oracle, golden, tag):
    sd, eng = ctx[tag]
    g = golden(f"unet64_{tag}")
    cond = torch.from_numpy(g["cond"]).cuda()
    noises = torch.from_numpy(g["noises"]).cuda()
    ref = torch.from_numpy(g["sr"])
    sr = eng.sample(cond, noise=noises).cpu()
    assert sr.shape == ref.shape
    # PSNR delta against a synthetic HR (cond + low-passed noise): |PSNR(ours,HR) - PSNR(ref,HR)| <= 0.05 dB
    gen = torch.Generator().manual_seed(9)
    hr = (torch.from_numpy(g["cond"]) + 0.1 * torch.nn.functional.avg_pool2d(
        torch.randn(1, 3, 64, 64, generator=gen), 3, 1, 1)).clamp(-1, 1)
    p_ours = oracle.psnr_u8(oracle.to_u8(sr[0]), oracle.to_u8(hr[0]))
    p_ref = oracle.psnr_u8(oracle.to_u8(ref[0]), oracle.to_u8(hr[0]))
    print(f"[{tag}] PSNR ours {p_ours:.4f} dB, reference {p_ref:.4f} dB, PSNR(ours,ref) "
          f"{oracle.psnr_u8(oracle.to_u8(sr[0]), oracle.to_u8(ref[0])):.1f} dB")
    assert abs(p_ours - p_ref) <= 0.05
    assert rel_l2(sr, ref) <= 1e-2
    # continous=True layout at B=1 is the reference's (1+7,3,H,W)
    sr2, tr = eng.sample(cond, noise=noises, trace=True)
    refc = torch.from_numpy(g["sr_continous"])
    assert tuple(tr.shape) == (1, 8, 3, 64, 64)
    assert torch.equal(sr2.cpu(), sr)
    assert rel_l2(tr[0].cpu(), refc) <= 1e-2
    assert torch.equal(tr[0, -1].cpu(), sr[0])


def test_batch_equals_per_image_and_graph_equals_stream(ctx):
    """B>1 (where the reference crashes, SURVEY F2) == B=1 per image; CUDA-graph replay == stream launches."""
    _, eng = ctx["default"]
    g = torch.Generator().manual_seed(2)
    B = 3
    cond = (torch.rand(B, 3, 64, 64, generator=g) * 2 - 1).cuda()
    noises = torch.randn(20, B, 3, 64, 64, generator=g).cuda()
    eng.set_use_graph(True)
    full = eng.sample(cond, noise=noises)
    again = eng.sample(cond, noise=noises)
    assert torch.equal(full, again)        # deterministic replay
    eng.set_use_graph(False)
    plain = eng.sample(cond, noise=noises)
    eng.set_use_graph(True)
    assert (full - plain).abs().max().item() <= 1e-5
    for b in range(B):
        one = eng.sample(cond[b:b + 1].contiguous(), noise=noises[:, b:b + 1].contiguous())
        assert (one[0] - full[b]).abs().max().item() <= 1e-5


def test_builtin_noise_is_gaussian_and_seeded(ctx):
    _, eng = ctx["default"]
    cond = torch.zeros(2, 3, 64, 64, device="cuda")
    a = eng.sample(cond, seed=1)
    b = eng.sample(cond, seed=1)
    c = eng.sample(cond, seed=2)
    assert torch.equal(a, b) and not torch.equal(a, c)
    assert torch.isfinite(a).all() and a.abs().max() <= 1.5 + 1e-6


def test_bicubic_bit_exact(ctx, golden_dir):
    _, eng = ctx["default"]
    g = np.load(os.path.join(golden_dir, "bicubic.npz"))
    lr = torch.from_numpy(np.stack([g["lr0"], g["lr1"]])).cuda()
    u8, cond = eng.bicubic_u8(lr, 512, 512)
    rows = g["rows"]                                        # the rows of the 512x512 outputs the fixture stores
    ref = np.stack([g["sr0"], g["sr1"]])
    assert np.array_equal(u8.cpu().numpy()[:, rows], ref)   # the reference's own UC-Merced fixtures
    refc = torch.from_numpy(ref).float().div(255.0).mul(2.0).sub(1.0).permute(0, 3, 1, 2)
    assert torch.equal(cond.cpu()[:, :, rows], refc)
    for h in (64, 32):
        u8, _ = eng.bicubic_u8(torch.from_numpy(g[f"syn_lr_{h}"])[None].cuda(), 256, 256)
        assert np.array_equal(u8[0].cpu().numpy(), g[f"syn_sr_{h}"])


def test_bicubic_ragged_vs_oracle(ctx, oracle):
    _, eng = ctx["default"]
    rng = np.random.default_rng(3)
    for (h, w, H, W) in ((8, 16, 64, 32), (5, 7, 40, 56), (16, 16, 16, 16)):
        a = rng.integers(0, 256, size=(2, h, w, 3), dtype=np.uint8)
        u8, _ = eng.bicubic_u8(torch.from_numpy(a).cuda(), H, W)
        for b in range(2):
            assert np.array_equal(u8[b].cpu().numpy(), oracle.pil_bicubic_u8(a[b], H, W))


def test_sse_u8_matches_tensor2img(ctx, oracle):
    _, eng = ctx["default"]
    g = torch.Generator().manual_seed(4)
    a = torch.randn(3, 3, 64, 64, generator=g) * 0.7
    b = a + 0.05 * torch.randn(3, 3, 64, 64, generator=g)
    sse = eng.sse_u8(a.cuda(), b.cuda()).cpu().numpy()
    for i in range(3):
        ua, ub = oracle.to_u8(a[i]).astype(np.int64), oracle.to_u8(b[i]).astype(np.int64)
        assert sse[i] == float(((ua - ub) ** 2).sum())


def test_host_buffer_path_equals_device_path(ctx, oracle):
    _, eng = ctx["default"]
    rng = np.random.default_rng(8)
    lr = rng.integers(0, 256, size=(2, 16, 16, 3), dtype=np.uint8)
    noises = torch.randn(20, 2, 3, 64, 64, generator=torch.Generator().manual_seed(1)).cuda()
    out = eng.super_resolve_u8_host(lr, 64, 64, noise=noises)
    _, cond = eng.bicubic_u8(torch.from_numpy(lr).cuda(), 64, 64)
    ref = eng.sample(cond, noise=noises).cpu().numpy()
    assert np.array_equal(out, ref)


def test_define_G_drop_in(ctx, oracle, golden):
    """The reference-facing API: define_G -> .to(cuda) -> set_new_noise_schedule -> super_resolution."""
    import fastdiffsr_b200 as F
    opt = F.config.default_config()
    opt["model"]["compute_dtype"] = ctx["dtype"]
    netG = F.define_G(opt)
    sd = oracle.make_state_dict(oracle.DEFAULT_UNET, seed=0)
    netG.load_state_dict(sd, strict=False)
    netG.to("cuda")
    netG.set_loss("cuda")
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cuda")
    netG.eval()
    g = golden("unet64_default")
    cond, noises = torch.from_numpy(g["cond"]).cuda(), torch.from_numpy(g["noises"]).cuda()
    sr = netG.super_resolution(cond, False, noise=noises)
    assert rel_l2(sr.cpu(), torch.from_numpy(g["sr"])) <= 1e-2
    cont = netG.super_resolution(cond, True, noise=noises)
    assert tuple(cont.shape) == (8, 3, 64, 64)
    assert torch.isfinite(netG.super_resolution(cond, False)).all()   # unseeded, like the reference


def test_full_size_step_vs_oracle(ctx, oracle, schedule):
    """256x256 (BASELINE config shape): one UNet step, B=1, oracle computed live on the host (~1-2 s)."""
    sd, eng = ctx["default"]
    cfg = ctx["cfg"]
    g = torch.Generator().manual_seed(13)
    cond = torch.rand(1, 3, 256, 256, generator=g) * 2 - 1
    x = torch.randn(1, 3, 256, 256, generator=g)
    t = 9
    nl = torch.full((1, 1), float(np.float32(schedule["sqrt_alphas_cumprod_prev"][t + 1])))
    ref = oracle.unet_forward(sd, cfg, torch.cat([cond, x], 1), nl)
    eps = eng.unet_forward(cond.cuda(), x.cuda(), t).cpu()
    r = rel_l2(eps, ref)
    print(f"[{ctx['dtype']}] 256x256 eps rel-L2 {r:.3e}")
    assert r <= EPS_TOL
    assert abs(eng.unet_flops() / 1e9 - 268.31) < 0.05      # SURVEY: 268.31 GFLOP per image-step at 256^2


def test_full_batch_properties(ctx):
    """BASELINE configs[1] shape (B=16, 256^2): size-independent properties — per-image independence
    (a batch slot does not depend on its neighbours), finiteness, output range of res2img."""
    _, eng = ctx["default"]
    g = torch.Generator().manual_seed(17)
    cond = (torch.rand(16, 3, 256, 256, generator=g) * 2 - 1).cuda()
    a = eng.sample(cond, seed=5)
    assert torch.isfinite(a).all()
    assert (a - cond).abs().max().item() <= 0.5 + 1e-6          # clamp(x,-1,1)/2 + cond
    perm = torch.arange(15, -1, -1, device="cuda")
    # the builtin RNG is indexed by batch position, so compare with injected noise instead
    noises = torch.randn(20, 4, 3, 256, 256, generator=g).cuda()
    c4 = cond[:4].contiguous()
    s1 = eng.sample(c4, noise=noises)
    s2 = eng.sample(c4.flip(0).contiguous(), noise=noises.flip(1).contiguous())
    assert (s1 - s2.flip(0)).abs().max().item() <= 1e-5
    del perm


def test_infer_x4_shape_properties(ctx, oracle):
    """BASELINE configs[3] shape (x4 128 -> 512, the UC-Merced infer config): bit-exact bicubic conditioning at
    512^2, one UNet step against the oracle at a 128x512 strip of it (same tiles_x, ragged tile rows), and
    size-independent properties of the full 20-step sampler at 512^2: finite, range of res2img, per-image
    independence of batch neighbours."""
    sd, eng = ctx["default"]
    cfg = ctx["cfg"]
    g = torch.Generator().manual_seed(23)
    lr = torch.randint(0, 256, (2, 128, 128, 3), generator=g, dtype=torch.uint8)
    up8, cond = eng.bicubic_u8(lr.cuda(), 512, 512)
    for b in range(2):
        assert np.array_equal(up8[b].cpu().numpy(), oracle.pil_bicubic_u8(lr[b].numpy(), 512, 512))
    noises = torch.randn(20, 2, 3, 512, 512, generator=g).cuda()
    both = eng.sample(cond, noise=noises)
    assert torch.isfinite(both).all() and (both - cond).abs().max().item() <= 0.5 + 1e-6
    one = eng.sample(cond[1:2].contiguous(), noise=noises[:, 1:2].contiguous())
    assert (one[0] - both[1]).abs().max().item() <= 1e-5
    # one step on a 128 x 512 strip vs the oracle (a few seconds on the host)
    x6 = torch.cat([cond[:1, :, :128].cpu(), torch.randn(1, 3, 128, 512, generator=g)], 1)
    t = 4
    nl = torch.full((1, 1), float(np.float32(oracle.schedule_tables(oracle.make_beta_schedule(**oracle.DEFAULT_SCHEDULE))
                                             ["sqrt_alphas_cumprod_prev"][t + 1])))
    ref = oracle.unet_forward(sd, cfg, x6, nl)
    eps = eng.unet_forward(x6[:, :3].contiguous().cuda(), x6[:, 3:].contiguous().cuda(), t).cpu()
    r = rel_l2(eps, ref)
    print(f"128x512 strip eps rel-L2 {r:.3e}")
    assert r <= EPS_TOL


def test_x8_shape_bicubic_and_step(ctx, oracle):
    """BASELINE configs[2] shape (x8 32 -> 256): bit-exact x8 bicubic conditioning, sampler properties."""
    _, eng = ctx["default"]
    g = torch.Generator().manual_seed(29)
    lr = torch.randint(0, 256, (3, 32, 32, 3), generator=g, dtype=torch.uint8)
    up8, cond = eng.bicubic_u8(lr.cuda(), 256, 256)
    for b in range(3):
        assert np.array_equal(up8[b].cpu().numpy(), oracle.pil_bicubic_u8(lr[b].numpy(), 256, 256))
    a = eng.sample(cond, seed=3)
    again = eng.sample(cond, seed=3)
    assert torch.equal(a, again) and torch.isfinite(a).all()
    assert not torch.equal(a, eng.sample(cond, seed=4))

"""fp32 parity mode (dtype="fp32": the same fused layer plan on the CUDA cores, fp32 end to end) against
the committed reference outputs and the oracle.  BASELINE.json north_star: per-step epsilon relative
L2 <= 1e-4 in fp32 mode.  Needs a B200: `pytest -m gpu`.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

EPS_TOL_FP32 = 1e-4     # north-star tolerance for the fp32 mode
LAYER_TOL_FP32 = 1e-4   # every intermediate activation


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def ctx32(oracle, schedule):
    from fastdiffsr_b200 import Engine
    assert torch.cuda.is_available(), "GPU tests need a CUDA device (no fallback exists)"
    cfg = dict(oracle.DEFAULT_UNET)
    out = {"cfg": cfg}
    for tag, jitter in (("default", 0.0), ("jitter", 0.2)):
        sd = oracle.make_state_dict(cfg, seed=0, gn_jitter=jitter)
        eng = Engine(cfg, "cuda:0", "fp32")
        eng.load_state_dict(sd)
        eng.set_schedule(schedule["betas"])
        out[tag] = (sd, eng)
    return out


@pytest.mark.parametrize("tag", ["default", "jitter"])
def test_fp32_unet_eps_vs_reference_golden(ctx32, golden, tag):
    sd, eng = ctx32[tag]
    g = golden(f"unet64_{tag}")
    x6 = torch.from_numpy(g["x6"]).cuda()
    for i, t in enumerate((19, 7)):
        eps = eng.unet_forward(x6[:, :3].contiguous(), x6[:, 3:].contiguous(), t).cpu()
        r = rel_l2(eps, torch.from_numpy(g["eps"][i]))
        print(f"[fp32 {tag}] t={t}: eps rel-L2 vs reference = {r:.3e}")
        assert r <= EPS_TOL_FP32


def test_fp32_every_layer_vs_oracle(ctx32, oracle, schedule):
    """Non-square input with partial tiles at every level; every intermediate tensor of the plan."""
    sd, eng = ctx32["jitter"]
    cfg = ctx32["cfg"]
    g = torch.Generator().manual_seed(5)
    B, H, W = 2, 64, 96
    cond = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    x = torch.randn(B, 3, H, W, generator=g)
    t = 11
    taps = {}
    nl = torch.full((B, 1), float(np.float32(schedule["sqrt_alphas_cumprod_prev"][t + 1])))
    eps_ref = oracle.unet_forward(sd, cfg, torch.cat([cond, x], 1), nl, taps=taps)
    eps = eng.unet_forward(cond.cuda(), x.cuda(), t).cpu()
    worst = 0.0
    for name in eng.tensor_names():
        if name in taps:
            got = eng.read_tensor(name, B, taps[name].numel()).cpu()
            r = rel_l2(got, taps[name])
            worst = max(worst, r)
            assert r <= LAYER_TOL_FP32, (name, r)
    print(f"[fp32] worst layer rel-L2 {worst:.3e}, eps {rel_l2(eps, eps_ref):.3e}")
    assert rel_l2(eps, eps_ref) <= EPS_TOL_FP32


def test_fp32_sampler_vs_reference_golden(ctx32, oracle, golden):
    """The whole 20-step chain with the reference's injected noise: trajectory stays within 1e-3 of the
    reference (the clamp and 20 accumulated steps amplify the per-step 1e-5), PSNR delta <= 0.05 dB."""
    sd, eng = ctx32["default"]
    g = golden("unet64_default")
    cond = torch.from_numpy(g["cond"]).cuda()
    noises = torch.from_numpy(g["noises"]).cuda()
    ref = torch.from_numpy(g["sr"])
    sr = eng.sample(cond, noise=noises).cpu()
    r = rel_l2(sr, ref)
    p = oracle.psnr_u8(oracle.to_u8(sr[0]), oracle.to_u8(ref[0]))
    print(f"[fp32] 20-step SR rel-L2 vs reference {r:.3e}, PSNR(ours, reference) {p:.1f} dB")
    assert r <= 1e-3
    gen = torch.Generator().manual_seed(9)
    hr = (torch.from_numpy(g["cond"]) + 0.1 * torch.nn.functional.avg_pool2d(
        torch.randn(1, 3, 64, 64, generator=gen), 3, 1, 1)).clamp(-1, 1)
    assert abs(oracle.psnr_u8(oracle.to_u8(sr[0]), oracle.to_u8(hr[0])) -
               oracle.psnr_u8(oracle.to_u8(ref[0]), oracle.to_u8(hr[0]))) <= 0.05


def test_fp32_per_step_eps_teacher_forced(ctx32, oracle, schedule):
    sd, eng = ctx32["default"]
    cfg = ctx32["cfg"]
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
        assert r <= EPS_TOL_FP32, (st["t"], r)
    print(f"[fp32] worst teacher-forced eps rel-L2 over 20 steps: {worst:.3e}")

"""The kernel's alternative code paths against each other (B200, `pytest -m gpu`): where the automatic per-layer choice
picks between two forms of a computation, each for some supported layer or configuration, an environment switch read at
context creation forces one form everywhere, and the two forms must agree — bitwise where the arithmetic is identical,
within 16-bit rounding noise where the association changes (a one-ulp change of an early activation reshuffles every
later rounding: the whole-network difference is the same ~1e-3 as between either form and the fp32 reference).

  FDSR_UP_PHASES=0   nearest-upsample convs: nine-tap form on the gathered 2x patch  vs  four 2x2 phase convs with
                     pre-summed weights on the low-resolution input (exact identity up to the rounding of the sums)
  FDSR_RESID_MMA=0   identity residual of the N = 64 layers added by the epilogue    vs  an identity-matrix K chunk
  FDSR_SPLIT_N=0     256-wide low-resolution layers on one CTA per tile              vs  two 128-column halves
  FDSR_PAIR=0        every layer on single CTAs (tcgen05.mma.cta_group::1)           vs  CTA pairs (cta_group::2, M = 256,
                     each CTA staging half of the weight columns) where the tile rows are even
  FDSR_HALF_TILES=0  32 x 8 tiles everywhere (split-N / single accumulator at <= 64^2)  vs  16 x 8 half tiles as CTA pairs
  FDSR_EPI2=0        one epilogue team for every layer                               vs  producer warps 12..19 as a second
                     epilogue team (odd 32-column blocks) in the layers that have no producer work
  FDSR_TAIL_HELP=0   the last tile of every CTA drained by warps 4..11 alone        vs  producer warps 12..19 joining as a
                     second team for that one tile (its epilogue is exposed: nothing left to overlap it with)
  FDSR_FUSED_TAIL=0  sampler: pack_input / final conv -> eps / posterior kernels    vs  the final conv's epilogue doing the
                     posterior update in registers and rewriting the next step's input (checked on the sampler)
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def make(oracle, schedule, env=None):
    from fastdiffsr_b200 import Engine
    cfg = dict(oracle.DEFAULT_UNET)
    sd = oracle.make_state_dict(cfg, seed=0, gn_jitter=0.2)
    env = env or {}
    os.environ.update(env)
    try:
        eng = Engine(cfg, "cuda:0", "fp16")     # the switches are read when the context is created
    finally:
        for k in env:
            os.environ.pop(k, None)
    eng.load_state_dict(sd)
    eng.set_schedule(schedule["betas"])
    return eng


@pytest.fixture(scope="module")
def inputs():
    g = torch.Generator().manual_seed(17)
    B, H, W = 2, 128, 96
    return (torch.rand(B, 3, H, W, generator=g) * 2 - 1).cuda(), torch.randn(B, 3, H, W, generator=g).cuda()


@pytest.fixture(scope="module")
def base(oracle, schedule, inputs):
    eng = make(oracle, schedule)
    return eng, eng.unet_forward(inputs[0], inputs[1], 9)


@pytest.mark.parametrize("switch,tol", [("FDSR_SPLIT_N", 0.0), ("FDSR_HALF_TILES", 0.0), ("FDSR_EPI2", 0.0),
                                        ("FDSR_TAIL_HELP", 0.0), ("FDSR_PAIR", 3e-3), ("FDSR_RESID_MMA", 3e-3),
                                        ("FDSR_UP_PHASES", 3e-3)])
def test_alternative_paths_agree(oracle, schedule, inputs, base, switch, tol):
    eng0, eps0 = base
    eng1 = make(oracle, schedule, {switch: "0"})
    eps1 = eng1.unet_forward(inputs[0], inputs[1], 9)
    r = rel_l2(eps1, eps0)
    print(f"{switch}=0 vs default: eps rel-L2 {r:.3e}")
    if tol == 0.0:
        assert torch.equal(eps1, eps0), (switch, r)
    elif switch == "FDSR_PAIR":
        assert r <= tol, (switch, r)            # (measured: bit-identical — cta_group::2 accumulates like ::1)
    else:
        assert 0.0 < r <= tol, (switch, r)      # (a zero difference would mean the switch did nothing)


def test_phase_upsample_layers_vs_oracle(oracle, schedule, inputs, base):
    """The three upsample convs themselves, against the oracle's nearest-upsample + conv3x3."""
    eng, _ = base
    cfg = dict(oracle.DEFAULT_UNET)
    sd = oracle.make_state_dict(cfg, seed=0, gn_jitter=0.2)
    taps = {}
    import numpy as np
    B = inputs[0].shape[0]
    nl = torch.full((B, 1), float(np.float32(schedule["sqrt_alphas_cumprod_prev"][10])))
    oracle.unet_forward(sd, cfg, torch.cat([inputs[0].cpu(), inputs[1].cpu()], 1), nl, taps=taps)
    for name in ("ups.3", "ups.7", "ups.11"):
        got = eng.read_tensor(name, B, taps[name].numel()).cpu()
        assert got.shape == taps[name].shape
        assert rel_l2(got, taps[name]) <= 5e-3, name


@pytest.mark.parametrize("dtype", ["fp16", "bf16"])
def test_fused_tail_equals_separate_kernels(oracle, schedule, dtype):
    """The sampler with the posterior update fused into the final conv's epilogue (default) equals, bit for bit, the
    sampler that writes eps, runs posterior_kernel and re-packs the input each step — with injected noise, with the
    built-in generator, and with the continous=True trace (diffusion.py:157-221)."""
    from fastdiffsr_b200 import Engine
    cfg = dict(oracle.DEFAULT_UNET)
    sd = oracle.make_state_dict(cfg, seed=0, gn_jitter=0.1)

    def mk(env):
        os.environ.update(env)
        try:
            e = Engine(cfg, "cuda:0", dtype)
        finally:
            for k in env:
                os.environ.pop(k, None)
        e.load_state_dict(sd)
        e.set_schedule(schedule["betas"])
        return e

    fused, plain = mk({}), mk({"FDSR_FUSED_TAIL": "0"})
    g = torch.Generator().manual_seed(31)
    cond = (torch.rand(3, 3, 64, 96, generator=g) * 2 - 1).cuda()
    noises = torch.randn(20, 3, 3, 64, 96, generator=g).cuda()
    a, ta = fused.sample(cond, noise=noises, trace=True)
    b, tb = plain.sample(cond, noise=noises, trace=True)
    assert torch.equal(a, b) and torch.equal(ta, tb)
    assert torch.equal(fused.sample(cond, seed=5, image_offset=7), plain.sample(cond, seed=5, image_offset=7))
    assert fused.launch_count() < plain.launch_count()      # two launches fewer per step
    fused.close()
    plain.close()

"""The oracle (oracle/fdsr_oracle.py) against the committed reference outputs in tests/golden/
(written by oracle/make_golden.py from the real reference).  CPU only."""
import os

import numpy as np
import pytest
import torch


def test_schedule_tables_match_reference(oracle, schedule, golden_dir):
    g = np.load(os.path.join(golden_dir, "schedule_T20.npz"))
    for k in g.files:
        ref = g[k]
        mine = schedule[k]
        if ref.dtype == np.float32:
            assert np.array_equal(ref, mine.astype(np.float32)), k
        else:
            assert np.array_equal(ref, mine), k


def test_schedule_known_answers(schedule):
    # SURVEY 8(c): values derived from the reference code
    assert abs(schedule["betas"][0] - 0.01598644) < 1e-8
    assert abs(schedule["betas"][16] - 0.86728909) < 1e-8
    assert schedule["betas"][17] == 0.999 and schedule["betas"][19] == 0.999
    assert abs(schedule["alphas_cumprod"][0] - 9.84013557e-01) < 1e-9
    assert abs(schedule["sqrt_alphas_cumprod_prev"][1] - 0.991974575) < 1e-9
    assert np.float32(schedule["posterior_mean_coef1"][0]) == 1.0 and schedule["posterior_mean_coef2"][0] == 0.0
    assert abs(schedule["posterior_log_variance_clipped"][0] - np.log(1e-20)) < 1e-12
    assert abs(schedule["sqrt_recip_alphas_cumprod"][19] - 1.5072739e06) < 1.0


def test_state_dict_spec(oracle):
    spec = oracle.state_dict_spec(oracle.DEFAULT_UNET)
    assert len(spec) == 317
    n = sum(int(np.prod(s)) for _, s, _, _ in spec)
    assert n == 23_802_277  # SURVEY section 6
    dead = 0
    for k, shp, _, _ in spec:
        stem = k.rsplit(".", 1)[0]
        if stem.endswith(".conv") and (stem + ".weight", ) and any(
                kk == stem + ".weight" and ss[2] == 1 for kk, ss, _, _ in spec if len(ss) == 4):
            dead += int(np.prod(shp))
    assert dead == 892_864  # the 22 never-executed 1x1 convs (SURVEY F9)


@pytest.mark.parametrize("tag", ["default", "jitter"])
def test_unet_and_sampler_match_reference(oracle, schedule, golden, tag):
    g = golden(f"unet64_{tag}")
    cfg = dict(oracle.DEFAULT_UNET)
    sd = oracle.make_state_dict(cfg, seed=int(g["seed"]), gn_jitter=float(g["gn_jitter"]))
    x6 = torch.from_numpy(g["x6"])
    for i, nl in enumerate(g["noise_levels"]):
        eps = oracle.unet_forward(sd, cfg, x6, torch.full((x6.shape[0], 1), float(nl)))
        assert np.abs(eps.numpy() - g["eps"][i]).max() <= 1e-5
    cond, noises = torch.from_numpy(g["cond"]), torch.from_numpy(g["noises"])
    trace = []
    sr = oracle.sample_loop(sd, cfg, schedule, cond, noises, False, trace=trace)
    assert np.abs(sr.numpy() - g["sr"]).max() <= 1e-4
    assert np.abs(trace[0]["eps"].numpy() - g["eps_first"]).max() <= 1e-5
    assert np.abs(trace[-1]["eps"].numpy() - g["eps_last"]).max() <= 1e-4
    src = oracle.sample_loop(sd, cfg, schedule, cond, noises, True)
    assert src.shape == g["sr_continous"].shape == (8, 3, 64, 64)
    assert np.abs(src.numpy() - g["sr_continous"]).max() <= 1e-4


@pytest.mark.parametrize("image_size", [256, 64])
def test_sr3_unet_and_sampler_match_reference(oracle, golden, image_size):
    """SR3 baseline restatement (ddpm_modules) against the reference's outputs (tests/golden/sr3_*.npz, stored at the
    image rows `rows`)."""
    import json
    g = golden(f"sr3_{image_size}")
    rows = g["rows"]
    cfg = dict(oracle.SR3_UNET)
    spec = oracle.sr3_state_dict_spec(cfg, image_size)
    assert len(spec) == 421
    sd = oracle.make_state_dict(cfg, seed=int(g["seed"]), gn_jitter=float(g["gn_jitter"]), spec=spec)
    x6 = torch.from_numpy(g["x6"])
    for i, t in enumerate(g["steps"][:1] if image_size == 256 else g["steps"]):
        eps = oracle.sr3_unet_forward(sd, cfg, x6, torch.full((x6.shape[0],), int(t), dtype=torch.long), image_size)
        assert np.abs(eps.numpy()[..., rows, :] - g["eps"][i]).max() <= 1e-5
    if image_size == 256:
        return  # (the 128x128 sampler costs ~10 s of CPU; the 64x64 fixture covers the loop)
    tab = oracle.schedule_tables(oracle.make_beta_schedule(**json.loads(str(g["sched"]))))
    cond = torch.from_numpy(g["cond"])
    H = cond.shape[-1]
    noises = torch.randn(12, 1, 3, H, H, generator=torch.Generator().manual_seed(int(g["noise_seed"])))
    assert abs(float(noises.double().sum()) - float(g["noise_sum"])) < 1e-6
    sr = oracle.sr3_sample_loop(sd, cfg, tab, cond, noises, image_size, False)
    assert np.abs(sr[0].numpy()[..., rows, :] - g["sr"]).max() <= 1e-4
    src = oracle.sr3_sample_loop(sd, cfg, tab, cond, noises, image_size, True)
    assert tuple(src.shape) == (13, 3, H, H)
    assert np.abs(src[::4].numpy()[..., rows, :] - g["sr_continous"]).max() <= 1e-4


def test_sr3_attention_layout(oracle):
    """SelfAttention flags follow the configured image_size, not the input (ddpm_modules/unet.py:184, 211)."""
    for image_size, level in ((256, 4), (64, 2), (512, 5)):
        downs, mid, ups, last = oracle.sr3_unet_layers(oracle.SR3_UNET, image_size)
        flagged = [e[1] for e in downs + ups if e[0] == "res" and e[4]]
        assert len(flagged) == 5 and mid[0][4] and not mid[1][4] and last == 64
        widths = [64, 64, 128, 128, 256, 256]
        assert all(e[3] == widths[level] for e in downs + ups if e[0] == "res" and e[4])


def test_film_table_matches_forward(oracle, schedule):
    cfg = dict(oracle.DEFAULT_UNET)
    sd = oracle.make_state_dict(cfg, seed=1)
    tab = oracle.film_table(sd, cfg, schedule)
    assert set(tab) == {e[1] for grp in oracle.unet_layers(cfg)[:3] for e in grp if e[0] == "res"}
    assert tab["downs.1"].shape == (20, 64) and tab["ups.0"].shape == (20, 256)


def test_bicubic_bit_exact_on_reference_fixtures(oracle, golden_dir):
    g = np.load(os.path.join(golden_dir, "bicubic.npz"))
    for i in range(2):  # UC-Merced lr_128 -> sr_128_512 from the reference tree (stored at the rows `rows`)
        assert np.array_equal(oracle.pil_bicubic_u8(g[f"lr{i}"], 512, 512)[g["rows"]], g[f"sr{i}"])
    for h in (64, 32):  # Pillow outputs for the x4 / x8 shapes
        assert np.array_equal(oracle.pil_bicubic_u8(g[f"syn_lr_{h}"], 256, 256), g[f"syn_sr_{h}"])


def test_bicubic_edge_cases(oracle):
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, size=(8, 16, 3), dtype=np.uint8)
    assert np.array_equal(oracle.pil_bicubic_u8(img, 8, 16), img)          # identity size
    flat = np.full((8, 8, 3), 200, dtype=np.uint8)
    assert np.array_equal(oracle.pil_bicubic_u8(flat, 32, 32), np.full((32, 32, 3), 200, np.uint8))
    try:
        from PIL import Image
    except Exception:
        return
    for (h, w, H, W) in ((8, 16, 64, 32), (5, 7, 40, 56), (16, 16, 128, 128)):   # ragged / non-square
        a = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        pil = np.array(Image.fromarray(a).resize((W, H), Image.BICUBIC))
        assert np.array_equal(oracle.pil_bicubic_u8(a, H, W), pil)


def test_posterior_extremes(oracle, schedule):
    # first steps: x0 is pure clamp saturation (SURVEY hard part 5); last step adds no noise
    x = torch.randn(1, 3, 8, 8)
    eps = torch.randn(1, 3, 8, 8)
    xp, _, x0 = oracle.p_sample_step(None, None, schedule, x, 19, None, torch.randn(1, 3, 8, 8), eps=eps)
    assert (x0.abs() == 1).all() and torch.isfinite(xp).all()
    xp0, _, x00 = oracle.p_sample_step(None, None, schedule, x, 0, None, None, eps=eps)
    assert torch.equal(xp0, x00)  # fp32 coef1 = 1, coef2 = 0, z = 0

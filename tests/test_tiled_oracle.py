"""Tiled sampling (fdsr_sample_tiled) in its CPU restatement: the grid and weight rule, and the two cases in which the tiled
sampler must reproduce the plain one bit for bit (tests/tiled_oracle.py against the oracle's sample_loop).  CPU only."""
import pytest
import torch

import tiled_oracle as TO


def _cover(starts, t_e, L):
    cov = torch.zeros(L, dtype=torch.int64)
    for s in starts:
        cov[s:s + t_e] += 1
    return cov


@pytest.mark.parametrize("t", [8, 16, 64, 256])
@pytest.mark.parametrize("overlap", [0, 4, 16, 32, 1000])
def test_grid_rule(t, overlap):
    for L in range(8, 601):
        starts, t_e, o_e = TO.tile_starts(L, t, overlap)
        s = t_e - o_e
        assert t_e % 8 == 0 and 8 <= t_e <= min(t, L) and s >= 8
        assert starts[0] == 0 and starts[-1] == L - t_e
        assert all(b - a > 0 and b - a <= s for a, b in zip(starts, starts[1:]))
        assert bool((_cover(starts, t_e, L) > 0).all())


def test_weights():
    for tey, tex, ov in [(64, 64, 16), (48, 64, 32), (8, 256, 0), (256, 256, 32), (16, 8, 1000)]:
        w = TO.tile_weights(tey, tex, ov)
        assert w.shape == (tey, tex) and w.dtype == torch.float32 and bool((w > 0).all())
        assert torch.equal(w, w.round())                       # integers
        assert torch.equal(w / w, torch.ones_like(w))          # a pixel covered by one tile keeps its eps exactly
    # the ramps rise over the overlap and are flat inside
    w = TO.tile_weights(64, 64, 16)
    assert w[0, 0] == 1 and w[16, 16] == 17 * 17 and w[32, 32] == 17 * 17 and w[63, 0] == 1
    # no overlap: every weight is 1
    assert torch.equal(TO.tile_weights(64, 128, 0), torch.ones(64, 128))


@pytest.fixture(scope="module")
def small(oracle):
    cfg = dict(oracle.DEFAULT_UNET)
    sd = oracle.make_state_dict(cfg, seed=0, gn_jitter=0.1)
    tab = oracle.schedule_tables(oracle.make_beta_schedule(**oracle.DEFAULT_SCHEDULE))
    return cfg, sd, tab


def test_one_tile_equals_sample_loop(oracle, small):
    cfg, sd, tab = small
    g = torch.Generator().manual_seed(1)
    cond = torch.rand(1, 3, 64, 64, generator=g) * 2 - 1
    noises = torch.randn(20, 1, 3, 64, 64, generator=g)
    ref = oracle.sample_loop(sd, cfg, tab, cond, noises, continous=True)
    assert torch.equal(TO.tiled_sample_loop(sd, cfg, tab, cond, noises, 64, 32, continous=True), ref)
    # a tile larger than the canvas shrinks to it
    assert torch.equal(TO.tiled_sample_loop(sd, cfg, tab, cond, noises, (256, 128), 32, continous=True), ref)


def test_partition_equals_per_crop_sample_loop(oracle, small):
    cfg, sd, tab = small
    g = torch.Generator().manual_seed(2)
    cond = torch.rand(1, 3, 64, 128, generator=g) * 2 - 1
    noises = torch.randn(20, 1, 3, 64, 128, generator=g)
    out = TO.tiled_sample_loop(sd, cfg, tab, cond, noises, 64, 0)
    for x0 in (0, 64):
        crop = oracle.sample_loop(sd, cfg, tab, cond[..., x0:x0 + 64].contiguous(), noises[..., x0:x0 + 64].contiguous())
        assert torch.equal(out[..., x0:x0 + 64], crop), x0

"""The per-launch float64 reference (tests/layer_reference.py) without a GPU: its op mirror reproduces the oracle, and
its comparator passes a kernel whose only error is the output rounding while failing each of a set of small,
localised corruptions of the kind a tile schedule gets wrong."""
import math

import pytest
import torch

import layer_reference as R


def _inputs(cfg, B, H, W, seed=0):
    g = torch.Generator().manual_seed(seed)
    C = cfg["out_channel"]
    return (torch.rand(B, C, H, W, generator=g) * 2 - 1, torch.randn(B, C, H, W, generator=g),
            torch.full((B, 1), 0.63))


@pytest.mark.parametrize("name", ["default"] + sorted(R.CONFIGS))
def test_op_mirror_matches_oracle(oracle, name):
    cfg, (B, H, W) = (oracle.DEFAULT_UNET, (2, 40, 72)) if name == "default" else R.CONFIGS[name][:2]
    sd = R.exact_weights(oracle.make_state_dict(cfg, seed=0, gn_jitter=0.2))
    cond, x, nl = _inputs(cfg, B, H, W)
    taps = {}
    eps = oracle.unet_forward(sd, cfg, torch.cat([cond, x], 1), nl, taps=taps)
    t = R.chain(sd, cfg, cond, x, nl)
    names = [op["name"] for op in R.plan_ops(cfg)]
    assert len(names) == len(set(names))
    assert set(taps) <= set(t)
    for k, v in list(taps.items()) + [("eps", eps)]:
        r = ((t[k] - v.double()).norm() / v.double().norm()).item()
        assert r < 1e-5, (name, k, r)        # fp32 oracle against the float64 mirror


def test_xin_packing():
    cond, x = torch.randn(2, 3, 4, 5), torch.randn(2, 3, 4, 5)
    p = R.xin_pack(cond, x)
    assert torch.equal(p[:, :3], x) and torch.equal(p[:, 4:7], cond)
    assert not p[:, 3].any() and not p[:, 7:].any()
    c8, x8 = torch.randn(1, 8, 2, 2), torch.randn(1, 8, 2, 2)
    p = R.xin_pack(c8, x8)
    assert torch.equal(p[:, :8], x8) and torch.equal(p[:, 8:], c8)


def test_exact_weights_are_exact_in_both_formats(oracle):
    sd = R.exact_weights(oracle.make_state_dict(oracle.DEFAULT_UNET, seed=0))
    for k, v in sd.items():
        if k.endswith(".weight") and v.dim() >= 2:
            assert torch.equal(v.half().float(), v) and torch.equal(v.bfloat16().float(), v), k


# --------------------------------------------------------------------------------------------- comparator sensitivity
B, H, W = 2, 40, 72   # every level has ragged tiles in y (level 0) or in x and y (levels 1-3)


@pytest.fixture(scope="module", params=["fp16", "bf16"])
def rounded(request, oracle):
    """Every op of the default network on the previous ops' outputs rounded to the mode's storage format, as the GPU
    stores them: (mode, cfg, sd, temb, tensors)."""
    cfg = oracle.DEFAULT_UNET
    sd = R.exact_weights(oracle.make_state_dict(cfg, seed=0, gn_jitter=0.2))
    cond, x, nl = _inputs(cfg, B, H, W, seed=3)
    t = R.chain(sd, cfg, cond, x, nl, mode=request.param)
    return request.param, cfg, sd, R.time_embedding(sd, cfg, nl), t


def _tile(out, b, ty, tx):
    return (b, slice(None), slice(ty * R.TILE_H, min((ty + 1) * R.TILE_H, out.shape[2])),
            slice(tx * R.TILE_W, min((tx + 1) * R.TILE_W, out.shape[3])))


def _corruptions(op, ref, sd, temb, cfg, t, mode):
    """(label, corrupted output) pairs; the perfect output is ref rounded to the storage format."""
    perfect = R.store(ref, op, mode)
    Ho, Wo = ref.shape[2:]
    tx = 1 if Wo > R.TILE_W else 0
    out = []
    if Wo > R.TILE_W:   # one 32 x 8 tile replaced by its x-neighbour (the columns that exist)
        c = perfect.clone()
        n = min(R.TILE_W, Wo - R.TILE_W)
        c[0, :, :R.TILE_H, :n] = perfect[0, :, :R.TILE_H, R.TILE_W:R.TILE_W + n]
        out.append(("tile <- x-neighbour", c))
    c = perfect.clone()  # one tile row shifted by one column
    c[0, :, :R.TILE_H, 1:] = perfect[0, :, :R.TILE_H, :-1]
    out.append(("tile row shifted", c))
    if op["kind"] != "gates":  # one tap (centre, first K chunk) dropped for one tile
        wkey = op["keys"][0] if op["kind"] in ("stem", "down", "up") else op["keys"][2]
        sd2 = dict(sd)
        w = sd[wkey].clone()
        ky = kx = w.shape[-1] // 2
        w[:, :64, ky, kx] = 0
        sd2[wkey] = w
        ref2, _ = R.reference(op, t, sd2, temb, cfg)
        c = perfect.clone()
        c[_tile(c, 1, 0, tx)] = R.store(ref2, op, mode)[_tile(c, 1, 0, tx)]
        out.append(("tap dropped", c))
    if op["kind"] != "final":  # one element off by 4 ulp (the final conv stores fp32 eps: 4 ulp are below its bound)
        c = perfect.clone()
        i = int(torch.argmax(ref.abs()))
        v = float(c.view(-1)[i])
        c.view(-1)[i] = v + 4 * 2.0 ** (math.floor(math.log2(abs(v))) - (10 if mode == "fp16" else 7))
        out.append(("4 ulp", c))
    c = perfect.clone()  # the valid part of the ragged last tile zeroed
    c[_tile(c, 1, (Ho - 1) // R.TILE_H, (Wo - 1) // R.TILE_W)] = 0
    out.append(("ragged last tile zeroed", c))
    c = perfect.clone()  # one tile of image 0 taken from image 1
    c[_tile(c, 0, 0, tx)] = perfect[_tile(c, 1, 0, tx)]
    out.append(("tile from the next image", c))
    return perfect, out


def test_comparator_passes_rounding_and_fails_corruptions(rounded):
    mode, cfg, sd, temb, t = rounded
    worst = 0.0
    for op in R.plan_ops(cfg):
        ref, terms = R.reference(op, t, sd, temb, cfg)
        perfect, bad = _corruptions(op, ref, sd, temb, cfg, t, mode)
        r, ex, loc = R.check(op, perfect, ref, terms, mode)
        worst = max(worst, r)
        assert r <= 1.0 and ex <= 1e-3, (mode, op["name"], r, ex, loc)   # the rounding part covers rounding alone
        for label, c in bad:
            r, ex, loc = R.check(op, c, ref, terms, mode)
            assert r > 1.0, (mode, op["name"], label, r, loc)
    print(f"[{mode}] rounding-only kernel: largest ratio {worst:.3f}")

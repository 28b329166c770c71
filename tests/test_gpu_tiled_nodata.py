"""Tiled sampling and metrics of scenes with nodata (fdsr_sample_tiled_masked, fdsr_metrics_masked, Engine.sample_tiled /
metrics_u8 / metrics_u16 (valid=...), super_resolution(valid=...), infer.py --nodata) on the GPU: bit identity with the
unmasked sampler where the rule demands it, parity with masked_tiled_sample_loop (tests/masked_oracle.py), launch counts,
the masked metrics against their restatement, and input validation.  Needs a B200: `pytest -m gpu`."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

import fastdiffsr_b200 as F
import masked_oracle as MO
import u16_reference as U
from test_gpu_launch_counts import op_launches, trace_frames

pytestmark = pytest.mark.gpu

DTYPES16 = ["fp16", "bf16"]


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def sd(oracle):
    return oracle.make_state_dict(dict(oracle.DEFAULT_UNET), seed=0, gn_jitter=0.1)


@pytest.fixture(scope="module")
def engines(oracle, schedule, sd):
    made = {}

    def get(dtype):
        if dtype not in made:
            e = F.Engine(dict(oracle.DEFAULT_UNET), "cuda:0", dtype)
            e.load_state_dict(sd)
            e.set_schedule(schedule["betas"])
            made[dtype] = e
        return made[dtype]
    yield get
    for e in made.values():
        e.close()


def _inputs(seed, B, H, W, T=20):
    g = torch.Generator().manual_seed(seed)
    cond = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    noise = torch.randn(T, B, 3, H, W, generator=g)
    return cond.cuda(), noise.cuda()


def _footprint(B, H, W):
    """Canvas 0: the upper-left triangle x/W + y/H < 0.9 with a 10 x 10 hole at (20, 20); canvas 1: its mirror image.
    With tile 64 / overlap 16 on 100 x 140 the far corner tile of each canvas holds no valid pixel."""
    y = torch.arange(H)[:, None].float()
    x = torch.arange(W)[None, :].float()
    v = torch.stack([(x / W + y / H < 0.9), ((W - 1 - x) / W + y / H < 0.9)][:B])
    v[:, 20:30, 20:30] = False
    return v.cuda()


def _check_masked(out, ref, cond, valid):
    """valid pixels: ref's bits; invalid pixels: cond's bits.  out / ref / cond: (B,C,H,W)."""
    v = valid[:, None].expand_as(out)
    assert torch.equal(out[v], ref[v])
    assert torch.equal(out[~v], cond[~v])


@pytest.mark.parametrize("dtype", ["fp32"] + DTYPES16)
def test_every_tile_active_equals_sample_tiled(engines, dtype):
    """(a) all-valid, and holes that leave every tile active: valid pixels are sample_tiled's bits, invalid ones cond."""
    e = engines(dtype)
    B, H, W = 2, 100, 140
    cond, noise = _inputs(11, B, H, W)
    holes = torch.rand(B, H, W, generator=torch.Generator().manual_seed(5)) > 0.3
    holes[:, 40:60, 10:130] = False
    n_tiles = B * 2 * 3
    for valid in (torch.ones(B, H, W, dtype=torch.bool, device="cuda"), holes.cuda()):
        assert len(MO.active_tiles(valid.cpu(), 64, 16)) == n_tiles
        for nz in (noise, None):
            ref, ref_tr = e.sample_tiled(cond, 64, overlap=16, noise=nz, seed=3, trace=True, image_offset=2, tile_batch=5)
            out, tr = e.sample_tiled(cond, 64, overlap=16, noise=nz, seed=3, trace=True, image_offset=2, tile_batch=5,
                                     valid=valid)
            _check_masked(out, ref, cond, valid)
            for f in range(tr.shape[1]):
                _check_masked(tr[:, f], ref_tr[:, f], cond, valid)
        # uint8 masks give the bool mask's bits
        assert torch.equal(e.sample_tiled(cond, 64, overlap=16, noise=noise, valid=valid.to(torch.uint8) * 7),
                           e.sample_tiled(cond, 64, overlap=16, noise=noise, valid=valid))
    e.check_overflow()


@pytest.mark.parametrize("dtype", DTYPES16)
def test_partition_skips_whole_tiles(engines, dtype):
    """(b) overlap 0, a mask invalid exactly on two of the six tiles: the valid pixels are sample of the other crops."""
    e = engines(dtype)
    cond, noise = _inputs(12, 1, 128, 192)
    valid = torch.ones(1, 128, 192, dtype=torch.bool, device="cuda")
    valid[:, 0:64, 64:128] = False
    valid[:, 64:128, 128:192] = False
    out = e.sample_tiled(cond, 64, overlap=0, noise=noise, valid=valid)
    wins = [(0, 0), (0, 128), (64, 0), (64, 64)]
    crops = torch.cat([cond[:, :, y:y + 64, x:x + 64] for y, x in wins]).contiguous()
    ncrops = torch.cat([noise[:, :, :, y:y + 64, x:x + 64] for y, x in wins], dim=1).contiguous()
    ref = e.sample(crops, noise=ncrops)
    for i, (y, x) in enumerate(wins):
        assert torch.equal(out[0, :, y:y + 64, x:x + 64], ref[i]), (y, x)
    inv = ~valid[:, None].expand_as(out)
    assert torch.equal(out[inv], cond[inv])
    e.check_overflow()


@pytest.mark.parametrize("dtype", DTYPES16)
def test_tile_batch_invariance(engines, dtype):
    """(c) the result does not depend on tile_batch."""
    e = engines(dtype)
    B, H, W = 2, 100, 140
    cond, noise = _inputs(13, B, H, W)
    valid = _footprint(B, H, W)
    n_active = len(MO.active_tiles(valid.cpu(), 64, 16))
    assert n_active == 10
    ref = e.sample_tiled(cond, 64, overlap=16, noise=noise, valid=valid, tile_batch=n_active)
    for tb in (1, 3, 4, 16):
        assert torch.equal(e.sample_tiled(cond, 64, overlap=16, noise=noise, valid=valid, tile_batch=tb), ref), tb
    built = e.sample_tiled(cond, 64, overlap=16, seed=4, valid=valid, tile_batch=3)
    assert torch.equal(built, e.sample_tiled(cond, 64, overlap=16, seed=4, valid=valid, tile_batch=7))
    e.check_overflow()


@pytest.fixture(scope="module")
def oracle_canvas(oracle, schedule, sd):
    cond, noise = _inputs(14, 2, 100, 140)
    valid = _footprint(2, 100, 140)
    ref = MO.masked_tiled_sample_loop(sd, dict(oracle.DEFAULT_UNET), schedule, cond.cpu(), noise.cpu(), valid.cpu(),
                                      64, 16)
    return cond, noise, valid, ref


@pytest.mark.parametrize("dtype", ["fp32"] + DTYPES16)
def test_masked_vs_oracle(engines, oracle, oracle_canvas, dtype):
    """(d) parity with masked_tiled_sample_loop, with test_tiled_vs_oracle's bars."""
    cond, noise, valid, ref = oracle_canvas
    e = engines(dtype)
    sr = e.sample_tiled(cond, 64, overlap=16, noise=noise, valid=valid).cpu()
    e.check_overflow()
    inv = ~valid.cpu()[:, None].expand_as(sr)
    assert torch.equal(sr[inv], cond.cpu()[inv])
    r = rel_l2(sr, ref)
    print(f"[{dtype}] masked tiled 100x140 B=2 T=20 SR rel-L2 vs oracle {r:.3e}")
    if dtype == "fp32":
        assert r <= 1e-4
        return
    assert r <= 1e-2
    gen = torch.Generator().manual_seed(9)
    c = cond.cpu()
    hr = (c + 0.1 * torch.nn.functional.avg_pool2d(torch.randn(c.shape, generator=gen), 3, 1, 1)).clamp(-1, 1)
    for b in range(2):
        p_ours = oracle.psnr_u8(oracle.to_u8(sr[b]), oracle.to_u8(hr[b]))
        p_ref = oracle.psnr_u8(oracle.to_u8(ref[b]), oracle.to_u8(hr[b]))
        assert abs(p_ours - p_ref) <= 0.05, (b, p_ours, p_ref)


@pytest.mark.parametrize("trace", [False, True], ids=["plain", "trace"])
def test_launch_count(engines, trace):
    """(e) 1 + sample_tiled's count over n_active tiles; no active tile: no UNet launch, and the output is cond."""
    e = engines("fp16")
    T, ops = e.T, op_launches(e.op_names(), "fp16")
    B, H, W, tb = 2, 100, 140, 3
    cond, _ = _inputs(15, B, H, W)
    for valid in (_footprint(B, H, W), torch.zeros(B, H, W, dtype=torch.bool, device="cuda")):
        k = len(MO.active_tiles(valid.cpu(), 64, 16))
        n_chunks = -(-k // tb)
        expect = 1 + 2 + T * (n_chunks * (1 + ops) + 1) + (trace_frames(T) if trace else 0) + 1
        before = e.launch_count()
        res = e.sample_tiled(cond, 64, overlap=16, tile_batch=tb, seed=1, trace=trace, valid=valid)
        torch.cuda.synchronize()
        assert e.launch_count() - before == expect, (k, e.launch_count() - before, expect)
        if k == 0:
            out, tr = res if trace else (res, None)
            assert torch.equal(out, cond)
            if trace:
                assert torch.equal(tr, cond[:, None].expand_as(tr))
    e.check_overflow()


def _levels(x, M):
    return U.quantise(x.permute(0, 2, 3, 1).cpu().numpy(), M)


def test_masked_metrics(engines):
    """(f) all-valid: metrics_u8 / metrics_u16 bitwise; random masks: the restatement; the NaN cases."""
    e = engines("fp16")
    g = torch.Generator().manual_seed(16)
    B, H, W = 3, 45, 61
    a = (torch.rand(B, 3, H, W, generator=g) * 2 - 1).cuda()
    b = (a.cpu() + 0.05 * torch.randn(B, 3, H, W, generator=g)).clamp(-1, 1).cuda()
    ones = torch.ones(B, H, W, dtype=torch.bool, device="cuda")
    assert torch.equal(e.metrics_u8(a, b, 4.0, valid=ones), e.metrics_u8(a, b, 4.0))
    for M in (255, 4095, 65535):
        assert torch.equal(e.metrics_u16(a, b, M, 3.0, valid=ones), e.metrics_u16(a, b, M, 3.0))
        for density in (0.97, 0.6):
            valid = torch.rand(B, H, W, generator=g) < density
            valid[:, 5:25, 5:30] = True                        # some wholly valid windows
            got = e.metrics_u16(a, b, M, 3.0, valid=valid.cuda()).cpu().numpy()
            la, lb = _levels(a, M), _levels(b, M)
            for i in range(B):
                ref = MO.masked_metrics(la[i], lb[i], valid[i].numpy(), M, 3.0)
                assert got[i, 0] == ref[0], (M, density, i)
                assert abs(got[i, 1] - ref[1]) <= 1e-13 * abs(ref[1])
                assert abs(got[i, 3] - ref[3]) <= 1e-13 * abs(ref[3])
                assert abs(got[i, 2] - ref[2]) <= 1e-9, (got[i, 2], ref[2])
    none = torch.zeros(B, H, W, dtype=torch.bool, device="cuda")
    assert torch.isnan(e.metrics_u8(a, b, valid=none)).all()
    sparse = none.clone()
    sparse[:, ::3, ::3] = True
    m = e.metrics_u8(a, b, valid=sparse)
    assert torch.isfinite(m[:, [0, 1, 3]]).all() and torch.isnan(m[:, 2]).all()


def test_validation_c_abi(engines):
    """(g) the new exports' argument checks."""
    e = engines("fp16")
    lib, h = e.lib, e._h
    cond = torch.zeros(1, 3, 64, 64, device="cuda")
    out = torch.empty_like(cond)
    valid = torch.ones(1, 64, 64, dtype=torch.uint8, device="cuda")
    res = torch.empty(1, 4, dtype=torch.float64, device="cuda")
    st = e._stream()
    P = lambda t: C.c_void_p(t.data_ptr())
    null = C.c_void_p(0)

    def call(cond_p, valid_p, out_p, B=1, H=64, W=64, th=64, tw=64, ov=16, tb=16):
        return lib.fdsr_sample_tiled_masked(h, cond_p, valid_p, null, 0, out_p, null, B, H, W, th, tw, ov, tb, st)

    assert call(P(cond), P(valid), P(out)) == 0
    assert call(P(cond), null, P(out)) == -1 and "valid" in lib.fdsr_last_error(h).decode()
    for cp, op in ((null, P(out)), (P(cond), null)):
        assert call(cp, P(valid), op) == -1 and "null argument" in lib.fdsr_last_error(h).decode()
    for kw, msg in [(dict(th=60), "multiples of 8"), (dict(H=7), ">= 8"), (dict(tb=0), "tile_batch"),
                    (dict(ov=-1), "overlap"), (dict(B=0), "B must be")]:
        assert call(P(cond), P(valid), P(out), **kw) == -1, kw
        assert msg in lib.fdsr_last_error(h).decode(), (kw, lib.fdsr_last_error(h))

    def metrics(valid_p, M=255, B=1):
        return lib.fdsr_metrics_masked(h, P(cond), P(out), valid_p, B, 64, 64, M, 4.0, P(res), st)

    assert metrics(P(valid)) == 0
    assert metrics(null) == -1 and "valid" in lib.fdsr_last_error(h).decode()
    assert metrics(P(valid), M=0) == -1 and "max_value" in lib.fdsr_last_error(h).decode()
    assert metrics(P(valid), B=0) == -1
    for bad in (torch.ones(1, 64, 63, dtype=torch.bool, device="cuda"), torch.ones(1, 64, 64, device="cuda"),
                torch.ones(1, 64, 64, dtype=torch.bool)):
        with pytest.raises(F.FdsrError):
            e.sample_tiled(cond, 64, valid=bad)
        with pytest.raises(F.FdsrError):
            e.metrics_u8(cond, out, valid=bad)


@pytest.fixture(scope="module")
def netG():
    opt = F.config.default_config()
    torch.manual_seed(0)
    n = F.define_G(opt).to("cuda")
    n.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cuda")
    return n.eval()


def test_drop_in(netG):
    """(g) super_resolution(valid=...): the engine's result, and the argument rules."""
    g = torch.Generator().manual_seed(8)
    x = (torch.rand(2, 3, 100, 140, generator=g) * 2 - 1).cuda()
    valid = _footprint(2, 100, 140)
    sr = netG.super_resolution(x, seed=7, tile=64, tile_overlap=16, valid=valid)
    assert torch.equal(sr, netG.engine().sample_tiled(x, 64, overlap=16, seed=7, valid=valid))
    seq = netG.super_resolution(x[:1], True, seed=7, tile=64, tile_overlap=16, valid=valid[:1])
    assert torch.equal(seq[-1], sr[0])
    with pytest.raises(ValueError):
        netG.super_resolution(x, seed=7, valid=valid)
    with pytest.raises(NotImplementedError):
        netG.super_resolution(x, seed=7, tile=64, tile_split=True, valid=valid)


def test_infer_script_nodata(tmp_path):
    """(h) infer.py --tile 64 --nodata 0: fill written as 0, scores over the valid pixels, an all-fill image left out."""
    from PIL import Image
    from fastdiffsr_b200.data import nodata_mask
    from fastdiffsr_b200.evaluate import main
    root = tmp_path / "ds"
    rng = np.random.default_rng(0)
    for d in ("hr_512", "lr_128"):
        os.makedirs(root / d)
    lrs = []
    for i, (h, w) in enumerate([(20, 26), (17, 23), (12, 12)]):
        lr = rng.integers(1, 256, (h, w, 3), dtype=np.uint8)
        lr[:3], lr[:, -4:] = 0, 0                               # a fill border
        lr[8:10, 8:11] = 0                                      # and a fill hole
        if i == 2:
            lr[:] = 0                                           # all fill: no score
        hr = np.repeat(np.repeat(lr, 4, 0), 4, 1)
        hr = np.clip(hr.astype(np.int64) + rng.integers(-6, 7, hr.shape), 0, 255).astype(np.uint8)
        Image.fromarray(hr).save(root / "hr_512" / f"img{i}.png")
        Image.fromarray(lr).save(root / "lr_128" / f"img{i}.png")
        lrs.append((lr, hr))
    opt = json.loads(json.dumps(F.config.default_config("sr_fastdiffsr_infer_x4")))
    opt["datasets"]["val"]["dataroot"] = str(root)
    opt["path"] = {"results": str(tmp_path / "results"), "log": None, "resume_state": None}
    cfg = tmp_path / "cfg.json"
    cfg.write_text(json.dumps(opt))
    res = main(["-c", str(cfg), "--tile", "64", "--tile-overlap", "16", "--tile-batch", "4", "--nodata", "0"],
               default_config=str(cfg), prog="infer.py")
    assert res["n"] == 3 and res["n_excluded"] == 1
    psnr = []
    for i, (lr, hr) in enumerate(lrs):
        valid = nodata_mask(torch.from_numpy(lr)[None], 0, hr.shape[0], hr.shape[1])[0].numpy()
        img = np.asarray(Image.open(tmp_path / "results" / f"0_{i + 1}_sr.png"))
        assert img.shape == hr.shape and (img[~valid] == 0).all()
        if i < 2:
            psnr.append(MO.masked_metrics(img.astype(np.int64), hr.astype(np.int64), valid, 255)[1])
    assert abs(res["sr_psnr"] - sum(psnr) / 2) <= 1e-9 * abs(res["sr_psnr"])

"""Tiled sampling of canvases of any size (fdsr_sample_tiled, Engine.sample_tiled, super_resolution(tile=...)) on the
GPU: bit-identity with the plain sampler where the definition demands it, parity with tiled_sample_loop (tests/tiled_oracle.py),
invariances, input validation, the drop-in surface and the evaluation driver.  Needs a B200: `pytest -m gpu`."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

import fastdiffsr_b200 as F
import tiled_oracle as TO

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


def _builtin_noise(e, B, H, W, seed, image_offset=0):
    """The built-in generator's draws in the injected-noise order: x_T (stream T), then the z of t = T-1 .. 1."""
    T = e.T
    return torch.stack([e.debug_noise(B, H, W, seed, T if k == 0 else T - k, image_offset) for k in range(T)])


@pytest.mark.parametrize("dtype", DTYPES16)
def test_one_tile_equals_sample(engines, dtype):
    e = engines(dtype)
    cond, noise = _inputs(1, 2, 64, 96)
    for nz in (noise, None):
        ref, ref_tr = e.sample(cond, noise=nz, seed=11, trace=True, image_offset=5)
        out, tr = e.sample_tiled(cond, (64, 96), overlap=32, noise=nz, seed=11, trace=True, image_offset=5)
        assert torch.equal(out, ref) and torch.equal(tr, ref_tr)
        out = e.sample_tiled(cond, (64, 96), noise=nz, seed=11, image_offset=5, tile_batch=1)
        assert torch.equal(out, ref)
    e.check_overflow()


@pytest.mark.parametrize("dtype", DTYPES16)
def test_partition_equals_stacked_crops(engines, dtype):
    e = engines(dtype)
    cond, noise = _inputs(2, 1, 128, 192)
    out = e.sample_tiled(cond, 64, overlap=0, noise=noise)
    wins = [(y0, x0) for y0 in (0, 64) for x0 in (0, 64, 128)]
    crops = torch.cat([cond[:, :, y:y + 64, x:x + 64] for y, x in wins]).contiguous()
    ncrops = torch.cat([noise[:, :, :, y:y + 64, x:x + 64] for y, x in wins], dim=1).contiguous()
    ref = e.sample(crops, noise=ncrops)
    for i, (y, x) in enumerate(wins):
        assert torch.equal(out[0, :, y:y + 64, x:x + 64], ref[i]), (y, x)
    e.check_overflow()


@pytest.fixture(scope="module")
def oracle_canvas(oracle, schedule, sd):
    """Two 100 x 140 canvases (not multiples of 8), tile 64, overlap 16: 2 x 3 tiles each, flush last tiles."""
    cond, noise = _inputs(3, 2, 100, 140)
    ref = TO.tiled_sample_loop(sd, dict(oracle.DEFAULT_UNET), schedule, cond.cpu(), noise.cpu(), 64, 16)
    return cond, noise, ref


@pytest.mark.parametrize("dtype", ["fp32"] + DTYPES16)
def test_tiled_vs_oracle(engines, oracle, oracle_canvas, dtype):
    cond, noise, ref = oracle_canvas
    e = engines(dtype)
    sr = e.sample_tiled(cond, 64, overlap=16, noise=noise).cpu()
    e.check_overflow()
    r = rel_l2(sr, ref)
    print(f"[{dtype}] tiled 100x140 B=2 T=20 SR rel-L2 vs oracle {r:.3e}")
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


@pytest.mark.parametrize("dtype", DTYPES16)
def test_invariances(engines, dtype):
    e = engines(dtype)
    B, H, W = 2, 100, 140
    cond, noise = _inputs(4, B, H, W)
    n_tiles = B * 2 * 3
    ref = e.sample_tiled(cond, 64, overlap=16, noise=noise, tile_batch=n_tiles)
    for tb in (1, 3):
        assert torch.equal(e.sample_tiled(cond, 64, overlap=16, noise=noise, tile_batch=tb), ref), tb
    assert torch.equal(e.sample_tiled(cond, 64, overlap=16, noise=noise, tile_batch=n_tiles), ref)
    # built-in noise is the debug hook's canvas noise, and canvas k's noise depends on its global index only
    built = e.sample_tiled(cond, 64, overlap=16, seed=21, image_offset=7, tile_batch=5)
    inj = e.sample_tiled(cond, 64, overlap=16, noise=_builtin_noise(e, B, H, W, 21, 7), tile_batch=5)
    assert torch.equal(built, inj)
    for k in range(B):
        alone = e.sample_tiled(cond[k:k + 1], 64, overlap=16, seed=21, image_offset=7 + k, tile_batch=5)
        assert torch.equal(alone[0], built[k]), k
    e.check_overflow()


def test_plain_sampler_unaffected(engines):
    e = engines("fp16")
    cond, noise = _inputs(5, 2, 64, 64)
    a = e.sample(cond, noise=noise)
    caps = e.graph_captures()
    big, bnoise = _inputs(6, 1, 100, 140)
    e.sample_tiled(big, 64, overlap=16, noise=bnoise, tile_batch=2)     # chunks of the plain batch's shape
    assert e.graph_captures() == caps                                   # neither captures nor evicts a graph
    assert torch.equal(e.sample(cond, noise=noise), a)
    assert e.graph_captures() == caps
    e.sample_tiled(big, 32, overlap=8, noise=bnoise, tile_batch=3)       # another chunk shape
    assert torch.equal(e.sample(cond, noise=noise), a)
    e.check_overflow()


def test_validation_c_abi(engines, oracle):
    e = engines("fp16")
    lib, h = e.lib, e._h
    cond = torch.zeros(1, 3, 64, 64, device="cuda")
    out = torch.empty_like(cond)
    st = e._stream()
    P = lambda t: C.c_void_p(t.data_ptr())
    null = C.c_void_p(0)

    def call(cond_p, out_p, B=1, H=64, W=64, th=64, tw=64, ov=16, tb=16):
        return lib.fdsr_sample_tiled(h, cond_p, null, 0, out_p, null, B, H, W, th, tw, ov, tb, st)

    assert call(P(cond), P(out)) == 0
    for cp, op in ((null, P(out)), (P(cond), null)):
        assert call(cp, op) == -1 and "null argument" in lib.fdsr_last_error(h).decode()
    for kw, msg in [(dict(th=60), "multiples of 8"), (dict(tw=0), "multiples of 8"), (dict(th=4, tw=4), "multiples of 8"),
                    (dict(H=7), ">= 8"), (dict(W=5), ">= 8"), (dict(H=65536, W=65536), "2^32"),
                    (dict(tb=0), "tile_batch"), (dict(ov=-1), "overlap"), (dict(B=0), "B must be")]:
        assert call(P(cond), P(out), **kw) == -1, kw
        assert msg in lib.fdsr_last_error(h).decode(), (kw, lib.fdsr_last_error(h))
    sr3 = F.Engine(dict(oracle.SR3_UNET, model="ddpm", image_size=64), "cuda:0", "fp16")
    try:
        assert sr3.lib.fdsr_sample_tiled(sr3._h, P(cond), null, 0, P(out), null, 1, 64, 64, 64, 64, 16, 16, st) == -1
        assert "SR3" in sr3.lib.fdsr_last_error(sr3._h).decode()
    finally:
        sr3.close()


@pytest.fixture(scope="module")
def netG():
    opt = F.config.default_config()
    torch.manual_seed(0)
    n = F.define_G(opt).to("cuda")
    n.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cuda")
    return n.eval()


def test_validation_drop_in(netG):
    x = torch.zeros(1, 3, 64, 64, device="cuda")
    for kw in (dict(tile=60), dict(tile=0), dict(tile=64, tile_batch=0), dict(tile=64, tile_overlap=-1)):
        with pytest.raises(F.FdsrError):
            netG.super_resolution(x, seed=0, **kw)
    with pytest.raises(F.FdsrError):
        netG.super_resolution(torch.zeros(1, 3, 7, 64, device="cuda"), seed=0, tile=64)
    opt = F.config.default_config("sr_ddpm_test_64_256")
    sr3 = F.define_G(opt).to("cuda")
    sr3.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cuda")
    with pytest.raises(NotImplementedError):
        sr3.super_resolution(x, seed=0, tile=64)


def test_drop_in(netG):
    g = torch.Generator().manual_seed(8)
    x = (torch.rand(1, 3, 100, 140, generator=g) * 2 - 1).cuda()
    sr = netG.super_resolution(x, seed=7, tile=64, tile_overlap=16)
    assert sr.shape == x.shape
    assert torch.equal(sr, netG.engine().sample_tiled(x, 64, overlap=16, seed=7))
    seq = netG.super_resolution(x, True, seed=7, tile=64, tile_overlap=16)
    plain = netG.super_resolution(x[..., :64, :64].contiguous(), True, seed=7)
    assert seq.shape == (plain.shape[0], 3, 100, 140)                  # (1 + frames, 3, H, W), the untiled layout
    assert torch.equal(seq[-1], sr[0])
    assert torch.equal(seq[0], x[0].clamp(-1, 1) / 2.0 + x[0])            # res2img(cond, cond), as untiled


def test_infer_script_tiled(tmp_path):
    """infer.py --tile on LR images of different sizes that are not multiples of 8: one canvas per call, SR = 4 x LR."""
    from PIL import Image
    from fastdiffsr_b200.evaluate import main
    root = tmp_path / "ds"
    rng = np.random.default_rng(0)
    sizes = [(13, 21), (19, 10)]                                        # LR (h, w)
    for d in ("hr_512", "lr_128"):
        os.makedirs(root / d)
    for i, (h, w) in enumerate(sizes):
        hr = Image.fromarray(rng.integers(0, 256, (4 * h, 4 * w, 3), dtype=np.uint8))
        hr.save(root / "hr_512" / f"img{i}.png")
        hr.resize((w, h), Image.BICUBIC).save(root / "lr_128" / f"img{i}.png")
    opt = json.loads(json.dumps(F.config.default_config("sr_fastdiffsr_infer_x4")))
    opt["datasets"]["val"]["dataroot"] = str(root)
    opt["path"] = {"results": str(tmp_path / "results"), "log": None, "resume_state": None}
    cfg = tmp_path / "cfg.json"
    cfg.write_text(json.dumps(opt))
    res = main(["-c", str(cfg), "--tile", "64", "--tile-overlap", "16", "--tile-batch", "4"],
               default_config=str(cfg), prog="infer.py")
    assert res["n"] == 2 and all(np.isfinite(res[k]) for k in res if k != "n")
    for i, (h, w) in enumerate(sizes):
        img = np.asarray(Image.open(tmp_path / "results" / f"0_{i + 1}_sr.png"))
        assert img.shape == (4 * h, 4 * w, 3), (i, img.shape)

"""Exact kernel-launch counts (Engine.launch_count, i.e. fdsr_launch_count) of every entry point, derived from the op
list and T: the counter is documented as the library's kernel launches, and the benchmark reports it per step.
Default network in fp16, bf16 and fp32, and the SR3 baseline in fp16.  Needs a B200: run with `pytest -m gpu`."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

CONFIGS = [("fp16", "fastdiffsr"), ("bf16", "fastdiffsr"), ("fp32", "fastdiffsr"), ("fp16", "ddpm")]
IDS = [f"{m}-{d}" for d, m in CONFIGS]
B, H = 2, 32   # H: a multiple of 2^(levels - 1) for both networks
GN_CONVS = (".block1", ".block2", ".attn.q", ".attn.k", ".attn.v", "final_conv")   # convs with a GroupNorm prologue


def op_launches(names, dtype):
    """Launches of one pass over the op list: one per conv (the fp32 parity mode adds a GroupNorm-table kernel to each
    conv with a GroupNorm prologue), four for CLAM/SLAM, one for a SelfAttention core."""
    n = 0
    for nm in names:
        if nm.endswith(".clam_slam"):
            n += 4
        elif nm.endswith(".attn.core"):
            n += 1
        else:
            n += 1 + int(dtype == "fp32" and nm.endswith(GN_CONVS))
    return n


def trace_frames(T):
    """The conditioning frame, then one after every step t with t % (1 | T // 10) == 0."""
    return 1 + sum(t % (1 | T // 10) == 0 for t in range(T))


def tile_count(L, t, overlap):
    """Tiles along one canvas axis (the tile-grid rule of fdsr_sample_tiled)."""
    te = min(t, L // 8 * 8)
    s = te - min(overlap, te - 8)
    return (L - te + s - 1) // s + 1 if L > te else 1


@pytest.fixture(scope="module")
def engines(oracle):
    from fastdiffsr_b200 import Engine
    betas = oracle.schedule_tables(oracle.make_beta_schedule(**oracle.DEFAULT_SCHEDULE))["betas"]
    cache = {}

    def get(dtype, model, fused_tail=True):
        key = (dtype, model, fused_tail)
        if key not in cache:
            if model == "ddpm":
                cfg = dict(oracle.SR3_UNET)
                sd = oracle.make_state_dict(cfg, seed=3, spec=oracle.sr3_state_dict_spec(cfg, 64))
                cfg = dict(cfg, model="ddpm", image_size=64)
            else:
                cfg = dict(oracle.DEFAULT_UNET)
                sd = oracle.make_state_dict(cfg, seed=0)
            if not fused_tail:
                os.environ["FDSR_FUSED_TAIL"] = "0"
            try:
                eng = Engine(cfg, "cuda:0", dtype)
            finally:
                os.environ.pop("FDSR_FUSED_TAIL", None)
            eng.load_state_dict(sd)
            eng.set_schedule(betas)
            cache[key] = eng
        return cache[key]

    yield get
    for eng in cache.values():
        eng.close()


def launches(eng, fn):
    l0 = eng.launch_count()
    fn()
    torch.cuda.synchronize()
    return eng.launch_count() - l0


def images(n=B, h=H, w=H, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(n, 3, h, w, generator=g) * 2 - 1).cuda()


@pytest.mark.parametrize("dtype,model", CONFIGS, ids=IDS)
def test_unet_forward(engines, dtype, model):
    eng = engines(dtype, model)
    cond, x = images(seed=1), images(seed=2)
    # pack_input, then the ops
    assert launches(eng, lambda: eng.unet_forward(cond, x, 3)) == 1 + op_launches(eng.op_names(), dtype)


@pytest.mark.parametrize("fused_tail", [True, False], ids=["fused", "unfused"])
@pytest.mark.parametrize("graph", [True, False], ids=["graph", "stream"])
@pytest.mark.parametrize("trace", [False, True], ids=["plain", "trace"])
@pytest.mark.parametrize("dtype,model", CONFIGS, ids=IDS)
def test_sample(engines, dtype, model, trace, graph, fused_tail):
    eng = engines(dtype, model, fused_tail)
    T, ops = eng.T, op_launches(eng.op_names(), dtype)
    fused = fused_tail and dtype != "fp32" and model == "fastdiffsr"
    # set_args, x_T, [pack_input once], T steps (fused: the ops; else pack_input, the ops, posterior), frames, result
    expect = 2 + (1 + T * ops if fused else T * (ops + 2)) + (trace_frames(T) if trace else 0) + 1
    cond = images(seed=3)
    eng.set_use_graph(graph)
    try:
        for _ in range(2):   # graph: the capturing call and a replay count the same
            assert launches(eng, lambda: eng.sample(cond, seed=5, trace=trace)) == expect
    finally:
        eng.set_use_graph(True)


@pytest.mark.parametrize("trace", [False, True], ids=["plain", "trace"])
@pytest.mark.parametrize("dtype", ["fp16", "bf16", "fp32"])
def test_sample_tiled(engines, dtype, trace):
    eng = engines(dtype, "fastdiffsr")
    T, ops = eng.T, op_launches(eng.op_names(), dtype)
    n, Hc, Wc, tile, overlap, tile_batch = 1, 48, 40, 32, 16, 3
    n_tiles = n * tile_count(Hc, tile, overlap) * tile_count(Wc, tile, overlap)
    n_chunks = -(-n_tiles // tile_batch)
    # set_args, x_T, T steps of (per chunk: tile_pack and the ops) and the blended posterior, frames, result
    expect = 2 + T * (n_chunks * (1 + ops) + 1) + (trace_frames(T) if trace else 0) + 1
    cond = images(n, Hc, Wc, seed=4)
    got = launches(eng, lambda: eng.sample_tiled(cond, tile, overlap=overlap, tile_batch=tile_batch, seed=6, trace=trace))
    assert got == expect


@pytest.mark.parametrize("dtype,model", CONFIGS, ids=IDS)
def test_image_and_debug_entry_points(engines, dtype, model):
    eng = engines(dtype, model)
    a, b = images(seed=7), images(seed=8)
    lr = (torch.rand(B, H // 4, H // 4, 3, generator=torch.Generator().manual_seed(9)) * 255).to(torch.uint8).cuda()
    assert launches(eng, lambda: eng.bicubic_u8(lr, H, H)) == 2
    assert launches(eng, lambda: eng.sse_u8(a, b)) == 1
    assert launches(eng, lambda: eng.metrics_u8(a, b)) == 2
    assert launches(eng, lambda: eng.debug_noise(B, H, H, seed=1, stream_id=0)) == 2


@pytest.mark.parametrize("dtype,model", CONFIGS, ids=IDS)
def test_read_tensor(engines, dtype, model):
    eng = engines(dtype, model)
    eng.unet_forward(images(seed=1), images(seed=2), 0)
    name = eng.tensor_names()[1]
    assert launches(eng, lambda: eng.read_tensor(name, B, B * 256 * H * H)) == 1

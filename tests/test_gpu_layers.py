"""Every launch of the CUDA UNet against a float64 reference of that launch on the inputs it actually read (B200,
`pytest -m gpu`), over a matrix of shapes that drives each per-layer schedule decision both ways.

Each op of tests/layer_reference.py's plan (the conv launches and the CLAM/SLAM gates) is evaluated in float64 on the
GPU's stored 16-bit input tensors, with GroupNorm statistics recomputed from them, and the stored output must lie
within the per-element bound of layer_reference.py.  Weights are snapped by `exact_weights`, so weight rounding drops
out.  Unlike the whole-network comparisons of test_gpu_parity.py, nothing accumulates over layers here: one wrong
tile, one stale halo column or one tile of the wrong image fails its layer.

Calibration: the rho values of layer_reference.RHO are estimates from the error model, not yet measured on a B200.
test_zz_calibration_table prints, per mode and op kind, the largest share of the modelled (rho) part of the bound that
any element used; the values and the maxima belong here once measured, with rho set so that no share exceeds 0.5.

Batch invariance (b) is bitwise: every intermediate tensor and eps of image b in a batch equals image b run alone.
"""
import os

import numpy as np
import pytest
import torch

import layer_reference as R

pytestmark = pytest.mark.gpu

# (B, H, W): what each shape exercises with the default network (64 x [1, 2, 4, 4])
SHAPES = [
    (1, 8, 8),        # smallest legal: level 3 is 1 x 1, every tile ragged
    (3, 40, 72),      # ragged tiles in x and y; tiles_x 9/5/3/2: pairs only at level 3
    (2, 64, 128),     # half tiles and split-N at the low-resolution levels
    (1, 256, 256),    # half tiles at level 1; ranges of 1 to 2 tiles
    (2, 256, 512),    # about 7 tiles per CTA at full resolution; ranges cross images and phases
    (16, 256, 256),   # the benchmark shape: reference for images 0, 7 and 15 only (all images: see (b))
]
BENCH_IMAGES = [0, 7, 15]
MODES = ["fp16", "bf16"]
T_STEP = 11

EXCESS = {}     # (mode, kind) -> largest excess seen
SCHEDULES = {}  # mode -> [(label, op name, schedule dict)]


def _engine(cfg, mode, sd, schedule, env=None):
    from fastdiffsr_b200 import Engine
    env = env or {}
    os.environ.update(env)
    try:
        eng = Engine(cfg, "cuda:0", mode)   # the switches are read when the context is created
    finally:
        for k in env:
            os.environ.pop(k, None)
    eng.load_state_dict(sd)
    eng.set_schedule(schedule["betas"])
    return eng


def _sd(oracle, cfg):
    return R.exact_weights(oracle.make_state_dict(cfg, seed=0, gn_jitter=0.2))


def _noise_level(schedule, B):
    return torch.full((B, 1), float(np.float32(schedule["sqrt_alphas_cumprod_prev"][T_STEP + 1])))


def _inputs(cfg, B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    C = cfg["out_channel"]
    return torch.rand(B, C, H, W, generator=g) * 2 - 1, torch.randn(B, C, H, W, generator=g)


def _read_all(eng, B, H, W, images=None):
    out = {}
    for name in eng.tensor_names():
        v = eng.read_tensor(name, B, B * 256 * H * W)
        out[name] = (v if images is None else v[images]).cpu().double()
    return out


def check_network(eng, cfg, sd, schedule, mode, B, H, W, label, images=None, seed=0):
    """One forward at (B, H, W); every op against its float64 reference.  Returns the failures (empty = pass) and
    records the largest excess per op kind and the schedule of every conv op."""
    cond, x = _inputs(cfg, B, H, W, seed)
    eps = eng.unet_forward(cond.cuda(), x.cuda(), T_STEP).cpu().double()
    ops = R.plan_ops(cfg)
    assert eng.op_names() == [op["name"] for op in ops]
    sel = images if images is not None else list(range(B))
    t = _read_all(eng, B, H, W, images)
    t["eps"] = eps[sel]
    # the packed network input: x_t and cond at their documented channels, rounded to the storage format
    xin = R.xin_pack(cond[sel].double(), x[sel].double()).to(R.STORE[mode]).double()
    assert torch.equal(t["xin"], xin), label
    temb = R.time_embedding(sd, cfg, _noise_level(schedule, B)[sel])
    fails = []
    for i, op in enumerate(ops):
        sch = eng.op_schedule(i) if (op["kind"] != "gates" and mode != "fp32") else None
        if sch is not None:
            SCHEDULES.setdefault(mode, []).append((label, op["name"], sch))
        ref, terms = R.reference(op, t, sd, temb, cfg)
        ratio, ex, loc = R.check(op, t[op["output"]], ref, terms, mode, sch["tile_h"] if sch else R.TILE_H)
        key = (mode, op["kind"])
        EXCESS[key] = max(EXCESS.get(key, 0.0), ex)
        if not ratio <= 1.0:
            fails.append((op["name"], round(ratio, 3), loc, sch))
    return fails


# ------------------------------------------------------------------------------------ (a) the default network
@pytest.fixture(scope="module", params=MODES)
def default_engine(request, oracle, schedule):
    cfg = dict(oracle.DEFAULT_UNET)
    sd = _sd(oracle, cfg)
    eng = _engine(cfg, request.param, sd, schedule)
    yield request.param, cfg, sd, eng
    eng.close()


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_every_op_vs_float64(default_engine, schedule, shape):
    mode, cfg, sd, eng = default_engine
    B, H, W = shape
    images = BENCH_IMAGES if B == 16 else None
    fails = check_network(eng, cfg, sd, schedule, mode, B, H, W, f"64x1244 {B}x{H}x{W}", images, seed=B * 7 + H)
    assert not fails, fails


# ------------------------------------------------------------------------------------ (d) other configurations
@pytest.mark.parametrize("mode", MODES + ["fp32"])
@pytest.mark.parametrize("name", sorted(R.CONFIGS))
def test_configurations_vs_float64(oracle, schedule, name, mode):
    cfg, small, multi = R.CONFIGS[name]
    sd = _sd(oracle, cfg)
    eng = _engine(cfg, mode, sd, schedule)
    try:
        fails = []
        for shape in ([small] if mode == "fp32" else [small, multi]):
            fails += check_network(eng, cfg, sd, schedule, mode, *shape, f"{name} {'x'.join(map(str, shape))}", seed=5)
        assert not fails, fails
    finally:
        eng.close()


# ------------------------------------------------------------------------------------ (f) the switches
SWITCHES = ["FDSR_PAIR", "FDSR_HALF_TILES", "FDSR_SPLIT_N", "FDSR_EPI2", "FDSR_TAIL_HELP", "FDSR_RESID_MMA",
            "FDSR_UP_PHASES"]   # (FDSR_FUSED_TAIL only changes the sampler, not a UNet forward)


@pytest.mark.parametrize("switch", SWITCHES)
def test_switch_off_vs_float64(oracle, schedule, switch):
    cfg = dict(oracle.DEFAULT_UNET)
    sd = _sd(oracle, cfg)
    eng = _engine(cfg, "fp16", sd, schedule, {switch: "0"})
    try:
        fails = check_network(eng, cfg, sd, schedule, "fp16", 2, 64, 128, f"{switch}=0 2x64x128", seed=9)
        assert not fails, fails
    finally:
        eng.close()


# ------------------------------------------------------------------------------------ (e) widths that are refused
@pytest.mark.parametrize("model", ["fastdiffsr", "ddpm"])
@pytest.mark.parametrize("inner,mults", [(64, [1, 3]), (192, [1]), (64, [1, 2, 3])])
def test_192_wide_levels_are_refused(oracle, model, inner, mults):
    from fastdiffsr_b200 import Engine, FdsrError
    cfg = dict(oracle.DEFAULT_UNET, inner_channel=inner, channel_multiplier=mults, model=model, image_size=64,
               attn_res=[16])
    with pytest.raises(FdsrError, match="every level width must be 64, 128 or 256"):
        Engine(cfg, "cuda:0", "fp16")


# ------------------------------------------------------------------------------------ (b) bitwise batch invariance
@pytest.mark.parametrize("mode,B,H,W", [("fp16", 16, 256, 256), ("bf16", 16, 256, 256), ("fp16", 32, 512, 512)])
def test_every_tensor_is_batch_invariant(oracle, schedule, mode, B, H, W):
    cfg = dict(oracle.DEFAULT_UNET)
    sd = _sd(oracle, cfg)
    full, one = _engine(cfg, mode, sd, schedule), _engine(cfg, mode, sd, schedule)
    try:
        cond, x = (v.cuda() for v in _inputs(cfg, B, H, W, seed=B + H))
        eps = full.unet_forward(cond, x, T_STEP)
        names = full.tensor_names()
        for b in range(B):
            e1 = one.unet_forward(cond[b:b + 1].contiguous(), x[b:b + 1].contiguous(), T_STEP)
            assert torch.equal(e1[0], eps[b]), ("eps", b)
            for name in names:
                a = full.read_tensor(name, B, B * 256 * H * W)[b]
                s = one.read_tensor(name, 1, 256 * H * W)[0]
                assert torch.equal(a, s), (name, b)
    finally:
        full.close()
        one.close()


# ------------------------------------------------------------------------------------ (c) coverage of the decisions
COVER = {"pair": {0, 1}, "tile_h": {16, 32}, "nsplit": {1, 2}, "group": {1, 2}, "epi2": {0, 1}, "tail2": {0, 1},
         "nR": {0, 2}, "phases": {1, 4}}


@pytest.mark.parametrize("mode", MODES)
def test_schedule_coverage(oracle, schedule, mode):
    """Across the shapes of (a) and the configurations of (d), every schedule decision is taken both ways, some CTA
    runs more tiles than its patch ring has stages, and some CTA range crosses an image and a phase boundary."""
    rows = []
    runs = [(dict(oracle.DEFAULT_UNET), "64x1244", s) for s in SHAPES]
    runs += [(R.CONFIGS[n][0], n, s) for n in sorted(R.CONFIGS) for s in R.CONFIGS[n][1:]]
    for cfg, cname, (B, H, W) in runs:
        eng = _engine(cfg, mode, _sd(oracle, cfg), schedule)
        try:
            cond, x = _inputs(cfg, B, H, W, seed=1)
            eng.unet_forward(cond.cuda(), x.cuda(), T_STEP)
            for i, name in enumerate(eng.op_names()):
                if not name.endswith((".clam_slam", ".attn.core")):
                    rows.append((f"{cname} {B}x{H}x{W}", name, eng.op_schedule(i)))
        finally:
            eng.close()
    seen = {k: {} for k in COVER}
    for label, name, s in rows:
        for k in COVER:
            seen[k].setdefault(s[k], []).append(f"{label} {name}")
    print(f"\n[{mode}] schedule decisions: value -> shapes (first layer)")
    for k in COVER:
        for v, where in sorted(seen[k].items()):
            shapes = sorted({w.rsplit(' ', 1)[0] for w in where})
            print(f"  {k:7s}= {v:3d}: {len(where):4d} layers, e.g. {where[0]};  shapes: {', '.join(shapes)}")
    for k, vals in COVER.items():
        assert vals <= set(seen[k]), (k, sorted(seen[k]))
    wraps = [(l, n) for l, n, s in rows if s["max_tiles"] > s["nG"] + s["nR"]]
    img = [(l, n) for l, n, s in rows if s["spans_image"]]
    ph = [(l, n) for l, n, s in rows if s["spans_phase"]]
    print(f"  ring wraps over tiles: {len(wraps)} layers, e.g. {wraps[:1]}; ranges across images: {len(img)}, "
          f"e.g. {img[:1]}; across phases: {len(ph)}, e.g. {ph[:1]}")
    assert wraps and img and ph


def test_zz_calibration_table():
    """Prints the largest share of the modelled bound used per (mode, op kind) by the checks above (runs last in this
    module): the calibration data of layer_reference.RHO (see the module docstring)."""
    if not EXCESS:
        pytest.skip("no per-op check ran in this session")
    print("\nlargest share of the rho part of the bound used, per mode and op kind:")
    for (mode, kind), v in sorted(EXCESS.items()):
        print(f"  {mode:5s} {kind:7s} excess {v:.3f}")

"""One tiled canvas split over ranks (fdsr_sample_tiled_part, Engine.sample_tiled_part, parallel.split_sample_tiled,
super_resolution(tile_split=True), evaluate(tile_split=True)): the gathered result equals sample_tiled bit for bit.
The first tests run 2-4 processes on one GPU, each with its own context, exchanging eps through host memory over gloo
(parallel.tile_exchange); the NCCL test needs two or more GPUs.  Needs a B200: `pytest -m gpu`."""
import ctypes as C
import json
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import fastdiffsr_b200 as F
from fastdiffsr_b200 import parallel as P

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _inputs(seed, B, H, W, T=20):
    g = torch.Generator().manual_seed(seed)
    cond = torch.rand(B, 3, H, W, generator=g) * 2 - 1
    noise = torch.randn(T, B, 3, H, W, generator=g)
    return cond.cuda(), noise.cuda()


# (dtype, world, (B, H, W), tile, overlap, noise: "inj" | (seed, image_offset), trace)
CANVAS = (2, 100, 140)            # ranges span canvases and partial tile rows
CASES = {
    2: [("fp16", CANVAS, 64, 16, "inj", False), ("bf16", CANVAS, 64, 16, "inj", False),
        ("fp16", CANVAS, 64, 16, (21, 7), True), ("fp32", CANVAS, 64, 16, "inj", False)],
    3: [("fp16", CANVAS, 64, 16, "inj", True), ("bf16", CANVAS, 64, 16, (5, 3), False),
        ("fp16", (1, 64, 64), 64, 16, (9, 0), True)],                       # one tile: ranks 0 and 1 own nothing
    4: [("fp16", CANVAS, 64, 16, "inj", False), ("bf16", CANVAS, 64, 16, "inj", True),
        ("fp16", CANVAS, 64, 48, (13, 2), False)],                           # stride 16: non-adjacent senders
}


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import fdsr_oracle as O
    from test_gpu_launch_counts import op_launches, trace_frames
    failures, engines = [], {}
    try:
        torch.cuda.set_device(0)
        sd = O.make_state_dict(dict(O.DEFAULT_UNET), seed=0, gn_jitter=0.1)
        betas = O.schedule_tables(O.make_beta_schedule(**O.DEFAULT_SCHEDULE))["betas"]
        for i, (dtype, (B, H, W), tile, overlap, nz, trace) in enumerate(CASES[world]):
            if dtype not in engines:
                engines[dtype] = F.Engine(dict(O.DEFAULT_UNET), "cuda:0", dtype)
                engines[dtype].load_state_dict(sd)
                engines[dtype].set_schedule(betas)
            e = engines[dtype]
            cond, noise = _inputs(100 + i, B, H, W)
            kw = dict(noise=noise) if nz == "inj" else dict(seed=nz[0], image_offset=nz[1])
            plan = e.tiled_plan(B, H, W, tile, overlap, world, rank)
            tile_batch = 1 + rank                                             # may differ per rank
            l0 = e.launch_count()
            res = e.sample_tiled_part(cond, tile, overlap=overlap, tile_batch=tile_batch, trace=trace, rank=rank,
                                      world=world, exchange=P.tile_exchange(plan), **kw)
            torch.cuda.synchronize()
            got = e.launch_count() - l0
            chunks = -(-(plan["own"][1] - plan["own"][0]) // tile_batch)
            want = 2 + e.T * (chunks * (1 + op_launches(e.op_names(), dtype)) + 1) + (trace_frames(e.T) if trace else 0) + 1
            if got != want:
                failures.append(f"case {i} rank {rank}: {got} launches, expected {want}")
            e.check_overflow()
            parts = res if trace else (res,)
            whole = []
            for t in parts:
                bits = t.cpu().view(torch.int32).clone()
                dist.all_reduce(bits, op=dist.ReduceOp.SUM)
                whole.append(bits)
            if rank == 0:
                ref = e.sample_tiled(cond, tile, overlap=overlap, trace=trace, **kw)
                for name, a, b in zip(("sr", "trace"), whole, ref if trace else (ref,)):
                    if not torch.equal(a, b.cpu().view(torch.int32)):
                        failures.append(f"case {i} ({dtype}, world {world}, tile {tile}/{overlap}, {nz}): {name} differs "
                                        f"at {int((a != b.cpu().view(torch.int32)).sum())} values")
                e.check_overflow()
            dist.barrier()
    finally:
        for e in engines.values():
            e.close()
        dist.destroy_process_group()
    with open(os.path.join(out_dir, f"rank{rank}.json"), "w") as f:
        json.dump(failures, f)


@pytest.mark.parametrize("world", sorted(CASES))
def test_split_equals_sample_tiled_one_gpu(world, tmp_path):
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    failures = [f for r in range(world) for f in json.load(open(tmp_path / f"rank{r}.json"))]
    assert not failures, "\n".join(failures)


@pytest.fixture(scope="module")
def engine(oracle, schedule):
    e = F.Engine(dict(oracle.DEFAULT_UNET), "cuda:0", "fp16")
    e.load_state_dict(oracle.make_state_dict(dict(oracle.DEFAULT_UNET), seed=0))
    e.set_schedule(schedule["betas"])
    yield e
    e.close()


def test_validation(engine):
    e = engine
    cond = torch.zeros(1, 3, 100, 140, device="cuda")
    out = torch.empty_like(cond)
    store = torch.empty(6, 3, 64, 64, device="cuda")
    P = lambda t: C.c_void_p(t.data_ptr())
    null = C.c_void_p(0)

    def call(store_p, rank, world, fn=F._lib.TILE_EXCHANGE_FN()):
        return e.lib.fdsr_sample_tiled_part(e._h, P(cond), null, 0, P(out), null, 1, 100, 140, 64, 64, 16, 4, rank, world,
                                            store_p, fn, null, e._stream())

    assert call(P(store), 0, 1) == 0                                   # one rank: nothing to exchange
    for args, msg in [((P(store), 0, 2), "exchange callback is required"), ((null, 0, 1), "eps_store"),
                      ((P(store), 2, 2), "rank must be"), ((P(store), -1, 2), "rank must be"),
                      ((P(store), 0, 0), "world must be")]:
        assert call(*args) == -1, args
        assert msg in e.lib.fdsr_last_error(e._h).decode(), (args, e.lib.fdsr_last_error(e._h))
    with pytest.raises(F.FdsrError, match="exchange callback is required"):
        e.sample_tiled_part(cond, 64, overlap=16, rank=1, world=2)
    torch.cuda.synchronize()

    def broken(step, store):
        raise KeyError("no peer")
    with pytest.raises(KeyError, match="no peer"):                     # re-raised after the aborted call
        e.sample_tiled_part(cond, 64, overlap=16, rank=0, world=2, exchange=broken)
    torch.cuda.synchronize()
    # the context stays usable
    assert torch.equal(e.sample_tiled_part(cond, 64, overlap=16, seed=3), e.sample_tiled(cond, 64, overlap=16, seed=3))


def _make_dataset(root):
    """Two LR/HR pairs whose sizes are not multiples of 8 (SR = 4 x LR)."""
    from PIL import Image
    rng = np.random.default_rng(0)
    for d in ("hr_512", "lr_128"):
        os.makedirs(root / d)
    for i, (h, w) in enumerate([(13, 21), (19, 10)]):
        hr = Image.fromarray(rng.integers(0, 256, (4 * h, 4 * w, 3), dtype=np.uint8))
        hr.save(root / "hr_512" / f"img{i}.png")
        hr.resize((w, h), Image.BICUBIC).save(root / "lr_128" / f"img{i}.png")


def _infer_config(tmp_path, root):
    opt = json.loads(json.dumps(F.config.default_config("sr_fastdiffsr_infer_x4")))
    opt["datasets"]["val"]["dataroot"] = str(root)
    opt["path"] = {"results": str(tmp_path / "results"), "log": None, "resume_state": None}
    cfg = tmp_path / "cfg.json"
    cfg.write_text(json.dumps(opt))
    return str(cfg)


def _netG(dev):
    opt = F.config.default_config()
    torch.manual_seed(0)
    n = F.define_G(opt).to(dev)
    n.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], dev)
    return n.eval()


def _drop_in_checks(rank, dev, failures):
    """super_resolution(tile_split=True) against the one-GPU tile= result, with and without the trace, and seed=None."""
    netG = _netG(dev)
    g = torch.Generator().manual_seed(8)
    x = (torch.rand(2, 3, 100, 140, generator=g) * 2 - 1).to(dev)
    for cont in (False, True):
        split = netG.super_resolution(x, cont, seed=7, image_offset=3, tile=64, tile_overlap=16, tile_split=True)
        one = netG.super_resolution(x, cont, seed=7, image_offset=3, tile=64, tile_overlap=16)
        if not torch.equal(split.view(torch.int32), one.view(torch.int32)):
            failures.append(f"rank {rank}: tile_split (continous={cont}) differs from the one-GPU result")
    a = netG.super_resolution(x, tile=64, tile_overlap=16, tile_split=True)     # seed=None: rank 0's, broadcast
    b = a.clone()
    dist.broadcast(b, src=0)
    if not torch.equal(a, b):
        failures.append(f"rank {rank}: seed=None gives a different result than rank 0's")


def _gloo_drop_in_worker(rank, world, port, out_dir, cfg):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    failures = []
    _drop_in_checks(rank, "cuda:0", failures)
    from fastdiffsr_b200.evaluate import main
    torch.manual_seed(rank)       # a different random init per rank: --tile-split must run rank 0's network everywhere
    res = main(["-c", cfg, "--tile", "64", "--tile-overlap", "16", "--tile-batch", "4", "--tile-split", "--no-save"],
               default_config=cfg, prog="infer.py")                      # destroys the process group
    with open(os.path.join(out_dir, f"eval{rank}.json"), "w") as f:
        json.dump({k: v for k, v in res.items() if k not in ("seconds", "images_per_s")}, f)
    with open(os.path.join(out_dir, f"rank{rank}.json"), "w") as f:
        json.dump(failures, f)


def test_split_drop_in_one_gpu(tmp_path):
    """split_sample_tiled through super_resolution(tile_split=True) and `infer.py --tile-split`, two ranks on one GPU
    over gloo: the same bits as one rank, and the same metrics as a single-process --tile run of rank 0's network."""
    root = tmp_path / "ds"
    _make_dataset(root)
    cfg = _infer_config(tmp_path, root)
    mp.spawn(_gloo_drop_in_worker, args=(2, _free_port(), str(tmp_path), cfg), nprocs=2, join=True)
    failures = [f for r in range(2) for f in json.load(open(tmp_path / f"rank{r}.json"))]
    assert not failures, "\n".join(failures)
    from fastdiffsr_b200.evaluate import main
    torch.manual_seed(0)
    ref = main(["-c", cfg, "--tile", "64", "--tile-overlap", "16", "--tile-batch", "4", "--no-save"], default_config=cfg,
               prog="infer.py")
    ref = {k: v for k, v in ref.items() if k not in ("seconds", "images_per_s")}
    for r in range(2):
        assert json.load(open(tmp_path / f"eval{r}.json")) == ref, r


# ---- NCCL: one process per GPU
def _nccl_worker(rank, world, port, out_dir, cfg):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    failures = []
    _drop_in_checks(rank, f"cuda:{rank}", failures)
    from fastdiffsr_b200.evaluate import main
    torch.manual_seed(rank)
    res = main(["-c", cfg, "--tile", "64", "--tile-overlap", "16", "--tile-batch", "4", "--tile-split", "--no-save"],
               default_config=cfg, prog="infer.py")                      # destroys the process group
    with open(os.path.join(out_dir, f"eval{rank}.json"), "w") as f:
        json.dump({k: v for k, v in res.items() if k not in ("seconds", "images_per_s")}, f)
    with open(os.path.join(out_dir, f"rank{rank}.json"), "w") as f:
        json.dump(failures, f)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="NCCL puts one rank on each GPU: needs two or more GPUs")
def test_nccl_split(tmp_path):
    root = tmp_path / "ds"
    _make_dataset(root)
    cfg = _infer_config(tmp_path, root)
    world = min(4, torch.cuda.device_count())
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path), cfg), nprocs=world, join=True)
    failures = [f for r in range(world) for f in json.load(open(tmp_path / f"rank{r}.json"))]
    assert not failures, "\n".join(failures)
    from fastdiffsr_b200.evaluate import main
    torch.manual_seed(0)
    ref = main(["-c", cfg, "--tile", "64", "--tile-overlap", "16", "--tile-batch", "4", "--no-save"], default_config=cfg,
               prog="infer.py")
    ref = {k: v for k, v in ref.items() if k not in ("seconds", "images_per_s")}
    for r in range(world):
        assert json.load(open(tmp_path / f"eval{r}.json")) == ref, r

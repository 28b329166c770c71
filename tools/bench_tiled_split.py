"""One tiled canvas split over the GPUs of a box (fdsr_sample_tiled_part with the NCCL eps exchange of
parallel.tile_exchange, the path of parallel.split_sample_tiled): one JSON line per case, written by rank 0, with the
device name and power limit (read in the same run), seconds per canvas (median of --reps timed calls after a warm-up,
between barriers, ending on a device synchronise), the tiles and UNet chunks of every rank, the bytes each rank
receives per step, the exchange's milliseconds per step as the stream sees it (CUDA events around the callback's work
on the stream, mean over the steps of the timed calls: the transfers plus the time this rank's stream waits for peers
that reach the step later, e.g. ranks with more chunks, so an upper bound on the transfer time), and whether the
gathered result equals sample_tiled of the same inputs on rank 0 bit for bit (checked outside the timed region).

Cases: `2048` = 2048^2 (9 x 9 tiles), `8192` = 8192^2 (37 x 37 tiles); tile 256, overlap 32, tile_batch 16, T = 20.
Random-init weights: the time does not depend on the values.

  torchrun --nproc_per_node N tools/bench_tiled_split.py --case 2048 8192 [--out profiles/tiled/bench_tiled_split.jsonl]
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fastdiffsr_b200 as F  # noqa: E402
from fastdiffsr_b200.parallel import gather_owned, tile_exchange  # noqa: E402
from bench_tiled import device_info  # noqa: E402

CASES = {"2048": dict(H=2048, W=2048), "8192": dict(H=8192, W=8192)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", nargs="+", default=["2048", "8192"], choices=sorted(CASES))
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tile", type=int, default=256)
    ap.add_argument("--overlap", type=int, default=32)
    ap.add_argument("--tile-batch", type=int, default=16)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file (rank 0)")
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29531")
    os.environ.setdefault("RANK", "0")
    os.environ.setdefault("WORLD_SIZE", "1")
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    opt = F.config.default_config()
    opt["model"]["compute_dtype"] = args.dtype
    torch.manual_seed(0)
    netG = F.define_G(opt).to(dev)
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], dev)
    eng = netG.engine()
    info = device_info(dev)
    infos = [None] * world
    dist.all_gather_object(infos, info)
    tile, ov, tb = args.tile, args.overlap, args.tile_batch
    for name in args.case:
        H, W = CASES[name]["H"], CASES[name]["W"]
        g = torch.Generator(device=dev).manual_seed(1)
        cond = (torch.rand(1, 3, H, W, device=dev, generator=g) * 2 - 1).contiguous()   # the same on every rank
        plan = eng.tiled_plan(1, H, W, tile, ov, world, rank)
        exch = tile_exchange(plan)
        events = []

        def timed_exchange(step, store):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            exch(step, store)
            e1.record()
            events.append((e0, e1))

        def run():
            sr = eng.sample_tiled_part(cond, tile, overlap=ov, tile_batch=tb, seed=1, rank=rank, world=world,
                                       exchange=timed_exchange)
            return gather_owned(sr)

        run()                                        # warm-up: modules, allocations, layer uploads, NCCL channels
        torch.cuda.synchronize()
        events.clear()
        ts = []
        for _ in range(args.reps):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sr = run()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        eng.check_overflow()
        exch_ms = statistics.mean(a.elapsed_time(b) for a, b in events) if events else 0.0
        tile_floats = eng.C * plan["te"][0] * plan["te"][1]
        mine = dict(rank=rank, tiles=plan["own"][1] - plan["own"][0],
                    chunks=-(-(plan["own"][1] - plan["own"][0]) // tb),
                    recv_bytes_per_step=sum(hi - lo for lo, hi in plan["recv"]) * tile_floats * 4,
                    exchange_ms_per_step_incl_peer_wait=round(exch_ms, 4), seconds=ts)
        ranks = [None] * world
        dist.all_gather_object(ranks, mine)
        identical = None
        if rank == 0:
            ref = eng.sample_tiled(cond, tile, overlap=ov, tile_batch=tb, seed=1)
            identical = bool(torch.equal(ref.view(torch.int32), sr.view(torch.int32)))
            eng.check_overflow()
            del ref
        dist.barrier()
        if rank == 0:
            sec = statistics.median(max(r["seconds"][i] for r in ranks) for i in range(args.reps))
            rec = dict(info, devices=sorted({i["device"] for i in infos}),
                       power_limits_w=sorted({i.get("power_limit_w") for i in infos}, key=str), case=name,
                       gpus=world, dtype=args.dtype, T=eng.T, canvas=[H, W], tile=tile, overlap=ov, tile_batch=tb,
                       n_tiles=plan["n_tiles"], seconds_per_canvas=sec, ranks=ranks, bit_identical=identical)
            line = json.dumps(rec)
            print(line, flush=True)
            if args.out:
                os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
                with open(args.out, "a") as f:
                    f.write(line + "\n")
        del cond, sr
        torch.cuda.empty_cache()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Tiled sampling (fdsr_sample_tiled) of large canvases on one GPU: one JSON line per case with the device name and
power limit (read in the same run), the canvas and tile parameters, the tile count and redundancy (tile pixels over
canvas pixels), the memory the call needs (activation workspace of one chunk + the canvas state and per-tile eps
store), seconds per canvas from CUDA events (one warm-up call, then --reps timed calls) and output megapixels per
second.  For canvases up to 2048^2 the untiled fdsr_sample of the same canvas is timed too (a 2048^2 canvas is
~16 GB of activations; 8192^2 would be ~252 GB and does not fit a B200), and the ratio of the two rates reported.

Cases: `2048` = a 512^2 LR scene at x4, tile 256, overlap 32 (9 x 9 tiles); `8192` = 8192^2, tile 256, overlap 32
(37 x 37 tiles).  Random-init weights: the time does not depend on the values.

  python tools/bench_tiled.py --case 2048 8192 [--dtype fp16] [--reps 3] [--out profiles/tiled/bench_tiled.jsonl]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fastdiffsr_b200 as F  # noqa: E402

CASES = {"2048": dict(H=2048, W=2048, tile=256, overlap=32, untiled=True),
         "8192": dict(H=8192, W=8192, tile=256, overlap=32, untiled=False)}


def axis(L, t, overlap):
    """Tile count and effective extent of one axis (the grid rule of include/fdsr.h)."""
    te = min(t, 8 * (L // 8))
    s = te - min(overlap, te - 8)
    return (math.ceil((L - te) / s) + 1 if L > te else 1), te


def device_info(dev):
    info = {"device": torch.cuda.get_device_name(dev), "power_limit_w": None}
    try:
        q = subprocess.run(["nvidia-smi", f"--id={dev.index or 0}", "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, mx = [v.strip() for v in q.stdout.strip().split(",")]
        info["power_limit_w"], info["sm_max_mhz"] = float(pl), float(mx)
    except Exception as e:  # the number is still stated, with the reason the limit is missing
        info["power_limit_error"] = repr(e)
    return info


def timed(fn, reps):
    fn()                                   # warm-up: loads modules, grows the allocations, uploads the layers
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    return ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", nargs="+", default=["2048", "8192"], choices=sorted(CASES))
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tile-batch", type=int, default=16)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    opt = F.config.default_config()
    opt["model"]["compute_dtype"] = args.dtype
    torch.manual_seed(0)
    netG = F.define_G(opt).to(dev)
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], dev)
    eng = netG.engine()
    info = device_info(dev)
    for name in args.case:
        c = CASES[name]
        H, W, tile, ov = c["H"], c["W"], c["tile"], c["overlap"]
        cond = (torch.rand(1, 3, H, W, device=dev) * 2 - 1).contiguous()
        ny, tey = axis(H, tile, ov)
        nx, tex = axis(W, tile, ov)
        n_tiles = ny * nx
        n_chunks = math.ceil(n_tiles / args.tile_batch)
        bc = math.ceil(n_tiles / n_chunks)
        ts = timed(lambda: eng.sample_tiled(cond, tile, overlap=ov, tile_batch=args.tile_batch, seed=1), args.reps)
        eng.check_overflow()
        ws = eng.workspace_bytes()
        canvas_bytes = 3 * H * W * 4 + n_chunks * bc * 3 * tey * tex * 4   # x_t canvas + per-tile eps store
        sec = sorted(ts)[len(ts) // 2]
        rec = dict(info, case=name, dtype=args.dtype, T=eng.T, canvas=[H, W], tile=tile, overlap=ov,
                   tile_batch=args.tile_batch, n_tiles=n_tiles, tiles_yx=[ny, nx], n_chunks=n_chunks, chunk=bc,
                   padding_slots=n_chunks * bc - n_tiles, redundancy=round(n_tiles * tey * tex / (H * W), 4),
                   workspace_bytes=ws, canvas_buffer_bytes=canvas_bytes, caller_buffer_bytes=2 * 3 * H * W * 4,
                   seconds_per_canvas=sec, seconds_all=ts, mpx_per_s=H * W / sec / 1e6)
        if c["untiled"]:
            tu = timed(lambda: eng.sample(cond, seed=1), args.reps)
            eng.check_overflow()
            su = sorted(tu)[len(tu) // 2]
            rec.update(untiled_seconds_per_canvas=su, untiled_seconds_all=tu, untiled_mpx_per_s=H * W / su / 1e6,
                       untiled_workspace_bytes=eng.workspace_bytes(), tiled_over_untiled_rate=su / sec,
                       expected_min_ratio=round(0.85 / rec["redundancy"], 4))
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
            with open(args.out, "a") as f:
                f.write(line + "\n")
        del cond
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""Sampling speed against the band count C (out_channel = C, in_channel = 2C): one JSON line per C with the device name
and power limit (read in the same run), images per second and milliseconds per UNet step.

Shape: BASELINE configs[1] (x4 64 -> 256, 16 images per call, T = 20).  One timed call = PIL-exact bicubic of the
uint8 LR batch on the device + the 20-step sampler with built-in noise (fdsr_bicubic_u8 + fdsr_sample, one captured
graph); CUDA events around --reps calls after --warmup calls.  The C values run interleaved for --rounds rounds, so
that drifting clocks affect every C alike; each line reports the median round and the spread.  Random-init weights:
the time does not depend on the values.

  python tools/bench_bands.py [--bands 1 3 4 8] [--dtype fp16] [--out profiles/bands/bench_bands.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import fastdiffsr_b200 as F  # noqa: E402
from bench_tiled import device_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bands", type=int, nargs="+", default=[1, 3, 4, 8])
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    B, h, H = args.batch, 64, 256
    runs = {}
    for C in args.bands:
        opt = F.config.default_config()
        opt["model"]["unet"]["in_channel"], opt["model"]["unet"]["out_channel"] = 2 * C, C
        opt["model"]["compute_dtype"] = args.dtype
        torch.manual_seed(0)
        netG = F.define_G(opt).to(dev)
        netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], dev)
        eng = netG.engine()
        lr = torch.randint(0, 256, (B, h, h, C), dtype=torch.uint8, device=dev)

        def call(eng=eng, lr=lr):
            _, cond = eng.bicubic_u8(lr, H, H, want_u8=False)
            return eng.sample(cond, seed=1)
        for _ in range(args.warmup):
            call()
        eng.check_overflow()
        runs[C] = (eng, call, [])
    T = next(iter(runs.values()))[0].T
    for _ in range(args.rounds):
        for C, (eng, call, ts) in runs.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.reps):
                call()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) / 1e3 / args.reps)
    info = device_info(dev)
    lines = []
    for C, (eng, call, ts) in runs.items():
        s = statistics.median(ts)
        lines.append(dict(info, bench="bands", bands=C, in_channel=2 * C, dtype=args.dtype, batch=B, lr=h, sr=H, T=T,
                          reps=args.reps, rounds=args.rounds, seconds_per_call=s, images_per_s=B / s,
                          ms_per_unet_step=1e3 * s / T, spread_pct=100.0 * (max(ts) - min(ts)) / s))
    base = next((l for l in lines if l["bands"] == 3), None)
    for l in lines:
        if base is not None:
            l["vs_c3_pct"] = 100.0 * (l["images_per_s"] / base["images_per_s"] - 1.0)
        print(json.dumps(l), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()

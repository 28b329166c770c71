#!/usr/bin/env python
"""16-bit boundary kernels against their 8-bit counterparts, and evaluate() on the same 4-band data stored at 8 and
16 bits.  One JSON line per measurement, each with the device name and power limit read in the same run.

Kernels (CUDA events around --reps calls after one warm-up call; the 8- and 16-bit forms run interleaved for
--rounds rounds and each line reports the median round and the spread):
  bicubic: fdsr_bicubic_u8 vs fdsr_bicubic_u16, conditioning output only (what evaluate() asks for);
  metrics: fdsr_metrics_u8 vs fdsr_metrics_u16 (M = 4095) of two fp32 images.
Cases: B = 16, C = 4, 64 -> 256 (the working set fits in the 126 MB L2, so this is a launch-and-L2 figure) and one
scene, C = 4, 2048^2 -> 8192^2 (about 1 GB of conditioning, far larger than L2).  GB/s counts the algorithmic bytes:
the inputs read once and the outputs written once (not the resize's intermediate, not the window re-reads), over
the HBM3e data-sheet bandwidth of 7.7 TB/s.

evaluate(): images/s of the whole loop (load, resize, 20-step sampling, metrics) on N random 64 -> 256 4-band images
stored as uint8 .npy and as uint16 .npy (max_value 65535), random-init weights, no images written; the two
datasets alternate for --rounds rounds after one warm-up pass each.

  python tools/bench_u16.py [--out profiles/u16/bench_u16.jsonl]
"""
import argparse
import json
import os
import statistics
import sys
import tempfile

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import fastdiffsr_b200 as F  # noqa: E402
from fastdiffsr_b200 import data as D  # noqa: E402
from bench_tiled import device_info  # noqa: E402

HBM_TBPS = 7.7
M = 4095


def _time(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def kernels(eng, dev, B, C, h, H, reps, rounds):
    g = torch.Generator(device=dev).manual_seed(0)
    lr8 = torch.randint(0, 256, (B, h, h, C), dtype=torch.uint8, device=dev, generator=g)
    lr16 = torch.from_numpy(np.random.default_rng(0).integers(0, 65536, (B, h, h, C), dtype=np.uint16)).to(dev)
    a = torch.rand((B, C, H, H), device=dev, generator=g) * 2 - 1
    b = (a + 0.05 * torch.randn(a.shape, device=dev, generator=g)).clamp_(-1, 1)
    out = a.numel() * 4
    ops = {
        ("bicubic", 8): (lambda: eng.bicubic_u8(lr8, H, H, want_u8=False), lr8.numel() + out),
        ("bicubic", 16): (lambda: eng.bicubic_u16(lr16, H, H, M, want_u16=False), lr16.numel() * 2 + out),
        ("metrics", 8): (lambda: eng.metrics_u8(a, b), 2 * out),
        ("metrics", 16): (lambda: eng.metrics_u16(a, b, M), 2 * out),
    }
    ts = {k: [] for k in ops}
    for fn, _ in ops.values():
        fn()
    for _ in range(rounds):
        for k, (fn, _) in ops.items():
            ts[k].append(_time(fn, reps))
    res = []
    for (op, bits), (_, nbytes) in ops.items():
        s = statistics.median(ts[(op, bits)])
        ts_k = ts[(op, bits)]
        gbps = nbytes / s / 1e9
        res.append(dict(bench="u16_kernels", op=op, bits=bits, B=B, C=C, lr=h, sr=H, reps=reps, rounds=rounds,
                        ms=1e3 * s, algorithmic_bytes=nbytes, gb_per_s=gbps, pct_of_hbm=100.0 * gbps / (HBM_TBPS * 1e3),
                        spread_pct=100.0 * (max(ts_k) - min(ts_k)) / s))
    return res


def evaluate_rate(dev, n, batch, rounds):
    from fastdiffsr_b200.evaluate import evaluate
    C, l, r = 4, 64, 256
    opt = F.config.default_config()
    opt["model"]["unet"]["in_channel"], opt["model"]["unet"]["out_channel"] = 2 * C, C
    torch.manual_seed(0)
    netG = F.define_G(opt).to(dev)
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], dev)
    netG.eval()
    rng = np.random.default_rng(0)
    with tempfile.TemporaryDirectory() as tmp:
        sets = {}
        for bits in (8, 16):
            root = os.path.join(tmp, f"u{bits}")
            for d in (f"hr_{r}", f"lr_{l}"):
                os.makedirs(os.path.join(root, d))
            for i in range(n):
                hr = rng.integers(0, 256, (r, r, C), dtype=np.uint8)
                lr = hr[::4, ::4]
                if bits == 16:
                    hr, lr = hr.astype(np.uint16) * 257, lr.astype(np.uint16) * 257
                np.save(os.path.join(root, f"hr_{r}", f"{i:04d}.npy"), np.ascontiguousarray(hr))
                np.save(os.path.join(root, f"lr_{l}", f"{i:04d}.npy"), np.ascontiguousarray(lr))
            sets[bits] = D.LRHRDataset(root, "img", l, r, channels=C, max_value=None if bits == 8 else 65535)
        rates = {8: [], 16: []}
        for ds in sets.values():
            evaluate(netG, ds, batch_size=batch, scale=4)
        for _ in range(rounds):
            for bits, ds in sets.items():
                rates[bits].append(evaluate(netG, ds, batch_size=batch, scale=4)["images_per_s"])
    return [dict(bench="u16_evaluate", bits=bits, max_value=None if bits == 8 else 65535, C=C, lr=l, sr=r, n=n,
                 batch=batch, T=netG.engine().T, rounds=rounds, images_per_s=statistics.median(v),
                 spread_pct=100.0 * (max(v) - min(v)) / statistics.median(v)) for bits, v in rates.items()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--eval-images", type=int, default=64)
    ap.add_argument("--eval-rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    eng = F.Engine(dict(in_channel=8, out_channel=4, inner_channel=64, norm_groups=32, channel_multiplier=[1, 2, 4, 4],
                        res_blocks=2), dev, "fp16")
    lines = kernels(eng, dev, 16, 4, 64, 256, args.reps, args.rounds)
    lines += kernels(eng, dev, 1, 4, 2048, 8192, max(args.reps // 4, 3), args.rounds)
    eng.close()
    torch.cuda.empty_cache()
    lines += evaluate_rate(dev, args.eval_images, 16, args.eval_rounds)
    info = device_info(dev)
    lines = [dict(info, **l) for l in lines]
    for l in lines:
        print(json.dumps(l), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()

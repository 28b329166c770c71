#!/usr/bin/env python
"""Tiled sampling of scenes with nodata (fdsr_sample_tiled_masked) against the unmasked call on one GPU: one JSON line
per (canvas, mask) with the device name and power limit (read in the same run), n_active / n_tiles, the chunk counts
of both calls, seconds per canvas of both (CUDA events; one warm-up call each, then --reps calls of each, masked and
unmasked alternated; median reported), and the bit check of the rule: the masked call's valid pixels equal the
unmasked call's bits when every tile is active, and its invalid pixels equal cond.

Masks (fp16, T = 20, tile 256, overlap 32, tile_batch 16; random-init weights, the time does not depend on them):
  all      every pixel valid, through the masked call (every tile active: the masked call's overhead);
  rotated  a square rotated by 12 degrees that touches the canvas edges (a Landsat path/row footprint, ~71 % valid);
  swath    a diagonal swath edge, x + y < 0.8 (W + H) / 2 (~32 % valid).
The expectation that the time follows the chunk count is what the numbers test.

--compare-dump ROOT also runs `bench.py --gpus 1 --steps 2 --warmup 1 --dump-outputs` from this tree and from the
checkout at ROOT (e.g. the parent commit, built) and records whether the dumped files are byte-identical.

  python tools/bench_tiled_nodata.py [--case 2048 8192] [--reps 3] [--out profiles/tiled/bench_tiled_nodata.jsonl]
"""
import argparse
import filecmp
import json
import math
import os
import subprocess
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import fastdiffsr_b200 as F  # noqa: E402
from bench_tiled import axis, device_info  # noqa: E402

CASES = {"2048": 2048, "8192": 8192}
MASKS = ("all", "rotated", "swath")


def make_mask(kind, L, dev):
    y = torch.arange(L, device=dev, dtype=torch.float64)[:, None]
    x = torch.arange(L, device=dev, dtype=torch.float64)[None, :]
    if kind == "all":
        return torch.ones(1, L, L, dtype=torch.bool, device=dev)
    if kind == "swath":
        return (x + y < 0.8 * L)[None]
    th = math.radians(12.0)
    side = L / (math.cos(th) + math.sin(th))           # the rotated square's bounding box is the canvas
    cy = cx = (L - 1) / 2
    u = (x - cx) * math.cos(th) + (y - cy) * math.sin(th)
    v = -(x - cx) * math.sin(th) + (y - cy) * math.cos(th)
    return ((u.abs() <= side / 2) & (v.abs() <= side / 2))[None]


def active_count(valid, tile, overlap):
    """Tiles of the grid whose window holds a valid pixel (the rule of include/fdsr.h, restated on the host)."""
    L = valid.shape[1]
    n, te = axis(L, tile, overlap)
    s = te - min(overlap, te - 8)
    starts = [min(i * s, L - te) if i + 1 < n else L - te for i in range(n)]
    v = valid[0]
    return sum(bool(v[y0:y0 + te, x0:x0 + te].any()) for y0 in starts for x0 in starts), n * n


def compare_dump(other_root):
    """bench.py --dump-outputs from this tree and from `other_root`: {file: identical}."""
    res, other_root = {}, os.path.abspath(other_root)
    with tempfile.TemporaryDirectory() as tmp:
        dirs = []
        for i, root in enumerate((ROOT, other_root)):
            d = os.path.join(tmp, str(i))
            subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup",
                            "1", "--dump-outputs", d], check=True, cwd=root, stdout=subprocess.DEVNULL)
            dirs.append(d)
        for f in sorted(os.listdir(dirs[0])):
            res[f] = filecmp.cmp(os.path.join(dirs[0], f), os.path.join(dirs[1], f), shallow=False)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", nargs="+", default=["2048", "8192"], choices=sorted(CASES))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tile-batch", type=int, default=16)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--compare-dump", metavar="ROOT", default=None)
    ap.add_argument("--compare-label", default=None, help="what ROOT is, for the record (default: its directory name)")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    opt = F.config.default_config()
    opt["model"]["compute_dtype"] = "fp16"
    torch.manual_seed(0)
    netG = F.define_G(opt).to(dev)
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], dev)
    eng = netG.engine()
    info = device_info(dev)
    tile, overlap, tb = 256, 32, args.tile_batch

    def emit(rec):
        print(json.dumps(rec), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as f:
                f.write(json.dumps(rec) + "\n")
    for name in args.case:
        L = CASES[name]
        g = torch.Generator(device=dev).manual_seed(1)
        cond = torch.rand(1, 3, L, L, generator=g, device=dev) * 2 - 1
        for kind in MASKS:
            valid = make_mask(kind, L, dev)
            n_active, n_tiles = active_count(valid, tile, overlap)

            def plain():
                return eng.sample_tiled(cond, tile, overlap=overlap, tile_batch=tb, seed=5)

            def masked():
                return eng.sample_tiled(cond, tile, overlap=overlap, tile_batch=tb, seed=5, valid=valid)
            ref, out = plain(), masked()                  # warm-up of both, and the outputs of the bit check
            torch.cuda.synchronize()
            v = valid[:, None].expand_as(out)
            bits = {"invalid_equal_cond": bool(torch.equal(out[~v], cond[~v]))}
            if n_active == n_tiles:
                bits["valid_equal_unmasked"] = bool(torch.equal(out[v], ref[v]))
            del ref, out, v
            ts = {"plain": [], "masked": []}
            for _ in range(args.reps):
                for key, fn in (("plain", plain), ("masked", masked)):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn()
                    e1.record()
                    e1.synchronize()
                    ts[key].append(e0.elapsed_time(e1) / 1e3)
            eng.check_overflow()
            med = {k: sorted(t)[len(t) // 2] for k, t in ts.items()}
            rec = dict(info, case=name, mask=kind, dtype="fp16", T=eng.T, canvas=[L, L], tile=tile, overlap=overlap,
                       tile_batch=tb, valid_fraction=round(float(valid.float().mean()), 4), n_tiles=n_tiles,
                       n_active=n_active, chunks_unmasked=-(-n_tiles // tb), chunks_masked=-(-n_active // tb),
                       seconds_per_canvas_unmasked=med["plain"], seconds_per_canvas_masked=med["masked"],
                       seconds_all_unmasked=ts["plain"], seconds_all_masked=ts["masked"],
                       masked_over_unmasked_time=med["masked"] / med["plain"],
                       chunk_ratio=(-(-n_active // tb)) / (-(-n_tiles // tb)), bit_check=bits)
            emit(rec)
    if args.compare_dump:
        label = args.compare_label or os.path.basename(os.path.abspath(args.compare_dump))
        emit(dict(info, check="bench.py --dump-outputs of this tree and of " + label,
                  identical=compare_dump(args.compare_dump)))


if __name__ == "__main__":
    main()

"""Batch sharding of LR images over ranks (one process per GPU, torch.distributed), and the split of one tiled canvas
over ranks.

The sampling path has no exchange step: every image's T-step chain is independent (GroupNorm is
per-sample, SURVEY 8(e)).  Ranks therefore run the full loop on their shard with no data-path
collective; NCCL (gloo in CPU tests) is used only after the loop to all-gather SR shards and to
all-reduce metric accumulators — the two collectives the reference's single-GPU evaluation loop
(sr_mfe.py:258-386) would need when spread over GPUs.

A tiled canvas (split_sample_tiled) is the exception: its tiles share one chain, so the ranks that split its tiles
exchange the eps of the tiles at their borders once per step (DESIGN §4.4).
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from ._lib import FdsrOverflowError


def shard_bounds(n_items: int, rank: int, world: int):
    """Contiguous, padded-even split: every rank gets ceil(n/world) slots; trailing slots of the
    last ranks may be empty.  Returns (start, stop, per_rank)."""
    per = (n_items + world - 1) // world
    start = min(rank * per, n_items)
    stop = min(start + per, n_items)
    return start, stop, per


def shard_batch(x: torch.Tensor, rank: int, world: int):
    """Slice dim 0 for this rank and zero-pad to the common per-rank size (collectives need equal shapes).
    Returns (local, n_valid)."""
    start, stop, per = shard_bounds(x.shape[0], rank, world)
    local = x[start:stop]
    n_valid = local.shape[0]
    if n_valid < per:
        pad = torch.zeros((per - n_valid,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
        local = torch.cat([local, pad], dim=0)
    return local.contiguous(), n_valid


def gather_batch(local: torch.Tensor, n_items: int, group=None):
    """all_gather per-rank shards (equal shapes) back into the global batch, dropping the padding."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local[:n_items]
    world = dist.get_world_size(group)
    out = torch.empty((world * local.shape[0],) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, local.contiguous(), group=group)
    return out[:n_items]


def reduce_sums(acc: torch.Tensor, group=None):
    """all_reduce(SUM) of a small fp64 accumulator vector, e.g. [sum_sse, sum_psnr, n_images]."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=group)
    return acc


def psnr_from_sse(sse: torch.Tensor, numel_per_image: int):
    """PSNR per image from uint8 squared-error sums (core/metrics.py:94-101)."""
    mse = sse / float(numel_per_image)
    return torch.where(mse > 0, 10.0 * torch.log10(255.0 ** 2 / mse.clamp_min(1e-300)),
                       torch.full_like(mse, float("inf")))


@torch.no_grad()
def sharded_super_resolution(netG, cond_global: torch.Tensor, noise_global=None, seed: int = 0, group=None):
    """Run netG.super_resolution on this rank's shard of `cond_global` (B,C,H,W) and return the
    gathered (B,C,H,W) result on every rank.  `noise_global`, if given, is (T,B,C,H,W)."""
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    local, _ = shard_batch(cond_global, rank, world)
    noise = None
    if noise_global is not None:
        start, stop, per = shard_bounds(cond_global.shape[0], rank, world)
        noise = noise_global[:, start:stop]
        if noise.shape[1] < per:
            pad = torch.zeros((noise.shape[0], per - noise.shape[1]) + tuple(noise.shape[2:]), dtype=noise.dtype,
                              device=noise.device)
            noise = torch.cat([noise, pad], dim=1)
        noise = noise.contiguous()
    # same seed on every rank + the global index of the shard's first image: the built-in noise of image k does not
    # depend on the world size, so the gathered result equals the single-rank one bit for bit (SURVEY 4(4))
    start, _, _ = shard_bounds(cond_global.shape[0], rank, world)
    sr_local = netG.super_resolution(local, False, noise=noise, seed=seed, image_offset=start)
    if sr_local.dim() == 3:   # SR3 baseline, one image per rank: ret_img[-1] has no batch axis
        sr_local = sr_local[None]
    return gather_batch(sr_local, cond_global.shape[0], group)


def tile_exchange(plan, group=None):
    """exchange(step, eps_store) of Engine.sample_tiled_part for the ranks of `group`: the plan's slot ranges as
    point-to-point sends / receives.  NCCL moves the device slots directly, ordered on and waited for by the current
    stream; a backend that sends host tensors only (gloo) gets them staged through host memory, after the stream's
    prior work and copied back on the stream."""
    peer = (lambda q: q) if group is None else (lambda q: dist.get_global_rank(group, q))
    sends = [(peer(q), lo, hi) for q, (lo, hi) in enumerate(plan["send"]) if hi > lo]
    recvs = [(peer(q), lo, hi) for q, (lo, hi) in enumerate(plan["recv"]) if hi > lo]
    on_device = "nccl" in str(dist.get_backend(group))

    def exchange(step, store):
        if not (sends or recvs):
            return
        if on_device:
            ops = [dist.P2POp(dist.isend, store[lo:hi], q, group) for q, lo, hi in sends]
            ops += [dist.P2POp(dist.irecv, store[lo:hi], q, group) for q, lo, hi in recvs]
            for req in dist.batch_isend_irecv(ops):
                req.wait()
            return
        out = [store[lo:hi].cpu() for _, lo, hi in sends]     # synchronises with the stream's prior work
        inc = [torch.empty(store[lo:hi].shape) for _, lo, hi in recvs]
        reqs = [dist.isend(t, q, group) for t, (q, _, _) in zip(out, sends)]
        reqs += [dist.irecv(t, q, group) for t, (q, _, _) in zip(inc, recvs)]
        for req in reqs:
            req.wait()
        for t, (_, lo, hi) in zip(inc, recvs):
            store[lo:hi].copy_(t)
    return exchange


def gather_owned(t: torch.Tensor, group=None):
    """The whole fp32 tensor from the ranks' parts of it (each rank's part, +0.0 elsewhere): an integer sum of the bit
    patterns, so the exact bits, -0.0 included, with no floating-point addition."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t.view(torch.int32), op=dist.ReduceOp.SUM, group=group)
    return t


@torch.no_grad()
def split_sample_tiled(engine, cond, tile, overlap: int = 32, tile_batch: int = 16, noise=None, seed: int = 0,
                       trace: bool = False, image_offset: int = 0, group=None):
    """engine.sample_tiled(cond, ...) split over the ranks of `group` (default: the default process group): every rank
    passes the same arguments (tile_batch may differ), samples its share of the tiles (Engine.sample_tiled_part) with
    an eps exchange every step (tile_exchange: NCCL, or gloo through host memory), and gets the whole result (and
    trace), bit for bit sample_tiled's.  The ranks' networks must hold the same weights.  fp16 mode: the
    overflow flags are combined over the ranks, so all of them raise FdsrOverflowError together."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    B, _, H, W = cond.shape
    # the ranks must agree on the job, or the exchange would pair mismatched ranges and hang
    th, tw = (tile, tile) if isinstance(tile, int) else (int(tile[0]), int(tile[1]))
    key = torch.tensor([B, H, W, th, tw, int(overlap), int(image_offset), int(seed) % (2 ** 62), noise is not None,
                        bool(trace)], dtype=torch.int64, device=engine.device)
    both = torch.cat([key, -key])
    dist.all_reduce(both, op=dist.ReduceOp.MAX, group=group)
    if not torch.equal(both[:key.numel()], -both[key.numel():]):
        raise ValueError("split_sample_tiled: the ranks were called with different canvas, tile, seed or noise arguments")
    plan = engine.tiled_plan(B, H, W, (th, tw), overlap, world, rank)
    res = engine.sample_tiled_part(cond, (th, tw), overlap=overlap, tile_batch=tile_batch, noise=noise, seed=seed,
                                   trace=trace, image_offset=image_offset, rank=rank, world=world,
                                   exchange=tile_exchange(plan, group))
    overflow = torch.zeros(1, dtype=torch.int32, device=engine.device)
    try:
        engine.check_overflow()
    except FdsrOverflowError:
        overflow.fill_(1)
    dist.all_reduce(overflow, op=dist.ReduceOp.MAX, group=group)
    if overflow.item():
        raise FdsrOverflowError("split_sample_tiled: an activation left the fp16 range on at least one rank")
    if not trace:
        return gather_owned(res, group)
    sr, tr = res
    both = gather_owned(torch.cat([sr.reshape(-1), tr.reshape(-1)]), group)   # one collective for both
    return both[:sr.numel()].view(sr.shape), both[sr.numel():].view(tr.shape)

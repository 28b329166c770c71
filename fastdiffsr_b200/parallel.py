"""Batch sharding of LR images over ranks (one process per GPU, torch.distributed).

The sampling path has no exchange step: every image's T-step chain is independent (GroupNorm is
per-sample, SURVEY 8(e)).  Ranks therefore run the full loop on their shard with no data-path
collective; NCCL (gloo in CPU tests) is used only after the loop to all-gather SR shards and to
all-reduce metric accumulators — the two collectives the reference's single-GPU evaluation loop
(sr_mfe.py:258-386) would need when spread over GPUs.
"""
from __future__ import annotations

import torch
import torch.distributed as dist


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

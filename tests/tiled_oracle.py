"""CPU restatement of tiled sampling (fdsr_sample_tiled in include/fdsr.h): the checker the tiled tests compare the CUDA
path against.  New functionality with no reference counterpart, so it lives with the tests rather than in the oracle,
whose functions are pinned to the reference; it is built from the oracle's pieces (unet_forward, p_sample_step,
res2img), one tile at a time with B = 1.  Test infrastructure only."""
import numpy as np
import torch

from fdsr_oracle import p_sample_step, res2img, unet_forward


def tile_starts(L, t, overlap):
    """Tile grid of one axis of length L for tile size t: (starts, t_e, o_e).  The effective extent t_e is the largest
    multiple of 8 that fits (at most t), the overlap is capped so that the stride t_e - o_e stays >= 8, and the last
    tile is flush with the far edge."""
    t_e = min(t, 8 * (L // 8))
    o_e = min(overlap, t_e - 8)
    s = t_e - o_e
    starts = []
    while len(starts) * s < L - t_e:
        starts.append(len(starts) * s)
    return starts + [L - t_e], t_e, o_e


def tile_weights(t_e_y, t_e_x, overlap):
    """(t_e_y, t_e_x) fp32 blending weights r_y(i) * r_x(j), r(i) = min(i+1, t_e-i, o_e+1) with o_e = min(overlap,
    t_e-8) per axis: integer ramps over the overlap, flat inside."""
    def ramp(t_e):
        i = np.arange(t_e)
        return np.minimum(np.minimum(i + 1, t_e - i), min(overlap, t_e - 8) + 1).astype(np.int64)
    return torch.from_numpy((ramp(t_e_y)[:, None] * ramp(t_e_x)[None, :]).astype(np.float32))


@torch.no_grad()
def tiled_sample_loop(sd, cfg, tables, cond, noises, tile, overlap, continous=False):
    """sample_loop on canvases of any size (H, W >= 8) as overlapping tiles on one shared chain.  Every step, each
    tile's eps is the UNet on its window of [cond | x_t] alone (B = 1); per pixel, over the covering tiles in global
    order (row start, then column start), n_k = w_k / sum(w) and eps = sum n_k eps_k in fp32, both sums starting from
    their first term; then one posterior update (p_sample_step) on the canvas.  `tile`: int or (th, tw); cond, noises
    and the output as in sample_loop."""
    th, tw = (tile, tile) if isinstance(tile, int) else tile
    B, _, H, W = cond.shape
    ys, tey, _ = tile_starts(H, th, overlap)
    xs, tex, _ = tile_starts(W, tw, overlap)
    wt = tile_weights(tey, tex, overlap)
    T = len(tables["betas"])
    sample_inter = 1 | (T // 10)
    x = noises[0]
    frames = []
    for k, t in enumerate(reversed(range(T))):
        nl = torch.full((1, 1), float(np.float32(tables["sqrt_alphas_cumprod_prev"][t + 1])), dtype=torch.float32)
        eps = torch.empty_like(x)
        for b in range(B):
            wins = [(slice(y0, y0 + tey), slice(x0, x0 + tex)) for y0 in ys for x0 in xs]
            wsum = torch.zeros(H, W)
            seen = torch.zeros(H, W, dtype=torch.bool)
            for wy, wx in wins:
                wsum[wy, wx] = torch.where(seen[wy, wx], wsum[wy, wx] + wt, wt)
                seen[wy, wx] = True
            acc = torch.zeros(3, H, W)
            seen.zero_()
            for wy, wx in wins:
                e = unet_forward(sd, cfg, torch.cat([cond[b:b + 1, :, wy, wx], x[b:b + 1, :, wy, wx]], dim=1), nl)[0]
                term = (wt / wsum[wy, wx]) * e
                acc[:, wy, wx] = torch.where(seen[wy, wx], acc[:, wy, wx] + term, term)
                seen[wy, wx] = True
            eps[b] = acc
        z = noises[k + 1] if t > 0 else None
        x, _, _ = p_sample_step(sd, cfg, tables, x, t, cond, z, eps=eps)
        if t % sample_inter == 0:
            frames.append(x)
    img = res2img(x, cond)
    if not continous:
        return img
    per = []
    for b in range(B):
        seq = [cond[b:b + 1]] + [f[b:b + 1] for f in frames]
        per.append(torch.cat([res2img(s, cond[b:b + 1]) for s in seq], dim=0))
    return torch.cat(per, dim=0)

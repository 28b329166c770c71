"""CPU restatement of tiled sampling with a validity mask (fdsr_sample_tiled_masked in include/fdsr.h) and of the masked
metrics (fdsr_metrics_masked): the checkers the nodata tests compare the CUDA path against.  Built from
tiled_oracle's grid and weights and the oracle's UNet and posterior.  Test infrastructure only."""
import math

import numpy as np
import torch

from fdsr_oracle import p_sample_step, res2img, unet_forward
from tiled_oracle import tile_starts, tile_weights


def active_tiles(valid, tile, overlap):
    """[(b, y0, x0)] of the tiles whose window holds a valid pixel, in global order.  valid: (B,H,W) bool."""
    th, tw = (tile, tile) if isinstance(tile, int) else tile
    B, H, W = valid.shape
    ys, tey, _ = tile_starts(H, th, overlap)
    xs, tex, _ = tile_starts(W, tw, overlap)
    return [(b, y0, x0) for b in range(B) for y0 in ys for x0 in xs if bool(valid[b, y0:y0 + tey, x0:x0 + tex].any())]


@torch.no_grad()
def masked_tiled_sample_loop(sd, cfg, tables, cond, noises, valid, tile, overlap, continous=False):
    """tiled_sample_loop over the active tiles only: per pixel, the blend runs over its active covering tiles in global
    order (both sums starting from the first active term); the result and the trace frames are res2img(x) at valid
    pixels and cond at invalid ones.  valid: (B,H,W) bool; everything else as in tiled_sample_loop."""
    th, tw = (tile, tile) if isinstance(tile, int) else tile
    B, C, H, W = cond.shape
    _, tey, _ = tile_starts(H, th, overlap)
    _, tex, _ = tile_starts(W, tw, overlap)
    wt = tile_weights(tey, tex, overlap)
    act = active_tiles(valid, tile, overlap)
    T = len(tables["betas"])
    sample_inter = 1 | (T // 10)
    x = noises[0]
    frames = []
    for k, t in enumerate(reversed(range(T))):
        nl = torch.full((1, 1), float(np.float32(tables["sqrt_alphas_cumprod_prev"][t + 1])), dtype=torch.float32)
        eps = torch.zeros_like(x)     # pixels with no active tile: invalid, so their x never reaches the output
        for b in range(B):
            wins = [(slice(y0, y0 + tey), slice(x0, x0 + tex)) for bb, y0, x0 in act if bb == b]
            wsum = torch.zeros(H, W)
            seen = torch.zeros(H, W, dtype=torch.bool)
            for wy, wx in wins:
                wsum[wy, wx] = torch.where(seen[wy, wx], wsum[wy, wx] + wt, wt)
                seen[wy, wx] = True
            acc = torch.zeros(C, H, W)
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
    keep = valid[:, None]

    def out(s, c, v):
        return torch.where(v, res2img(s, c), c)
    img = out(x, cond, keep)
    if not continous:
        return img
    per = []
    for b in range(B):
        seq = [cond[b:b + 1]] + [f[b:b + 1] for f in frames]
        per.append(torch.cat([out(s, cond[b:b + 1], keep[b:b + 1]) for s in seq], dim=0))
    return torch.cat(per, dim=0)


def masked_metrics(a, b, valid, M, scale=4.0):
    """(mse, psnr, ssim, ergas) of two (H,W,C) level images at white level M over the valid pixels (fdsr_metrics_masked),
    float64: MSE and the ERGAS mean over the C |V| valid values, SSIM the mean over the channels and the cropped-interior
    positions whose 7x7 window is wholly valid of u16_reference.metrics's SSIM map; NaN where nothing qualifies."""
    from scipy.ndimage import minimum_filter, uniform_filter
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    valid = np.asarray(valid, bool)
    if not valid.any():
        return (math.nan,) * 4
    C = a.shape[2]
    d = (a - b)[valid]
    mse = float(np.sum(d * d) / d.size)
    psnr = 10.0 * math.log10(float(M) * float(M) / mse) if mse > 0 else math.inf
    win, R = 7, float(M)
    cov = 49.0 / 48.0
    C1, C2 = (0.01 * R) ** 2, (0.03 * R) ** 2
    whole = minimum_filter(valid.astype(np.uint8), size=win, mode="constant", cval=0)[3:-3, 3:-3].astype(bool)
    vals = []
    for ch in range(C):
        X, Y = a[..., ch], b[..., ch]
        ux, uy = uniform_filter(X, size=win), uniform_filter(Y, size=win)
        vx = cov * (uniform_filter(X * X, size=win) - ux * ux)
        vy = cov * (uniform_filter(Y * Y, size=win) - uy * uy)
        vxy = cov * (uniform_filter(X * Y, size=win) - ux * uy)
        S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux ** 2 + uy ** 2 + C1) * (vx + vy + C2))
        vals.append(S[3:-3, 3:-3][whole])
    vals = np.concatenate(vals)
    ssim = float(np.mean(vals)) if vals.size else math.nan
    mean = float(np.sum(a[valid]) / d.size)
    ergas = float(100.0 * np.sqrt(mse / mean ** 2 / C) / scale)
    return mse, psnr, ssim, ergas

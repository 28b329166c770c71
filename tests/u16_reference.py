"""Float64 numpy restatement of the 16-bit boundary (DESIGN.md §4.6), for tests and for debugging without a GPU:
Pillow's BICUBIC resize of an 'I;16' band with its store quirk, the normalisation at white level M, the 16-bit
tensor2img and the metrics of fdsr_metrics_u16."""
import math

import numpy as np


def _cubic(x, a=-0.5):
    x = abs(x)
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1.0
    if x < 2.0:
        return (((x - 5.0) * x + 8.0) * x - 4.0) * a
    return 0.0


def coeffs(in_size, out_size):
    """Per output index (xmin, normalised double weights): Pillow precompute_coeffs for the full-image box."""
    scale = in_size / out_size
    fscale = max(scale, 1.0)
    support = 2.0 * fscale
    ss = 1.0 / fscale
    out = []
    for i in range(out_size):
        center = (i + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        n = min(int(center + support + 0.5), in_size) - xmin
        k = [_cubic((x + xmin - center + 0.5) * ss) for x in range(n)]
        ww = 0.0
        for w in k:
            ww += w
        out.append((xmin, [w / ww if ww != 0.0 else w for w in k]))
    return out


def store_i16(v):
    """Pillow's byte-wise I;16 store of the rounded int64 sums v: lo = CLIP8(v % 256) (C remainder), hi = CLIP8(v >> 8)."""
    return np.where(v < 0, 0, np.where(v > 65535, 65280 + v % 256, v)).astype(np.uint16)


def _pass_axis0(img, out_size):
    src = img.astype(np.float64)
    res = np.empty((out_size,) + img.shape[1:], dtype=np.uint16)
    for i, (xmin, k) in enumerate(coeffs(img.shape[0], out_size)):
        ss = np.zeros(img.shape[1:], dtype=np.float64)
        for j, w in enumerate(k):          # one rounded multiply and one rounded add per tap, in tap order
            ss = ss + src[xmin + j] * w
        v = np.where(ss >= 0, np.floor(ss + 0.5), -np.floor(-ss + 0.5)).astype(np.int64)
        res[i] = store_i16(v)
    return res


def pil_bicubic_u16(img, out_h, out_w):
    """(h,w,C) or (h,w) uint16 -> (out_h,out_w,...) uint16, each band as Pillow resizes an I;16 image: horizontal pass,
    uint16 intermediate, vertical pass."""
    img = np.asarray(img, dtype=np.uint16)
    t = np.swapaxes(_pass_axis0(np.swapaxes(img, 0, 1), out_w), 0, 1)
    return np.ascontiguousarray(_pass_axis0(t, out_h))


def u16_to_cond(img, M):
    """(..., H, W, C) uint16 -> fp32 (min(v, M) / M) * 2 - 1 in the input layout, every step in fp32."""
    v = np.minimum(np.asarray(img).astype(np.int64), M).astype(np.float32)
    return (v / np.float32(M)) * np.float32(2.0) - np.float32(1.0)


def quantise(x, M):
    """The 16-bit tensor2img: rint(((clamp(x, -1, 1) + 1) / 2) * M) in fp32, ties to even, as int64."""
    x = np.clip(np.asarray(x, dtype=np.float32), np.float32(-1), np.float32(1))
    return np.rint(((x + np.float32(1)) / np.float32(2)) * np.float32(M)).astype(np.int64)


def metrics(a, b, M, scale=4.0):
    """(mse, psnr, ssim, ergas) of two (H,W,C) level images at white level M (fdsr_metrics_u16), float64."""
    from scipy.ndimage import uniform_filter
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    mse = float(np.mean((a - b) ** 2))
    psnr = 10.0 * math.log10(float(M) * float(M) / mse) if mse > 0 else float("inf")
    win, R = 7, float(M)
    cov = 49.0 / 48.0
    C1, C2 = (0.01 * R) ** 2, (0.03 * R) ** 2
    vals = []
    for ch in range(a.shape[2]):
        X, Y = a[..., ch], b[..., ch]
        ux, uy = uniform_filter(X, size=win), uniform_filter(Y, size=win)
        vx = cov * (uniform_filter(X * X, size=win) - ux * ux)
        vy = cov * (uniform_filter(Y * Y, size=win) - uy * uy)
        vxy = cov * (uniform_filter(X * Y, size=win) - ux * uy)
        S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux ** 2 + uy ** 2 + C1) * (vx + vy + C2))
        vals.append(S[3:-3, 3:-3].mean())
    ssim = float(np.mean(vals))
    ergas = float(100.0 * np.sqrt(mse / np.mean(a) ** 2 / a.shape[2]) / scale)
    return mse, psnr, ssim, ergas

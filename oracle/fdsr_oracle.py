"""CPU oracle for the FastDiffSR T=20 conditional sampling path.  TEST INFRASTRUCTURE ONLY.

This file is a from-scratch, functional restatement (plain numpy for the integer / table work,
torch-CPU fp32 for the floating-point UNet) of the reference algorithm.  It is the checker for
the CUDA path: only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import it.  The product package never does (it fails loudly when
its CUDA library is missing).

Parity pinning: ``oracle/make_golden.py`` imports the real reference from a checkout of the
original FastDiffSR repository, asserts that every function below reproduces it, and
writes ``tests/golden/*.npz``; ``tests/test_oracle_golden.py`` re-checks this file against those
fixtures anywhere.  The bicubic restatement is additionally pinned by the reference's own
UC-Merced fixtures (lr_128 -> sr_128_512, bit-exact).

Reference locations restated here (paths relative to the original FastDiffSR repository):
  make_beta_schedule            model/fastdiffsr_modules/diffusion.py:21-64
  schedule tables               model/fastdiffsr_modules/diffusion.py:109-155
  p_mean_variance / p_sample    model/fastdiffsr_modules/diffusion.py:157-190
  p_sample_loop / res2img       model/fastdiffsr_modules/diffusion.py:192-221, 275-281
  UNet and its blocks           model/fastdiffsr_modules/unet.py:22-173, 206-323
  PIL bicubic conditioning      data/prepare_data_mfe_dm.py:30-40 (Pillow ImagingResample)
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------------------
# Config helpers
# --------------------------------------------------------------------------------------

DEFAULT_UNET = dict(in_channel=6, out_channel=3, inner_channel=64, norm_groups=32,
                    channel_multiplier=[1, 2, 4, 4], attn_res=[16], res_blocks=2, dropout=0.2)
DEFAULT_SCHEDULE = dict(schedule="linear_cosine", n_timestep=20, linear_start=1e-6, linear_end=1e-2)


def unet_layers(cfg):
    """Ordered structural plan of the UNet (unet.py:224-297).

    Returns (downs, mid, ups) where every entry is a tuple
      ("stem", name, cin, cout) | ("res", name, cin, cout, with_attn) | ("down", name, c) |
      ("up", name, c)
    ``cin`` of an ``ups`` res entry already includes the skip channels.
    """
    inner = cfg["inner_channel"]
    mults = list(cfg["channel_multiplier"])
    nres = cfg["res_blocks"]
    pre = inner
    feat = [pre]
    downs = [("stem", "downs.0", cfg["in_channel"], inner)]
    for li, m in enumerate(mults):
        cm = inner * m
        for _ in range(nres):
            downs.append(("res", f"downs.{len(downs)}", pre, cm, False))
            feat.append(cm)
            pre = cm
        if li != len(mults) - 1:
            downs.append(("down", f"downs.{len(downs)}", pre))
            feat.append(pre)
    mid = [("res", "mid.0", pre, pre, True), ("res", "mid.1", pre, pre, False)]
    ups = []
    for li in reversed(range(len(mults))):
        cm = inner * mults[li]
        for _ in range(nres + 1):
            ups.append(("res", f"ups.{len(ups)}", pre + feat.pop(), cm, False))
            pre = cm
        if li >= 1:
            ups.append(("up", f"ups.{len(ups)}", pre))
    return downs, mid, ups, pre


def state_dict_spec(cfg):
    """[(key, shape, kind, fan_in)] in the reference's state_dict order (317-12 = 305 tensors for
    the shipped config).  kind in {"w", "b", "gamma", "beta"}."""
    inner = cfg["inner_channel"]
    out = []

    def conv(name, co, ci, k, bias=True):
        out.append((name + ".weight", (co, ci, k, k), "w", ci * k * k))
        if bias:
            out.append((name + ".bias", (co,), "b", ci * k * k))

    def lin(name, co, ci):
        out.append((name + ".weight", (co, ci), "w", ci))
        out.append((name + ".bias", (co,), "b", ci))

    def gn(name, c):
        out.append((name + ".weight", (c,), "gamma", 0))
        out.append((name + ".bias", (c,), "beta", 0))

    def res(name, ci, co, attn):
        lin(f"{name}.res_block.noise_func.noise_func.0", co, inner)
        gn(f"{name}.res_block.block1.block.0", ci)
        conv(f"{name}.res_block.block1.block.3", co, ci, 3)
        gn(f"{name}.res_block.block2.block.0", co)
        conv(f"{name}.res_block.block2.block.3", co, co, 3)
        if ci != co:
            conv(f"{name}.res_block.res_conv", co, ci, 1)
        conv(f"{name}.conv", co, co, 1)  # constructed, never executed (unet.py:212)
        if attn:
            conv(f"{name}.ca.fc1", co // 16, co, 1, bias=False)
            conv(f"{name}.ca.fc2", co, co // 16, 1, bias=False)
            conv(f"{name}.sa.conv1", 1, 2, 7, bias=False)

    lin("noise_level_mlp.1", inner * 4, inner)
    lin("noise_level_mlp.3", inner, inner * 4)
    downs, mid, ups, last = unet_layers(cfg)
    for grp in (downs, mid, ups):
        for e in grp:
            if e[0] == "stem":
                conv(e[1], e[3], e[2], 3)
            elif e[0] == "res":
                res(e[1], e[2], e[3], e[4])
            else:
                conv(e[1] + ".conv", e[2], e[2], 3)
    gn("final_conv.block.0", last)
    conv("final_conv.block.3", cfg["out_channel"], last, 3)
    return [("denoise_fn." + k, s, kind, f) for (k, s, kind, f) in out]


def make_state_dict(cfg, seed=0, gn_jitter=0.0, spec=None):
    """Deterministic, machine-independent random weights with PyTorch's default-init statistics
    (conv/linear: U(-1/sqrt(fan_in), 1/sqrt(fan_in)); GroupNorm: gamma=1, beta=0, optionally
    jittered so that the affine path is exercised).  numpy PCG64, one stream per tensor.
    ``spec`` defaults to the FastDiffSR UNet's; pass ``sr3_state_dict_spec(...)`` for the SR3 baseline."""
    sd = {}
    for idx, (key, shape, kind, fan_in) in enumerate(spec if spec is not None else state_dict_spec(cfg)):
        rng = np.random.default_rng([seed, idx])
        if kind == "inv_freq":  # TimeEmbedding buffer (ddpm_modules/unet.py:22-27), not random
            dim = 2 * shape[0]
            sd[key] = torch.exp(torch.arange(0, dim, 2, dtype=torch.float32) * (-math.log(10000) / dim))
            continue
        if kind in ("w", "b"):
            bound = 1.0 / math.sqrt(fan_in)
            a = rng.uniform(-bound, bound, size=shape)
        elif kind == "gamma":
            a = 1.0 + gn_jitter * rng.standard_normal(shape)
        else:
            a = gn_jitter * rng.standard_normal(shape)
        sd[key] = torch.from_numpy(a.astype(np.float32))
    return sd


# --------------------------------------------------------------------------------------
# Schedule (float64 numpy, exactly as the reference derives it)
# --------------------------------------------------------------------------------------

def make_beta_schedule(schedule, n_timestep, linear_start=1e-4, linear_end=2e-2, cosine_s=8e-3):
    if schedule == "linear":
        return np.linspace(linear_start, linear_end, n_timestep, dtype=np.float64)
    if schedule == "quad":
        return np.linspace(linear_start ** 0.5, linear_end ** 0.5, n_timestep, dtype=np.float64) ** 2
    if schedule == "const":
        return linear_end * np.ones(n_timestep, dtype=np.float64)
    if schedule == "jsd":
        return 1.0 / np.linspace(n_timestep, 1, n_timestep, dtype=np.float64)
    if schedule in ("warmup10", "warmup50"):
        frac = 0.1 if schedule == "warmup10" else 0.5
        betas = linear_end * np.ones(n_timestep, dtype=np.float64)
        w = int(n_timestep * frac)
        betas[:w] = np.linspace(linear_start, linear_end, w, dtype=np.float64)
        return betas
    if schedule == "linear_cosine":
        lin = np.linspace(linear_start, linear_end, n_timestep, dtype=np.float64)
        steps = n_timestep + 1
        x = np.linspace(0, steps, steps)
        ac = np.cos(((x / steps) + cosine_s) / (1 + cosine_s) * np.pi * 0.5) ** 2
        ac = ac / ac[0]
        cos_b = np.clip(1 - (ac[1:] / ac[:-1]), 0, 0.999)
        return np.clip(lin + (cos_b + cos_b), 0, 0.999)   # code is truth: linear + 2*cosine
    raise NotImplementedError(schedule)


def schedule_tables(betas):
    """All tables of set_new_noise_schedule, float64; callers cast to fp32 like the reference."""
    betas = np.asarray(betas, dtype=np.float64)
    alphas = 1.0 - betas
    ac = np.cumprod(alphas, axis=0)
    ac_prev = np.append(1.0, ac[:-1])
    pv = betas * (1.0 - ac_prev) / (1.0 - ac)
    return dict(
        betas=betas, alphas_cumprod=ac, alphas_cumprod_prev=ac_prev,
        sqrt_alphas_cumprod=np.sqrt(ac), sqrt_one_minus_alphas_cumprod=np.sqrt(1.0 - ac),
        log_one_minus_alphas_cumprod=np.log(1.0 - ac),
        sqrt_recip_alphas_cumprod=np.sqrt(1.0 / ac), sqrt_recipm1_alphas_cumprod=np.sqrt(1.0 / ac - 1),
        posterior_variance=pv, posterior_log_variance_clipped=np.log(np.maximum(pv, 1e-20)),
        posterior_mean_coef1=betas * np.sqrt(ac_prev) / (1.0 - ac),
        posterior_mean_coef2=(1.0 - ac_prev) * np.sqrt(alphas) / (1.0 - ac),
        sqrt_alphas_cumprod_prev=np.sqrt(np.append(1.0, ac)),   # noise levels, length T+1
    )


# --------------------------------------------------------------------------------------
# UNet (functional, fp32)
# --------------------------------------------------------------------------------------

def _swish(x):
    return x * torch.sigmoid(x)


def noise_embedding(noise_level, dim):
    """unet.py:22-35 — noise_level (B,1) -> (B,1,dim)."""
    count = dim // 2
    step = torch.arange(count, dtype=noise_level.dtype, device=noise_level.device) / count
    enc = noise_level.unsqueeze(1) * torch.exp(-math.log(1e4) * step.unsqueeze(0))
    return torch.cat([torch.sin(enc), torch.cos(enc)], dim=-1)


def _gn_swish_conv(sd, pfx, x, groups):
    h = F.group_norm(x, groups, sd[pfx + ".block.0.weight"], sd[pfx + ".block.0.bias"], eps=1e-5)
    return F.conv2d(_swish(h), sd[pfx + ".block.3.weight"], sd[pfx + ".block.3.bias"], padding=1)


def _res_block(sd, name, x, temb, groups, with_attn):
    p = f"denoise_fn.{name}.res_block"
    h = _gn_swish_conv(sd, p + ".block1", x, groups)
    film = F.linear(temb, sd[p + ".noise_func.noise_func.0.weight"], sd[p + ".noise_func.noise_func.0.bias"])
    h = h + film.view(x.shape[0], -1, 1, 1)
    h = _gn_swish_conv(sd, p + ".block2", h, groups)
    if p + ".res_conv.weight" in sd:
        x = F.conv2d(x, sd[p + ".res_conv.weight"], sd[p + ".res_conv.bias"])
    y = h + x
    if with_attn:
        q = f"denoise_fn.{name}"
        w1, w2 = sd[q + ".ca.fc1.weight"], sd[q + ".ca.fc2.weight"]
        avg = F.adaptive_avg_pool2d(y, 1)
        mx = F.adaptive_max_pool2d(y, 1)
        gate = F.conv2d(F.relu(F.conv2d(avg, w1)), w2) + F.conv2d(F.relu(F.conv2d(mx, w1)), w2)
        y = torch.sigmoid(gate) * y
        sp = torch.cat([y.mean(dim=1, keepdim=True), y.max(dim=1, keepdim=True)[0]], dim=1)
        y = torch.sigmoid(F.conv2d(sp, sd[q + ".sa.conv1.weight"], padding=3)) * y
    return y


@torch.no_grad()
def unet_forward(sd, cfg, x, noise_level, taps=None):
    """eps = UNet(cat[cond, x_t], noise_level).  x: (B,6,H,W) fp32, noise_level: (B,1).
    ``taps`` (optional dict) receives named intermediate tensors for layer-level debugging."""
    groups = cfg.get("norm_groups") or 32
    inner = cfg["inner_channel"]
    downs, mid, ups, _ = unet_layers(cfg)
    t = noise_embedding(noise_level, inner)
    t = F.linear(t, sd["denoise_fn.noise_level_mlp.1.weight"], sd["denoise_fn.noise_level_mlp.1.bias"])
    t = F.linear(_swish(t), sd["denoise_fn.noise_level_mlp.3.weight"], sd["denoise_fn.noise_level_mlp.3.bias"])
    feats = []
    for e in downs:
        if e[0] == "stem":
            x = F.conv2d(x, sd[f"denoise_fn.{e[1]}.weight"], sd[f"denoise_fn.{e[1]}.bias"], padding=1)
        elif e[0] == "res":
            x = _res_block(sd, e[1], x, t, groups, e[4])
        else:
            x = F.conv2d(x, sd[f"denoise_fn.{e[1]}.conv.weight"], sd[f"denoise_fn.{e[1]}.conv.bias"],
                         stride=2, padding=1)
        feats.append(x)
        if taps is not None:
            taps[e[1]] = x
    for e in mid:
        x = _res_block(sd, e[1], x, t, groups, e[4])
        if taps is not None:
            taps[e[1]] = x
    for e in ups:
        if e[0] == "res":
            x = _res_block(sd, e[1], torch.cat((x, feats.pop()), dim=1), t, groups, e[4])
        else:
            x = F.interpolate(x, scale_factor=2, mode="nearest")
            x = F.conv2d(x, sd[f"denoise_fn.{e[1]}.conv.weight"], sd[f"denoise_fn.{e[1]}.conv.bias"], padding=1)
        if taps is not None:
            taps[e[1]] = x
    h = F.group_norm(x, groups, sd["denoise_fn.final_conv.block.0.weight"],
                     sd["denoise_fn.final_conv.block.0.bias"], eps=1e-5)
    return F.conv2d(_swish(h), sd["denoise_fn.final_conv.block.3.weight"],
                    sd["denoise_fn.final_conv.block.3.bias"], padding=1)


def film_table(sd, cfg, tables):
    """Per-step additive FiLM vectors: the noise level depends on t only (diffusion.py:169-170), so
    every ResnetBlock's Linear(temb) is a constant per step.  Returns {block_name: (T, Cout)}."""
    inner = cfg["inner_channel"]
    T = len(tables["betas"])
    nl = torch.tensor(tables["sqrt_alphas_cumprod_prev"][1:T + 1], dtype=torch.float32).view(T, 1)
    t = noise_embedding(nl, inner)
    t = F.linear(t, sd["denoise_fn.noise_level_mlp.1.weight"], sd["denoise_fn.noise_level_mlp.1.bias"])
    t = F.linear(_swish(t), sd["denoise_fn.noise_level_mlp.3.weight"], sd["denoise_fn.noise_level_mlp.3.bias"])
    out = {}
    downs, mid, ups, _ = unet_layers(cfg)
    for e in downs + mid + ups:
        if e[0] == "res":
            p = f"denoise_fn.{e[1]}.res_block.noise_func.noise_func.0"
            out[e[1]] = F.linear(t, sd[p + ".weight"], sd[p + ".bias"]).view(T, -1)
    return out


# --------------------------------------------------------------------------------------
# Sampler
# --------------------------------------------------------------------------------------

def _f32(tables, key, t):
    return torch.tensor(tables[key][t], dtype=torch.float32)


@torch.no_grad()
def p_sample_step(sd, cfg, tables, x, t, cond, z, eps=None):
    """One ancestral step (diffusion.py:167-190).  Returns (x_prev, eps, x0_clipped).
    ``eps`` may be supplied to bypass the UNet (used to test the posterior arithmetic alone)."""
    B = x.shape[0]
    if eps is None:
        nl = torch.full((B, 1), float(np.float32(tables["sqrt_alphas_cumprod_prev"][t + 1])), dtype=torch.float32,
                        device=x.device)
        eps = unet_forward(sd, cfg, torch.cat([cond, x], dim=1), nl)
    x0 = _f32(tables, "sqrt_recip_alphas_cumprod", t) * x - _f32(tables, "sqrt_recipm1_alphas_cumprod", t) * eps
    x0 = x0.clamp(-1.0, 1.0)
    mean = _f32(tables, "posterior_mean_coef1", t) * x0 + _f32(tables, "posterior_mean_coef2", t) * x
    if t > 0:
        x_prev = mean + z * (0.5 * _f32(tables, "posterior_log_variance_clipped", t)).exp()
    else:
        x_prev = mean + torch.zeros_like(x) * (0.5 * _f32(tables, "posterior_log_variance_clipped", t)).exp()
    return x_prev, eps, x0


def res2img(res, cond):
    return res.clamp(-1, 1) / 2.0 + cond


@torch.no_grad()
def sample_loop(sd, cfg, tables, cond, noises, continous=False, trace=None):
    """p_sample_loop (diffusion.py:192-221) with injected noise.

    cond   : (B,3,H,W) bicubic conditioning in [-1,1]
    noises : (T,B,3,H,W); noises[0] is x_T, noises[k] (k=1..T-1) is the z drawn at step t=T-k
             (the reference's draw order: one randn, then randn_like for t=T-1..1; t=0 draws none).
    continous=True reproduces the reference's B=1 layout: [res2img(cond,cond), frames at
    t % sample_inter == 0] -> (1+n_frames, 3, H, W); for B>1 (where the reference crashes,
    SURVEY F2) frames are stacked per sample along dim 0 in the same order, sample-major.
    """
    T = len(tables["betas"])
    sample_inter = 1 | (T // 10)
    x = noises[0]
    frames = []
    for k, t in enumerate(reversed(range(T))):
        z = noises[k + 1] if t > 0 else None
        x_in = x
        x, eps, x0 = p_sample_step(sd, cfg, tables, x, t, cond, z)
        if trace is not None:
            trace.append(dict(t=t, x_t=x_in, eps=eps, x_prev=x))
        if t % sample_inter == 0:
            frames.append(x)
    img = res2img(x, cond)
    if not continous:
        return img
    B = cond.shape[0]
    per = []
    for b in range(B):
        seq = [cond[b:b + 1]] + [f[b:b + 1] for f in frames]
        per.append(torch.cat([res2img(s, cond[b:b + 1]) for s in seq], dim=0))
    return torch.cat(per, dim=0)


# --------------------------------------------------------------------------------------
# PIL-exact bicubic (integer arithmetic; numpy)
# --------------------------------------------------------------------------------------

_PREC = 22  # Pillow's PRECISION_BITS = 32 - 8 - 2


def _cubic(x, a=-0.5):
    x = abs(x)
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1.0
    if x < 2.0:
        return (((x - 5.0) * x + 8.0) * x - 4.0) * a
    return 0.0


def bicubic_coeffs(in_size, out_size):
    """Per-output-index (xmin, int32 taps) exactly as Pillow's precompute_coeffs + normalize_coeffs_8bpc
    for the full-image box: support 2 (scaled up when down-sampling), window clipped at the border and
    renormalised, taps quantised to 22-bit fixed point."""
    scale = in_size / out_size
    fscale = max(scale, 1.0)
    support = 2.0 * fscale
    ksize = int(math.ceil(support)) * 2 + 1
    bounds, taps = [], np.zeros((out_size, ksize), dtype=np.int64)
    for i in range(out_size):
        center = (i + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), in_size) - xmin
        w = np.array([_cubic((x + xmin - center + 0.5) / fscale) for x in range(xmax)], dtype=np.float64)
        w = w / w.sum()
        q = np.where(w < 0, np.trunc(-0.5 + w * (1 << _PREC)), np.trunc(0.5 + w * (1 << _PREC))).astype(np.int64)
        taps[i, :xmax] = q
        bounds.append((xmin, xmax))
    return bounds, taps


def _resample_axis0(img, out_size):
    """img (L, ...) uint8 -> (out_size, ...) uint8 along axis 0."""
    bounds, taps = bicubic_coeffs(img.shape[0], out_size)
    out = np.empty((out_size,) + img.shape[1:], dtype=np.uint8)
    src = img.astype(np.int64)
    for i, (xmin, n) in enumerate(bounds):
        acc = np.tensordot(taps[i, :n], src[xmin:xmin + n], axes=(0, 0)) + (1 << (_PREC - 1))
        out[i] = np.clip(acc >> _PREC, 0, 255).astype(np.uint8)
    return out


def pil_bicubic_u8(img, out_h, out_w):
    """(H,W,C) uint8 -> (out_h,out_w,C) uint8, bit-exact with PIL Image.resize(BICUBIC):
    horizontal pass first, uint8 rounding/clipping between the passes."""
    img = np.ascontiguousarray(img)
    if img.shape[1] != out_w:
        img = np.swapaxes(_resample_axis0(np.swapaxes(img, 0, 1), out_w), 0, 1)
    if img.shape[0] != out_h:
        img = _resample_axis0(img, out_h)
    return np.ascontiguousarray(img)


def u8_to_cond(img_u8):
    """(B,H,W,C) or (H,W,C) uint8 -> NCHW fp32 in [-1,1] (data/util.py:66-75: ToTensor then *2-1)."""
    a = torch.from_numpy(np.asarray(img_u8)).to(torch.float32) / 255.0
    a = a * 2.0 - 1.0
    if a.dim() == 3:
        return a.permute(2, 0, 1).contiguous()
    return a.permute(0, 3, 1, 2).contiguous()


# --------------------------------------------------------------------------------------
# Metrics used by the end-to-end parity bar
# --------------------------------------------------------------------------------------

def to_u8(img):
    """core/metrics.py:16-42 tensor2img for a single image, min_max=(-1,1): (3,H,W) -> (H,W,3) uint8."""
    a = img.detach().float().clamp(-1, 1)
    a = (a + 1) / 2
    return (a.permute(1, 2, 0).numpy() * 255.0).round().astype(np.uint8)


def psnr_u8(a, b):
    """core/metrics.py:94-101."""
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    if mse == 0:
        return float("inf")
    return 20 * math.log10(255.0 / math.sqrt(mse))


def mse_u8(a, b):
    """skimage.measure.compare_mse as sr_mfe.py:315 calls it (uint8 HWC images -> float64)."""
    return float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))


def ssim_u8(a, b):
    """skimage.measure.compare_ssim(a, b, multichannel=True) as sr_mfe.py:317 calls it, restated from the
    published algorithm of scikit-image 0.15 (`skimage/measure/_structural_similarity.py`; the package is
    pinned in the reference's requirements.txt:6 but absent here and the reference holds no fixture with a
    recorded SSIM value, so this restatement is PARITY UNPINNED): win_size 7 uniform filter, K1 = 0.01,
    K2 = 0.03, data_range 255 (uint8), use_sample_covariance=True, float64; per channel the map is cropped by
    (win_size-1)//2 on each side and averaged; channels are averaged."""
    from scipy.ndimage import uniform_filter
    assert a.shape == b.shape and a.ndim == 3
    win, K1, K2, R = 7, 0.01, 0.03, 255.0
    NP = win ** 2
    cov_norm = NP / (NP - 1.0)
    C1, C2 = (K1 * R) ** 2, (K2 * R) ** 2
    pad = (win - 1) // 2
    vals = []
    for ch in range(a.shape[2]):
        X = a[..., ch].astype(np.float64)
        Y = b[..., ch].astype(np.float64)
        ux, uy = uniform_filter(X, size=win), uniform_filter(Y, size=win)
        uxx, uyy, uxy = uniform_filter(X * X, size=win), uniform_filter(Y * Y, size=win), uniform_filter(X * Y, size=win)
        vx, vy, vxy = cov_norm * (uxx - ux * ux), cov_norm * (uyy - uy * uy), cov_norm * (uxy - ux * uy)
        S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux ** 2 + uy ** 2 + C1) * (vx + vy + C2))
        vals.append(S[pad:-pad, pad:-pad].mean())
    return float(np.mean(vals))


def ergas_u8(a, b, scale=4):
    """core/metrics.py:88-93 calculate_ergas(img1, img2, scale)."""
    mean2 = np.mean(a, dtype=np.float64) ** 2
    return float(100.0 * np.sqrt(mse_u8(a, b) / mean2 / a.shape[2]) / scale)


# --------------------------------------------------------------------------------------
# SR3 baseline (which_model_G == "ddpm"): the comparison model of the paper, SURVEY section 8(f) N3.
# Restates model/ddpm_modules/unet.py (TimeEmbedding :19-33, ResnetBlock :79-97, SelfAttention
# :100-131, ResnetBlocWithAttn :134-147, UNet :150-243) and the sampler of
# model/ddpm_modules/diffusion.py (:159-199 posterior / p_sample, :201-231 p_sample_loop).
# Pinned against the real reference by oracle/make_golden.py (tests/golden/sr3_*.npz).
# --------------------------------------------------------------------------------------

SR3_UNET = dict(in_channel=6, out_channel=3, inner_channel=64, norm_groups=32,
                channel_multiplier=[1, 1, 2, 2, 4, 4], attn_res=[16], res_blocks=2, dropout=0.2)
SR3_SCHEDULE = dict(schedule="linear", n_timestep=1000, linear_start=1e-4, linear_end=2e-2)


def sr3_unet_layers(cfg, image_size=256):
    """Structural plan of the SR3 UNet (ddpm_modules/unet.py:178-225): like ``unet_layers`` but a
    block carries SelfAttention when the resolution *of the configured image_size* at its level is in
    attn_res (the flag does not depend on the actual input size), and mid[0] always does."""
    inner = cfg["inner_channel"]
    mults = list(cfg["channel_multiplier"])
    nres = cfg["res_blocks"]
    attn_res = list(cfg["attn_res"])
    pre = inner
    feat = [pre]
    now = image_size
    downs = [("stem", "downs.0", cfg["in_channel"], inner)]
    for li, m in enumerate(mults):
        cm = inner * m
        for _ in range(nres):
            downs.append(("res", f"downs.{len(downs)}", pre, cm, now in attn_res))
            feat.append(cm)
            pre = cm
        if li != len(mults) - 1:
            downs.append(("down", f"downs.{len(downs)}", pre))
            feat.append(pre)
            now //= 2
    mid = [("res", "mid.0", pre, pre, True), ("res", "mid.1", pre, pre, False)]
    ups = []
    for li in reversed(range(len(mults))):
        cm = inner * mults[li]
        for _ in range(nres + 1):
            ups.append(("res", f"ups.{len(ups)}", pre + feat.pop(), cm, now in attn_res))
            pre = cm
        if li >= 1:
            ups.append(("up", f"ups.{len(ups)}", pre))
            now *= 2
    return downs, mid, ups, pre


def sr3_state_dict_spec(cfg, image_size=256):
    """[(key, shape, kind, fan_in)] in the reference's state_dict order for the SR3 UNet."""
    inner = cfg["inner_channel"]
    out = [("time_mlp.0.inv_freq", (inner // 2,), "inv_freq", 0)]

    def conv(name, co, ci, k, bias=True):
        out.append((name + ".weight", (co, ci, k, k), "w", ci * k * k))
        if bias:
            out.append((name + ".bias", (co,), "b", ci * k * k))

    def lin(name, co, ci):
        out.append((name + ".weight", (co, ci), "w", ci))
        out.append((name + ".bias", (co,), "b", ci))

    def gn(name, c):
        out.append((name + ".weight", (c,), "gamma", 0))
        out.append((name + ".bias", (c,), "beta", 0))

    def res(name, ci, co, attn):
        lin(f"{name}.res_block.mlp.1", co, inner)
        gn(f"{name}.res_block.block1.block.0", ci)
        conv(f"{name}.res_block.block1.block.3", co, ci, 3)
        gn(f"{name}.res_block.block2.block.0", co)
        conv(f"{name}.res_block.block2.block.3", co, co, 3)
        if ci != co:
            conv(f"{name}.res_block.res_conv", co, ci, 1)
        if attn:
            gn(f"{name}.attn.norm", co)
            conv(f"{name}.attn.qkv", 3 * co, co, 1, bias=False)
            conv(f"{name}.attn.out", co, co, 1)

    lin("time_mlp.1", inner * 4, inner)
    lin("time_mlp.3", inner, inner * 4)
    downs, mid, ups, last = sr3_unet_layers(cfg, image_size)
    for grp in (downs, mid, ups):
        for e in grp:
            if e[0] == "stem":
                conv(e[1], e[3], e[2], 3)
            elif e[0] == "res":
                res(e[1], e[2], e[3], e[4])
            else:
                conv(e[1] + ".conv", e[2], e[2], 3)
    gn("final_conv.block.0", last)
    conv("final_conv.block.3", cfg["out_channel"], last, 3)
    return [("denoise_fn." + k, s, kind, f) for (k, s, kind, f) in out]


def sr3_time_embedding(sd, cfg, time):
    """time_mlp (ddpm_modules/unet.py:165-171): time (B,) -> (B, inner)."""
    inv = sd["denoise_fn.time_mlp.0.inv_freq"]
    sinus = torch.ger(time.view(-1).float(), inv)
    t = torch.cat([sinus.sin(), sinus.cos()], dim=-1)
    t = F.linear(t, sd["denoise_fn.time_mlp.1.weight"], sd["denoise_fn.time_mlp.1.bias"])
    return F.linear(_swish(t), sd["denoise_fn.time_mlp.3.weight"], sd["denoise_fn.time_mlp.3.bias"])


def sr3_self_attention(sd, pfx, x, groups, taps=None, name=None):
    """SelfAttention.forward, n_head = 1 (ddpm_modules/unet.py:110-131): note the 1/sqrt(channel) scale."""
    B, C, H, W = x.shape
    n = F.group_norm(x, groups, sd[pfx + ".norm.weight"], sd[pfx + ".norm.bias"], eps=1e-5)
    qkv = F.conv2d(n, sd[pfx + ".qkv.weight"]).view(B, 1, 3 * C, H, W)
    q, k, v = qkv.chunk(3, dim=2)
    attn = torch.einsum("bnchw, bncyx -> bnhwyx", q, k).contiguous() / math.sqrt(C)
    attn = torch.softmax(attn.view(B, 1, H, W, -1), -1).view(B, 1, H, W, H, W)
    o = torch.einsum("bnhwyx, bncyx -> bnchw", attn, v).contiguous().view(B, C, H, W)
    if taps is not None:
        taps[name + ".attn.q"] = q.reshape(B, C, H, W)
        taps[name + ".attn.k"] = k.reshape(B, C, H, W)
        taps[name + ".attn.v"] = v.reshape(B, C, H, W)
        taps[name + ".attn.o"] = o
    return F.conv2d(o, sd[pfx + ".out.weight"], sd[pfx + ".out.bias"]) + x


def _sr3_res_block(sd, name, x, temb, groups, with_attn, taps=None):
    p = f"denoise_fn.{name}.res_block"
    h = _gn_swish_conv(sd, p + ".block1", x, groups)
    h = h + F.linear(_swish(temb), sd[p + ".mlp.1.weight"], sd[p + ".mlp.1.bias"])[:, :, None, None]
    h = _gn_swish_conv(sd, p + ".block2", h, groups)
    if p + ".res_conv.weight" in sd:
        x = F.conv2d(x, sd[p + ".res_conv.weight"], sd[p + ".res_conv.bias"])
    y = h + x
    if with_attn:
        if taps is not None:
            taps[name + ".res"] = y
        y = sr3_self_attention(sd, f"denoise_fn.{name}.attn", y, groups, taps, name)
    return y


@torch.no_grad()
def sr3_unet_forward(sd, cfg, x, time, image_size=256, taps=None):
    """eps = UNet(cat[cond, x_t], t) of the SR3 baseline.  x: (B,6,H,W) fp32, time: (B,) integer steps."""
    groups = cfg.get("norm_groups") or 32
    downs, mid, ups, _ = sr3_unet_layers(cfg, image_size)
    t = sr3_time_embedding(sd, cfg, time)
    feats = []
    for e in downs:
        if e[0] == "stem":
            x = F.conv2d(x, sd[f"denoise_fn.{e[1]}.weight"], sd[f"denoise_fn.{e[1]}.bias"], padding=1)
        elif e[0] == "res":
            x = _sr3_res_block(sd, e[1], x, t, groups, e[4], taps)
        else:
            x = F.conv2d(x, sd[f"denoise_fn.{e[1]}.conv.weight"], sd[f"denoise_fn.{e[1]}.conv.bias"],
                         stride=2, padding=1)
        feats.append(x)
        if taps is not None:
            taps[e[1]] = x
    for e in mid:
        x = _sr3_res_block(sd, e[1], x, t, groups, e[4], taps)
        if taps is not None:
            taps[e[1]] = x
    for e in ups:
        if e[0] == "res":
            x = _sr3_res_block(sd, e[1], torch.cat((x, feats.pop()), dim=1), t, groups, e[4], taps)
        else:
            x = F.interpolate(x, scale_factor=2, mode="nearest")
            x = F.conv2d(x, sd[f"denoise_fn.{e[1]}.conv.weight"], sd[f"denoise_fn.{e[1]}.conv.bias"], padding=1)
        if taps is not None:
            taps[e[1]] = x
    h = F.group_norm(x, groups, sd["denoise_fn.final_conv.block.0.weight"],
                     sd["denoise_fn.final_conv.block.0.bias"], eps=1e-5)
    return F.conv2d(_swish(h), sd["denoise_fn.final_conv.block.3.weight"],
                    sd["denoise_fn.final_conv.block.3.bias"], padding=1)


@torch.no_grad()
def sr3_sample_loop(sd, cfg, tables, cond, noises, image_size=256, continous=False, trace=None):
    """p_sample_loop of the SR3 baseline (ddpm_modules/diffusion.py:201-231) with injected noise.

    noises: (T,B,3,H,W) in the draw order x_T, then z for t = T-1 .. 1.  (The reference also draws a
    tensor at t = 0 and multiplies it by the zero mask, :196-199; it does not enter the result.)
    The image itself is predicted (no res2img).  Returns (B,3,H,W); the reference returns
    ``ret_img[-1]`` = the last image without the batch axis (identical for B = 1 up to that axis).
    continous=True: [cond, frames at t % (1 | T//10) == 0] stacked per sample along dim 0."""
    T = len(tables["betas"])
    sample_inter = 1 | (T // 10)
    x = noises[0]
    B = cond.shape[0]
    frames = []
    for k, t in enumerate(reversed(range(T))):
        x_in = x
        eps = sr3_unet_forward(sd, cfg, torch.cat([cond, x], dim=1), torch.full((B,), t, dtype=torch.long), image_size)
        x0 = _f32(tables, "sqrt_recip_alphas_cumprod", t) * x - _f32(tables, "sqrt_recipm1_alphas_cumprod", t) * eps
        x0 = x0.clamp(-1.0, 1.0)
        mean = _f32(tables, "posterior_mean_coef1", t) * x0 + _f32(tables, "posterior_mean_coef2", t) * x
        sigma = (0.5 * _f32(tables, "posterior_log_variance_clipped", t)).exp()
        x = mean + (sigma * noises[k + 1] if t > 0 else 0.0)
        if trace is not None:
            trace.append(dict(t=t, x_t=x_in, eps=eps, x_prev=x))
        if t % sample_inter == 0:
            frames.append(x)
    if not continous:
        return x
    return torch.cat([torch.cat([cond[b:b + 1]] + [f[b:b + 1] for f in frames], dim=0) for b in range(B)], dim=0)


# --------------------------------------------------------------------------------------
# Golden fixtures (tests/golden/*.npz, written by oracle/make_golden.py)
# --------------------------------------------------------------------------------------

def golden_inputs(name):
    """The seeded inputs of fixture `name`, in the order make_golden.py draws them.  The fixture stores the float64 sum
    of each (`<input>_sum`) instead of the tensor; the tests regenerate the input here and check that sum."""
    if name.startswith("unet64_"):
        g = torch.Generator().manual_seed(11)
        x6 = torch.randn(2, 6, 64, 64, generator=g)
        cond = torch.rand(1, 3, 64, 64, generator=g) * 2 - 1
        return dict(x6=x6, cond=cond, noises=torch.randn(20, 1, 3, 64, 64, generator=g))
    if name.startswith("sr3_"):
        H = {"sr3_256": 128, "sr3_64": 64}[name]
        g = torch.Generator().manual_seed(21)
        x6 = torch.randn(2, 6, H, H, generator=g).half().float()   # exactly representable in fp16
        return dict(x6=x6, cond=torch.rand(1, 3, H, H, generator=g) * 2 - 1)
    return {}

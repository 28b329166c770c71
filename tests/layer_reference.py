"""Per-launch float64 reference of the FastDiffSR UNet: the conv and gate ops in the order the library launches them,
each evaluated on the very inputs the GPU read (its stored 16-bit tensors, exact in float64), with a per-element
error bound.  CPU only; used by tests/test_layer_reference.py (the mirror against the oracle, the comparator's
sensitivity) and tests/test_gpu_layers.py (every launch of the CUDA path).

Error bound of one output element (sums over the products w_k a_k that feed it):

    |got - ref| <= u_out |ref| + rho_op sqrt(sum_k w_k^2 (|a_k| + |g_k|)^2) + rho_acc sum_k |w_k a_k| + floor

  u_out    rounding of the stored output: 2^-11 (fp16), 2^-8 (bf16), 2^-24 (fp32 parity mode); 0 for the final conv's
           fp32 eps in the 16-bit modes.
  rho_op   operand error of the GroupNorm chunks: g_k = GroupNorm output before Swish, a_k = swish(g_k); covers the
           16-bit scale / shift table, the f16x2 affine, tanh.approx and the fp16 operand (fp16 in both 16-bit modes).
           Nearest-upsample convs get the same term with g_k = 0 and their own coefficient rho_w: their phase form
           sums two to four 3x3 weights into one weight rounded to the raw-chunk format, fp16 or bf16, so rho_w scales
           with that format's unit roundoff (2^-11 or 2^-8).
  rho_acc  fp32 accumulation; the sum also holds |bias| + |FiLM| + |identity residual| and the 1x1 residual conv's
           products.  The CLAM/SLAM gates have no matmul: their fp32 chain (a channel mean, two small MLPs, a 7x7 conv
           and three products) is bounded as (C + 98) |ref| in the same term.
  floor    one ulp of the output format at its smallest normal.

With `exact_weights` every conv weight is exact in fp16 and bf16, so weight rounding drops out; the raw chunks (stem,
stride-2 convs, 1x1 residual, identity) then have exact fp32 products and only rho_acc remains.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

import fdsr_oracle as O

U_OUT = {"fp16": 2.0 ** -11, "bf16": 2.0 ** -8, "fp32": 2.0 ** -24}
FLOOR = {"fp16": 2.0 ** -24, "bf16": 2.0 ** -133, "fp32": 2.0 ** -149}
STORE = {"fp16": torch.float16, "bf16": torch.bfloat16, "fp32": torch.float32}
# (rho_op, rho_acc) per mode: first estimates from the error model above (a few fp16 unit roundoffs per GroupNorm
# operand; fp32 accumulation at a few 2^-24 per term), not yet calibrated on a B200.  The target is that no element uses
# more than half of the rho part of its bound (`check`'s excess <= 0.5, printed by tests/test_gpu_layers.py); the
# comparator's sensitivity to small corruptions at these values is tests/test_layer_reference.py's check.
RHO = {"fp16": (2.0 ** -9, 2.0 ** -17), "bf16": (2.0 ** -9, 2.0 ** -17), "fp32": (2.0 ** -20, 2.0 ** -20)}
# rho_w of the nearest-upsample convs: four unit roundoffs of the format their summed weights are stored in
RHO_W = {"fp16": 4 * 2.0 ** -11, "bf16": 4 * 2.0 ** -8, "fp32": 2.0 ** -20}
TILE_H, TILE_W = 32, 8


def unet_cfg(inner=64, mults=(1, 2, 4, 4), res_blocks=2, bands=3):
    cfg = dict(O.DEFAULT_UNET)
    cfg.update(inner_channel=inner, channel_multiplier=list(mults), res_blocks=res_blocks, in_channel=2 * bands,
               out_channel=bands)
    return cfg


# Network configurations beyond the shipped one, each with a small shape and a multi-tile shape (B, H, W):
#   128x[1,2]       N = 128 stem, 256-wide concats at full resolution, final conv over two 64-channel chunks
#   64x[2,4]        1x1 res_conv at level 0 (64 -> 128)
#   256x[1]         one level: no down / up convs, gates on 256 channels at full resolution, GroupNorm width 512,
#                   H and W not multiples of 8
#   64x[1,1,2,2,4,4] (res_blocks 1 and 3): six levels; the 64-wide up conv runs the nine-tap gather form
#   C = 1 / C = 8   band counts of the packed input
CONFIGS = {
    "128x12": (unet_cfg(128, (1, 2)), (1, 24, 40), (2, 128, 192)),
    "64x24": (unet_cfg(64, (2, 4)), (2, 16, 24), (2, 128, 192)),
    "256x1": (unet_cfg(256, (1,)), (1, 20, 44), (3, 100, 132)),
    "sr6_rb1": (unet_cfg(64, (1, 1, 2, 2, 4, 4), 1), (1, 32, 64), (2, 128, 224)),
    "sr6_rb3": (unet_cfg(64, (1, 1, 2, 2, 4, 4), 3), (1, 32, 32), (2, 128, 256)),
    "c1": (unet_cfg(bands=1), (2, 16, 24), (2, 128, 192)),
    "c8": (unet_cfg(bands=8), (2, 16, 24), (2, 128, 192)),
}


def _p(name):
    return f"denoise_fn.{name}"


def plan_ops(cfg):
    """The ops of the UNet in launch order, named as fdsr_debug_op_name names them.  Each is a dict:
      name    op name ("downs.0", "downs.1.block1", "mid.0.clam_slam", "ups.3", "final_conv", ...)
      kind    "stem" | "block1" (GroupNorm + Swish conv, FiLM) | "block2" (GroupNorm + Swish conv + residual) | "down" |
              "up" | "gates" (CLAM + SLAM) | "final"
      inputs  tensor names read, in order (block1: the concat sources; block2: "<res>.h", then the residual sources)
      output  tensor name written ("eps" for the final conv)
      resid   block2 only: "res_conv" or "identity"
      keys    state_dict keys the op reads
      block   ResnetBlock name (block1 / block2)"""
    downs, mid, ups, _ = O.unet_layers(cfg)
    ops = []

    def res(name, srcs, out, cin, cout):
        p = _p(name) + ".res_block"
        ops.append(dict(name=name + ".block1", kind="block1", inputs=list(srcs), output=name + ".h", block=name,
                        keys=[p + ".block1.block.0.weight", p + ".block1.block.0.bias", p + ".block1.block.3.weight",
                              p + ".block1.block.3.bias", p + ".noise_func.noise_func.0.weight",
                              p + ".noise_func.noise_func.0.bias"]))
        k2 = [p + ".block2.block.0.weight", p + ".block2.block.0.bias", p + ".block2.block.3.weight",
              p + ".block2.block.3.bias"]
        if cin != cout:
            k2 += [p + ".res_conv.weight", p + ".res_conv.bias"]
        ops.append(dict(name=name + ".block2", kind="block2", inputs=[name + ".h"] + list(srcs), output=out,
                        block=name, resid="res_conv" if cin != cout else "identity", keys=k2))

    cur, feats = None, []
    for e in downs:
        if e[0] == "stem":
            ops.append(dict(name=e[1], kind="stem", inputs=["xin"], output=e[1],
                            keys=[_p(e[1]) + ".weight", _p(e[1]) + ".bias"]))
        elif e[0] == "res":
            res(e[1], [cur], e[1], e[2], e[3])
        else:
            ops.append(dict(name=e[1], kind="down", inputs=[cur], output=e[1],
                            keys=[_p(e[1]) + ".conv.weight", _p(e[1]) + ".conv.bias"]))
        cur = e[1]
        feats.append(cur)
    c = mid[0][3]
    res("mid.0", [cur], "mid.0.res", c, c)
    q = _p("mid.0")
    ops.append(dict(name="mid.0.clam_slam", kind="gates", inputs=["mid.0.res"], output="mid.0",
                    keys=[q + ".ca.fc1.weight", q + ".ca.fc2.weight", q + ".sa.conv1.weight"]))
    res("mid.1", ["mid.0"], "mid.1", c, c)
    cur = "mid.1"
    for e in ups:
        if e[0] == "res":
            res(e[1], [cur, feats.pop()], e[1], e[2], e[3])
        else:
            ops.append(dict(name=e[1], kind="up", inputs=[cur], output=e[1],
                            keys=[_p(e[1]) + ".conv.weight", _p(e[1]) + ".conv.bias"]))
        cur = e[1]
    ops.append(dict(name="final_conv", kind="final", inputs=[cur], output="eps",
                    keys=[_p("final_conv.block.0.weight"), _p("final_conv.block.0.bias"),
                          _p("final_conv.block.3.weight"), _p("final_conv.block.3.bias")]))
    return ops


def exact_weights(sd):
    """Every conv / linear weight snapped to the bf16 grid, |w| < 2^-14 set to 0: exact in fp16 and in bf16, so that the
    library's weight rounding is the identity.  Biases and GroupNorm parameters are kept (the kernels use them in
    fp32)."""
    out = {}
    for k, v in sd.items():
        if k.endswith(".weight") and v.dim() >= 2:
            w = v.to(torch.bfloat16).to(torch.float32)
            out[k] = torch.where(w.abs() < 2.0 ** -14, torch.zeros_like(w), w)
        else:
            out[k] = v
    return out


def xin_pack(cond, x):
    """The packed 16-channel network input (fdsr.h, fdsr_create): x_t in channels [0, C), cond in [P, P + C) with P = 4
    for C <= 4 and 8 otherwise, every other channel 0."""
    B, C, H, W = cond.shape
    P = 4 if C <= 4 else 8
    out = torch.zeros(B, 16, H, W, dtype=cond.dtype)
    out[:, :C] = x
    out[:, P:P + C] = cond
    return out


def time_embedding(sd, cfg, noise_level):
    """(B, inner) noise-level embedding (unet.py:22-35, 242-248) in float64."""
    d = torch.float64
    inner = cfg["inner_channel"]
    t = O.noise_embedding(noise_level.to(d), inner).reshape(noise_level.shape[0], inner)
    t = F.linear(t, sd[_p("noise_level_mlp.1.weight")].to(d), sd[_p("noise_level_mlp.1.bias")].to(d))
    t = F.linear(O._swish(t), sd[_p("noise_level_mlp.3.weight")].to(d), sd[_p("noise_level_mlp.3.bias")].to(d))
    return t


def _gn(x, gamma, beta, groups):
    """GroupNorm in float64 with the statistics of x itself (the tensor the kernel read)."""
    B, C, H, W = x.shape
    xg = x.reshape(B, groups, -1)
    mean = xg.mean(-1, keepdim=True)
    var = ((xg - mean) ** 2).mean(-1, keepdim=True)
    g = ((xg - mean) / torch.sqrt(var + 1e-5)).reshape(B, C, H, W)
    return g * gamma.view(1, -1, 1, 1) + beta.view(1, -1, 1, 1)


class _Acc:
    """ref (float64) and the two bound sums (float32 is plenty for a bound)."""

    def __init__(self):
        self.ref, self.op2, self.acc = 0.0, 0.0, 0.0

    def conv(self, a, w, g=None, **kw):
        """sum_k w_k a_k over conv taps; g given: the operand-error term of a GroupNorm (or phase) chunk."""
        self.ref = self.ref + F.conv2d(a, w.to(torch.float64), **kw)
        a32, w32 = a.float(), w.float()
        self.acc = self.acc + F.conv2d(a32.abs(), w32.abs(), **kw)
        if g is not None:
            self.op2 = self.op2 + F.conv2d((a32.abs() + g.float().abs()) ** 2, w32 * w32, **kw)

    def add(self, v):
        self.ref = self.ref + v
        self.acc = self.acc + v.float().abs()


def reference(op, inputs, sd, temb, cfg):
    """Evaluate `op` in float64 on `inputs` ({tensor name: (B,C,H,W)}, the tensors the kernel read).
    temb: (B, inner) float64 `time_embedding`.  Returns (ref, terms) with terms = {"op": sqrt-sum of the GroupNorm /
    phase operand term, "acc": sum of |w a| (+ |bias| ...)}, each shaped like ref."""
    d = torch.float64
    groups = cfg.get("norm_groups") or 32
    x = [inputs[n].to(d) for n in op["inputs"]]
    S = _Acc()
    kind = op["kind"]
    if kind == "gates":
        q = _p("mid.0")
        y = x[0]
        w1, w2, w7 = (sd[q + s].to(d) for s in (".ca.fc1.weight", ".ca.fc2.weight", ".sa.conv1.weight"))
        avg, mx = F.adaptive_avg_pool2d(y, 1), F.adaptive_max_pool2d(y, 1)
        gate = F.conv2d(F.relu(F.conv2d(avg, w1)), w2) + F.conv2d(F.relu(F.conv2d(mx, w1)), w2)
        y = torch.sigmoid(gate) * y
        sp = torch.cat([y.mean(dim=1, keepdim=True), y.max(dim=1, keepdim=True)[0]], dim=1)
        ref = torch.sigmoid(F.conv2d(sp, w7, padding=3)) * y
        n = y.shape[1] + 98
        return ref, {"op": torch.zeros_like(ref, dtype=torch.float32), "acc": ref.float().abs() * n}
    if kind == "stem":
        C = cfg["out_channel"]
        P = 4 if C <= 4 else 8
        xin = x[0]
        S.conv(torch.cat([xin[:, P:P + C], xin[:, :C]], 1), sd[op["keys"][0]], padding=1)
        S.add(sd[op["keys"][1]].to(d).view(1, -1, 1, 1).expand_as(S.ref))
    elif kind == "down":
        S.conv(x[0], sd[op["keys"][0]], stride=2, padding=1)
        S.add(sd[op["keys"][1]].to(d).view(1, -1, 1, 1).expand_as(S.ref))
    elif kind == "up":
        u = F.interpolate(x[0], scale_factor=2, mode="nearest")
        S.conv(u, sd[op["keys"][0]], g=torch.zeros_like(u), padding=1)
        S.add(sd[op["keys"][1]].to(d).view(1, -1, 1, 1).expand_as(S.ref))
    else:  # block1, block2, final: GroupNorm + Swish over the (virtual) concat of the GroupNorm sources
        gsrc = x[:len(x) if kind != "block2" else 1]
        cat = torch.cat(gsrc, 1) if len(gsrc) > 1 else gsrc[0]
        g = _gn(cat, sd[op["keys"][0]].to(d), sd[op["keys"][1]].to(d), groups)
        a = O._swish(g)
        S.conv(a, sd[op["keys"][2]], g=g, padding=1)
        S.add(sd[op["keys"][3]].to(d).view(1, -1, 1, 1).expand_as(S.ref))
        if kind == "block1":
            p = _p(op["block"]) + ".res_block.noise_func.noise_func.0"
            film = F.linear(temb.to(d), sd[p + ".weight"].to(d), sd[p + ".bias"].to(d))
            S.add(film.view(film.shape[0], -1, 1, 1).expand_as(S.ref))
        elif kind == "block2":
            r = torch.cat(x[1:], 1) if len(x) > 2 else x[1]
            if op["resid"] == "res_conv":
                p = _p(op["block"]) + ".res_block.res_conv"
                S.conv(r, sd[p + ".weight"])
                S.add(sd[p + ".bias"].to(d).view(1, -1, 1, 1).expand_as(S.ref))
            else:
                S.add(r)
    return S.ref, {"op": torch.sqrt(S.op2) if torch.is_tensor(S.op2) else torch.zeros_like(S.ref, dtype=torch.float32),
                   "acc": S.acc}


def bound(op, ref, terms, mode):
    """(rounding part u_out |ref| + floor, modelled part rho_op ... + rho_acc ...) of the allowed |got - ref|."""
    rho_op, rho_acc = RHO[mode]
    if op["kind"] == "up":
        rho_op = RHO_W[mode]
    final16 = op["kind"] == "final" and mode != "fp32"
    u = 0.0 if final16 else U_OUT[mode]
    floor = FLOOR["fp32" if final16 else mode]
    return u * ref.abs() + floor, rho_op * terms["op"].double() + rho_acc * terms["acc"].double()


def check(op, got, ref, terms, mode, tile_h=TILE_H):
    """(ratio, excess, loc):
      ratio   largest |got - ref| / bound; the op passes with ratio <= 1;
      excess  largest (|got - ref| - rounding part) / modelled part: how much of the rho terms the op used (the
              rounding part is exact theory, so the calibration keeps excess <= 0.5 rather than ratio);
      loc     where the ratio peaks: dict(image, y, x, channel, tile=(ty, tx) on the tile_h x 8 grid, got, ref, err,
              bound).
    A non-finite `got` gives infinite ratios."""
    got = got.to(torch.float64)
    rnd, mod = bound(op, ref, terms, mode)
    err = (got - ref).abs()
    bad = ~torch.isfinite(got)
    ratio = torch.where(bad, torch.full_like(err, math.inf), err / (rnd + mod))
    excess = torch.where(bad, torch.full_like(err, math.inf), (err - rnd).clamp_min(0) / mod.clamp_min(1e-300))
    i = int(torch.argmax(ratio))
    b, c, y, x = (int(v) for v in torch.unravel_index(torch.tensor(i), ratio.shape))
    loc = dict(image=b, y=y, x=x, channel=c, tile=(y // tile_h, x // TILE_W), got=float(got[b, c, y, x]),
               ref=float(ref[b, c, y, x]), err=float(err[b, c, y, x]), bound=float((rnd + mod)[b, c, y, x]))
    return float(ratio[b, c, y, x]), float(excess.max()), loc


def store(ref, op, mode):
    """What a kernel without error would store: ref rounded to the output format (fp32 for the final conv's eps)."""
    fmt = torch.float32 if op["kind"] == "final" else STORE[mode]
    return ref.to(fmt).to(torch.float64)


def chain(sd, cfg, cond, x, noise_level, mode=None):
    """Run every op of plan_ops(cfg) on the previous ops' reference outputs (rounded to `mode`'s storage format if
    given, else kept in float64).  Returns {tensor name: tensor} including "xin" and "eps"."""
    temb = time_embedding(sd, cfg, noise_level)
    t = {"xin": xin_pack(cond.double(), x.double())}
    if mode is not None:
        t["xin"] = t["xin"].to(STORE[mode]).double()
    for op in plan_ops(cfg):
        ref, _ = reference(op, t, sd, temb, cfg)
        t[op["output"]] = ref if mode is None else store(ref, op, mode)
    return t

"""Python owner of one libfdsr context: device memory and streams come from torch, compute from
the C ABI.  One Engine per (process, GPU)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import FdsrConfig, FdsrError, FdsrOverflowError

_DTYPES = {"auto": _lib.DTYPE_FP16, "fp16": _lib.DTYPE_FP16, "float16": _lib.DTYPE_FP16, "bf16": _lib.DTYPE_BF16, "bfloat16": _lib.DTYPE_BF16,
           "fp32": _lib.DTYPE_FP32, "float32": _lib.DTYPE_FP32}  # fp32 = CUDA-core parity mode (slow)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class Engine:
    def __init__(self, unet_cfg: dict, device, dtype: str = "fp16"):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise FdsrError("fastdiffsr_b200 runs on CUDA (sm_100a) devices only; there is no CPU fallback")
        mults = list(unet_cfg["channel_multiplier"])
        cfg = FdsrConfig()
        cfg.in_channel = unet_cfg["in_channel"]
        cfg.out_channel = unet_cfg["out_channel"]
        cfg.inner_channel = unet_cfg["inner_channel"]
        cfg.norm_groups = unet_cfg.get("norm_groups") or 32
        cfg.n_levels = len(mults)
        for i, m in enumerate(mults):
            cfg.channel_mults[i] = m
        cfg.res_blocks = unet_cfg["res_blocks"]
        cfg.dtype = _DTYPES[dtype]
        # which_model_G: "fastdiffsr" (default) or "ddpm" = the SR3 baseline, whose ResnetBlocks carry SelfAttention
        # where the resolution of the *configured* image_size is in attn_res (ddpm_modules/unet.py:184, 211)
        self.model = unet_cfg.get("model", "fastdiffsr")
        if self.model not in ("fastdiffsr", "ddpm"):
            raise FdsrError(f"unknown model {self.model!r}")
        cfg.model = _lib.MODEL_SR3 if self.model == "ddpm" else _lib.MODEL_FASTDIFFSR
        cfg.attn_levels = 0
        if self.model == "ddpm":
            res = int(unet_cfg.get("image_size", 256))
            for i in range(len(mults)):
                if res in list(unet_cfg["attn_res"]):
                    cfg.attn_levels |= 1 << i
                res //= 2
        self.dtype = dtype
        self.C = int(cfg.out_channel)  # image bands: every image tensor is (B,C,H,W), u8 images (B,h,w,C)
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            rc = self.lib.fdsr_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise FdsrError("fdsr_create: " + self.lib.fdsr_global_error().decode())
        self.T = 0

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.fdsr_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc < 0:
            cls = FdsrOverflowError if rc == _lib.E_OVERFLOW else FdsrError
            raise cls(f"{what}: {self.lib.fdsr_last_error(self._h).decode()} (code {rc})")
        return rc

    def _call(self, fn_name, *args):
        """self.lib.<fn_name>(handle, *args) on this engine's device; a negative return code raises."""
        with torch.cuda.device(self.device):
            return self._check(getattr(self.lib, fn_name)(self._h, *args), fn_name)

    def check_overflow(self):
        """fp16 mode: synchronise the current stream and raise FdsrOverflowError if an activation left the fp16 range
        since the last check (the value was stored saturated; the result is not the network's output)."""
        if self.dtype not in ("fp16", "float16"):
            return
        self._call("fdsr_check_overflow", self._stream())

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- weights / schedule
    def load_state_dict(self, sd: dict):
        """Tensors that already live on this engine's GPU are handed over as device pointers (fdsr_load_weights_dev);
        anything else goes through host memory (fdsr_load_weights)."""
        items = [(k, v.detach()) for k, v in sd.items() if k.startswith("denoise_fn.")]
        on_dev = bool(items) and all(v.device == self.device for _, v in items)
        items = [(k, v.to(torch.float32).contiguous() if on_dev else v.to("cpu", torch.float32).contiguous())
                 for k, v in items]
        n = len(items)
        names = (C.c_char_p * n)(*[k.encode() for k, _ in items])
        ptrs = (C.c_void_p * n)(*[v.data_ptr() for _, v in items])
        numels = (C.c_int64 * n)(*[v.numel() for _, v in items])
        if on_dev:
            self._call("fdsr_load_weights_dev", names, ptrs, numels, n, self._stream())
        else:
            self._call("fdsr_load_weights", names, ptrs, numels, n)

    def set_schedule(self, betas):
        b = np.ascontiguousarray(np.asarray(betas, dtype=np.float64))
        self._call("fdsr_set_schedule", b.ctypes.data_as(C.POINTER(C.c_double)), len(b))
        self.T = len(b)

    def table(self, name: str):
        buf = (C.c_double * (self.T + 1))()
        n = self._call("fdsr_get_table", name.encode(), buf, self.T + 1)
        return np.array(buf[:n], dtype=np.float64)

    # ---- compute
    def _img(self, t, name):
        if t.device != self.device or t.dtype != torch.float32 or t.dim() != 4 or t.shape[1] != self.C:
            raise FdsrError(f"{name} must be a (B,{self.C},H,W) fp32 tensor on {self.device}")
        return t.contiguous()

    def unet_forward(self, cond, x_t, t: int):
        cond, x_t = self._img(cond, "cond"), self._img(x_t, "x_t")
        B, _, H, W = cond.shape
        out = torch.empty_like(cond)
        self._call("fdsr_unet_forward", _ptr(cond), _ptr(x_t), t, _ptr(out), B, H, W, self._stream())
        return out

    def posterior_step(self, x_t, eps, z, t: int):
        x_t, eps = x_t.contiguous(), eps.contiguous()
        z = z.contiguous() if z is not None else None
        out = torch.empty_like(x_t)
        self._call("fdsr_posterior_step", _ptr(x_t), _ptr(eps), _ptr(z), t, _ptr(out), x_t.numel(), self._stream())
        return out

    def trace_frames(self):
        return self.lib.fdsr_trace_frames(self._h)

    def _sample_io(self, cond, noise, trace, image_offset):
        """The preamble of sample / sample_tiled: image offset, checked inputs, output and trace tensors."""
        self._call("fdsr_set_image_offset", int(image_offset))
        cond = self._img(cond, "cond")
        B, _, H, W = cond.shape
        if noise is not None:
            if tuple(noise.shape) != (self.T, B, self.C, H, W) or noise.dtype != torch.float32 or noise.device != self.device:
                raise FdsrError(f"noise must be ({self.T},{B},{self.C},{H},{W}) fp32 on {self.device}")
            noise = noise.contiguous()
        out = torch.empty_like(cond)
        tr = torch.empty((B, self.trace_frames(), self.C, H, W), device=self.device, dtype=torch.float32) if trace else None
        return cond, noise, out, tr

    def sample(self, cond, noise=None, seed: int = 0, trace: bool = False, image_offset: int = 0):
        """T-step sampling of a batch.  `image_offset` = global index of cond[0] in the whole job: the built-in noise of
        an image depends on (seed, global index, step) only, so shards of a job reproduce the unsharded result."""
        cond, noise, out, tr = self._sample_io(cond, noise, trace, image_offset)
        B, _, H, W = cond.shape
        self._call("fdsr_sample", _ptr(cond), _ptr(noise), seed, _ptr(out), _ptr(tr), B, H, W, self._stream())
        return (out, tr) if trace else out

    def _valid(self, valid, B, H, W):
        """A (B,H,W) bool or uint8 validity mask on this engine's device (nonzero = valid), as contiguous uint8."""
        if (not isinstance(valid, torch.Tensor) or valid.dtype not in (torch.bool, torch.uint8)
                or tuple(valid.shape) != (B, H, W) or valid.device != self.device):
            raise FdsrError(f"valid must be a ({B},{H},{W}) bool or uint8 tensor on {self.device}")
        valid = valid.contiguous()
        return valid.view(torch.uint8) if valid.dtype == torch.bool else valid

    def sample_tiled(self, cond, tile, overlap: int = 32, tile_batch: int = 16, noise=None, seed: int = 0,
                     trace: bool = False, image_offset: int = 0, valid=None):
        """T-step sampling of (B,C,H,W) canvases of any size (H, W >= 8) as overlapping tiles blended at every step
        (fdsr_sample_tiled).  `tile`: int or (th, tw), multiples of 8; `tile_batch`: tiles per UNet call (the activation
        workspace scales with it, not with the canvas).  Noise, seed, image_offset and the trace are as in `sample`.
        `valid`: a (B,H,W) bool / uint8 mask, nonzero = valid (fdsr_sample_tiled_masked): only the tiles that hold a
        valid pixel go through the UNet, and invalid pixels of the result and trace are cond itself."""
        th, tw = (tile, tile) if isinstance(tile, int) else (int(tile[0]), int(tile[1]))
        cond, noise, out, tr = self._sample_io(cond, noise, trace, image_offset)
        B, _, H, W = cond.shape
        if valid is None:
            self._call("fdsr_sample_tiled", _ptr(cond), _ptr(noise), seed, _ptr(out), _ptr(tr), B, H, W, th, tw,
                       int(overlap), int(tile_batch), self._stream())
        else:
            valid = self._valid(valid, B, H, W)
            self._call("fdsr_sample_tiled_masked", _ptr(cond), _ptr(valid), _ptr(noise), seed, _ptr(out), _ptr(tr), B,
                       H, W, th, tw, int(overlap), int(tile_batch), self._stream())
        return (out, tr) if trace else out

    @staticmethod
    def tiled_plan(B: int, H: int, W: int, tile, overlap: int, world: int, rank: int):
        """The exchange plan of `rank` for a tiled job split over `world` ranks (fdsr_tiled_plan; host only, no
        context or GPU needed): {"n_tiles", "te": (te_y, te_x), "own": (lo, hi), "send": [(lo, hi)] * world,
        "recv": [(lo, hi)] * world}, ranges of global tile slots, (0, 0) = nothing."""
        th, tw = (tile, tile) if isinstance(tile, int) else (int(tile[0]), int(tile[1]))
        lib = _lib.load()
        buf = (C.c_int64 * (5 + 4 * max(int(world), 1)))()
        rc = lib.fdsr_tiled_plan(B, H, W, th, tw, int(overlap), int(world), int(rank), buf, len(buf))
        if rc < 0:
            raise FdsrError(f"fdsr_tiled_plan: {lib.fdsr_global_error().decode()} (code {rc})")
        peers = [tuple(buf[5 + 4 * q:9 + 4 * q]) for q in range(world)]
        return {"n_tiles": buf[0], "te": (buf[1], buf[2]), "own": (buf[3], buf[4]),
                "send": [p[:2] for p in peers], "recv": [p[2:] for p in peers]}

    def sample_tiled_part(self, cond, tile, overlap: int = 32, tile_batch: int = 16, noise=None, seed: int = 0,
                          trace: bool = False, image_offset: int = 0, rank: int = 0, world: int = 1, exchange=None):
        """Rank `rank`'s part of sample_tiled split over `world` ranks (fdsr_sample_tiled_part): every rank passes the
        same arguments except tile_batch.  Allocates the (n_tiles, C, te_y, te_x) fp32 eps store and calls
        exchange(step, eps_store) once per step, on the host, between the own tiles' eps and the blend: it must move the
        plan's slot ranges (tiled_plan) on the current stream.  Returns the rank's pixels of the result (and trace),
        +0.0 elsewhere: the int32 bit patterns of all ranks sum to sample_tiled's bits.  An exception raised by
        `exchange` aborts the call and is re-raised here."""
        th, tw = (tile, tile) if isinstance(tile, int) else (int(tile[0]), int(tile[1]))
        cond, noise, out, tr = self._sample_io(cond, noise, trace, image_offset)
        B, _, H, W = cond.shape
        plan = self.tiled_plan(B, H, W, (th, tw), overlap, world, rank)
        store = torch.empty((plan["n_tiles"], self.C) + tuple(plan["te"]), dtype=torch.float32, device=self.device)
        errors = []

        def call_exchange(user, step, stream):
            try:
                exchange(int(step), store)
                return 0
            except BaseException as e:     # never unwind through the C frames
                errors.append(e)
                return 1
        fn = _lib.TILE_EXCHANGE_FN(call_exchange) if exchange is not None else _lib.TILE_EXCHANGE_FN()
        with torch.cuda.device(self.device):
            rc = self.lib.fdsr_sample_tiled_part(self._h, _ptr(cond), _ptr(noise), seed, _ptr(out), _ptr(tr), B, H, W,
                                                 th, tw, int(overlap), int(tile_batch), int(rank), int(world),
                                                 _ptr(store), fn, None, self._stream())
        if errors:
            raise errors[0]
        self._check(rc, "fdsr_sample_tiled_part")
        return (out, tr) if trace else out

    def bicubic_u8(self, lr_u8, H: int, W: int, want_u8=True, want_cond=True):
        """lr_u8: (B,h,w,C) uint8 on device -> (u8 (B,H,W,C) | None, cond (B,C,H,W) fp32 | None)."""
        if lr_u8.dtype != torch.uint8 or lr_u8.dim() != 4 or lr_u8.shape[3] != self.C or lr_u8.device != self.device:
            raise FdsrError(f"lr must be (B,h,w,{self.C}) uint8 on the engine's device")
        lr_u8 = lr_u8.contiguous()
        B, h, w, _ = lr_u8.shape
        o8 = torch.empty((B, H, W, self.C), dtype=torch.uint8, device=self.device) if want_u8 else None
        oc = torch.empty((B, self.C, H, W), dtype=torch.float32, device=self.device) if want_cond else None
        self._call("fdsr_bicubic_u8", _ptr(lr_u8), B, h, w, H, W, _ptr(o8), _ptr(oc), self._stream())
        return o8, oc

    def bicubic_u16(self, lr_u16, H: int, W: int, max_value: int, want_u16=True, want_cond=True):
        """lr_u16: (B,h,w,C) torch.uint16 on device -> (u16 (B,H,W,C) | None, cond (B,C,H,W) fp32 | None): each band
        resized as Pillow resizes an 'I;16' image, cond = (min(v, max_value) / max_value) * 2 - 1 (fdsr_bicubic_u16)."""
        if lr_u16.dtype != torch.uint16 or lr_u16.dim() != 4 or lr_u16.shape[3] != self.C or lr_u16.device != self.device:
            raise FdsrError(f"lr must be (B,h,w,{self.C}) uint16 on the engine's device")
        lr_u16 = lr_u16.contiguous()
        B, h, w, _ = lr_u16.shape
        o16 = torch.empty((B, H, W, self.C), dtype=torch.uint16, device=self.device) if want_u16 else None
        oc = torch.empty((B, self.C, H, W), dtype=torch.float32, device=self.device) if want_cond else None
        self._call("fdsr_bicubic_u16", _ptr(lr_u16), B, h, w, H, W, int(max_value), _ptr(o16), _ptr(oc), self._stream())
        return o16, oc

    def debug_noise(self, B: int, H: int, W: int, seed: int, stream_id: int, image_offset: int = 0):
        """(B,C,H,W) N(0,1) values of the built-in generator for step stream `stream_id` (T: x_T, t: z of step t)."""
        out = torch.empty((B, self.C, H, W), dtype=torch.float32, device=self.device)
        self._call("fdsr_debug_noise", _ptr(out), B, H, W, int(seed), int(image_offset), int(stream_id), self._stream())
        return out

    def graph_captures(self):
        return int(self.lib.fdsr_graph_captures(self._h))

    def _host_u8(self, lr_host):
        lr_host = np.ascontiguousarray(lr_host, dtype=np.uint8)
        if lr_host.ndim != 4 or lr_host.shape[3] != self.C:
            raise FdsrError(f"lr must be a (B,h,w,{self.C}) uint8 array")
        return lr_host

    def super_resolve_u8_host(self, lr_host: np.ndarray, H: int, W: int, noise=None, seed: int = 0, out=None,
                              image_offset: int = 0):
        """Host uint8 (B,h,w,C) -> host fp32 (B,C,H,W): H2D, bicubic, T-step sampling, D2H.
        `out`: optional caller-owned C-contiguous float32 (B,C,H,W) array to fill (avoids a fresh allocation per call)."""
        lr_host = self._host_u8(lr_host)
        B, h, w, _ = lr_host.shape
        if out is None:
            out = np.empty((B, self.C, H, W), dtype=np.float32)
        elif out.shape != (B, self.C, H, W) or out.dtype != np.float32 or not out.flags["C_CONTIGUOUS"]:
            raise FdsrError(f"out must be a C-contiguous float32 array of shape {(B, self.C, H, W)}")
        self._call("fdsr_set_image_offset", int(image_offset))
        self._call("fdsr_super_resolve_u8", lr_host.ctypes.data_as(C.c_void_p), B, h, w, H, W, _ptr(noise), seed,
                   out.ctypes.data_as(C.c_void_p), self._stream())
        return out

    def super_resolve_u8_submit(self, slot: int, lr_host: np.ndarray, H: int, W: int, noise=None, seed: int = 0,
                                image_offset: int = 0):
        """Pipelined host path: enqueue one batch into `slot` (0 / 1) and return; see super_resolve_u8_wait."""
        lr_host = self._host_u8(lr_host)
        B, h, w, _ = lr_host.shape
        self._call("fdsr_set_image_offset", int(image_offset))
        self._call("fdsr_super_resolve_u8_submit", slot, lr_host.ctypes.data_as(C.c_void_p), B, h, w, H, W, _ptr(noise),
                   seed, self._stream())
        return (B, self.C, H, W)

    def super_resolve_u8_wait(self, slot: int, out: np.ndarray):
        """Block until the batch in `slot` is on the host; fills the C-contiguous float32 array `out`."""
        if out.dtype != np.float32 or not out.flags["C_CONTIGUOUS"]:
            raise FdsrError("out must be a C-contiguous float32 array")
        self._call("fdsr_super_resolve_u8_wait", slot, out.ctypes.data_as(C.c_void_p))
        return out

    def sse_u8(self, a, b):
        a, b = self._img(a, "a"), self._img(b, "b")
        B, _, H, W = a.shape
        out = torch.empty(B, dtype=torch.float64, device=self.device)
        self._call("fdsr_sse_u8", _ptr(a), _ptr(b), B, H, W, _ptr(out), self._stream())
        return out

    def metrics_u8(self, a, b, scale: float = 4.0, valid=None):
        """Per-image (mse, psnr, ssim, ergas) of `a` (SR or bicubic image) against `b` (HR), both (B,C,H,W) fp32
        in [-1,1]: the reference's evaluation block (sr_mfe.py:315-345) on the device.  Returns (B,4) float64.
        `valid`: a (B,H,W) bool / uint8 mask: score the valid pixels only (fdsr_metrics_masked at 255)."""
        if valid is not None:
            return self.metrics_u16(a, b, 255, scale, valid=valid)
        a, b = self._img(a, "a"), self._img(b, "b")
        B, _, H, W = a.shape
        out = torch.empty((B, 4), dtype=torch.float64, device=self.device)
        self._call("fdsr_metrics_u8", _ptr(a), _ptr(b), B, H, W, float(scale), _ptr(out), self._stream())
        return out

    def metrics_u16(self, a, b, max_value: int, scale: float = 4.0, valid=None):
        """metrics_u8 on images quantised to levels 0..max_value instead of 0..255 (fdsr_metrics_u16): PSNR against
        max_value^2, SSIM with data_range max_value.  max_value = 255 gives metrics_u8's bits.  Returns (B,4) float64.
        `valid`: a (B,H,W) bool / uint8 mask: MSE, PSNR and ERGAS over the valid pixels, SSIM over the windows that
        are wholly valid, NaN where nothing qualifies (fdsr_metrics_masked)."""
        a, b = self._img(a, "a"), self._img(b, "b")
        B, _, H, W = a.shape
        out = torch.empty((B, 4), dtype=torch.float64, device=self.device)
        if valid is None:
            self._call("fdsr_metrics_u16", _ptr(a), _ptr(b), B, H, W, int(max_value), float(scale), _ptr(out),
                       self._stream())
        else:
            valid = self._valid(valid, B, H, W)
            self._call("fdsr_metrics_masked", _ptr(a), _ptr(b), _ptr(valid), B, H, W, int(max_value), float(scale),
                       _ptr(out), self._stream())
        return out

    # ---- hooks
    def tensor_names(self):
        n = self.lib.fdsr_debug_num_tensors(self._h)
        return [self.lib.fdsr_debug_tensor_name(self._h, i).decode() for i in range(n)]

    def read_tensor(self, name: str, B: int, max_elems: int):
        buf = torch.empty(max_elems, dtype=torch.float32, device=self.device)
        c, h, w = C.c_int32(), C.c_int32(), C.c_int32()
        self._call("fdsr_debug_read_tensor", name.encode(), _ptr(buf), max_elems, C.byref(c), C.byref(h), C.byref(w),
                   self._stream())
        n = B * c.value * h.value * w.value
        return buf[:n].view(B, c.value, h.value, w.value)

    def op_flops_executed(self):
        """Executed conv FLOPs per op (phase-decomposed upsample convs at 4/9 of their nine-tap cost)."""
        n = self.lib.fdsr_debug_num_ops(self._h)
        return [float(self.lib.fdsr_debug_op_flops_executed(self._h, i)) for i in range(n)]

    OP_SCHEDULE_FIELDS = ("N", "pair", "tile_h", "nsplit", "group", "grid", "ntiles", "max_tiles", "epi2", "tail2", "nR",
                          "nG", "phases", "a_tma", "spans_image", "spans_phase", "nchunks")

    def op_names(self):
        return [self.lib.fdsr_debug_op_name(self._h, i).decode() for i in range(self.lib.fdsr_debug_num_ops(self._h))]

    def op_schedule(self, op: int):
        """The launch schedule of conv op `op` at the shape of the last forward (fdsr_debug_op_schedule), as a dict."""
        buf = (C.c_int32 * len(self.OP_SCHEDULE_FIELDS))()
        n = self._call("fdsr_debug_op_schedule", op, buf, len(buf))
        return dict(zip(self.OP_SCHEDULE_FIELDS, buf[:n]))

    def profile_unet(self, t: int, reps: int = 3):
        """[(op name, mean ms, algorithmic conv FLOPs)] for one UNet evaluation at the current shape."""
        n = self.lib.fdsr_debug_num_ops(self._h)
        ms = (C.c_float * n)()
        self._call("fdsr_debug_profile_unet", t, reps, ms, n, self._stream())
        return [(self.lib.fdsr_debug_op_name(self._h, i).decode(), float(ms[i]),
                 float(self.lib.fdsr_debug_op_flops(self._h, i))) for i in range(n)]

    def role_cycles(self, op: int, t: int = 0):
        """(n_cta, 5 roles, 8 slots) cycle counters of conv op `op` (FDSR_PROFILE builds only)."""
        n = 148 * 40 * 2
        buf = (C.c_int64 * n)()
        m = self._call("fdsr_debug_role_cycles", op, t, buf, n, self._stream())
        return np.array(buf[:m], dtype=np.int64).reshape(-1, 5, 8)

    def timeline(self, t: int = 0, reps: int = 3):
        """(n_ops, n_sms, 5 roles, 8 slots): the same counters of every conv op inside a running UNet evaluation
        (FDSR_PROFILE builds only; tools/timeline.py)."""
        nops = int(self.lib.fdsr_debug_num_ops(self._h))
        nsm = torch.cuda.get_device_properties(self.device).multi_processor_count
        out = np.zeros((nops, nsm, 5, 8), dtype=np.int64)
        self._call("fdsr_debug_timeline", t, reps, out.ctypes.data_as(C.POINTER(C.c_int64)), out.size, self._stream())
        return out

    def launch_count(self):
        return int(self.lib.fdsr_launch_count(self._h))

    def unet_flops(self):
        return float(self.lib.fdsr_unet_flops(self._h))

    def reserve(self, B, H, W):
        self._call("fdsr_reserve", B, H, W)

    def workspace_bytes(self):
        return int(self.lib.fdsr_workspace_bytes(self._h))

    def set_use_graph(self, enable: bool):
        self.lib.fdsr_set_use_graph(self._h, 1 if enable else 0)

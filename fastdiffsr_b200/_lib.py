"""ctypes binding of libfdsr.so (the C ABI declared in include/fdsr.h).

There is deliberately no fallback: if the shared library is missing, or no sm_100 GPU is
visible when a context is created, the caller gets an exception.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FDSR_LIB", os.path.join(_HERE, "libfdsr.so"))
CSRC = os.path.join(_HERE, "csrc")
MAX_LEVELS = 8
DTYPE_FP16, DTYPE_BF16, DTYPE_FP32 = 0, 1, 2
MODEL_FASTDIFFSR, MODEL_SR3 = 0, 1

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


class FdsrConfig(C.Structure):
    _fields_ = [("in_channel", C.c_int32), ("out_channel", C.c_int32), ("inner_channel", C.c_int32),
                ("norm_groups", C.c_int32), ("n_levels", C.c_int32), ("channel_mults", C.c_int32 * MAX_LEVELS),
                ("res_blocks", C.c_int32), ("dtype", C.c_int32), ("model", C.c_int32), ("attn_levels", C.c_int32)]


class FdsrError(RuntimeError):
    pass


class FdsrOverflowError(FdsrError, FloatingPointError):
    """fp16 mode: an activation left the fp16 range during the call (FDSR_E_OVERFLOW)."""


E_OVERFLOW = -5

# fdsr_tile_exchange_fn: int (*)(void* user, int32_t step, void* stream)
TILE_EXCHANGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int32, C.c_void_p)


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile libfdsr.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    newest = max(os.path.getmtime(s) for s in srcs + [os.path.join(_HERE, "..", "include", "fdsr.h")])
    if not force and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= newest:
        return LIB_PATH
    cmd = ["nvcc", *NVCC_FLAGS, "-o", LIB_PATH, os.path.join(CSRC, "api.cu")]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB_PATH


_lib = None

_SIGS = {
    "fdsr_create": (C.c_int, [C.POINTER(FdsrConfig), C.POINTER(C.c_void_p)]),
    "fdsr_destroy": (C.c_int, [C.c_void_p]),
    "fdsr_last_error": (C.c_char_p, [C.c_void_p]),
    "fdsr_global_error": (C.c_char_p, []),
    "fdsr_load_weights": (C.c_int, [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(C.c_void_p),
                                    C.POINTER(C.c_int64), C.c_int32]),
    "fdsr_load_weights_dev": (C.c_int, [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(C.c_void_p),
                                        C.POINTER(C.c_int64), C.c_int32, C.c_void_p]),
    "fdsr_set_schedule": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_int32]),
    "fdsr_get_table": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double), C.c_int32]),
    "fdsr_reserve": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32]),
    "fdsr_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "fdsr_unet_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                    C.c_int32, C.c_int32, C.c_void_p]),
    "fdsr_posterior_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                      C.c_int64, C.c_void_p]),
    "fdsr_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                              C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "fdsr_sample_tiled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_void_p]),
    "fdsr_tiled_plan": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_int32, C.POINTER(C.c_int64), C.c_int64]),
    "fdsr_sample_tiled_part": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                         C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                         C.c_int32, C.c_int32, C.c_void_p, TILE_EXCHANGE_FN, C.c_void_p, C.c_void_p]),
    "fdsr_sample_tiled_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p,
                                           C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                           C.c_int32, C.c_int32, C.c_void_p]),
    "fdsr_trace_frames": (C.c_int32, [C.c_void_p]),
    "fdsr_super_resolve_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_int32, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "fdsr_super_resolve_u8_submit": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                               C.c_int32, C.c_int32, C.c_void_p, C.c_uint64, C.c_void_p]),
    "fdsr_super_resolve_u8_wait": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "fdsr_bicubic_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    "fdsr_sse_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                              C.c_void_p]),
    "fdsr_metrics_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_double,
                                  C.c_void_p, C.c_void_p]),
    "fdsr_bicubic_u16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "fdsr_metrics_u16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_double, C.c_void_p, C.c_void_p]),
    "fdsr_metrics_masked": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.c_void_p]),
    "fdsr_debug_num_tensors": (C.c_int32, [C.c_void_p]),
    "fdsr_debug_tensor_name": (C.c_char_p, [C.c_void_p, C.c_int32]),
    "fdsr_debug_read_tensor": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int32),
                                         C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_void_p]),
    "fdsr_debug_num_ops": (C.c_int32, [C.c_void_p]),
    "fdsr_debug_op_name": (C.c_char_p, [C.c_void_p, C.c_int32]),
    "fdsr_debug_op_flops": (C.c_double, [C.c_void_p, C.c_int32]),
    "fdsr_debug_op_flops_executed": (C.c_double, [C.c_void_p, C.c_int32]),
    "fdsr_debug_op_schedule": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32]),
    "fdsr_debug_profile_unet": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.c_int32,
                                          C.c_void_p]),
    "fdsr_debug_role_cycles": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.c_int32,
                                         C.c_void_p]),
    "fdsr_debug_timeline": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.c_int64, C.c_void_p]),
    "fdsr_check_overflow": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fdsr_set_image_offset": (C.c_int, [C.c_void_p, C.c_uint64]),
    "fdsr_debug_noise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_uint64,
                                   C.c_int32, C.c_void_p]),
    "fdsr_graph_captures": (C.c_int64, [C.c_void_p]),
    "fdsr_launch_count": (C.c_int64, [C.c_void_p]),
    "fdsr_unet_flops": (C.c_double, [C.c_void_p]),
    "fdsr_set_use_graph": (C.c_int, [C.c_void_p, C.c_int32]),
}
EXPORTS = tuple(_SIGS)


def load():
    """Load libfdsr.so (once) and attach argument/return types."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FdsrError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU or PyTorch fallback for this path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib

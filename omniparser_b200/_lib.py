"""ctypes binding of ``libb200parse.so`` (the C-ABI declared in ``include/b200parse.h``).

The product path has no CPU fallback: if the shared library is missing, or a
call fails, this module raises.  ``build()`` compiles it in-tree with nvcc.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

HERE = Path(__file__).resolve().parent
LIB_PATH = HERE / "libb200parse.so"
CSRC = HERE / "csrc"

_lib = None

vp, i32, i64, f32, f64 = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_double

# name -> (restype, argtypes); mirrors include/b200parse.h
PROTOTYPES = {
    "b2p_last_error": (C.c_char_p, []),
    "b2p_launch_count": (i64, []),
    "b2p_trace_read": (i32, [vp, vp, i32]),
    "b2p_abi_version": (i32, []),
    "b2p_gemm": (i32, [vp, i64, vp, i32, i32, i32, vp, i64, vp, vp, i64, i32, i32, vp]),
    "b2p_conv3x3": (i32, [vp, i64, i32, i32, i32, i32, i32, vp, i32, vp, i64, vp, vp, i64, i32, i32, vp]),
    "b2p_gemm_planes": (i32, [vp, i64, vp, i32, i32, i32, vp, i64, vp, vp, i64, i32, i32, i64, i64, i64, vp]),
    "b2p_conv3x3_planes": (i32, [vp, i64, i32, i32, i32, i32, i32, vp, i32, vp, i64, vp, vp, i64, i32, i32, i64, i64, i64, vp]),
    "b2p_adown_pool": (i32, [vp, i64, i32, i32, i32, i32, vp, i64, vp, i64, vp]),
    "b2p_adown_pool_x3": (i32, [vp, i64, i32, i32, i32, i32, vp, i64, vp, i64, i64, i64, i64, vp]),
    "b2p_maxpool_s1_x3": (i32, [vp, i64, i32, i32, i32, i32, i32, vp, i64, i64, i64, vp]),
    "b2p_upsample2x_x3": (i32, [vp, i64, i32, i32, i32, i32, vp, i64, i64, i64, vp]),
    "b2p_cbfuse_x3": (i32, [i32, C.POINTER(vp), C.POINTER(i64), C.POINTER(i32), C.POINTER(i64), vp, i64, i32, i32, i32, i32, vp, i64, i64, i64, vp]),
    "b2p_maxpool_s1": (i32, [vp, i64, i32, i32, i32, i32, i32, vp, i64, vp]),
    "b2p_upsample2x": (i32, [vp, i64, i32, i32, i32, i32, vp, i64, vp]),
    "b2p_cbfuse": (i32, [i32, C.POINTER(vp), C.POINTER(i64), C.POINTER(i32), vp, i64, i32, i32, i32, i32, vp, i64, vp]),
    "b2p_yolo_decode": (i32, [C.POINTER(vp), C.POINTER(vp), C.POINTER(i32), C.POINTER(i32), i32, i32, f32, vp, vp, vp,
                              i32, vp, vp, vp, vp, vp, vp, vp]),
    "b2p_batched_nms": (i32, [vp, vp, vp, vp, i32, i32, f64, i32, vp, vp, vp, vp, vp, vp, vp]),
    "b2p_lanczos_coeffs_host": (i32, [i32, i32, C.POINTER(i32), vp, vp, i32]),
    "b2p_letterbox": (i32, [vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp, vp, vp]),
    "b2p_resize_u8": (i32, [vp, i32, i32, i32, i32, i32, i32, vp, vp, vp]),
    "b2p_im2col3x3": (i32, [vp, i64, i32, i32, i32, i32, i32, i32, vp, vp]),
    "b2p_im2col_u8": (i32, [vp, i32, i32, i32, i32, i32, i32, i32, vp, vp, i32, vp]),
    "b2p_overlap_filter": (i32, [vp, vp, i32, i32, vp, vp, vp, vp, i32, f64, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "b2p_crop_resize": (i32, [vp, vp, vp, vp, vp, i32, i32, vp, vp, vp]),
    "b2p_layernorm": (i32, [vp, i64, vp, vp, f32, i32, i32, vp, i64, vp, i64, i32, vp]),
    "b2p_dwconv_ln": (i32, [vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, f32, vp, i32, vp]),
    "b2p_window_attn": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, vp, i32, vp]),
    "b2p_channel_attn": (i32, [vp, i32, i32, i32, i32, vp, i32, vp]),
    "b2p_mha": (i32, [vp, i64, vp, vp, i64, i32, i32, i32, i32, vp, i64, i32, vp]),
    "b2p_mha_cached": (i32, [vp, i64, vp, vp, i64, vp, vp, i32, vp, i32, i32, vp, i64, i32, vp]),
    "b2p_encoder_embed": (i32, [vp, i32, vp, vp, i32, vp, i32, i32, vp, vp]),
    "b2p_decoder_embed": (i32, [vp, vp, i32, vp, vp, i32, i32, vp, vp]),
    "b2p_projector_prep": (i32, [vp, vp, i32, i32, i32, vp, i32, vp]),
    "b2p_greedy_pick": (i32, [vp, i64, i32, i32, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, vp]),
    "b2p_step_advance": (i32, [vp, vp]),
}


class B2PError(RuntimeError):
    pass


def build(force: bool = False) -> Path:
    """Compile every CUDA source for sm_100a into ``libb200parse.so`` (nvcc cross-compiles without a GPU)."""
    srcs = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [CSRC / "Makefile"]
    if not force and LIB_PATH.is_file() and all(LIB_PATH.stat().st_mtime >= s.stat().st_mtime for s in srcs):
        return LIB_PATH
    r = subprocess.run(["make", "-C", str(CSRC), "-j", str(os.cpu_count() or 4)], capture_output=True, text=True)
    if r.returncode != 0:
        raise B2PError("building libb200parse.so failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not LIB_PATH.is_file():
            raise B2PError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(the product path has no CPU fallback)")
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(l, name)   # raises AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise B2PError(lib().b2p_last_error().decode("utf-8", "replace"))


def launch_count() -> int:
    return int(lib().b2p_launch_count())

"""ctypes binding of libvgen_b200.so (the C ABI declared in include/vgen_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, a
`VgenError` is raised.  PyTorch is used by callers only for device memory and streams.
"""
from __future__ import annotations

import ctypes
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("VGEN_B200_LIB", _PKG / "libvgen_b200.so"))


class VgenError(RuntimeError):
    pass


class Epilogue(ctypes.Structure):
    """struct vgen_epilogue (include/vgen_b200.h)."""
    _fields_ = [
        ("alpha", ctypes.c_float),
        ("bias", ctypes.c_void_p),
        ("group_bias", ctypes.c_void_p),
        ("group_bias_ld", ctypes.c_int64),
        ("group_bias_div", ctypes.c_int64),
        ("residual", ctypes.c_void_p),
        ("residual_ld", ctypes.c_int64),
        ("geglu", ctypes.c_int),
        ("bn", ctypes.c_int),
        ("row_stats", ctypes.c_void_p),
        ("col_sum", ctypes.c_void_p),
    ]


_lib = None

_vp, _i64, _i32, _f32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_float
_EP = ctypes.POINTER(Epilogue)

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/vgen_b200.h 1:1.
_SIGNATURES = {
    "vgen_abi_version": [],
    "vgen_last_error": [],
    "vgen_launch_count": [],
    "vgen_set_tapgemm_impl": [_i32],
    "vgen_linear": [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _EP, _vp],
    "vgen_conv2d_3x3": [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _EP, _vp],
    "vgen_tconv3": [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _EP, _vp],
    "vgen_tconv3_batch": [_vp, _i64, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _EP, _vp],
    "vgen_group_norm_workspace_bytes": [_i64],
    "vgen_group_norm": [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _f32, _i32, _vp, _vp],
    "vgen_layer_norm": [_vp, _vp, _i64, _i64, _i64, _i64, _vp, _vp, _f32, _vp],
    "vgen_row_stats": [_vp, _i64, _i64, _i64, _f32, _vp, _vp],
    "vgen_attention_d64": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _f32, _vp],
    "vgen_attention_d512": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _f32, _vp],
    "vgen_attention_d64_debug": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _f32, _vp, _vp],
    "vgen_attention_temporal": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _f32, _vp],
    "vgen_softmax_rows": [_vp, _i64, _i64, _i64, _f32, _vp],
    "vgen_attention_cross_small": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i32, _f32, _vp],
    "vgen_embed_tokens": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp],
    "vgen_add_rows_f32": [_vp, _vp, _i64, _i64, _vp],
    "vgen_interp_linear_rows": [_vp, _vp, _i64, _i64, _i64, _i64, _vp],
    "vgen_fourier_lowfreq_filter": [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _i64, _f32, _vp],
    "vgen_upsample_nearest2x_rows": [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _vp],
    "vgen_scale_copy2d": [_vp, _i64, _vp, _i64, _i64, _i64, _f32, _vp],
    "vgen_cp_to_pc": [_vp, _i32, _vp, _i64, _i64, _i64, _i64, _vp],
    "vgen_pc_to_cp": [_vp, _i64, _vp, _i32, _i64, _i64, _i64, _vp],
    "vgen_im2col": [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i32, _vp],
    "vgen_upsample_nearest2x": [_vp, _vp, _i64, _i64, _i64, _i64, _vp],
    "vgen_copy2d": [_vp, _i64, _vp, _i64, _i64, _i64, _vp],
    "vgen_eltwise": [_i32, _vp, _vp, _vp, _i64, _f32, _vp],
    "vgen_linear_small": [_vp, _i64, _i64, _i64, _vp, _vp, _i64, _vp, _i64, _vp, _i64, _i32, _i32, _vp],
    "vgen_sinusoidal_embedding": [_vp, _vp, _i64, _i64, _vp],
    "vgen_adaptive_avgpool": [_vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i32, _vp],
    "vgen_cond_stem": [_vp, _i32, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _i64, _i64, _i64, _vp, _vp],
    "vgen_cond_sum": [ctypes.POINTER(ctypes.c_void_p), _i32, _i64, _i64, _i64, _vp, _i64, _vp],
    "vgen_vae_sample": [_vp, _vp, _vp, _i64, _i64, _i64, _f32, _vp],
    "vgen_ddim_step": [_vp, _vp, _vp, _vp, _i64, _f32, _vp, _i32, _vp, _vp],
    "vgen_cfg_combine": [_vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp],
    "vgen_gauss_x0": [_vp, _vp, _vp, _f32, _f32, _f32, _i32, _vp, _i64, _i64, _vp],
    "vgen_video_to_rgb8": [_vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp],
    "vgen_lincomb_f32": [_vp, _i64, _vp, _f32, _vp, _f32, _vp, _f32, _vp, _f32, _vp],
}
_RESTYPES = {"vgen_last_error": ctypes.c_char_p, "vgen_launch_count": ctypes.c_int64,
             "vgen_group_norm_workspace_bytes": ctypes.c_int64}


def declared_symbols():
    return sorted(_SIGNATURES)


def load():
    """Load the shared library once; raise VgenError if it is absent (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise VgenError(
            f"{LIB_PATH} not found: build it with `python -m vgen_b200.build` "
            "(vgen_b200 has no CPU or PyTorch fallback path)")
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, ctypes.c_int)
    if lib.vgen_abi_version() != 2:
        raise VgenError(f"ABI version mismatch: library {lib.vgen_abi_version()} != binding 2")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().vgen_last_error()
        raise VgenError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")


def launch_count() -> int:
    return int(load().vgen_launch_count())

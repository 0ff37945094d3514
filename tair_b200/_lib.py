"""ctypes binding of the C ABI declared in ``include/tair_b200.h``.

The library is the product: there is no Python/torch fallback.  Importing this
module never touches the GPU; ``lib()`` loads ``libtair_b200.so`` (built in-tree
by ``tair_b200.build``) and raises ``TairLibraryError`` if it is missing.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtair_b200.so")


class TairLibraryError(RuntimeError):
    pass


class TairError(RuntimeError):
    """A C-ABI call returned a negative status."""


class Epilogue(C.Structure):
    """Mirror of ``tair_epilogue`` (include/tair_b200.h)."""

    _fields_ = [
        ("out", C.c_void_p),
        ("ldc", C.c_int64),
        ("out_fp32", C.c_int32),
        ("act", C.c_int32),
        ("bias", C.c_void_p),
        ("residual", C.c_void_p),
        ("ldr", C.c_int64),
        ("rowgroup", C.c_void_p),
        ("ldg", C.c_int64),
        ("rows_per_group", C.c_int32),
        ("rowgroup_bf16", C.c_int32),
        ("workspace", C.c_void_p),
        ("workspace_bytes", C.c_int64),
        ("ln_row_stats", C.c_void_p),
        ("ln_col_sum", C.c_void_p),
    ]


ACT_NONE, ACT_GEGLU, ACT_GELU, ACT_SILU, ACT_RELU = 0, 1, 2, 3, 4

_i32, _i64, _f32, _vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p

# name -> (restype, argtypes); must list every symbol of include/tair_b200.h
SIGNATURES = {
    "tair_last_error": (C.c_char_p, []),
    "tair_abi_version": (C.c_int, []),
    "tair_launch_count": (C.c_int64, []),
    "tair_launch_count_reset": (None, []),
    "tair_gemm_bf16": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _i32, C.POINTER(Epilogue), _vp]),
    "tair_conv3x3_bf16": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, C.POINTER(Epilogue), _vp]),
    "tair_attention_bf16": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _f32, _i32, _vp]),
    "tair_groupnorm_workspace_bytes": (C.c_int64, [_i32, _i32]),
    "tair_groupnorm_nhwc": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _f32, _i32, _vp, _vp]),
    "tair_row_stats": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _f32, _vp]),
    "tair_layernorm": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _f32, _vp]),
    "tair_sampler_update": (C.c_int, [_vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    "tair_sampler_multistep_update": (C.c_int, [_vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    "tair_sampler_unipc_update": (C.c_int, [_vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "tair_timestep_embedding": (C.c_int, [_vp, _vp, _i32, _i32, _f32, _vp]),
    "tair_nchw_to_nhwc_bf16": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "tair_nhwc_to_nchw_f32": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _i32, _vp]),
    "tair_concat_add": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp]),
    "tair_add_bf16": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "tair_upsample2x_nhwc": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "tair_msda_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "tair_attention_windows_bf16": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _i64, _i32, _i32, _i64, _vp, _i32, _f32, _vp]),
    "tair_layernorm_ragged": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _f32, _vp]),
    "tair_gather_rows_bf16": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _i64, _i32, _vp]),
    "tair_leaky_relu_bf16": (C.c_int, [_vp, _vp, _i64, _f32, _vp]),
    "tair_tiles_bicubic_u8": (C.c_int, [_vp, _i32, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp]),
    "tair_blend_tiles": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "tair_msda_fused": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _i32, _i64, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "tair_attention_seq_bf16": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _i64, _i32, _i32, _i64, _i32, _i64, _i64, _i64, _f32, _vp]),
    "tair_attention_seq32_bf16": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _i64, _i32, _i32, _i64, _i32, _i64, _i64, _i64, _f32, _vp]),
    "tair_testr_postprocess": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _f32, _f32, _vp]),
    "tair_softmax_rows_bf16": (C.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _f32, _vp]),
    "tair_transpose_bf16": (C.c_int, [_vp, _i64, _i64, _vp, _i64, _i64, _i32, _i32, _i32, _vp]),
}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        # the stamp of the prebuilt library must match the sources on disk; a stale or missing library is rebuilt
        # in-tree (nvcc cross-compiles sm_100a) — and if that is impossible the call fails: there is no fallback
        try:
            from . import build as _build
            _build.ensure()
        except Exception as e:
            raise TairLibraryError(
                f"{LIB_PATH} is missing or stale and could not be rebuilt ({e}); build it with "
                "`python -m tair_b200.build` (tair_b200 has no CPU / PyTorch fallback)") from e
        try:
            handle = C.CDLL(LIB_PATH)
        except OSError as e:  # pragma: no cover
            raise TairLibraryError(f"cannot load {LIB_PATH}: {e}") from e
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(handle, name)
            except AttributeError as e:
                raise TairLibraryError(f"{LIB_PATH} does not export {name}") from e
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().tair_last_error().decode("utf-8", "replace")
        raise TairError(f"{what} failed (code {rc}): {msg}")

"""ctypes binding of libgramhead.so (C ABI: include/gramhead.h). There is no fallback: if the library is missing or a
call fails, this raises."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_int, c_longlong, c_void_p, POINTER, c_uint

from .build import LIB_PATH

_LIB = None

GH_DTYPE_F32 = 0
GH_DTYPE_BF16 = 1
GH_ERR_BAD_ARG = -1
GH_ERR_UNSUPPORTED = -2

_P = c_void_p
_SIGNATURES = {
    "gh_version": (c_int, []),
    "gh_sm_count": (c_int, []),
    "gh_set_option": (c_int, [ctypes.c_char_p, c_int]),
    "gh_last_device_error": (c_int, [POINTER(c_uint)]),
    "gh_gram_pool_fwd": (c_int, [_P, c_int, c_longlong, c_longlong, c_longlong, c_int, c_int, c_int, c_int, _P, c_int,
                                  c_int, c_int, c_int, _P]),
    "gh_gram_dense_fwd": (c_int, [_P, c_int, c_longlong, c_longlong, c_longlong, c_int, c_int, c_int, _P, c_int, c_int,
                                   _P]),
    "gh_adaptive_pool_fwd": (c_int, [_P, c_int, c_int, c_int, _P, c_int, c_int, _P]),
    "gh_adaptive_pool_bwd": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "gh_gram_pool_bwd": (c_int, [_P, c_int, c_longlong, c_longlong, c_longlong, c_int, c_int, c_int, c_int, _P, c_int,
                                  c_int, _P, c_int, c_longlong, c_longlong, c_longlong, c_int, _P]),
    "gh_gram_dense_bwd": (c_int, [_P, c_int, c_longlong, c_longlong, c_longlong, c_int, c_int, c_int, _P, _P, c_int,
                                   c_longlong, c_longlong, c_longlong, c_int, _P]),
    "gh_attn_head_fwd": (c_int, [_P] * 7 + [c_int] * 4 + [_P] * 5 + [_P]),
    "gh_transpose_cast": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, c_longlong, _P]),
    "gh_preprocess_frame": (c_int, [_P, c_longlong, c_int, c_int, c_int, _P, _P, _P, c_int, _P, _P, _P, c_int, _P, _P, _P,
                                     c_int, c_int, _P]),
    "gh_preprocess_frames": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, _P, c_int, c_int, _P, _P]),
    "gh_preprocess_frames_smem": (c_int, [c_int, c_int]),
    "gh_frame_tables": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "gh_frame_tables_stride": (c_longlong, [c_int, c_int, c_int, c_int]),
    "gh_normalize_u8": (c_int, [_P, _P, c_longlong, c_int, c_longlong, _P, _P, _P]),
    "gh_gemm_f32": (c_int, [_P, c_longlong, c_longlong, _P, c_longlong, c_longlong, _P, _P, c_longlong, c_int, c_int,
                             c_int, _P]),
    "gh_maxpool2d_nhwc": (c_int, [_P, c_int, _P] + [c_int] * 7 + [_P]),
    "gh_stem_space_to_depth": (c_int, [_P] + [c_longlong] * 4 + [c_int] * 3 + [_P, c_int, _P]),
    "gh_stem_conv_pool_nhwc": (c_int, [_P] + [c_longlong] * 4 + [c_int] * 3 + [_P] * 4),
    "gh_stem_conv_pool_u8_nhwc": (c_int, [_P] + [c_longlong] * 4 + [c_int] * 3 + [_P] * 6),
    "gh_patch_gram_workspace": (c_longlong, [c_int, c_int, c_int]),
    "gh_patch_gram_fwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "gh_patch_attn_fwd": (c_int, [_P] * 11 + [c_int] * 5 + [_P, _P, _P]),
    "gh_gemm_f32_fixed": (c_int, [_P, c_longlong, c_longlong, _P, c_longlong, c_longlong, _P, _P, c_longlong, c_int,
                                   c_int, c_int, _P]),
    "gh_colsum_f32": (c_int, [_P, c_longlong, c_int, c_int, _P, _P]),
    "gh_patch_bwd_workspace": (c_longlong, [c_int, c_int, c_int]),
    "gh_patch_gram_bwd": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P]),
    "gh_patch_pool_bwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "gh_patch_attn_bwd": (c_int, [_P] * 12 + [c_int] * 5 + [_P] * 5 + [_P]),
    "gh_attn_head_bwd_workspace": (c_longlong, [c_int, c_int, c_int]),
    "gh_attn_head_bwd": (c_int, [_P] * 10 + [c_int] * 4 + [_P] * 8 + [_P]),
    "gh_gram_mse_blocks": (c_int, [c_longlong]),
    "gh_gram_mse": (c_int, [_P, _P, c_longlong, _P, _P, _P]),
    "gh_gram_mse_images_blocks": (c_int, [c_longlong]),
    "gh_gram_mse_images": (c_int, [_P, _P, c_int, c_longlong, _P, _P, _P]),
    "gh_split_bf16": (c_int, [_P, _P, c_longlong, c_longlong, _P]),
    "gh_gemm_planes": (c_int, [_P, c_longlong, c_longlong, c_int, _P, c_longlong, c_longlong, c_int, _P, _P, _P,
                                c_longlong, c_longlong, c_int, c_int, c_int, c_int, _P]),
    "gh_tgemm_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "gh_gram_bwd_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, POINTER(c_int)]),
    "gh_attn_head_fwd2": (c_int, [_P] * 7 + [c_int] * 4 + [_P] * 6 + [_P]),
    "gh_attn_head_bwd2_workspace": (c_longlong, [c_int, c_int, c_int]),
    "gh_attn_head_bwd2": (c_int, [_P] * 10 + [c_int] * 4 + [_P] * 8 + [_P]),
    "gh_jpeg_table_ints": (c_int, []),
    "gh_jpeg_records_bytes": (c_longlong, [c_longlong, c_int, c_int]),
    "gh_jpeg_check": (c_int, [c_longlong, c_int, c_int, c_longlong, c_longlong, c_int, c_int]),
    "gh_jpeg_decode": (c_int, [_P, c_longlong, _P, c_int, _P, c_int, _P, c_longlong, c_longlong, c_int, _P, _P, _P, _P,
                               _P, c_int, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class GramHeadError(RuntimeError):
    pass


def library_path() -> str:
    return os.environ.get("GRAMHEAD_LIB", LIB_PATH)


def lib() -> ctypes.CDLL:
    """Loads the library once. Raises GramHeadError when it has not been built (python -m ...build)."""
    global _LIB
    if _LIB is None:
        path = library_path()
        if not os.path.isfile(path):
            raise GramHeadError(
                f"gramhead: {path} not found. Build it with `python -m heuristique_style_transfer_code_b200.build` "
                "(needs nvcc, targets sm_100a). There is no CPU or PyTorch fallback for the Gram + attention head.")
        handle = ctypes.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = handle
        _apply_env_options(handle)
    return _LIB


def _apply_env_options(handle) -> None:
    """GRAMHEAD_OPTIONS="name=value,name=value": tuning knobs of gh_set_option (include/gramhead.h) for processes whose
    code cannot be touched (the reference's unmodified scripts, profiler drivers). An unknown name or a rejected value
    raises: a silently ignored knob would make a measurement lie."""
    spec = os.environ.get("GRAMHEAD_OPTIONS", "").strip()
    if not spec:
        return
    for item in spec.split(","):
        name, sep, value = item.strip().partition("=")
        if not sep or not name:
            raise GramHeadError(f"gramhead: GRAMHEAD_OPTIONS: expected name=value, got {item!r}")
        try:
            ivalue = int(value)
        except ValueError:
            raise GramHeadError(f"gramhead: GRAMHEAD_OPTIONS: {name}: {value!r} is not an integer") from None
        if handle.gh_set_option(name.encode(), ivalue) != 0:
            raise GramHeadError(f"gramhead: GRAMHEAD_OPTIONS: gh_set_option({name!r}, {ivalue}) was rejected")


def check(code: int, what: str) -> None:
    if code == 0:
        return
    if code == GH_ERR_BAD_ARG:
        raise GramHeadError(f"gramhead: {what}: bad argument")
    if code == GH_ERR_UNSUPPORTED:
        raise GramHeadError(f"gramhead: {what}: shape not supported by this entry point")
    raise GramHeadError(f"gramhead: {what}: CUDA error {code}")


def last_device_error():
    out = (c_uint * 4)()
    rc = lib().gh_last_device_error(out)
    return rc, tuple(out)

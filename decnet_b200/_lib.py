"""ctypes binding of libdecnet_b200.so (the C ABI declared in include/decnet_b200.h).

There is NO fallback: if the shared library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("DECNET_B200_LIB", _PKG / "libdecnet_b200.so"))

ABI_VERSION = 2
_ptr = C.c_void_p          # a device or host pointer of any element type (fp32, bf16, uint8, uint16, int64, ...)
_i = C.c_int

# name -> (restype, argtypes); mirrors include/decnet_b200.h one to one.
SIGNATURES = {
    "decnet_abi_version": (_i, []),
    "decnet_last_error": (C.c_char_p, []),
    "decnet_device_info": (_i, [C.POINTER(_i)] * 3),
    "decnet_launch_count": (C.c_int64, []),
    "decnet_reset_launch_count": (None, []),
    "decnet_spamat_fwd": (_i, [_ptr] * 7 + [_i] * 5 + [C.c_void_p]),
    "decnet_spavar_fwd": (_i, [_ptr] * 8 + [_i] * 5 + [C.c_void_p]),
    "decnet_spamat_spavar_fwd": (_i, [_ptr] * 8 + [_i] * 5 + [C.c_void_p]),
    "decnet_spamat_spavar_fwd_levels": (_i, [_i] + [C.c_void_p] * 13 + [C.c_void_p]),
    "decnet_spamat_bwd": (_i, [_ptr] * 10 + [_i] * 5 + [C.c_void_p]),
    "decnet_spavar_bwd": (_i, [_ptr] * 12 + [_i] * 5 + [C.c_void_p]),
    "decnet_candidate_signature": (_i, [_ptr] * 4 + [_i] * 4 + [C.c_void_p]),
    "decnet_costvol_fwd": (_i, [_ptr] * 3 + [_i] * 5 + [C.c_void_p]),
    "decnet_costvol_bf16_ndhwc": (_i, [_ptr] * 3 + [_i] * 6 + [C.c_void_p]),
    "decnet_conv3d_bf16": (_i, [_ptr] * 5 + [_i] * 8 + [C.c_void_p]),
    "decnet_conv3d_bf16_band": (_i, [_ptr] * 5 + [_i] * 7 + [C.c_void_p]),
    "decnet_conv3d_bf16_softargmin": (_i, [_ptr] * 5 + [_i] * 7 + [C.c_void_p]),
    "decnet_costvol_bf16_ndhwc_rows": (_i, [_ptr] * 3 + [_i] * 8 + [C.c_void_p]),
    "decnet_refine_pack_rows": (_i, [_ptr] * 4 + [_i] * 6 + [C.c_void_p]),
    "decnet_conv2d_tf32_nhwc": (_i, [_ptr] * 4 + [_i] * 7 + [C.c_void_p]),
    "decnet_conv2d_tf32_supported": (_i, [_i] * 5),
    "decnet_conv2d_tf32_packed_floats": (_i, [_i] * 2),
    "decnet_conv2d_tf32_nchw": (_i, [_ptr] * 4 + [_i] * 7 + [C.c_void_p]),
    "decnet_conv2d_tf32_nchw_cat": (_i, [C.c_void_p, C.c_void_p, _i] + [_ptr] * 3 + [_i] * 7 + [C.c_void_p]),
    "decnet_conv2d_tc_supported": (_i, [_i] * 6),
    "decnet_conv2d_tc_packed_floats": (_i, [_i] * 3),
    "decnet_conv2d_tc_nchw_cat": (_i, [C.c_void_p, C.c_void_p, _i] + [_ptr] * 3 + [_i] * 8 + [C.c_void_p]),
    "decnet_conv2d_tc_nchw_cat_add": (_i, [C.c_void_p, C.c_void_p, _i] + [_ptr] * 4 + [_i] * 8 + [C.c_void_p]),
    "decnet_conv2d_tc_nhwc_halo": (_i, [_ptr] * 4 + [_i] * 8 + [C.c_void_p]),
    "decnet_conv2d_nhwc_set_variant": (None, [_i]),
    "decnet_conv2d_tc_nhwc_halo_ldc": (_i, [_ptr] * 4 + [_i] * 8 + [C.c_void_p]),
    "decnet_gemm_tc_nhwc": (_i, [_ptr] * 4 + [C.c_longlong] + [_i] * 10 + [C.c_void_p]),
    "decnet_im2col3x3": (_i, [_ptr] * 2 + [_i] * 4 + [C.c_longlong] * 4 + [_i] * 5 + [C.c_void_p]),
    "decnet_deconv3x3s3_shuffle": (_i, [_ptr] * 2 + [_i] * 7 + [C.c_void_p]),
    "decnet_nhwc_to_nchw": (_i, [_ptr] * 2 + [_i] * 6 + [C.c_void_p]),
    "decnet_conv3x3s3_nchw": (_i, [_ptr] * 4 + [_i] * 6 + [C.c_void_p]),
    "decnet_conv2d_tf32_rows_supported": (_i, [_i] * 5),
    "decnet_conv2d_tf32_rows_nchw_cat": (_i, [C.c_void_p, C.c_void_p, _i] + [_ptr] * 3 + [_i] * 6 + [C.c_void_p]),
    "decnet_conv2d_tf32_nhwc_halo": (_i, [_ptr] * 4 + [_i] * 7 + [C.c_void_p]),
    "decnet_nchw_cat_to_nhwc_pad": (_i, [C.c_void_p, C.c_void_p, _i, _ptr] + [_i] * 5 + [C.c_void_p]),
    "decnet_nhwc_pad_to_nchw": (_i, [_ptr] * 2 + [_i] * 5 + [C.c_void_p]),
    "decnet_conv3d_debug_timing": (None, [C.c_void_p]),
    "decnet_conv2d_nhwc_debug_trace": (None, [C.c_void_p]),
    "decnet_conv2d_tf32_debug": (None, [_i, C.c_void_p]),
    "decnet_conv3d_set_variant": (None, [_i]),
    "decnet_softargmin": (_i, [_ptr] * 2 + [_i] * 4 + [C.c_void_p]),
    "decnet_mask_threshold": (_i, [_ptr] * 2 + [C.c_float] + [_ptr] * 4 + [_i] * 3 + [C.c_void_p]),
    "decnet_dynup_pack": (_i, [_ptr] * 3 + [_i] * 4 + [C.c_void_p]),
    "decnet_dynup_glue": (_i, [_ptr] * 3 + [_i] * 3 + [C.c_void_p]),
    "decnet_dynup_pack_nhwc": (_i, [_ptr] * 3 + [_i] * 7 + [C.c_void_p]),
    "decnet_dynup_set_disp_nhwc": (_i, [_ptr] * 2 + [_i] * 6 + [C.c_void_p]),
    "decnet_dynup_glue_nhwc": (_i, [_ptr] * 3 + [_i] * 5 + [C.c_void_p]),
    "decnet_bicubic_up3": (_i, [_ptr] * 2 + [_i] * 5 + [C.c_void_p]),
    "decnet_sqdiff_pair": (_i, [_ptr] * 6 + [C.c_longlong, C.c_void_p]),
    "decnet_detail_head": (_i, [_ptr] * 3 + [C.c_float, C.c_float] + [_ptr] * 2 + [_i] * 3 + [C.c_void_p]),
    "decnet_detail_level_scratch_floats": (C.c_longlong, [_i] * 3),
    "decnet_detail_level": (_i, [_ptr] * 4 + [C.c_float] + [_i] * 3 + [C.c_void_p]),
    "decnet_image_prepare_u8": (_i, [_ptr] * 5 + [_i] * 5 + [C.c_void_p]),
    "decnet_image_prepare_u8_shift": (_i, [_ptr] * 5 + [_i] * 6 + [C.c_void_p]),
    "decnet_disp_to_u16": (_i, [_ptr] * 2 + [_i] * 5 + [C.c_void_p]),
    "decnet_disp_add": (_i, [_ptr, C.c_float, C.c_longlong, C.c_void_p]),
    "decnet_epe_3px": (_i, [_ptr] * 2 + [C.c_float, _ptr, C.c_longlong, C.c_void_p]),
    "decnet_mirror_swap_u8": (_i, [_ptr] * 4 + [_i] * 3 + [C.c_void_p]),
    "decnet_lr_check": (_i, [_ptr] + [_i] * 5 + [C.c_float] + [_ptr] * 3 + [C.c_void_p]),
    "decnet_lr_check_fill": (_i, [_ptr] + [_i] * 5 + [C.c_float] + [_ptr] * 4 + [C.c_void_p]),
    "decnet_lr_guided_fill_scratch_floats": (C.c_longlong, [_i] * 3),
    "decnet_lr_check_guided_fill": (_i, [_ptr] * 2 + [_i] * 5 + [C.c_float] + [C.c_double] * 2 + [_ptr] * 5 + [C.c_void_p]),
    "decnet_lr_speckle_scratch_bytes": (C.c_longlong, [_i] * 4),
    "decnet_lr_check_speckle": (_i, [_ptr] * 2 + [_i] * 5 + [C.c_float, _i, C.c_float, _i] + [C.c_double] * 2 + [_ptr] * 5
                                + [C.c_void_p]),
    "decnet_attn_pack": (_i, [_ptr] * 6 + [_i] * 4 + [C.c_void_p]),
    "decnet_blend": (_i, [_ptr] * 5 + [_i] * 3 + [C.c_void_p]),
    "decnet_warp_bilinear": (_i, [_ptr] * 3 + [_i] * 4 + [C.c_void_p]),
    "decnet_refine_pack": (_i, [_ptr] * 4 + [_i] * 4 + [C.c_void_p]),
    "decnet_haar_level": (_i, [_ptr] * 6 + [_i] * 3 + [C.c_void_p]),
    "decnet_conv2d_small_supported": (_i, [_i] * 3),
    "decnet_conv2d_set_variant": (None, [_i]),
    "decnet_conv2d_small": (_i, [_ptr] * 5 + [_i] * 8 + [C.c_void_p]),
    "decnet_deconv3x3s3": (_i, [_ptr] * 4 + [_i] * 6 + [C.c_void_p]),
    "decnet_last_sparse_path": (_i, []),
    "decnet_set_sparse_path": (None, [_i]),
    "decnet_last_sparse_variant": (_i, []),
    "decnet_set_sparse_variant": (None, [_i]),
}


class DecnetError(RuntimeError):
    pass


_lib = None


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raise loudly if it is absent."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise DecnetError(
                f"{LIB_PATH} not found: build it with `python -m decnet_b200.build` "
                "(there is no CPU or PyTorch fallback for these ops)")
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError here == header/library mismatch
            fn.restype = res
            fn.argtypes = args
        if handle.decnet_abi_version() != ABI_VERSION:
            raise DecnetError("libdecnet_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().decnet_last_error().decode("utf-8", "replace")
        raise DecnetError(f"{what} failed with status {status}: {msg}")

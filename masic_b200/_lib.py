"""ctypes binding of libmasic_b200.so (the C ABI declared in include/masic_b200.h).

There is deliberately no fallback: if the shared object is missing or a call returns a
non-zero status the caller gets an exception.  Nothing in this module computes on the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libmasic_b200.so"

ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
GDN_NONE, GDN_FWD, GDN_INV = 0, 1, 2
IMG_XOFF, IMG_XPAD = 2, 8       # MASIC_IMG_XOFF / MASIC_IMG_XPAD
CONV, DECONV_S2, DECONV_S2_SUBPIX, CONV_XFOLD4, CONV_XFOLD8 = 0, 1, 2, 3, 4
# 16-bit activation / operand formats (MASIC_FMT_*, csrc/cvt16.cuh): the training step runs in bf16 (gradients need
# fp32's exponent range), the inference engines in fp16 (8x finer rounding at the same tensor-core rate)
FMT_BF16, FMT_F16 = 0, 1
FMT_SPLIT = 2      # or-ed in by image producers: pixels of <= 4 channels as [hi | lo] (see include/masic_b200.h)


def act_dtype(f16):
    import torch
    return torch.float16 if (f16 & 1) else torch.bfloat16

_ERRORS = {-1: "MASIC_EINVAL (bad argument)", -2: "MASIC_ENOSUP (not implemented)",
           -3: "MASIC_EDRIVER (cuTensorMapEncodeTiled unavailable or failed)"}


class MasicError(RuntimeError):
    pass


class ConvDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int), ("ksize", C.c_int), ("stride", C.c_int), ("tap_mask", C.c_uint32),
        ("n", C.c_int), ("h_in", C.c_int), ("w_in", C.c_int),
        ("c_in", C.c_int), ("c_out", C.c_int), ("c_out_pad", C.c_int), ("n_tile", C.c_int),
        ("in_", C.c_void_p), ("in_cpitch", C.c_int), ("in_coff", C.c_int),
        ("w_packed", C.c_void_p),
        ("bias", C.c_void_p),
        ("out", C.c_void_p), ("out_cpitch", C.c_int), ("out_coff", C.c_int), ("out_fp32", C.c_int),
        ("act", C.c_uint8 * 32),
        ("gdn", C.c_int), ("gamma_packed", C.c_void_p), ("beta", C.c_void_p),
        ("rowscale", C.c_void_p), ("rs_stride", C.c_int), ("rs_off", C.c_int),
        ("residual0", C.c_void_p), ("res0_cpitch", C.c_int), ("res0_coff", C.c_int),
        ("residual1", C.c_void_p), ("res1_cpitch", C.c_int), ("res1_coff", C.c_int),
        ("nt_in_coff", C.POINTER(C.c_int)), ("nt_out_coff", C.POINTER(C.c_int)), ("nt_out_img", C.POINTER(C.c_int)),
        ("out_images", C.c_int), ("cta_pairs", C.c_int), ("f16", C.c_int), ("pdl", C.c_int),
        ("in_row_pixels", C.c_int), ("out_blk_images", C.c_int),
    ]


class PackJob(C.Structure):
    _fields_ = [
        ("w", C.c_void_p), ("dst", C.c_void_p), ("bias_src", C.c_void_p), ("bias_dst", C.c_void_p),
        ("kind", C.c_int), ("transposed", C.c_int), ("ksize", C.c_int), ("c_in", C.c_int), ("c_out", C.c_int),
        ("c_out_pad", C.c_int),
    ]


class WgradDesc(C.Structure):
    _fields_ = [
        ("ksize", C.c_int), ("stride", C.c_int), ("tap_mask", C.c_uint32),
        ("n", C.c_int), ("h_lo", C.c_int), ("w_lo", C.c_int),
        ("lo", C.c_void_p), ("lo_cpitch", C.c_int), ("lo_coff", C.c_int), ("c_lo", C.c_int),
        ("hi", C.c_void_p), ("hi_cpitch", C.c_int), ("hi_coff", C.c_int), ("c_hi", C.c_int),
        ("dw", C.c_void_p), ("accumulate", C.c_int),
    ]


_lib = None


def load() -> C.CDLL:
    """Load the shared object, failing loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("MASIC_B200_LIB", LIB_PATH))
    if not path.exists():
        raise MasicError(
            f"{path} not found: build it with `python -m masic_b200.build` (nvcc, sm_100a). "
            "masic_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(str(path))
    _declare(lib)
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status == 0:
        return
    if status < 0:
        raise MasicError(f"{what}: {_ERRORS.get(status, status)}")
    raise MasicError(f"{what}: CUDA error {status}")


def _declare(lib: C.CDLL) -> None:
    vp, i, u32, f = C.c_void_p, C.c_int, C.c_uint32, C.c_float
    i64 = C.c_int64
    sig = {
        "masic_abi_version": (i, []),
        "masic_build_info": (C.c_char_p, []),
        "masic_conv_plan_create": (i, [C.POINTER(ConvDesc), C.POINTER(vp)]),
        "masic_conv_plan_launch": (i, [vp, vp]),
        "masic_conv_plan_destroy": (None, [vp]),
        "masic_conv_plan_info": (i, [vp, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                     C.POINTER(i), C.POINTER(i)]),
        "masic_conv_plan_trace": (i, [vp, vp]),
        "masic_conv_plan_set_act_out": (i, [vp, vp, i, i]),
        "masic_packed_weight_bytes": (i64, [i, i, i, i]),
        "masic_pack_conv_weights": (i, [vp, i, i, i, i, i, i, vp, i, vp]),
        "masic_pack_batch_create": (i, [C.POINTER(PackJob), i, C.POINTER(vp)]),
        "masic_pack_batch_launch": (i, [vp, vp]),
        "masic_pack_batch_destroy": (None, [vp]),
        "masic_gdn_prepare": (i, [vp, vp, i, f, vp, vp, vp, i, vp]),
        "masic_conv_direct_nhwc": (i, [vp, i, i, i, i, i, i, vp, i, i, i, u32, vp, i, vp, i, i, i, i, vp]),
        "masic_gmm_likelihood_fwd": (i, [vp, vp, vp, vp, i, i, i, i, i, i, f, vp, vp, vp, i, vp, i, i,
                                         vp, i, i, i, vp]),
        "masic_gc_likelihood_fwd": (i, [vp, vp, vp, i64, f, vp, vp, vp, vp]),
        "masic_gc_build_indexes": (i, [vp, i64, vp, i, f, vp, vp]),
        "masic_eb_fwd": (i, [vp, i, i, i, i, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), vp, vp, vp, vp,
                             i, vp, i, i, vp]),
        "masic_quantize": (i, [vp, vp, i64, vp, vp, vp]),
        "masic_latent_prep": (i, [vp, i64, i, vp, i, vp, i, i, vp, i, i, i, vp]),
        "masic_pmf_to_quantized_cdf": (i, [vp, i, i, vp]),
        "masic_pmf_table_to_cdf": (i, [vp, i, i, vp, vp, i, i, vp]),
        "masic_gmm_symbol_cdfs": (i, [vp, vp, vp, i, i, i, i64, vp, i, i, f, vp, vp, vp, vp]),
        "masic_range_encode": (i, [vp, i64, vp, i64, C.POINTER(i64)]),
        "masic_range_decoder_create": (i, [vp, i64, C.POINTER(vp)]),
        "masic_range_decode_rows": (i, [vp, vp, i, i, vp]),
        "masic_range_decoder_destroy": (None, [vp]),
        "masic_range_encode_channels": (i, [vp, i64, i, vp, i64, vp]),
        "masic_range_streams_init": (i, [vp, vp, i, vp, vp]),
        "masic_range_decode_wave": (i, [vp, i, i, i, vp, vp, vp, vp, i, vp, i, i, vp, vp, i, vp, vp]),
        "masic_wave_gather": (i, [vp, i, i, vp, i, i, i, vp, vp, i, vp, vp, vp, vp]),
        "masic_wave_center": (i, [vp, i, i, i, i, vp, vp]),
        "masic_gmm_symbol_cdfs_pairs": (i, [vp, vp, vp, i, i, i, i64, i64, vp, vp, vp, i, i, f, vp, vp, i, vp, vp]),
        "masic_wave_gather_pairs": (i, [vp, i, i, i, vp, i, i, i, vp, vp, i, i, i, vp, vp, vp, vp]),
        "masic_range_decode_wave_pairs": (i, [vp, i, i, i, vp, vp, vp, vp, vp, vp, i, vp, i, i, i, vp, vp, i, vp, vp]),
        "masic_range_encode_streams": (i, [vp, vp, vp, i64, i, vp, i64, vp, vp, vp]),
        "masic_pack_streams": (i, [vp, i64, vp, i, vp, vp, vp]),
        "masic_rans_encoder_create": (i, [C.POINTER(vp)]),
        "masic_rans_encoder_push": (i, [vp, vp, vp, i64, vp, i, i, vp, vp]),
        "masic_rans_encoder_flush": (i, [vp, C.POINTER(vp), C.POINTER(i64)]),
        "masic_rans_encoder_destroy": (None, [vp]),
        "masic_rans_decoder_create": (i, [vp, i64, C.POINTER(vp)]),
        "masic_rans_decoder_decode": (i, [vp, vp, i64, vp, i, i, vp, vp, vp]),
        "masic_rans_decoder_destroy": (None, [vp]),
        "masic_deconv_img_weight_bytes": (i64, []),
        "masic_deconv_img_pack_weights": (i, [vp, vp, i, vp]),
        "masic_deconv_img_plan_create": (i, [vp, i, i, i, i, vp, vp, i, vp, vp, vp, i, C.POINTER(vp)]),
        "masic_deconv_img_plan_launch": (i, [vp, vp]),
        "masic_deconv_img_plan_set_out16": (i, [vp, vp, i, i, i, i, i]),
        "masic_deconv_img_plan_destroy": (None, [vp]),
        "masic_maxpool2_nhwc_bf16": (i, [vp, i, i, i, i, vp, i, vp]),
        "masic_fc_pack_weights": (i, [vp, i, i, i, vp, i, vp]),
        "masic_fc_bf16": (i, [vp, i, vp, vp, i, i, i, i, vp, vp, i, i, vp]),
        "masic_homography_from_delta": (i, [vp, vp, i, i, i, i, i, i, vp, vp]),
        "masic_homography_pad": (i, [vp, i, i, i, vp, vp]),
        "masic_warp_prepare": (i, [vp, i, i, i, i, i, i, vp, vp]),
        "masic_warp_perspective_fwd": (i, [vp, i, i, i, i, i, i, vp, vp, vp, i, i, i, i, vp, i, i, i, i, i, vp, vp]),
        "masic_conv_small_nchw": (i, [vp, i, vp, i, i, i, i, vp, i, vp, i, i, i, i, i, vp, vp, f, vp, vp, i, i, i, i, vp]),
        "masic_mask2weights": (i, [vp, i, i, i, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "masic_subpix_to_nchw": (i, [vp, i, i, i, i, i, vp, vp, f, vp, vp, i, i, vp]),
        "masic_gdn_nchw": (i, [vp, i, i, i, vp, vp, f, i, vp, vp]),
        "masic_softmax_channels": (i, [vp, i, i, i, vp, vp, vp]),
        "masic_nchw_to_nhwc_bf16": (i, [vp, i, i, i, i, vp, i, i, i, i, vp]),
        "masic_u8_to_unit_f32": (i, [vp, i64, vp, vp]),
        "masic_pad_image": (i, [vp, i, i, i, i, i, i, i, i, i, vp, vp, vp]),
        "masic_nhwc_to_nchw_f32": (i, [vp, i, i, i, i, vp, vp]),
        "masic_wgrad_plan_create": (i, [C.POINTER(WgradDesc), C.POINTER(vp)]),
        "masic_wgrad_plan_workspace_bytes": (i64, [vp]),
        "masic_wgrad_plan_launch": (i, [vp, vp, vp]),
        "masic_wgrad_plan_info": (i, [vp, C.POINTER(C.c_double), C.POINTER(i)]),
        "masic_wgrad_plan_destroy": (None, [vp]),
        "masic_wgrad_small": (i, [vp, i, i, vp, i, i, i, i, vp, vp]),
        "masic_gmm_likelihood_train": (i, [vp, vp, vp, vp, vp, i64, i, i, f, f, vp, vp, i, vp, vp, vp, vp, vp, vp]),
        "masic_eb_train": (i, [vp, vp, i, i, i, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), f, vp, vp, vp, i,
                               vp, vp, vp]),
        "masic_eb_aux_loss": (i, [vp, i, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(f), vp, vp, vp]),
        "masic_act_bwd_bias": (i, [vp, i, i, vp, i, i, i, i64, i, vp, vp]),
        "masic_act_bwd_bias_out": (i, [vp, i, i, vp, i, i, i, i64, i, vp, i, i, vp, vp]),
        "masic_gdn_square": (i, [vp, vp, i64, vp]),
        "masic_gdn_apply": (i, [vp, vp, i, vp, i64, vp]),
        "masic_gdn_bwd_a": (i, [vp, vp, vp, i, vp, i64, i, vp, vp]),
        "masic_gdn_bwd_b": (i, [vp, vp, vp, i64, i, vp, vp]),
        "masic_reparam_bwd": (i, [vp, vp, i, f, i, vp, vp]),
        "masic_reparam_batch_create": (i, [vp, vp, vp, vp, vp, vp, i, C.POINTER(vp)]),
        "masic_reparam_batch_launch": (i, [vp, vp]),
        "masic_reparam_batch_destroy": (None, [vp]),
        "masic_latent_prep_train": (i, [vp, vp, i64, i, vp, i, vp, i, vp]),
        "masic_latent_merge_bwd": (i, [vp, vp, vp, vp, vp, i64, vp, vp]),
        "masic_add_f32_bf16": (i, [vp, vp, i64, vp, vp]),
        "masic_mask_fuse_fwd": (i, [vp, vp, i, vp, vp, i, vp, i64, vp, vp]),
        "masic_mask_fuse_bwd": (i, [vp, vp, vp, i, vp, vp, i, vp, i64, vp, vp, vp, vp, vp]),
        "masic_mse_grad": (i, [vp, vp, vp, f, i64, vp, vp]),
        "masic_warp_perspective_bwd": (i, [vp, vp, i, i, i, i, i, i, vp, vp, vp]),
        "masic_conv_small_bwd": (i, [vp, i, vp, i, i, i, i, vp, i, i, i, i, vp, vp, vp, vp, vp, vp, vp]),
        "masic_gdn_small_bwd": (i, [vp, vp, i, i, i, vp, vp, f, i, vp, vp, vp, vp]),
        "masic_softmax_channels_bwd": (i, [vp, vp, i, i, i, vp, vp]),
        "masic_colsum_nchw": (i, [vp, i, i, i64, vp, vp]),
        "masic_cqe_mask_weights": (i, [vp, i, i, i, C.POINTER(vp), C.POINTER(vp), i, vp, vp]),
        "masic_cqe_blend_images": (i, [vp, vp, vp, i, i, i, vp, i, vp]),
        "masic_cqe_feature_fuse": (i, [vp, i, vp, i, i, vp, vp, i, i, i, vp, i, i, vp]),
        "masic_cqe_residual_image": (i, [vp, i, vp, i, i, i, vp, vp]),
        "masic_cqe_feature_fuse_bwd": (i, [vp, i, vp, i, vp, i, i, vp, vp, i, i, i, vp, i, vp, i, vp, vp]),
        "masic_cqe_blend_images_bwd": (i, [vp, i, vp, vp, i, i, i, vp, vp]),
        "masic_rd_metrics_scratch_bytes": (i64, []),
        "masic_rd_metrics": (i, [C.POINTER(vp), C.POINTER(i64), vp, vp, vp, vp, i, i, i, i, f, vp, vp, vp]),
        "masic_ms_ssim_scratch_bytes": (i64, [i, i, i, i, i]),
        "masic_ms_ssim": (i, [vp, vp, i, i, i, i, i, f, f, f, C.POINTER(f), i, vp, vp, vp]),
        "masic_ms_ssim_bwd_work_bytes": (i64, [i, i, i, i, i]),
        "masic_ms_ssim_bwd": (i, [vp, vp, i, i, i, i, i, f, f, f, C.POINTER(f), i, vp, f, vp, vp, vp, vp]),
        "masic_lpips_prep": (i, [vp, i, i, i, i, C.POINTER(f), C.POINTER(f), vp, vp]),
        "masic_maxpool3s2_nhwc": (i, [vp, i, i, i, i, i, i, i, i, vp, vp]),
        "masic_lpips_distance_scratch_bytes": (i64, [i, i, i]),
        "masic_lpips_distance": (i, [C.POINTER(vp), C.POINTER(vp), i, i, i, vp, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)      # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    lib._masic_declared = tuple(sig)


def declared_symbols() -> tuple:
    return load()._masic_declared

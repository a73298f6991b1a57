"""ctypes binding of libiswm_b200.so (the C ABI declared in include/iswm_b200.h).

The library is the product; there is no fallback. Importing this module never fails
(so CPU-only tooling can import the package), but the first call that needs the
library raises if the shared object is missing, and every op raises on a non-zero
return code with the library's own error text.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ISWM_B200_LIB selects an alternative build of the SAME library (e.g. the -DISWM_EPI_TIMING debug build of tools/)
LIB_PATH = os.environ.get("ISWM_B200_LIB") or os.path.join(_HERE, "libiswm_b200.so")

MAX_TAPS = 32
TTA_MAX_VIEWS = 8
U8, I32, I64 = 0, 1, 2
F32, BF16, E4M3 = 0, 1, 2
EPI_AFFINE, EPI_RELU, EPI_RESIDUAL, EPI_STATS, EPI_OUT_F32, EPI_RES_MASK = 1, 2, 4, 8, 16, 32


class ConvDesc(C.Structure):
    """Mirror of iswm_conv_desc."""

    _fields_ = [
        ("B", C.c_int32), ("Hi", C.c_int32), ("Wi", C.c_int32), ("Cin", C.c_int32),
        ("in_ld", C.c_int32), ("n_img", C.c_int32),
        ("Ho", C.c_int32), ("Wo", C.c_int32), ("Cout", C.c_int32),
        ("out_ld", C.c_int32), ("res_ld", C.c_int32), ("ntaps", C.c_int32),
        ("dh", C.c_int8 * MAX_TAPS), ("dw", C.c_int8 * MAX_TAPS), ("phase", C.c_int8 * MAX_TAPS),
        ("coff", C.c_int16 * MAX_TAPS), ("wtap", C.c_int8 * MAX_TAPS),
        ("flags", C.c_int32), ("out_ws", C.c_int32), ("out_hs", C.c_int32), ("out_bs", C.c_int64),
        ("w_ntaps", C.c_int32), ("stats_replicas", C.c_int32), ("in_phase_view", C.c_int32), ("reserved2_", C.c_int32),
    ]


class BnSide(C.Structure):
    """Mirror of iswm_bn_side."""

    _fields_ = [("stats", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p), ("running_mean", C.c_void_p),
                ("running_var", C.c_void_p), ("num_batches_tracked", C.c_void_p), ("save_mean", C.c_void_p), ("save_invstd", C.c_void_p),
                ("stats_replicas", C.c_int32)]


class PackJob(C.Structure):
    """Mirror of iswm_pack_job."""

    _fields_ = [("w", C.c_void_p), ("dst", C.c_void_p), ("Cout", C.c_int32), ("Cin", C.c_int32), ("RS", C.c_int32),
                ("pad", C.c_int32), ("row_ld", C.c_int32), ("mode", C.c_int32), ("blk_begin", C.c_int32), ("blk_count", C.c_int32)]


class SgdPackJob(C.Structure):
    """Mirror of iswm_sgd_pack_job."""

    _fields_ = [("w", C.c_void_p), ("g", C.c_void_p), ("m", C.c_void_p), ("dst_f", C.c_void_p), ("dst_d", C.c_void_p), ("n", C.c_int64),
                ("Cout", C.c_int32), ("Cin", C.c_int32), ("RS", C.c_int32), ("pad_f", C.c_int32), ("row_ld_f", C.c_int32),
                ("pad_d", C.c_int32), ("row_ld_d", C.c_int32), ("mode", C.c_int32), ("TC", C.c_int32),
                ("blk_begin", C.c_int32), ("blk_count", C.c_int32)]


class UnpackJob(C.Structure):
    """Mirror of iswm_unpack_job."""

    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("Cout", C.c_int32), ("Cin", C.c_int32), ("RS", C.c_int32),
                ("chunks", C.c_int32), ("blk_begin", C.c_int32), ("pad_", C.c_int32)]


class TtaView(C.Structure):
    """Mirror of IswmTtaView."""

    _fields_ = [("lo", C.c_void_p), ("Hi", C.c_int32), ("Wi", C.c_int32), ("Hv", C.c_int32), ("Wv", C.c_int32), ("flip", C.c_int32)]


class SyncBnJob(C.Structure):
    """Mirror of iswm_syncbn_job."""

    _fields_ = [("src_off", C.c_int64), ("dst", C.c_void_p), ("n", C.c_int32), ("replicas", C.c_int32)]


def fill_unpack_jobs(jobs):
    """jobs: list of (src_ptr, dst_ptr, Cout, Cin, RS) -> (ctypes array, total_blocks)."""
    arr = (UnpackJob * len(jobs))()
    begin = 0
    for i, (src, dst, Cout, Cin, RS) in enumerate(jobs):
        chunks = (Cin + 511) // 512
        arr[i].src, arr[i].dst, arr[i].Cout, arr[i].Cin, arr[i].RS, arr[i].chunks, arr[i].blk_begin = src, dst, Cout, Cin, RS, chunks, begin
        begin += Cout * chunks
    return arr, begin


def fill_pack_jobs(jobs):
    """jobs: list of (w_ptr, dst_ptr, Cout, Cin, RS, pad, row_ld, mode) -> (ctypes array, total_blocks); thread
    blocks are dealt to jobs in proportion to their element count (one per 16 Ki elements, 1..256)."""
    arr = (PackJob * len(jobs))()
    begin = 0
    for i, j in enumerate(jobs):
        arr[i].w, arr[i].dst, arr[i].Cout, arr[i].Cin, arr[i].RS, arr[i].pad, arr[i].row_ld, arr[i].mode = j
        n = j[2] * j[3] * j[4]
        arr[i].blk_begin = begin
        arr[i].blk_count = max(1, min(256, (n + 16383) // 16384))
        begin += arr[i].blk_count
    return arr, begin


_p, _i, _i64, _f, _u64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64

# name -> (restype, argtypes); kept in the order of include/iswm_b200.h
SIGNATURES = {
    "iswm_last_error": (C.c_char_p, []),
    "iswm_version": (_i, []),
    "iswm_launch_count": (_i64, []),
    "iswm_reset_launch_count": (None, []),
    "iswm_debug_abort_code": (_i, []),
    "iswm_debug_set_skip": (None, [_i]),
    "iswm_class_hist": (_i, [_p, _i, _i64, _i, _p, _p]),
    "iswm_wce_fwd_bwd": (_i, [_p, _i, _p, _i, _p, _p, _i64, _i, _i64, _i, _f, _p, _p, _p, _p]),
    "iswm_confusion": (_i, [_p, _i, _p, _i, _i64, _i, _p, _p]),
    "iswm_argmax_confusion": (_i, [_p, _i, _p, _i, _i64, _i, _i64, _i, _f, _p, _p, _p, _p]),
    "iswm_predict_epilogue": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _f, _p, _i, _p, _p, _p, _p]),
    "iswm_resize_flip_f32": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_predict_tta_epilogue": (_i, [C.POINTER(TtaView), _i, _i, _i, _i, _i, _i, _f, _p, _i, _p, _p, _p, _p]),
    "iswm_window_gather_f32": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_predict_window_epilogue": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _p, _i, _p, _p, _p, _p]),
    "iswm_focal_fwd_bwd": (_i, [_p, _i, _p, _i, _p, _i64, _i, _i64, _i, _f, _f, _i, _p, _p, _p, _p]),
    "iswm_conv_igemm": (_i, [C.POINTER(ConvDesc), _p, _p, _p, _p, _p, _p, _p, _p]),
    "iswm_conv_igemm_ex": (_i, [C.POINTER(ConvDesc), _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "iswm_conv_igemm_f8": (_i, [C.POINTER(ConvDesc), _p, _p, _p, _p, _p, _p, _f, _i, _p]),
    "iswm_aspp_bwd": (_i, [_p, _i, _p, _i, _i, _i, _i, _i, C.POINTER(C.c_int), _p, _i, _i, _p]),
    "iswm_peer_barrier": (_i, [C.POINTER(_p), _i, _i, _p, _p]),
    "iswm_peer_allreduce_f32": (_i, [C.POINTER(_p), _i, _i, _i64, _i64, _i, _p]),
    "iswm_peer_small_publish": (_i, [C.POINTER(_p), _i, _i, _p, _i, _i, _i, _p]),
    "iswm_peer_small_sum": (_i, [C.POINTER(_p), _i, _p, _i, _i, _i, _p]),
    "iswm_syncbn_exchange": (_i, [C.POINTER(SyncBnJob), _i, C.POINTER(_p), C.POINTER(_p), _i, _i, C.c_double, _p, _p]),
    "iswm_conv_wgrad": (_i, [C.POINTER(ConvDesc), _p, _p, _p, _p]),
    "iswm_conv_wgrad_grouped": (_i, [C.POINTER(ConvDesc), C.POINTER(_p), C.POINTER(_p), C.POINTER(_p), _i, _p]),
    "iswm_conv_wgrad_ex": (_i, [C.POINTER(ConvDesc), _p, _p, _p, _i, _p]),
    "iswm_pack_weight_fwd": (_i, [_p, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_pack_weight_dgrad": (_i, [_p, _i, _i, _i, _i, _p, _p]),
    "iswm_pack_weights_batched": (_i, [_p, _i, _i, _p]),
    "iswm_sgd_pack_batched": (_i, [_p, _i, _i, _f, _f, _f, _i, _i, _p, _p]),
    "iswm_unpack_wgrad": (_i, [_p, _i, _i, _i, _i, _i, _f, _p, _p]),
    "iswm_unpack_wgrad_batched": (_i, [_p, _i, _i, _p]),
    "iswm_bn_train_apply": (_i, [_p, _i, _p, _i, _i64, _i, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p, _i, _i, _f, _u64, _p, _p, _i, _p, _p]),
    "iswm_bn_train_apply_global": (_i, [_p, _i, _p, _i64, _i, _p, _p, _f, _f, _p, _p, _p, _p, _p, _p, _i, _i, _f, _u64, _p, _p, _i, _p, _p]),
    "iswm_bn_fold": (_i, [_p, _p, _p, _p, _f, _i, _p, _p, _p]),
    "iswm_bn_bwd_reduce": (_i, [_p, _i, _p, _i, _p, _i, _i64, _i, _p, _p, _p, _p, _i, _f, _u64, _p, _p, _p]),
    "iswm_bn_bwd_apply": (_i, [_p, _i, _p, _i, _p, _i, _i64, _i, _p, _p, _p, _p, _p, _i, _f, _u64, _p, _p, _i, _p, _i, _p, _p, _p]),
    "iswm_bn_bwd_apply_global": (_i, [_p, _i, _p, _i, _p, _i, _i64, _i, _p, _p, _p, _p, _p, _p, _i, _f, _u64, _p, _p, _i, _p, _i, _p, _p, _p]),
    "iswm_bn_dual_train_apply": (_i, [_p, _i, C.POINTER(BnSide), _p, _i, C.POINTER(BnSide), _i64, _i, _f, _f, _p, _i, _p, _p]),
    "iswm_bn_dual_bwd_reduce": (_i, [_p, _i, _p, _p, _i, C.POINTER(BnSide), _p, _i, C.POINTER(BnSide), _i64, _i, _p, _p, _p]),
    "iswm_bn_dual_bwd_apply": (_i, [_p, _i, _p, _p, _i, C.POINTER(BnSide), _p, _p, _i, C.POINTER(BnSide), _p, _i64, _i, _p, _i, _p, _i,
                                    _p, _p, _p, _p, _p]),
    "iswm_bn_dual_train_apply_global": (_i, [_p, _i, C.POINTER(BnSide), _p, _i, C.POINTER(BnSide), _i64, _i, _f, _f, _p, _i, _p, _p]),
    "iswm_bn_dual_bwd_apply_global": (_i, [_p, _i, _p, _p, _i, C.POINTER(BnSide), _p, _p, _p, _i, C.POINTER(BnSide), _p, _p, _i64, _i, _p, _i,
                                           _p, _i, _p, _p, _p, _p, _p]),
    "iswm_stem_pool_fwd": (_i, [_p, C.POINTER(BnSide), _i, _i, _i, _i, _i, _i, _f, _f, _p, _p, _p]),
    "iswm_stem_pool_fwd_global": (_i, [_p, C.POINTER(BnSide), _i, _i, _i, _i, _i, _i, _f, _f, _p, _p, _p]),
    "iswm_stem_rows": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_unpack_wgrad_stem": (_i, [_p, _i, _i, _i, _i, _f, _p, _p]),
    "iswm_stem_im2col": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_maxpool_fwd": (_i, [_p, _i, _i, _i, _i, _i, _i, _p, _p, _p]),
    "iswm_maxpool_bwd": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_gap_fwd": (_i, [_p, _i, _i, _i64, _i, _p, _p]),
    "iswm_broadcast_hw": (_i, [_p, _i, _i64, _i, _p, _i, _p]),
    "iswm_sum_hw": (_i, [_p, _i, _i, _i64, _i, _p, _p]),
    "iswm_gap_bwd_add": (_i, [_p, _i, _i64, _i, _p, _i, _p]),
    "iswm_bilinear_fwd": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p]),
    "iswm_bilinear_bwd": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _p, _i, _p]),
    "iswm_logits_up_fwd": (_i, [_p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_logits_up_bwd": (_i, [_p, _i, _i, _i, _i, _i, _i, _p, _i, _p, _p]),
    "iswm_pack_weight_f8": (_i, [_p, _i, _i, _i, _i, _p, _p, _p]),
    "iswm_maxpool_fwd_f8": (_i, [_p, _i, _i, _i, _i, _i, _i, _f, _p, _p]),
    "iswm_gap_fwd_f8": (_i, [_p, _i, _i, _i64, _i, _f, _p, _p]),
    "iswm_broadcast_hw_f8": (_i, [_p, _i, _i64, _i, _f, _p, _i, _p]),
    "iswm_bilinear_fwd_f8": (_i, [_p, _i, _i, _i, _i, _i, _i, _i, _f, _p, _i, _p]),
    "iswm_phase_split_b8": (_i, [_p, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_subsample2_b8": (_i, [_p, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_phase_split": (_i, [_p, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_subsample2": (_i, [_p, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_zero_stuff2": (_i, [_p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_scatter2_add": (_i, [_p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "iswm_add_bf16": (_i, [_p, _p, _i64, _p, _p]),
    "iswm_nhwc_to_nchw_f32": (_i, [_p, _i, _i, _i64, _i, _p, _p]),
    "iswm_nchw_f32_to_nhwc": (_i, [_p, _i, _i64, _i, _p, _i, _p]),
    "iswm_bias_grad_nchw": (_i, [_p, _i, _i, _i64, _p, _p]),
    "iswm_scale_by_device_scalar": (_i, [_p, _i, _i64, _p, _p]),
    "iswm_sgd_step": (_i, [_p, _p, _p, _i64, _f, _f, _f, _i, _i, _p, _p]),
    "iswm_adam_step": (_i, [_p, _p, _p, _p, _i64, _f, _f, _f, _f, _f, _i, _i64, _p, _p, _p]),
    "iswm_u8_to_f32_norm": (_i, [_p, _i, _i, _i, _i, _p, _p, C.POINTER(C.c_float), C.POINTER(C.c_float), _i, _i, _p, _p]),
    "iswm_crop_flip_u8": (_i, [_p, _i, _i, _i, _p, _p, _i, _i, _p, _p]),
    "iswm_random_scale_table_words": (_i64, [_i, _i, _i]),
    "iswm_tail_fwd": (_i, [_p, _i, _i, _i, _p, _i, _i, _i, _p, _i, _p, _p, _p, _p]),
    "iswm_tail_loss": (_i, [_p, _p, _p, _i, _p, _p]),
    "iswm_tail_bwd": (_i, [_p, _i, _i, _i, _p, _p, _i, _p, _p, _i, _p, _p, _p]),
    "iswm_mask_work_bytes": (_i64, [_i, _i, _i]),
    "iswm_mask_preprocess": (_i, [_p, _i, _i, _i, _i, C.c_double, _p, _p, _p, _p, _p]),
    "iswm_region_components": (_i, [_p, _i, _p, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p]),
    "iswm_front_nearest": (_i, [_p, _p, _i, _i, _p, _p, _p]),
    "iswm_front_window_diff": (_i, [_p, _p, _i, _i, _i, _i, _p, _p]),
    "iswm_random_scale_crop": (_i, [_p, _p, _i, _i, _i, _i, _p, _i, _i, _i, _p, C.POINTER(C.c_float), C.POINTER(C.c_float), _i, _i, _p, _p, _p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raise loudly if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). iswm_b200 has no CPU or PyTorch fallback."
            )
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().iswm_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libiswm_b200 {what} failed (rc={rc}): {msg}")


def launch_count() -> int:
    return int(lib().iswm_launch_count())

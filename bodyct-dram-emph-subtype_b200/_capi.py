"""ctypes binding of libdram_b200.so (include/dram_b200.h).

This is the only place that touches the shared library.  Loading never needs a GPU (the
library links cudart statically and resolves the driver lazily), so the symbol table can be
checked on a CPU box; every compute entry point needs a B200.
There is no fallback: if the library is missing, `load()` raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# DRAM_B200_LIB selects another build of the same sources (kernel tuning experiments, build.build_variant)
LIB_PATH = os.environ.get("DRAM_B200_LIB") or os.path.join(HERE, "libdram_b200.so")

DRAM_OK = 0
DRAM_DTYPE_BF16 = 0
DRAM_DTYPE_F16 = 1
CONV_ALGO = {"auto": 0, "tiles": 1, "planes": 2}
CONV_EPILOGUE = {"auto": 0, "direct": 1, "staged": 2}
LOSS_COEF_HEAD = 16  # DRAM_LOSS_COEF_HEAD
PEER_HANDLE_BYTES = 64  # DRAM_PEER_HANDLE_BYTES


class ConvDesc(C.Structure):
    """Mirror of `dram_conv_desc` (include/dram_b200.h)."""

    _fields_ = [
        ("n", C.c_int32), ("di", C.c_int32), ("hi", C.c_int32), ("wi", C.c_int32),
        ("c1", C.c_int32), ("c2", C.c_int32),
        ("cout", C.c_int32),
        ("kd", C.c_int32), ("kh", C.c_int32), ("kw", C.c_int32),
        ("sd", C.c_int32), ("sh", C.c_int32), ("sw", C.c_int32),
        ("dd", C.c_int32), ("dh", C.c_int32), ("dw", C.c_int32),
        ("pd", C.c_int32), ("ph", C.c_int32), ("pw", C.c_int32),
        ("relu", C.c_int32),
        ("res_c", C.c_int32), ("res_stride", C.c_int32),
        ("res_d", C.c_int32), ("res_h", C.c_int32), ("res_w", C.c_int32),
        ("n_heads", C.c_int32), ("head_ch", C.c_int32 * 2), ("head_sigmoid", C.c_int32),
        ("store_out", C.c_int32),
        ("tw", C.c_int32), ("th", C.c_int32), ("td", C.c_int32),
        ("dtype", C.c_int32),
        ("algo", C.c_int32),
        ("src1_up2x", C.c_int32),
        ("epilogue", C.c_int32),
    ]


_vp, _i32, _i64, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_size_t
_pi32 = C.POINTER(C.c_int32)

# name -> (restype, argtypes); must list every symbol include/dram_b200.h declares.
SIGNATURES = {
    "dram_version": (C.c_int, []),
    "dram_last_error": (C.c_int, [C.c_char_p, _sz]),
    "dram_sm_count": (C.c_int, []),
    "dram_set_saturation_counter": (C.c_int, [_vp]),
    "dram_conv3d_out_dims": (C.c_int, [C.POINTER(ConvDesc), _pi32, _pi32, _pi32]),
    "dram_conv3d_plan_create": (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _vp, _vp, C.POINTER(_vp)]),
    "dram_conv3d_plan_destroy": (C.c_int, [_vp]),
    "dram_conv3d_run": (C.c_int, [_vp, _i32, _vp]),
    "dram_conv3d_plan_info": (C.c_int, [_vp, C.POINTER(_i64), _pi32, _pi32, _pi32, _pi32]),
    "dram_conv3d_plan_executed_flops": (C.c_int, [_vp, C.POINTER(_i64)]),
    "dram_conv3d_worklist_size": (C.c_int, [_vp, _pi32]),
    "dram_conv3d_worklist": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "dram_conv3d_run_listed": (C.c_int, [_vp, _vp, _vp, _i32, _vp]),
    "dram_stem_expand": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_stem_weight_bytes": (_sz, []),
    "dram_stem_conv7": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_stem_conv7_hu": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32,
                                     _i32, _vp]),
    "dram_maxpool3d": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_upsample2x": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_upsample2x_plan_create": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, C.POINTER(_vp)]),
    "dram_upsample2x_plan_destroy": (C.c_int, [_vp]),
    "dram_upsample2x_plan_run": (C.c_int, [_vp, _i32, _vp]),
    "dram_upsample2x_worklist_size": (C.c_int, [_vp, _pi32]),
    "dram_upsample2x_worklist": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "dram_upsample2x_plan_run_listed": (C.c_int, [_vp, _vp, _vp, _i32, _vp]),
    "dram_decoder_support": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "dram_upconv_axis": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i64, _i32, _i32, _i32, _vp]),
    "dram_pool_workspace_bytes": (_sz, [_i32, _i32]),
    "dram_masked_pool": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_dram_workspace_bytes": (_sz, [_i32]),
    "dram_dram_upsample_mask": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32,
                                          _i32, _i32, _i32, _i32, _vp]),
    "dram_lobe_workspace_bytes": (_sz, [_i32, _i64]),
    "dram_lobe_sums": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _vp]),
    "dram_preprocess_workspace_bytes": (_sz, []),
    "dram_window_standardize": (C.c_int, [_vp, _vp, _vp, _vp, _i64, C.c_float, C.c_float, _vp]),
    "dram_preprocess_workspace_bytes_n": (_sz, [_i32]),
    "dram_window_standardize_batch": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, C.c_float, C.c_float, _vp]),
    "dram_window_stats": (C.c_int, [_vp, _vp, _vp, _i32, _i64, C.c_float, C.c_float, _vp]),
    "dram_window_lut": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, C.c_float, C.c_float, _vp]),
    "dram_resize_image": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_resize_mask": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_resize_labels": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_mask_bbox": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp]),
    "dram_lung_crop_workspace_bytes": (_sz, [_i32, _i32, _i32]),
    "dram_lung_crop": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "dram_label_counts": (C.c_int, [_vp, _i64, _vp, _vp]),
    "dram_label_hu_hist": (C.c_int, [_vp, _vp, _i64, _vp, _i32, _vp, _vp, _vp]),
    "dram_heatmap_u8": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_conv3d_wgrad_workspace_bytes": (_i64, [C.POINTER(ConvDesc)]),
    "dram_conv3d_wgrad_plan_create": (C.c_int, [C.POINTER(ConvDesc), _vp, _vp, _vp, _i32, _i32, _vp, _i64, C.POINTER(_vp)]),
    "dram_conv3d_wgrad_plan_destroy": (C.c_int, [_vp]),
    "dram_conv3d_wgrad_plan_info": (C.c_int, [_vp, C.POINTER(_i64), _pi32, _pi32, _pi32]),
    "dram_conv3d_wgrad_run": (C.c_int, [_vp, _i32, _i32, _vp]),
    "dram_bn_workspace_bytes": (_i64, [_i32]),
    "dram_bn_stats": (C.c_int, [_vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "dram_bn_finalize": (C.c_int, [_vp, C.c_double, _vp, _vp, C.c_float, C.c_float, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "dram_bn_apply": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _i64, _i32, _i32, _vp]),
    "dram_bn_backward_reduce": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "dram_bn_backward_apply": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _i64, _i32, _i32, _vp]),
    "dram_upsample2x_backward": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_maxpool3d_backward_workspace_bytes": (_i64, [_i32, _i32, _i32, _i32, _i32]),
    "dram_maxpool3d_backward": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_heads_workspace_bytes": (_i64, []),
    "dram_heads_sigmoid_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "dram_heads_sigmoid_backward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    "dram_peer_exchange_bytes": (_i64, []),
    "dram_peer_alloc": (C.c_int, [_i64, C.POINTER(_vp), _vp]),
    "dram_peer_open": (C.c_int, [_vp, C.POINTER(_vp)]),
    "dram_peer_close": (C.c_int, [_vp]),
    "dram_peer_free": (C.c_int, [_vp]),
    "dram_peer_allreduce_f64": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _i32, C.c_uint64, _vp, _vp]),
    "dram_train_loss_workspace_bytes": (_i64, [_i32]),
    "dram_train_loss_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32,
                                          _i32, _i32, C.c_float, C.c_float, _vp, _vp, _vp]),
    "dram_train_loss_backward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32,
                                           _i32, _vp, _vp, _vp]),
    "dram_adam_step": (C.c_int, [_vp, _vp, _vp, _vp, _i64, C.c_double, C.c_double, C.c_double, C.c_double, _i32,
                                 C.c_float, _vp]),
    "dram_pack_conv_weight": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_ncdhw_f32_to_ndhwc_16": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "dram_ndhwc_16_to_ncdhw_f32": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
}

_lib = None


class DramError(RuntimeError):
    """A libdram_b200 call returned a negative status."""


def load():
    """Loads the library once and types every entry point.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python {os.path.join(HERE, 'build.py')}` "
            "(there is no CPU or library fallback for this path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    buf = C.create_string_buffer(512)
    load().dram_last_error(buf, len(buf))
    return buf.value.decode("utf-8", "replace")


def check(status, what):
    if status != DRAM_OK:
        raise DramError(f"{what} failed ({status}): {last_error()}")

"""ctypes binding of libtrainner_b200.so (the C ABI declared in include/trainner_b200.h).

There is NO fallback: if the shared library is missing the import of any compute module raises,
and every compute entry point raises RuntimeError with the library's message on failure.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtrainner_b200.so")

MAX_TAPS = 16


class ConvDesc(C.Structure):
    _fields_ = [
        ("n", C.c_int32), ("h_in", C.c_int32), ("w_in", C.c_int32),
        ("cx", C.c_int32), ("cin_off", C.c_int32), ("cin", C.c_int32),
        ("h_out", C.c_int32), ("w_out", C.c_int32),
        ("h_buf", C.c_int32), ("w_buf", C.c_int32), ("cy", C.c_int32),
        ("cout_off", C.c_int32), ("cout", C.c_int32),
        ("ntaps", C.c_int32),
        ("tap_dy", C.c_int8 * MAX_TAPS), ("tap_dx", C.c_int8 * MAX_TAPS), ("tap_w", C.c_int8 * MAX_TAPS),
        ("in_stride", C.c_int32), ("in_off_y", C.c_int32), ("in_off_x", C.c_int32),
        ("out_mul_y", C.c_int32), ("out_off_y", C.c_int32), ("out_mul_x", C.c_int32), ("out_off_x", C.c_int32),
        ("upsample2x", C.c_int32),
        ("w_taps", C.c_int32), ("w_cout_pad", C.c_int32), ("w_cin_pad", C.c_int32),
        ("alpha", C.c_float), ("act", C.c_int32), ("slope", C.c_float),
        ("beta1", C.c_float), ("beta2", C.c_float),
        ("res_nch", C.c_int32),
        ("res1_c", C.c_int32), ("res1_coff", C.c_int32), ("res2_c", C.c_int32), ("res2_coff", C.c_int32),
        ("accumulate", C.c_int32),
        ("mask_c", C.c_int32), ("mask_coff", C.c_int32), ("mask_lo", C.c_int32), ("mask_hi", C.c_int32),
        ("mask_slope", C.c_float),
        ("parity_classes", C.c_int32),
    ]


class FlatDesc(C.Structure):
    _fields_ = [
        ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
        ("cx", C.c_int32), ("cin_off", C.c_int32), ("cin", C.c_int32),
        ("cx2", C.c_int32), ("cin2_off", C.c_int32), ("cin2", C.c_int32),
        ("cy", C.c_int32), ("cout_off", C.c_int32), ("cout", C.c_int32),
        ("tap_dy", C.c_int8 * 9), ("tap_dx", C.c_int8 * 9), ("tap_w", C.c_int8 * 9),
        ("out_mode", C.c_int32),
        ("w_taps", C.c_int32), ("w_cout_pad", C.c_int32), ("w_cin_pad", C.c_int32),
        ("alpha", C.c_float), ("act", C.c_int32), ("slope", C.c_float),
        ("beta1", C.c_float), ("beta2", C.c_float),
        ("res_nch", C.c_int32), ("res1_c", C.c_int32), ("res1_coff", C.c_int32),
        ("res2_c", C.c_int32), ("res2_coff", C.c_int32),
        ("accumulate", C.c_int32),
        ("mask_c", C.c_int32), ("mask_coff", C.c_int32), ("mask_lo", C.c_int32), ("mask_hi", C.c_int32),
        ("mask_slope", C.c_float),
    ]


class WgradDesc(C.Structure):
    _fields_ = [
        ("n", C.c_int32), ("h_in", C.c_int32), ("w_in", C.c_int32), ("cx", C.c_int32),
        ("x_coff", C.c_int32), ("cin", C.c_int32),
        ("h_out", C.c_int32), ("w_out", C.c_int32), ("cdy", C.c_int32), ("dy_coff", C.c_int32),
        ("cout", C.c_int32),
        ("kh", C.c_int32), ("kw", C.c_int32), ("stride", C.c_int32), ("pad", C.c_int32),
        ("scale", C.c_float),
    ]


class WgradRdbEntry(C.Structure):
    _fields_ = [("dw", C.c_void_p * 5), ("scale5", C.c_float), ("pad_", C.c_int32)]


class ColsumEntry(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("npix", C.c_int64),
                ("pitch", C.c_int32), ("coff", C.c_int32), ("c", C.c_int32), ("scale", C.c_float)]


class BnFinalizeEntry(C.Structure):
    _fields_ = [("stats", C.c_void_p), ("mean_invstd", C.c_void_p), ("running_mean", C.c_void_p),
                ("running_var", C.c_void_p), ("npix", C.c_int64), ("c", C.c_int32), ("momentum", C.c_float),
                ("eps", C.c_float), ("pad_", C.c_int32)]


class PackCatEntry(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p),
                ("cout", C.c_int32), ("cin", C.c_int32), ("taps", C.c_int32), ("ci_off", C.c_int32),
                ("n_rows", C.c_int32), ("rows_pad", C.c_int32), ("cols_pad", C.c_int32), ("col_off", C.c_int32),
                ("scale", C.c_float), ("row_off", C.c_int32), ("mode", C.c_int32), ("pad_", C.c_int32)]


class ChainStage(C.Structure):
    _fields_ = [("out", C.c_void_p), ("bias", C.c_void_p), ("mask", C.c_void_p), ("res1", C.c_void_p),
                ("res2", C.c_void_p),
                ("out_c", C.c_int32), ("out_coff", C.c_int32), ("mask_c", C.c_int32), ("mask_coff", C.c_int32),
                ("res1_c", C.c_int32), ("res1_coff", C.c_int32), ("res2_c", C.c_int32), ("res2_coff", C.c_int32),
                ("alpha", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("slope", C.c_float),
                ("mask_slope", C.c_float), ("act", C.c_int32), ("pad_", C.c_int32 * 2)]


class ChainDesc(C.Structure):
    _fields_ = [("n_total", C.c_int32), ("img0", C.c_int32), ("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("cx", C.c_int32), ("x_coff", C.c_int32), ("n_blocks", C.c_int32), ("flip_taps", C.c_int32)]


class PackEntry(C.Structure):
    _fields_ = [
        ("src", C.c_void_p), ("dst", C.c_void_p),
        ("cout", C.c_int32), ("cin", C.c_int32), ("taps", C.c_int32),
        ("rows_pad", C.c_int32), ("cols_pad", C.c_int32), ("mode", C.c_int32),
        ("co_mul", C.c_int32), ("co_off", C.c_int32),
    ]


_P, _I, _L, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_float

_SIGNATURES = {
    "b200_conv_igemm": [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P, _P, _P],
    "b200_conv_igemm_stats": [_P, _P, _P, _P, _P, _P, _P],
    "b200_conv3x3_flat": [C.POINTER(FlatDesc), _P, _P, _P, _P, _P, _P, _P, _P, _P],
    "b200_pack_cat": [_P, _I, _I, _P],
    "b200_rdb_chain": [C.POINTER(ChainDesc), _P, _P, _P, _P, _L, _P, _P],
    "b200_rdb_chain_geometry": [_I, _I, _I, _P, _P],
    "b200_pad_copy": [_P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P],
    "b200_unpad_add": [_P, _I, _P, _I, _I, _P, _I, _I, _I, _I, _I, _P],
    "b200_conv_wgrad": [C.POINTER(WgradDesc), _P, _P, _P, _P, _P],
    "b200_wgrad_rdb_make_maps": [_P, _I, _P, _P, _P, _P, _I, _I, _I, _I],
    "b200_wgrad_rdb": [_P, _P, _I, _I, _I, _I, _I, _I, _P, _L, _P],
    "b200_colsum_multi": [_P, _I, _P],
    "b200_pack_weights": [_P, _I, _I, _P],
    "b200_conv3x3_thin_to_wide": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _I, _F,
                                  _P, _I, _I, _F, _P],
    "b200_conv3x3_wide_to_thin": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _F, _P],
    "b200_conv3x3_thin_wgrad": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P],
    "b200_bn_stats_finalize": [_P, _P, _P, _P, _P, _L, _I, _F, _F, _P],
    "b200_bn_partials_finalize": [_P, _I, _P, _P, _P, _P, _L, _I, _F, _F, _P],
    "b200_bn_finalize_multi": [_P, _I, _I, _P],
    "b200_bn_apply_lrelu": [_P, _P, _P, _P, _P, _L, _I, _F, _P],
    "b200_bn_bwd_reduce": [_P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _P],
    "b200_bn_bwd_apply": [_P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _I, _P],
    "b200_maxpool2x2": [_P, _P, _I, _I, _I, _I, _P],
    "b200_maxpool2x2_bwd": [_P, _P, _P, _I, _I, _I, _I, _P],
    "b200_sumpool2x2_mask": [_P, _P, _P, _I, _I, _I, _I, _F, _P],
    "b200_pixel_shuffle2": [_P, _P, _I, _I, _I, _I, _I, _F, _P],
    "b200_pixel_unshuffle2": [_P, _P, _I, _I, _I, _I, _P],
    "b200_l1_loss_f32": [_P, _P, _P, _P, _L, _F, _P],
    "b200_l1_loss_bf16": [_P, _P, _P, _P, _L, _F, _P],
    "b200_lrelu_mask_mul": [_P, _P, _P, _L, _F, _P],
    "b200_nchw_f32_to_nhwc_bf16": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
    "b200_nhwc_bf16_to_nchw_f32": [_P, _P, _I, _I, _I, _I, _I, _I, _P],
}

EXPORTED_SYMBOLS = sorted(list(_SIGNATURES) + ["b200_last_error", "b200_version", "b200_device_ok",
                                                "b200_launch_count", "b200_tensor_map_bytes",
                                                "b200_wgrad_rdb_ws_bytes", "b200_conv_igemm_stat_rows"])


def _load():
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "trainner_b200: %s not found. Build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a). There is no CPU / PyTorch fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, args in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.b200_last_error.restype = C.c_char_p
    lib.b200_version.restype = C.c_int
    lib.b200_device_ok.restype = C.c_int
    lib.b200_launch_count.restype = C.c_int64
    lib.b200_tensor_map_bytes.restype = C.c_int
    lib.b200_tensor_map_bytes.argtypes = []
    lib.b200_conv_igemm_stat_rows.restype = C.c_int
    lib.b200_conv_igemm_stat_rows.argtypes = [C.POINTER(ConvDesc)]
    lib.b200_wgrad_rdb_ws_bytes.restype = C.c_int64
    lib.b200_wgrad_rdb_ws_bytes.argtypes = [_I, _I, _I, _I]
    return lib


lib = _load()


def check(rc, what=""):
    if rc != 0:
        raise RuntimeError("trainner_b200 %s failed: %s" % (what, lib.b200_last_error().decode()))


def launch_count():
    return int(lib.b200_launch_count())

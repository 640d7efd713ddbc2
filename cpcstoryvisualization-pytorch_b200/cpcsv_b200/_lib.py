"""ctypes binding of libcpcsv.so (the C ABI declared in include/cpcsv.h).

The library is loaded lazily on first use and the load fails loudly: there is no CPU or
PyTorch fallback for any kernel (BASELINE.json north_star).  The shared object is built
in-tree by ``csrc/Makefile`` (``__graft_entry__.build()``).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcpcsv.so")
MAX_TAPS = 16


class View5(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("dims", C.c_int64 * 5), ("strides", C.c_int64 * 5)]


class Tap(C.Structure):
    _fields_ = [("a", C.c_int32 * 4), ("b", C.c_int32 * 4), ("out_off", C.c_int64)]


class Gemm(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("dtype", C.c_int32), ("planes", C.c_int32),
        ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("tile_n", C.c_int32), ("tile_h", C.c_int32), ("tile_w", C.c_int32),
        ("groups", C.c_int32), ("taps_per_group", C.c_int32), ("k_blocks", C.c_int32),
        ("m_valid", C.c_int32), ("n_valid", C.c_int32), ("block_n", C.c_int32),
        ("n_tiles", C.c_int32), ("splits", C.c_int32), ("accumulate", C.c_int32), ("cta_pair", C.c_int32),
        ("out_stride_n", C.c_int64), ("out_stride_h", C.c_int64), ("out_stride_w", C.c_int64),
        ("ldc", C.c_int64),
        ("alpha", C.c_void_p), ("out", C.c_void_p), ("stats", C.c_void_p), ("stats_ld", C.c_int64),
        ("a", View5 * 2), ("b", View5 * 2),
        ("taps", Tap * MAX_TAPS),
    ]


MAX_PLANES = 6


class AdamHyper(C.Structure):
    _fields_ = [("lr", C.c_void_p), ("bc", C.c_void_p), ("beta1", C.c_double), ("beta2", C.c_double),
                ("eps", C.c_double)]


class AdamTensor(C.Structure):
    _fields_ = [("p", C.c_void_p), ("g", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("n", C.c_int64)]


class Plane(C.Structure):
    _fields_ = [("kind", C.c_int32), ("dtype", C.c_int32), ("rows_pad", C.c_int32), ("cols_pad", C.c_int32),
                ("hi", C.c_void_p), ("lo", C.c_void_p)]


_i32, _i64, _f32, _p = C.c_int32, C.c_int64, C.c_float, C.c_void_p

# name -> argument ctypes (every function returns int unless noted)
SIGNATURES = {
    "cpcsv_conv_gemm": [C.POINTER(Gemm), _p],
    "cpcsv_bn_stats": [_p, _i64, _i32, _i64, _p, _p],
    "cpcsv_bn_finalize": [_p, _i64, _i32, _p, _p, _p, _p, _p, _i32, _f32, _f32, _p, _p, _p, _p, _p],
    "cpcsv_bn_act_pack": [_p, _i64, _i32, _i64, _p, _p, _i32, _p, _i64, _p, _i64, _p, _p, _i64, _i32, _p],
    "cpcsv_bn_bwd_reduce": [_p, _p, _i64, _i32, _i64, _i64, _p, _p, _p, _p, _i32, _p, _i64, _p, _p],
    "cpcsv_bn_bwd_apply": [_p, _p, _i64, _i32, _i64, _i64, _p, _p, _p, _p, _p, _p, _i32, _i32, _p, _i64,
                           _p, _i32, _p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _p, _p],
    "cpcsv_bn_norm_act_pack": [_p, _i64, _i32, _i64, _p, _p, _p, _p, _p, _p, _i32, _f32, _f32, _p, _i32, _p, _i64,
                               _p, _i64, _p, _p, _i64, _i32, _p],
    "cpcsv_bn_add_act_pack": [_p, _i64, _i32, _i64, _p, _p, _p, _i64, _p, _p, _i32, _p, _i64, _p, _p, _i64, _i32,
                              _p],
    "cpcsv_resize_im2col": [_p, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _i32, _f32, _f32, _p, _p, _i32, _i32, _p],
    "cpcsv_pool3x3": [_p, _i32, _i32, _i32, _i32, _i64, _i64, _i64, _i32, _i32, _p, _i64, _i64, _i64, _p, _p, _i64,
                      _i64, _i64, _i32, _p],
    "cpcsv_ssim": [_p, _p, _i32, _i32, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _i64,
                   _f32, _f32, _p, _p],
    "cpcsv_images_to_u8": [_p, _i32, _i32, _i32, _i64, _i64, _i64, _p, _p],
    "cpcsv_pack_nchw": [_p, _i32, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _p, _i32, _i64, _p, _p,
                        _i32, _i32, _p],
    "cpcsv_im2col_small": [_p, _i32, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _i32, _i32, _i32, _p, _p,
                           _i32, _i32, _p],
    "cpcsv_enc0_lrelu_fwd": [_p, _i32, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _p, _i32, _p, _f32, _p, _p, _i32,
                             _i32, _p],
    "cpcsv_lrelu_bwd16": [_p, _p, _i64, _f32, _p, _p],
    "cpcsv_col2im_small": [_p, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p],
    "cpcsv_head_gather_tanh": [_p, _i64, _i32, _i32, _i32, _i32, _p, _p],
    "cpcsv_tanh_bwd_im2col": [_p, _i64, _i64, _i64, _i64, _p, _i32, _i32, _i32, _i32, _p, _i32, _i32, _p],
    "cpcsv_pack_matrix": [_p, _i64, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _i64, _i32, _p],
    "cpcsv_scatter_rows_f32": [_p, _i64, _p, _p, _i64, _i64, _i64, _p],
    "cpcsv_pack_conv_weight": [_p, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _i32, _p],
    "cpcsv_unpack_conv_wgrad": [_p, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _p, _p, _p],
    "cpcsv_linear_f32": [_p, _i64, _p, _i64, _p, _p, _i64, _i32, _i32, _i32, _i32, _p],
    "cpcsv_linear_tn_f32": [_p, _i64, _p, _i64, _p, _i64, _i32, _i32, _i32, _i32, _p],
    "cpcsv_linear_nn_f32": [_p, _i64, _p, _i64, _p, _i64, _i32, _i32, _i32, _i32, _p],
    "cpcsv_gru_gates_fwd": [_p, _p, _p, _i32, _i32, _p, _p, _p],
    "cpcsv_gru_gates_bwd": [_p, _p, _p, _i32, _i32, _p, _p, _p, _p],
    "cpcsv_ca_fwd": [_p, _p, _i32, _i32, _p, _p, _p, _p],
    "cpcsv_ca_bwd": [_p, _p, _p, _p, _p, _i32, _i32, _p, _p],
    "cpcsv_dfn1d_fwd": [_p, _p, _i32, _i32, _i32, _i32, _p, _p],
    "cpcsv_dfn1d_bwd": [_p, _p, _p, _i32, _i32, _i32, _i32, _p, _p, _p],
    "cpcsv_tanh_fwd": [_p, _p, _i64, _p],
    "cpcsv_tanh_bwd": [_p, _p, _p, _i64, _p],
    "cpcsv_affine_sigmoid_fwd": [_p, _p, _p, _p, _i64, _p],
    "cpcsv_affine_sigmoid_bwd": [_p, _p, _p, _p, _p, _i64, _p],
    "cpcsv_spectral_sigma": [_p, _i32, _i32, _p, _p, _i32, _f32, _p, _p, _p, _p],
    "cpcsv_spectral_bwd": [_p, _p, _p, _p, _p, _i32, _i32, _p, _p, _p],
    "cpcsv_spectral_bwd_apply": [_p, _p, _p, _p, _p, _i32, _i32, _p, _p],
    "cpcsv_unpack_conv_wgrad_dot": [_p, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p],
    "cpcsv_adam_tick": [_p, C.c_double, C.c_double, _p, _p],
    "cpcsv_adam_multi": [C.POINTER(AdamTensor), _i32, C.POINTER(AdamHyper), _p],
    "cpcsv_adam_pack_conv": [_p, _p, _p, _p, _i32, _i32, _i32, _i32, C.POINTER(AdamHyper), C.POINTER(Plane),
                             _i32, _p],
    "cpcsv_adam_pack_fc": [_p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, C.POINTER(AdamHyper), _p, _p, _p, _p,
                           _p],
}
OTHER_SYMBOLS = ("cpcsv_version", "cpcsv_last_error_string", "cpcsv_launch_count",
                 "cpcsv_bn_workspace_doubles")

_lib = None


def load():
    """Load libcpcsv.so (once).  Raises RuntimeError when the extension is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libcpcsv.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (there is no CPU / PyTorch fallback for the CP-CSV kernels)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    lib.cpcsv_version.restype = C.c_int
    lib.cpcsv_last_error_string.restype = C.c_char_p
    lib.cpcsv_launch_count.restype = C.c_int64
    lib.cpcsv_bn_workspace_doubles.argtypes = [C.c_int64, C.c_int32]
    lib.cpcsv_bn_workspace_doubles.restype = C.c_int64
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().cpcsv_last_error_string().decode("utf-8", "replace")
        raise RuntimeError("%s failed (rc=%d): %s" % (what, rc, msg))


def launch_count():
    return int(load().cpcsv_launch_count())

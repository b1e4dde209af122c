"""ctypes binding of libopenstereo_b200.so (the C ABI in include/openstereo_b200.h).

There is deliberately NO fallback: if the shared library is missing or a symbol is absent the
import fails loudly, and every compute entry point raises when it is handed a non-CUDA tensor.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libopenstereo_b200.so")

_f32p = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_s = ctypes.c_void_p

# name -> argtypes; every name must be exported by the library and declared in the header.
SIGNATURES = {
    "osb_gwc_volume_fwd": [_f32p, _f32p, _f32p, _i, _i, _i, _i, _i, _i, _s],
    "osb_concat_volume_fwd": [_f32p, _f32p, _f32p, _i, _i, _i, _i, _i, _i, _s],
    "osb_gwc_concat_volume_fwd": [_f32p, _f32p, _f32p, _f32p, _f32p, _i, _i, _i, _i, _i, _i, _i, _s],
    "osb_corr_volume_fwd": [_f32p, _f32p, _f32p, _i, _i, _i, _i, _i, _s],
    "osb_softargmin_fwd": [_f32p, _f32p, _i, _i, _i, _i, _f, _f, _f, _i, _s],
    "osb_upsample_softargmin_fwd": [_f32p, _f32p, _i, _i, _i, _i, _i, _i, _i, _i, _s],
    "osb_epe_partial_fwd": [_f32p, _f32p, _f32p, _i, _i, _f, _s],
    "osb_conv3d_k3_bn_act_fwd": [_f32p] * 7 + [_i] * 8 + [_s],
    "osb_deconv3d_bn_act_fwd": [_f32p] * 6 + [_i] * 8 + [_s],
    "osb_conv3d_1x1_bn_act_fwd": [_f32p, _f32p, _i] + [_f32p] * 6 + [_i] * 8 + [_s],
    "osb_conv3d_tc_supported": [_i, _i, _i, _i],
    "osb_conv3d_tc_kc": [_i, _i, _i, _i],
    "osb_tc_general_width": [_i],
    "osb_conv3d_s2_tc_supported": [_i, _i, _i, _i, _i],
    "osb_deconv3d_tc_supported": [_i, _i, _i],
    "osb_deconv3d_k3_tc_fwd": [_f32p] * 6 + [_i] * 9 + [_s],
    "osb_conv3d_k3_s2_tc_fwd": [_f32p] * 6 + [_i] * 9 + [_s],
    "osb_conv3d_k3_tc_fwd": [_f32p] * 6 + [_i] * 9 + [_s],
    "osb_conv3d_k3_tc_ncdhw_fwd": [_f32p] * 6 + [_i] * 9 + [_s],
    "osb_conv3d_k3_tc_gate_fwd": [_f32p] * 7 + [_i] * 7 + [_s],
    "osb_deconv3d_k4_tc_supported": [_i, _i, _i],
    "osb_conv3d_k3_tc_cs_fwd": [_f32p] * 7 + [_i] * 8 + [_s],
    "osb_conv3d_k3_s2_tc_cs_fwd": [_f32p] * 5 + [_i] * 8 + [_s],
    "osb_deconv3d_k4_tc_cs_fwd": [_f32p] * 5 + [_i] * 8 + [_s],
    "osb_deconv3d_k4_tc_fwd": [_f32p] * 6 + [_i] * 10 + [_s],
    "osb_conv1x1_ndhwc_cat_fwd": [_f32p, _f32p, _i, _i, _f32p, _f32p, _f32p, _f32p, ctypes.c_longlong, _i, _i, _s],
    "osb_feature_att_gate_fwd": [_f32p] * 8 + [_i] * 7 + [_s],
    "osb_ncdhw_to_ndhwc_pad": [_f32p, _f32p, _i, _i, _i, _i, _i, _i, _s],
    "osb_conv1x1_ndhwc_fwd": [_f32p] * 5 + [ctypes.c_longlong, _i, _i, _i, _s],
    "osb_conv3d_k3_c1_ndhwc_fwd": [_f32p] * 5 + [_i] * 5 + [_s],
    "osb_avgpool_pairs_fwd": [_f32p, _f32p, ctypes.c_longlong, _i, ctypes.c_longlong, _s],
    "osb_geo_lookup_fwd": [_f32p] * 11 + [_i] * 8 + [_s],
    "osb_context_upsample_fwd": [_f32p] * 3 + [_i] * 4 + [_s],
    "osb_conv2d_tc_kc": [_i] * 4,
    "osb_conv2d_k3_tc_fwd": [_f32p] * 6 + [_i] * 9 + [_s],
    "osb_ncdhw_to_ndhwc": [_f32p, _f32p, _i, _i, _i, _i, _i, _s],
    "osb_gwc_volume_sum_fwd": [_f32p, _f32p, _f32p, _i, _i, _i, _i, _i, _i, _s],
    "osb_group_l2_normalize_fwd": [_f32p, _f32p, _i, _i, _i, _i, _i, _f, _s],
    "osb_sub_volume_fwd": [_f32p, _f32p, _f32p, _i, _i, _i, _i, _i, _s],
    "osb_regression_values_fwd": [_f32p, _f32p, _f32p, _i, _i, _i, _i, _s],
    "osb_gwc_volume_bwd": [_f32p] * 5 + [_i] * 7 + [_s],
    "osb_concat_volume_bwd": [_f32p] * 3 + [_i] * 6 + [_s],
    "osb_softargmin_bwd": [_f32p] * 3 + [_i] * 4 + [_f, _f, _f, _i, _s],
    "osb_dwconv2d_fwd": [_f32p] * 6 + [_i] * 8 + [_s],
    "osb_deconv2d_k3s2_fwd": [_f32p] * 6 + [_i] * 6 + [_s],
    "osb_conv3d_tc_h16_supported": [_i, _i, _i],
    "osb_conv3d_s2_tc_h16_supported": [_i] * 5,
    "osb_conv3d_k3_tc_h16_fwd": [_f32p] * 5 + [_i] * 7 + [_s],
    "osb_conv3d_k3_tc_gate_h16_fwd": [_f32p] * 6 + [_i] * 7 + [_s],
    "osb_conv3d_k3_s2_tc_h16_fwd": [_f32p] * 5 + [_i] * 7 + [_s],
    "osb_deconv3d_k4_tc_h16_fwd": [_f32p] * 5 + [_i] * 9 + [_s],
    "osb_conv3d_k3_tc_cs_h16_fwd": [_f32p] * 6 + [_i] * 8 + [_s],
    "osb_conv3d_k3_s2_tc_cs_h16_fwd": [_f32p] * 5 + [_i] * 8 + [_s],
    "osb_deconv3d_k4_tc_cs_h16_fwd": [_f32p] * 5 + [_i] * 8 + [_s],
    "osb_conv1x1_ndhwc_cat_h16_fwd": [_f32p, _f32p, _i, _i, _f32p, _f32p, _f32p, _f32p, ctypes.c_longlong, _i, _i, _s],
    "osb_ncdhw_to_ndhwc_pad_h16": [_f32p, _f32p, _i, _i, _i, _i, _i, _i, _s],
}


class NativeLibraryError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            "%s not found: build it with `python -m openstereo_b200.build` (there is no CPU/PyTorch fallback)"
            % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.osb_abi_version.restype = ctypes.c_int
    lib.osb_last_error.restype = ctypes.c_char_p
    lib.osb_launch_count.restype = ctypes.c_uint64
    lib.osb_tc_overflow_count.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_uint)]
    lib.osb_tc_overflow_count.restype = ctypes.c_int
    lib.osb_tc_overflow_poll.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.osb_tc_overflow_poll.restype = ctypes.c_int
    lib.osb_tc_overflow_flag.argtypes = []
    lib.osb_tc_overflow_flag.restype = ctypes.c_void_p
    lib.osb_set_rz_kappa.argtypes = [ctypes.c_float]
    lib.osb_set_rz_kappa.restype = ctypes.c_float
    for name, argtypes in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise NativeLibraryError("%s does not export %s" % (LIB_PATH, name)) from exc
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int
    return lib


lib = _load()

_ERRORS = {1: ValueError, 2: RuntimeError, 3: NotImplementedError}


def call(name, *args):
    """Invoke an entry point; translate OSB_E* into the exception class the reference would raise."""
    if len(args) != len(SIGNATURES[name]):          # ctypes would silently pass extra args as 32-bit ints
        raise TypeError("%s takes %d arguments (%d given)" % (name, len(SIGNATURES[name]), len(args)))
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = (lib.osb_last_error() or b"").decode("utf-8", "replace")
        raise _ERRORS.get(rc, RuntimeError)("%s: %s" % (name, msg))


def launch_count():
    return int(lib.osb_launch_count())

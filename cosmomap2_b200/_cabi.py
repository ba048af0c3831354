"""
ctypes binding of libcosmomap2_b200.so (the C ABI declared in include/cosmomap2_b200.h).

There is no CPU fallback: if the shared library is missing the import fails loudly, and every
entry point raises ``RuntimeError`` with the library's error text on a non-zero status.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CM2_LIB") or os.path.join(_HERE, "csrc", "libcosmomap2_b200.so")

_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_int = ctypes.c_int
_f64 = ctypes.c_double

# name -> (restype, argtypes); mirrors include/cosmomap2_b200.h one to one
SIGNATURES = {
    "cm2_version": (_int, []),
    "cm2_last_error": (ctypes.c_char_p, []),
    "cm2_device_info": (_int, [ctypes.POINTER(_int), ctypes.POINTER(_i64), ctypes.POINTER(_int)]),
    "cm2_launch_count": (_i64, []),
    "cm2_pointing_apply": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _vp, _vp]),
    "cm2_pointing_apply_t": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _vp, _i64, _vp]),
    "cm2_pointing_apply_t_sorted": (_int, [_vp, _vp, _vp, _vp, _int, _vp, _vp, _i64, _vp]),
    "cm2_hits_i64": (_int, [_vp, _i64, _i64, _vp, _vp]),
    "cm2_angles": (_int, [_vp, _i64, _vp, _vp, _vp]),
    "cm2_pix_narrow": (_int, [_vp, _i64, _vp, _vp]),
    "cm2_pix_widen": (_int, [_vp, _i64, _vp, _vp]),
    "cm2_weights_moments": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _i64, _int, _vp, _i64, _vp]),
    "cm2_weights_moments_sorted": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _vp, _int, _vp, _i64, _vp]),
    "cm2_weights_mask": (_int, [_vp, _i64, _int, _f64, _vp, _vp]),
    "cm2_scan_scratch_bytes": (_i64, [_i64]),
    "cm2_weights_old2new": (_int, [_vp, _i64, _vp, _vp, _vp, _vp]),
    "cm2_compact_rows_f64": (_int, [_vp, _vp, _i64, _int, _vp, _vp]),
    "cm2_compact_rows_i64": (_int, [_vp, _vp, _i64, _int, _vp, _vp]),
    "cm2_relabel": (_int, [_vp, _i64, _vp, _vp]),
    "cm2_bd_build": (_int, [_vp, _i64, _int, _vp, _vp]),
    "cm2_bd_apply": (_int, [_vp, _i64, _int, _vp, _vp, _vp]),
    "cm2_bdfwd_apply": (_int, [_vp, _i64, _int, _vp, _vp, _vp]),
    "cm2_noise_white_apply": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _i64, _vp]),
    "cm2_toeplitz_scratch_bytes": (_i64, [_i64]),
    "cm2_noise_toeplitz_apply": (_int, [_vp, _int, _i64, _i64, _vp, _vp, _vp, _i64, _vp, _vp]),
    "cm2_toeplitz_fft_points": (_int, []),
    "cm2_toeplitz_fft_scratch_bytes": (_i64, [_i64]),
    "cm2_noise_toeplitz_fft_apply": (_int, [_vp, _int, _i64, _i64, _vp, _vp, _vp, _i64, _vp, _int, _int, _vp]),
    "cm2_noise_psd_scratch_bytes": (_i64, [_i64]),
    "cm2_noise_psd": (_int, [_vp, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _vp, _int, _vp]),
    "cm2_filter_offset_apply": (_int, [_vp, _vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    "cm2_amatvec_white": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _vp, _i64, _i64, _vp, _vp, _vp, _i64, _i64, _vp]),
    "cm2_pack_pointing": (_int, [_vp, _i64, _vp, _vp, _vp]),
    "cm2_amatvec_white_set_stage": (_int, [_int]),
    "cm2_amatvec_filter": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _vp, _i64, _vp, _vp, _i64, _vp]),
    "cm2_filter_runs_mark": (_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    "cm2_filter_runs_fill": (_int, [_vp, _vp, _vp, _int, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cm2_filter_seg_mean": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _vp, _vp, _vp]),
    "cm2_amatvec_filter_mu": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i64, _i64, _vp]),
    "cm2_filter_poly_gram": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _vp, _vp]),
    "cm2_filter_poly_runs_fill": (_int, [_vp, _vp, _vp, _int, _vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cm2_filter_poly_seg_coef": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _int, _vp, _vp, _vp, _vp]),
    "cm2_amatvec_filter_poly_mu": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _i64, _int, _vp, _vp,
                                          _i64, _int, _i64, _vp]),
    "cm2_pointing_filter_mu": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    "cm2_amatvec_toeplitz_max_band": (_int, []),
    "cm2_amatvec_toeplitz": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _int, _i64, _i64, _vp, _vp, _vp, _i64, _vp]),
    "cm2_filter_poly_max_order": (_int, []),
    "cm2_filter_poly_set_tma": (_int, [_int]),
    "cm2_filter_poly_apply": (_int, [_vp, _vp, _vp, _i64, _i64, _int, _int, _vp, _vp, _i64, _vp]),
    "cm2_amatvec_filter_poly_max_order": (_int, []),
    "cm2_amatvec_filter_poly": (_int, [_vp, _vp, _vp, _i64, _int, _vp, _vp, _i64, _i64, _int, _vp, _vp, _i64, _vp]),
    "cm2_ground_filter_apply": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "cm2_ground_filter_sub": (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "cm2_reorganize_map": (_int, [_vp, _vp, _i64, _int, _i64, _vp, _vp]),
    "cm2_defl_work_doubles": (_i64, [_int]),
    "cm2_defl_zt_apply": (_int, [_vp, _i64, _int, _i64, _vp, _int, _i64, _vp, _vp, _vp]),
    "cm2_defl_z_apply": (_int, [_vp, _i64, _int, _i64, _vp, _f64, _f64, _vp, _vp, _vp]),
    "cm2_coarse_apply": (_int, [_vp, _int, _vp, _vp, _vp]),
    "cm2_m2_apply": (_int, [_vp, _vp, _i64, _int, _i64, _vp, _vp, _i64, _int, _vp, _vp, _vp, _vp]),
    "cm2_m2_banded_apply": (_int, [_vp, _vp, _int, _vp, _vp, _i64, _int, _vp, _vp, _vp, _vp]),
    "cm2_dense_gram_work_doubles": (_i64, []),
    "cm2_dense_gram": (_int, [_vp, _i64, _int, _vp, _i64, _int, _i64, _vp, _i64, _vp, _vp]),
    "cm2_dense_combine": (_int, [_vp, _i64, _i64, _int, _vp, _i64, _int, _vp, _i64, _vp]),
    "cm2_dot": (_int, [_vp, _vp, _i64, _vp, _vp]),
    "cm2_axpby": (_int, [_f64, _vp, _f64, _vp, _i64, _vp]),
    "cm2_pcg_reset": (_int, [_vp, _i64, _vp, _f64, _vp]),
    "cm2_pcg_update_p": (_int, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "cm2_pcg_update_xr": (_int, [_vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "cm2_pcg_bd_reset": (_int, [_vp, _i64, _int, _vp, _vp, _vp, _f64, _f64, _vp, _vp, _vp, _vp]),
    "cm2_pcg_bd_iter": (_int, [_vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cm2_pcg_bd_update_p": (_int, [_vp, _vp, _i64, _vp, _vp]),
    "cm2_pcg_bd_update": (_int, [_vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cm2_allreduce_p2p_signal_bytes": (_i64, []),
    "cm2_allreduce_p2p": (_int, [_vp, _vp, _vp, _int, _int, _i64, ctypes.c_uint32, _vp]),
    "cm2_enable_peer_access": (_int, [_int]),
    "cm2_allreduce_p2p_set_timeout": (_f64, [_f64]),
    "cm2_pcg_bd_iter_refuse": (_int, [_int]),
    "cm2_pcg_bd_iter_max_npix": (_i64, [_int]),
    "cm2_pcg_bd_tail_strided": (_int, [_int]),
    "cm2_pcg_sharded_signal_bytes": (_i64, []),
    "cm2_pcg_sharded_work_doubles": (_i64, []),
    "cm2_pcg_bd_sharded": (_int, [_int, _int, _int, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                  _vp, ctypes.c_uint32, _f64, _f64, _f64, _vp]),
}

# entry points that return a size/count rather than a status
_NOT_STATUS = {"cm2_version", "cm2_last_error", "cm2_launch_count", "cm2_scan_scratch_bytes",
               "cm2_toeplitz_scratch_bytes", "cm2_defl_work_doubles", "cm2_allreduce_p2p_signal_bytes",
               "cm2_toeplitz_fft_points", "cm2_toeplitz_fft_scratch_bytes", "cm2_noise_psd_scratch_bytes",
               "cm2_filter_poly_max_order", "cm2_filter_poly_set_tma",
               "cm2_amatvec_filter_poly_max_order", "cm2_amatvec_toeplitz_max_band",
               "cm2_allreduce_p2p_set_timeout", "cm2_pcg_bd_iter_refuse", "cm2_pcg_bd_iter_max_npix",
               "cm2_pcg_bd_tail_strided",
               "cm2_pcg_sharded_signal_bytes", "cm2_pcg_sharded_work_doubles", "cm2_dense_gram_work_doubles"}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "cosmomap2_b200: %s is missing. Build it with `python cosmomap2_b200/csrc/build.py` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


class Cm2Error(RuntimeError):
    pass


def last_error():
    msg = lib.cm2_last_error()
    return msg.decode() if msg else ""


def call(name, *args):
    """Invoke a status-returning entry point; raise on a non-zero status."""
    rc = getattr(lib, name)(*args)
    if name in _NOT_STATUS:
        return rc
    if rc != 0:
        raise Cm2Error("%s failed (%d): %s" % (name, rc, last_error()))
    return rc


def launch_count():
    return int(lib.cm2_launch_count())

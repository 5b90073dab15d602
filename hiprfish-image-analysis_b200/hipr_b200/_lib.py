"""ctypes binding of libhipr_b200.so (include/hipr_b200.h).  There is no fallback: if the CUDA
library is missing or a call fails, this raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "libhipr_b200.so")

F32, F64, I32, I64, U8 = 0, 1, 2, 3, 4
FLAVOURS = {"F1": 1, "F2": 2, "F3": 3, "ME2": 4, "V3": 5}

_vp, _i, _i64 = C.c_void_p, C.c_int, C.c_int64
_SIGNATURES = {
    "hipr_abi_version": (_i, []),
    "hipr_error_string": (C.c_char_p, [_i]),
    "hipr_launch_count": (_i64, []),
    "hipr_sm_count": (_i, []),
    "hipr_chansum": (_i, [_vp, _vp, _i64, _i, _vp, _i, _vp, _vp]),
    "hipr_chansum_raw": (_i, [_vp, _i, C.c_double, _i64, _i, _vp, _vp, _vp]),
    "hipr_register_stacks": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "hipr_xcorr2d_workspace_bytes": (_i64, [_i, _i, _i]),
    "hipr_register_translation_2d": (_i, [_vp, _vp, _i, _i, _i, _vp, _i64, _vp, _vp, _vp]),
    "hipr_excitation_shifts": (_i, [_vp, _vp, _i, _i, _i, _i, C.c_double, _vp, _i64, _vp, _vp]),
    "hipr_image_range": (_i, [_vp, _i, _i64, _vp, _vp]),
    "hipr_normalize_cast": (_i, [_vp, _i64, _vp, _vp, _vp]),
    "hipr_normalize": (_i, [_vp, _i, _i64, _vp, _vp]),
    "hipr_maxkey_decode": (_i, [_vp, _vp, _vp]),
    "hipr_range_decode": (_i, [_vp, _vp, _vp]),
    "hipr_range_encode": (_i, [_vp, _vp, _vp]),
    "hipr_denoise_nl_means_2d": (_i, [_vp, _i, _i, _i, _i, _i, C.c_double, _vp, _vp]),
    "hipr_denoise_nl_means_3d": (_i, [_vp, _i, _i, _i, _i, _i, _i, C.c_double, _vp, _vp, _i64, _vp]),
    "hipr_denoise_nl_means_3d_workspace": (_i64, [_i, _i, _i, _i]),
    "hipr_line_profile_2d": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "hipr_lne2d": (_i, [_vp, _i, _i, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "hipr_lne2d_q": (_i, [_vp, _i, _i, _i64, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "hipr_neighbor2d": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _i, _vp]),
    "hipr_neighbor2d_fused": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _vp]),
    "hipr_line_profile_3d": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "hipr_lne3d_dirs": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "hipr_lne3d": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp, _vp]),
    "hipr_lne3d_q": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp]),
    "hipr_label_max": (_i, [_vp, _i, _i64, _vp, _vp]),
    "hipr_cell_spectra_accumulate": (_i, [_vp, _vp, _i, _i64, _i64, _i, _i64, _vp, _vp, _vp, _vp]),
    "hipr_cell_spectra_reset": (_i, [_vp, _vp, _i64, _i, _vp]),
    "hipr_cell_spectra_finalize": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hipr_cell_moments": (_i, [_vp, _i, _i, _i, _i64, _vp, _vp]),
    "hipr_cell_geometry_finalize": (_i, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hipr_paint_labels": (_i, [_vp, _i, _i64, _vp, _i, _i64, _i, _vp, _vp]),
    "hipr_label_workspace_bytes": (_i64, [_i, _i, _i, _i]),
    "hipr_label": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i64, _vp, _i, _vp, _vp]),
    "hipr_label_counts": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i64, _vp, _vp, _vp]),
    "hipr_label_clear": (_i, [_vp, _i, _vp, _i64, _vp, _i64, _vp, _vp]),
    "hipr_watershed_workspace_bytes": (_i64, [_i, _i, _i, _i, _i, _i]),
    "hipr_watershed": (_i, [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _i64, _vp, _vp, _vp]),
    "hipr_kmeans1d_workspace_bytes": (_i64, []),
    "hipr_kmeans1d_uniforms": (_i, [_i, _i]),
    "hipr_kmeans1d": (_i, [_vp, _i, _i64, _i, C.c_double, _i, _i, _i, _vp, _i, C.c_double, _vp, _vp, _i, _vp, _vp, _vp]),
    "hipr_mosaic_p2p_bytes": (_i64, [_i, _i, _i]),
    "hipr_p2p_alloc": (_i, [C.POINTER(_vp), _i64]),
    "hipr_p2p_free": (_i, [_vp]),
    "hipr_p2p_get_handle": (_i, [_vp, _vp]),
    "hipr_p2p_open_handle": (_i, [_vp, C.POINTER(_vp)]),
    "hipr_p2p_close_handle": (_i, [_vp]),
    "hipr_mosaic_p2p_rows_ptr": (_i, [_vp, _i, _i, _i, _i, _i, C.POINTER(_vp)]),
    "hipr_mosaic_p2p_exchange": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, C.c_uint64, _vp, _vp, _vp]),
    "hipr_mosaic_p2p_set_timeout_ms": (_i, [C.c_double]),
    "hipr_mosaic_p2p_guard": (_i, [_vp, _vp, _i64, _vp]),
    "hipr_mosaic_p2p_score": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, C.c_uint64, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "hipr_neighbor2d_host": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    "hipr_line_profile_2d_host": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "hipr_lne3d_dirs_host": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "hipr_line_profile_3d_host": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "hipr_neighbor3d_host": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "hipr_neighbor3d_host_denoise": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, C.c_double, _i, _vp]),
    "hipr_neighbor2d_host_denoise": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _i, C.c_double, _vp, _vp]),
    "hipr_neighbor2d_host_batch": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _i, C.c_double, _vp]),
    "hipr_neighbor2d_host_raw": (_i, [_vp, _i, C.c_double, _i, _i, _i, _i, _i, _vp, _i, _vp, _vp]),
    "hipr_cell_spectra_host": (_i, [_vp, _vp, _i, _i64, _i64, _i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hipr_cell_spectra_host_fetch": (_i, [_i64, _vp, _vp, _vp, _vp]),
    "hipr_fov_upload": (_i, [_vp, _i, _i, _i, C.POINTER(_vp)]),
    "hipr_fov_score": (_i, [_vp, _i, _i, _vp, _i, _vp, _vp]),
    "hipr_fov_cell_spectra": (_i, [_vp, _vp, _i, _i64, _vp, _vp, _vp, _vp, _vp]),
    "hipr_fov_device_arrays": (_i, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "hipr_fov_release": (_i, [_vp]),
    "hipr_host_last_elapsed_ms": (C.c_double, []),
    "hipr_host_alloc": (_i, [C.POINTER(_vp), _i64]),
    "hipr_host_free": (_i, [_vp]),
    "hipr_host_release_workspace": (_i, []),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


class HiprError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libhipr_b200.so not found at %s: build it with "
                "`python hiprfish-image-analysis_b200/build.py` (nvcc, sm_100a). "
                "There is no CPU fallback." % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.hipr_abi_version() != 1:
            raise ImportError("libhipr_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(code, what):
    """Maps the ABI's return code to the exception classes the Cython modules raise."""
    if code == 0:
        return
    msg = lib().hipr_error_string(code).decode()
    if code in (-1, -3, -4, -5, -6, -7, -9):
        raise ValueError("%s: %s" % (what, msg))
    if code == -2:
        raise TypeError("%s: %s" % (what, msg))
    raise HiprError("%s: CUDA error %d: %s" % (what, code, msg))

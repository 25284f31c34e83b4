"""ctypes binding of libhydrodem_b200.so (the C ABI declared in include/hydrodem_b200.h).

The product path fails loudly: if the library has not been built, or a call
returns a negative status, a DeviceError / reference exception is raised.
Nothing here falls back to the CPU.
"""
import ctypes
import os

from .exceptions import DeviceError, WindowSizeEvenError, WindowSizeHighError

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhydrodem_b200.so")

# hd_status / hd_dtype / op codes (mirrors of the header enums)
HD_OK, HD_ERR_NULL, HD_ERR_WINDOW_HIGH, HD_ERR_WINDOW_EVEN = 0, -1, -2, -3
HD_ERR_ALIGN, HD_ERR_CUDA, HD_ERR_UNSUPPORTED, HD_ERR_ARG, HD_ERR_WORKSPACE = -4, -5, -6, -7, -8
U8, F32, F64, I64, C64, C128, I32, I16, BOOL = range(9)
OP_COPY, OP_MUL, OP_ADD, OP_RSUB, OP_LT, OP_GT, OP_ABS, OP_RINT, OP_XOR, OP_TRUNC = range(10)
MORPH_ERODE, MORPH_DILATE, MORPH_CLOSE, MORPH_OPEN = range(4)
WARP_NEAREST, WARP_BILINEAR = range(2)
HD_SCATTER_MAX_SEGS = 16

_p, _i, _i64, _d = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double

# name -> (restype, argtypes).  tests/test_abi.py checks this table against the header.
SIGNATURES = {
    "hd_version": (_i, []),
    "hd_status_string": (ctypes.c_char_p, [_i]),
    "hd_last_cuda_error": (_i, []),
    "hd_last_cuda_error_string": (ctypes.c_char_p, []),
    "hd_device_count": (_i, []),
    "hd_launch_count": (_i64, []),
    "hd_reset_launch_count": (None, []),
    "hd_profile_enable": (_i, [_i]),
    "hd_profile_report": (_i64, [ctypes.c_char_p, _i64]),
    "hd_pitch_elems": (_i64, [_i64, _i]),
    "hd_memcpy2d_h2d": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p]),
    "hd_memcpy2d_d2h": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p]),
    "hd_stream_synchronize": (_i, [_p]),
    "hd_host_widen_f32_f64": (_i, [_p, _p, _i64, _i]),
    "hd_host_widen_i16": (_i, [_p, _i, _p, _i64, _i]),
    "hd_host_lzw_decode": (_i64, [_p, _i64, _p, _i64]),
    "hd_host_inflate": (_i64, [_p, _i64, _p, _i64]),
    "hd_host_tiff_lzw": (_i64, [_p, _i64, _p, _i64]),
    "hd_confusion_counts": (_i, [_p, _i, _i64, _p, _i, _i64, _i64, _i64, ctypes.c_double, _p, _p]),
    "hd_pack_i16": (_i, [_p, _i64, _p, _i64, _i64, _p, _p]),
    "hd_elementwise": (_i, [_i, _p, _i, _i64, _p, _i, _i64, _p, _i, _p, _i, _i64, _i64, _i64, _p]),
    "hd_final_terms": (_i, [_p, _i, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _i, _i64, _i64, _i64, _p]),
    "hd_final_mean3": (_i, [_p, _i64, _p, _i64, _p, _i64, _p, _i64, _p, _i64, _i64, _i64, _p]),
    "hd_expand": (_i, [_p, _i, _i64, _p, _i, _i64, _i64, _i64, _i, _p]),
    "hd_expand_select": (_i, [_p, _i, _i64, _p, _i64, _p, _i64, _i64, _i64, _i, _p]),
    "hd_majority": (_i, [_p, _i64, _p, _i, _i64, _i64, _i64, _i, _i, _p]),
    "hd_nanfix": (_i, [_p, _i64, _p, _i64, _i, _i64, _i64, _p]),
    "hd_isolated": (_i, [_p, _i64, _p, _i64, _i, _i64, _i64, _p]),
    "hd_route_rivers": (_i, [_p, _i64, _p, _i64, _p, _i64, _i64, _i64, _i, _p, _i64, _p]),
    "hd_quadratic": (_i, [_p, _i64, _p, _i64, _i, _i64, _i64, _i, _p]),
    "hd_groves_correction": (_i, [_p, _i, _i64, _p, _i64, _p, _i, _i64, _i64, _i64, _i, _d, _p]),
    "hd_groves_tile_count": (_i64, [_i64, _i64]),
    "hd_groves_correction_tiles": (_i, [_p, _i64, _p, _i64, _p, _i64, _i64, _i64, _i, _d, _p, _i, _p]),
    "hd_median": (_i, [_p, _i64, _p, _i64, _i64, _i64, _i, _i, _p]),
    "hd_hollow_mean_detect": (_i, [_p, _i64, _p, _i64, _p, _i, _i64, _p, _i64, _i64, _i64, _i, _i, _d, _p]),
    "hd_hollow_tile_count": (_i64, [_i64, _i64]),
    "hd_hollow_mean_detect_tiles": (_i, [_p, _i64, _p, _i64, _p, _i, _i64, _p, _i64, _i64, _i64, _i, _i, _d, _p, _p, _p]),
    "hd_fourier_mask_assemble": (_i, [_p, _i64, _p, _i64, _p, _i, _i64, _i64, _i64, _i, _i, _p]),
    "hd_fft2_plan_create": (_i, [_i64, _i64, ctypes.POINTER(_p)]),
    "hd_fft2_plan_destroy": (_i, [_p]),
    "hd_fft_plan_info": (_i, [_p, _i, ctypes.POINTER(_i64)]),
    "hd_fft2_workspace_bytes": (_i64, [_i64, _i64]),
    "hd_fft2_forward_shift_abs": (_i, [_p, _p, _i64, _p, _i64, _p, _i64, _p, _i64, _p]),
    "hd_fft2_masked_inverse_abs": (_i, [_p, _p, _i64, _p, _i64, _p, _i, _i64, _p, _i64, _p]),
    "hd_fft2_c2c": (_i, [_p, _p, _i, _i64, _p, _i64, _i, _p, _i64, _p]),
    "hd_fft_rows": (_i, [_p, _p, _i, _i64, _p, _i64, _i64, _i, _i, _p, _i64, _p]),
    "hd_fft_band_workspace_bytes": (_i64, [_i64, _i64]),
    "hd_fft_band_pass": (_i, [_p, _i, _i, _p, _i64, _i64, _p, _i64, _i, _i, _i, _p, _i64, _i64, _p, _i64, _p]),
    "hd_fft_band_pass_scatter": (_i, [_p, _i, _i, _p, _i64, _i64, _p, _i64, _i, _i, _i, _p, _i64, _p, _i64, _p]),
    "hd_ipc_export": (_i, [_p, _p, ctypes.POINTER(_i64)]),
    "hd_ipc_import": (_i, [_p, ctypes.POINTER(_p)]),
    "hd_ipc_close": (_i, [_p]),
    "hd_klayout_rows": (_i64, [_i64, _i64, _i64]),
    "hd_klayout_ky": (_i64, [_i64, _i64, _i64, _i64]),
    "hd_hermitian_complete": (_i, [_p, _i64, _p, _i64, _p, _i64, _i64, _i64, _i64, _i64, _p]),
    "hd_conj_mirror_fill": (_i, [_p, _i64, _i64, _i64, _p]),
    "hd_fourier_mask_assemble_rows": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p, _i64, _i64, _i64, _i64, _i64, _i64, _i, _p]),
    "hd_fftshift2": (_i, [_p, _i64, _p, _i64, _i, _i64, _i64, _i, _p]),
    "hd_pdfill_workspace_bytes": (_i64, [_i64, _i64]),
    "hd_pdfill": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p, _i64, ctypes.POINTER(_i), _p]),
    "hd_pdfill_band": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p, _i64, _i, ctypes.POINTER(_i), _p]),
    "hd_pdfill_d8": (_i, [_p, _i64, _p, _i64, _p, _i64, _i64, _i64, _p, _i64, ctypes.POINTER(_i), _p]),
    "hd_pdfill_finish_d8": (_i, [_p, _i64, _p, _i64, _p, _i64, _i64, _i64, _p, _p]),
    "hd_pdfill_status": (_i, [_p, ctypes.POINTER(_i), _p]),
    "hd_halo_min_flag": (_i, [_p, _p, _i64, _p, _p]),
    "hd_fill_pool_band": (_i, [_p, _i64, _i64, _i64, _p, _p, _i64, _i, _p, _p]),
    "hd_pdfill_coarse": (_i, [_p, _p, _i64, _i64, _i64, _p, _i64, _p]),
    "hd_pdfill_band_start": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p, _i64, _i, _p, _i64, _i64, _p]),
    "hd_d8": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p]),
    "hd_binary_morph": (_i, [_p, _i, _i64, _p, _i64, _i64, _i64, _i, _i, _i, _p]),
    "hd_max_filter": (_i, [_p, _i64, _p, _i64, _i, _i64, _i64, _i, _p]),
    "hd_tidy_lagoons": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p]),
    "hd_convolve3": (_i, [_p, _i64, _p, _i64, _i, _i64, _i64, ctypes.POINTER(_d), _d, _i, _p, _i64, _p]),
    "hd_correlate": (_i, [_p, _i64, _p, _i64, _i, _i64, _i64, _i, ctypes.POINTER(_i), ctypes.POINTER(_i),
                          ctypes.POINTER(_d), _d, _p]),
    "hd_binary_morph_struct": (_i, [_p, _i, _i64, _p, _i64, _i64, _i64, _i, _i, ctypes.POINTER(_i), ctypes.POINTER(_i),
                                    _i, _p, _p]),
    "hd_max_filter_rect": (_i, [_p, _i64, _p, _i64, _i, _i64, _i64, _i, _i, _p, _i64, _p]),
    "hd_warp": (_i, [_p, _i, _i64, _i64, _i64, ctypes.POINTER(_d), _i, _d, _p, _i64, _i64, _i64, ctypes.POINTER(_d), _i64,
                     ctypes.POINTER(_d), _i, _p]),
    "hd_warp_mosaic": (_i, [_p, _i64, _p, _p, ctypes.POINTER(_i64), _i, ctypes.POINTER(_d), _i, _d, _p, _i64, _i64, _i64,
                            ctypes.POINTER(_d), _i64, ctypes.POINTER(_d), _i, _p]),
    "hd_host_tm_inverse": (_i, [ctypes.POINTER(_d), _p, _p, _i64, _p, _p]),
    "hd_host_tm_forward": (_i, [ctypes.POINTER(_d), _p, _p, _i64, _p, _p]),
    "hd_rasterize_workspace_bytes": (_i64, [_i64]),
    "hd_rasterize_lines": (_i, [_p, _p, _i64, _p, _p, _i64, _p, _i64, _p, _i64, _i64, _i64, ctypes.POINTER(_d), _i64,
                                ctypes.POINTER(_d), _p, _i64, _p]),
    "hd_tiff_decode_workspace_bytes": (_i64, [_i64, _i64, _i64, _i]),
    "hd_tiff_decode": (_i, [_p, _i64, _p, _i64, _i, _i, _i, _i, _p, _i64, _i64, _i64, _i64, _i64, _p, _p, _i64, _p]),
}



class ScatterSeg(ctypes.Structure):
    _fields_ = [("row0", _i64), ("row1", _i64), ("base", _p), ("pitch", _i64), ("dst_row0", _i64)]


class Scatter(ctypes.Structure):
    """hd_scatter of include/hydrodem_b200.h."""
    _fields_ = [("nseg", ctypes.c_int32), ("ncolseg", ctypes.c_int32), ("seg", ScatterSeg * HD_SCATTER_MAX_SEGS),
                ("col_local0", _i64 * 2), ("col_dst0", _i64 * 2), ("col_len", _i64 * 2)]


_lib = None


def load():
    """Load the shared library (once).  Raises DeviceError if it was never built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DeviceError(f"{LIB_PATH} is missing: run `python -m hydrodem_b200.build` "
                              "(there is no CPU fallback for the conditioning path)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(status, *, window_size=None, shape=None):
    """Map a negative hd_status to the reference's exception classes."""
    if status == HD_OK:
        return
    lib = load()
    if status == HD_ERR_WINDOW_HIGH:
        raise WindowSizeHighError(window_size, shape)
    if status == HD_ERR_WINDOW_EVEN:
        raise WindowSizeEvenError(window_size)
    msg = lib.hd_status_string(status).decode()
    if status == HD_ERR_CUDA:
        msg += f": {lib.hd_last_cuda_error_string().decode()} ({lib.hd_last_cuda_error()})"
    raise DeviceError(f"libhydrodem_b200: {msg}")

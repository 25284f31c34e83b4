"""CPU: the C-ABI library builds, loads, exports every symbol the header declares, and fails loudly
(no CPU fallback) when no GPU is present."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from hydrodem_b200 import _lib
from hydrodem_b200.exceptions import DeviceError

from conftest import REPO

HEADER = os.path.join(REPO, "include", "hydrodem_b200.h")


def declared():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for m in re.finditer(r"\b(?:int64_t|int|void|const char\*)\s+(hd_\w+)\s*\(([^;]*?)\)\s*;", src, flags=re.S):
        args = m.group(2).strip()
        out[m.group(1)] = 0 if args in ("", "void") else len(args.split(","))
    return out


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        from hydrodem_b200.build import build
        build()
    return _lib.load()


def test_header_symbols_exported(lib):
    decl = declared()
    assert len(decl) >= 15
    for name, nargs in decl.items():
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
        assert name in _lib.SIGNATURES, f"{name} has no ctypes signature"
        assert len(_lib.SIGNATURES[name][1]) == nargs, f"{name}: header has {nargs} args"
    assert set(_lib.SIGNATURES) <= set(decl), set(_lib.SIGNATURES) - set(decl)


def test_runtime_helpers(lib):
    assert lib.hd_version() >= 100
    assert lib.hd_status_string(_lib.HD_ERR_WINDOW_EVEN) == b"window size is even"
    assert lib.hd_pitch_elems(3601, _lib.F32) == 3616 and lib.hd_pitch_elems(3601, _lib.F64) == 3616
    assert lib.hd_pitch_elems(3601, _lib.U8) == 3712


def test_argument_errors_need_no_gpu(lib):
    p = ctypes.c_void_p(1 << 20)
    assert lib.hd_expand(None, _lib.F32, 64, p, _lib.U8, 64, 64, 64, 7, None) == _lib.HD_ERR_NULL
    assert lib.hd_expand(p, _lib.F32, 64, p, _lib.U8, 64, 64, 64, 6, None) == _lib.HD_ERR_WINDOW_EVEN
    assert lib.hd_expand(p, _lib.F32, 64, p, _lib.U8, 64, 5, 64, 6, None) == _lib.HD_ERR_WINDOW_HIGH   # high before even
    assert lib.hd_majority(p, 64, p, _lib.F64, 64, 64, 64, 11, 40, None) == _lib.HD_ERR_UNSUPPORTED
    with pytest.raises(DeviceError):
        _lib.check(_lib.HD_ERR_ARG)


def test_fill_argument_errors_need_no_gpu(lib):
    """The fill family rejects bad arguments before it touches the device."""
    p = ctypes.c_void_p(1 << 20)
    need = lib.hd_pdfill_workspace_bytes(300, 400)
    assert lib.hd_pdfill(None, 400, p, 400, 300, 400, p, need, None, None) == _lib.HD_ERR_NULL
    assert lib.hd_pdfill(p, 400, p, 400, 300, 400, None, need, None, None) == _lib.HD_ERR_NULL
    assert lib.hd_pdfill(p, 399, p, 400, 300, 400, p, need, None, None) == _lib.HD_ERR_ARG
    assert lib.hd_pdfill(p, 400, p, 400, 0, 400, p, need, None, None) == _lib.HD_ERR_ARG
    assert lib.hd_pdfill(p, 400, p, 400, 300, 400, p, need - 1, None, None) == _lib.HD_ERR_WORKSPACE
    # a later round continues after a halo exchange; the first round is hd_pdfill_band_start
    for flags in (1, 3, 7, 8):
        assert lib.hd_pdfill_band(p, 400, p, 400, 300, 400, p, need, flags, None, None) == _lib.HD_ERR_ARG
    assert lib.hd_pdfill_band(p, 400, p, 400, 300, 400, p, need - 1, 6, None, None) == _lib.HD_ERR_WORKSPACE
    assert lib.hd_pdfill_band_start(p, 400, p, 400, 300, 400, p, need, 1, p, 64, 0, None) == _lib.HD_ERR_ARG
    assert lib.hd_fill_pool_band(p, 400, 300, 400, p, p, 64, 1, p, None) == _lib.HD_ERR_ARG
    assert lib.hd_pdfill_d8(p, 400, p, 400, p, 400, 300, 400, p, need - 1, None, None) == _lib.HD_ERR_WORKSPACE


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback(lib):
    """Without a device the product path must raise, never compute on the host."""
    from hydrodem_b200.filters.custom_filters import ExpandFilter
    assert lib.hd_device_count() == 0
    with pytest.raises(DeviceError):
        ExpandFilter(window_size=3).apply(np.zeros((8, 8), dtype=np.float32))
    p = ctypes.c_void_p(1 << 20)
    assert lib.hd_expand(p, _lib.F32, 64, p, _lib.U8, 64, 64, 64, 7, None) == _lib.HD_ERR_CUDA


def test_host_widen_helpers_are_exact():
    """hd_host_widen_*: HOST functions of the C ABI (no device needed): int16 / float32 results widened to the
    reference dtypes on several threads, any alignment, every value exact."""
    import ctypes
    import numpy as np
    from hydrodem_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(5)
    n = 200_003
    src16 = rng.integers(-32768, 32768, n + 9).astype(np.int16)
    src32 = rng.standard_normal(n + 9).astype(np.float32) * 1e3
    for off in (0, 1, 3):
        for threads in (1, 5):
            for dt, code in ((np.float32, _lib.F32), (np.float64, _lib.F64)):
                dst = np.full(n + 8, -7, dtype=dt)
                rc = lib.hd_host_widen_i16(ctypes.c_void_p(dst.ctypes.data + dst.itemsize * off), code,
                                           ctypes.c_void_p(src16.ctypes.data + 2 * off), n, threads)
                assert rc == 0
                np.testing.assert_array_equal(dst[off:off + n], src16[off:off + n].astype(dt))
                assert (dst[:off] == -7).all() and (dst[off + n:] == -7).all()
            dst = np.full(n + 8, -7.0)
            rc = lib.hd_host_widen_f32_f64(ctypes.c_void_p(dst.ctypes.data + 8 * off),
                                           ctypes.c_void_p(src32.ctypes.data + 4 * off), n, threads)
            assert rc == 0
            np.testing.assert_array_equal(dst[off:off + n], src32[off:off + n].astype(np.float64))
            assert (dst[:off] == -7).all() and (dst[off + n:] == -7).all()
    assert lib.hd_host_widen_i16(None, _lib.F32, None, 4, 1) != 0

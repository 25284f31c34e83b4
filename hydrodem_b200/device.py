"""Device rasters: pitched HBM buffers behind the filter API.

PyTorch is used for plumbing only -- device memory (its caching allocator),
the current CUDA stream and pinned host buffers.  Every computation goes
through the C ABI (``_lib``) on raw device pointers.

Layout: a raster of (ny, nx) cells is a row-major ``(ny, pitch)`` buffer whose
pitch is rounded up so that each row starts on a 128-byte boundary
(``hd_pitch_elems``) -- the TMA tile loads need 16-byte aligned rows, and
128 bytes keeps every row on a fresh cache line.  A raster remembers
``ref_dtype``: the NumPy dtype the reference would hold at this point of the
chain (e.g. Expand stores 0/1 as uint8 on the device but the reference
returns float64); the conversion happens once, on the device, at download.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from .exceptions import DeviceError, NumpyArrayExpectedError

_NP2HD = {np.dtype(np.uint8): _lib.U8, np.dtype(np.bool_): _lib.U8, np.dtype(np.float32): _lib.F32,
          np.dtype(np.float64): _lib.F64, np.dtype(np.int64): _lib.I64, np.dtype(np.int32): _lib.I32,
          np.dtype(np.complex64): _lib.C64, np.dtype(np.complex128): _lib.C128, np.dtype(np.int16): _lib.I16}
_HD2TORCH = {_lib.U8: torch.uint8, _lib.F32: torch.float32, _lib.F64: torch.float64, _lib.I64: torch.int64,
             _lib.I32: torch.int32, _lib.C64: torch.complex64, _lib.C128: torch.complex128, _lib.I16: torch.int16}
_HD2NP = {_lib.U8: np.dtype(np.uint8), _lib.F32: np.dtype(np.float32), _lib.F64: np.dtype(np.float64),
          _lib.I64: np.dtype(np.int64), _lib.I32: np.dtype(np.int32), _lib.C64: np.dtype(np.complex64),
          _lib.C128: np.dtype(np.complex128), _lib.I16: np.dtype(np.int16)}


def hd_dtype_of(np_dtype):
    try:
        return _NP2HD[np.dtype(np_dtype)]
    except KeyError:
        raise DeviceError(f"dtype {np_dtype} is not supported on the device path") from None


def require_cuda():
    if not torch.cuda.is_available():
        raise DeviceError("no CUDA device visible: the conditioning path has no CPU fallback")
    _lib.load()


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def device():
    return torch.device("cuda", torch.cuda.current_device())


class DeviceRaster:
    """A pitched 2-D raster in HBM."""

    __slots__ = ("buf", "ny", "nx", "dtype", "ref_dtype", "_y0", "_x0")

    def __init__(self, buf, ny, nx, dtype, ref_dtype=None, y0=0, x0=0):
        self.buf, self.ny, self.nx, self.dtype = buf, int(ny), int(nx), dtype
        self.ref_dtype = np.dtype(ref_dtype) if ref_dtype is not None else _HD2NP[dtype]
        self._y0, self._x0 = y0, x0

    @property
    def pitch(self):
        return self.buf.shape[1]

    @property
    def itemsize(self):
        return _HD2NP[self.dtype].itemsize

    @property
    def ptr(self):
        return ctypes.c_void_p(self.buf.data_ptr() + (self._y0 * self.pitch + self._x0) * self.itemsize)

    @property
    def shape(self):
        return (self.ny, self.nx)

    def sub(self, y0, y1, x0, x1):
        """A view of rows y0:y1, columns x0:x1 (same buffer, same pitch)."""
        return DeviceRaster(self.buf, y1 - y0, x1 - x0, self.dtype, self.ref_dtype, self._y0 + y0, self._x0 + x0)

    def with_ref(self, ref_dtype):
        return DeviceRaster(self.buf, self.ny, self.nx, self.dtype, ref_dtype, self._y0, self._x0)

    def tensor(self):
        """torch view (ny, nx) of the valid cells (plumbing / debugging only)."""
        return self.buf[self._y0:self._y0 + self.ny, self._x0:self._x0 + self.nx]


def empty(ny, nx, dtype, ref_dtype=None):
    require_cuda()
    pitch = _lib.load().hd_pitch_elems(nx, dtype)
    buf = torch.empty((ny, pitch), dtype=_HD2TORCH[dtype], device=device())
    return DeviceRaster(buf, ny, nx, dtype, ref_dtype)


def zeros(ny, nx, dtype, ref_dtype=None):
    r = empty(ny, nx, dtype, ref_dtype)
    r.buf.zero_()
    return r


def upload(array, ref_dtype=None):
    """Host ndarray -> device raster of the same dtype (bool travels as uint8)."""
    if not isinstance(array, np.ndarray):
        raise NumpyArrayExpectedError(array)
    if array.ndim != 2:
        raise DeviceError(f"expected a 2-D raster, got shape {array.shape}")
    require_cuda()
    host = np.ascontiguousarray(array)
    dt = hd_dtype_of(host.dtype)
    ny, nx = host.shape
    r = empty(ny, nx, dt, ref_dtype if ref_dtype is not None else array.dtype)
    es = host.dtype.itemsize
    if ny and nx:
        _lib.check(_lib.load().hd_memcpy2d_h2d(r.ptr, r.pitch * es, ctypes.c_void_p(host.ctypes.data), nx * es, nx * es,
                                               ny, stream_ptr()))
        if not _is_pinned(host):
            # a pageable source may be released by the caller as soon as we return
            _lib.check(_lib.load().hd_stream_synchronize(stream_ptr()))
    return r


def _is_pinned(host):
    try:
        return torch.from_numpy(host).is_pinned()
    except Exception:      # noqa: BLE001  (read-only arrays, exotic dtypes)
        return False


def convert(src, dtype, ref_dtype=None):
    """Device-side dtype conversion (HD_OP_COPY) with the semantics of ``astype`` (to bool: ``!= 0``)."""
    to_bool = ref_dtype is not None and np.dtype(ref_dtype) == np.bool_ and src.ref_dtype != np.bool_
    if src.dtype == dtype and not to_bool:
        return src if ref_dtype is None else src.with_ref(ref_dtype)
    dst = empty(src.ny, src.nx, dtype, ref_dtype if ref_dtype is not None else src.ref_dtype)
    elementwise(_lib.OP_COPY, src, None, dst)
    return dst


def _tag(raster):
    """hd_dtype of a raster's storage, HD_BOOL for a byte raster that holds a bool reference."""
    return _lib.BOOL if raster.dtype == _lib.U8 and raster.ref_dtype == np.bool_ else raster.dtype


def elementwise(op, a, b, out, compute=None, scalar=None):
    """out = op(a, b) in ``compute``, the NumPy dtype of the ufunc loop (default: a's storage dtype).  Without a
    raster ``b``, ``scalar`` is the second operand: a Python scalar, NumPy scalar or 0-d array, cast to ``compute``
    as NumPy casts an operand into the loop."""
    lib = _lib.load()
    cdt = np.dtype(compute) if compute is not None else _HD2NP[a.dtype]
    ctag = _lib.BOOL if cdt == np.bool_ else hd_dtype_of(cdt)
    bp, bd, bpitch = (b.ptr, _tag(b), b.pitch) if b is not None else (None, 0, 0)
    host = None
    if b is None and scalar is not None:
        with np.errstate(all="ignore"):
            host = np.asarray(scalar, dtype=cdt) if isinstance(scalar, (bool, int, float, complex)) \
                else np.asarray(scalar).astype(cdt)
    sp = ctypes.c_void_p(host.ctypes.data) if host is not None else None
    _lib.check(lib.hd_elementwise(op, a.ptr, _tag(a), a.pitch, bp, bd, bpitch, sp, ctag, out.ptr, _tag(out), out.pitch,
                                  a.ny, a.nx, stream_ptr()))
    return out


def pinned_empty(shape, np_dtype):
    """Pinned host array from torch's caching host allocator (returned to the cache when dropped)."""
    dt = np.dtype(np_dtype)
    tdt = torch.uint8 if dt == np.bool_ else torch.from_numpy(np.empty(0, dtype=dt)).dtype
    a = torch.empty(shape, dtype=tdt, pin_memory=True).numpy()
    return a.view(np.bool_) if dt == np.bool_ else a


def download(raster, out=None):
    """Device raster -> host ndarray in the raster's ``ref_dtype``.

    The conversion to ``ref_dtype`` runs on the device; the copy lands in a
    pinned buffer (or straight in ``out`` when given: the in-place filters of
    the reference return the caller's own array)."""
    lib = _lib.load()
    ref = raster.ref_dtype
    dev = convert(raster, hd_dtype_of(ref))
    if out is not None and out.flags.c_contiguous and out.dtype == ref and out.shape == dev.shape:
        host = out
    else:
        host = pinned_empty(dev.shape, ref)
    es = ref.itemsize
    if dev.ny and dev.nx:
        _lib.check(lib.hd_memcpy2d_d2h(ctypes.c_void_p(host.ctypes.data), dev.nx * es, dev.ptr, dev.pitch * es,
                                       dev.nx * es, dev.ny, stream_ptr()))
        _lib.check(lib.hd_stream_synchronize(stream_ptr()))
    if out is not None and host is not out:
        np.copyto(out, host, casting="unsafe")
        return out
    return host


def upload_async(array, stream):
    """Pinned host ndarray -> device raster on ``stream`` (a torch.cuda.Stream); no host synchronisation.
    Returns (raster, event).  The caller keeps ``array`` alive until the event has completed."""
    if not isinstance(array, np.ndarray):
        raise NumpyArrayExpectedError(array)
    require_cuda()
    host = np.ascontiguousarray(array)
    dt = hd_dtype_of(host.dtype)
    ny, nx = host.shape
    r = empty(ny, nx, dt, array.dtype)
    es = host.dtype.itemsize
    _lib.check(_lib.load().hd_memcpy2d_h2d(r.ptr, r.pitch * es, ctypes.c_void_p(host.ctypes.data), nx * es, nx * es, ny,
                                           ctypes.c_void_p(stream.cuda_stream)))
    ev = torch.cuda.Event()
    ev.record(stream)
    return r, ev


def upload_into(raster, array, stream):
    """Pinned host ndarray -> an existing device raster of the same shape / dtype, on ``stream``; returns the event."""
    if array.shape != raster.shape or hd_dtype_of(array.dtype) != raster.dtype:
        raise DeviceError("upload_into: shape / dtype mismatch")
    es = array.dtype.itemsize
    ny, nx = array.shape
    _lib.check(_lib.load().hd_memcpy2d_h2d(raster.ptr, raster.pitch * es, ctypes.c_void_p(array.ctypes.data), nx * es,
                                           nx * es, ny, ctypes.c_void_p(stream.cuda_stream)))
    ev = torch.cuda.Event()
    ev.record(stream)
    return ev


def download_async(raster, stream, record=True):
    """Device raster (already in its reference dtype) -> pinned host array on ``stream``; returns (array, event)."""
    ref = raster.ref_dtype
    if hd_dtype_of(ref) != raster.dtype:
        raise DeviceError("download_async needs a raster stored in its reference dtype")
    host = pinned_empty(raster.shape, ref)
    es = ref.itemsize
    _lib.check(_lib.load().hd_memcpy2d_d2h(ctypes.c_void_p(host.ctypes.data), raster.nx * es, raster.ptr, raster.pitch * es,
                                           raster.nx * es, raster.ny, ctypes.c_void_p(stream.cuda_stream)))
    if record:
        raster.buf.record_stream(stream)
    ev = torch.cuda.Event()
    ev.record(stream)
    return host, ev


# ---- FFT plans and scratch --------------------------------------------------------------------------
_FFT_PLANS = {}


def fft_plan(ny, nx):
    """Cached hd_fft2 plan (twiddle / chirp tables in device memory) for one raster shape."""
    key = (torch.cuda.current_device(), int(ny), int(nx))
    plan = _FFT_PLANS.get(key)
    if plan is None:
        handle = ctypes.c_void_p()
        _lib.check(_lib.load().hd_fft2_plan_create(ny, nx, ctypes.byref(handle)))
        plan = _FFT_PLANS[key] = handle
    return plan


def scratch(nbytes):
    """Uninitialised device scratch of at least ``nbytes`` (256-byte aligned by the caching allocator)."""
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device())

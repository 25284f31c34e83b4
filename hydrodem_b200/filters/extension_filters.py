"""Wrapped numpy / scipy filters (reference: ``filters/extension_filters.py``),
re-implemented as CUDA kernels behind the same class names.

The reference delegates these to ``numpy``, ``scipy.ndimage`` and
``scipy.fftpack``; here they are launches of libhydrodem_b200 (see
include/hydrodem_b200.h for the contract of each entry point).
"""
import copy
import ctypes
import operator

import numpy as np

from . import DeviceFilter, Filter
from .. import _lib, device as dev
from ..exceptions import DeviceError
from .simple_filters import binary_op


class BitwiseXOR(DeviceFilter):
    """``np.bitwise_xor(operand, image)`` (extension_filters.py:12-60)."""

    def __init__(self, *, operand):
        self.operand = operand if isinstance(operand, dev.DeviceRaster) else copy.deepcopy(operand)

    def run_device(self, raster):
        return binary_op(_lib.OP_XOR, raster, self.operand, np.bitwise_xor)


class AbsoluteValues(DeviceFilter):
    """``np.abs(image)`` (extension_filters.py:63-95); complex -> real."""

    def run_device(self, raster):
        ref = np.abs(np.zeros(0, dtype=raster.ref_dtype)).dtype
        if np.dtype(raster.ref_dtype).kind == "c" and raster.dtype not in (_lib.C64, _lib.C128):
            raise DeviceError("complex raster stored as a real dtype")
        out = dev.empty(raster.ny, raster.nx, dev.hd_dtype_of(ref), ref)
        return dev.elementwise(_lib.OP_ABS, raster, None, out, raster.ref_dtype)


class Around(DeviceFilter):
    """``np.around(image)`` -- round half to even, both parts of a complex (extension_filters.py:98-130)."""

    def run_device(self, raster):
        ref = np.around(np.zeros(0, dtype=raster.ref_dtype)).dtype
        out = dev.empty(raster.ny, raster.nx, dev.hd_dtype_of(ref), ref)
        return dev.elementwise(_lib.OP_RINT, raster, None, out, raster.ref_dtype)


# ---- general footprints: host-side plans --------------------------------------------------------------------------
# scipy.ndimage puts the centre of an axis of length k at k // 2 + origin, so footprint index j sits at offset
# j - (k // 2 + origin) from the output cell.  A convolution, a binary dilation and grey_dilation reverse the footprint
# and turn origin 0 into -1 on an axis of even length (scipy's _correlate_or_convolve, binary_dilation, grey_dilation).
MAX_FOOTPRINT = 31          # Convolve weights and BinaryClosing structures, per axis
MAX_GREY_SIZE = 255         # GreyDilation size, per axis
DBL_EPSILON = np.finfo(np.float64).eps
MORPH_STEPS_PER_LAUNCH = 8  # hd_binary_morph's cap for erosions with the cross
STABLE_STEPS_PER_LAUNCH = 15  # cross erosions per hd_binary_morph_struct launch when iterating until stable
STABLE_LAUNCHES_PER_READ = 8  # launches between two host reads of their changed flags
_CROSS = np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]], dtype=bool)


def _centre(k, reversed_):
    return k // 2 + (-1 if reversed_ and k % 2 == 0 else 0)


def _offsets(mask, reversed_):
    """(dy, dx) of the True cells of a 2-D footprint, row-major; `reversed_` flips it with the even-axis origin shift."""
    if reversed_:
        mask = mask[::-1, ::-1]
    cy, cx = _centre(mask.shape[0], reversed_), _centre(mask.shape[1], reversed_)
    iy, ix = np.nonzero(mask)                                           # row-major
    return (iy - cy).astype(np.int32), (ix - cx).astype(np.int32)


def _footprint_2d(a, what):
    if a.ndim != 2:
        raise DeviceError(f"{what} must be 2-D like the raster (got shape {a.shape})")
    if a.size == 0:
        raise DeviceError(f"{what} must not be empty (got shape {a.shape})")
    if max(a.shape) > MAX_FOOTPRINT:
        raise DeviceError(f"{what}: at most {MAX_FOOTPRINT}x{MAX_FOOTPRINT} on the device (got {a.shape})")


def convolve_taps(weights):
    """NI_Correlate's footprint of scipy.ndimage.convolve(image, weights) as (dy, dx, w) in summation order: the flipped
    weights, origin -1 on even axes, entries with |w| <= DBL_EPSILON left out (a NaN weight too: its |w| > eps is false)."""
    w = np.asarray(weights, dtype=np.float64)
    _footprint_2d(w, "Convolve weights")
    with np.errstate(invalid="ignore"):
        keep = np.abs(w) > DBL_EPSILON
    dy, dx = _offsets(keep, reversed_=True)
    return dy, dx, w[::-1, ::-1][keep[::-1, ::-1]]


def closing_taps(structure):
    """binary_closing(structure): (dilation taps, erosion taps), each (dy, dx).  None = the cross."""
    s = _CROSS if structure is None else np.asarray(structure)
    _footprint_2d(s, "BinaryClosing structure")
    s = s.astype(bool)                                                  # non-zero (NaN included) is True
    return _offsets(s, reversed_=True), _offsets(s, reversed_=False)


def grey_sizes(size):
    """(a, b) of grey_dilation(size=...): an int for both axes or a pair, each 1 ... MAX_GREY_SIZE."""
    pair = (size, size) if np.ndim(size) == 0 else tuple(np.asarray(size).ravel())
    if np.ndim(size) > 1 or len(pair) != 2:
        raise DeviceError(f"GreyDilation: size must be an int or a pair (got {size!r})")
    try:
        pair = tuple(operator.index(s) for s in pair)
    except TypeError:
        raise DeviceError(f"GreyDilation: sizes must be integers (got {size!r})") from None
    for s in pair:
        if s < 1:
            raise DeviceError(f"GreyDilation: sizes must be >= 1 (got {size!r})")
        if s > MAX_GREY_SIZE:
            raise DeviceError(f"GreyDilation: sizes up to {MAX_GREY_SIZE} on the device (got {size!r})")
    return pair


def _int_array(v):
    v = np.ascontiguousarray(v, dtype=np.int32)
    return v, v.ctypes.data_as(ctypes.POINTER(ctypes.c_int))


class _CheckedFilter(DeviceFilter):
    """A filter whose arguments are validated on the host (``plan``) before the raster goes to the device."""

    def plan(self, shape):
        raise NotImplementedError

    def apply(self, image_to_filter):
        Filter.apply(self, image_to_filter)
        self.plan(np.shape(image_to_filter))
        return DeviceFilter.apply(self, image_to_filter)


class Convolve(_CheckedFilter):
    """``scipy.ndimage.convolve(image, weights) / weights.size`` with the default
    mode='reflect' (extension_filters.py:133-184).  3x3 weights (the pipeline's ones((3, 3))) run on
    hd_convolve3; any other 2-D weights up to 31x31 on hd_correlate."""

    def __init__(self, weights=np.ones((3, 3))):
        self.weights = weights

    def plan(self, shape):
        """("conv3", None) or ("correlate", (dy, dx, w))."""
        w = np.asarray(self.weights, dtype=np.float64)
        if w.shape == (3, 3):
            return "conv3", None
        return "correlate", convolve_taps(w)

    def run_device(self, raster, do_round=False, copy32=None):
        """``copy32``: optional F32 device raster that receives a float32 copy of the result (chain plumbing)."""
        path, taps = self.plan(raster.shape)
        w = np.asarray(self.weights, dtype=np.float64)
        ref = np.dtype(raster.ref_dtype)
        work = np.float32 if ref == np.float32 else np.float64       # ndimage keeps float dtypes, else float64
        if path == "correlate" and (do_round or copy32 is not None):
            raise DeviceError("Convolve: rounding and the float32 copy are only fused into the 3x3 path")
        src = dev.convert(raster, dev.hd_dtype_of(work))
        out = dev.empty(raster.ny, raster.nx, src.dtype, work)
        if path == "correlate":
            dy, dx, tw = taps
            (dy, pdy), (dx, pdx) = _int_array(dy), _int_array(dx)
            tw = np.ascontiguousarray(tw, dtype=np.float64)
            _lib.check(_lib.load().hd_correlate(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, src.ny, src.nx, len(tw),
                                                pdy, pdx, tw.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                                float(w.size), dev.stream_ptr()))
            return out
        corr = np.ascontiguousarray(w[::-1, ::-1])                    # convolution = correlation with the flipped kernel
        cw = (ctypes.c_double * 9)(*corr.ravel())
        _lib.check(_lib.load().hd_convolve3(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, src.ny, src.nx, cw,
                                            float(w.size), int(do_round), copy32.ptr if copy32 is not None else None,
                                            copy32.pitch if copy32 is not None else 0, dev.stream_ptr()))
        return out


class BinaryErosion(_CheckedFilter):
    """``scipy.ndimage.binary_erosion(image, iterations=n)`` (extension_filters.py:187-235):
    cross structuring element, border_value 0, bool result.  n >= 1 is n erosions (hd_binary_morph, up to 8 per
    launch); n < 1 repeats until the result stops changing, as scipy does."""

    def __init__(self, *, iterations):
        self.iterations = iterations

    def plan(self, shape):
        """("erode", [steps per launch]) or ("stable", None)."""
        n = int(self.iterations)
        if n < 1:
            return "stable", None
        k = MORPH_STEPS_PER_LAUNCH
        return "erode", [k] * (n // k) + ([n % k] if n % k else [])

    def run_device(self, raster):
        path, launches = self.plan(raster.shape)
        if path == "erode":
            out = raster
            for n in launches:
                out = _morph(out, _lib.MORPH_ERODE, None, n)
            return out
        return _erode_until_stable(raster)


class BinaryClosing(_CheckedFilter):
    """``scipy.ndimage.binary_closing(image, structure=...)`` (extension_filters.py:238-293).  None, the 3x3 cross and
    the 3x3 square run on hd_binary_morph; any other 2-D structure up to 31x31 is a dilation and an erosion on
    hd_binary_morph_struct."""

    def __init__(self, *, structure=None):
        self.structure = structure

    def plan(self, shape):
        """("morph3", None) or ("struct", (dilation taps, erosion taps))."""
        if self.structure is None:
            return "morph3", None
        s = np.asarray(self.structure)
        if s.shape == (3, 3) and ((s != 0).all() or ((s != 0) == _CROSS).all()):
            return "morph3", None
        return "struct", closing_taps(s)

    def run_device(self, raster):
        path, taps = self.plan(raster.shape)
        if path == "morph3":
            return _morph(raster, _lib.MORPH_CLOSE, self.structure, 1)
        dil, ero = taps
        src = raster if raster.dtype in (_lib.U8, _lib.F32) else dev.convert(raster, _lib.U8, np.bool_)
        return _morph_struct(_morph_struct(src, 1, dil, 1), 0, ero, 1)


def _morph_struct(src, dilate, taps, iterations, changed=None):
    dy, dx = taps
    (dy, pdy), (dx, pdx) = _int_array(dy), _int_array(dx)
    out = dev.empty(src.ny, src.nx, _lib.U8, np.bool_)
    _lib.check(_lib.load().hd_binary_morph_struct(src.ptr, src.dtype, src.pitch, out.ptr, out.pitch, src.ny, src.nx, dilate,
                                                  len(dy), pdy, pdx, iterations, changed, dev.stream_ptr()))
    return out


def _erode_until_stable(raster):
    """Cross erosions until the result stops changing: launches of STABLE_STEPS_PER_LAUNCH erosions, each with its own
    device flag "output != input", read once per STABLE_LAUNCHES_PER_READ launches.  Erosion with a structure that holds
    its centre only removes cells, so a launch that changes nothing has reached the fixed point, and launches after it
    return the same raster."""
    import torch
    taps = _offsets(_CROSS, reversed_=False)
    flags = torch.zeros(STABLE_LAUNCHES_PER_READ, dtype=torch.int32, device=dev.device())
    cur = raster if raster.dtype in (_lib.U8, _lib.F32) else dev.convert(raster, _lib.U8, np.bool_)
    while True:
        for i in range(STABLE_LAUNCHES_PER_READ):
            cur = _morph_struct(cur, 0, taps, STABLE_STEPS_PER_LAUNCH, ctypes.c_void_p(flags.data_ptr() + 4 * i))
        if bool((flags == 0).any().item()):                             # the one host read of these launches
            return cur


def _morph(raster, op, structure, iterations):
    if structure is None:
        full = 0
    else:
        s = np.asarray(structure) != 0
        cross = np.array([[0, 1, 0], [1, 1, 1], [0, 1, 0]], dtype=bool)
        if s.shape == (3, 3) and s.all():
            full = 1
        elif s.shape == (3, 3) and (s == cross).all():
            full = 0
        else:
            raise DeviceError("binary morphology: only the 3x3 cross and the 3x3 square are implemented on the device")
    src = raster if raster.dtype in (_lib.U8, _lib.F32) else dev.convert(raster, _lib.U8, np.bool_)
    out = dev.empty(raster.ny, raster.nx, _lib.U8, np.bool_)
    _lib.check(_lib.load().hd_binary_morph(src.ptr, src.dtype, src.pitch, out.ptr, out.pitch, src.ny, src.nx, op, full,
                                           int(iterations), dev.stream_ptr()))
    return out


class GreyDilation(_CheckedFilter):
    """``scipy.ndimage.grey_dilation(image, size=(a, b))`` (extension_filters.py:296-345):
    flat rectangular maximum filter, mode='reflect'.  Odd square sizes up to 17 that fit the raster run on
    hd_max_filter; any other size 1 ... 255 per axis on hd_max_filter_rect."""

    def __init__(self, *, size):
        self.size = size

    def plan(self, shape):
        """("square", (s, s)) or ("rect", (a, b))."""
        a, b = grey_sizes(self.size)
        if a == b and a % 2 == 1 and a <= 17 and a <= min(shape):
            return "square", (a, b)
        return "rect", (a, b)

    def run_device(self, raster):
        path, (a, b) = self.plan(raster.shape)
        ref = np.dtype(raster.ref_dtype)
        if ref == np.float64 and raster.dtype == _lib.F32:
            src = raster                                              # narrow-exact storage (e.g. majority values)
        else:
            src = dev.convert(raster, _lib.F32 if ref == np.float32 else _lib.F64)
        out = dev.empty(raster.ny, raster.nx, src.dtype, ref)
        if path == "square":
            _lib.check(_lib.load().hd_max_filter(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, src.ny, src.nx, a,
                                                 dev.stream_ptr()))
            return out
        nbytes = src.ny * src.nx * src.itemsize
        work = dev.scratch(nbytes)
        _lib.check(_lib.load().hd_max_filter_rect(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, src.ny, src.nx, a, b,
                                                  ctypes.c_void_p(work.data_ptr()), nbytes, dev.stream_ptr()))
        return out


def _complex_ref(ref_dtype):
    """Result dtype of scipy.fftpack.fft2 / ifft2: single precision stays single, everything else complex128."""
    return np.dtype(np.complex64) if np.dtype(ref_dtype) in (np.float32, np.complex64) else np.dtype(np.complex128)


def _fft2(raster, inverse):
    ref = np.dtype(raster.ref_dtype)
    if ref.kind == "c":
        src = dev.convert(raster, _lib.C64)
    else:
        src = dev.convert(raster, _lib.F32)
    out = dev.empty(raster.ny, raster.nx, _lib.C64, _complex_ref(ref))
    lib = _lib.load()
    plan = dev.fft_plan(raster.ny, raster.nx)
    nbytes = lib.hd_fft2_workspace_bytes(raster.ny, raster.nx)
    work = dev.scratch(nbytes)
    _lib.check(lib.hd_fft2_c2c(plan, src.ptr, src.dtype, src.pitch, out.ptr, out.pitch, int(inverse),
                               ctypes.c_void_p(work.data_ptr()), nbytes, dev.stream_ptr()))
    return out


class FourierTransform(DeviceFilter):
    """``scipy.fftpack.fft2(image)`` (extension_filters.py:348-379).  Computed in complex64 on the
    device (float32 input gives complex64 exactly like scipy; wider inputs are returned as
    complex128 but carry single-precision accuracy -- tolerance class)."""

    def run_device(self, raster):
        return _fft2(raster, inverse=False)


class FourierITransform(DeviceFilter):
    """``scipy.fftpack.ifft2(image)`` (extension_filters.py:382-414); see FourierTransform."""

    def run_device(self, raster):
        return _fft2(raster, inverse=True)


def _shift(raster, inverse):
    out = dev.empty(raster.ny, raster.nx, raster.dtype, raster.ref_dtype)
    src = raster
    if raster.itemsize not in (4, 8, 16):
        src = dev.convert(raster, _lib.F32)
        out = dev.empty(raster.ny, raster.nx, _lib.F32, raster.ref_dtype)
    _lib.check(_lib.load().hd_fftshift2(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, src.ny, src.nx, int(inverse),
                                        dev.stream_ptr()))
    return out


class FourierShift(DeviceFilter):
    """``scipy.fftpack.fftshift(image)`` (extension_filters.py:417-447)."""

    def run_device(self, raster):
        return _shift(raster, inverse=False)


class FourierIShift(DeviceFilter):
    """``scipy.fftpack.ifftshift(image)`` (extension_filters.py:450-480)."""

    def run_device(self, raster):
        return _shift(raster, inverse=True)

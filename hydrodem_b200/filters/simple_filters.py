"""Elementwise filters (reference: ``filters/simple_filters.py``), device backed.

Same class names and constructor signatures as the reference
(``LowerThan(*, value)``, ``ProductFilter(factor=1)`` ...).  Each is one
``hd_elementwise`` launch; operands may be scalars, ndarrays or device rasters.
The result dtype follows NumPy's promotion rules, evaluated on empty host
arrays so that the reference's dtype flow (SURVEY.md A.3) is reproduced.
"""
import numpy as np

from . import DeviceFilter
from .. import _lib, device as dev


def _operand(value, like):
    """-> (DeviceRaster | None, scalar | None, prototype of the operand for NumPy's promotion).  Python scalars stay
    Python scalars (weak under NEP 50); NumPy scalars and 0-d arrays keep their dtype."""
    if isinstance(value, dev.DeviceRaster):
        return value, None, np.zeros(0, dtype=value.ref_dtype)
    if isinstance(value, np.ndarray) and value.ndim:
        if value.shape != like.shape:
            raise ValueError(f"operand shape {value.shape} does not match raster shape {like.shape}")
        return dev.upload(value), None, np.zeros(0, dtype=value.dtype)
    return None, value, value


def binary_op(op, raster, operand, np_func):
    """out = np_func(operand, raster) on the device, in NumPy's result dtype, which is also the dtype of its loop.
    Raises what NumPy raises (TypeError for a missing loop, OverflowError for a Python int out of range)."""
    b, scalar, proto = _operand(operand, raster)
    ref = np_func(proto, np.zeros(0, dtype=raster.ref_dtype)).dtype
    out = dev.empty(raster.ny, raster.nx, dev.hd_dtype_of(ref), ref)
    return dev.elementwise(op, raster, b, out, ref, scalar)


def compare(op, raster, value):
    """image < value / image > value -> bool, in the dtype NumPy compares in.  NumPy compares a Python int outside
    the range of an integer loop exactly (np.less(uint8, 300) is all True); against an integer raster that int acts
    like an infinity of its sign, so it is compared as one, in float64."""
    b, scalar, proto = _operand(value, raster)
    loop = np.result_type(raster.ref_dtype, proto)
    if type(scalar) is int and loop.kind in "iu" and not np.iinfo(loop).min <= scalar <= np.iinfo(loop).max:
        loop, scalar = np.dtype(np.float64), np.inf if scalar > 0 else -np.inf
    out = dev.empty(raster.ny, raster.nx, _lib.U8, np.bool_)
    return dev.elementwise(op, raster, b, out, loop, scalar)


class LowerThan(DeviceFilter):
    """``image < value`` -> bool (simple_filters.py:7-50)."""

    def __init__(self, *, value):
        self.value = value

    def run_device(self, raster):
        return compare(_lib.OP_LT, raster, self.value)


class GreaterThan(DeviceFilter):
    """``image > value`` -> bool (simple_filters.py:53-96)."""

    def __init__(self, *, value):
        self.value = value

    def run_device(self, raster):
        return compare(_lib.OP_GT, raster, self.value)


class BooleanToInteger(DeviceFilter):
    """``image * 1`` (simple_filters.py:99-131): bool -> int64, other dtypes unchanged."""

    def run_device(self, raster):
        return binary_op(_lib.OP_MUL, raster, 1, np.multiply)


class ProductFilter(DeviceFilter):
    """``factor * image`` (simple_filters.py:134-180)."""

    def __init__(self, factor=1):
        self.factor = factor

    def run_device(self, raster):
        return binary_op(_lib.OP_MUL, raster, self.factor, np.multiply)


class AdditionFilter(DeviceFilter):
    """``addend + image`` (simple_filters.py:183-229)."""

    def __init__(self, addend=0):
        self.addend = addend

    def run_device(self, raster):
        return binary_op(_lib.OP_ADD, raster, self.addend, np.add)


class SubtractionFilter(DeviceFilter):
    """``minuend - image`` (simple_filters.py:232-275)."""

    def __init__(self, *, minuend=0.0):
        self.minuend = minuend

    def run_device(self, raster):
        return binary_op(_lib.OP_RSUB, raster, self.minuend, np.subtract)

    def apply(self, subtracting):  # pylint: disable=arguments-renamed
        # the reference skips the ndarray check here (simple_filters.py:261-275)
        if not isinstance(subtracting, np.ndarray):
            return self.minuend - subtracting
        return dev.download(self.run_device(dev.upload(subtracting)))

"""hd_elementwise against NumPy, bit for bit: every op, raster dtype and operand kind of the elementwise filters, and
every device dtype conversion.

The reference is the NumPy expression each reference class evaluates (np.multiply(factor, image), np.less(image,
value), image.astype(dst) ...), run on the host under np.errstate(all="ignore").  Where NumPy raises, the class must
raise the same exception type.  Results compare bytewise: integers and bools as unsigned integers of their width (a
bool holding 2 fails), floats and each part of a complex as unsigned bits with the sign of a zero counted; a NaN only
has to be NaN in both.

The kernel implements NumPy's complex multiply and complex |z| with the formulas of NumPy's loops.  The CPU half of
this file pins those formulas against the host's NumPy with exact rational arithmetic, so that a NumPy built with
other loops fails there, by name, rather than in the GPU tests without an explanation.  The CPU half also checks that
the raster generators hold the edge values they are written for."""
import math
import warnings
from fractions import Fraction

import numpy as np
import pytest
import scipy.ndimage as ndi
import torch

from hydrodem_b200 import _lib, device as dev
from hydrodem_b200.filters.extension_filters import (AbsoluteValues, Around, BinaryClosing, BinaryErosion,
                                                     BitwiseXOR)
from hydrodem_b200.filters.simple_filters import (AdditionFilter, BooleanToInteger, GreaterThan, LowerThan,
                                                  ProductFilter, SubtractionFilter)

DTYPES = [np.dtype(d) for d in (np.bool_, np.uint8, np.int16, np.int32, np.int64, np.float32, np.float64,
                                np.complex64, np.complex128)]
assert set(DTYPES) == set(dev._NP2HD)


def gpu(test):
    """Marks one test as needing the device (the CPU tests of this file carry no mark)."""
    return pytest.mark.gpu(pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")(test))


# ---- bitwise comparison -------------------------------------------------------------------------------------------
def _real_bad(got, want):
    if got.dtype.kind == "f":
        nan_g, nan_w = np.isnan(got), np.isnan(want)
        u = np.dtype(f"u{got.dtype.itemsize}")
        return (nan_g != nan_w) | (~nan_g & ~nan_w & (got.view(u) != want.view(u)))
    return got.view(f"u{got.dtype.itemsize}") != want.view(f"u{want.dtype.itemsize}")


def bits_equal(got, want, what=""):
    """Bytewise equality of two arrays of the same dtype and shape (see the module docstring)."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.dtype == want.dtype, (what, got.dtype, want.dtype)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if got.dtype.kind == "c":
        bad = _real_bad(got.real.copy(), want.real.copy()) | _real_bad(got.imag.copy(), want.imag.copy())
    else:
        bad = _real_bad(got, want)
    if bad.any():
        idx = np.argwhere(bad.reshape(got.shape))
        first = tuple(idx[0])
        raise AssertionError(f"{what}: {len(idx)} of {bad.size} cells differ, first at {first}: "
                             f"got {got[first]!r}, want {want[first]!r}")


# ---- raster generators --------------------------------------------------------------------------------------------
F32_NEAR = [np.float32(0.1), np.float32(1.1)]


def float_edges(dt):
    dt = np.dtype(dt)
    fi = np.finfo(dt)
    v = [0.0, -0.0, 1.0, -1.0, fi.smallest_subnormal, -fi.smallest_subnormal, fi.max, -fi.max, np.inf, -np.inf,
         np.nan, 0.5, -0.5, 1.5, -1.5, 2.5, -2.5]
    for c in F32_NEAR:
        v += [np.nextafter(c, np.float32(-1)), c, np.nextafter(c, np.float32(2))]
    return np.array(v, dtype=dt)


def int_edges(dt):
    dt = np.dtype(dt)
    ii = np.iinfo(dt)
    v = [ii.min, ii.max, ii.min + 1, ii.max - 1, 0, 1, 2, 3, 255, 256, 32767, ii.max // 3 + 1, ii.max // 255 + 1]
    if ii.min < 0:
        v += [-1, -2, -3, -256, -(ii.max // 3) - 1]
    if dt == np.int64:
        v += [2 ** 53 + 1, -(2 ** 53 + 1), 2 ** 62 + 1]
    return np.array([x for x in v if ii.min <= x <= ii.max], dtype=dt)


def edge_values(dt):
    dt = np.dtype(dt)
    if dt == np.bool_:
        return np.array([False, True])
    if dt.kind in "iu":
        return int_edges(dt)
    if dt.kind == "f":
        return float_edges(dt)
    part = float_edges(np.float32 if dt == np.complex64 else np.float64)
    re, im = np.meshgrid(part, part)
    z = np.empty(re.size, dtype=dt)
    z.real, z.imag = re.ravel(), im.ravel()
    return z


def random_fill(dt, n, rng):
    dt = np.dtype(dt)
    if dt == np.bool_:
        return rng.random(n) < 0.5
    if dt.kind in "iu":
        ii = np.iinfo(dt)
        return rng.integers(ii.min, ii.max, n, dtype=dt, endpoint=True)
    if dt.kind == "f":
        return np.round(rng.normal(300, 200, n), int(rng.integers(0, 3))).astype(dt) if n else np.zeros(0, dt)
    z = np.empty(n, dtype=dt)
    z.real, z.imag = rng.normal(300, 200, n), rng.normal(0, 200, n)
    return z


def raster(dt, ny, nx, seed=0):
    """(ny, nx) raster of dtype dt: its edge values first (as many as fit), the rest random, in shuffled order."""
    rng = np.random.default_rng(seed)
    e = edge_values(dt)[: ny * nx]
    v = np.concatenate([e, random_fill(dt, ny * nx - len(e), rng)]).astype(dt)
    return rng.permutation(v).reshape(ny, nx)


# ---- operands -----------------------------------------------------------------------------------------------------
PY_SCALARS = ([True, False]
              + [0, 1, -1, 3, 255, 256, 32767, 2 ** 31, 2 ** 53 + 1, 2 ** 63 - 1]
              + [0.0, -0.0, 0.1, 1.1, 1 / 3, 1.5, 1e-40, 1e39, math.nan, math.inf, -math.inf]
              + [1j, 0.5 - 2j])


def np_scalars():
    out = []
    for d in DTYPES:
        out.append(d.type(True) if d == np.bool_ else d.type(3))
    out += [np.float32(0.1), np.float64(1.1), np.complex64(0.1 - 1.1j)]
    return out


ZERO_D = [np.array(np.float32(1.1)), np.array(3, dtype=np.int16), np.array(True)]


def operands(shape):
    """(label, host operand, device operand) for every operand kind of the matrix."""
    out = [(repr(v), v, v) for v in PY_SCALARS]
    out += [(f"{type(v).__name__}({v!r})", v, v) for v in np_scalars()]
    out += [(f"0-d {v.dtype}", v, v) for v in ZERO_D]
    for i, d in enumerate(DTYPES):
        arr = raster(d, *shape, seed=100 + i)
        out.append((f"ndarray {d}", arr, arr))
    u8 = (np.random.default_rng(7).random(shape) < 0.5).astype(np.uint8)
    out.append(("DeviceRaster u8 / ref float64", u8.astype(np.float64), ("u8f64", u8)))
    return out


def _device_operand(op):
    if isinstance(op, tuple) and op and op[0] == "u8f64":
        return dev.upload(op[1]).with_ref(np.float64)
    return op


# ---- the classes and their NumPy expressions ----------------------------------------------------------------------
BINARY = {
    "ProductFilter": (lambda v: ProductFilter(factor=v), lambda v, x: np.multiply(v, x)),
    "AdditionFilter": (lambda v: AdditionFilter(addend=v), lambda v, x: np.add(v, x)),
    "SubtractionFilter": (lambda v: SubtractionFilter(minuend=v), lambda v, x: np.subtract(v, x)),
    "LowerThan": (lambda v: LowerThan(value=v), lambda v, x: np.less(x, v)),
    "GreaterThan": (lambda v: GreaterThan(value=v), lambda v, x: np.greater(x, v)),
    "BitwiseXOR": (lambda v: BitwiseXOR(operand=v), lambda v, x: np.bitwise_xor(v, x)),
}
UNARY = {
    "BooleanToInteger": (BooleanToInteger, lambda x: x * 1),
    "AbsoluteValues": (AbsoluteValues, np.abs),
    "Around": (Around, np.around),
}
SHAPE = (23, 24)                     # room for the 23 x 23 part combinations of a complex raster


def run_filter(flt, host):
    return dev.download(flt.run_device(dev.upload(host)))


def check_against_numpy(make, expr, host, label):
    """The class raises what NumPy raises, or returns NumPy's bytes."""
    try:
        with np.errstate(all="ignore"):
            want = expr()
    except Exception as e:                                              # noqa: BLE001
        with pytest.raises(type(e)):
            with np.errstate(all="ignore"):
                run_filter(make(), host)
        return
    if want.dtype not in dev._NP2HD:                                    # e.g. np.around(bool) is float16
        with pytest.raises(dev.DeviceError):
            run_filter(make(), host)
        return
    bits_equal(run_filter(make(), host), want, label)


@gpu
@pytest.mark.parametrize("dtype", [d.name for d in DTYPES])
@pytest.mark.parametrize("name", list(BINARY))
def test_binary_op_matches_numpy(name, dtype):
    make, expr = BINARY[name]
    host = raster(dtype, *SHAPE)
    for label, h_op, d_op in operands(SHAPE):
        check_against_numpy(lambda: make(_device_operand(d_op)), lambda: expr(h_op, host), host,
                            f"{name}({label}) on {dtype}")


@gpu
@pytest.mark.parametrize("dtype", [d.name for d in DTYPES])
@pytest.mark.parametrize("name", list(UNARY))
def test_unary_op_matches_numpy(name, dtype):
    cls, expr = UNARY[name]
    host = raster(dtype, *SHAPE)
    check_against_numpy(cls, lambda: expr(host), host, f"{name} on {dtype}")


def astype_defined(src, dst):
    """Cells of `src` whose conversion to `dst` astype defines: in range (after truncation) for an integer target."""
    dst = np.dtype(dst)
    if dst.kind not in "iu" or src.dtype.kind in "biu":
        return np.ones(src.shape, bool)
    re = src.real if src.dtype.kind == "c" else src
    ii = np.iinfo(dst)
    with np.errstate(all="ignore"):
        t = np.trunc(re.astype(np.float64))
        return np.isfinite(t) & (t >= ii.min) & (t <= ii.max)


@gpu
@pytest.mark.parametrize("src", [d.name for d in DTYPES])
def test_convert_and_download_match_astype(src):
    host = raster(src, 29, 31, seed=3)
    r = dev.upload(host)
    for dst in DTYPES:
        keep = astype_defined(host, dst)
        with np.errstate(all="ignore"), warnings.catch_warnings():
            warnings.simplefilter("ignore")                             # complex -> real drops the imaginary part
            want = host.astype(dst)
        got = dev.download(dev.convert(r, dev.hd_dtype_of(dst), dst))
        bits_equal(np.where(keep, got, 0).astype(dst), np.where(keep, want, 0).astype(dst), f"convert {src} -> {dst}")
        if dev.hd_dtype_of(dst) == r.dtype:
            continue                  # a byte raster with a bool ref holds 0 / 1 already: download copies it as is
        got = dev.download(r.with_ref(dst))                             # the conversion inside download
        bits_equal(np.where(keep, got, 0).astype(dst), np.where(keep, want, 0).astype(dst), f"download {src} -> {dst}")


@gpu
@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_trunc_in_place(dtype):
    """HD_OP_TRUNC with `a is out`, as _InPlace3 calls it: truncation toward zero, NaN -> 0."""
    host = raster(dtype, 37, 41, seed=5)
    r = dev.upload(host)
    dev.elementwise(_lib.OP_TRUNC, r, None, r)
    with np.errstate(all="ignore"):
        want = np.where(np.isnan(host), 0, np.trunc(host)).astype(dtype)
    bits_equal(dev.download(r), want, f"trunc {dtype}")


# ---- shapes -------------------------------------------------------------------------------------------------------
def _shape_cases():
    return [(1, 1), (1, 97), (97, 1), (13, 17), (2049, 1537)]


@gpu
@pytest.mark.parametrize("shape", _shape_cases(), ids=lambda s: f"{s[0]}x{s[1]}")
def test_shapes(shape):
    a = raster(np.float32, *shape, seed=11)
    b = raster(np.float32, *shape, seed=12)
    bits_equal(run_filter(ProductFilter(factor=0.1), a), np.multiply(0.1, a), f"mul 0.1 {shape}")
    bits_equal(run_filter(AdditionFilter(addend=b), a), np.add(b, a), f"add array {shape}")
    bits_equal(run_filter(GreaterThan(value=np.float32(0.1)), a), np.greater(a, np.float32(0.1)), f"gt {shape}")
    c = raster(np.complex64, *shape, seed=13)
    with np.errstate(all="ignore"):
        bits_equal(run_filter(ProductFilter(factor=0.5 - 2j), c), np.multiply(0.5 - 2j, c), f"cmul {shape}")


@gpu
def test_one_row_longer_than_the_grid_stride():
    """One row of SMs * 16 * 256 + 5 cells: the grid-stride loop advances along x only (CellIter's sy = 0)."""
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    n = sms * 16 * 256 + 5
    a = raster(np.float32, 1, n, seed=17)
    with np.errstate(all="ignore"):
        bits_equal(run_filter(ProductFilter(factor=1.1), a), np.multiply(1.1, a), "long row mul")
        bits_equal(run_filter(SubtractionFilter(minuend=0.1), a), np.subtract(0.1, a), "long row rsub")
    i = raster(np.int16, 1, n, seed=18)
    bits_equal(dev.download(dev.convert(dev.upload(i), _lib.U8, np.bool_)), i.astype(bool), "long row bool")


@gpu
def test_views_with_three_pitches():
    """a, b and out as sub() views of parents of three widths; cells outside the out view stay untouched."""
    ny, nx = 23, 19
    pa, pb, po = raster(np.float32, 40, 20, seed=21), raster(np.float64, 40, 50, seed=22), np.full((40, 100), 7, np.float64)
    da, db, do = dev.upload(pa), dev.upload(pb), dev.upload(po)
    assert len({da.pitch * 4, db.pitch * 8, do.pitch * 8}) == 3
    a, b, out = da.sub(3, 3 + ny, 1, 1 + nx), db.sub(5, 5 + ny, 30, 30 + nx), do.sub(2, 2 + ny, 60, 60 + nx)
    dev.elementwise(_lib.OP_MUL, a, b, out, np.float64)
    want = po.copy()
    want[2:2 + ny, 60:60 + nx] = np.multiply(pb[5:5 + ny, 30:30 + nx], pa[3:3 + ny, 1:1 + nx])
    bits_equal(dev.download(do), want, "pitched views")


# ---- binary morphology of non-bool rasters ------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", ["float64", "int32", "int64"])
def test_binary_morphology_treats_nan_as_foreground(dtype):
    """BinaryErosion / BinaryClosing turn a raster into `!= 0` as scipy does: NaN is foreground.  (scipy refuses
    complex input.)"""
    rng = np.random.default_rng(31)
    host = np.where(rng.random((40, 45)) < 0.8, 1.5, 0).astype(dtype)
    if host.dtype.kind != "i":
        host[rng.random(host.shape) < 0.3] = np.nan
    bits_equal(run_filter(BinaryErosion(iterations=1), host), ndi.binary_erosion(host, iterations=1), "erosion")
    bits_equal(run_filter(BinaryClosing(), host), ndi.binary_closing(host), "closing")


# ---- CPU: generators ----------------------------------------------------------------------------------------------
def _has(arr, v):
    arr = np.asarray(arr)
    if isinstance(v, float) and math.isnan(v):
        return bool(np.isnan(arr).any())
    if isinstance(v, float) and v == 0:
        return bool(((arr == 0) & (np.signbit(arr) == (math.copysign(1, v) < 0))).any())
    return bool((arr == v).any())


@pytest.mark.parametrize("dtype", [d.name for d in DTYPES])
def test_rasters_hold_the_edge_values(dtype):
    dt = np.dtype(dtype)
    r = raster(dt, *SHAPE)
    assert r.shape == SHAPE and r.dtype == dt
    if dt.kind in "iu":
        ii = np.iinfo(dt)
        need = [ii.min, ii.max, ii.min + 1, ii.max - 1, 0, 1] + ([-1] if ii.min < 0 else [])
        if dt == np.int64:
            need += [2 ** 53 + 1, -(2 ** 53 + 1), 2 ** 62 + 1]
        for v in need:
            assert _has(r, v), (dtype, v)
        # a value whose product or sum with the operands overflows
        assert (np.abs(r.astype(object)) * 3 > ii.max).any() and (r.astype(object) + 256 > ii.max).any()
    elif dt.kind == "f":
        fi = np.finfo(dt)
        for v in [0.0, -0.0, 1.0, -1.0, float(fi.smallest_subnormal), float(fi.max), math.inf, -math.inf, math.nan,
                  0.5, -0.5, 1.5, -1.5, 2.5, -2.5]:
            assert _has(r, v), (dtype, v)
        for c in F32_NEAR:
            for v in (np.nextafter(c, np.float32(-1)), c, np.nextafter(c, np.float32(2))):
                assert _has(r, float(v)), (dtype, v)
    elif dt.kind == "c":
        for part in (r.real, r.imag):
            for v in (0.0, -0.0, math.inf, -math.inf, math.nan, 2.5):
                assert _has(part, v), (dtype, v)
        assert ((r.real == 0) & np.signbit(r.real) & (r.imag == 0) & ~np.signbit(r.imag)).any()
    else:
        assert r.any() and not r.all()


# ---- CPU: NumPy's complex loops -----------------------------------------------------------------------------------
def _round(q, dt):
    """Correctly rounded value of the rational q in float dtype dt."""
    try:
        d = float(q)                                                    # correctly rounded to double
    except OverflowError:
        d = math.inf if q > 0 else -math.inf
    if dt == np.float64:
        return np.float64(d)
    with np.errstate(over="ignore"):
        f = np.float32(d)
    if np.isinf(f):
        return f
    cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
    return min((c for c in cands if np.isfinite(c)),
               key=lambda c: (abs(Fraction(float(c)) - q), int(np.array(c).view(np.uint32)) & 1))


def _fma(x, y, z, dt):
    x, y, z = float(x), float(y), float(z)
    if math.isfinite(x) and math.isfinite(y) and not math.isfinite(z):
        return dt(z)                                                    # the exact product is finite
    if not (math.isfinite(x) and math.isfinite(y) and math.isfinite(z)):
        with np.errstate(all="ignore"):                                 # x * y is not finite: no rounding
            return dt(np.float64(x) * np.float64(y) + np.float64(z))
    q = Fraction(x) * Fraction(y) + Fraction(z)
    if q == 0:                      # an exact zero is -0 only when the product and z are both -0 (round to nearest)
        neg = (x == 0 or y == 0) and math.copysign(1, x) * math.copysign(1, y) < 0 and z == 0 and math.copysign(1, z) < 0
        return dt(-0.0 if neg else 0.0)
    return _round(q, dt)


def cmul_formula(x, y, dt):
    """re = fma(xr, yr, -(xi * yi)), im = fma(xr, yi, xi * yr), as the kernel computes x * y."""
    return (_fma(x.real, y.real, -(x.imag * y.imag), dt), _fma(x.real, y.imag, x.imag * y.real, dt))


def cabs_formula(z, dt):
    """hi * sqrt(fma(r, r, 1)), r = lo / hi; inf / NaN / 0 cases as the kernel handles them."""
    a, b = abs(dt(z.real)), abs(dt(z.imag))
    if np.isinf(a) or np.isinf(b):
        return dt(np.inf)
    if np.isnan(a) or np.isnan(b):
        return dt(np.nan)
    hi, lo = max(a, b), min(a, b)
    if hi == 0:
        return dt(0)
    with np.errstate(all="ignore"):
        r = dt(lo / hi)
        return dt(hi * dt(np.sqrt(_fma(r, r, dt(1), dt))))


def _complex_samples(cdt, n, seed):
    rng = np.random.default_rng(seed)
    z = np.empty(n, cdt)
    z.real = rng.normal(300, 200, n) * 10.0 ** rng.integers(-3, 4, n)
    z.imag = rng.normal(0, 200, n) * 10.0 ** rng.integers(-3, 4, n)
    return z


@pytest.mark.parametrize("cdt", ["complex64", "complex128"])
def test_numpy_complex_multiply_is_the_pinned_fma_formula(cdt):
    dt = np.float32 if cdt == "complex64" else np.float64
    e = edge_values(cdt)
    pick = np.random.default_rng(4).integers(0, len(e), (2, 4000))
    x = np.concatenate([_complex_samples(cdt, 4000, 1), e[pick[0]]])
    y = np.concatenate([_complex_samples(cdt, 4000, 2), e[pick[1]]])
    with np.errstate(all="ignore"):
        got = np.multiply(x, y)
    for i in range(len(x)):
        with np.errstate(all="ignore"):
            re, im = cmul_formula(x[i], y[i], dt)
        want = np.array([complex(re, im)], np.dtype(cdt))
        want.real, want.imag = re, im
        assert not (_real_bad(got[i:i + 1].real.copy(), want.real.copy()) |
                    _real_bad(got[i:i + 1].imag.copy(), want.imag.copy())).any(), (
            f"this NumPy's {cdt} multiply is not re = fma(xr, yr, -(xi*yi)), im = fma(xr, yi, xi*yr): "
            f"{x[i]!r} * {y[i]!r} = {got[i]!r}, formula gives {complex(re, im)!r}")


@pytest.mark.parametrize("cdt", ["complex64", "complex128"])
def test_numpy_complex_abs_is_the_pinned_scaled_formula(cdt):
    dt = np.float32 if cdt == "complex64" else np.float64
    z = np.concatenate([_complex_samples(cdt, 4000, 3), edge_values(cdt)])
    with np.errstate(all="ignore"):
        got = np.abs(z)
        want = np.array([cabs_formula(v, dt) for v in z], dt)
    bad = _real_bad(got, want)
    assert not bad.any(), (f"this NumPy's {cdt} abs is not hi * sqrt(fma(r, r, 1)), r = lo / hi: "
                           f"|{z[bad][0]!r}| = {got[bad][0]!r}, formula gives {want[bad][0]!r}")

"""The scipy.ndimage wrappers with every argument the reference's classes accept, bit for bit against scipy itself.

Convolve takes any 2-D weights up to 31 x 31, BinaryErosion any iteration count (< 1 = until nothing changes),
BinaryClosing any 2-D structure up to 31 x 31 and GreyDilation any size 1 ... 255 per axis.  The arguments the chain uses
keep their kernels (3 x 3 weights, the cross or the square, odd square sizes up to 17 that fit the raster); everything
else runs on hd_correlate, hd_binary_morph_struct and hd_max_filter_rect.  Shapes: 1 x 1, thin rasters, rasters smaller
than the footprint, one cell either side of the 32 x 128 tile seams, and one raster with more tiles than the persistent
grid holds.  Results are compared bitwise (the same-width unsigned integers; a NaN only has to be NaN in both), so the
sign of a zero counts, except for the sign of a zero maximum of the grey dilation (DESIGN.md section 7).

The CPU tests restate the host-side footprint, origin and tap-list construction in NumPy and check it against scipy on
small cases, check which path each argument selects, and check that over-limit and malformed arguments raise before any
device work."""
import ctypes
import os
import warnings

import numpy as np
import pytest
import scipy.ndimage as ndi

from hydrodem_b200 import _lib
from hydrodem_b200 import device as dev
from hydrodem_b200.exceptions import DeviceError
from hydrodem_b200.filters import extension_filters as ef
from test_gpu_window_paths import BIG, SEAMS, SUBNORMAL, _out, bits_equal, gen_grey, gen_morph, gpu

CONV_SIZES = [1, 2, 3, 4, 5, 8, 15, 16, 31]
GREY_SIZES = [1, 2, 3, 4, 8, 17, 18, 31, 64, 255]
EPS = np.finfo(np.float64).eps
TINY = np.array([EPS, -EPS, 1e-17, 2.3e-16, -2.3e-16, EPS * 0.5], dtype=np.float64)   # at, below and above DBL_EPSILON


# ---- NumPy restatements of the host-side plans ------------------------------------------------------------------
def reflect_periodic(i, n):
    m = np.mod(i, 2 * n)
    return np.where(m < n, m, 2 * n - 1 - m)


def correlate_taps_ref(a, dy, dx, w, size):
    """The double sum over the taps in their order, from +0.0, each product and sum rounded; cast; / size."""
    ny, nx = a.shape
    yy, xx = np.mgrid[0:ny, 0:nx]
    acc = np.zeros(a.shape, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        for y, x, v in zip(dy, dx, w):
            acc = acc + a[reflect_periodic(yy + y, ny), reflect_periodic(xx + x, nx)].astype(np.float64) * v
        return acc.astype(a.dtype) / a.dtype.type(size)


def morph_taps_ref(a, taps, dilate):
    """Erosion (AND) or dilation (OR) over the tap offsets, cells outside the raster False."""
    ny, nx = a.shape
    pad = np.zeros((ny + 64, nx + 64), dtype=bool)
    pad[32:32 + ny, 32:32 + nx] = a != 0
    out = np.zeros(a.shape, dtype=bool) if dilate else np.ones(a.shape, dtype=bool)
    for y, x in zip(*taps):
        s = pad[32 + y:32 + y + ny, 32 + x:32 + x + nx]
        out = (out | s) if dilate else (out & s)
    return out


def grey_window_ref(a, sy, sx, skip_nan=False):
    """Maximum over [i - lo, i - lo + k - 1] per axis, lo = k // 2 - 1 on even axes, periodic reflect."""
    ny, nx = a.shape
    out = a
    for axis, k in ((0, sy), (1, sx)):
        n = out.shape[axis]
        lo = k // 2 - (1 if k % 2 == 0 else 0)
        idx = reflect_periodic(np.arange(n)[:, None] - lo + np.arange(k)[None, :], n)      # (n, k)
        v = out[idx, :] if axis == 0 else out[:, idx]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            out = (np.nanmax if skip_nan else np.max)(v, axis=axis + 1)
    return out


# ---- generators ---------------------------------------------------------------------------------------------------
def gen_weights(kh, kw, seed):
    """Normal weights of both signs with 20 % zeros and 25 % entries at, just below and just above DBL_EPSILON."""
    rng = np.random.default_rng(seed)
    w = rng.standard_normal((kh, kw))
    r = rng.random((kh, kw))
    w[r < 0.2] = 0.0
    tiny = (r >= 0.2) & (r < 0.45)
    w[tiny] = TINY[rng.integers(0, len(TINY), int(tiny.sum()))]
    return w


def gen_conv(shape, dtype, seed):
    """Values of both signs; in the left third NaN runs, +-inf, subnormals and blocks of +-0 (all -0.0 windows too)."""
    rng = np.random.default_rng(seed)
    ny, nx = shape
    a = (rng.standard_normal(shape) * 100).astype(dtype)
    third = max(1, nx // 3)
    left = a[:, :third]
    sub = np.finfo(dtype).smallest_subnormal
    special = np.array([np.inf, -np.inf, sub, -sub, 0.0, -0.0], dtype=dtype)
    pick = rng.random(left.shape) < 0.08
    left[pick] = special[rng.integers(0, len(special), int(pick.sum()))]
    for _ in range(max(1, ny * third // 300)):
        y, x = int(rng.integers(0, ny)), int(rng.integers(0, third))
        left[y, x:x + int(rng.integers(2, 6))] = np.nan
    if ny > 4 and nx > 8:
        a[ny // 2:, nx - 6:] = dtype(-0.0)
    return a


def shapes_small(k):
    """1 x 1, thin rasters, one smaller than a k x k footprint, and a tile seam."""
    small = (max(1, k // 2), max(1, k - 1))
    return [(1, 1), (1, 40), (40, 1), small, SEAMS[1]]


# ---- device calls -------------------------------------------------------------------------------------------------
def run_correlate(a, weights):
    """hd_correlate straight from the ABI (also for 3 x 3 weights, which the class sends to hd_convolve3)."""
    dy, dx, w = ef.convolve_taps(weights)
    (dy, pdy), (dx, pdx) = ef._int_array(dy), ef._int_array(dx)
    w = np.ascontiguousarray(w)
    ny, nx = a.shape
    src = dev.upload(a)
    out = _out(ny, nx, src.dtype)
    _lib.check(_lib.load().hd_correlate(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, ny, nx, len(w), pdy, pdx,
                                        w.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), float(np.size(weights)),
                                        dev.stream_ptr()))
    return dev.download(out)


def conv_want(a, w):
    with np.errstate(invalid="ignore", over="ignore"):
        return ndi.convolve(a, w, mode="reflect") / w.size


# ---- CPU: plans against scipy -------------------------------------------------------------------------------------
@pytest.mark.parametrize("kh,kw", [(1, 1), (1, 2), (2, 1), (2, 2), (3, 4), (4, 3), (5, 2), (8, 5), (7, 7)])
def test_convolve_taps_follow_scipy(kh, kw):
    """The tap list (flip, even-axis origin, DBL_EPSILON rule, order) summed in NumPy equals scipy bit for bit, with
    periodic reflection on rasters smaller than the weights."""
    for shape in [(1, 1), (2, 3), (5, 7), (9, 11)]:
        w = gen_weights(kh, kw, kh * 10 + kw)
        a = gen_conv(shape, np.float64, kh + kw + shape[0])
        got = correlate_taps_ref(a, *ef.convolve_taps(w), w.size)
        bits_equal(got, conv_want(a, w), f"{(kh, kw)} {shape}")


def test_convolve_epsilon_rule_and_reflection():
    """The cases quoted by the issue of this feature, from scipy 1.18.1."""
    x = np.ones((3, 3))
    x[1, 1] = np.nan
    assert np.isfinite(conv_want(x, np.full((3, 3), 1e-17))).all()
    assert np.isnan(conv_want(x, np.full((3, 3), 2.3e-16))[1, 1])
    dy, dx, w = ef.convolve_taps(np.full((3, 3), EPS))
    assert len(w) == 0
    bits_equal(conv_want(np.array([[1.0, 2.0]]), np.ones((1, 7))), np.array([[11.0, 10.0]]) / 7)
    bits_equal(correlate_taps_ref(np.array([[1.0, 2.0]]), *ef.convolve_taps(np.ones((1, 7))), 7),
               np.array([[11.0, 10.0]]) / 7)
    bits_equal(correlate_taps_ref(np.full((4, 4), -0.0), *ef.convolve_taps(np.ones((2, 2))), 4), np.zeros((4, 4)))


STRUCTS = {
    "1x1": np.ones((1, 1)), "2x2": np.ones((2, 2)), "line_h4": np.ones((1, 4)), "line_v5": np.ones((5, 1)),
    "diag3": np.eye(3), "asym2x3": np.array([[1, 0, 0], [1, 1, 0]]), "even4x6": None, "empty": np.zeros((3, 3)),
    "no_centre": np.array([[1, 0, 1], [0, 0, 0], [0, 1, 0]]),
}


def _structure(name, seed=0):
    s = STRUCTS[name]
    if s is None:
        s = np.random.default_rng(seed).random((4, 6)) < 0.5
    return s


@pytest.mark.parametrize("name", list(STRUCTS))
def test_closing_taps_follow_scipy(name):
    s = _structure(name)
    dil, ero = ef.closing_taps(s)
    for shape in [(1, 1), (3, 2), (9, 13)]:
        a = gen_morph(shape, True, shape[0] + shape[1])
        got = morph_taps_ref(morph_taps_ref(a, dil, True), ero, False)
        want = ndi.binary_closing(a, structure=s, border_value=0)
        bits_equal(got, want, f"{name} {shape}")
        bits_equal(morph_taps_ref(a, dil, True), ndi.binary_dilation(a, structure=s, border_value=0), name)
        bits_equal(morph_taps_ref(a, ero, False), ndi.binary_erosion(a, structure=s, border_value=0), name)


def test_grey_window_follows_scipy():
    rng = np.random.default_rng(3)
    ramp = np.arange(12.0).reshape(3, 4)
    bits_equal(grey_window_ref(ramp, 2, 3), ndi.grey_dilation(ramp, size=(2, 3)))
    for sy, sx in [(1, 1), (2, 2), (4, 3), (8, 1), (9, 18), (17, 4)]:
        for shape in [(1, 1), (1, 5), (3, 7), (12, 10)]:
            a = rng.standard_normal(shape)
            bits_equal(grey_window_ref(a, sy, sx), ndi.grey_dilation(a, size=(sy, sx), mode="reflect"),
                       f"{(sy, sx)} {shape}")


def test_path_selection():
    """Today's arguments keep today's kernels; everything else goes to the new entry points."""
    assert ef.Convolve().plan((5, 5))[0] == "conv3"
    assert ef.Convolve(weights=np.arange(9.0).reshape(3, 3)).plan((1, 1))[0] == "conv3"
    for shape in [(1, 1), (2, 2), (5, 5), (3, 1), (31, 31)]:
        assert ef.Convolve(weights=np.ones(shape)).plan((50, 50))[0] == "correlate", shape
    assert ef.BinaryErosion(iterations=1).plan((9, 9)) == ("erode", [1])
    assert ef.BinaryErosion(iterations=8).plan((9, 9)) == ("erode", [8])
    assert ef.BinaryErosion(iterations=20).plan((9, 9)) == ("erode", [8, 8, 4])
    assert ef.BinaryErosion(iterations=16).plan((9, 9)) == ("erode", [8, 8])
    assert ef.BinaryErosion(iterations=0).plan((9, 9))[0] == "stable"
    assert ef.BinaryErosion(iterations=-1).plan((9, 9))[0] == "stable"
    cross = ndi.generate_binary_structure(2, 1)
    for s in (None, np.ones((3, 3)), cross, cross.astype(np.float32) * 7):
        assert ef.BinaryClosing(structure=s).plan((9, 9))[0] == "morph3"
    for s in (np.ones((1, 1)), np.ones((3, 2)), np.eye(3), np.zeros((3, 3)), np.ones((31, 31))):
        assert ef.BinaryClosing(structure=s).plan((9, 9))[0] == "struct"
    for size in (1, 3, 7, 17, (5, 5)):
        assert ef.GreyDilation(size=size).plan((40, 40))[0] == "square", size
    for size, shape in [(2, (40, 40)), ((3, 5), (40, 40)), (19, (40, 40)), (7, (6, 40)), (255, (300, 300))]:
        assert ef.GreyDilation(size=size).plan(shape)[0] == "rect", size


@pytest.mark.parametrize("make", [
    lambda: ef.Convolve(weights=np.ones((32, 3))),
    lambda: ef.Convolve(weights=np.ones(5)),
    lambda: ef.Convolve(weights=np.ones((3, 3, 3))),
    lambda: ef.Convolve(weights=np.ones((0, 3))),
    lambda: ef.BinaryClosing(structure=np.ones((3, 32))),
    lambda: ef.BinaryClosing(structure=np.ones(3)),
    lambda: ef.BinaryClosing(structure=np.ones((2, 0))),
    lambda: ef.GreyDilation(size=256),
    lambda: ef.GreyDilation(size=(3, 300)),
    lambda: ef.GreyDilation(size=0),
    lambda: ef.GreyDilation(size=(3, -1)),
    lambda: ef.GreyDilation(size=(3, 3, 3)),
    lambda: ef.GreyDilation(size=2.5),
], ids=["conv_32", "conv_1d", "conv_3d", "conv_empty", "close_32", "close_1d", "close_empty", "grey_256",
        "grey_300", "grey_0", "grey_neg", "grey_3d", "grey_float"])
def test_bad_arguments_raise_before_device_work(make, monkeypatch):
    def no_device(*args, **kwargs):
        raise AssertionError("the raster reached the device")
    monkeypatch.setattr(dev, "upload", no_device)
    with pytest.raises(DeviceError) as err:
        make().apply(np.ones((40, 40), dtype=np.float32))
    assert "device" in str(err.value) or "must" in str(err.value)


def test_limit_messages_name_the_limit():
    with pytest.raises(DeviceError, match="31x31"):
        ef.Convolve(weights=np.ones((32, 3))).plan((9, 9))
    with pytest.raises(DeviceError, match="31x31"):
        ef.BinaryClosing(structure=np.ones((3, 32))).plan((9, 9))
    with pytest.raises(DeviceError, match="255"):
        ef.GreyDilation(size=(256, 3)).plan((9, 9))
    with pytest.raises(DeviceError, match=">= 1"):
        ef.GreyDilation(size=(0, 3)).plan((9, 9))


def test_abi_refuses_beyond_its_limits():
    if not os.path.exists(_lib.LIB_PATH):
        from hydrodem_b200.build import build
        build()
    lib = _lib.load()
    p = ctypes.c_void_p(1 << 20)
    I = ctypes.c_int
    D = ctypes.c_double

    def ints(*v):
        return (I * len(v))(*v)
    w1 = (D * 1)(1.0)
    assert lib.hd_correlate(p, 64, p, 64, _lib.F32, 64, 64, 1, ints(16), ints(0), w1, 1.0, None) == _lib.HD_ERR_UNSUPPORTED
    assert lib.hd_correlate(p, 64, p, 64, _lib.F32, 64, 64, 1, ints(0), ints(-16), w1, 1.0, None) == _lib.HD_ERR_UNSUPPORTED
    n = 962
    assert lib.hd_correlate(p, 64, p, 64, _lib.F64, 64, 64, n, (I * n)(), (I * n)(), (D * n)(), 1.0,
                            None) == _lib.HD_ERR_UNSUPPORTED
    assert lib.hd_correlate(p, 64, p, 64, _lib.U8, 64, 64, 1, ints(0), ints(0), w1, 1.0, None) == _lib.HD_ERR_UNSUPPORTED
    assert lib.hd_correlate(None, 64, p, 64, _lib.F32, 64, 64, 1, ints(0), ints(0), w1, 1.0, None) == _lib.HD_ERR_NULL
    assert lib.hd_binary_morph_struct(p, _lib.U8, 256, p, 256, 64, 64, 0, 1, ints(1), ints(0), 16, None,
                                      None) == _lib.HD_ERR_UNSUPPORTED
    assert lib.hd_binary_morph_struct(p, _lib.U8, 256, p, 256, 64, 64, 0, 1, ints(0), ints(8), 2, None,
                                      None) == _lib.HD_ERR_UNSUPPORTED
    assert lib.hd_binary_morph_struct(p, _lib.U8, 256, p, 256, 64, 64, 0, 1, ints(0), ints(0), 0, None,
                                      None) == _lib.HD_ERR_ARG
    assert lib.hd_binary_morph_struct(p, _lib.F64, 256, p, 256, 64, 64, 0, 1, ints(0), ints(0), 1, None,
                                      None) == _lib.HD_ERR_UNSUPPORTED
    assert lib.hd_max_filter_rect(p, 64, p, 64, _lib.F32, 64, 64, 256, 3, p, 1 << 20, None) == _lib.HD_ERR_UNSUPPORTED
    assert lib.hd_max_filter_rect(p, 64, p, 64, _lib.F32, 64, 64, 0, 3, p, 1 << 20, None) == _lib.HD_ERR_ARG
    assert lib.hd_max_filter_rect(p, 64, p, 64, _lib.F32, 64, 64, 3, 3, p, 64 * 64 * 4 - 1, None) == _lib.HD_ERR_WORKSPACE
    assert lib.hd_max_filter_rect(p, 64, p, 64, _lib.F32, 64, 64, 3, 3, None, 1 << 20, None) == _lib.HD_ERR_NULL


# ---- GPU: Convolve ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("kh", CONV_SIZES)
@gpu
def test_convolve_every_weight_shape(kh, dtype):
    """(kh, kw) over CONV_SIZES^2 on a tile-seam raster, through the class and (3 x 3 too) through hd_correlate; the
    small shapes for the square weights."""
    for kw in CONV_SIZES:
        w = gen_weights(kh, kw, 31 * kh + kw)
        a = gen_conv(SEAMS[0], dtype, kh * 100 + kw)
        want = conv_want(a, w)
        bits_equal(run_correlate(a, w), want, f"hd_correlate {(kh, kw)} {SEAMS[0]}")
        bits_equal(ef.Convolve(weights=w).apply(a), want, f"Convolve {(kh, kw)} {SEAMS[0]}")
    for shape in shapes_small(kh):
        w = gen_weights(kh, kh, kh)
        a = gen_conv(shape, dtype, kh + shape[0] * 7 + shape[1])
        bits_equal(run_correlate(a, w), conv_want(a, w), f"hd_correlate {(kh, kh)} {shape}")


@gpu
def test_convolve_epsilon_weights_skip_nan():
    """NaN under a weight |w| <= DBL_EPSILON does not reach the result; under 2.3e-16 it does."""
    a = gen_conv(SEAMS[2], np.float64, 5)
    a[::2, ::3] = np.nan                  # on even output rows the NaN rows fall under the tiny weight rows only
    for tiny in (1e-17, EPS, -EPS, 2.3e-16):
        w = np.ones((5, 4))
        w[::2, :] = tiny
        want = conv_want(a, w)
        if abs(tiny) <= EPS:
            assert np.isfinite(want[:, 100:]).sum() > 1000
        else:
            assert np.isnan(want[:, 100:]).all()
        bits_equal(ef.Convolve(weights=w).apply(a), want, f"tiny={tiny}")
        bits_equal(ef.Convolve(weights=w).apply(a.astype(np.float32)), conv_want(a.astype(np.float32), w), f"f32 {tiny}")


@gpu
def test_convolve_more_tiles_than_grid():
    for w, dtype in ((gen_weights(5, 5, 1), np.float32), (gen_weights(4, 7, 2), np.float64)):
        a = gen_conv(BIG, dtype, 9)
        bits_equal(ef.Convolve(weights=w).apply(a), conv_want(a, w), f"{w.shape} {BIG}")


# ---- GPU: BinaryErosion -------------------------------------------------------------------------------------------
def erosion_inputs(shape, seed):
    a = gen_morph(shape, False, seed)                  # F32 with NaN (True) and -0.0 (False)
    u8 = gen_morph(shape, True, seed + 1)
    return {"f32": a, "u8": u8, "bool": u8 != 0, "i16": np.where(u8 != 0, np.int16(-300), np.int16(0))}


@pytest.mark.parametrize("iterations", list(range(1, 21)) + [0, -1])
@gpu
def test_binary_erosion_every_iteration_count(iterations):
    for shape in [(1, 1), (1, 40), (40, 1), SEAMS[0], SEAMS[1], (70, 90)]:
        for tag, a in erosion_inputs(shape, shape[0] + shape[1] + iterations).items():
            if shape == (70, 90):
                a = a.copy()
                a[5:65, 5:85] = 1                          # a large blob, so many iterations still change something
            want = ndi.binary_erosion(a, iterations=iterations, border_value=0)
            bits_equal(ef.BinaryErosion(iterations=iterations).apply(a), want, f"x{iterations} {tag} {shape}")


@gpu
def test_binary_erosion_until_stable_all_true():
    a = np.ones((9, 9), dtype=bool)
    assert not ef.BinaryErosion(iterations=0).apply(a).any()
    big = np.ones((600, 700), dtype=np.uint8)            # 300 erosions: 20 launches, 3 host reads
    bits_equal(ef.BinaryErosion(iterations=-1).apply(big), np.zeros(big.shape, dtype=bool), "600 x 700")


@gpu
def test_binary_erosion_more_tiles_than_grid():
    a = gen_morph(BIG, False, 3)
    a[100:1900, 100:1400] = 1.0
    bits_equal(ef.BinaryErosion(iterations=20).apply(a), ndi.binary_erosion(a, iterations=20, border_value=0), f"{BIG}")


# ---- GPU: BinaryClosing -------------------------------------------------------------------------------------------
def closing_structures():
    rng = np.random.default_rng(17)
    out = {name: _structure(name, 5) for name in STRUCTS}
    for k in (5, 8, 16, 31):
        out[f"random{k}"] = rng.random((k, k)) < 0.4
        out[f"random{k}x{k // 2 + 1}"] = rng.random((k, k // 2 + 1)) < 0.5
    out["line_h31"] = np.ones((1, 31))
    out["line_v30"] = np.ones((30, 1))
    out["square31"] = np.ones((31, 31))
    yy, xx = np.mgrid[-3:4, -3:4]
    out["disc7"] = (yy ** 2 + xx ** 2) <= 9
    out["nan_float"] = np.where(rng.random((4, 5)) < 0.5, np.nan, 0.0)
    out["none"] = None
    out["ones3"] = np.ones((3, 3))
    return out


@pytest.mark.parametrize("name", list(closing_structures()))
@gpu
def test_binary_closing_every_structure(name):
    s = closing_structures()[name]
    k = 3 if s is None else max(np.shape(s))
    for shape in shapes_small(k) + [SEAMS[0], SEAMS[2]]:
        for u8 in (False, True):
            a = gen_morph(shape, u8, shape[0] * 3 + shape[1] + k)
            want = ndi.binary_closing(a, structure=s, border_value=0)
            bits_equal(ef.BinaryClosing(structure=s).apply(a), want, f"{name} u8={u8} {shape}")


@gpu
def test_binary_closing_more_tiles_than_grid():
    yy, xx = np.mgrid[-3:4, -3:4]
    for s in ((yy ** 2 + xx ** 2) <= 9, np.ones((4, 6))):
        a = gen_morph(BIG, False, 21)
        bits_equal(ef.BinaryClosing(structure=s).apply(a), ndi.binary_closing(a, structure=s, border_value=0), f"{BIG}")


# ---- GPU: GreyDilation --------------------------------------------------------------------------------------------
GREY_CASES = [s for s in GREY_SIZES] + [(a, b) for a in GREY_SIZES for b in GREY_SIZES if a != b]


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("size", GREY_CASES, ids=[str(s) for s in GREY_CASES])
@gpu
def test_grey_dilation_every_size(size, dtype):
    a_, b_ = (size, size) if np.ndim(size) == 0 else size
    shapes = [(1, 1), (1, 300), (300, 1), (max(1, a_ // 2), max(1, b_ - 1)), SEAMS[1]]
    for shape in shapes:
        a = gen_grey(shape, dtype, a_ * 1000 + b_ + shape[0])
        want = ndi.grey_dilation(a, size=(a_, b_), mode="reflect")
        bits_equal(ef.GreyDilation(size=size).apply(a), want, f"size={size} {shape}", zero_sign=False)


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@gpu
def test_grey_dilation_skips_nan(dtype):
    for size in ((2, 3), 8, (31, 4), 64):
        a = gen_grey(SEAMS[2], dtype, 3)
        rng = np.random.default_rng(4)
        a[rng.random(a.shape) < 0.2] = np.nan
        a[10:25, 40:120] = np.nan
        sy, sx = (size, size) if np.ndim(size) == 0 else size
        bits_equal(ef.GreyDilation(size=size).apply(a), grey_window_ref(a, sy, sx, skip_nan=True), f"size={size}",
                   zero_sign=False)


@gpu
def test_grey_dilation_more_tiles_than_grid():
    for size, dtype in (((18, 31), np.float32), ((3, 64), np.float64)):
        a = gen_grey(BIG, dtype, 8)
        bits_equal(ef.GreyDilation(size=size).apply(a), ndi.grey_dilation(a, size=size, mode="reflect"), f"{size} {BIG}",
                   zero_sign=False)

"""Every window size and dtype path of the exact windowed kernels against independent references, bit for bit.

The C ABI accepts more than the chain uses: majority at ws 3 ... 15 with F32 or F64 output, expand at ws 3 ... 15 from
U8 or F32 into U8 / F32 / F64, binary morphology as erode / dilate (up to 8 iterations) and close / open (up to 4) with
the cross or the full 3x3 structure, the grey dilation at every odd size 1 ... 17 in F32 (one path for 7, a generic one
for the rest) and F64, and the quadratic smoother at ws 3 ... 15.  Each of them runs here on the shapes where tiled
kernels go wrong: the smallest raster the window allows, thin rasters, one cell either side of the 32 x 128 tile seams,
and one raster with more tiles than the persistent grid holds.

References are plain restatements, independent of the kernels' algorithms:
  * majority: collections.Counter over each corner-less window, as MajorityFilter.apply does (custom_filters.py:48-73);
  * expand: "any non-NaN cell of the corner-less window is > 0", and the product with `select` in float32 NumPy;
  * morphology and grey dilation: scipy.ndimage itself, which is what the reference's classes call;
  * quadratic: oracle.stencils.quadratic, with the stage's relative tolerance of 1e-5.
Exact kernels are compared bitwise (the same-width unsigned integers; a NaN only has to be NaN in both), so the sign of
a zero counts.  The one exception is the sign of a zero maximum of the grey dilation, which scipy leaves to its scan
order (DESIGN.md section 7).

The input generators assert on the CPU that they reach the edges they are written for; those checks, the Counter
reference against oracle.stencils.majority, and the ABI's refusals need no GPU and carry no `gpu` mark."""
import collections
import ctypes
import os
import warnings

import numpy as np
import pytest
import scipy.ndimage as ndi
import torch
from numpy.lib.stride_tricks import sliding_window_view

from hydrodem_b200 import _lib
from oracle import stencils


def gpu(test):
    """Marks one test as needing the device (the CPU tests of this file carry no mark)."""
    return pytest.mark.gpu(pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")(test))


if torch.cuda.is_available():
    from hydrodem_b200 import device as dev
    from hydrodem_b200.filters import custom_filters as cf
    from oracle import clib

WINDOWS = [3, 5, 7, 9, 11, 13, 15]
SEAMS = [(33, 129), (31, 127), (65, 257)]
BIG = (2049, 1537)                   # 65 x 13 = 845 tiles: more than the persistent grid of any of these kernels holds
SUBNORMAL = np.float32(1e-45)         # the smallest positive float32 subnormal
F32_OUT = {_lib.F32: np.float32, _lib.F64: np.float64}


def shapes_for(ws):
    """The smallest raster, two thin ones, and the tile-seam shapes (those the window fits in)."""
    return [(ws, ws), (ws, 300), (300, ws)] + [s for s in SEAMS if min(s) >= ws]


# ---- comparison ---------------------------------------------------------------------------------------------------
def bits_equal(got, want, what="", zero_sign=True):
    """Bitwise equality of two arrays of the same dtype and shape.  NaN only has to be NaN in both (payloads are not
    part of any contract); with zero_sign=False, -0.0 and +0.0 are taken as equal."""
    assert got.dtype == want.dtype, (what, got.dtype, want.dtype)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if got.dtype.kind == "f":
        nan_g, nan_w = np.isnan(got), np.isnan(want)
        bad = nan_g != nan_w
        if not zero_sign:
            got, want = got + got.dtype.type(0), want + want.dtype.type(0)      # -0.0 + 0.0 == +0.0
        u = np.dtype(f"u{got.dtype.itemsize}")
        bad |= ~nan_g & ~nan_w & (got.view(u) != want.view(u))
    else:
        bad = got != want
    if bad.any():
        idx = np.argwhere(bad)
        y, x = idx[0]
        raise AssertionError(f"{what}: {len(idx)} of {bad.size} cells differ, first at ({y}, {x}): "
                             f"got {got[y, x]!r}, want {want[y, x]!r}")


# ---- references ---------------------------------------------------------------------------------------------------
def majority_counter(image, ws, min_count=None):
    """MajorityFilter.apply restated directly: the float32 window with its four corners set to NaN, a Counter over it in
    row-major order, most_common(1), kept when count > (ws^2 - 1) * 0.7 -- or count >= min_count when one is given
    (the C ABI's parameter).  Returns (float64 result, mode count per cell; 0 on the border).

    The window travels as Python floats: float32 -> float is exact and keeps ==, so each NaN is its own key (every
    NaN is a distinct object) and -0.0 / +0.0 share one, whose sign is that of the first one inserted."""
    g = np.asarray(image).astype(np.float32)
    ny, nx = g.shape
    h = ws // 2
    out = np.zeros(g.shape)
    counts = np.zeros(g.shape, dtype=np.int64)
    rows = g.tolist()
    thr = (ws ** 2 - 1) * 0.7
    for y in range(h, ny - h):
        band = rows[y - h:y + h + 1]
        for x in range(h, nx - h):
            win = [v for r in band for v in r[x - h:x + h + 1]]
            win[0], win[ws - 1], win[-ws], win[-1] = float("nan"), float("nan"), float("nan"), float("nan")
            value, count = collections.Counter(win).most_common(1)[0]
            counts[y, x] = count
            if (count > thr) if min_count is None else (count >= min_count):
                out[y, x] = value
    return out, counts


def expand_ref(image, ws):
    """ExpandFilter.apply: 1 where any non-NaN cell of the corner-less window is > 0, 0 elsewhere and on the border."""
    pos = np.asarray(image).astype(np.float32) > 0
    h = ws // 2
    fp = np.ones((ws, ws), dtype=bool)
    fp[0, 0] = fp[0, -1] = fp[-1, 0] = fp[-1, -1] = False
    out = np.zeros(pos.shape, dtype=bool)
    out[h:pos.shape[0] - h, h:pos.shape[1] - h] = (sliding_window_view(pos, (ws, ws)) & fp).any(axis=(-1, -2))
    return out


def nanmax_reflect(a, size):
    """Maximum of the size x size window over mode='reflect' (d c b a | a b c d), NaN cells skipped."""
    h = size // 2
    view = sliding_window_view(np.pad(a, h, mode="symmetric"), (size, size))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)        # "All-NaN slice encountered": NaN, as the kernel gives
        return np.nanmax(view, axis=(-1, -2))


# ---- input generators ---------------------------------------------------------------------------------------------
def nwin(ws):
    return ws * ws - 4


def gen_threshold(shape, ws, min_count, seed):
    """Small alphabet with a biased fill: a dominant value per cell with probability p, chosen so that the mode count
    of a window is min_count - 1 or min_count about as often as anything else.  The dominant value changes in vertical
    bands so that warps also see several candidates."""
    rng = np.random.default_rng(seed)
    ny, nx = shape
    alphabet = np.array([3.0, -1.5, 7.25, 0.5], dtype=np.float32)
    p = min(1.0, (min_count - 0.5) / nwin(ws))
    dom = np.zeros(nx, dtype=np.int64)
    x = 0
    while x < nx:
        w = int(rng.integers(40, 200))
        dom[x:x + w] = rng.integers(0, len(alphabet))
        x += w
    idx = np.broadcast_to(dom, shape).copy()
    other = rng.random(shape) >= p
    idx[other] = (idx[other] + rng.integers(1, len(alphabet), int(other.sum()))) % len(alphabet)
    return alphabet[idx]


def gen_stripes(shape, ws, seed):
    """Vertical stripes of two or three plateau values, narrower than a warp, with 3 % noise: aligned 32-cell warp
    segments hold several distinct winners, so the verification loop runs once per candidate."""
    rng = np.random.default_rng(seed)
    ny, nx = shape
    levels = np.array([2.0, 5.0, 9.0][:int(rng.integers(2, 4))], dtype=np.float32)
    col = np.zeros(nx, dtype=np.float32)
    x, k = 0, 0
    while x < nx:
        w = int(rng.integers(max(2, ws - 3), 31))
        col[x:x + w] = levels[k % len(levels)]
        x, k = x + w, k + 1
    a = np.broadcast_to(col, shape).copy()
    a[rng.random(shape) < 0.03] = np.float32(-4.0)
    return a


def gen_specials(shape, seed):
    """Mostly zeros of random sign, so the winner of most windows is the +-0 class and the sign returned is that of the
    first zero in the row-major scan; 20 % other cells so that this first zero is often not the first cell.  Plateaus
    of +inf, -inf and of +-subnormals, and horizontal runs of NaN."""
    rng = np.random.default_rng(seed)
    ny, nx = shape
    a = np.where(rng.random(shape) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
    a[rng.random(shape) < 0.2] = np.float32(1.0)
    specials = np.array([np.inf, -np.inf, SUBNORMAL, -SUBNORMAL, 1.0], dtype=np.float32)
    for k in range(max(1, ny * nx // 500)):
        y, x = int(rng.integers(0, ny)), int(rng.integers(0, nx))
        hh, ww = int(rng.integers(8, 30)), int(rng.integers(8, 30))
        blk = a[y:y + hh, x:x + ww]
        blk[rng.random(blk.shape) < 0.95] = specials[k % len(specials)]
    for _ in range(max(1, ny * nx // 150)):
        y, x = int(rng.integers(0, ny)), int(rng.integers(0, nx))
        a[y, x:x + int(rng.integers(3, 11))] = np.nan
    return a


def gen_equal_distinct(shape, seed):
    """Left: one constant value (every window count = ws^2 - 4).  Right: every cell a distinct value (count 1)."""
    ny, nx = shape
    a = np.full(shape, np.float32(4.0), dtype=np.float32)
    half = nx // 2
    a[:, half:] = (np.float32(1000.0) + np.arange(ny * (nx - half), dtype=np.float32).reshape(ny, nx - half)
                   * np.float32(0.5))
    return np.ascontiguousarray(a)


def majority_inputs(shape, ws, seed):
    mc = stencils.majority_min_count(ws)
    return {"threshold": gen_threshold(shape, ws, mc, seed), "stripes": gen_stripes(shape, ws, seed + 1),
            "specials": gen_specials(shape, seed + 2), "equal_distinct": gen_equal_distinct(shape, seed + 3)}


def gen_expand(shape, ws, u8, seed):
    """Sparse positives (about one per window, so both outcomes are common and a positive often sits on a corner only)
    among cells that must not count: 0, -0.0, NaN, negatives.  F32 positives are values in (0, 1), subnormals and
    large values; U8 positives take every value 1 ... 255."""
    rng = np.random.default_rng(seed)
    pos = rng.random(shape) < 1.0 / nwin(ws)
    if u8:
        return np.where(pos, rng.integers(1, 256, shape), 0).astype(np.uint8)
    neg = np.array([0.0, -0.0, np.nan, -1.0, -SUBNORMAL, -np.inf], dtype=np.float32)
    good = np.array([0.25, 0.999, SUBNORMAL, 1.0, 300.0, np.inf], dtype=np.float32)
    return np.where(pos, good[rng.integers(0, len(good), shape)], neg[rng.integers(0, len(neg), shape)])


def gen_morph(shape, u8, seed):
    """Blobs of many sizes with salt and pepper.  True cells take non-zero values (NaN included, which scipy counts as
    True), False cells 0 or -0.0; values in (0, 1) and subnormals are True."""
    rng = np.random.default_rng(seed)
    m = ndi.uniform_filter(rng.random(shape), size=5, mode="reflect") > 0.5
    m ^= rng.random(shape) < 0.03
    if u8:
        return np.where(m, rng.integers(1, 256, shape), 0).astype(np.uint8)
    true = np.array([1.0, np.nan, 0.3, SUBNORMAL, -2.0, 255.0], dtype=np.float32)
    false = np.array([0.0, -0.0], dtype=np.float32)
    return np.where(m, true[rng.integers(0, len(true), shape)], false[rng.integers(0, 2, shape)])


def gen_grey(shape, dtype, seed):
    """NaN-free values of both signs, with zeros of both signs, subnormals and +-inf mixed in."""
    rng = np.random.default_rng(seed)
    a = (rng.standard_normal(shape) * 100).astype(dtype)
    special = np.array([0.0, -0.0, SUBNORMAL, -SUBNORMAL, np.inf, -np.inf], dtype=dtype)
    pick = rng.random(shape) < 0.05
    a[pick] = special[rng.integers(0, len(special), int(pick.sum()))]
    return a


def gen_dem(shape, dtype, seed):
    ny, nx = shape
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:ny, 0:nx]
    a = 800 + 300 * np.sin(y / 17.0) * np.cos(x / 23.0) + rng.standard_normal(shape) * 5
    return a.astype(dtype)


# ---- device calls -------------------------------------------------------------------------------------------------
def _out(ny, nx, hd):
    """An output raster filled with a value no kernel writes, so a cell the kernel skips shows up."""
    out = dev.empty(ny, nx, hd)
    if hd == _lib.U8:
        out.buf.fill_(0xAB)
    else:
        out.buf.fill_(float("nan"))
    return out


def run_majority(a, ws, out_hd, min_count):
    ny, nx = a.shape
    src, out = dev.upload(np.ascontiguousarray(a, dtype=np.float32)), _out(ny, nx, out_hd)
    _lib.check(_lib.load().hd_majority(src.ptr, src.pitch, out.ptr, out_hd, out.pitch, ny, nx, ws, min_count,
                                       dev.stream_ptr()))
    return dev.download(out)


def run_expand(a, ws, out_hd):
    ny, nx = a.shape
    src, out = dev.upload(a), _out(ny, nx, out_hd)
    _lib.check(_lib.load().hd_expand(src.ptr, src.dtype, src.pitch, out.ptr, out_hd, out.pitch, ny, nx, ws,
                                     dev.stream_ptr()))
    return dev.download(out)


def run_expand_select(a, sel, ws):
    ny, nx = a.shape
    src, s, out = dev.upload(a), dev.upload(sel), _out(ny, nx, _lib.F32)
    _lib.check(_lib.load().hd_expand_select(src.ptr, src.dtype, src.pitch, s.ptr, s.pitch, out.ptr, out.pitch, ny, nx,
                                            ws, dev.stream_ptr()))
    return dev.download(out)


def run_morph(a, op, full, iterations):
    ny, nx = a.shape
    src, out = dev.upload(a), _out(ny, nx, _lib.U8)
    _lib.check(_lib.load().hd_binary_morph(src.ptr, src.dtype, src.pitch, out.ptr, out.pitch, ny, nx, op, int(full),
                                           iterations, dev.stream_ptr()))
    return dev.download(out)


def run_max_filter(a, size):
    ny, nx = a.shape
    src = dev.upload(a)
    out = _out(ny, nx, src.dtype)
    _lib.check(_lib.load().hd_max_filter(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, ny, nx, size,
                                         dev.stream_ptr()))
    return dev.download(out)


def run_quadratic(a, ws):
    ny, nx = a.shape
    src = dev.upload(a)
    out = _out(ny, nx, src.dtype)
    _lib.check(_lib.load().hd_quadratic(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, ny, nx, ws,
                                        dev.stream_ptr()))
    return dev.download(out)


# ---- CPU: references and generators ------------------------------------------------------------------------------
_REF = {}


def majority_reference(tag, a, ws, min_count=None):
    """Counter reference, cached per input so that the F32 and F64 outputs share it."""
    key = (tag, a.shape, ws, min_count)
    if key not in _REF:
        _REF[key] = majority_counter(a, ws, min_count)
    return _REF[key]


@pytest.mark.parametrize("ws", WINDOWS)
def test_counter_reference_agrees_with_sort_oracle(ws):
    """The Counter restatement and the sort-based oracle give the same values (== treats -0.0 as 0.0: the oracle's
    sign of a zero winner comes from an unstable sort)."""
    shape = (40, 90)
    for tag, a in majority_inputs(shape, ws, 100 + ws).items():
        got, _ = majority_counter(a, ws)
        np.testing.assert_array_equal(got, stencils.majority(a, ws), err_msg=f"{tag} ws={ws}")


def _warp_segments_with_winners(result):
    """Number of aligned 32-cell segments of an output row that hold >= 2 distinct non-zero winners."""
    ny, nx = result.shape
    n = 0
    for y in range(ny):
        for x0 in range(0, nx, 32):
            seg = result[y, x0:x0 + 32]
            if len(np.unique(seg[seg != 0])) >= 2:
                n += 1
    return n


@pytest.mark.parametrize("ws", [5, 9, 11, 15])
def test_majority_generators_reach_their_edges(ws):
    shape = SEAMS[2]
    mc = stencils.majority_min_count(ws)
    inputs = majority_inputs(shape, ws, 7 * ws)
    res, counts = majority_counter(inputs["threshold"], ws)
    assert (counts == mc - 1).sum() >= 300 and (counts == mc).sum() >= 300, \
        ((counts == mc - 1).sum(), (counts == mc).sum())
    res, _ = majority_counter(inputs["stripes"], ws)
    assert _warp_segments_with_winners(res) >= 100
    a = inputs["specials"]
    res, counts = majority_counter(a, ws)
    zero = (res == 0) & (counts > (ws ** 2 - 1) * 0.7)
    assert (zero & np.signbit(res)).sum() >= 100 and (zero & ~np.signbit(res)).sum() >= 100
    for v in (np.inf, -np.inf, SUBNORMAL, -SUBNORMAL):
        assert (res == v).sum() >= 5, v
    assert np.isnan(a).sum() >= 100
    assert (a != 0).mean() > 0.15          # so the first zero of the scan is often not the first non-corner cell
    res, counts = majority_counter(inputs["equal_distinct"], ws)
    h = ws // 2
    assert (counts[h:-h, h:-h] == nwin(ws)).sum() >= 100 and (counts[h:-h, h:-h] == 1).sum() >= 100


@pytest.mark.parametrize("ws", [3, 9, 15])
def test_window_generators_reach_their_edges(ws):
    shape = SEAMS[2]
    h = ws // 2
    for u8 in (False, True):
        a = gen_expand(shape, ws, u8, ws)
        e = expand_ref(a, ws)[h:-h, h:-h]
        assert 0.1 < e.mean() < 0.9, e.mean()
        # windows whose only positive cell sits on a corner: the corner rule decides them
        pos = a.astype(np.float32) > 0
        corners = sliding_window_view(pos, (ws, ws))[..., [0, 0, -1, -1], [0, -1, 0, -1]].any(axis=-1)
        assert (corners & ~e).sum() >= 20
    a = gen_expand(shape, ws, False, ws)
    for v in (SUBNORMAL, -SUBNORMAL, np.float32(0.25)):
        assert (a == v).sum() >= 5, v
    assert np.isnan(a).sum() >= 100 and (np.signbit(a) & (a == 0)).sum() >= 100
    m = gen_morph(shape, False, ws)
    assert np.isnan(m).sum() >= 100 and ((m == 0) & np.signbit(m)).sum() >= 100 and (m == SUBNORMAL).sum() >= 100
    assert 0.3 < (m != 0).mean() < 0.7


def test_abi_refuses_what_it_does_not_support():
    """The smallest min_count below an absolute majority and iteration counts beyond the cap are refused before any
    device work."""
    if not os.path.exists(_lib.LIB_PATH):
        from hydrodem_b200.build import build
        build()
    lib = _lib.load()
    p = ctypes.c_void_p(1 << 20)
    for ws in WINDOWS:
        below = (ws * ws - 4) // 2
        assert lib.hd_majority(p, 64, p, _lib.F32, 64, 64, 64, ws, below, None) == _lib.HD_ERR_UNSUPPORTED
    for op, cap in ((_lib.MORPH_ERODE, 8), (_lib.MORPH_DILATE, 8), (_lib.MORPH_CLOSE, 4), (_lib.MORPH_OPEN, 4)):
        for dt in (_lib.U8, _lib.F32):
            assert lib.hd_binary_morph(p, dt, 256, p, 256, 64, 64, op, 0, cap + 1, None) == _lib.HD_ERR_UNSUPPORTED


# ---- GPU: majority ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("out_hd", [_lib.F32, _lib.F64], ids=["f32", "f64"])
@pytest.mark.parametrize("ws", WINDOWS)
@gpu
def test_majority_every_window_and_output(ws, out_hd):
    mc = stencils.majority_min_count(ws)
    for shape in shapes_for(ws):
        for tag, a in majority_inputs(shape, ws, shape[0] * 7 + shape[1] + ws).items():
            want, _ = majority_reference(tag, a, ws)
            got = run_majority(a, ws, out_hd, mc)
            bits_equal(got, want.astype(F32_OUT[out_hd]), f"ws={ws} {shape} {tag}")


@pytest.mark.parametrize("ws", WINDOWS)
@gpu
def test_majority_class_every_window(ws):
    """The drop-in class: its own threshold and the widening to float64 on download."""
    a = gen_specials(SEAMS[0], 500 + ws)
    want, _ = majority_reference("class", a, ws)
    got = cf.MajorityFilter(window_size=ws).apply(a)
    bits_equal(got, want, f"MajorityFilter(window_size={ws})")


@pytest.mark.parametrize("ws", [5, 11])
@gpu
def test_majority_min_count_range(ws):
    """min_count from the smallest value the kernel accepts (an absolute majority of the ws^2 - 4 cells) through the
    reference threshold to ws^2 - 4, each on inputs biased to sit at that count."""
    n = nwin(ws)
    for mc in (stencils.majority_min_count(ws), n // 2 + 1, n):
        for shape in (SEAMS[0], SEAMS[2]):
            a = gen_threshold(shape, ws, mc, mc)
            if mc == n:
                a[:, :shape[1] // 3] = np.float32(3.0)          # whole windows of one value
            want, counts = majority_reference(f"mc{mc}", a, ws, mc)
            assert (counts == mc).sum() >= 10 and (counts == mc - 1).sum() >= 10
            for out_hd in (_lib.F32, _lib.F64):
                got = run_majority(a, ws, out_hd, mc)
                bits_equal(got, want.astype(F32_OUT[out_hd]), f"ws={ws} min_count={mc} {shape}")
    lib = _lib.load()
    src, out = dev.upload(np.zeros(SEAMS[0], np.float32)), _out(*SEAMS[0], _lib.F32)
    assert lib.hd_majority(src.ptr, src.pitch, out.ptr, _lib.F32, out.pitch, *SEAMS[0], ws, n // 2,
                           dev.stream_ptr()) == _lib.HD_ERR_UNSUPPORTED


@gpu
def test_majority_more_tiles_than_grid():
    """845 tiles: every CTA of the persistent grid loops, through both stage buffers.  Values from the C oracle; the
    inputs hold no zero, so there is no sign of zero to check."""
    ws = 11
    mc = stencils.majority_min_count(ws)
    a = gen_threshold(BIG, ws, mc, 2049)
    a[:, :600] = gen_stripes((BIG[0], 600), ws, 1537)
    want = clib.majority(a, ws, mc)
    assert (want != 0).sum() > 100000
    for out_hd in (_lib.F32, _lib.F64):
        bits_equal(run_majority(a, ws, out_hd, mc), want.astype(F32_OUT[out_hd]), f"{BIG}")


# ---- GPU: expand --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("in_u8", [False, True], ids=["in_f32", "in_u8"])
@pytest.mark.parametrize("ws", WINDOWS)
@gpu
def test_expand_every_window_and_dtype(ws, in_u8):
    for shape in shapes_for(ws):
        a = gen_expand(shape, ws, in_u8, shape[0] * 3 + shape[1] + ws)
        want = expand_ref(a, ws)
        for out_hd, dt in ((_lib.U8, np.uint8), (_lib.F32, np.float32), (_lib.F64, np.float64)):
            bits_equal(run_expand(a, ws, out_hd), want.astype(dt), f"ws={ws} {shape} out={dt.__name__}")
        sel = gen_grey(shape, np.float32, ws)
        sel[::7, ::3] = np.nan
        sel[1::5, ::2] = -np.abs(sel[1::5, ::2]) - 1
        prod = sel * want.astype(np.float32)
        assert np.signbit(prod[prod == 0]).any() and np.isnan(prod).any()
        bits_equal(run_expand_select(a, sel, ws), prod, f"select ws={ws} {shape}")


@gpu
def test_expand_more_tiles_than_grid():
    ws = 7
    for in_u8 in (False, True):
        a = gen_expand(BIG, ws, in_u8, 11)
        want = clib.expand(a, ws)
        bits_equal(run_expand(a, ws, _lib.F64), want, f"{BIG} u8={in_u8}")
        bits_equal(run_expand(a, ws, _lib.U8), want.astype(np.uint8), f"{BIG} u8={in_u8}")


# ---- GPU: binary morphology ---------------------------------------------------------------------------------------
MORPH_CASES = ([(_lib.MORPH_ERODE, n) for n in range(1, 9)] + [(_lib.MORPH_DILATE, n) for n in range(1, 9)]
               + [(_lib.MORPH_CLOSE, n) for n in range(1, 5)] + [(_lib.MORPH_OPEN, n) for n in range(1, 5)])
MORPH_NAMES = {_lib.MORPH_ERODE: "erode", _lib.MORPH_DILATE: "dilate", _lib.MORPH_CLOSE: "close",
               _lib.MORPH_OPEN: "open"}
SCIPY_MORPH = {_lib.MORPH_ERODE: ndi.binary_erosion, _lib.MORPH_DILATE: ndi.binary_dilation,
               _lib.MORPH_CLOSE: ndi.binary_closing, _lib.MORPH_OPEN: ndi.binary_opening}
CROSS = ndi.generate_binary_structure(2, 1)


@pytest.mark.parametrize("op,iterations", MORPH_CASES, ids=[f"{MORPH_NAMES[o]}{n}" for o, n in MORPH_CASES])
@gpu
def test_binary_morph_every_op_and_iteration(op, iterations):
    steps = iterations * (2 if op in (_lib.MORPH_CLOSE, _lib.MORPH_OPEN) else 1)
    span = 2 * steps + 1
    for shape in [(span, span), (span, 300), (300, span)] + SEAMS:
        for full in (False, True):
            st = np.ones((3, 3), dtype=bool) if full else CROSS
            for u8 in (False, True):
                a = gen_morph(shape, u8, shape[0] + shape[1] * 5 + op * 11 + iterations)
                want = SCIPY_MORPH[op](a, structure=st, iterations=iterations, border_value=0).astype(np.uint8)
                got = run_morph(a, op, full, iterations)
                bits_equal(got, want, f"{MORPH_NAMES[op]} x{iterations} full={full} u8={u8} {shape}")


@gpu
def test_binary_morph_more_tiles_than_grid():
    for op, it in ((_lib.MORPH_DILATE, 3), (_lib.MORPH_OPEN, 2)):
        a = gen_morph(BIG, False, op)
        want = SCIPY_MORPH[op](a, structure=np.ones((3, 3), bool), iterations=it, border_value=0).astype(np.uint8)
        bits_equal(run_morph(a, op, True, it), want, f"{MORPH_NAMES[op]} {BIG}")


# ---- GPU: grey dilation -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("size", list(range(1, 18, 2)))
@gpu
def test_max_filter_every_size(size, dtype):
    """scipy.ndimage.grey_dilation(size=(s, s), mode='reflect'); the sign of a zero maximum is not compared."""
    for shape in shapes_for(size):
        a = gen_grey(shape, dtype, size * 1000 + shape[0] + shape[1])
        want = ndi.grey_dilation(a, size=(size, size), mode="reflect")
        bits_equal(run_max_filter(a, size), want, f"size={size} {shape}", zero_sign=False)


@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@gpu
def test_max_filter_skips_nan(dtype):
    """The header's rule: NaN cells are skipped by the maximum (a window of NaN only gives NaN)."""
    for size in (3, 7, 9):
        a = gen_grey(SEAMS[2], dtype, size)
        rng = np.random.default_rng(size)
        a[rng.random(a.shape) < 0.2] = np.nan
        a[10:25, 40:70] = np.nan
        bits_equal(run_max_filter(a, size), nanmax_reflect(a, size), f"size={size}", zero_sign=False)


@gpu
def test_max_filter_more_tiles_than_grid():
    for size, dtype in ((9, np.float32), (7, np.float32), (5, np.float64)):
        a = gen_grey(BIG, dtype, size)
        want = ndi.grey_dilation(a, size=(size, size), mode="reflect")
        bits_equal(run_max_filter(a, size), want, f"size={size} {BIG}", zero_sign=False)


# ---- GPU: quadratic -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("ws", WINDOWS)
@gpu
def test_quadratic_every_window(ws, dtype):
    """Tolerance class: 1e-5 relative (DESIGN.md section 2, A5)."""
    for shape in shapes_for(ws):
        a = gen_dem(shape, dtype, ws + shape[0])
        got = run_quadratic(a, ws)
        assert got.dtype == a.dtype
        np.testing.assert_allclose(got, stencils.quadratic(a, ws), rtol=1e-5, err_msg=f"ws={ws} {shape}")


@gpu
def test_quadratic_more_tiles_than_grid():
    a = gen_dem(BIG, np.float32, 5)
    np.testing.assert_allclose(run_quadratic(a, 5), stencils.quadratic(a, 5), rtol=1e-5)

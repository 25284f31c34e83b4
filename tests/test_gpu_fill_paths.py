"""Sink-fill and D8 on the inputs where the worklist, the multigrid start and the banded Schwarz loop go wrong, against
exact fixed points, on one GPU and on row bands.

The fill (csrc/hydro.cu) has three parts that synthetic terrain barely reaches: the asynchronous worklist (persistent
CTAs, the poke / ticket protocol, the spin limit), the multigrid start from 8x8 block maxima and, on row bands, the
overlapping Schwarz loop.  The inputs here are built to reach them:

  * serpentine mazes: one-cell corridors between one-cell walls of +inf, one outlet on the frame.  Every 8x8 block holds
    a wall, so every block maximum is +inf and the multigrid start contributes nothing: the worklist has to carry the
    whole wave, tile after tile, along a path of up to 1.57 M cells.  On row bands a column maze crosses every cut once
    per corridor, so the Schwarz loop needs one round per crossing;
  * special values (+-0, +-1, +-1e-45, +-inf, NaN, the float32 extremes) on the tile and block seam shapes, and whole
    rasters of them (all NaN, all +inf, a NaN frame, a -inf interior, ...);
  * degenerate shapes from 1 x 1 up to 3 x 20000, float64 / int16 / uint8 input, and device views whose column offset
    puts the fill on its scalar load path.

A maze has a closed-form fixed point that needs no fill algorithm: the filled surface is the running maximum of the
floor along the corridor, measured from the outlet (with an outlet at either end, or a NaN cell inside the corridor, the
minimum of the two running maxima).  The row-end cells next to a turn can be bypassed diagonally; their floor is -inf,
so the bypass cannot matter.  On the CPU the closed form is checked against both oracles (priority flood, and the
iterative Planchon-Darboux on small mazes), and on special-value grids the two oracles are checked against each other.

The two oracles agree on every value and every NaN position but not on the sign of a zero, and the GPU's racy update
order leaves that sign to the schedule; the fill therefore writes every zero as +0.0 (DESIGN.md section 6).  Results
are compared with the oracles with zero signs folded, and with each other (one CTA or four per SM, SinkFill against
SinkFillD8, a repeated run, one GPU against row bands) bit for bit, sign of zero included.

CPU checks carry no mark; the tests that need the device carry `gpu`."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import clib, hydrology


def gpu(test):
    """Marks one test as needing the device (the CPU tests of this file carry no mark)."""
    return pytest.mark.gpu(pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")(test))


if torch.cuda.is_available():
    from hydrodem_b200 import _lib, device as dev, sharding
    from hydrodem_b200.exceptions import DeviceError
    from hydrodem_b200.filters import new_filters as nf

INF = np.float32(np.inf)
F32_MAX = np.finfo(np.float32).max
F32_TINY = np.finfo(np.float32).tiny                 # smallest normal
SUB = np.float32(1e-45)                              # smallest subnormal
FLOORS = np.array([0.0, -0.0, 1e-45, -2.0, 3.0, 7.5, 100.0, 1.7e38], dtype=np.float32)
SPECIALS = np.array([0.0, -0.0, 1.0, -1.0, 1e-45, -1e-45, np.inf, -np.inf, np.nan, F32_MAX, -F32_MAX, F32_TINY,
                     -F32_TINY], dtype=np.float32)
SEAMS = [(63, 65), (64, 64), (65, 129), (200, 333)]
DEGENERATE = [(1, 1), (1, 2), (1, 300), (300, 1), (2, 2), (2, 300), (300, 2), (3, 3), (7, 9), (8, 8), (9, 9),
              (3, 20000), (20000, 3)]


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


def negative_zeros(a):
    return int(((a == 0) & np.signbit(a)).sum())


# ---- mazes --------------------------------------------------------------------------------------------------------
class Maze:
    """A serpentine maze and its closed-form fill.

    z: float32 raster; path: (n, 2) cell coordinates in corridor order, outlets included; kind: per path cell 0 =
    floor, 1 = frame outlet (W = z), 2 = NaN cell (an outlet at -inf that stays NaN)."""

    def __init__(self, z, path, kind):
        self.z, self.path, self.kind = z, path, kind

    @property
    def shape(self):
        return self.z.shape

    def fill(self):
        """The closed form: per path cell the smaller of the running maxima of the floor from the nearest outlet
        before it and after it along the corridor; walls keep +inf, NaN cells stay NaN."""
        ys, xs = self.path[:, 0], self.path[:, 1]
        lev = self.z[ys, xs].copy()
        lev[self.kind == 2] = -INF
        outlet = self.kind != 0

        def running(lv, out):
            r = np.full(len(lv), INF, dtype=np.float32)        # no outlet before the cell: +inf
            cuts = list(np.flatnonzero(out)) + [len(lv)]
            for a, b in zip(cuts[:-1], cuts[1:]):
                r[a:b] = np.maximum.accumulate(lv[a:b])
            return r

        w = np.minimum(running(lev, outlet), running(lev[::-1], outlet[::-1])[::-1])
        out = np.full(self.shape, INF, dtype=np.float32)
        out[ys, xs] = w
        out[np.isnan(self.z)] = np.nan
        return out


def maze(ny, nx, *, cols=False, side="left", second_outlet=False, nan_at=None, seed=0):
    """Serpentine maze of ny x nx cells.  cols: the corridors run along columns (the transpose of a row maze); side:
    the frame side of the outlet ("left", "right", "top", "bottom"); second_outlet: another frame outlet at the far
    end of the corridor; nan_at: a NaN cell at that fraction of the corridor.  Floors: mostly a ramp that rises along
    the corridor (so that the running maximum keeps changing), a third of them drawn from FLOORS."""
    if cols:                                            # transpose of a row maze: the sides swap with the axes
        t = maze(nx, ny, side={"left": "top", "right": "bottom", "top": "left", "bottom": "right"}[side],
                 second_outlet=second_outlet, nan_at=nan_at, seed=seed)
        return Maze(np.ascontiguousarray(t.z.T), t.path[:, ::-1].copy(), t.kind)
    flip_y, flip_x = side == "bottom", side == "right"
    base = "top" if side in ("top", "bottom") else "left"
    assert ny >= 3 and nx >= 5, (ny, nx)
    rng = np.random.default_rng(seed)
    z = np.full((ny, nx), INF, dtype=np.float32)
    path = [(0, 1) if base == "top" else (1, 0)]       # the outlet first
    end_x = None
    for i, y in enumerate(range(1, ny - 1, 2)):
        xs = range(1, nx - 1) if i % 2 == 0 else range(nx - 2, 0, -1)
        if end_x is not None:
            path.append((y - 1, end_x))                 # the turn gap in the wall row above
        path += [(y, x) for x in xs]
        end_x = xs[-1]
    if second_outlet:
        last_y = path[-1][0]
        path.append((last_y, nx - 1 if end_x == nx - 2 else 0))
    path = np.array(path, dtype=np.int64)
    n = len(path)
    kind = np.zeros(n, dtype=np.int8)
    kind[0] = 1
    if second_outlet:
        kind[-1] = 1
    ramp = np.floor(np.arange(n) * (60.0 / n) + rng.integers(-3, 4, n)).astype(np.float32)
    floor = np.where(rng.random(n) < 1 / 3, FLOORS[rng.integers(0, len(FLOORS), n)], ramp).astype(np.float32)
    floor[n - max(1, n // 50):] = np.where(rng.random(max(1, n // 50)) < 0.1, np.float32(1.7e38),
                                           floor[n - max(1, n // 50):])
    floor[kind == 1] = FLOORS[rng.integers(0, 3, int(kind.sum()))]        # outlets at +0, -0 or 1e-45
    # cells that a later path cell touches diagonally can be bypassed: -inf, so that the bypass cannot matter
    index = -np.ones((ny, nx), dtype=np.int64)
    index[path[:, 0], path[:, 1]] = np.arange(n)
    for k, (y, x) in enumerate(path):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                yy, xx = y + dy, x + dx
                if 0 <= yy < ny and 0 <= xx < nx and index[yy, xx] > k + 1:
                    floor[k + 1:index[yy, xx]] = -INF
    z[path[:, 0], path[:, 1]] = floor
    if nan_at is not None:
        m = int(n * nan_at)
        while kind[m] or floor[m] == -INF:
            m += 1
        z[path[m, 0], path[m, 1]] = np.nan
        kind[m] = 2
    if flip_y:
        z, path[:, 0] = z[::-1], ny - 1 - path[:, 0]
    if flip_x:
        z, path[:, 1] = z[:, ::-1], nx - 1 - path[:, 1]
    return Maze(np.ascontiguousarray(z), path, kind)


def check_maze(m):
    """The maze is what the closed form assumes: a simple 8-connected chain of distinct cells; path cells that are not
    consecutive touch only where every cell between them is -inf; outlets on the frame; walls (+inf) at or above
    every floor."""
    ny, nx = m.shape
    p = m.path
    assert len({(int(y), int(x)) for y, x in p}) == len(p)
    assert (np.abs(np.diff(p, axis=0)).max(axis=1) == 1).all()                         # 8-connected chain
    index = -np.ones(m.shape, dtype=np.int64)
    index[p[:, 0], p[:, 1]] = np.arange(len(p))
    floor = m.z[p[:, 0], p[:, 1]]
    for k, (y, x) in enumerate(p):
        nb = index[max(0, y - 1):y + 2, max(0, x - 1):x + 2]
        for j in nb[nb > k + 1]:
            assert (floor[k + 1:j] == -INF).all(), ("shortcut", k, int(j))
    for y, x in p[m.kind == 1]:
        assert y in (0, ny - 1) or x in (0, nx - 1)
    assert not np.isnan(floor[m.kind != 2]).any() and np.isnan(floor[m.kind == 2]).all()
    walls = m.z[index < 0]
    assert (walls == INF).all() and walls.min() >= floor[m.kind != 2].max()


MAZES_CPU = [dict(ny=33, nx=41), dict(ny=40, nx=33, cols=True, side="top"), dict(ny=17, nx=129, side="right"),
             dict(ny=31, nx=35, side="bottom", second_outlet=True), dict(ny=35, nx=30, cols=True, nan_at=0.5),
             dict(ny=257, nx=130, side="top", second_outlet=True, nan_at=0.3)]


@pytest.mark.parametrize("kw", MAZES_CPU, ids=lambda kw: "-".join(f"{k}{v}" for k, v in kw.items()))
def test_maze_closed_form_matches_both_oracles(kw):
    """The closed form equals the priority flood, and (up to about 64 x 64: one Jacobi sweep per path cell) the
    iterative Planchon-Darboux fixed point, with zero signs folded."""
    m = maze(**kw, seed=5)
    check_maze(m)
    want = m.fill()
    assert np.isfinite(want).sum() > len(m.path) // 2
    bits_equal(hydrology.sinkfill(m.z), want, f"priority flood {kw}", zero_sign=False)
    if max(m.shape) <= 64:
        it, sweeps = hydrology.sinkfill_iterative(m.z)
        bits_equal(it, want, f"iterative {kw}", zero_sign=False)
        assert sweeps > len(m.path) // 4                  # the wave really runs the whole corridor


@pytest.mark.parametrize("side", ["left", "right", "top", "bottom"])
@pytest.mark.parametrize("cols", [False, True])
def test_maze_generator_sides(side, cols):
    """Every outlet side in both orientations: the outlet is on that side of the frame and the fill matches the
    priority flood."""
    m = maze(23, 27, cols=cols, side=side, second_outlet=True, seed=3)
    check_maze(m)
    y, x = m.path[0]
    ny, nx = m.shape
    assert {"left": x == 0, "right": x == nx - 1, "top": y == 0, "bottom": y == ny - 1}[side]
    bits_equal(hydrology.sinkfill(m.z), m.fill(), f"{side} {cols}", zero_sign=False)


def test_maze_needs_a_long_wave_and_no_coarse_help():
    """Walls of +inf put +inf into every 8x8 block maximum (the multigrid start learns nothing), and the filled
    corridor holds values the wave has carried from the outlet across the whole raster."""
    m = maze(129, 257, seed=9)
    ny, nx = m.shape
    blocks = np.pad(m.z, ((0, -ny % 8), (0, -nx % 8)), constant_values=INF).reshape(-(-ny // 8), 8, -(-nx // 8), 8)
    assert (blocks.max(axis=(1, 3)) == INF).all()
    w = m.fill()
    far = m.path[-1]
    assert np.isfinite(w[far[0], far[1]])


# ---- special values -----------------------------------------------------------------------------------------------
def special_grid(shape, seed, values=SPECIALS):
    rng = np.random.default_rng(seed)
    return values[rng.integers(0, len(values), shape)].astype(np.float32)


def whole_raster_cases(ny, nx, seed=0):
    """Rasters made of one kind of value, or of one value inside a frame of another."""
    rng = np.random.default_rng(seed)
    r = special_grid((ny, nx), seed)
    frame = np.zeros((ny, nx), dtype=bool)
    frame[0, :] = frame[-1, :] = frame[:, 0] = frame[:, -1] = True
    sub = (rng.integers(1, 8, (ny, nx)) * rng.choice([-1, 1], (ny, nx)) * SUB).astype(np.float32)
    cases = {"all_nan": np.full((ny, nx), np.nan, np.float32), "all_inf": np.full((ny, nx), INF),
             "zeros": np.zeros((ny, nx), np.float32), "neg_zeros": np.full((ny, nx), -0.0, np.float32),
             "nan_frame": np.where(frame, np.float32(np.nan), r), "nan_inside": np.where(frame, r, np.float32(np.nan)),
             "ninf_inside": np.where(frame, r, -INF), "subnormal": sub,
             "mixed_zeros": np.where(rng.random((ny, nx)) < 0.5, np.float32(0.0), np.float32(-0.0))}
    return {k: v.astype(np.float32) for k, v in cases.items()}


@pytest.mark.parametrize("seed", range(6))
def test_oracles_agree_on_special_values(seed):
    """On grids of {+-0, +-1, +-1e-45, +-inf, NaN, float32 extremes} the priority flood and the iterative fill agree on
    every value and every NaN position (not on the sign of a zero): the contract the device fill is held to."""
    shape = [(23, 31), (63, 65), (64, 64), (9, 9), (3, 40), (40, 3)][seed]
    z = special_grid(shape, seed)
    bits_equal(hydrology.sinkfill(z), hydrology.sinkfill_iterative(z)[0], f"specials {shape}", zero_sign=False)
    for name, c in whole_raster_cases(*shape, seed).items():
        bits_equal(hydrology.sinkfill(c), hydrology.sinkfill_iterative(c)[0], f"{name} {shape}", zero_sign=False)


def test_zero_sign_is_not_pinned_by_the_oracles():
    """Why the sign of a zero needs a rule of its own: on signed-zero grids the two oracles do not agree on it."""
    diff = 0
    for seed in range(5):
        z = special_grid((23, 31), seed, np.array([0.0, -0.0, 1.0, -1.0, 1e-45, -1e-45, np.inf, -np.inf, np.nan],
                                                   dtype=np.float32))
        a, b = hydrology.sinkfill(z), hydrology.sinkfill_iterative(z)[0]
        bits_equal(a, b, "specials", zero_sign=False)
        diff += int((np.signbit(a) != np.signbit(b))[a == 0].sum())
    assert diff > 0


# ---- one GPU ------------------------------------------------------------------------------------------------------
def _status(work):
    st = ctypes.c_int(-1)
    _lib.check(_lib.load().hd_pdfill_status(ctypes.c_void_p(work.data_ptr()), ctypes.byref(st), dev.stream_ptr()))
    return st.value


def run_fill(z):
    """SinkFill, SinkFillD8 and D8FlowDirection on z: (filled, filled of the fused call, d8 of the fused call, d8 of
    the separate pass), each status word checked."""
    f = nf.SinkFill()
    w1 = f.apply(z)
    assert _status(f._work) == 0
    fd = nf.SinkFillD8()
    w2, d2 = fd.apply(z)
    assert fd.status() == 0
    d1 = nf.D8FlowDirection().apply(w1)
    return w1, w2, d2, d1


def check_fill(z, want, what):
    """Every device path against the oracle's fill (zero signs folded) and the oracles' D8, the two fills against each
    other bit for bit, and no -0.0 anywhere in the result."""
    w1, w2, d2, d1 = run_fill(z)
    bits_equal(w1, want, f"SinkFill {what}", zero_sign=False)
    bits_equal(w2, want, f"SinkFillD8 {what}", zero_sign=False)
    bits_equal(w1, w2, f"SinkFill vs SinkFillD8 {what}")
    assert negative_zeros(w1) == 0 and negative_zeros(w2) == 0, what
    d_want = hydrology.d8(want)
    bits_equal(clib.d8(want), d_want, f"the two D8 oracles {what}")
    bits_equal(d1, d_want, f"D8FlowDirection {what}")
    bits_equal(d2, d_want, f"fused D8 {what}")
    return w1


MAZES_GPU = [dict(ny=17, nx=129), dict(ny=129, nx=17, cols=True, side="bottom"),
             dict(ny=200, nx=333, side="right", second_outlet=True), dict(ny=333, nx=200, cols=True, nan_at=0.6),
             dict(ny=2049, nx=1537, side="top"), dict(ny=2049, nx=1537, cols=True, side="left", nan_at=0.8),
             dict(ny=5, nx=131073), dict(ny=131073, nx=5, cols=True, side="right")]


@gpu
@pytest.mark.parametrize("ctas", ["1", "4"])
@pytest.mark.parametrize("kw", MAZES_GPU, ids=lambda kw: "-".join(f"{k}{v}" for k, v in kw.items()))
def test_maze_fill(kw, ctas, monkeypatch):
    """The worklist alone carries the wave along corridors of up to 1.57 M cells (2049 x 1537), or 262 k cells through
    a raster with three coarse levels (5 x 131073): the closed form, bit for bit, with one and four CTAs per SM."""
    monkeypatch.setenv("HD_FILL_CTAS_PER_SM", ctas)
    m = maze(**kw, seed=11)
    want = m.fill()
    bits_equal(hydrology.sinkfill(m.z), want, "oracle", zero_sign=False)
    check_fill(m.z, want, str(kw))


@gpu
@pytest.mark.parametrize("shape", SEAMS)
def test_special_values_on_seams(shape):
    for seed in range(3):
        z = special_grid(shape, seed)
        check_fill(z, hydrology.sinkfill(z), f"specials {shape} seed {seed}")


@gpu
@pytest.mark.parametrize("shape", [(64, 64), (65, 129), (200, 333)])
def test_whole_raster_special_cases(shape):
    for name, z in whole_raster_cases(*shape).items():
        want = hydrology.sinkfill(z)
        check_fill(z, want, f"{name} {shape}")
        if max(shape) <= 129:
            bits_equal(hydrology.sinkfill_iterative(z)[0], want, f"iterative {name}", zero_sign=False)


@gpu
@pytest.mark.parametrize("shape", DEGENERATE, ids=lambda s: f"{s[0]}x{s[1]}")
def test_degenerate_shapes(shape):
    """Single rows and columns, rasters thinner than one 8-row coarse block, a 3 x 20000 strip with two coarse levels."""
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    z = rng.integers(0, 10, shape).astype(np.float32)
    z[rng.random(shape) < 0.05] = np.nan
    z[rng.random(shape) < 0.05] = -0.0
    z[rng.random(shape) < 0.02] = np.inf
    check_fill(z, hydrology.sinkfill(z), f"{shape}")
    s = special_grid(shape, 1)
    check_fill(s, hydrology.sinkfill(s), f"specials {shape}")


@gpu
def test_input_dtypes():
    """float64 (values that round on the cast to float32 and values beyond its range), int16 and uint8 input: the fill
    of astype(np.float32)."""
    rng = np.random.default_rng(4)
    shape = (130, 197)
    z64 = rng.integers(0, 50, shape).astype(np.float64) + np.array([0.0, 0.1, 1 + 2.0 ** -30, 1e-300])[
        rng.integers(0, 4, shape)]
    z64[rng.random(shape) < 0.02] = 1e39
    z64[rng.random(shape) < 0.02] = -1e39
    z64[rng.random(shape) < 0.02] = -1e-50                  # rounds to -0.0
    z64[rng.random(shape) < 0.02] = np.nan
    z64[40:60, 50:90] -= 30
    assert (z64.astype(np.float32).astype(np.float64) != z64).sum() > 1000
    z16 = rng.integers(-32768, 32767, shape, dtype=np.int64).astype(np.int16)
    z16[40:60, 50:90] = -32768
    z8 = rng.integers(0, 256, shape).astype(np.uint8)
    z8[40:60, 50:90] = 0
    for z in (z64, z16, z8):
        f32 = z.astype(np.float32)
        w = check_fill(z, hydrology.sinkfill(f32), str(z.dtype))
        assert w.dtype == np.float32


def _upload_offset(a, off):
    """A device view of ``a`` whose first column sits ``off`` cells after an aligned row start (same pitch)."""
    ny, nx = a.shape
    wide = np.zeros((ny, nx + off), dtype=a.dtype)
    wide[:, off:] = a
    return dev.upload(wide).sub(0, ny, off, off + nx)


@gpu
@pytest.mark.parametrize("off", [1, 2, 3])
def test_unaligned_views(off):
    """z and W at column offsets 1, 2, 3 (no 16-byte loads or stores: the scalar paths of fill_async_kernel and the
    finish passes): the oracle's bits, or a clean DeviceError -- never other bits."""
    lib = _lib.load()
    for what, z in (("maze", maze(67, 131, side="right", seed=off).z), ("specials", special_grid((130, 257), off))):
        want = hydrology.sinkfill(z)
        d_want = hydrology.d8(want)
        ny, nx = z.shape
        zv = _upload_offset(z, off)
        try:
            w1 = nf.SinkFill().run_device(zv)
            w2, d2 = nf.SinkFillD8().run_device(zv)
            d1 = nf.D8FlowDirection().run_device(_upload_offset(dev.download(w1), off))
            # W and the flow directions written through views at the same offset
            wv = dev.empty(ny, nx + off, _lib.F32).sub(0, ny, off, off + nx)
            dv = dev.empty(ny, nx + off, _lib.U8).sub(0, ny, off, off + nx)
            nbytes = lib.hd_pdfill_workspace_bytes(ny, nx)
            work = dev.scratch(nbytes)
            _lib.check(lib.hd_pdfill_d8(zv.ptr, zv.pitch, wv.ptr, wv.pitch, dv.ptr, dv.pitch, ny, nx,
                                        ctypes.c_void_p(work.data_ptr()), nbytes, None, dev.stream_ptr()))
            assert _status(work) == 0
            w3, d3 = dev.download(wv), dev.download(dv)
            _lib.check(lib.hd_pdfill(zv.ptr, zv.pitch, wv.ptr, wv.pitch, ny, nx, ctypes.c_void_p(work.data_ptr()),
                                     nbytes, None, dev.stream_ptr()))
            assert _status(work) == 0
            w4 = dev.download(wv)
        except DeviceError:
            continue                                      # a refusal is a clean answer; other bits are not
        for k, w in enumerate((dev.download(w1), dev.download(w2), w3, w4)):
            bits_equal(w, want, f"{what} offset {off} fill {k}", zero_sign=False)
            assert negative_zeros(w) == 0
        for k, d in enumerate((dev.download(d1), dev.download(d2), d3)):
            bits_equal(d, d_want, f"{what} offset {off} d8 {k}")


# ---- determinism --------------------------------------------------------------------------------------------------
def zero_heavy(shape, seed):
    """Signed zeros in pits, on the frame and under NaN outlets: many cells whose fill is a zero of either sign."""
    rng = np.random.default_rng(seed)
    z = np.where(rng.random(shape) < 0.5, np.float32(0.0), np.float32(-0.0)).astype(np.float32)
    z[rng.random(shape) < 0.15] = 1.0
    z[rng.random(shape) < 0.05] = -1e-45
    z[rng.random(shape) < 0.02] = np.nan
    z[rng.random(shape) < 0.05] = np.inf
    return z


@gpu
@pytest.mark.parametrize("shape", [(200, 333), (700, 900)])
def test_fill_is_deterministic_to_the_sign_of_zero(shape, monkeypatch):
    """One CTA against four per SM, SinkFill against SinkFillD8 and a repeated run: the same bits, sign of zero
    included, and every zero of the result is +0.0."""
    cases = [zero_heavy(shape, 1), maze(*shape, seed=2).z, special_grid(shape, 3)]
    for k, z in enumerate(cases):
        want = hydrology.sinkfill(z)
        runs = {}
        for ctas in ("1", "4"):
            monkeypatch.setenv("HD_FILL_CTAS_PER_SM", ctas)
            runs[ctas] = run_fill(z)
            runs[ctas + "again"] = run_fill(z)
        ref = runs["4"][0]
        bits_equal(ref, want, f"case {k}", zero_sign=False)
        assert negative_zeros(ref) == 0
        assert k == 1 or (ref == 0).sum() > 100          # (the maze's zeros depend on its floors)
        for key, (w1, w2, d2, d1) in runs.items():
            bits_equal(w1, ref, f"case {k} SinkFill {key}")
            bits_equal(w2, ref, f"case {k} SinkFillD8 {key}")
            bits_equal(d1, runs["4"][3], f"case {k} D8 {key}")
            bits_equal(d2, runs["4"][3], f"case {k} fused D8 {key}")


# ---- row bands ----------------------------------------------------------------------------------------------------
def run_bands(z, world, max_rounds=10000):
    def fn(comm):
        band = sharding.Band(comm, *z.shape)
        w, d8 = band.sinkfill(dev.upload(band.take(z)), max_rounds=max_rounds)
        return dev.download(w), dev.download(d8), band.fill_rounds, band.fill_status(), band.fill_overlap, band.bounds

    res = sharding.ThreadComm.run(world, fn)
    return (np.concatenate([r[0] for r in res]), np.concatenate([r[1] for r in res]), [r[2] for r in res],
            [r[3] for r in res], res[0][4], res[0][5])


def check_bands(z, world, want, what):
    """Row bands against the oracle (zero signs folded) and against the single-GPU bits (sign of zero included); every
    rank's status word 0 and the same round count on every rank.  Returns (rounds, overlap, bounds)."""
    w, d8, rounds, status, ov, bounds = run_bands(z, world)
    bits_equal(w, want, f"bands {what}", zero_sign=False)
    bits_equal(d8, hydrology.d8(want), f"bands d8 {what}")
    w1, d1 = nf.SinkFillD8().apply(z)
    bits_equal(w, w1, f"bands vs one GPU {what}")
    bits_equal(d8, d1, f"bands vs one GPU d8 {what}")
    assert status == [0] * world, status
    assert len(set(rounds)) == 1, rounds
    return rounds[0], ov, bounds


# (world, ny, nx): bands of 24 to 40 rows (world 8: the 24-row minimum the halo allows) -- all thinner than 128, so
# the overlap shrinks to 8 -- and one case with the default overlap of 64
BAND_MAZES = [(2, 80, 101), (3, 100, 121), (4, 96, 91), (8, 192, 61), (8, 320, 41), (2, 400, 61)]


@gpu
@pytest.mark.parametrize("overlap", ["8", None])
@pytest.mark.parametrize("world,ny,nx", BAND_MAZES)
def test_banded_column_maze(world, ny, nx, overlap, monkeypatch):
    """A column maze crosses every cut once per corridor, so the drainage path crosses each cut many times and the
    Schwarz loop needs about one round per crossing: the closed form, and the single-GPU bits."""
    if overlap is None:
        monkeypatch.delenv("HD_FILL_OVERLAP", raising=False)
    else:
        monkeypatch.setenv("HD_FILL_OVERLAP", overlap)
    m = maze(ny, nx, cols=True, side="top", seed=world)
    want = m.fill()
    bits_equal(hydrology.sinkfill(m.z), want, "oracle", zero_sign=False)
    rounds, ov, bounds = check_bands(m.z, world, want, f"maze world {world}")
    crossings = (nx - 1) // 2 * (world - 1)
    print(f"world {world} {ny}x{nx} overlap {ov}: {crossings} cut crossings, {rounds} rounds, "
          f"bands {[b - a for a, b in bounds]}")
    thinnest = min(b - a for a, b in bounds)
    want_ov = 8 if overlap == "8" else 64
    assert ov == (want_ov if thinnest >= 2 * want_ov else max(8, thinnest // 16 * 8))
    assert rounds > 1 and crossings < 1000


@gpu
@pytest.mark.parametrize("swap", [False, True])
@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_banded_special_rows_on_cuts(world, swap):
    """Whole NaN rows and +inf rows on the cuts: on the first owned row of the band below a cut (NaN at odd cuts, or at
    even ones with swap) and on the last owned row of the band above it (+inf at the others), over pits and signed
    zeros.  Then a special-value raster on the same bands."""
    ny, nx = 40 * world, 150
    bounds = sharding.band_bounds(ny, world, 8)
    rng = np.random.default_rng(world)
    z = (rng.integers(0, 20, (ny, nx)) - 10 * (rng.random((ny, nx)) < 0.3)).astype(np.float32)
    z[z == 0] = np.where(rng.random(int((z == 0).sum())) < 0.5, np.float32(0.0), np.float32(-0.0))
    for k in range(1, world):
        if (k % 2 == 1) != swap:
            z[bounds[k][0]] = np.nan                    # first owned row of band k
        else:
            z[bounds[k - 1][1] - 1] = INF                # last owned row of band k - 1
    if world == 2:                                       # one cut: the other kind of row right next to it
        if swap:
            z[bounds[0][1] - 2] = np.nan
        else:
            z[bounds[1][0] + 1] = INF
    want = hydrology.sinkfill(z)
    rounds, ov, _ = check_bands(z, world, want, f"special rows world {world} swap {swap}")
    print(f"world {world}, overlap {ov}: special rows, {rounds} rounds")
    s = special_grid((ny, nx), world + 10 * swap)
    check_bands(s, world, hydrology.sinkfill(s), f"specials world {world}")


@gpu
def test_banded_fill_stops_at_max_rounds():
    """A maze that needs more rounds than max_rounds raises DeviceError on every rank (no rank waits in a collective
    alone)."""
    m = maze(96, 41, cols=True, seed=1)

    def fn(comm):
        band = sharding.Band(comm, *m.shape)
        with pytest.raises(DeviceError, match="did not converge"):
            band.sinkfill(dev.upload(band.take(m.z)), max_rounds=5)
        return True

    assert sharding.ThreadComm.run(4, fn) == [True] * 4

"""CPU: host-side logic that needs no GPU -- reference-compatible surface of the filter package, band
partitioning, and the halo-exchange communicator over gloo (world_size 2)."""
import inspect
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import hydrodem_b200
from hydrodem_b200 import _lib, sharding
from hydrodem_b200.exceptions import (CenterCloseBorderError, HydroDEMException, NumpyArrayExpectedError,
                                      WindowSizeEvenError, WindowSizeHighError)
from hydrodem_b200.filters import ComposedFilter, ComposedFilterResults, Filter, custom_filters as cf
from hydrodem_b200.filters import extension_filters as ef, simple_filters as sf


def test_reference_class_surface():
    """Every filter class of the reference's three modules exists with the same constructor keywords."""
    want = {
        cf: dict(MajorityFilter=["window_size"], ExpandFilter=["window_size"], QuadraticFilter=["window_size"],
                 CorrectNANValues=["window_size"], IsolatedPoints=["window_size"], BlanksFourier=["window_size"],
                 DetectBlanksFourier=[], MaskNegatives=[], MaskPositives=[], MaskTallGroves=[], MaskFourier=[],
                 TidyingLagoons=[], LagoonsDetection=[], GrovesCorrection=["groves_class"],
                 GrovesCorrectionsIter=["groves_class", "iterations"], FourierInitial=[],
                 FourierProcessQuarters=["fft_transform_abs"], DetectApplyFourier=[], PostProcessingFinal=[]),
        ef: dict(BitwiseXOR=["operand"], AbsoluteValues=[], Around=[], Convolve=["weights"], BinaryErosion=["iterations"],
                 BinaryClosing=["structure"], GreyDilation=["size"], FourierTransform=[], FourierITransform=[],
                 FourierShift=[], FourierIShift=[]),
        sf: dict(LowerThan=["value"], GreaterThan=["value"], BooleanToInteger=[], ProductFilter=["factor"],
                 AdditionFilter=["addend"], SubtractionFilter=["minuend"]),
    }
    for mod, classes in want.items():
        for name, params in classes.items():
            cls = getattr(mod, name)
            assert issubclass(cls, Filter), name
            got = [] if cls.__init__ is object.__init__ else \
                [p for p in inspect.signature(cls.__init__).parameters if p != "self"]
            assert got == params, (name, got)
    # keyword-only constructors as in the reference (custom_filters.py:39, simple_filters.py:24, ...)
    with pytest.raises(TypeError):
        cf.MajorityFilter(11)
    with pytest.raises(TypeError):
        sf.LowerThan(0.0)
    assert sf.ProductFilter(3).factor == 3 and sf.AdditionFilter(2).addend == 2


def test_exceptions_match_reference_messages():
    assert str(WindowSizeHighError(7, (5, 5))) == "Window size: 7 cannot be higher than grid dimensions: (5, 5)"
    assert str(WindowSizeEvenError(4)) == "Window size: 4 cannot be an even number"
    assert str(CenterCloseBorderError((0, 1), 3)) == "Center of window: (0, 1) too close of border. Window size: 3"
    assert "Expected numpy ndarray type" in str(NumpyArrayExpectedError([1]))
    assert issubclass(WindowSizeEvenError, HydroDEMException)


def test_boundary_checks_run_before_any_device_work():
    """The reference's argument errors do not need a GPU (sliding_window.py:130-156 order)."""
    with pytest.raises(NumpyArrayExpectedError):
        cf.MajorityFilter(window_size=11).apply([[1.0]])
    with pytest.raises(WindowSizeHighError):
        cf.ExpandFilter(window_size=7).apply(np.zeros((5, 9)))
    with pytest.raises(WindowSizeEvenError):
        cf.QuadraticFilter(window_size=4).apply(np.zeros((9, 9)))
    with pytest.raises(WindowSizeHighError):
        cf.ExpandFilter(window_size=6).apply(np.zeros((5, 9)))      # too large wins over even
    assert isinstance(cf.LagoonsDetection(), ComposedFilterResults) and isinstance(cf.MaskFourier(), ComposedFilter)


def test_install_as_reference_filters():
    saved = {k: sys.modules.get(k) for k in ("filters", "filters.custom_filters", "exceptions")}
    try:
        hydrodem_b200.install_as_reference_filters()
        from filters.custom_filters import MajorityFilter          # the reference's flat import style
        from filters import Filter as F2
        from exceptions import WindowSizeEvenError as E2
        assert MajorityFilter is cf.MajorityFilter and F2 is Filter and E2 is WindowSizeEvenError
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_band_bounds():
    assert sharding.band_bounds(10, 3) == [(0, 4), (4, 7), (7, 10)]
    b = sharding.band_bounds(36000, 8)
    assert b[0] == (0, 4500) and b[-1] == (31500, 36000)
    for ny, w in ((3601, 8), (5, 5), (18000, 4)):
        bb = sharding.band_bounds(ny, w)
        assert bb[0][0] == 0 and bb[-1][1] == ny and all(a[1] == c[0] for a, c in zip(bb, bb[1:]))
    # aligned starts (two rows share one transform on the device: the pairs must not straddle a cut)
    for ny, w in ((3601, 8), (421, 3), (36000, 8), (10801, 4)):
        bb = sharding.band_bounds(ny, w, 2)
        assert bb[0][0] == 0 and bb[-1][1] == ny and all(a[1] == c[0] for a, c in zip(bb, bb[1:]))
        assert all(a % 2 == 0 for a, _ in bb) and max(b - a for a, b in bb) - min(b - a for a, b in bb) <= 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _check_exchanges(comm, ny=23, nx=17, h=3):
    """Halo exchange (grouped send / recv into the margin rows), the transposing all-to-all of the sharded Fourier
    stage and redistribute_rows between two row layouts, on CPU tensors."""
    world, rank = comm.world, comm.rank
    mosaic = torch.arange(ny * nx, dtype=torch.float32).reshape(ny, nx)
    bounds = sharding.band_bounds(ny, world)
    r0, r1 = bounds[rank]
    up, down = (h if rank > 0 else 0), (h if rank < world - 1 else 0)
    ext = torch.full((up + r1 - r0 + down, nx), -1.0)
    ext[up:up + r1 - r0] = mosaic[r0:r1]
    sends, recvs = [], []
    if up:
        sends.append((ext[up:up + h], rank - 1)); recvs.append((ext[:up], rank - 1))
    if down:
        sends.append((ext[up + r1 - r0 - h:up + r1 - r0], rank + 1)); recvs.append((ext[up + r1 - r0:], rank + 1))
    comm.p2p(sends, recvs)
    ok = bool(torch.equal(ext, mosaic[r0 - up:r1 + down]))
    # transposing all-to-all: block (rows of rank i, columns of rank j) lands on rank j
    cols_b = sharding.band_bounds(nx, world)
    t = mosaic[r0:r1].t().contiguous()
    c0, c1 = cols_b[rank]
    bufs = [torch.empty((c1 - c0, b - a)) for a, b in bounds]
    comm.p2p([(t[a:b], j) for j, (a, b) in enumerate(cols_b)], [(bufs[i], i) for i in range(world)])
    ok &= bool(torch.equal(torch.cat(bufs, dim=1), mosaic[:, c0:c1].t()))
    # row redistribution: contiguous bands -> overlapping slabs in another order
    src_ids = [torch.arange(a, b).numpy() for a, b in bounds]
    dst_ids = [((torch.arange(0, ny // 2 + 2) + 3 * k) % ny).numpy() for k in range(world)]
    dst = torch.full((len(dst_ids[rank]), nx), -1.0)
    sharding.redistribute_rows(comm, mosaic[r0:r1].clone(), src_ids, dst_ids, dst)
    ok &= bool(torch.equal(dst, mosaic[torch.from_numpy(dst_ids[rank])]))
    flag = torch.tensor([1 if rank == 1 else 0], dtype=torch.int32)
    ok &= int(comm.allreduce_max_(flag)[0]) == 1
    ok &= int(comm.allreduce_max_(torch.zeros(1, dtype=torch.int32))[0]) == 0
    return ok


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        out[rank] = int(_check_exchanges(sharding.DistComm()))
    finally:
        dist.destroy_process_group()


def test_exchanges_gloo_world2():
    world = 2
    out = mp.Array("i", [0] * world)
    port = _free_port()
    procs = [mp.Process(target=_gloo_worker, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert list(out) == [1, 1]


def test_exchanges_thread_comm():
    assert sharding.ThreadComm.run(3, _check_exchanges) == [True, True, True]
    assert sharding.ThreadComm.run(4, lambda c: _check_exchanges(c, 41, 9, 2)) == [True] * 4


def test_band_rejects_thin_bands_on_every_rank():
    """Bands thinner than the halo are refused before any collective, by a test that only depends on (ny, world)."""
    def fn(comm):
        try:
            sharding.Band(comm, 60, 50)
        except ValueError:
            return "refused"
        return "ok"
    assert sharding.ThreadComm.run(3, fn) == ["refused"] * 3


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        from hydrodem_b200.build import build
        build()
    return _lib.load()


@pytest.mark.parametrize("shape", [(36000, 36000), (18000, 18000), (3601, 3601), (301, 333), (420, 333)])
def test_fourier_exchanges_cover_every_cell_once(shape, lib):
    """The four exchanges of the sharded Fourier stage on 1 ... 8 ranks (host geometry only): every cell the next step
    reads from a destination buffer is written by exactly one (rank, local row, row of the transposed result), it
    holds the row / column the next step takes it for, and every pass fits the limits of hd_scatter."""
    ny, nx = shape
    nh = nx // 2 + 1
    odd = ny % 2 == 1 and nx % 2 == 1
    n_out = {"F1": nh, "F2": ny, "I1": nx, "I2": ny}              # rows of the transposed result T of each pass
    read_cols = {"F1": ny, "F2": nh, "I1": ny // 2 + 1 if odd else ny, "I2": nx}   # odd x odd: conj mirror fills the rest
    for world in range(1, 9):
        bounds = sharding.band_bounds(ny, world, 8)
        KL, ex = sharding.fourier_exchanges(ny, nx, bounds)
        assert [(k, e.dest) for k, e in ex.items()] == [("F1", "at"), ("F2", "half"), ("I1", "bt"), ("I2", "dem")]
        # what rank j's local row k is before each pass: a y row, a kx column, a ky row (K layout), an x column
        held = {"F1": [np.arange(a, b) for a, b in bounds]}
        for name, nxt in (("F1", "F2"), ("F2", "I1"), ("I1", "I2"), ("I2", None)):
            e = ex[name]
            assert sum(b > a for r in e.ranges for a, b in r) <= _lib.HD_SCATTER_MAX_SEGS, (world, name)
            assert all(len(segs) <= 2 for segs in e.colsegs), (world, name)
            # rows: every row of T goes to exactly one place, so every buffer row receives exactly one row of T
            hits = np.zeros(n_out[name], dtype=np.int64)
            for r in e.ranges:
                for a, b in r:
                    assert 0 <= a <= b <= n_out[name]
                    hits[a:b] += 1
            assert (hits == 1).all(), (world, name)
            # columns: rank i's local rows land once each, at the column of the row / frequency they hold
            cols = np.zeros(e.cols, dtype=np.int64)
            for i, segs in enumerate(e.colsegs):
                nrows = max((l0 + ln for l0, _, ln in segs), default=0)
                assert nrows == len(held[name][i]) or (name == "I1" and nrows < len(held[name][i]))
                where = np.full(nrows, -1, dtype=np.int64)
                for l0, c0, ln in segs:
                    assert 0 <= l0 and 0 <= c0 and c0 + ln <= e.cols and (where[l0:l0 + ln] == -1).all()
                    where[l0:l0 + ln] = np.arange(c0, c0 + ln)
                    cols[c0:c0 + ln] += 1
                np.testing.assert_array_equal(where, held[name][i][:nrows])
            assert (cols[:read_cols[name]] == 1).all() and (cols[read_cols[name]:] == 0).all(), (world, name)
            held[nxt] = [np.concatenate([np.arange(a, b) for a, b in r]) for r in e.ranges]
        # the spectrum rows arrive in the K layout; I1 transforms all of them (only ky <= ny/2 on odd x odd);
        # the DEM rows land on the owned rows of each band
        for j, k in enumerate(KL):
            np.testing.assert_array_equal(held["I1"][j], k["ky"])
            assert max(l0 + ln for l0, _, ln in ex["I1"].colsegs[j]) == (k["nlo"] if odd else k["rows"])
            np.testing.assert_array_equal(held[None][j], np.arange(*bounds[j]))


def test_device_mosaic_is_cut_independent():
    """bench.py's mosaic generator: every cell is a pure function of (y, x, seed), so the bands of any cut reassemble
    to the same mosaic (strong scaling at N = 1, 2, 4, 8 works on ONE mosaic)."""
    from hydrodem_b200.synth import DeviceMosaic
    ny, nx = 700, 640
    m = DeviceMosaic(ny, nx, 1005, device="cpu")
    whole = m.band(0, ny)
    for cuts in ([0, 350, 700], [0, 234, 468, 700], [0, 96, 300, 301, 700]):
        parts = [m.band(a, b) for a, b in zip(cuts, cuts[1:])]
        for k in range(3):
            assert torch.equal(torch.cat([p[k] for p in parts]), whole[k]), (cuts, k)
    srtm, groves, hsheds = (t.numpy() for t in whole)
    assert groves.dtype == np.uint8 and 0.002 < groves.mean() < 0.05
    assert (hsheds == np.round(hsheds)).all() and (hsheds == -32768).sum() >= 1
    assert 60 < np.median(srtm) < 160

"""GPU: hd_warp_mosaic (several sources sampled as one virtual raster, DESIGN.md §9c) against hd_warp on the materialised
mosaic and against the float64 oracle: seams, last-wins order, nodata transparency, bin-size invariance, row bands, the
file-level entry points and CUDA-graph capture."""
import itertools
import struct

import numpy as np
import pytest
import torch

from oracle import mosaic as om
from oracle import warp as ow
from test_warp_mosaic import GEOGRAPHIC, PROJECTED, _tags

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200 import device as dev, geotiff
    from hydrodem_b200 import warp as hw
    from hydrodem_b200.pipeline import ConditioningChain
    from hydrodem_b200.synth import SynthScene

D = 1.0 / 3600.0
LON0, LAT0 = -64.0, -34.0
T = 361                                                   # tile side: 0.1 degree at 1" plus the shared edge
NANF = float("nan")


def _info(shape, dtype, geo, nodata=None, keys=GEOGRAPHIC):
    """A GeoTiffInfo for a raster held in memory (NaN nodata included)."""
    info = geotiff.GeoTiffInfo()
    info.height, info.width = shape
    info.dtype = np.dtype(dtype)
    x0, dx, y0, dy = geo
    info.tags = _tags(x0, y0, dx, dy, keys)
    info.nodata = None if nodata is None else float(nodata)
    return info


def _value(U, V, dtype, nodata):
    """A function of the global lattice pixel, so that shared edges agree; nodata on a sparse hash of the pixel."""
    if dtype == np.uint8:
        a = ((U * 7 + V * 3) % 251).astype(np.uint8)
    elif dtype == np.int16:
        a = ((U * 37 + V * 101) % 6000 - 300).astype(np.int16)
    else:
        a = (np.sin(U * 0.013) * 800 + V * 0.731 + 50).astype(np.float32)
    if nodata is not None:
        a[(U * 7919 + V * 104729) % 53 == 0] = nodata
    return a


def _geo_tiles(rows=3, cols=4, dtype=np.int16, nodata=None, order=None):
    """SRTM-like tiles: 0.1 degree at 1", 361 x 361, sharing edge rows and columns.  (array, geo, nodata) in list order,
    top-left first unless ``order`` permutes them."""
    out = []
    for r, c in itertools.product(range(rows), range(cols)):
        V, U = np.mgrid[360 * r:360 * r + T, 360 * c:360 * c + T].astype(np.int64)
        out.append((_value(U, V, dtype, nodata), (LON0 + 0.1 * c - 0.5 * D, D, LAT0 - 0.1 * r + 0.5 * D, D), nodata))
    return [out[k] for k in order] if order is not None else out


PX0, PY0, PRES = 4412345.0, 6151234.0, 30.0                # projected tiles: 30 m pixels, 361 x 361 sharing edges


def _proj_tiles(rows=3, cols=4, dtype=np.int16, nodata=None):
    out = []
    for r, c in itertools.product(range(rows), range(cols)):
        V, U = np.mgrid[360 * r:360 * r + T, 360 * c:360 * c + T].astype(np.int64)
        out.append((_value(U, V, dtype, nodata), (PX0 + 360 * c * PRES, PRES, PY0 - 360 * r * PRES, PRES), nodata))
    return out


def _pairs(tiles, keys=GEOGRAPHIC):
    return [(a, _info(a.shape, a.dtype, g, nd, keys)) for a, g, nd in tiles]


def _geo_grid():
    """About 470 x 430 cells at 90 m: crosses every seam of the 3 x 4 geographic mosaic and sticks out past all its edges
    (origin off the metre grid)."""
    x0, y1 = ow.tm_forward(LON0 - 0.03, LAT0 + 0.02)
    x1, y0 = ow.tm_forward(LON0 + 0.43, LAT0 - 0.33)
    return hw.Grid(float(x0) + 0.37, float(y1) - 0.81, 90.0, int((x1 - x0) / 90), int((y1 - y0) / 90))


def _proj_grid():
    return hw.Grid(PX0 - 1000.37, PY0 + 777.7, 90.0, 520, 400)           # 4 x 3 tiles are 43 km x 32 km


def _materialised(tiles, keys):
    arr, geo, has = om.mosaic(tiles)
    nd = tiles[0][2]
    return arr, geo, has, (arr, _info(arr.shape, arr.dtype, geo, nd, keys))


def _near_integer(t):
    return np.abs(t - np.rint(t)) < 1e-6


CASES = [(np.int16, None), (np.int16, -32768), (np.uint8, None), (np.float32, None), (np.float32, NANF)]


@pytest.mark.parametrize("resample", ["nearest", "bilinear"])
@pytest.mark.parametrize("dtype,nodata", CASES)
@pytest.mark.parametrize("crs", ["geographic", "projected"])
def test_same_bits_as_hd_warp_on_the_materialised_mosaic(crs, dtype, nodata, resample):
    tiles, keys, grid = ((_geo_tiles(dtype=dtype, nodata=nodata), GEOGRAPHIC, _geo_grid()) if crs == "geographic" else
                         (_proj_tiles(dtype=dtype, nodata=nodata), PROJECTED, _proj_grid()))
    arr, geo, has, whole = _materialised(tiles, keys)
    assert geo == tiles[0][1] and arr.shape == (1081, 1441) and has.sum() > 0.9 * has.size
    got = dev.download(hw.warp_to_device(_pairs(tiles, keys), grid, resample))
    want = dev.download(hw.warp_to_device(whole, grid, resample))
    fill = 0.0 if nodata is None else nodata
    edge = got == np.float32(fill) if not np.isnan(fill) else np.isnan(got)
    assert edge.any() and (~edge).sum() > 0.5 * got.size              # the grid sticks out and covers the mosaic
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))


RECTS = [(0, 0, 300, 400), (250, 120, 320, 260), (100, 280, 200, 300)]    # (U, V, ny, nx); a gap at the bottom left


def _overlapping(dtype, nodata, keys, order):
    """Three overlapping sources with conflicting values (1000 (k + 1) + a pattern), nodata holes in each, and a gap no
    source covers; listed in ``order``.  Geographic: 1" pixels; projected: 30 m."""
    rng = np.random.default_rng(17)
    d, x0, y0 = (D, LON0, LAT0) if keys is GEOGRAPHIC else (PRES, PX0, PY0)
    srcs = []
    for k, (U, V, ny, nx) in enumerate(RECTS):
        a = (1000 * (k + 1) + rng.integers(0, 500, (ny, nx))).astype(dtype)
        if nodata is not None:
            a[rng.random(a.shape) < 0.1] = nodata
            a[10:60, 20:90] = nodata                                           # a block hole: lower sources show
        srcs.append((a, (x0 + U * d, d, y0 - V * d, d), nodata))
    return [srcs[k] for k in order]


def _overlap_grid(keys):
    if keys is PROJECTED:
        return hw.Grid(PX0 - 400.3, PY0 + 300.1, 90.0, 190, 160)
    x0, y1 = ow.tm_forward(LON0 - 0.01, LAT0 + 0.01)
    return hw.Grid(float(x0) + 0.29, float(y1) - 0.13, 90.0, 190, 190)


@pytest.mark.parametrize("resample", ["nearest", "bilinear"])
@pytest.mark.parametrize("crs", ["geographic", "projected"])
def test_last_wins_and_nodata_transparency(crs, resample):
    keys = GEOGRAPHIC if crs == "geographic" else PROJECTED
    tm = hw.EPSG22184 if crs == "geographic" else None
    grid = _overlap_grid(keys)
    for dtype, nodata in ((np.int16, -32768), (np.float32, None)):
        seen = set()
        for order in itertools.permutations(range(3)):
            srcs = _overlapping(dtype, nodata, keys, order)
            arr, geo, has = om.mosaic(srcs)
            assert not has.all()                                               # a gap
            got = dev.download(hw.warp_to_device(_pairs(srcs, keys), grid, resample))
            # (u, v) from the first listed source's corner, as the kernel computes them; the materialised raster's
            # pixel (0, 0) sits at the integer lattice offset of the mosaic's top-left corner from it
            first = RECTS[order[0]]
            origin = (min(r[0] for r in RECTS) - first[0], min(r[1] for r in RECTS) - first[1])
            u, v = ow.pixel_coords((grid.x0, grid.res, grid.y0, grid.res), grid.ny, grid.nx, srcs[0][1], tm)
            want = om.sample(arr, u, v, resample, nodata, valid=has, origin=origin).astype(np.float32)
            seen.add(want.tobytes())
            if crs == "projected":
                np.testing.assert_array_equal(got, want)
            elif resample == "nearest":
                assert not np.any((got != want) & ~(_near_integer(u) | _near_integer(v)))
            else:
                ok = ~(_near_integer(u - 0.5) | _near_integer(v - 0.5))
                np.testing.assert_allclose(got[ok], want[ok], rtol=1e-5)
        assert len(seen) == 6                                                  # every order gives its own raster


@pytest.mark.parametrize("resample", ["nearest", "bilinear"])
def test_bin_size_and_one_source_invariance(resample):
    tiles = _geo_tiles(nodata=-32768)
    grid = _geo_grid()
    pairs = _pairs(tiles)
    outs = []
    for bin_size in (1, 37, 100000):
        m = hw.Mosaic(pairs, grid, bin_size=bin_size)
        outs.append(dev.download(m.launch(dev.empty(grid.ny, grid.nx, hw._lib.F32, np.float32), grid, resample)))
    assert m.nbins == 1
    for o in outs[1:]:
        np.testing.assert_array_equal(o.view(np.uint32), outs[0].view(np.uint32))
    np.testing.assert_array_equal(dev.download(hw.warp_to_device(pairs, grid, resample)), outs[0])
    # a one-source mosaic is hd_warp
    one = [pairs[5]]
    np.testing.assert_array_equal(dev.download(hw.warp_to_device(one, grid, resample)).view(np.uint32),
                                  dev.download(hw.warp_to_device(pairs[5], grid, resample)).view(np.uint32))


@pytest.mark.parametrize("resample", ["nearest", "bilinear"])
def test_row_bands_are_bit_identical(resample):
    pairs = _pairs(_geo_tiles(nodata=-32768))
    x0, y1 = ow.tm_forward(LON0 - 0.03, LAT0 - 0.01)                 # every row meets the mosaic: a band always reads
    x1, y0 = ow.tm_forward(LON0 + 0.43, LAT0 - 0.29)
    grid = hw.Grid(float(x0) + 0.37, float(y1) - 0.81, 90.0, int((x1 - x0) / 90), int((y1 - y0) / 90))
    full = dev.download(hw.warp_to_device(pairs, grid, resample))
    n_full = len(hw.select_sources([i for _, i in pairs], grid))
    fewer = 0
    for r0, r1 in ((0, 1), (1, 40), (40, 200), (200, 201), (201, grid.ny - 1), (grid.ny - 1, grid.ny), (0, grid.ny)):
        band = grid.rows(r0, r1)
        n = len(hw.select_sources([i for _, i in pairs], band))
        fewer += n < n_full
        got = dev.download(hw.warp_to_device(pairs, band, resample))
        np.testing.assert_array_equal(got.view(np.uint32), full[r0:r1].view(np.uint32))
    assert fewer >= 3


def _write_tiles(tmp_path, tiles, prefix, keys=GEOGRAPHIC):
    paths = []
    for k, (a, (x0, dx, y0, dy), nd) in enumerate(tiles):
        p = str(tmp_path / f"{prefix}{k}.tif")
        geotiff.write_geotiff(p, a, geo_tags=_tags(x0, y0, dx, dy, keys), nodata=nd)
        paths.append(p)
    return paths


def test_resample_and_cut_over_tile_files(tmp_path):
    grid = _geo_grid()
    for dtype, nodata in ((np.int16, -32768), (np.float32, NANF), (np.uint8, None)):
        paths = _write_tiles(tmp_path, _geo_tiles(dtype=dtype, nodata=nodata), f"{np.dtype(dtype).name}_")
        out = str(tmp_path / f"cut_{np.dtype(dtype).name}.tif")
        assert hw.resample_and_cut(paths, out, grid, resample="bilinear") is grid
        info = geotiff.read_info(out)
        assert info.dtype == np.float32 and info.shape == grid.shape and info.geotransform() == grid.geotransform()
        assert (info.nodata is None) if nodata is None else (info.nodata == nodata or np.isnan(info.nodata) and
                                                             np.isnan(nodata))
        want = dev.download(hw.warp_to_device(paths, grid, "bilinear"))
        np.testing.assert_array_equal(geotiff.read_array(out).view(np.uint32), want.view(np.uint32))


def _cut(a, rows, cols):
    """A raster split into rows x cols tiles that share their edge rows and columns, top-left first."""
    ny, nx = a.shape
    ys = np.linspace(0, ny - 1, rows + 1).astype(int)
    xs = np.linspace(0, nx - 1, cols + 1).astype(int)
    return [(ys[r], xs[c], a[ys[r]:ys[r + 1] + 1, xs[c]:xs[c + 1] + 1]) for r in range(rows) for c in range(cols)]


def test_process_geotiffs_on_tile_lists(tmp_path):
    """Tile lists plus an envelope shapefile in: the same bits as the chain run on the warped mosaics, which are the
    warps of the whole rasters the tiles were cut from."""
    sc = SynthScene(1500, 1800, 9)
    rasters = {"srtm": (sc.srtm().astype(np.float32), -32768), "groves": (sc.groves().astype(np.uint8), None),
               "hsheds": (sc.hsheds().astype(np.float32), -32768)}
    lists, whole = {}, {}
    for k, (a, nd) in rasters.items():
        whole[k] = str(tmp_path / f"{k}.tif")
        geotiff.write_geotiff(whole[k], a, geo_tags=_tags(LON0, LAT0, D, D, GEOGRAPHIC), nodata=nd)
        tiles = [(t, (LON0 + x * D, D, LAT0 - y * D, D), nd) for y, x, t in _cut(a, 2, 3)]
        tiles = tiles[:1] + tiles[1:][::-1]                       # first listed: top-left; the rest in any order
        lists[k] = _write_tiles(tmp_path, tiles, f"{k}_")
    x0, y1 = ow.tm_forward(LON0 + 0.05, LAT0 - 0.05)
    box = (float(x0), float(y1) - 90 * 300, float(x0) + 90 * 340, float(y1))
    shp = str(tmp_path / "aoi.shp")
    with open(shp, "wb") as f:
        f.write(struct.pack(">i", 9994) + b"\0" * 20 + struct.pack(">i", 50) + struct.pack("<ii", 1000, 5) +
                struct.pack("<8d", *box, 0, 0, 0, 0))
    grid = hw.Grid.from_envelope(shp)
    chain = ConditioningChain()
    final = str(tmp_path / "final.tif")
    out = geotiff.process_geotiffs(lists["srtm"], lists["groves"], lists["hsheds"], final, chain=chain, envelope=shp)
    warped = []
    for k in ("srtm", "groves", "hsheds"):
        w = dev.download(hw.warp_to_device(lists[k], grid))
        np.testing.assert_array_equal(w, dev.download(hw.warp_to_device(whole[k], grid)))
        warped.append(w)
    want = chain.apply(*warped)
    np.testing.assert_array_equal(out["final"], want.final)
    np.testing.assert_array_equal(out["filled"], want.filled)
    np.testing.assert_array_equal(out["d8"], want.d8)
    info = geotiff.read_info(final)
    assert info.geo_keys()[3072] == 22184 and info.geotransform() == grid.geotransform()


@pytest.mark.parametrize("resample", ["nearest", "bilinear"])
def test_capture_replays_the_same_bits(resample):
    grid = _geo_grid()
    m = hw.Mosaic(_pairs(_geo_tiles(dtype=np.float32, nodata=NANF)), grid)
    want = dev.download(hw.warp_to_device(_pairs(_geo_tiles(dtype=np.float32, nodata=NANF)), grid, resample))
    out = dev.empty(grid.ny, grid.nx, hw._lib.F32, np.float32)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        m.launch(out, grid, resample)
    out.buf.fill_(-1.0)
    g.replay()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(dev.download(out).view(np.uint32), want.view(np.uint32))

"""CPU: the host side of mosaics (several sources sampled as one virtual raster, DESIGN.md §9c): the lattice and its
rejections, source selection on grids and row bands, the bin index of hd_warp_mosaic, the oracle's materialised mosaic,
and the C entry's argument errors."""
import ctypes
import itertools
import os

import numpy as np
import pytest

from hydrodem_b200 import _lib, geotiff
from hydrodem_b200 import warp as hw
from hydrodem_b200.geotiff import GeoTiffError
from oracle import mosaic as om
from oracle import warp as ow

D = 1.0 / 3600.0
LON0, LAT0 = -64.0, -34.0
GEOGRAPHIC = [1, 1, 0, 3, 1024, 0, 1, 2, 1025, 0, 1, 1, 2048, 0, 1, 4326]
PROJECTED = [1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 22184]


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        from hydrodem_b200.build import build
        build()
    return _lib.load()


def _tags(x0, y0, dx, dy, keys):
    return {33550: (12, 3, np.array([dx, dy, 0.0], "<f8").tobytes()),
            33922: (12, 6, np.array([0, 0, 0, x0, y0, 0], "<f8").tobytes()),
            34735: (3, len(keys), np.array(keys, "<u2").tobytes())}


def _info(path, x0, y0, d, shape=(361, 361), dtype=np.int16, nodata=None, keys=GEOGRAPHIC, dy=None):
    geotiff.write_geotiff(str(path), np.zeros(shape, dtype), geo_tags=_tags(x0, y0, d, d if dy is None else dy, keys),
                          nodata=nodata)
    return geotiff.read_info(str(path))


def _tile_corner(r, c):
    """SRTM-like 0.1 degree tiles at 1": 361 x 361 cells whose edge rows and columns are shared with the neighbours."""
    return LON0 + 0.1 * c - 0.5 * D, LAT0 - 0.1 * r + 0.5 * D


def _tiles(tmp_path, rows, cols, **kw):
    out = []
    for r, c in itertools.product(range(rows), range(cols)):
        x0, y0 = _tile_corner(r, c)
        out.append(_info(tmp_path / f"t{r}_{c}.tif", x0, y0, D, **kw))
    return out


# ---- the lattice ---------------------------------------------------------------------------------------------------
def test_lattice_offsets(tmp_path):
    infos = _tiles(tmp_path, 3, 4, nodata=-32768)
    lat = hw.lattice(infos)
    assert lat.frame == hw.source_georeference(infos[0])[0] and lat.tm == hw.EPSG22184
    assert lat.dtype == _lib.I16 and lat.nodata == -32768
    want = [(360 * c, 360 * r) for r, c in itertools.product(range(3), range(4))]
    assert [tuple(o) for o in lat.offsets] == want
    # the anchor is the first listed source, whichever it is: offsets may be negative
    lat = hw.lattice(infos[::-1])
    assert tuple(lat.offsets[0]) == (0, 0) and tuple(lat.offsets[-1]) == (-3 * 360, -2 * 360)
    # PixelIsPoint tiles: the half-pixel shift of source_georeference applies before the lattice
    point = list(GEOGRAPHIC)
    point[11] = 2
    p = _info(tmp_path / "point.tif", LON0 + 0.1, LAT0, D, nodata=-32768, keys=point)   # tiepoint: a pixel centre
    assert tuple(hw.lattice([infos[0], p]).offsets[1]) == (360, 0)


def test_lattice_rejections(tmp_path):
    a = _info(tmp_path / "a.tif", *_tile_corner(0, 0), D, nodata=-32768)

    def bad(info, match):
        with pytest.raises(GeoTiffError, match=match) as e:
            hw.lattice([a, info], ["a.tif", "b.tif"])
        assert "b.tif" in str(e.value)

    x0, y0 = _tile_corner(0, 1)
    bad(_info(tmp_path / "b.tif", x0, y0, D * (1 + 1e-8), nodata=-32768), "pixel size")
    bad(_info(tmp_path / "b.tif", x0, y0, D, nodata=-32768, dy=D * (1 - 1e-8)), "pixel size")
    bad(_info(tmp_path / "b.tif", x0 + 1e-5 * D, y0, D, nodata=-32768), "off the first source's lattice")
    bad(_info(tmp_path / "b.tif", x0, y0 - 0.5 * D, D, nodata=-32768), "off the first source's lattice")
    bad(_info(tmp_path / "b.tif", 4.4e6, 6.1e6, 30.0, nodata=-32768, keys=PROJECTED), "CRS")
    bad(_info(tmp_path / "b.tif", x0, y0, D, dtype=np.float32, nodata=-32768), "sample type")
    bad(_info(tmp_path / "b.tif", x0, y0, D, nodata=-9999), "nodata")
    bad(_info(tmp_path / "b.tif", x0, y0, D), "nodata")
    # within the tolerances: accepted
    ok = _info(tmp_path / "b.tif", x0 + 1e-8 * D, y0, D * (1 + 1e-10), nodata=-32768)
    assert tuple(hw.lattice([a, ok]).offsets[1]) == (360, 0)
    nan_a = _info(tmp_path / "na.tif", *_tile_corner(0, 0), D, dtype=np.float32, nodata=float("nan"))
    nan_b = _info(tmp_path / "nb.tif", x0, y0, D, dtype=np.float32, nodata=float("nan"))
    assert np.isnan(hw.lattice([nan_a, nan_b]).nodata)
    with pytest.raises(GeoTiffError, match="sample type"):
        hw.lattice([_info(tmp_path / "f64.tif", x0, y0, D, dtype=np.float64)])
    with pytest.raises(GeoTiffError, match="at least one"):
        hw.lattice([])


# ---- selection -----------------------------------------------------------------------------------------------------
def _grid_over(lon0, lat0, lon1, lat1):
    x0, y1 = ow.tm_forward(lon0, lat1)
    x1, y0 = ow.tm_forward(lon1, lat0)
    return hw.Grid.from_bounds(float(x0), float(y0), float(x1), float(y1))


def _brute_select(infos, grid):
    """Every source whose padded extent contains a tap of some destination cell: the oracle's projection of every pixel
    centre, no outline argument."""
    lat = hw.lattice(infos)
    u, v = ow.pixel_coords((grid.x0, grid.res, grid.y0, grid.res), grid.ny, grid.nx, lat.frame, row0=grid.row0)
    out = []
    for k, ((U, V), (ny, nx)) in enumerate(zip(lat.offsets, lat.shapes)):
        tu, tv = u - U, v - V
        if np.any((tu > -1.5) & (tu < nx + 1.5) & (tv > -1.5) & (tv < ny + 1.5)):
            out.append(k)
    return out


def test_selection_on_grids_and_row_bands(tmp_path, lib):
    infos = _tiles(tmp_path, 3, 4)
    grid = _grid_over(LON0 + 0.12, LAT0 - 0.27, LON0 + 0.29, LAT0 - 0.03)
    sel = hw.select_sources(infos, grid)
    assert sel == sorted(sel) and 1 < len(sel) < len(infos)
    assert set(_brute_select(infos, grid)) <= set(sel)
    band_sels = []
    for r0, r1 in ((0, 1), (0, grid.ny // 3), (grid.ny // 3, grid.ny - 5), (grid.ny - 1, grid.ny), (0, grid.ny)):
        band = grid.rows(r0, r1)
        s = hw.select_sources(infos, band)
        assert set(s) <= set(sel) and set(_brute_select(infos, band)) <= set(s)
        band_sels.append(s)
    assert band_sels[-1] == sel
    assert len(band_sels[0]) < len(sel)                        # the first row reads strictly fewer tiles than its grid
    # a grid over one tile's interior selects that tile only; one far away selects none
    assert hw.select_sources(infos, _grid_over(LON0 + 0.14, LAT0 - 0.16, LON0 + 0.16, LAT0 - 0.14)) == [5]
    far = _grid_over(LON0 + 3.0, LAT0 - 3.2, LON0 + 3.1, LAT0 - 3.0)
    assert hw.select_sources(infos, far) == []
    paths = [str(tmp_path / f"t{r}_{c}.tif") for r, c in itertools.product(range(3), range(4))]
    with pytest.raises(GeoTiffError, match="does not overlap any"):
        hw.warp_to_device(paths, far)                          # raised from the headers, before any device work


def test_selection_pads_two_source_pixels(tmp_path, lib):
    """A projected source 40 px east of a grid's last pixel centre is not read; one 1 px east of it is."""
    grid = hw.Grid(4500000.0, 6100000.0, 90.0, 50, 40)
    last_centre = grid.x0 + (grid.nx - 0.5) * grid.res
    near = _info(tmp_path / "n.tif", last_centre + 30.0, grid.y0, 30.0, shape=(200, 200), keys=PROJECTED)
    far = _info(tmp_path / "f.tif", last_centre + 40 * 30.0, grid.y0, 30.0, shape=(200, 200), keys=PROJECTED)
    assert hw.select_sources([near, far], grid) == [0]
    src_geo, tm = hw.source_georeference(far)
    with pytest.raises(GeoTiffError, match="does not overlap"):
        hw.check_overlap(src_geo, far.shape, tm, grid)
    src_geo, tm = hw.source_georeference(near)
    hw.check_overlap(src_geo, near.shape, tm, grid)


def test_process_geotiffs_list_needs_an_envelope(tmp_path):
    with pytest.raises(GeoTiffError, match="envelope"):
        geotiff.process_geotiffs(["a.tif", "b.tif"], "g.tif", "h.tif", str(tmp_path / "o.tif"))


def test_mosaic_source_kinds():
    assert hw._is_mosaic(["a.tif"]) and hw._is_mosaic(("a.tif", "b.tif"))
    assert hw._is_mosaic(((np.zeros((2, 2)), None), (np.zeros((2, 2)), None)))
    assert not hw._is_mosaic((np.zeros((2, 2)), geotiff.GeoTiffInfo())) and not hw._is_mosaic("a.tif")


# ---- the bin index -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(6))
def test_index_lists_match_brute_force(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 14))
    rects = np.stack([rng.integers(-300, 300, n), rng.integers(-200, 200, n), rng.integers(1, 250, n),
                      rng.integers(1, 250, n)], axis=1)
    for bin_size in (1, 7, 64, 100, 1000):
        (iu0, iv0, bw, bh, nbu, nbv), start, lst = hw.mosaic_index(rects, bin_size)
        assert (iu0, iv0) == (rects[:, 0].min(), rects[:, 1].min()) and bw == bh == bin_size
        assert iu0 + nbu * bw >= (rects[:, 0] + rects[:, 3]).max() > iu0 + (nbu - 1) * bw
        assert iv0 + nbv * bh >= (rects[:, 1] + rects[:, 2]).max() > iv0 + (nbv - 1) * bh
        assert start[0] == 0 and start[-1] == lst.size and np.all(np.diff(start) >= 0)
        for bv, bu in itertools.product(range(nbv), range(nbu)):
            b0u, b0v = iu0 + bu * bw, iv0 + bv * bh
            want = [k for k in range(n - 1, -1, -1)
                    if rects[k, 0] < b0u + bw and b0u < rects[k, 0] + rects[k, 3] and
                    rects[k, 1] < b0v + bh and b0v < rects[k, 1] + rects[k, 2]]
            b = bv * nbu + bu
            assert list(lst[start[b]:start[b + 1]]) == want, (bin_size, bu, bv)


def test_default_bin_size_bounds_the_index():
    rects = np.array([[0, 0, 3601, 3601], [3600, 0, 3601, 3601]])
    assert hw._default_bin_size(rects) == 900
    tiny = np.array([[0, 0, 1, 1], [10 ** 6, 10 ** 6, 2, 2]])
    b = hw._default_bin_size(tiny)
    assert (-(-(10 ** 6 + 2) // b)) ** 2 <= 1 << 22


# ---- the oracle's materialised mosaic --------------------------------------------------------------------------------
def _pixel_loop(sources):
    """The virtual-pixel rule, one pixel at a time: the last listed source that covers the pixel with a valid value."""
    x0, dx, y0, dy = sources[0][1]
    offs = [(round((g[0] - x0) / dx), round((y0 - g[2]) / dy)) for _, g, _ in sources]
    u0, v0 = min(o[0] for o in offs), min(o[1] for o in offs)
    u1 = max(o[0] + a.shape[1] for o, (a, _, _) in zip(offs, sources))
    v1 = max(o[1] + a.shape[0] for o, (a, _, _) in zip(offs, sources))
    nd = sources[0][2]
    out = np.full((v1 - v0, u1 - u0), 0 if nd is None else nd, dtype=sources[0][0].dtype)
    has = np.zeros(out.shape, bool)
    for V, U in itertools.product(range(v0, v1), range(u0, u1)):
        for (ou, ov), (a, _, _) in reversed(list(zip(offs, sources))):
            j, i = V - ov, U - ou
            if 0 <= j < a.shape[0] and 0 <= i < a.shape[1]:
                s = a[j, i]
                if nd is not None and (s == nd or (np.isnan(nd) and np.isnan(s))):
                    continue
                out[V - v0, U - u0], has[V - v0, U - u0] = s, True
                break
    return out, (x0 + u0 * dx, dx, y0 - v0 * dy, dy), has


@pytest.mark.parametrize("seed", range(8))
def test_oracle_mosaic_is_the_pixel_rule(seed):
    rng = np.random.default_rng(seed)
    dtype, nodata = [(np.int16, -32768), (np.float32, float("nan")), (np.uint8, None), (np.float32, None)][seed % 4]
    srcs = []
    for _ in range(int(rng.integers(1, 6))):
        ny, nx = rng.integers(1, 12, 2)
        a = rng.integers(0, 100, (ny, nx)).astype(dtype)
        if nodata is not None:
            a[rng.random(a.shape) < 0.3] = nodata
        u, v = rng.integers(-10, 10, 2)
        srcs.append((a, (100.0 + u * 0.5, 0.5, 50.0 - v * 0.5, 0.5), nodata))
    got, geo, has = om.mosaic(srcs)
    want, wgeo, whas = _pixel_loop(srcs)
    assert geo == wgeo
    np.testing.assert_array_equal(has, whas)
    np.testing.assert_array_equal(got, want)
    assert got.dtype == want.dtype


def test_oracle_sample_valid_mask():
    src = np.array([[1.0, 2.0], [3.0, 4.0]])
    valid = np.array([[True, False], [True, True]])
    u, v = np.array([0.5, 1.5, 1.0]), np.array([0.5, 0.5, 1.0])
    np.testing.assert_array_equal(om.sample(src, u, v, "nearest", nodata=-9, valid=valid), [1.0, -9.0, 4.0])
    got = om.sample(src, u, v, "bilinear", valid=valid)
    # (1.5, 0.5): the one tap of non-zero weight holds no sample -> fill; (1, 1): taps 1, 3 and 4 of weight 1/4 each
    np.testing.assert_allclose(got, [1.0, 0.0, 8.0 / 3.0])


@pytest.mark.parametrize("resample", ["nearest", "bilinear"])
def test_mosaic_oracle_sample_is_the_warp_oracles(resample):
    """Without a mask or an origin the mosaic oracle's sampler gives oracle.warp.sample's bits; an integer origin only
    moves the array in the (u, v) frame (coordinates on a 1/64 px lattice, so that the shift is exact)."""
    rng = np.random.default_rng(3)
    src = rng.integers(0, 50, (40, 60)).astype(np.float64)
    src[rng.random(src.shape) < 0.2] = -32768
    u, v = rng.integers(-200, 64 * 63, 5000) / 64.0, rng.integers(-200, 64 * 43, 5000) / 64.0
    u[:3], v[3:6] = np.nan, 1e300
    for nodata in (None, -32768):
        want = ow.sample(src, u, v, resample, nodata)
        np.testing.assert_array_equal(om.sample(src, u, v, resample, nodata).view(np.uint64), want.view(np.uint64))
        shifted = om.sample(src, u - 7.0, v + 5.0, resample, nodata, origin=(-7, 5))
        np.testing.assert_array_equal(shifted.view(np.uint64), want.view(np.uint64))


# ---- the C entry ---------------------------------------------------------------------------------------------------
def test_warp_mosaic_argument_errors_need_no_gpu(lib):
    q = ctypes.c_void_p(1 << 20)
    g = (ctypes.c_double * 4)(0.0, 1.0, 0.0, 1.0)
    tm = (ctypes.c_double * 7)(*ow.EPSG22184)

    def call(n=1, bins=(0, 0, 16, 16, 2, 2), sources=q, start=q, lst=q, dtype=_lib.I16, frame=g, dst_ny=10, dst_nx=10,
             dst_pitch=16, dg=g, row0=0, tmb=tm, resample=0, dst=q):
        return lib.hd_warp_mosaic(sources, n, start, lst, (ctypes.c_int64 * 6)(*bins) if bins else None, dtype, frame,
                                  1, -32768.0, dst, dst_pitch, dst_ny, dst_nx, dg, row0, tmb, resample, None)

    assert call(sources=None) == _lib.HD_ERR_NULL and call(start=None) == _lib.HD_ERR_NULL
    assert call(lst=None) == _lib.HD_ERR_NULL and call(bins=None) == _lib.HD_ERR_NULL
    assert call(frame=None) == _lib.HD_ERR_NULL and call(dst=None) == _lib.HD_ERR_NULL
    assert call(n=0) == _lib.HD_ERR_ARG and call(dst_ny=0) == _lib.HD_ERR_ARG and call(dst_pitch=9) == _lib.HD_ERR_ARG
    assert call(row0=-1) == _lib.HD_ERR_ARG and call(resample=2) == _lib.HD_ERR_ARG
    for bins in ((0, 0, 0, 16, 2, 2), (0, 0, 16, 0, 2, 2), (0, 0, 16, 16, 0, 2), (0, 0, 16, 16, 2, -1),
                 (0, 0, 1 << 40, 16, 1 << 20, 2), (1 << 53, 0, 16, 16, 2, 2), (0, -(1 << 53), 16, 16, 2, 2)):
        assert call(bins=bins) == _lib.HD_ERR_ARG, bins
    assert call(frame=(ctypes.c_double * 4)(0.0, -1.0, 0.0, 1.0)) == _lib.HD_ERR_ARG
    assert call(dg=(ctypes.c_double * 4)(float("nan"), 1.0, 0.0, 1.0)) == _lib.HD_ERR_ARG
    assert call(tmb=(ctypes.c_double * 7)(-1.0, *ow.EPSG22184[1:])) == _lib.HD_ERR_ARG
    assert call(dtype=_lib.F64) == _lib.HD_ERR_UNSUPPORTED

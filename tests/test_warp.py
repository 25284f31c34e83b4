"""CPU: the float64 reprojection oracle (Transverse Mercator of EPSG:22184) against independent known answers, the host
inverse projection the library shares with its kernel, and the host logic of hydrodem_b200.warp (georeference parsing,
envelopes, grids, errors raised before any device work)."""
import ctypes
import math
import os
import struct

import numpy as np
import pytest
from scipy import integrate

from hydrodem_b200 import _lib, geotiff
from hydrodem_b200 import warp as hw
from hydrodem_b200.geotiff import GeoTiffError
from oracle import warp as ow

A_WGS84, F_WGS84 = 6378137.0, 1.0 / 298.257223563


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        from hydrodem_b200.build import build
        build()
    return _lib.load()


def _geo_tags(x0, y0, dx, dy, keys, doubles=(), ascii_=""):
    """GeoTIFF georeference tags: tiepoint at pixel (0, 0), keys = [(id, location, count, value)]."""
    d = [1, 1, 0, len(keys)] + [v for k in keys for v in k]
    tags = {33550: (12, 3, np.array([dx, dy, 0.0], "<f8").tobytes()),
            33922: (12, 6, np.array([0, 0, 0, x0, y0, 0], "<f8").tobytes()),
            34735: (3, len(d), np.array(d, "<u2").tobytes())}
    if doubles:
        tags[34736] = (12, len(doubles), np.array(doubles, "<f8").tobytes())
    if ascii_:
        s = ascii_.encode() + b"\0"
        tags[34737] = (2, len(s), s)
    return tags


GEOGRAPHIC = [(1024, 0, 1, 2), (1025, 0, 1, 1), (2048, 0, 1, 4326)]


def _write_shp(path, box, prj=None):
    head = struct.pack(">i", 9994) + b"\0" * 20 + struct.pack(">i", 50) + struct.pack("<ii", 1000, 5)
    head += struct.pack("<4d", *box) + struct.pack("<4d", 0, 0, 0, 0)
    assert len(head) == 100
    with open(path, "wb") as f:
        f.write(head)
    if prj is not None:
        with open(os.path.splitext(path)[0] + ".prj", "w") as f:
            f.write(prj)


# ---- the projection ------------------------------------------------------------------------------------------------
def test_known_answers_epsg22184():
    e, n = ow.tm_forward(-63.0, 0.0)
    assert abs(e - 4500000.0) < 1e-3
    assert abs(n - 10001965.729) < 1e-3                   # the WGS84 meridian quadrant
    e, n = ow.tm_forward(-63.0, -90.0)
    assert abs(n) < 1e-6 and abs(e - 4500000.0) < 1e-6


def test_central_meridian_northing_is_the_meridian_arc():
    e2 = F_WGS84 * (2 - F_WGS84)

    def arc(phi):
        return integrate.quad(lambda t: A_WGS84 * (1 - e2) / (1 - e2 * math.sin(t) ** 2) ** 1.5, -math.pi / 2, phi,
                              epsabs=1e-7, epsrel=1e-15, limit=200)[0]

    for lat in np.arange(-20.0, -55.01, -2.5):
        e, n = ow.tm_forward(-63.0, lat)
        assert abs(e - 4500000.0) < 1e-9
        assert abs(n - arc(math.radians(lat))) < 1e-4, lat


def test_round_trip():
    lon, lat = np.meshgrid(np.linspace(-67.0, -59.0, 81), np.linspace(-55.0, -20.0, 141))
    x, y = ow.tm_forward(lon, lat)
    lon2, lat2 = ow.tm_inverse(x, y)
    assert np.abs(lon2 - lon).max() < 1e-9 and np.abs(lat2 - lat).max() < 1e-9
    x2, y2 = ow.tm_forward(lon2, lat2)
    assert np.abs(x2 - x).max() < 1e-6 and np.abs(y2 - y).max() < 1e-6


def test_library_inverse_matches_the_oracle(lib):
    """hd_host_tm_inverse runs the kernel's own __host__ __device__ projection code on the CPU."""
    rng = np.random.default_rng(3)
    lon, lat = rng.uniform(-67, -59, 5000), rng.uniform(-55, -20, 5000)
    x, y = ow.tm_forward(lon, lat)
    x, y = np.ascontiguousarray(x), np.ascontiguousarray(y)
    glon, glat = np.empty_like(x), np.empty_like(y)
    p = lambda a: ctypes.c_void_p(a.ctypes.data)                                       # noqa: E731
    tm = (ctypes.c_double * 7)(*ow.EPSG22184)
    assert lib.hd_host_tm_inverse(tm, p(x), p(y), x.size, p(glon), p(glat)) == _lib.HD_OK
    olon, olat = ow.tm_inverse(x, y)
    assert np.abs(glon - olon).max() < 1e-11 and np.abs(glat - olat).max() < 1e-11
    assert np.abs(glon - lon).max() < 1e-9 and np.abs(glat - lat).max() < 1e-9
    bad = (ctypes.c_double * 7)(-1.0, *ow.EPSG22184[1:])
    assert lib.hd_host_tm_inverse(bad, p(x), p(y), x.size, p(glon), p(glat)) == _lib.HD_ERR_ARG


def test_warp_argument_errors_need_no_gpu(lib):
    q = ctypes.c_void_p(1 << 20)
    g = (ctypes.c_double * 4)(0.0, 1.0, 0.0, 1.0)
    tm = (ctypes.c_double * 7)(*ow.EPSG22184)

    def call(src_ny=10, src_nx=10, src_pitch=16, dst_ny=10, dst_nx=10, dst_pitch=16, sg=g, dg=g, row0=0, resample=0,
             dtype=_lib.F32, src=q):
        return lib.hd_warp(src, dtype, src_pitch, src_ny, src_nx, sg, 0, 0.0, q, dst_pitch, dst_ny, dst_nx, dg, row0, tm,
                           resample, None)

    assert call(src=None) == _lib.HD_ERR_NULL
    assert call(src_ny=0) == _lib.HD_ERR_ARG and call(dst_nx=0) == _lib.HD_ERR_ARG
    assert call(src_pitch=9) == _lib.HD_ERR_ARG and call(dst_pitch=9) == _lib.HD_ERR_ARG
    assert call(sg=(ctypes.c_double * 4)(0.0, 0.0, 0.0, 1.0)) == _lib.HD_ERR_ARG
    assert call(dg=(ctypes.c_double * 4)(0.0, 1.0, 0.0, -90.0)) == _lib.HD_ERR_ARG
    assert call(resample=2) == _lib.HD_ERR_ARG and call(row0=-1) == _lib.HD_ERR_ARG


# ---- the oracle's sampling rules ----------------------------------------------------------------------------------
def test_oracle_sampling_rules():
    src = np.array([[1.0, 2.0, 3.0], [4.0, -32768.0, 6.0]])
    u = np.array([0.0, 2.99, 3.0, -1e-12, 1.5, 0.5])
    v = np.array([0.0, 1.99, 0.5, 0.5, 0.5, 1.0])
    got = ow.sample(src, u, v, "nearest", nodata=-32768)
    np.testing.assert_array_equal(got, [1.0, 6.0, -32768, -32768, 2.0, 4.0])
    # bilinear at a pixel centre is the pixel; between centres the taps are weighted; nodata taps are dropped
    got = ow.sample(src, np.array([0.5, 1.0, 1.5, 2.5]), np.array([0.5, 0.5, 1.0, 1.5]), "bilinear", nodata=-32768)
    np.testing.assert_allclose(got, [1.0, 1.5, (2.0 * 0.5) / 0.5, 6.0])
    # corner (0, 0): only the tap (0, 0) is inside, with weight 1/4; renormalised to the pixel's value
    np.testing.assert_allclose(ow.sample(src, np.array([0.0]), np.array([0.0]), "bilinear"), [1.0])
    # every tap invalid: fill value
    assert ow.sample(src, np.array([-5.0]), np.array([0.5]), "bilinear", nodata=-9)[0] == -9


# ---- host logic ---------------------------------------------------------------------------------------------------
def test_geo_keys_round_trip(tmp_path):
    g = hw.Grid(4412345.5, 6201234.25, 90.0, 17, 11)
    path = str(tmp_path / "g.tif")
    geotiff.write_geotiff(path, np.zeros(g.shape, np.float32), geo_tags=g.geo_tags(), nodata=-32768)
    info = geotiff.read_info(path)
    assert info.geo_keys() == {1024: 1, 1025: 1, 3072: 22184, 3076: 9001}
    assert info.geotransform() == g.geotransform() == (4412345.5, 90.0, 0.0, 6201234.25, 0.0, -90.0)
    assert info.nodata == -32768
    # keys held in GeoDoubleParams / GeoAsciiParams
    tags = _geo_tags(-64.0, -34.0, 1 / 3600, 1 / 3600, GEOGRAPHIC + [(1026, 34737, 7, 0), (2057, 34736, 1, 1)],
                     doubles=(1.5, 6378137.0), ascii_="WGS 84|")
    geotiff.write_geotiff(path, np.zeros((3, 4), np.int16), geo_tags=tags)
    keys = geotiff.read_info(path).geo_keys()
    assert keys[2048] == 4326 and keys[2057] == 6378137.0 and keys[1026] == "WGS 84"
    geotiff.write_geotiff(path, np.zeros((3, 4), np.int16))
    assert geotiff.read_info(path).geo_keys() == {}


def test_source_georeference_and_pixel_is_point(tmp_path):
    path = str(tmp_path / "s.tif")
    d = 1 / 3600
    geotiff.write_geotiff(path, np.zeros((5, 6), np.int16), geo_tags=_geo_tags(-64.0, -34.0, d, d, GEOGRAPHIC))
    geo, tm = hw.source_georeference(geotiff.read_info(path))
    assert geo == (-64.0, d, -34.0, d) and tm == hw.EPSG22184 == ow.EPSG22184
    point = [(1024, 0, 1, 2), (1025, 0, 1, 2), (2048, 0, 1, 4326)]
    geotiff.write_geotiff(path, np.zeros((5, 6), np.int16), geo_tags=_geo_tags(-64.0, -34.0, d, d, point))
    geo, _ = hw.source_georeference(geotiff.read_info(path))
    assert geo == (-64.0 - 0.5 * d, d, -34.0 + 0.5 * d, d)
    projected = [(1024, 0, 1, 1), (1025, 0, 1, 1), (3072, 0, 1, 22184)]
    geotiff.write_geotiff(path, np.zeros((5, 6), np.uint8), geo_tags=_geo_tags(4.4e6, 6.2e6, 30.0, 30.0, projected))
    geo, tm = hw.source_georeference(geotiff.read_info(path))
    assert geo == (4.4e6, 30.0, 6.2e6, 30.0) and tm is None


def test_envelope_from_shapefile_header(tmp_path):
    shp = str(tmp_path / "aoi.shp")
    _write_shp(shp, (4400000.0, 6100000.0, 4400000.0 + 90 * 20.4, 6100000.0 + 90 * 10.6))
    assert hw.read_envelope(shp) == (4400000.0, 6100000.0, 4400000.0 + 90 * 20.4, 6100000.0 + 90 * 10.6)
    g = hw.Grid.from_envelope(shp)
    assert (g.x0, g.y0, g.res, g.nx, g.ny) == (4400000.0, 6100000.0 + 90 * 10.6, 90.0, 20, 11)
    _write_shp(shp, (4400000.0, 6100000.0, 4401000.0, 6101000.0), prj='PROJCS["POSGAR 94 / Argentina 4",GEOGCS[...]]')
    assert hw.Grid.from_envelope(shp).shape == (11, 11)
    _write_shp(shp, (-64.0, -35.0, -63.0, -34.0), prj=' GEOGCS["GCS_WGS_1984",DATUM["D_WGS_1984"]]')
    with pytest.raises(GeoTiffError, match="geographic"):
        hw.Grid.from_envelope(shp)
    with open(shp, "r+b") as f:
        f.write(struct.pack(">i", 1234))
    with pytest.raises(GeoTiffError, match="9994"):
        hw.Grid.from_envelope(shp)


def test_grid_sizing_and_row_bands():
    g = hw.Grid.from_bounds(1000.0, 2000.0, 1000.0 + 90 * 10.49, 2000.0 + 90 * 4.5)
    assert (g.nx, g.ny, g.x0, g.y0) == (10, 5, 1000.0, 2000.0 + 405.0)
    band = g.rows(2, 4)
    assert band.shape == (2, 10) and band.row0 == 2 and band.y0 == g.y0
    assert band.geotransform() == (1000.0, 90.0, 0.0, g.y0 - 180.0, 0.0, -90.0)
    assert band.rows(1, 2).row0 == 3
    tie = np.frombuffer(band.geo_tags()[33922][2], "<f8")
    assert tie[3] == 1000.0 and tie[4] == g.y0 - 180.0
    for r0, r1 in ((0, 0), (3, 2), (-1, 2), (0, 6)):
        with pytest.raises(GeoTiffError):
            g.rows(r0, r1)
    with pytest.raises(GeoTiffError, match="empty"):
        hw.Grid.from_bounds(0.0, 0.0, 44.0, 900.0)
    with pytest.raises(GeoTiffError):
        hw.Grid(0.0, 0.0, 0.0, 4, 4)


def test_errors_before_any_device_work(tmp_path, lib):
    """Unsupported CRS, no georeference, and an envelope that misses the source raise GeoTiffError from the header alone."""
    d = 1 / 3600
    grid = hw.Grid.from_bounds(4420000.0, 6170000.0, 4430000.0, 6180000.0)
    path = str(tmp_path / "s.tif")
    geotiff.write_geotiff(path, np.zeros((20, 30), np.int16),
                          geo_tags=_geo_tags(-64.0, -34.0, d, d, [(1024, 0, 1, 1), (3072, 0, 1, 32720)]))
    with pytest.raises(GeoTiffError, match="32720"):
        hw.warp_to_device(path, grid)
    geotiff.write_geotiff(path, np.zeros((20, 30), np.int16), geo_tags=_geo_tags(-64.0, -34.0, d, d, [(1024, 0, 1, 2)]))
    with pytest.raises(GeoTiffError, match="not supported"):
        hw.resample_and_cut(path, str(tmp_path / "o.tif"), grid)
    geotiff.write_geotiff(path, np.zeros((20, 30), np.int16))
    with pytest.raises(GeoTiffError, match="no georeference"):
        hw.warp_to_device(path, grid)
    # a 30 x 20 arc-second source near (-64, -34), a grid ~100 km away from it
    geotiff.write_geotiff(path, np.zeros((20, 30), np.int16), geo_tags=_geo_tags(-64.0, -34.0, d, d, GEOGRAPHIC))
    with pytest.raises(GeoTiffError, match="does not overlap"):
        hw.warp_to_device(path, grid)
    x, y = ow.tm_forward(-64.0 + 10 * d, -34.0 - 10 * d)
    near = hw.Grid.from_bounds(x - 5000, y - 5000, x + 5000, y + 5000)
    src_geo, tm = hw.source_georeference(geotiff.read_info(path))
    hw.check_overlap(src_geo, (20, 30), tm, near)                                       # no error
    with pytest.raises(ValueError):
        hw.warp_to_device(path, near, resample="cubic")

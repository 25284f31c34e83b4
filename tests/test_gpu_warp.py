"""GPU: hd_warp (reprojection onto the EPSG:22184 grid) against the float64 NumPy oracle, and the file-level entry points
built on it."""
import struct

import numpy as np
import pytest
import torch

from oracle import warp as ow

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200 import device as dev, geotiff
    from hydrodem_b200 import warp as hw
    from hydrodem_b200.pipeline import ConditioningChain
    from hydrodem_b200.synth import SynthScene

D = 1.0 / 3600.0                                         # 1 arc-second
LON0, LAT0, SNY, SNX = -64.0, -34.0, 3600, 4320          # lon -64 ... -62.8, lat -35 ... -34: 15.6e6 cells < 2^24
GEOGRAPHIC = [1, 1, 0, 3, 1024, 0, 1, 2, 1025, 0, 1, 1, 2048, 0, 1, 4326]
PROJECTED = [1, 1, 0, 3, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 22184]


def _tags(x0, y0, dx, dy, keys):
    return {33550: (12, 3, np.array([dx, dy, 0.0], "<f8").tobytes()),
            33922: (12, 6, np.array([0, 0, 0, x0, y0, 0], "<f8").tobytes()),
            34735: (3, len(keys), np.array(keys, "<u2").tobytes())}


def _grid():
    """600 x 700 cells at 90 m inside the source, sticking out 10 km past its west edge (origin off the metre grid)."""
    x, _ = ow.tm_forward(LON0, LAT0 - 0.5)
    _, y = ow.tm_forward(LON0 + 0.6, LAT0 - 0.2)
    return hw.Grid(float(x) - 10000.37, float(y) + 0.81, 90.0, 700, 600)


def _write_src(path, a, nodata=None):
    geotiff.write_geotiff(path, a, geo_tags=_tags(LON0, LAT0, D, D, GEOGRAPHIC), nodata=nodata)
    return path


def _near_integer(t):
    return np.abs(t - np.rint(t)) < 1e-6


@pytest.fixture(scope="module")
def index_src(tmp_path_factory):
    a = np.arange(SNY * SNX, dtype=np.float32).reshape(SNY, SNX)       # value = row * ncols + col, exact below 2^24
    return _write_src(str(tmp_path_factory.mktemp("warp") / "index.tif"), a), a


def test_nearest_picks_the_oracles_cell(index_src):
    path, _ = index_src
    grid = _grid()
    got = dev.download(hw.warp_to_device(path, grid))
    u, v = ow.pixel_coords((grid.x0, grid.res, grid.y0, grid.res), grid.ny, grid.nx, (LON0, D, LAT0, D))
    inside = (u >= 0) & (u < SNX) & (v >= 0) & (v < SNY)
    assert inside.any() and (~inside).any()
    want = np.where(inside, np.floor(v).clip(0, SNY - 1) * SNX + np.floor(u).clip(0, SNX - 1), 0.0).astype(np.float32)
    assert np.all(got[~inside] == 0.0)                                  # no nodata in the source: fill 0
    differ = got != want
    ambiguous = _near_integer(u) | _near_integer(v)
    print(f"nearest: {int(differ.sum())} of {differ.size} cells differ, {int(ambiguous.sum())} lie within 1e-6 px of a "
          "cell edge")
    assert not np.any(differ & ~ambiguous)


def test_bilinear_with_nodata_taps(tmp_path):
    rng = np.random.default_rng(11)
    a = (rng.standard_normal((SNY, SNX)) * 50 + 800).astype(np.float32)
    a[rng.random(a.shape) < 0.02] = -32768
    a[:, 0] = -32768
    a[-1, :] = -32768
    path = _write_src(str(tmp_path / "b.tif"), a, nodata=-32768)
    grid = _grid()
    got = dev.download(hw.warp_to_device(path, grid, resample="bilinear"))
    u, v, want = ow.warp(a, (LON0, D, LAT0, D), (grid.x0, grid.res, grid.y0, grid.res), grid.ny, grid.nx, "bilinear",
                         nodata=-32768)
    ok = ~(_near_integer(u - 0.5) | _near_integer(v - 0.5))
    print(f"bilinear: {int((~ok).sum())} cells within 1e-6 px of a tap edge")
    assert (want == -32768).any() and (want != -32768).any()
    np.testing.assert_allclose(got[ok], want[ok], rtol=1e-5)


@pytest.mark.parametrize("resample", ["nearest", "bilinear"])
def test_sample_types_give_the_cells_of_their_float32_cast(tmp_path, resample):
    rng = np.random.default_rng(5)
    grid = _grid()
    i16 = rng.integers(-200, 3000, (SNY, SNX)).astype(np.int16)
    i16[rng.random(i16.shape) < 0.01] = -32768
    u8 = rng.integers(0, 3, (SNY, SNX)).astype(np.uint8)
    for a, nodata in ((i16, -32768), (u8, None)):
        p = _write_src(str(tmp_path / f"{a.dtype}.tif"), a, nodata)
        p32 = _write_src(str(tmp_path / f"{a.dtype}_f32.tif"), a.astype(np.float32), nodata)
        got = dev.download(hw.warp_to_device(p, grid, resample))
        want = dev.download(hw.warp_to_device(p32, grid, resample))
        np.testing.assert_array_equal(got, want)


def test_same_crs_is_numpy_index_arithmetic(tmp_path):
    """A source already in EPSG:22184 (NULL projection block): only the affine step runs."""
    grid = _grid()
    sx0, sy0, sres = grid.x0 + 1234.56, grid.y0 - 777.7, 30.0
    ny, nx = 1500, 1900
    a = np.arange(ny * nx, dtype=np.float32).reshape(ny, nx)
    path = str(tmp_path / "p.tif")
    geotiff.write_geotiff(path, a, geo_tags=_tags(sx0, sy0, sres, sres, PROJECTED))
    got = dev.download(hw.warp_to_device(path, grid))
    u, v, want = ow.warp(a, (sx0, sres, sy0, sres), (grid.x0, grid.res, grid.y0, grid.res), grid.ny, grid.nx, tm=None)
    assert (want == 0).sum() > 1000
    np.testing.assert_array_equal(got, want)
    got = dev.download(hw.warp_to_device(path, grid, "bilinear"))
    _, _, want = ow.warp(a, (sx0, sres, sy0, sres), (grid.x0, grid.res, grid.y0, grid.res), grid.ny, grid.nx,
                         "bilinear", tm=None)
    np.testing.assert_allclose(got, want, rtol=1e-6)


@pytest.mark.parametrize("resample", ["nearest", "bilinear"])
def test_row_bands_are_bit_identical(index_src, resample):
    path, _ = index_src
    grid = _grid()
    full = dev.download(hw.warp_to_device(path, grid, resample))
    for r0, r1 in ((0, 1), (1, 150), (150, 451), (451, 600)):
        band = dev.download(hw.warp_to_device(path, grid.rows(r0, r1), resample))
        np.testing.assert_array_equal(band, full[r0:r1])


def test_resample_and_cut_writes_the_grid(index_src, tmp_path):
    path, _ = index_src
    grid = _grid()
    out = str(tmp_path / "cut.tif")
    assert hw.resample_and_cut(path, out, grid) is grid
    info = geotiff.read_info(out)
    assert info.dtype == np.float32 and info.shape == grid.shape
    assert info.geo_keys()[3072] == 22184
    assert info.geotransform() == grid.geotransform()
    np.testing.assert_array_equal(geotiff.read_array(out), dev.download(hw.warp_to_device(path, grid)))


def test_process_geotiffs_on_an_envelope(tmp_path):
    """Raw geographic rasters plus an envelope shapefile in, the DEM on the envelope's grid out: the same bits as the
    chain run on the three warped rasters."""
    sc = SynthScene(1500, 1800, 9)
    srtm, groves, hsheds = sc.srtm().astype(np.float32), sc.groves().astype(np.uint8), sc.hsheds().astype(np.float32)
    paths = {k: str(tmp_path / f"{k}.tif") for k in ("srtm", "groves", "hsheds", "final")}
    _write_src(paths["srtm"], srtm, nodata=-32768)
    _write_src(paths["groves"], groves)
    _write_src(paths["hsheds"], hsheds, nodata=-32768)
    x0, y1 = ow.tm_forward(LON0 + 0.05, LAT0 - 0.05)
    box = (float(x0), float(y1) - 90 * 300, float(x0) + 90 * 340, float(y1))
    shp = str(tmp_path / "aoi.shp")
    with open(shp, "wb") as f:
        f.write(struct.pack(">i", 9994) + b"\0" * 20 + struct.pack(">i", 50) + struct.pack("<ii", 1000, 5) +
                struct.pack("<8d", *box, 0, 0, 0, 0))
    grid = hw.Grid.from_envelope(shp)
    assert grid.shape == (300, 340)
    chain = ConditioningChain()
    out = geotiff.process_geotiffs(paths["srtm"], paths["groves"], paths["hsheds"], paths["final"], chain=chain,
                                   envelope=shp)
    warped = [dev.download(hw.warp_to_device(paths[k], grid)) for k in ("srtm", "groves", "hsheds")]
    want = chain.apply(*warped)
    np.testing.assert_array_equal(out["final"], want.final)
    np.testing.assert_array_equal(out["filled"], want.filled)
    np.testing.assert_array_equal(out["d8"], want.d8)
    info = geotiff.read_info(paths["final"])
    assert info.geo_keys()[3072] == 22184 and info.geotransform() == grid.geotransform()
    np.testing.assert_array_equal(geotiff.read_array(paths["final"]), want.final.astype(np.float32))

"""GPU: hd_rasterize_lines (river polylines burned onto the EPSG:22184 grid) against the plain oracle -- every segment
direction, a random geographic network, REPLACE order, long and degenerate segments, row bands, CUDA-graph capture, and
the file-to-file entry point."""
import numpy as np
import pytest
import torch

from oracle import rasterize as orr
from oracle import warp as ow
from test_rasterize import EPSG_PRJ, GEOG_PRJ, write_shapefile

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200 import device as dev, geotiff
    from hydrodem_b200 import rasterize as hr
    from hydrodem_b200 import warp as hw

X0, Y0, RES = 4400000.0, 6200000.0, 90.0           # a projected grid corner (metres)


def _burn(lines, grid):
    return dev.download(hr.rasterize_to_device(lines, grid))


def _oracle(lines, grid):
    return orr.rasterize(lines.x, lines.y, lines.part_start, lines.part_feature, lines.values,
                         (grid.x0, grid.res, grid.y0, grid.res), grid.ny, grid.nx, grid.row0, lines.tm)


def _projected(parts_px, features, values, grid):
    """Lines in EPSG:22184 metres from vertices given in (fractional) pixel coordinates of ``grid``."""
    xs = np.concatenate([[grid.x0 + c * grid.res for c, _ in p] for p in parts_px]) if parts_px else np.zeros(0)
    ys = np.concatenate([[grid.y0 - r * grid.res for _, r in p] for p in parts_px]) if parts_px else np.zeros(0)
    starts = np.concatenate([[0], np.cumsum([len(p) for p in parts_px])])
    return hr.Lines(xs, ys, starts, features, values, None)


def test_every_direction_is_the_oracles_walk():
    """One segment for every (dx, dy) in [-64, 64]^2, each from the middle of its own 130 x 130 block; one grid per dy."""
    rng = np.random.default_rng(3)
    d = np.arange(-64, 65)
    for dy in d:
        grid = hw.Grid(X0, Y0, RES, 130 * d.size, 130)
        parts = []
        for b, dx in enumerate(d):
            fx, fy = rng.uniform(0.05, 0.95, 2)
            c0, r0 = 130 * b + 65, 65
            parts.append([(c0 + fx, r0 + fy), (c0 + dx + fy, r0 + dy + fx)])
        lines = _projected(parts, np.arange(d.size), np.arange(1, d.size + 1, dtype=np.float32) * 1.5, grid)
        px, py, want = _oracle(lines, grid)
        assert not np.any(np.abs(px - np.rint(px)) < 1e-6) and not np.any(np.abs(py - np.rint(py)) < 1e-6)
        got = _burn(lines, grid)
        assert (got > 0).sum() == sum(max(abs(int(dx)), abs(int(dy))) + 1 for dx in d)
        np.testing.assert_array_equal(got, want)


def _network(seed=11, features=2000):
    """Random-walk polylines of 15 arc-second steps about 63 W 34.5 S, 1-3 parts per feature, random UP_CELLS."""
    rng = np.random.default_rng(seed)
    nparts = rng.integers(1, 4, features)
    feature = np.repeat(np.arange(features), nparts)
    nv = rng.integers(20, 61, feature.size)
    start = np.concatenate([[0], np.cumsum(nv)])
    step = np.full(start[-1], 15.0 / 3600.0)
    head = rng.uniform(0, 2 * np.pi, feature.size)
    ang = np.repeat(head, nv) + rng.normal(0, 0.4, start[-1]).cumsum() * 0.1
    lon0 = np.repeat(rng.uniform(-63.3, -62.7, feature.size), nv)
    lat0 = np.repeat(rng.uniform(-34.8, -34.2, feature.size), nv)
    first = np.zeros(start[-1], bool)
    first[start[:-1]] = True
    dlon, dlat = np.where(first, 0, step * np.cos(ang)), np.where(first, 0, step * np.sin(ang))
    seg = np.repeat(np.arange(feature.size), nv)
    cum_lon = np.cumsum(dlon) - np.repeat(np.cumsum(dlon)[start[:-1]], nv)
    cum_lat = np.cumsum(dlat) - np.repeat(np.cumsum(dlat)[start[:-1]], nv)
    values = rng.integers(1, 5_000_000, features).astype(np.float32)
    assert seg.size - feature.size >= 100_000
    return hr.Lines(lon0 + cum_lon, lat0 + cum_lat, start, feature, values, ow.EPSG22184)


def _network_grid():
    """900 x 800 cells at 90 m over the east half of the network, sticking out of it to the north-east."""
    x, y = ow.tm_forward(-63.0, -34.3)
    return hw.Grid(float(x) + 0.37, float(y) + 20000.81, RES, 800, 900)


@pytest.fixture(scope="module")
def network():
    lines = _network()
    grid = _network_grid()
    px, py, want = _oracle(lines, grid)
    return lines, grid, px, py, want


def _allowed(lines, grid, px, py):
    """Cells any walk may reach when a vertex within 1e-6 px of a pixel edge floors to the other side."""
    amb = (np.abs(px - np.rint(px)) < 1e-6) | (np.abs(py - np.rint(py)) < 1e-6)
    mask = np.zeros(grid.shape, bool)
    ps = lines.part_start
    for v in np.flatnonzero(amb):
        for i in (v - 1, v):
            p = np.searchsorted(ps, i, side="right") - 1
            if i < 0 or i + 1 >= ps[p + 1] or not np.isfinite(px[i:i + 2]).all():
                continue
            for ax in (-1, 0, 1):
                for ay in (-1, 0, 1):
                    a = [int(np.floor(px[i])), int(np.floor(py[i]))]
                    b = [int(np.floor(px[i + 1])), int(np.floor(py[i + 1]))]
                    (a if i == v else b)[0] += ax
                    (a if i == v else b)[1] += ay
                    for x, y in orr.bresenham(a[0], a[1], b[0], b[1]):
                        if 0 <= x < grid.nx and 0 <= y - grid.row0 < grid.ny:
                            mask[y - grid.row0, x] = True
    return int(amb.sum()), mask


def test_random_geographic_network(network):
    lines, grid, px, py, want = network
    got = _burn(lines, grid)
    inside = (px >= 0) & (px < grid.nx) & (py >= 0) & (py < grid.ny)
    assert inside.any() and (~inside).any()                           # the grid cuts the network
    assert (want > 0).sum() > 50_000
    namb, allowed = _allowed(lines, grid, px, py)
    differ = got != want
    print(f"network: {lines.n_vertices} vertices, {int(differ.sum())} of {differ.size} cells differ, {namb} vertices lie "
          "within 1e-6 px of a pixel edge")
    assert not np.any(differ & ~allowed)


def test_row_bands_are_bit_identical(network):
    lines, grid, _, _, _ = network
    full = _burn(lines, grid)
    for r0, r1 in ((0, 1), (1, 150), (150, 451), (451, 900), (377, 378)):
        np.testing.assert_array_equal(_burn(lines, grid.rows(r0, r1)), full[r0:r1])


def test_replace_order():
    grid = hw.Grid(X0, Y0, RES, 40, 30)
    parts = [[(2.5, 10.5), (30.5, 10.5)],                 # feature 2: horizontal
             [(10.5, 2.5), (10.5, 25.5)],                 # feature 0: vertical, crosses it
             [(5.5, 10.5), (20.5, 10.5)],                 # feature 1: on top of feature 2's row
             [(1.5, 20.5), (30.5, 20.5)],                 # feature 3, two overlapping parts of one feature
             [(30.5, 20.5), (1.5, 20.6), (1.5, 28.5)],
             [(12.5, 0.5), (12.5, 29.5)]]                 # feature 4 (value 0, a blank): crosses everything
    lines = _projected(parts, np.array([2, 0, 1, 3, 3, 4]), np.float32([7, 11, 13, 17, 0]), grid)
    got = _burn(lines, grid)
    np.testing.assert_array_equal(got, _oracle(lines, grid)[2])
    assert got[10, 10] == 13 and got[10, 5] == 13 and got[10, 25] == 13 and got[10, 3] == 13
    assert got[5, 10] == 7 and got[20, 10] == 17 and got[10, 12] == 0 and got[27, 1] == 17


def test_long_and_degenerate_segments():
    grid = hw.Grid(X0, Y0, RES, 700, 500)
    nan, inf = float("nan"), float("inf")
    parts = [[(-1_000_000.3, -250.2), (1_000_400.7, 600.6)],        # ~2e6 px, a few hundred of them in the grid
             [(-900_000.5, 1_100_000.5), (800.5, -300.5)],           # major axis y, enters through the left edge
             [(50.5, 60.5), (50.7, 60.2)],                           # zero length: one pixel
             [(70.5, 70.5)],                                         # a single vertex: nothing
             [(80.5, 80.5), (nan, 90.5), (100.5, 100.5), (120.5, 90.5)],     # the NaN vertex drops two segments
             [(130.5, 130.5), (inf, 130.5)],
             [(140.5, 140.5), (6e8, 140.5)],                          # beyond 2^29 px: no vertex
             [(699.9, 499.9), (700.1, 500.1), (-0.1, -0.1), (0.1, 0.1)]]
    lines = _projected(parts, np.arange(len(parts)), np.arange(1, len(parts) + 1, dtype=np.float32), grid)
    got = _burn(lines, grid)
    want = _oracle(lines, grid)[2]
    np.testing.assert_array_equal(got, want)
    assert got[60, 50] == 3 and got[70, 70] == 0 and got[130, 131] == 0 and got[140, 141] == 0
    assert (got == 1).sum() > 300 and (got == 2).sum() > 100 and (got == 5).sum() == 21


def test_capture_replays_the_same_raster(network):
    lines, grid, _, _, _ = network
    dl = hr.DeviceLines(lines)
    want = dev.download(hr.rasterize_to_device(dl, grid))
    ws = dev.scratch(hr._lib.load().hd_rasterize_workspace_bytes(dl.n_vertices))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = hr.rasterize_to_device(dl, grid, workspace=ws)
    out.buf.fill_(-1.0)
    g.replay()
    np.testing.assert_array_equal(dev.download(out), want)


def test_rasterize_rivers_file_to_file(tmp_path):
    rng = np.random.default_rng(4)
    grid = hw.Grid(X0, Y0, RES, 300, 200)
    recs = [[[tuple(rng.uniform(-20, 320, 2)) for _ in range(rng.integers(2, 6))] for _ in range(rng.integers(1, 3))]
            for _ in range(60)]
    recs = [[[(X0 + c * RES, Y0 - r * RES * 0.7) for c, r in part] for part in rec] for rec in recs]
    recs[7] = None
    vals = [int(v) for v in rng.integers(1, 10**6, 60)]
    vals[3] = None
    shp = write_shapefile(tmp_path / "rivers.shp", recs, vals, shape_type=13, prj=EPSG_PRJ, deleted={5})
    out = str(tmp_path / "rivers.tif")
    assert hr.rasterize_rivers(shp, out, grid) is grid
    info = geotiff.read_info(out)
    assert info.dtype == np.float32 and info.shape == grid.shape
    assert info.geo_keys()[3072] == 22184 and info.geotransform() == grid.geotransform()
    got = geotiff.read_array(out)
    np.testing.assert_array_equal(got, dev.download(hr.rasterize_to_device(shp, grid)))
    lines = hr.read_lines(shp)
    np.testing.assert_array_equal(got, _oracle(lines, grid)[2])
    assert (got > 0).sum() > 1000
    geo = write_shapefile(tmp_path / "geo.shp", [[[(-63.0, -34.0), (-62.9, -34.1)]]], [5], prj=GEOG_PRJ)
    x, y = ow.tm_forward(-63.05, -33.95)
    g2 = hw.Grid(float(x), float(y), RES, 200, 200)
    assert (dev.download(hr.rasterize_to_device(geo, g2)) == 5).sum() > 100

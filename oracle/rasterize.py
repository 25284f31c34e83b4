"""Plain restatement of the river-line rasterization (utils_dem.rasterize_rivers, utils_dem.py:183-191, gdal.RasterizeLayer
with ATTRIBUTE=UP_CELLS) under this package's contract (DESIGN.md §9b).

The reference the GPU burn is tested against; it is not on the product path.  Vertices go through ``oracle.warp.tm_forward``
(term-by-term Krueger series), pixel coordinates are ``(X - x0) / res`` floored, each segment is walked by the sequential,
error-accumulating Bresenham loop of GDAL's ``GDALdllImageLine`` (not a closed form), and features are burned one after
another in file order, each write replacing what was there (MERGE_ALG=REPLACE).
"""
import math

import numpy as np

from . import warp as ow

PIX_LIMIT = 2.0 ** 29          # a pixel coordinate at or beyond it counts as no vertex (as a non-finite one)


def bresenham(x0, y0, x1, y1):
    """The pixels of GDALdllImageLine's walk from (x0, y0) to (x1, y1), in walk order, both ends included."""
    dx, dy = abs(x1 - x0), abs(y1 - y0)
    sx = -1 if x0 > x1 else 1
    sy = -1 if y0 > y1 else 1
    out = []
    x, y = x0, y0
    if dx >= dy:
        err, ex, ey = 2 * dy - dx, 2 * dy, 2 * dy - 2 * dx
        for _ in range(dx + 1):
            out.append((x, y))
            x += sx
            if err > 0:
                y += sy
                err += ey
            else:
                err += ex
    else:
        err, ey, ex = 2 * dx - dy, 2 * dx, 2 * dx - 2 * dy
        for _ in range(dy + 1):
            out.append((x, y))
            y += sy
            if err > 0:
                x += sx
                err += ex
            else:
                err += ey
    return out


def pixel_coords(x, y, grid_geo, tm=ow.EPSG22184):
    """Fractional (px, py) of vertices in the full grid's frame; tm None: the vertices are already EPSG:22184 metres.
    A vertex with |latitude| > 90 (geographic) becomes NaN."""
    x0, dx, y0, dy = grid_geo
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    if tm is not None:
        with np.errstate(invalid="ignore"):
            ok = np.abs(y) <= 90.0
            X, Y = ow.tm_forward(np.where(ok, x, 0.0), np.where(ok, y, 0.0), tm)
        X, Y = np.where(ok, X, np.nan), np.where(ok, Y, np.nan)
    else:
        X, Y = x, y
    return (X - x0) / dx, (y0 - Y) / dy


def floor_pixels(px, py):
    """int pixel or None per vertex (non-finite or too far from the grid: None)."""
    out = []
    for a, b in zip(px.tolist(), py.tolist()):
        if math.isfinite(a) and math.isfinite(b) and abs(a) < PIX_LIMIT and abs(b) < PIX_LIMIT:
            out.append((math.floor(a), math.floor(b)))
        else:
            out.append(None)
    return out


def burn(pixels, part_start, part_feature, values, ny, nx, row0=0):
    """float32 (ny, nx) raster of rows row0 ... row0 + ny - 1: the parts burned in file order of their features (a
    stable order: parts of one feature keep theirs), later writes replacing earlier ones; 0 where nothing burns."""
    out = np.zeros((ny, nx), np.float32)
    part_start = [int(v) for v in part_start]
    order = sorted(range(len(part_feature)), key=lambda p: int(part_feature[p]))
    for p in order:
        v = np.float32(values[int(part_feature[p])])
        for i in range(part_start[p], part_start[p + 1] - 1):
            a, b = pixels[i], pixels[i + 1]
            if a is None or b is None:
                continue
            for x, y in bresenham(a[0], a[1], b[0], b[1]):
                if 0 <= x < nx and row0 <= y < row0 + ny:
                    out[y - row0, x] = v
    return out


def rasterize(x, y, part_start, part_feature, values, grid_geo, ny, nx, row0=0, tm=ow.EPSG22184):
    """(px, py, raster): the fractional pixel coordinates of the vertices and the burned float32 raster."""
    px, py = pixel_coords(x, y, grid_geo, tm)
    return px, py, burn(floor_pixels(px, py), part_start, part_feature, values, ny, nx, row0)

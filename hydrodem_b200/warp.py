"""Reproject and cut input rasters onto the EPSG:22184 90 m grid on the GPU: utils_dem.resample_and_cut of the reference
(utils_dem.py:65-84; image_srtm.py:55-63 calls it from each image's ``_prepare``), which runs ``gdal.Warp`` to POSGAR 94 /
Argentina 4 with 90 m Float32 pixels cut to the area-of-interest envelope.

* ``Grid``                    the destination grid: from bounds, or from the bounding box of an envelope shapefile.
* ``warp_to_device(src, grid)``  a GeoTIFF (geographic WGS84 or EPSG:22184) -> F32 ``DeviceRaster`` on ``grid``
  (``hd_warp``: inverse Transverse Mercator per destination cell in float64, nearest or bilinear sampling).
* ``resample_and_cut(src_tif, dst_tif, envelope_or_grid)``  the same, file to file.

The contract is this module's own, stated exactly in DESIGN.md: destination pixel centres, the inverse projection by the
Krueger series to order n^6, floor() to the source cell (nearest) or renormalised bilinear taps that skip nodata.
Whether ``gdal.Warp`` picks the same source cell everywhere (it uses an approximate transformer by default) is not known.
Datum shifts are out of scope: POSGAR 94 is taken as WGS84.
"""
import ctypes
import math
import os
import struct

import numpy as np

from . import _lib
from .geotiff import GeoTiffError, GeoTiffInfo, read_info

# (a, f, lat0, lon0, k0, FE, FN) of EPSG:22184: WGS84 ellipsoid, Transverse Mercator on -63 deg, false easting 4 500 km
EPSG22184 = (6378137.0, 1.0 / 298.257223563, -90.0, -63.0, 1.0, 4500000.0, 0.0)
RESAMPLE = {"nearest": _lib.WARP_NEAREST, "bilinear": _lib.WARP_BILINEAR}

_D4, _D7 = ctypes.c_double * 4, ctypes.c_double * 7


class Grid:
    """A north-up EPSG:22184 grid of square ``res`` metre pixels: top-left corner (x0, y0), ``ny`` x ``nx`` cells.  A row
    band (``rows``) keeps its parent's corner and records its first row, so that a band computes the very same pixel
    centres as the full grid."""

    def __init__(self, x0, y0, res, nx, ny, row0=0):
        self.x0, self.y0, self.res = float(x0), float(y0), float(res)
        self.nx, self.ny, self.row0 = int(nx), int(ny), int(row0)
        if not (self.res > 0 and math.isfinite(self.res) and math.isfinite(self.x0) and math.isfinite(self.y0)):
            raise GeoTiffError(f"grid origin ({x0}, {y0}) / resolution {res} is not a finite positive-pixel grid")
        if self.nx < 1 or self.ny < 1 or self.row0 < 0:
            raise GeoTiffError(f"empty grid: {self.ny} x {self.nx} cells")

    @classmethod
    def from_bounds(cls, xmin, ymin, xmax, ymax, res=90.0):
        """Origin (xmin, ymax); nx = floor((xmax - xmin) / res + 1/2), ny likewise."""
        nx = math.floor((xmax - xmin) / res + 0.5)
        ny = math.floor((ymax - ymin) / res + 0.5)
        return cls(xmin, ymax, res, nx, ny)

    @classmethod
    def from_envelope(cls, shp_path, res=90.0):
        """The grid over the bounding box of a shapefile's main header (Xmin, Ymin, Xmax, Ymax), taken as EPSG:22184
        metres.  A ``.prj`` sidecar that describes a geographic CRS raises instead of being guessed at."""
        return cls.from_bounds(*read_envelope(shp_path), res=res)

    @property
    def shape(self):
        return self.ny, self.nx

    def rows(self, r0, r1):
        """The sub-grid of rows [r0, r1)."""
        if not 0 <= r0 < r1 <= self.ny:
            raise GeoTiffError(f"row band [{r0}, {r1}) is not inside a grid of {self.ny} rows")
        return Grid(self.x0, self.y0, self.res, self.nx, r1 - r0, self.row0 + r0)

    def geotransform(self):
        """GDAL-style (x0, dx, 0, y0, 0, -dy) of this grid's first row."""
        return (self.x0, self.res, 0.0, self.y0 - self.row0 * self.res, 0.0, -self.res)

    def geo_tags(self):
        """{tag: (type, count, little-endian bytes)} for ``write_geotiff``: ModelPixelScale, ModelTiepoint and a
        GeoKeyDirectory with GTModelType 1 (projected), GTRasterType 1 (PixelIsArea), ProjectedCSType 22184 and
        ProjLinearUnits 9001 (metre)."""
        gt = self.geotransform()
        scale = np.array([self.res, self.res, 0.0], dtype="<f8")
        tie = np.array([0.0, 0.0, 0.0, gt[0], gt[3], 0.0], dtype="<f8")
        keys = np.array([1, 1, 0, 4, 1024, 0, 1, 1, 1025, 0, 1, 1, 3072, 0, 1, 22184, 3076, 0, 1, 9001], dtype="<u2")
        return {33550: (12, 3, scale.tobytes()), 33922: (12, 6, tie.tobytes()), 34735: (3, len(keys), keys.tobytes())}

    def __repr__(self):
        return f"Grid(x0={self.x0}, y0={self.y0}, res={self.res}, nx={self.nx}, ny={self.ny}, row0={self.row0})"


def read_envelope(shp_path):
    """(Xmin, Ymin, Xmax, Ymax) from the 100-byte main header of an ESRI shapefile."""
    with open(shp_path, "rb") as f:
        head = f.read(100)
    if len(head) < 100 or struct.unpack(">i", head[:4])[0] != 9994:
        raise GeoTiffError(f"{shp_path}: not an ESRI shapefile (no file code 9994 in a 100-byte header)")
    box = struct.unpack("<4d", head[36:68])
    if not all(math.isfinite(v) for v in box) or box[2] <= box[0] or box[3] <= box[1]:
        raise GeoTiffError(f"{shp_path}: empty or invalid bounding box {box}")
    prj = os.path.splitext(str(shp_path))[0] + ".prj"
    if os.path.exists(prj):
        with open(prj, "r", errors="replace") as f:
            wkt = f.read().lstrip()
        if wkt.upper().startswith("GEOGCS"):
            raise GeoTiffError(f"{prj}: the envelope is in a geographic CRS; give its bounding box in EPSG:22184 metres")
    return box


def source_georeference(info, name="source"):
    """(src_geo, tm) of a GeoTIFF header: src_geo = (x0, dx, y0, dy) of the top-left pixel corner; tm = the EPSG:22184
    parameters when the source is geographic WGS84, None when it is already in EPSG:22184."""
    scale, tie = info.values(33550), info.values(33922)
    if not scale or not tie or len(tie) < 6 or len(scale) < 2:
        raise GeoTiffError(f"{name}: no georeference (ModelPixelScale / ModelTiepoint)")
    keys = info.geo_keys()
    model, geog, proj = keys.get(1024), keys.get(2048), keys.get(3072)
    if proj == 22184:
        tm = None
    elif model == 2 and geog == 4326:
        tm = EPSG22184
    else:
        raise GeoTiffError(f"{name}: CRS not supported (GTModelType {model}, GeographicType {geog}, ProjectedCSType {proj}); "
                           "geographic WGS84 (EPSG:4326) and EPSG:22184 sources are read")
    gt = info.geotransform()
    x0, dx, y0, dy = gt[0], gt[1], gt[3], -gt[5]
    if not (dx > 0 and dy > 0):
        raise GeoTiffError(f"{name}: pixel scale {scale[:2]} is not positive")
    if keys.get(1025) == 2:                    # PixelIsPoint: the tiepoint is a pixel centre, shift to its corner as GDAL does
        x0, y0 = x0 - 0.5 * dx, y0 + 0.5 * dy
    return (x0, dx, y0, dy), tm


def check_overlap(src_geo, src_shape, tm, grid, name="source", samples=64):
    """GeoTiffError unless the grid's outline, taken to source coordinates, has a bounding box that meets the source."""
    x1, y_top = grid.x0 + grid.nx * grid.res, grid.y0 - grid.row0 * grid.res
    y_bot = y_top - grid.ny * grid.res
    t = np.linspace(0.0, 1.0, samples)
    xs = np.concatenate([grid.x0 + t * (x1 - grid.x0)] * 2 + [np.full(samples, grid.x0), np.full(samples, x1)])
    ys = np.concatenate([np.full(samples, y_top), np.full(samples, y_bot)] + [y_bot + t * (y_top - y_bot)] * 2)
    if tm is not None:
        lon, lat = np.empty_like(xs), np.empty_like(ys)
        p = lambda a: ctypes.c_void_p(a.ctypes.data)                                       # noqa: E731
        _lib.check(_lib.load().hd_host_tm_inverse(_D7(*tm), p(xs), p(ys), xs.size, p(lon), p(lat)))
        xs, ys = lon, lat
    sx0, sdx, sy0, sdy = src_geo
    sny, snx = src_shape
    if xs.max() <= sx0 or xs.min() >= sx0 + snx * sdx or ys.max() <= sy0 - sny * sdy or ys.min() >= sy0:
        raise GeoTiffError(f"{name}: the grid {grid} does not overlap the source extent "
                           f"x [{sx0}, {sx0 + snx * sdx}], y [{sy0 - sny * sdy}, {sy0}]")


def warp_to_device(src, grid, resample="nearest"):
    """A source raster resampled onto ``grid`` as an F32 DeviceRaster (cells with no valid sample hold the source's
    nodata value, or 0 without one).  ``src``: a GeoTIFF path, or a pair (ndarray or DeviceRaster, GeoTiffInfo) for a
    raster already read.  Sources: U8 / I16 / F32 samples, geographic WGS84 or EPSG:22184."""
    if resample not in RESAMPLE:
        raise ValueError(f"resample must be one of {sorted(RESAMPLE)}, not {resample!r}")
    if isinstance(src, tuple):
        data, info = src
        name = "source"
        if not isinstance(info, GeoTiffInfo):
            raise TypeError("warp_to_device: a raster must come with its GeoTiffInfo")
    else:
        data, info, name = None, read_info(src), str(src)
    src_geo, tm = source_georeference(info, name)
    check_overlap(src_geo, info.shape, tm, grid, name)
    from . import device as dev
    from .geotiff import read_to_device
    if data is None:
        raster = read_to_device(src)
    elif isinstance(data, dev.DeviceRaster):
        raster = data
    else:
        raster = dev.upload(np.asarray(data))
    if raster.shape != info.shape:
        raise GeoTiffError(f"{name}: raster shape {raster.shape} differs from its header's {info.shape}")
    out = dev.empty(grid.ny, grid.nx, _lib.F32, np.float32)
    nodata = info.nodata
    _lib.check(_lib.load().hd_warp(raster.ptr, raster.dtype, raster.pitch, raster.ny, raster.nx, _D4(*src_geo),
                                   0 if nodata is None else 1, 0.0 if nodata is None else float(nodata), out.ptr,
                                   out.pitch, grid.ny, grid.nx, _D4(grid.x0, grid.res, grid.y0, grid.res), grid.row0,
                                   _D7(*tm) if tm is not None else None, RESAMPLE[resample], dev.stream_ptr()))
    return out


def as_grid(envelope_or_grid, res=90.0):
    return envelope_or_grid if isinstance(envelope_or_grid, Grid) else Grid.from_envelope(envelope_or_grid, res=res)


def resample_and_cut(src_tif, dst_tif, envelope_or_grid, resample="nearest", res=90.0):
    """The reference's resample-and-cut step as one call, file to file: ``src_tif`` (geographic WGS84 or EPSG:22184)
    reprojected to EPSG:22184 with ``res`` metre pixels over ``envelope_or_grid`` (a Grid, or an ESRI shapefile whose
    bounding box is the area of interest), written to ``dst_tif`` as a Float32 GeoTIFF with the grid's georeference and
    the source's nodata value.  Returns the Grid."""
    from . import device as dev
    from .geotiff import write_geotiff
    grid = as_grid(envelope_or_grid, res)
    info = read_info(src_tif)
    out = warp_to_device(src_tif, grid, resample)
    write_geotiff(dst_tif, dev.download(out), dtype=np.float32, geo_tags=grid.geo_tags(), nodata=info.nodata)
    return grid

"""Reproject and cut input rasters onto the EPSG:22184 90 m grid on the GPU: utils_dem.resample_and_cut of the reference
(utils_dem.py:65-84; image_srtm.py:55-63 calls it from each image's ``_prepare``), which runs ``gdal.Warp`` to POSGAR 94 /
Argentina 4 with 90 m Float32 pixels cut to the area-of-interest envelope.

* ``Grid``                    the destination grid: from bounds, or from the bounding box of an envelope shapefile.
* ``warp_to_device(src, grid)``  a GeoTIFF (geographic WGS84 or EPSG:22184) -> F32 ``DeviceRaster`` on ``grid``
  (``hd_warp``: inverse Transverse Mercator per destination cell in float64, nearest or bilinear sampling).
* ``resample_and_cut(src_tif, dst_tif, envelope_or_grid)``  the same, file to file.
* a list of sources (tiles) in place of one: a mosaic sampled as one virtual raster, last listed source on top
  (``hd_warp_mosaic``; ``lattice``, ``select_sources``, ``Mosaic``).

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


def footprint(grid, tm):
    """(xmin, xmax, ymin, ymax) in the source CRS (lon / lat degrees when ``tm`` is set, else metres) of the destination
    pixel centres of ``grid`` (a row band: its own rows).

    The outline of the centres, one point per cell along each edge, goes through ``hd_host_tm_inverse``, the kernel's own
    projection code.  The inverse projection is a diffeomorphism, so it maps the rectangle of centres onto a region whose
    boundary is the image of the rectangle's boundary, and the extremes of lon and lat over the region lie on that
    outline.  Between two outline points 90 m apart the projected edge deviates from its chord by far less than a
    nanodegree, far below a source pixel; callers pad source extents by whole source pixels."""
    xc = grid.x0 + (np.arange(grid.nx, dtype=np.float64) + 0.5) * grid.res
    yc = grid.y0 - (np.arange(grid.row0, grid.row0 + grid.ny, dtype=np.float64) + 0.5) * grid.res
    xs = np.concatenate([xc, xc, np.full(grid.ny, xc[0]), np.full(grid.ny, xc[-1])])
    ys = np.concatenate([np.full(grid.nx, yc[0]), np.full(grid.nx, yc[-1]), yc, yc])
    if tm is not None:
        lon, lat = np.empty_like(xs), np.empty_like(ys)
        p = lambda a: ctypes.c_void_p(a.ctypes.data)                                       # noqa: E731
        _lib.check(_lib.load().hd_host_tm_inverse(_D7(*tm), p(xs), p(ys), xs.size, p(lon), p(lat)))
        xs, ys = lon, lat
    return float(xs.min()), float(xs.max()), float(ys.min()), float(ys.max())


SELECT_PAD = 2      # source pixels around each extent: the bilinear taps (1.5 px) and host-vs-device projection rounding


def _meets(fp, src_geo, src_shape, pad=SELECT_PAD):
    """Does the footprint ``fp`` meet the source extent padded by ``pad`` source pixels?  (NaN meets nothing.)"""
    xmin, xmax, ymin, ymax = fp
    sx0, sdx, sy0, sdy = src_geo
    sny, snx = src_shape
    return (xmax > sx0 - pad * sdx and xmin < sx0 + (snx + pad) * sdx and
            ymax > sy0 - (sny + pad) * sdy and ymin < sy0 + pad * sdy)


def check_overlap(src_geo, src_shape, tm, grid, name="source"):
    """GeoTiffError unless the grid's pixel centres, taken to source coordinates (``footprint``), have a bounding box that
    meets the source extent padded by ``SELECT_PAD`` source pixels: otherwise no cell could get a sample."""
    if not _meets(footprint(grid, tm), src_geo, src_shape):
        sx0, sdx, sy0, sdy = src_geo
        sny, snx = src_shape
        raise GeoTiffError(f"{name}: the grid {grid} does not overlap the source extent "
                           f"x [{sx0}, {sx0 + snx * sdx}], y [{sy0 - sny * sdy}, {sy0}]")


# ---- mosaics: several sources sampled as one virtual raster (DESIGN.md §9c) -------------------------------------------
_MOSAIC_DTYPES = {("u", 1): _lib.U8, ("i", 2): _lib.I16, ("f", 4): _lib.F32}


class Lattice:
    """The checked lattice of a mosaic's sources (``lattice``): ``frame`` = (x0, dx, y0, dy) of the first listed source,
    ``tm`` the projection block (None: EPSG:22184 sources), ``offsets`` int64 (n, 2) of (U, V), ``shapes`` int64 (n, 2)
    of (ny, nx), ``geos`` each source's own (x0, dx, y0, dy), the common ``dtype`` code and ``nodata``."""

    def __init__(self, frame, tm, offsets, shapes, geos, dtype, nodata):
        self.frame, self.tm, self.offsets, self.shapes, self.geos = frame, tm, offsets, shapes, geos
        self.dtype, self.nodata = dtype, nodata


def _same_nodata(a, b):
    if a is None or b is None:
        return a is None and b is None
    return a == b or (math.isnan(a) and math.isnan(b))


def lattice(infos, names=None):
    """Check that the sources (GeoTiffInfo headers, in list order) lie on one lattice and return it as a ``Lattice``.
    Every source must share the first's CRS kind, sample type (U8 / I16 / F32), nodata (the same value, NaN included, or
    none) and pixel size (relative difference <= 1e-9).  Source i sits at (U, V) = (round((x0_i - x0_1) / dx),
    round((y0_1 - y0_i) / dy)) with its corner within 1e-6 px of that lattice point.  Violations raise GeoTiffError
    naming the source and the rule."""
    infos = list(infos)
    if not infos:
        raise GeoTiffError("a mosaic needs at least one source")
    names = list(names) if names is not None else [f"source {k}" for k in range(len(infos))]
    geos, tms = zip(*[source_georeference(info, name) for info, name in zip(infos, names)])
    x0, dx, y0, dy = frame = geos[0]
    kinds = [(np.dtype(i.dtype).kind, np.dtype(i.dtype).itemsize) for i in infos]
    if kinds[0] not in _MOSAIC_DTYPES:
        raise GeoTiffError(f"{names[0]}: sample type {infos[0].dtype} not supported; U8, I16 and F32 sources are read")
    offsets = np.zeros((len(infos), 2), np.int64)
    for k in range(1, len(infos)):
        name, (gx, gdx, gy, gdy) = names[k], geos[k]
        if (tms[k] is None) != (tms[0] is None):
            raise GeoTiffError(f"{name}: CRS differs from the first source's (geographic WGS84 and EPSG:22184 mixed)")
        if kinds[k] != kinds[0]:
            raise GeoTiffError(f"{name}: sample type {infos[k].dtype} differs from the first source's {infos[0].dtype}")
        if not _same_nodata(infos[k].nodata, infos[0].nodata):
            raise GeoTiffError(f"{name}: nodata {infos[k].nodata} differs from the first source's {infos[0].nodata}")
        if abs(gdx - dx) > 1e-9 * dx or abs(gdy - dy) > 1e-9 * dy:
            raise GeoTiffError(f"{name}: pixel size ({gdx}, {gdy}) differs from the first source's ({dx}, {dy})")
        fu, fv = (gx - x0) / dx, (y0 - gy) / dy
        if not (abs(fu) < 2.0 ** 52 and abs(fv) < 2.0 ** 52):
            raise GeoTiffError(f"{name}: corner ({gx}, {gy}) is off the first source's lattice")
        u, v = round(fu), round(fv)
        if abs(fu - u) > 1e-6 or abs(fv - v) > 1e-6:
            raise GeoTiffError(f"{name}: corner ({gx}, {gy}) is off the first source's lattice by "
                               f"({fu - u:.3g}, {fv - v:.3g}) px (more than 1e-6)")
        offsets[k] = u, v
    shapes = np.array([i.shape for i in infos], np.int64).reshape(-1, 2)
    return Lattice(frame, tms[0], offsets, shapes, geos, _MOSAIC_DTYPES[kinds[0]], infos[0].nodata)


def select_sources(infos, grid):
    """Indices, in list order, of the mosaic sources (GeoTiffInfo headers) that ``grid`` (or a row band of it) can read:
    those whose extent, padded by ``SELECT_PAD`` source pixels, meets the footprint of the grid's pixel centres.  The
    lattice is checked first (``lattice``)."""
    lat = infos if isinstance(infos, Lattice) else lattice(infos)
    fp = footprint(grid, lat.tm)
    return [k for k in range(len(lat.geos)) if _meets(fp, lat.geos[k], tuple(lat.shapes[k]))]


def mosaic_index(rects, bin_size):
    """The bin lists of ``hd_warp_mosaic`` for source rectangles ``rects`` (int64 (n, 4) of (U, V, ny, nx), in list
    order): a uniform grid of ``bin_size`` pixel square bins over their joint extent and, per bin, every source whose
    rectangle meets it, in descending list order.  Returns (bins, start, lst): bins = (iu0, iv0, bw, bh, nbu, nbv),
    start = int64[nbu * nbv + 1] CSR offsets, lst = int64 source indices."""
    rects = np.asarray(rects, np.int64).reshape(-1, 4)
    bw = bh = int(bin_size)
    if bw < 1:
        raise ValueError(f"bin size must be positive, not {bin_size}")
    iu0, iv0 = int(rects[:, 0].min()), int(rects[:, 1].min())
    nbu = -(-int((rects[:, 0] + rects[:, 3]).max() - iu0) // bw)
    nbv = -(-int((rects[:, 1] + rects[:, 2]).max() - iv0) // bh)
    ids, srcs = [], []
    for k in range(len(rects) - 1, -1, -1):                  # descending list order; the stable sort keeps it per bin
        u, v, ny, nx = (int(t) for t in rects[k])
        bu = np.arange((u - iu0) // bw, (u + nx - 1 - iu0) // bw + 1)
        bv = np.arange((v - iv0) // bh, (v + ny - 1 - iv0) // bh + 1)
        ids.append((bv[:, None] * nbu + bu[None, :]).ravel())
        srcs.append(np.full(bu.size * bv.size, k, np.int64))
    ids, srcs = np.concatenate(ids), np.concatenate(srcs)
    order = np.argsort(ids, kind="stable")
    start = np.zeros(nbu * nbv + 1, np.int64)
    np.cumsum(np.bincount(ids, minlength=nbu * nbv), out=start[1:])
    return (iu0, iv0, bw, bh, nbu, nbv), start, srcs[order]


def _default_bin_size(rects):
    """A quarter of the smallest source side (at least 16 px), doubled until there are at most 2^22 bins: most bins then
    lie inside one source, and the index stays a few MB."""
    rects = np.asarray(rects, np.int64).reshape(-1, 4)
    b = max(16, int(rects[:, 2:].min()) // 4)
    w = int((rects[:, 0] + rects[:, 3]).max() - rects[:, 0].min())
    h = int((rects[:, 1] + rects[:, 2]).max() - rects[:, 1].min())
    while -(-w // b) * -(-h // b) > 1 << 22:
        b *= 2
    return b


def _is_mosaic(src):
    """A list, or a tuple that is not one (raster, GeoTiffInfo) pair, is a mosaic."""
    if isinstance(src, list):
        return True
    return isinstance(src, tuple) and isinstance(src[0] if src else None, (str, os.PathLike, tuple))


def _source(src, name="source"):
    """(data or None, GeoTiffInfo, name) of one source: a path, or a (raster, GeoTiffInfo) pair."""
    if isinstance(src, tuple):
        data, info = src
        if not isinstance(info, GeoTiffInfo):
            raise TypeError("warp_to_device: a raster must come with its GeoTiffInfo")
        return data, info, name
    return None, read_info(src), str(src)


def _to_device(data, path, info, name):
    from . import device as dev
    from .geotiff import read_to_device
    if data is None:
        raster = read_to_device(path)
    elif isinstance(data, dev.DeviceRaster):
        raster = data
    else:
        raster = dev.upload(np.asarray(data))
    if raster.shape != info.shape:
        raise GeoTiffError(f"{name}: raster shape {raster.shape} differs from its header's {info.shape}")
    return raster


class Mosaic:
    """The selected sources of a mosaic on the device and its index, ready for ``hd_warp_mosaic`` onto ``grid`` or any
    row band of it inside the selection's footprint.  ``warp_to_device`` builds one per call and drops it on return."""

    def __init__(self, srcs, grid, bin_size=None):
        from . import device as dev
        import torch
        items = [_source(s, f"source {k}") for k, s in enumerate(srcs)]
        lat = lattice([i for _, i, _ in items], [n for _, _, n in items])
        self.selected = select_sources(lat, grid)
        if not self.selected:
            raise GeoTiffError(f"the grid {grid} does not overlap any of the {len(items)} sources of the mosaic")
        # one file after another: each read_to_device overlaps its own reads with its uploads
        self.rasters = [_to_device(items[k][0], srcs[k], items[k][1], items[k][2]) for k in self.selected]
        for k, r in zip(self.selected, self.rasters):
            if r.dtype != lat.dtype:
                raise GeoTiffError(f"{items[k][2]}: device raster type {r.dtype} differs from the mosaic's {lat.dtype}")
        rects = np.concatenate([lat.offsets[self.selected], lat.shapes[self.selected]], axis=1)
        self.bins, start, lst = mosaic_index(rects, bin_size or _default_bin_size(rects))
        table = np.array([[r.ptr.value, r.pitch] for r in self.rasters], np.int64)
        table = np.concatenate([table, rects], axis=1)                                    # ptr, pitch, U, V, ny, nx
        self.index = torch.from_numpy(np.concatenate([table.ravel(), start, lst])).to(dev.device())
        self.n, self.nbins, self.lattice = len(self.rasters), start.size - 1, lat

    def launch(self, out, grid, resample="nearest", stream=None):
        from . import device as dev
        lat, base, es = self.lattice, self.index.data_ptr(), 8
        nodata = lat.nodata
        _lib.check(_lib.load().hd_warp_mosaic(
            ctypes.c_void_p(base), self.n, ctypes.c_void_p(base + 6 * self.n * es),
            ctypes.c_void_p(base + (6 * self.n + self.nbins + 1) * es), (ctypes.c_int64 * 6)(*self.bins), lat.dtype,
            _D4(*lat.frame), 0 if nodata is None else 1, 0.0 if nodata is None else float(nodata), out.ptr, out.pitch,
            grid.ny, grid.nx, _D4(grid.x0, grid.res, grid.y0, grid.res), grid.row0,
            _D7(*lat.tm) if lat.tm is not None else None, RESAMPLE[resample],
            dev.stream_ptr() if stream is None else stream))
        return out


def warp_to_device(src, grid, resample="nearest"):
    """A source raster resampled onto ``grid`` as an F32 DeviceRaster (cells with no valid sample hold the source's
    nodata value, or 0 without one).  ``src``: a GeoTIFF path, or a pair (ndarray or DeviceRaster, GeoTiffInfo) for a
    raster already read.  Sources: U8 / I16 / F32 samples, geographic WGS84 or EPSG:22184.

    ``src`` may also be a list (or tuple) of such sources, a mosaic sampled as one virtual raster (DESIGN.md §9c): the
    last listed source with a valid value at a pixel gives it.  Only the sources the grid (or row band) can read are read
    and uploaded (``select_sources``), one after another, and released when the call returns."""
    if resample not in RESAMPLE:
        raise ValueError(f"resample must be one of {sorted(RESAMPLE)}, not {resample!r}")
    from . import device as dev
    if _is_mosaic(src):
        m = Mosaic(list(src), grid)
        return m.launch(dev.empty(grid.ny, grid.nx, _lib.F32, np.float32), grid, resample)
    data, info, name = _source(src)
    src_geo, tm = source_georeference(info, name)
    check_overlap(src_geo, info.shape, tm, grid, name)
    raster = _to_device(data, src, info, name)
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
    """The reference's resample-and-cut step as one call, file to file: ``src_tif`` (geographic WGS84 or EPSG:22184, or
    a list of tile files mosaicked as in ``warp_to_device``) reprojected to EPSG:22184 with ``res`` metre pixels over
    ``envelope_or_grid`` (a Grid, or an ESRI shapefile whose bounding box is the area of interest), written to
    ``dst_tif`` as a Float32 GeoTIFF with the grid's georeference and the source's nodata value (a mosaic's sources
    share one).  Returns the Grid."""
    from . import device as dev
    from .geotiff import write_geotiff
    grid = as_grid(envelope_or_grid, res)
    out = warp_to_device(src_tif, grid, resample)
    nodata = _source(src_tif[0] if _is_mosaic(src_tif) else src_tif)[1].nodata
    write_geotiff(dst_tif, dev.download(out), dtype=np.float32, geo_tags=grid.geo_tags(), nodata=nodata)
    return grid

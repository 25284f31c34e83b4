"""Rasterize the HydroSHEDS river polylines onto the EPSG:22184 grid on the GPU: rasterize_rivers of the reference
(utils_dem.py:183-191, ``gdal.RasterizeLayer`` with ``ATTRIBUTE=UP_CELLS``; ``Rivers.process``, image_hsheds.py:178-205).

* ``read_lines(shp)``                  an ESRI PolyLine shapefile (.shp + .shx + .dbf + .prj) -> vertex arrays, part starts,
  part -> feature, feature values and the CRS decision, parsed with NumPy vector operations (no loop per record).
* ``rasterize_to_device(shp, grid)``   -> F32 ``DeviceRaster`` on ``grid`` (``hd_rasterize_lines``), row bands included.
* ``rasterize_rivers(shp, dst_tif, envelope_or_grid)``  the same, file to file.

The contract is this module's own, modelled on GDAL's default line burning (no ALL_TOUCHED, MERGE_ALG=REPLACE) and stated
exactly in DESIGN.md §9b; parity with ``gdal.RasterizeLayer`` is not verified.
"""
import os
import re
import struct

import numpy as np

from . import _lib
from .geotiff import GeoTiffError
from .warp import _D4, _D7, EPSG22184, as_grid

POLYLINE_TYPES = {3: "PolyLine", 13: "PolyLineZ", 23: "PolyLineM"}


class Lines:
    """Polylines as flat arrays: vertex ``x``, ``y`` (float64; lon / lat degrees when ``tm`` is set, else EPSG:22184
    metres), ``part_start`` (int64, n_parts + 1: part p is vertices [part_start[p], part_start[p + 1])), ``part_feature``
    (int32, the feature of each part, in file order) and ``values`` (float32, one per feature)."""

    def __init__(self, x, y, part_start, part_feature, values, tm):
        self.x = np.ascontiguousarray(x, dtype=np.float64)
        self.y = np.ascontiguousarray(y, dtype=np.float64)
        self.part_start = np.ascontiguousarray(part_start, dtype=np.int64)
        self.part_feature = np.ascontiguousarray(part_feature, dtype=np.int32)
        self.values = np.ascontiguousarray(values, dtype=np.float32)
        self.tm = tm
        if self.x.shape != self.y.shape or self.part_start.size != self.part_feature.size + 1:
            raise ValueError("Lines: x / y or part_start / part_feature sizes disagree")

    @property
    def n_vertices(self):
        return self.x.size

    @property
    def n_parts(self):
        return self.part_feature.size

    def __repr__(self):
        crs = "geographic WGS84" if self.tm is not None else "EPSG:22184"
        return f"Lines({self.n_vertices} vertices, {self.n_parts} parts, {self.values.size} features, {crs})"


# ---- the shapefile -------------------------------------------------------------------------------------------------
def _read(path, what):
    try:
        return np.fromfile(path, dtype=np.uint8)
    except FileNotFoundError:
        raise GeoTiffError(f"{path}: missing ({what} is required)") from None


def _gather_i4(buf, pos):
    """Little-endian int32 at byte offsets ``pos`` (any alignment)."""
    b = buf[np.asarray(pos, dtype=np.int64)[:, None] + np.arange(4)]
    return b.view("<i4").ravel().astype(np.int64)


def _gather_f8(buf, pos):
    """float64 at byte offsets ``pos``: one aligned view of the buffer per offset class mod 8 (no per-element loop)."""
    out = np.empty(pos.size, dtype=np.float64)
    cls = pos & 7
    for a in range(8):
        sel = np.flatnonzero(cls == a)
        if sel.size:
            view = np.frombuffer(buf, dtype="<f8", count=(buf.size - a) // 8, offset=a)
            out[sel] = view[(pos[sel] - a) >> 3]
    return out


def _check_header(buf, path):
    if buf.size < 100 or struct.unpack(">i", buf[:4].tobytes())[0] != 9994:
        raise GeoTiffError(f"{path}: not an ESRI shapefile (no file code 9994 in a 100-byte header)")
    return struct.unpack("<i", buf[32:36].tobytes())[0]


def _read_dbf(path, attribute, n_shapes):
    """(values float64, deleted bool) of the numeric field ``attribute`` (case-insensitive), one per record."""
    buf = _read(path, "the .dbf attribute table")
    if buf.size < 33:
        raise GeoTiffError(f"{path}: truncated .dbf header")
    n, hlen, rlen = struct.unpack("<IHH", buf[4:12].tobytes())
    if hlen < 33 or rlen < 1 or (hlen - 1) % 32 or buf.size < hlen or buf[hlen - 1] != 0x0D:
        raise GeoTiffError(f"{path}: bad .dbf header (header length {hlen}, record length {rlen})")
    desc = buf[32:hlen - 1].reshape(-1, 32)
    names = [bytes(d[:11]).split(b"\0")[0].decode("ascii", "replace").strip() for d in desc]
    types = [chr(d[11]) for d in desc]
    widths = desc[:, 16].astype(np.int64)
    starts = 1 + np.concatenate([[0], np.cumsum(widths)[:-1]]).astype(np.int64)
    if widths.sum() + 1 > rlen:
        raise GeoTiffError(f"{path}: bad .dbf header (fields of {int(widths.sum())} bytes in records of {rlen})")
    if n != n_shapes:
        raise GeoTiffError(f"{path}: {n} attribute records for {n_shapes} shapes")
    if buf.size < hlen + n * rlen:
        raise GeoTiffError(f"{path}: truncated: {n} records of {rlen} bytes need {hlen + n * rlen} bytes, "
                           f"the file has {buf.size}")
    found = [i for i, nm in enumerate(names) if nm.upper() == attribute.upper()]
    if not found:
        raise GeoTiffError(f"{path}: no field {attribute!r}; the fields are {names}")
    k = found[0]
    if types[k] not in "NF":
        raise GeoTiffError(f"{path}: field {names[k]!r} has type {types[k]!r}, not numeric (N or F)")
    recs = buf[hlen:hlen + n * rlen].reshape(n, rlen)
    deleted = recs[:, 0] == ord("*")
    w = int(widths[k])
    text = np.ascontiguousarray(recs[:, starts[k]:starts[k] + w]).view(f"S{w}").ravel()
    text = np.char.strip(text)
    text = np.where(text == b"", b"0", text)                                      # a blank value counts as 0
    try:
        values = text.astype(np.float64)
    except ValueError as e:
        raise GeoTiffError(f"{path}: field {names[k]!r} holds a value that is not a number ({e})") from None
    return values, deleted


_PARAM = re.compile(r'PARAMETER\[\s*"([^"]+)"\s*,\s*([-+0-9.eE]+)\s*\]', re.I)
_SPHEROID = re.compile(r'SPHEROID\[\s*"[^"]*"\s*,\s*([-+0-9.eE]+)\s*,\s*([-+0-9.eE]+)', re.I)


def _wgs84_spheroid(wkt):
    m = _SPHEROID.search(wkt)
    return bool(m) and abs(float(m.group(1)) - 6378137.0) < 1e-3 and abs(float(m.group(2)) - 298.257223563) < 1e-6


def read_crs(shp_path):
    """The CRS of a shapefile's ``.prj``: ``EPSG22184`` (the projection block) when it is geographic on the WGS84
    ellipsoid, None when it is POSGAR 94 / Argentina 4 (EPSG:22184).  Anything else, or no ``.prj``, raises."""
    prj = os.path.splitext(str(shp_path))[0] + ".prj"
    if not os.path.exists(prj):
        raise GeoTiffError(f"{prj}: missing; without it the vertices' CRS is unknown")
    with open(prj, "r", errors="replace") as f:
        wkt = f.read().strip()
    head = wkt.upper()
    if head.startswith("GEOGCS"):
        if _wgs84_spheroid(wkt):
            return EPSG22184
        raise GeoTiffError(f"{prj}: a geographic CRS on an ellipsoid other than WGS84 is not supported")
    if head.startswith("PROJCS"):
        tail = re.findall(r'AUTHORITY\[\s*"EPSG"\s*,\s*"?(\d+)"?\s*\]\s*\]\s*$', wkt, re.I)
        if tail and tail[0] == "22184":
            return None
        params = {re.sub(r"[^a-z]", "", k.lower()): float(v) for k, v in _PARAM.findall(wkt)}
        want = {"centralmeridian": -63.0, "latitudeoforigin": -90.0, "scalefactor": 1.0, "falseeasting": 4500000.0,
                "falsenorthing": 0.0}
        if ("TRANSVERSE_MERCATOR" in head.replace(" ", "_") and _wgs84_spheroid(wkt) and
                all(k in params and abs(params[k] - v) < 1e-9 for k, v in want.items()) and
                re.search(r'UNIT\[\s*"(METER|METRE)"\s*,\s*1(\.0*)?\s*[,\]]', wkt, re.I)):
            return None
    raise GeoTiffError(f"{prj}: CRS not supported; geographic WGS84 and POSGAR 94 / Argentina 4 (EPSG:22184) are read")


def read_lines(shp, attribute="UP_CELLS"):
    """An ESRI shapefile of PolyLine / PolyLineZ / PolyLineM shapes -> ``Lines``.  Z and M are ignored, Null shapes and
    deleted records burn nothing, a blank value counts as 0; the value is the numeric ``.dbf`` field ``attribute``, cast
    once to float32 (round to nearest: UP_CELLS above 2^24 is rounded).  Record offsets come from the ``.shx``, which is
    required.  Corrupt or unsupported files raise ``GeoTiffError``."""
    shp = str(shp)
    base = os.path.splitext(shp)[0]
    tm = read_crs(shp)
    buf = _read(shp, "the .shp geometry")
    stype = _check_header(buf, shp)
    if stype not in POLYLINE_TYPES:
        raise GeoTiffError(f"{shp}: shape type {stype} is not supported; PolyLine (3), PolyLineZ (13) and PolyLineM (23) "
                           "are read")
    shx = _read(base + ".shx", "the .shx record index")
    _check_header(shx, base + ".shx")
    if (shx.size - 100) % 8:
        raise GeoTiffError(f"{base}.shx: truncated: {shx.size - 100} index bytes are not whole 8-byte entries")
    index = shx[100:].view(">i4").reshape(-1, 2).astype(np.int64)
    off, clen = 2 * index[:, 0], 2 * index[:, 1]
    n = off.size
    values, deleted = _read_dbf(base + ".dbf", attribute, n)

    if np.any(off < 100) or np.any(clen < 4) or np.any(off + 8 + clen > buf.size):
        r = int(np.flatnonzero((off < 100) | (clen < 4) | (off + 8 + clen > buf.size))[0])
        raise GeoTiffError(f"{shp}: truncated record {r}: {int(clen[r])} bytes at offset {int(off[r])} in a file of "
                           f"{buf.size} bytes")
    rtype = _gather_i4(buf, off + 8)
    bad = (rtype != 0) & (rtype != stype)
    if bad.any():
        r = int(np.flatnonzero(bad)[0])
        raise GeoTiffError(f"{shp}: record {r} has shape type {int(rtype[r])} in a {POLYLINE_TYPES[stype]} file")
    live = rtype != 0
    if np.any(live & (clen < 44)):
        raise GeoTiffError(f"{shp}: truncated record {int(np.flatnonzero(live & (clen < 44))[0])}")
    nparts = np.where(live, _gather_i4(buf, np.where(live, off + 44, 0)), 0)
    npts = np.where(live, _gather_i4(buf, np.where(live, off + 48, 0)), 0)
    bad = (nparts < 0) | (npts < 0) | (live & (44 + 4 * nparts + 16 * npts > clen))
    if bad.any():
        r = int(np.flatnonzero(bad)[0])
        raise GeoTiffError(f"{shp}: truncated record {r}: {int(nparts[r])} parts and {int(npts[r])} points do not fit "
                           f"its {int(clen[r])} bytes")
    # part indices of every record, checked: first 0, non-decreasing, inside the record's point count
    part_rec = np.repeat(np.arange(n), nparts)
    first_part = np.concatenate([[0], np.cumsum(nparts)[:-1]]).astype(np.int64)
    j = np.arange(part_rec.size) - first_part[part_rec]
    parts = _gather_i4(buf, off[part_rec] + 52 + 4 * j) if part_rec.size else np.zeros(0, np.int64)
    prev = np.concatenate([[0], parts[:-1]])
    bad = (parts < 0) | (parts >= npts[part_rec]) | ((j == 0) & (parts != 0)) | ((j > 0) & (parts < prev))
    if bad.any():
        r = int(part_rec[np.flatnonzero(bad)[0]])
        raise GeoTiffError(f"{shp}: record {r}: part index outside its {int(npts[r])} points (or out of order)")

    # keep the records that burn: neither Null nor deleted
    keep = live & ~deleted
    kpts = np.where(keep, npts, 0)
    vbase = np.concatenate([[0], np.cumsum(kpts)[:-1]]).astype(np.int64)
    vrec = np.repeat(np.arange(n), kpts)
    vj = np.arange(vrec.size) - vbase[vrec]
    pos = off[vrec] + 52 + 4 * nparts[vrec] + 16 * vj
    x, y = _gather_f8(buf, pos), _gather_f8(buf, pos + 8)
    pk = keep[part_rec]
    part_start = np.concatenate([vbase[part_rec[pk]] + parts[pk], [vrec.size]]).astype(np.int64)
    if n > np.iinfo(np.int32).max:
        raise GeoTiffError(f"{shp}: {n} records do not fit a 32-bit feature index")
    return Lines(x, y, part_start, part_rec[pk], values.astype(np.float32), tm)


# ---- the device ----------------------------------------------------------------------------------------------------
class DeviceLines:
    """``Lines`` uploaded to the device (torch tensors as plumbing)."""

    def __init__(self, lines):
        import torch
        from . import device as dev
        dev.require_cuda()
        d = dev.device()
        self.x, self.y = torch.from_numpy(lines.x).to(d), torch.from_numpy(lines.y).to(d)
        self.part_start = torch.from_numpy(lines.part_start).to(d)
        self.part_feature = torch.from_numpy(lines.part_feature).to(d)
        self.values = torch.from_numpy(lines.values).to(d)
        self.tm = lines.tm
        self.n_vertices, self.n_parts, self.n_features = lines.n_vertices, lines.n_parts, lines.values.size


def rasterize_to_device(shp_or_lines, grid, attribute="UP_CELLS", workspace=None):
    """Polylines burned onto ``grid`` (a ``warp.Grid``, row bands included) as an F32 DeviceRaster: each cell holds the
    value of the last feature, in file order, whose line walk touches it, 0 where none does.  ``shp_or_lines``: a
    shapefile path, ``Lines`` or ``DeviceLines``.  Launches only (no host synchronisation) when given ``DeviceLines`` and,
    optionally, a workspace of ``hd_rasterize_workspace_bytes`` bytes: capturable in a CUDA graph."""
    import ctypes
    from . import device as dev
    lines = shp_or_lines
    if not isinstance(lines, (Lines, DeviceLines)):
        lines = read_lines(lines, attribute)
    if isinstance(lines, Lines):
        lines = DeviceLines(lines)
    lib = _lib.load()
    need = lib.hd_rasterize_workspace_bytes(lines.n_vertices)
    if workspace is None:
        workspace = dev.scratch(need)
    out = dev.empty(grid.ny, grid.nx, _lib.F32, np.float32)
    p = lambda t: ctypes.c_void_p(t.data_ptr())                                           # noqa: E731
    _lib.check(lib.hd_rasterize_lines(p(lines.x), p(lines.y), lines.n_vertices, p(lines.part_start),
                                      p(lines.part_feature), lines.n_parts, p(lines.values), lines.n_features, out.ptr,
                                      out.pitch, grid.ny, grid.nx, _D4(grid.x0, grid.res, grid.y0, grid.res), grid.row0,
                                      _D7(*lines.tm) if lines.tm is not None else None, p(workspace),
                                      workspace.numel(), dev.stream_ptr()))
    return out


def rasterize_rivers(shp, dst_tif, envelope_or_grid, attribute="UP_CELLS", res=90.0):
    """The reference's river rasterization as one call, file to file: the polylines of ``shp`` (geographic WGS84 or
    EPSG:22184) burned with their ``attribute`` value onto ``envelope_or_grid`` (a Grid, or an ESRI shapefile whose
    bounding box is the area of interest) at ``res`` metres, written to ``dst_tif`` as a Float32 GeoTIFF with the grid's
    georeference.  Returns the Grid."""
    from . import device as dev
    from .geotiff import write_geotiff
    grid = as_grid(envelope_or_grid, res)
    out = rasterize_to_device(shp, grid, attribute)
    write_geotiff(dst_tif, dev.download(out), dtype=np.float32, geo_tags=grid.geo_tags())
    return grid

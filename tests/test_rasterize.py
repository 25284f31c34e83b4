"""CPU: the river-line rasterization's host side (hydrodem_b200/rasterize.py) -- the shapefile reader on files written here
with ``struct``, the oracle's Bresenham loop and its closed form, and the library's host forward projection against the
float64 oracle."""
import ctypes
import os
import struct

import numpy as np
import pytest

from hydrodem_b200 import _lib
from hydrodem_b200 import rasterize as hr
from hydrodem_b200.geotiff import GeoTiffError
from oracle import rasterize as orr
from oracle import warp as ow

GEOG_PRJ = ('GEOGCS["GCS_WGS_1984",DATUM["D_WGS_1984",SPHEROID["WGS_1984",6378137.0,298.257223563]],'
            'PRIMEM["Greenwich",0.0],UNIT["Degree",0.0174532925199433]]')
POSGAR4_PRJ = ('PROJCS["POSGAR_1994_Argentina_4",GEOGCS["GCS_POSGAR_1994",DATUM["D_POSGAR_1994",'
               'SPHEROID["WGS_1984",6378137.0,298.257223563]],PRIMEM["Greenwich",0.0],UNIT["Degree",0.0174532925199433]],'
               'PROJECTION["Transverse_Mercator"],PARAMETER["False_Easting",4500000.0],PARAMETER["False_Northing",0.0],'
               'PARAMETER["Central_Meridian",-63.0],PARAMETER["Scale_Factor",1.0],PARAMETER["Latitude_Of_Origin",-90.0],'
               'UNIT["Meter",1.0]]')
EPSG_PRJ = ('PROJCS["POSGAR 94 / Argentina 4",GEOGCS["POSGAR 94",DATUM["Posiciones_Geodesicas_Argentinas_1994",'
            'SPHEROID["WGS 84",6378137,298.257223563]],PRIMEM["Greenwich",0],UNIT["degree",0.0174532925199433]],'
            'PROJECTION["Transverse_Mercator"],PARAMETER["latitude_of_origin",-90],PARAMETER["central_meridian",-63],'
            'PARAMETER["scale_factor",1],PARAMETER["false_easting",4500000],PARAMETER["false_northing",0],'
            'UNIT["metre",1],AUTHORITY["EPSG","22184"]]')


def write_shapefile(path, records, values, shape_type=3, prj=GEOG_PRJ, field="UP_CELLS", deleted=(), width=12,
                    extra_fields=(("NAME", "C", 8),)):
    """ESRI shapefile of polylines.  records[i]: None (a Null shape) or a list of parts, each a list of (x, y).
    values[i]: a number, or None for a blank field.  Z / M values are written for types 13 / 23 and must be ignored."""
    recs = []
    for r in records:
        if r is None:
            recs.append(struct.pack("<i", 0))
            continue
        pts = [p for part in r for p in part]
        xs, ys = [p[0] for p in pts] or [0.0], [p[1] for p in pts] or [0.0]
        c = struct.pack("<i4dii", shape_type, min(xs), min(ys), max(xs), max(ys), len(r), len(pts))
        starts, k = [], 0
        for part in r:
            starts.append(k)
            k += len(part)
        c += struct.pack(f"<{len(r)}i", *starts)
        c += b"".join(struct.pack("<2d", *p) for p in pts)
        if shape_type == 13:
            c += struct.pack(f"<2d{len(pts)}d", -1.0, 1.0, *[1e9] * len(pts))
        if shape_type in (13, 23):
            c += struct.pack(f"<2d{len(pts)}d", 0.0, 5.0, *[-7.0] * len(pts))
        recs.append(c)

    def header(nbytes):
        return (struct.pack(">i", 9994) + b"\0" * 20 + struct.pack(">i", nbytes // 2) +
                struct.pack("<ii", 1000, shape_type) + struct.pack("<8d", 0, 0, 1, 1, 0, 0, 0, 0))

    body, index, off = b"", b"", 100
    for i, c in enumerate(recs):
        body += struct.pack(">ii", i + 1, len(c) // 2) + c
        index += struct.pack(">ii", off // 2, len(c) // 2)
        off += 8 + len(c)
    base = os.path.splitext(str(path))[0]
    with open(base + ".shp", "wb") as f:
        f.write(header(100 + len(body)) + body)
    with open(base + ".shx", "wb") as f:
        f.write(header(100 + len(index)) + index)
    fields = [(field, "N", width)] + list(extra_fields)
    rlen = 1 + sum(w for _, _, w in fields)
    hlen = 32 + 32 * len(fields) + 1
    dbf = struct.pack("<B3BIHH20x", 3, 126, 1, 1, len(records), hlen, rlen)
    for name, typ, w in fields:
        dbf += name.encode().ljust(11, b"\0") + typ.encode() + b"\0" * 4 + bytes([w, 0]) + b"\0" * 14
    dbf += b"\r"
    for i, v in enumerate(values):
        dbf += b"*" if i in deleted else b" "
        dbf += (b"" if v is None else repr(v).encode()).rjust(width)
        for _, _, w in fields[1:]:
            dbf += f"r{i}".encode().ljust(w)
    dbf += b"\x1a"
    with open(base + ".dbf", "wb") as f:
        f.write(dbf)
    if prj is not None:
        with open(base + ".prj", "w") as f:
            f.write(prj)
    return base + ".shp"


MULTI = [[[(0.5, 0.5), (3.5, 1.5)], [(10.0, 10.0), (11.0, 12.0), (12.5, 12.5)]],
         None,
         [[(-2.0, 5.0), (7.0, -3.0)]],
         [[(1.0, 1.0)]]]


# ---- the reader ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape_type", [3, 13, 23])
def test_reader_multipart_null_and_z_m(tmp_path, shape_type):
    shp = write_shapefile(tmp_path / "r.shp", MULTI, [5, 9, 7.5, 2], shape_type=shape_type)
    L = hr.read_lines(shp)
    assert L.tm == ow.EPSG22184
    pts = [p for r in MULTI if r for part in r for p in part]
    np.testing.assert_array_equal(L.x, [p[0] for p in pts])
    np.testing.assert_array_equal(L.y, [p[1] for p in pts])
    np.testing.assert_array_equal(L.part_start, [0, 2, 5, 7, 8])
    np.testing.assert_array_equal(L.part_feature, [0, 0, 2, 3])          # record 1 is Null: no part
    np.testing.assert_array_equal(L.values, np.float32([5, 9, 7.5, 2]))


def test_reader_deleted_blank_and_float32_rounding(tmp_path):
    recs = [[[(0.0, 0.0), (1.0, 1.0)]], [[(2.0, 2.0), (3.0, 3.0)]], [[(4.0, 4.0), (5.0, 5.0)]]]
    shp = write_shapefile(tmp_path / "d.shp", recs, [16777217, None, 3], deleted={2}, width=14)
    L = hr.read_lines(shp)
    np.testing.assert_array_equal(L.values, np.float32([16777216, 0, 3]))  # 2^24 + 1 rounds to even; blank is 0
    np.testing.assert_array_equal(L.part_feature, [0, 1])                 # the deleted record burns nothing
    np.testing.assert_array_equal(L.part_start, [0, 2, 4])
    np.testing.assert_array_equal(L.x, [0, 1, 2, 3])


def test_reader_field_name_and_missing_field(tmp_path):
    recs = [[[(0.0, 0.0), (1.0, 1.0)]]]
    shp = write_shapefile(tmp_path / "f.shp", recs, [4], field="up_cells")
    assert hr.read_lines(shp).values[0] == 4
    shp = write_shapefile(tmp_path / "g.shp", recs, [4], field="ORD_STRA")
    with pytest.raises(GeoTiffError, match=r"no field 'UP_CELLS'.*ORD_STRA.*NAME"):
        hr.read_lines(shp)
    assert hr.read_lines(shp, attribute="ORD_STRA").values[0] == 4
    with pytest.raises(GeoTiffError, match="not numeric"):
        hr.read_lines(shp, attribute="NAME")


def test_reader_crs(tmp_path):
    recs = [[[(4.4e6, 6.1e6), (4.41e6, 6.11e6)]]]
    for prj in (POSGAR4_PRJ, EPSG_PRJ):
        assert hr.read_lines(write_shapefile(tmp_path / "p.shp", recs, [1], prj=prj)).tm is None
    assert hr.read_lines(write_shapefile(tmp_path / "p.shp", recs, [1], prj=GEOG_PRJ)).tm == ow.EPSG22184
    utm = EPSG_PRJ.replace('"central_meridian",-63', '"central_meridian",-69').replace('"22184"', '"22182"')
    for bad in (utm, GEOG_PRJ.replace("298.257223563", "298.257222101"), 'LOCAL_CS["x"]'):
        with pytest.raises(GeoTiffError, match="not supported"):
            hr.read_lines(write_shapefile(tmp_path / "p.shp", recs, [1], prj=bad))
    shp = write_shapefile(tmp_path / "n.shp", recs, [1], prj=None)
    with pytest.raises(GeoTiffError, match=r"\.prj: missing"):
        hr.read_lines(shp)


def test_reader_missing_sidecars_and_wrong_type(tmp_path):
    recs = [[[(0.0, 0.0), (1.0, 1.0)]]]
    shp = write_shapefile(tmp_path / "a.shp", recs, [1])
    os.remove(str(tmp_path / "a.shx"))
    with pytest.raises(GeoTiffError, match=r"\.shx: missing"):
        hr.read_lines(shp)
    shp = write_shapefile(tmp_path / "b.shp", recs, [1])
    os.remove(str(tmp_path / "b.dbf"))
    with pytest.raises(GeoTiffError, match=r"\.dbf: missing"):
        hr.read_lines(shp)
    for t in (1, 5, 8, 15, 25):                                            # points, polygons, multipoints
        with pytest.raises(GeoTiffError, match=f"shape type {t} is not supported"):
            hr.read_lines(write_shapefile(tmp_path / "c.shp", recs, [1], shape_type=t))


def _patch(path, offset, data):
    with open(path, "r+b") as f:
        f.seek(offset)
        f.write(data)


def test_reader_corrupt_files(tmp_path):
    recs = [[[(0.0, 0.0), (1.0, 1.0), (2.0, 0.0)], [(5.0, 5.0), (6.0, 6.0)]], [[(1.0, 2.0), (3.0, 4.0)]]]
    mk = lambda: write_shapefile(tmp_path / "x.shp", recs, [1, 2])                   # noqa: E731
    base = str(tmp_path / "x")
    shp = mk()
    _patch(shp, 0, struct.pack(">i", 1234))
    with pytest.raises(GeoTiffError, match="9994"):
        hr.read_lines(shp)
    shp = mk()
    with open(shp, "r+b") as f:
        f.truncate(os.path.getsize(shp) - 9)
    with pytest.raises(GeoTiffError, match="truncated record 1"):
        hr.read_lines(shp)
    shp = mk()                                                             # record 0: 2 parts, 5 points
    _patch(shp, 100 + 48, struct.pack("<i", 50))
    with pytest.raises(GeoTiffError, match="truncated record 0"):
        hr.read_lines(shp)
    shp = mk()
    _patch(shp, 100 + 56, struct.pack("<i", 5))                         # second part starts at point 5 of 5
    with pytest.raises(GeoTiffError, match="part index"):
        hr.read_lines(shp)
    shp = mk()
    _patch(shp, 100 + 56, struct.pack("<i", -1))
    with pytest.raises(GeoTiffError, match="part index"):
        hr.read_lines(shp)
    shp = mk()
    with open(base + ".shx", "r+b") as f:
        f.truncate(100 + 8 + 3)
    with pytest.raises(GeoTiffError, match="shx: truncated"):
        hr.read_lines(shp)
    shp = mk()
    _patch(base + ".dbf", 8, struct.pack("<H", 40))                        # header length not 32 k + 1
    with pytest.raises(GeoTiffError, match="bad .dbf header"):
        hr.read_lines(shp)
    shp = mk()
    _patch(base + ".dbf", 4, struct.pack("<I", 3))
    with pytest.raises(GeoTiffError, match="3 attribute records for 2 shapes"):
        hr.read_lines(shp)
    shp = mk()
    with open(base + ".dbf", "r+b") as f:
        f.truncate(os.path.getsize(base + ".dbf") - 10)
    with pytest.raises(GeoTiffError, match="dbf: truncated"):
        hr.read_lines(shp)
    shp = write_shapefile(tmp_path / "x.shp", recs, [1, 2])
    _patch(base + ".dbf", 97 + 21 + 1, b"abc")                            # the second record's value: not a number
    with pytest.raises(GeoTiffError, match="not a number"):
        hr.read_lines(shp)


# ---- the line rule -------------------------------------------------------------------------------------------------
def test_closed_form_is_the_error_accumulating_loop():
    """floor((2 k |dy| + |dx| - 1) / (2 |dx|)) is GDALdllImageLine's minor offset after k steps: the nearest integer to
    k |dy| / |dx|, exact halves rounded toward the start vertex."""
    for adx in range(0, 200):
        for ady in range(0, adx + 1):
            walk = orr.bresenham(0, 0, adx, ady)
            closed = [(k, (2 * k * ady + adx - 1) // (2 * adx) if adx else 0) for k in range(adx + 1)]
            assert walk == closed, (adx, ady)
    assert orr.bresenham(0, 0, 2, 1) == [(0, 0), (1, 0), (2, 1)]          # the tie at k = 1 stays on the start row
    assert orr.bresenham(2, 1, 0, 0) == [(2, 1), (1, 1), (0, 0)]


def test_oracle_line_loop():
    rng = np.random.default_rng(1)
    for _ in range(2000):
        x0, y0, x1, y1 = (int(v) for v in rng.integers(-40, 40, 4))
        walk = orr.bresenham(x0, y0, x1, y1)
        assert walk[0] == (x0, y0) and walk[-1] == (x1, y1)
        assert len(walk) == max(abs(x1 - x0), abs(y1 - y0)) + 1
        assert all(max(abs(a[0] - b[0]), abs(a[1] - b[1])) == 1 for a, b in zip(walk, walk[1:]))      # 8-connected
    assert orr.bresenham(3, 4, 3, 4) == [(3, 4)]


def test_oracle_replace_order_and_degenerate_parts():
    pixels = [(0, 0), (4, 0), (2, 0), (2, 0), (1, 1), None, (3, 3), (9, 9), (0, 2)]
    # feature 1 (listed first) is later in file order than feature 0: its value wins where both burn
    out = orr.burn(pixels, [0, 2, 4, 5, 7, 8, 9], [1, 0, 0, 2, 2, 2], [10.0, 20.0, 30.0], 4, 5)
    assert out[0].tolist() == [20, 20, 20, 20, 20]                         # part 0 over the zero-length part 1
    assert out[1, 1] == 0                                                  # a single-vertex part burns nothing
    assert out[3, 3] == 0 and out[2, 0] == 0                               # segments with a missing end are skipped
    assert (out[3] == 0).all()
    band = orr.burn(pixels, [0, 2, 4, 5, 7, 8, 9], [1, 0, 0, 2, 2, 2], [10.0, 20.0, 30.0], 2, 5, row0=0)
    np.testing.assert_array_equal(band, out[:2])


# ---- the host forward projection -----------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        from hydrodem_b200.build import build
        build()
    return _lib.load()


def test_library_forward_matches_the_oracle(lib):
    rng = np.random.default_rng(7)
    lon, lat = rng.uniform(-75, -51, 20000), rng.uniform(-56, -21, 20000)
    lon[:3], lat[:3] = (-75.0, -63.0, -51.0), (-56.0, -21.0, -21.0)
    x, y = np.empty_like(lon), np.empty_like(lat)
    p = lambda a: ctypes.c_void_p(a.ctypes.data)                                       # noqa: E731
    tm = (ctypes.c_double * 7)(*ow.EPSG22184)
    assert lib.hd_host_tm_forward(tm, p(lon), p(lat), lon.size, p(x), p(y)) == _lib.HD_OK
    ox, oy = ow.tm_forward(lon, lat)
    assert np.abs(x - ox).max() < 1e-6 and np.abs(y - oy).max() < 1e-6
    glon, glat = np.empty_like(x), np.empty_like(y)
    assert lib.hd_host_tm_inverse(tm, p(x), p(y), x.size, p(glon), p(glat)) == _lib.HD_OK
    assert np.abs(glon - lon).max() < 1e-9 and np.abs(glat - lat).max() < 1e-9
    bad = (ctypes.c_double * 7)(6378137.0, 1.5, *ow.EPSG22184[2:])
    assert lib.hd_host_tm_forward(bad, p(lon), p(lat), lon.size, p(x), p(y)) == _lib.HD_ERR_ARG
    assert lib.hd_host_tm_forward(tm, None, p(lat), lon.size, p(x), p(y)) == _lib.HD_ERR_NULL


def test_rasterize_argument_errors_need_no_gpu(lib):
    q = ctypes.c_void_p(1 << 20)
    g = (ctypes.c_double * 4)(0.0, 90.0, 0.0, 90.0)
    need = lib.hd_rasterize_workspace_bytes(1000)
    assert need >= 1000 * 24 and lib.hd_rasterize_workspace_bytes(-1) == 0

    def call(nv=1000, nparts=10, nfeat=10, ny=64, nx=64, pitch=64, geo=g, row0=0, ws=need, dst=q, vx=q):
        return lib.hd_rasterize_lines(vx, q, nv, q, q, nparts, q, nfeat, dst, pitch, ny, nx, geo, row0, None, q, ws, None)

    assert call(dst=None) == _lib.HD_ERR_NULL and call(vx=None) == _lib.HD_ERR_NULL
    assert call(nv=-1) == _lib.HD_ERR_ARG and call(nparts=-1) == _lib.HD_ERR_ARG
    assert call(nfeat=2 ** 31) == _lib.HD_ERR_ARG                          # more features than a 32-bit index holds
    assert call(ny=0) == _lib.HD_ERR_ARG and call(pitch=63) == _lib.HD_ERR_ARG and call(row0=-1) == _lib.HD_ERR_ARG
    assert call(nx=2 ** 29 + 1, pitch=2 ** 29 + 1) == _lib.HD_ERR_ARG
    assert call(geo=(ctypes.c_double * 4)(0.0, -90.0, 0.0, 90.0)) == _lib.HD_ERR_ARG
    assert call(ws=need - 1) == _lib.HD_ERR_WORKSPACE
    bad = (ctypes.c_double * 7)(-1.0, *ow.EPSG22184[1:])
    assert lib.hd_rasterize_lines(q, q, 1000, q, q, 10, q, 10, q, 64, 64, 64, g, 0, bad, q, need, None) == _lib.HD_ERR_ARG


def test_rasterize_without_a_device_is_an_error(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("checks the no-GPU behaviour")
    q = ctypes.c_void_p(1 << 20)
    g = (ctypes.c_double * 4)(0.0, 90.0, 0.0, 90.0)
    need = lib.hd_rasterize_workspace_bytes(1000)
    assert lib.hd_rasterize_lines(q, q, 1000, q, q, 10, q, 10, q, 64, 64, 64, g, 0, None, q, need, None) == _lib.HD_ERR_CUDA

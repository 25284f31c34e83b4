"""GPU: compressed GeoTIFFs decoded on the device (hd_tiff_decode, DESIGN §9d).  read_to_device gives the same bits as
read_array on the host (sign of zero and NaN payloads included) for LZW and Deflate, every predictor, every device sample
type, both byte orders, strips and ragged tiles; the host fallback for over-long Deflate blocks and LZW zero padding;
corrupt blocks raise GeoTiffError naming the block and leave the device usable; compressed tile mosaics and
process_geotiffs give the bits of the same files uncompressed."""
import zlib

import numpy as np
import pytest
import torch
from PIL import Image

import tiff_builder as tb
from test_warp_mosaic import GEOGRAPHIC, _tags

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200 import device as dev, geotiff
    from hydrodem_b200 import warp as hw
    from hydrodem_b200.exceptions import DeviceError
    from hydrodem_b200.pipeline import ConditioningChain
    from hydrodem_b200.synth import SynthScene
    from oracle import warp as ow

DTYPES = [np.uint8, np.int16, np.int32, np.int64, np.float32, np.float64]
LAYOUTS = [{"rows": 1}, {"rows": 16}, {"tile": (16, 32)}]


def _raster(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    if np.dtype(dtype).kind == "f":
        a = np.round(rng.standard_normal(shape).cumsum(1) * 7.3, 2).astype(dtype)
        bits = a.view(np.uint32 if a.itemsize == 4 else np.uint64).reshape(-1)
        one = np.dtype(bits.dtype).type(1)
        sign = one << np.dtype(bits.dtype).type(8 * a.itemsize - 1)
        bits[:5] = [0, sign, np.array(np.nan, dtype).view(bits.dtype) | one,                    # +0, -0, NaN payloads
                    np.array(np.nan, dtype).view(bits.dtype) | sign | (one << 3),
                    np.array(np.inf, dtype).view(bits.dtype)]
        return a
    info = np.iinfo(dtype)
    smooth = (rng.standard_normal(shape).cumsum(1) * 40).astype(np.int64)
    a = smooth.astype(dtype) if info.bits == 64 else (smooth % (int(info.max) - int(info.min) + 1) + int(info.min)).astype(dtype)
    a[0, :4] = [info.min, info.max, 0, info.min]
    return a


def _same(got, want):
    assert got.dtype == want.dtype and got.shape == want.shape
    np.testing.assert_array_equal(got.view(np.uint8), np.ascontiguousarray(want).view(np.uint8))


def _check(path, **kw):
    want = geotiff.read_array(path, pinned=False)
    got = dev.download(geotiff.read_to_device(path, **kw))
    _same(got, want)
    return want


@pytest.mark.parametrize("bo", ["<", ">"])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("compression", [5, 8, 32946])
def test_same_bits_as_read_array(tmp_path, compression, dtype, bo):
    a = _raster((45, 70), dtype, 1)
    preds = (1, 3) if np.dtype(dtype).kind == "f" else (1, 2)
    for pred in preds:
        for k, layout in enumerate(LAYOUTS):
            p = tb.write(tmp_path / f"{pred}_{k}.tif", a, compression, pred, bo, **layout)
            _same(_check(p), a)


@pytest.mark.parametrize("comp", ["tiff_lzw", "tiff_adobe_deflate", "tiff_deflate"])
@pytest.mark.parametrize("mode,dtype,pred", [("L", np.uint8, 2), ("I", np.int32, 2), ("F", np.float32, 1)])
def test_files_written_by_libtiff(tmp_path, comp, mode, dtype, pred):
    yy, xx = np.mgrid[0:300, 0:400]
    a = np.round(100 + 20 * np.sin(xx / 40.0) + 15 * np.cos(yy / 55.0)).astype(dtype)
    p = tmp_path / "p.tif"
    im = Image.fromarray(a)
    assert im.mode == mode
    im.save(p, format="TIFF", compression=comp, tiffinfo={317: pred} if pred != 1 else {})
    assert len(geotiff.read_info(p).offsets) > 1
    _same(_check(p), a)


def test_unsupported_sample_type_raises_as_before(tmp_path):
    a = np.arange(600, dtype=np.uint16).reshape(20, 30)
    p = tmp_path / "u16.tif"
    Image.fromarray(a).save(p, format="TIFF", compression="tiff_lzw")
    with pytest.raises(DeviceError):
        geotiff.read_to_device(p)
    p = tb.write(tmp_path / "f2.tif", np.zeros((8, 8), np.float32), 8, 2)
    with pytest.raises(geotiff.GeoTiffError, match="horizontal predictor"):
        geotiff.read_to_device(p)


def test_thousands_of_blocks_and_many_batches(tmp_path):
    a = _raster((3001, 517), np.int16, 5)
    p = tb.write(tmp_path / "strips.tif", a, 8, 2, rows=1)
    assert len(geotiff.read_info(p).offsets) == 3001
    _check(p, chunk_bytes=40_000)
    _check(p)
    p = tb.write(tmp_path / "tiles.tif", a, 5, 2, tile=(16, 16))
    _check(p, chunk_bytes=30_000)


def test_host_fallback_for_long_deflate_blocks(tmp_path):
    """A Deflate block that decodes to more than the block holds is legal (the surplus is ignored): the device stops at the
    block's end, and the host decodes that block again."""
    a = _raster((40, 50), np.int16, 7)
    blocks = []
    for y0, _, b in tb.blocks_of(a, rows=16):
        raw = tb.predict(b, 2, np.dtype("<i2"))
        blocks.append(zlib.compress(raw + (b"extra bytes" * 9 if y0 == 16 else b"")))
    p = tb.write(tmp_path / "long.tif", a, 8, 2, rows=16, blocks=blocks)
    _same(_check(p, chunk_bytes=1), a)


def test_lzw_without_eoi_and_short_strips_are_zero_padded(tmp_path):
    a = _raster((40, 50), np.uint8, 8)
    blocks = []
    for y0, _, b in tb.blocks_of(a, rows=16):
        raw = tb.predict(b, 1, np.dtype("u1"))
        blocks.append(tb.lzw_encode(raw, eoi=False) if y0 == 0 else tb.lzw_encode(raw[:300]) if y0 == 16 else
                      tb.lzw_encode(raw))
    p = tb.write(tmp_path / "pad.tif", a, 5, 1, rows=16, blocks=blocks)
    want = _check(p)
    _same(want[:16], a[:16])
    assert (want[16:32].reshape(-1)[300:] == 0).all()


def test_corrupt_blocks_raise_and_the_device_stays_usable(tmp_path):
    a = _raster((64, 40), np.int16, 9)
    good = tb.write(tmp_path / "good.tif", a, 8, 2, rows=8)
    for comp, k, damage in ((8, 3, "adler"), (8, 5, "short"), (5, 6, "code"), (8, 0, "sparse")):
        blocks = [tb.compress(tb.predict(b, 2, np.dtype("<i2")), comp) for _, _, b in tb.blocks_of(a, rows=8)]
        if damage == "adler":
            blocks[k] = blocks[k][:-1] + bytes([blocks[k][-1] ^ 1])
        elif damage == "short":
            blocks[k] = zlib.compress(tb.predict(a[:7], 2, np.dtype("<i2")))       # decodes to 7 of the 8 rows
        elif damage == "code":
            blocks[k] = b"\x80\x3f\xff\xff\xff"                                  # Clear, then a code beyond the table
        else:
            blocks[k] = b""
        p = tb.write(tmp_path / f"bad_{damage}.tif", a, comp, 2, rows=8, blocks=blocks)
        with pytest.raises(geotiff.GeoTiffError, match=f"block {k}\\b"):
            geotiff.read_to_device(p)
        _same(dev.download(geotiff.read_to_device(good)), a)


# ---- the files-in path over compressed inputs -----------------------------------------------------------------------
D = 1.0 / 3600.0
LON0, LAT0 = -64.0, -34.0


def _tile_files(tmp_path, prefix, compression):
    """3 x 4 int16 1" tiles of 361 x 361 sharing their edges (nodata -32768), written uncompressed or with Deflate /
    LZW + predictor 2 in 256 x 256 tiles or 8-row strips."""
    paths = []
    for r in range(3):
        for c in range(4):
            V, U = np.mgrid[360 * r:360 * r + 361, 360 * c:360 * c + 361]
            a = ((U * 37 + V * 101) % 6000 - 300).astype(np.int16)
            a[(U * 7919 + V * 104729) % 53 == 0] = -32768
            tags = _tags(LON0 + 0.1 * c - 0.5 * D, LAT0 - 0.1 * r + 0.5 * D, D, D, GEOGRAPHIC)
            nd = b"-32768\0"
            tags[geotiff.GDAL_NODATA] = (2, len(nd), nd)
            p = tmp_path / f"{prefix}{r}{c}.tif"
            if compression is None:
                geotiff.write_geotiff(p, a, geo_tags=tags, nodata=-32768)
            else:
                layout = {"tile": (256, 256)} if (r + c) % 2 else {"rows": 8}
                tb.write(p, a, compression, 2, extra_tags=tags, **layout)
            paths.append(str(p))
    return paths


def test_warp_of_a_compressed_mosaic(tmp_path):
    plain = _tile_files(tmp_path, "plain", None)
    x0, y1 = ow.tm_forward(LON0 - 0.03, LAT0 + 0.02)
    x1, y0 = ow.tm_forward(LON0 + 0.43, LAT0 - 0.33)
    grid = hw.Grid(float(x0) + 0.37, float(y1) - 0.81, 90.0, int((x1 - x0) / 90), int((y1 - y0) / 90))
    for comp in (8, 5):
        packed = _tile_files(tmp_path, f"c{comp}_", comp)
        for resample in ("nearest", "bilinear"):
            want = dev.download(hw.warp_to_device(plain, grid, resample))
            got = dev.download(hw.warp_to_device(packed, grid, resample))
            np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))


def test_process_geotiffs_on_compressed_inputs(tmp_path):
    sc = SynthScene(900, 900, 9)
    rasters = {"srtm": (sc.srtm().astype(np.float32), 3), "groves": (sc.groves().astype(np.uint8), 1),
               "hsheds": (sc.hsheds().astype(np.float32), 3)}
    plain, packed = {}, {}
    for k, (a, pred) in rasters.items():
        tags = _tags(LON0, LAT0, D, D, GEOGRAPHIC)
        plain[k] = str(tmp_path / f"{k}.tif")
        geotiff.write_geotiff(plain[k], a, geo_tags=tags)
        packed[k] = str(tb.write(tmp_path / f"{k}_z.tif", a, 8, pred, tile=(128, 128), extra_tags=tags))
        _same(dev.download(geotiff.read_to_device(packed[k])), a)
    x0, y1 = ow.tm_forward(LON0 + 0.02, LAT0 - 0.02)
    grid = hw.Grid(float(x0), float(y1), 90.0, 200, 240)
    outs = []
    for files in (plain, packed):
        final = str(tmp_path / f"final_{len(outs)}.tif")
        outs.append(geotiff.process_geotiffs(files["srtm"], files["groves"], files["hsheds"], final,
                                             chain=ConditioningChain(), envelope=grid))
    for key in ("final", "filled", "d8"):
        np.testing.assert_array_equal(outs[1][key], outs[0][key])

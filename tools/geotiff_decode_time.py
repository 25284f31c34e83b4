"""Compressed GeoTIFF ingest on the GPU (hd_tiff_decode, DESIGN §9d):  python tools/geotiff_decode_time.py [--size N] [--only rasters|mosaic]

Writes seeded files into a temporary directory and prints one JSON record per case:
  * an 18000 x 18000 int16 DEM-like raster (the sum of two random walks, one along the rows and one along the columns,
    plus 0.5 m noise, rounded to metres) with Deflate + predictor 2 and with LZW + predictor 2, each in GDAL's default
    one-row strips and in 256 x 256 tiles (LZW blocks are encoded by libtiff through Pillow, one block per image);
  * the same field as float32 with Deflate + predictor 3 in one-row strips;
  * the §9c workload: a 4096 x 4096 90 m grid warped (nearest) from the 24 int16 1" tiles of 3601 x 3601 it meets, the
    tiles written with Deflate + predictor 2 in 256 x 256 tiles against the same tiles uncompressed.
Each record: the card's name and power limit (read in the same run); compressed and decoded bytes and the block count;
the decode + store kernel time (CUDA events around one hd_tiff_decode call over every block of the file, its compressed
bytes already on the device; best of 5 after warm-up) and the decoded GB/s it gives; read_to_device file -> device
against dev.upload(read_array(path)) on the same file, run alternately, best of 3 each; whether the files were in the page
cache (they were written by this run just before: yes).  Without a GPU it fails."""
import argparse
import concurrent.futures as cf
import ctypes
import io
import json
import os
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from hydrodem_b200 import _lib, device as dev, geotiff                                   # noqa: E402
from hydrodem_b200 import warp as hw                                                     # noqa: E402
import tiff_builder as tb                                                                # noqa: E402

dev.require_cuda()
lib = _lib.load()
POOL = cf.ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else "unknown"


def dem(ny, nx, seed):
    rng = np.random.default_rng(seed)
    z = (rng.standard_normal(ny, dtype=np.float32).cumsum()[:, None] * 2 +
         rng.standard_normal(nx, dtype=np.float32).cumsum()[None, :] * 2 + 300)
    z += rng.standard_normal((ny, nx), dtype=np.float32) * 0.5
    return np.round(z)


def lzw_block(block, predictor):
    """One block's LZW bytes as libtiff encodes them: int16 samples as a uint16 image of one strip (the same bytes)."""
    buf = io.BytesIO()
    Image.fromarray(np.ascontiguousarray(block).view(np.uint16)).save(
        buf, format="TIFF", compression="tiff_lzw", tiffinfo={317: predictor, 278: block.shape[0]})
    im = Image.open(io.BytesIO(buf.getvalue()))
    off, count = im.tag_v2[273][0], im.tag_v2[279][0]
    return buf.getvalue()[off:off + count]


def write(path, a, compression, predictor, layout, extra_tags=None):
    parts = tb.blocks_of(a, **layout)
    dt = np.dtype("<" + a.dtype.str[1:])
    if compression == 5:
        blocks = list(POOL.map(lambda p: lzw_block(p[2], predictor), parts))
    else:
        blocks = list(POOL.map(lambda p: zlib.compress(tb.predict(p[2], predictor, dt), 6), parts))
    tb.write(path, a, compression, predictor, extra_tags=extra_tags, blocks=blocks, **layout)
    return sum(len(b) for b in blocks), len(blocks)


def kernel_ms(path):
    """Best of 5 decode + store times (ms) of one hd_tiff_decode call over all blocks, after warm-up."""
    info = geotiff.read_info(path)
    tbl = geotiff._block_table(path, info)
    raw = np.fromfile(path, dtype=np.uint8)
    src = torch.from_numpy(raw).cuda()
    blocks = torch.from_numpy(np.ascontiguousarray(tbl[:, 1:])).cuda()
    native = info.dtype.newbyteorder("=")
    hd = dev.hd_dtype_of(native)
    out = dev.empty(info.height, info.width, hd, native)
    status = torch.zeros(len(tbl), dtype=torch.int32, device="cuda")
    wsb = lib.hd_tiff_decode_workspace_bytes(len(tbl), info.block_h, info.block_w, hd)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")

    def run():
        _lib.check(lib.hd_tiff_decode(ctypes.c_void_p(src.data_ptr()), raw.size, ctypes.c_void_p(blocks.data_ptr()),
                                      len(tbl), info.compression, info.predictor, hd, 0, out.ptr, out.pitch,
                                      info.height, info.width, info.block_h, info.block_w,
                                      ctypes.c_void_p(status.data_ptr()), ctypes.c_void_p(ws.data_ptr()), wsb,
                                      dev.stream_ptr()))
    run()
    torch.cuda.synchronize()
    assert int(status.max()) == 0, "a block did not decode on the device"
    best = float("inf")
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return best, out


def file_to_device(path, rounds=3):
    """Best of ``rounds`` of read_to_device and of upload(read_array), alternated; asserts the same bits."""
    t_dev, t_host = [], []
    for _ in range(rounds):
        torch.cuda.synchronize()
        t = time.perf_counter()
        a = geotiff.read_to_device(path)
        torch.cuda.synchronize()
        t_dev.append(time.perf_counter() - t)
        t = time.perf_counter()
        b = dev.upload(geotiff.read_array(path, pinned=True))
        torch.cuda.synchronize()
        t_host.append(time.perf_counter() - t)
    assert torch.equal(a.tensor().view(torch.uint8), b.tensor().view(torch.uint8))
    return min(t_dev), min(t_host)


def record(name, path, a, comp_bytes, nblocks, gpu):
    ms, out = kernel_ms(path)
    assert np.array_equal(dev.download(out).view(np.uint8), a.view(np.uint8))
    t_dev, t_host = file_to_device(path)
    rec = {"case": name, "card": gpu, "shape": list(a.shape), "dtype": a.dtype.name, "compressed_bytes": comp_bytes,
           "decoded_bytes": int(a.nbytes), "ratio": round(a.nbytes / comp_bytes, 2), "blocks": nblocks,
           "kernel_ms_best_of_5": round(ms, 3), "kernel_decoded_GBps": round(a.nbytes / ms / 1e6, 2),
           "read_to_device_s": round(t_dev, 4), "upload_read_array_s": round(t_host, 4),
           "speedup": round(t_host / t_dev, 2), "page_cache": True}
    print(json.dumps(rec), flush=True)


def mosaic_case(tmp, gpu):
    d = 1.0 / 3600.0
    keys = np.array([1, 1, 0, 3, 1024, 0, 1, 2, 1025, 0, 1, 1, 2048, 0, 1, 4326], "<u2")
    n = 4096                                             # tools/warp_time.py's grid: centred about 35 S on the meridian
    cx, cy = 4500000.0, 10001965.729312724 - 35.0 * 111000.0
    grid = hw.Grid(cx - n * 45.0, cy + n * 45.0, 90.0, n, n)
    lon0, lon1, lat0, lat1 = hw.footprint(grid, hw.EPSG22184)
    plain, packed, comp, nblk = [], [], 0, 0
    for lat in range(int(np.ceil(lat1)), int(np.floor(lat0)), -1):
        for lon in range(int(np.floor(lon0)), int(np.ceil(lon1))):
            a = dem(3601, 3601, 1000 + 7 * lat + lon).astype(np.int16)
            tags = {33550: (12, 3, np.array([d, d, 0.0], "<f8").tobytes()),
                    33922: (12, 6, np.array([0, 0, 0, lon - d / 2, lat + d / 2, 0], "<f8").tobytes()),
                    34735: (3, keys.size, keys.tobytes())}
            p = os.path.join(tmp, f"t{lat}_{lon}.tif")
            geotiff.write_geotiff(p, a, geo_tags=tags)
            plain.append(p)
            q = os.path.join(tmp, f"z{lat}_{lon}.tif")
            c, k = write(q, a, 8, 2, {"tile": (256, 256)}, extra_tags=tags)
            comp, nblk = comp + c, nblk + k
            packed.append(q)
    times = {"plain": [], "deflate": []}
    for _ in range(3):
        for key, files in (("deflate", packed), ("plain", plain)):
            torch.cuda.synchronize()
            t = time.perf_counter()
            r = hw.warp_to_device(files, grid)
            torch.cuda.synchronize()
            times[key].append(time.perf_counter() - t)
            times[key + "_out"] = r
    assert torch.equal(times["plain_out"].tensor(), times["deflate_out"].tensor())
    print(json.dumps({"case": "warp_to_device 4096^2 from 1\" tiles, deflate+pred2 256x256 tiles vs uncompressed",
                      "card": gpu, "tiles": len(plain), "compressed_bytes": comp, "decoded_bytes": len(plain) * 3601 ** 2 * 2,
                      "blocks": nblk, "warp_to_device_compressed_s": round(min(times["deflate"]), 4),
                      "warp_to_device_uncompressed_s": round(min(times["plain"]), 4), "page_cache": True}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=18000)
    ap.add_argument("--only", choices=["rasters", "mosaic"], help="run one half of the cases")
    args = ap.parse_args()
    gpu = card()
    n = args.size
    with tempfile.TemporaryDirectory() as tmp:
        if args.only == "mosaic":
            return mosaic_case(tmp, gpu)
        z = dem(n, n, 1)
        a = z.astype(np.int16)
        for comp, cname in ((8, "deflate"), (5, "lzw")):
            for layout, lname in (({"rows": 1}, "1-row strips"), ({"tile": (256, 256)}, "256x256 tiles")):
                p = os.path.join(tmp, f"{cname}_{lname[:3]}.tif")
                c, k = write(p, a, comp, 2, layout)
                record(f"int16 {cname}+pred2 {lname}", p, a, c, k, gpu)
                os.unlink(p)
        f = (z + np.float32(0.25)).astype(np.float32)
        del z, a
        p = os.path.join(tmp, "f32.tif")
        c, k = write(p, f, 8, 3, {"rows": 1})
        record("float32 deflate+pred3 1-row strips", p, f, c, k, gpu)
        os.unlink(p)
        del f
        if args.only != "rasters":
            mosaic_case(tmp, gpu)


if __name__ == "__main__":
    main()

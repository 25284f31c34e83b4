"""Reprojection of a tiled mosaic onto the EPSG:22184 grid (hd_warp_mosaic) on the GPU:  python tools/warp_mosaic_time.py
[--large]

Workload: the 4096 x 4096, 90 m destination of tools/warp_time.py (a 369 km square on the central meridian of zone 4,
centred about 35 S) from seeded int16 1 arc-second tiles laid out like SRTM: 1 x 1 degree, 3601 x 3601 cells, the edge
row and column shared with the neighbours, corners half a pixel off the degree lines; every tile the grid's footprint
meets, about 20 (540 MB, larger than the L2 cache).  The tiles are cut from one seeded raster, so shared edges agree and
the mosaic materialised on the host is that raster.  Prints, as one JSON line, for nearest and bilinear sampling: the
best kernel time of several runs (CUDA events around 10 launches, after warm-up) of hd_warp_mosaic over the tiles and of
hd_warp over the materialised mosaic, their ratio (the cost of the index lookup), with the two outputs asserted equal
bit for bit; then the end-to-end ``resample_and_cut`` time over the tile files, file to file (tiles and output in a
temporary directory, i.e. in the page cache); and the card's name and power limit read in the same run.  ``--large``
adds a 36000 x 36000 grid centred at 63 W 37 S over about 1000 tiles filled on the device with seeded random values,
timing the kernel only and reporting the peak device memory of the case.  Without a GPU it fails."""
import itertools
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hydrodem_b200 import _lib, device as dev, geotiff                                   # noqa: E402
from hydrodem_b200 import warp as hw                                                     # noqa: E402

D = 1.0 / 3600.0
T = 3601
KEYS = np.array([1, 1, 0, 3, 1024, 0, 1, 2, 1025, 0, 1, 1, 2048, 0, 1, 4326], "<u2")
dev.require_cuda()
lib = _lib.load()


def tags(x0, y0):
    return {33550: (12, 3, np.array([D, D, 0.0], "<f8").tobytes()),
            33922: (12, 6, np.array([0, 0, 0, x0, y0, 0], "<f8").tobytes()), 34735: (3, KEYS.size, KEYS.tobytes())}


def info_of(shape, x0, y0, nodata=-32768.0):
    info = geotiff.GeoTiffInfo()
    info.height, info.width = shape
    info.dtype, info.tags, info.nodata = np.dtype(np.int16), tags(x0, y0), nodata
    return info


def tile_range(grid):
    """Integer-degree tiles (lon, lat of the north-west corner) that cover the grid's footprint."""
    lon0, lon1, lat0, lat1 = hw.footprint(grid, hw.EPSG22184)
    return (range(math.floor(lon0), math.ceil(lon1)), range(math.ceil(lat1), math.floor(lat0), -1))


def best_ms(fn, reps=5, inner=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(inner):
            fn()
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b) / inner)
    return best


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
out = {"device": torch.cuda.get_device_name(), "nvidia_smi_name_power_limit_max_sm_clock": gpu[0] if gpu else None}

# ---- 4096^2 over ~20 tiles ------------------------------------------------------------------------------------------
n = 4096
centre_x, centre_y = 4500000.0, 10001965.729312724 - 35.0 * 111000.0
grid = hw.Grid(centre_x - n * 45.0, centre_y + n * 45.0, 90.0, n, n)
lons, lats = tile_range(grid)
rows, cols = len(lats), len(lons)
rng = np.random.default_rng(2024)
whole = rng.integers(-100, 4000, (3600 * rows + 1, 3600 * cols + 1), dtype=np.int16)
tiles = []                                                    # (array, x0, y0), north-west first, row-major
for r, c in itertools.product(range(rows), range(cols)):
    tiles.append((whole[3600 * r:3600 * r + T, 3600 * c:3600 * c + T], lons[c] - 0.5 * D, lats[r] + 0.5 * D))
x00, y00 = tiles[0][1], tiles[0][2]
pairs = [(dev.upload(np.ascontiguousarray(a)), info_of(a.shape, x0, y0)) for a, x0, y0 in tiles]
materialised = dev.upload(whole)
m = hw.Mosaic(pairs, grid)
out.update({"dst": [n, n], "dst_res_m": 90.0, "tiles": [rows, cols], "tile": [T, T], "tiles_selected": m.n,
            "tiles_MB": round(sum(a.nbytes for a, _, _ in tiles) / 1e6, 1), "bins": m.nbins, "bin_px": m.bins[2],
            "index_entries": int(m.index.numel() - 6 * m.n - m.nbins - 1)})
dst_m = dev.empty(n, n, _lib.F32, np.float32)
dst_w = dev.empty(n, n, _lib.F32, np.float32)
stream = dev.stream_ptr()


def warp_materialised(code):
    _lib.check(lib.hd_warp(materialised.ptr, materialised.dtype, materialised.pitch, materialised.ny, materialised.nx,
                           hw._D4(x00, D, y00, D), 1, -32768.0, dst_w.ptr, dst_w.pitch, n, n,
                           hw._D4(grid.x0, grid.res, grid.y0, grid.res), 0, hw._D7(*hw.EPSG22184), code, stream))


for name, code in (("nearest", _lib.WARP_NEAREST), ("bilinear", _lib.WARP_BILINEAR)):
    t_mosaic = best_ms(lambda: m.launch(dst_m, grid, name, stream))
    t_single = best_ms(lambda: warp_materialised(code))
    torch.cuda.synchronize()
    assert torch.equal(dst_m.tensor().view(torch.int32), dst_w.tensor().view(torch.int32)), name
    out[name] = {"mosaic_kernel_ms": round(t_mosaic, 3), "materialised_hd_warp_ms": round(t_single, 3),
                 "mosaic_over_materialised": round(t_mosaic / t_single, 3),
                 "mosaic_dst_Mcells_per_s": round(n * n / t_mosaic / 1e3, 1)}
del m, pairs, materialised

with tempfile.TemporaryDirectory() as tmp:
    paths = []
    for k, (a, x0, y0) in enumerate(tiles):
        paths.append(os.path.join(tmp, f"t{k}.tif"))
        geotiff.write_geotiff(paths[-1], np.ascontiguousarray(a), geo_tags=tags(x0, y0), nodata=-32768)
    dst_tif = os.path.join(tmp, "dst.tif")
    hw.resample_and_cut(paths, dst_tif, grid)                                              # warm-up
    ts = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hw.resample_and_cut(paths, dst_tif, grid)
        ts.append(time.perf_counter() - t0)
    out["resample_and_cut_tiles_file_to_file_s"] = round(min(ts), 3)
    got = geotiff.read_array(dst_tif)
    single = os.path.join(tmp, "whole.tif")
    geotiff.write_geotiff(single, whole, geo_tags=tags(x00, y00), nodata=-32768)
    assert np.array_equal(got, dev.download(hw.warp_to_device(single, grid)))
del tiles, whole

# ---- 36000^2 over ~1000 tiles generated on the device ---------------------------------------------------------------
if "--large" in sys.argv:
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    n = 36000
    cx, cy = 4500000.0, 10001965.729312724 - 37.0 * 111000.0
    big = hw.Grid(cx - n * 45.0, cy + n * 45.0, 90.0, n, n)
    lons, lats = tile_range(big)
    gen = torch.Generator(device=dev.device())
    gen.manual_seed(7)
    pairs = []
    for lat, lon in itertools.product(lats, lons):
        r = dev.empty(T, T, _lib.I16)
        r.buf.random_(-100, 4000, generator=gen)
        pairs.append((r, info_of((T, T), lon - 0.5 * D, lat + 0.5 * D)))
    t0 = time.perf_counter()
    m = hw.Mosaic(pairs, big)
    t_index = time.perf_counter() - t0
    dst = dev.empty(n, n, _lib.F32, np.float32)
    res = {"dst": [n, n], "tiles": len(pairs), "tiles_selected": m.n, "bins": m.nbins, "bin_px": m.bins[2],
           "select_and_index_s": round(t_index, 3)}
    for name in ("nearest", "bilinear"):
        res[name] = {"mosaic_kernel_ms": round(best_ms(lambda: m.launch(dst, big, name, stream), reps=3, inner=3), 2)}
    torch.cuda.synchronize()
    res["peak_device_GB"] = round(torch.cuda.max_memory_allocated() / 1e9, 2)
    out["large"] = res
print(json.dumps(out))

"""Reprojection onto the EPSG:22184 grid (hd_warp) on the GPU:  python tools/warp_time.py [n]

Workload: an n x n destination at 90 m (n = 4096: a 369 km square on the central meridian of zone 4, centred about 35 S)
from a seeded int16 1 arc-second geographic source that covers it (about 14 400 x 12 000 cells, 350 MB: larger than the
L2 cache).  Prints, as one JSON line, for nearest and bilinear sampling: the best kernel time of several runs (CUDA
events around 10 launches, after warm-up), destination Mcells/s, and the bytes the algorithm needs per second computed
from shapes (4 B written per cell plus one (nearest) or four (bilinear) 2-byte source taps); then the end-to-end
``resample_and_cut`` time, file to file (source and output in a temporary directory, i.e. in the page cache), and the
card's name and power limit read in the same run.  Without a GPU it fails."""
import ctypes
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

n = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
dev.require_cuda()
lib = _lib.load()
D = 1.0 / 3600.0

# the destination: an n x n, 90 m grid on the central meridian, centred about 35 S (northing from lat -90)
centre_x, centre_y = 4500000.0, 10001965.729312724 - 35.0 * 111000.0
grid = hw.Grid(centre_x - n * 45.0, centre_y + n * 45.0, 90.0, n, n)
# its outline in lon / lat (the library's host inverse projection), padded by 20 arc-seconds
t = np.linspace(0.0, 1.0, 257)
x1, y1 = grid.x0 + n * 90.0, grid.y0 - n * 90.0
xs = np.concatenate([grid.x0 + t * (x1 - grid.x0)] * 2 + [np.full(t.size, grid.x0), np.full(t.size, x1)])
ys = np.concatenate([np.full(t.size, grid.y0), np.full(t.size, y1), y1 + t * (grid.y0 - y1), y1 + t * (grid.y0 - y1)])
lon, lat = np.empty_like(xs), np.empty_like(ys)
p = lambda a: ctypes.c_void_p(a.ctypes.data)                                             # noqa: E731
_lib.check(lib.hd_host_tm_inverse(hw._D7(*hw.EPSG22184), p(xs), p(ys), xs.size, p(lon), p(lat)))
slon0 = math.floor((lon.min() - 20 * D) / D) * D
slat0 = math.ceil((lat.max() + 20 * D) / D) * D
snx = int(math.ceil((lon.max() + 20 * D - slon0) / D))
sny = int(math.ceil((slat0 - (lat.min() - 20 * D)) / D))
rng = np.random.default_rng(2024)
src = rng.integers(-100, 4000, (sny, snx), dtype=np.int16)
src_geo = (slon0, D, slat0, D)
keys = np.array([1, 1, 0, 3, 1024, 0, 1, 2, 1025, 0, 1, 1, 2048, 0, 1, 4326], "<u2")
tags = {33550: (12, 3, np.array([D, D, 0.0], "<f8").tobytes()),
        33922: (12, 6, np.array([0, 0, 0, slon0, slat0, 0], "<f8").tobytes()), 34735: (3, keys.size, keys.tobytes())}

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
out = {"device": torch.cuda.get_device_name(), "nvidia_smi_name_power_limit_max_sm_clock": gpu[0] if gpu else None,
       "dst": [n, n], "dst_res_m": 90.0, "src": [sny, snx], "src_dtype": "int16", "src_MB": round(src.nbytes / 1e6, 1)}

raster = dev.upload(src)
dst = dev.empty(n, n, _lib.F32, np.float32)
stream = dev.stream_ptr()


def launch(code):
    _lib.check(lib.hd_warp(raster.ptr, raster.dtype, raster.pitch, sny, snx, hw._D4(*src_geo), 1, -32768.0, dst.ptr,
                           dst.pitch, n, n, hw._D4(grid.x0, grid.res, grid.y0, grid.res), 0, hw._D7(*hw.EPSG22184), code,
                           stream))


for name, code, taps in (("nearest", _lib.WARP_NEAREST, 1), ("bilinear", _lib.WARP_BILINEAR, 4)):
    for _ in range(3):
        launch(code)
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(10):
            launch(code)
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b) / 10)
    cells = n * n
    out[name] = {"kernel_ms": round(best, 3), "dst_Mcells_per_s": round(cells / best / 1e3, 1),
                 "needed_GB_per_s": round(cells * (4 + 2 * taps) / best / 1e6, 1)}

with tempfile.TemporaryDirectory() as tmp:
    src_tif, dst_tif = os.path.join(tmp, "src.tif"), os.path.join(tmp, "dst.tif")
    geotiff.write_geotiff(src_tif, src, geo_tags=tags, nodata=-32768)
    hw.resample_and_cut(src_tif, dst_tif, grid)                                          # warm-up
    ts = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        hw.resample_and_cut(src_tif, dst_tif, grid)
        ts.append(time.perf_counter() - t0)
    out["resample_and_cut_file_to_file_s"] = round(min(ts), 3)
    want = dev.download(hw.warp_to_device(src_tif, grid))
    assert np.array_equal(geotiff.read_array(dst_tif), want)
print(json.dumps(out))

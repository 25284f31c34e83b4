"""River-line rasterization onto the EPSG:22184 grid (hd_rasterize_lines) on the GPU:  python tools/rasterize_time.py [n]

Workload: a seeded synthetic river network written as a geographic (WGS84) PolyLine shapefile -- 100 000 random-walk
polylines of 100 vertices (10^7 vertices) with 15 arc-second steps and random UP_CELLS, started uniformly over lon -75 ... -51,
lat -52 ... -22 -- burned onto an n x n, 90 m grid (n = 36000: a 3240 km square on the central meridian of zone 4 centred
at 37 S, which most of the network falls inside).  A second case adds 8 very long segments that cross the whole area.
Prints, as one JSON line per case: the time of ``read_lines`` (files in the page cache), of the upload, of the kernels
(CUDA events around 5 launches, best of 5, after warm-up), and of ``rasterize_rivers`` file to file (one call: read, upload,
burn, download and a 4n^2-byte GeoTIFF written to a temporary directory), with the card's name and power limit read in the
same run.  Without a GPU it fails."""
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hydrodem_b200 import _lib, device as dev                                            # noqa: E402
from hydrodem_b200 import rasterize as hr                                                # noqa: E402
from hydrodem_b200 import warp as hw                                                     # noqa: E402
from oracle import warp as ow                                                            # noqa: E402

GEOG_PRJ = ('GEOGCS["GCS_WGS_1984",DATUM["D_WGS_1984",SPHEROID["WGS_1984",6378137.0,298.257223563]],'
            'PRIMEM["Greenwich",0.0],UNIT["Degree",0.0174532925199433]]')


def network(features=100_000, nv=100, long_segments=0, seed=2024):
    """(lon, lat, vertices per feature, UP_CELLS): one part per feature."""
    rng = np.random.default_rng(seed)
    step = 15.0 / 3600.0
    ang = rng.uniform(0, 2 * np.pi, (features, 1)) + rng.normal(0, 0.3, (features, nv)).cumsum(axis=1)
    d = np.where(np.arange(nv) == 0, 0.0, step)
    lon = rng.uniform(-75, -51, (features, 1)) + (d * np.cos(ang)).cumsum(axis=1)
    lat = rng.uniform(-52, -22, (features, 1)) + (d * np.sin(ang)).cumsum(axis=1)
    counts = np.full(features, nv)
    lon, lat = lon.ravel(), lat.ravel()
    if long_segments:
        t = np.linspace(0, 1, long_segments)
        lon = np.concatenate([lon, np.stack([np.full_like(t, -76.0), np.full_like(t, -50.0)], 1).ravel()])
        lat = np.concatenate([lat, np.stack([-53 + 30 * t, -22 - 30 * t], 1).ravel()])
        counts = np.concatenate([counts, np.full(long_segments, 2)])
    return lon, lat, counts, rng.integers(1, 10_000_000, counts.size)


def write_network(base, lon, lat, counts, values):
    """.shp / .shx / .dbf / .prj of one-part PolyLine records, built with array operations."""
    n = counts.size
    clen = 44 + 4 + 16 * counts                                   # content bytes of each record
    off = 100 + np.concatenate([[0], np.cumsum(8 + clen)[:-1]])
    size = int(off[-1] + 8 + clen[-1])
    buf = np.zeros(size, np.uint8)
    head = np.zeros(100, np.uint8)
    head[:4] = np.frombuffer(np.int32(9994).byteswap().tobytes(), np.uint8)
    head[28:36] = np.frombuffer(np.array([1000, 3], "<i4").tobytes(), np.uint8)
    head[36:68] = np.frombuffer(np.array([lon.min(), lat.min(), lon.max(), lat.max()], "<f8").tobytes(), np.uint8)
    buf[:100] = head
    buf[24:28] = np.frombuffer(np.int32(size // 2).byteswap().tobytes(), np.uint8)
    be, le = buf.view(">i4"), buf.view("<i4")                     # every record starts 4 mod 8: int32 fields are aligned
    be[off // 4] = np.arange(1, n + 1)
    be[off // 4 + 1] = clen // 2
    le[off // 4 + 2] = 3
    le[off // 4 + 11] = 1
    le[off // 4 + 12] = counts
    le[off // 4 + 13] = 0
    first = np.concatenate([[0], np.cumsum(counts)[:-1]])
    rec = np.repeat(np.arange(n), counts)
    pos = off[rec] + 56 + 16 * (np.arange(lon.size) - first[rec])  # 4 mod 8: doubles of buf[4:] are aligned
    f8 = buf[4:4 + (size - 4) // 8 * 8].view("<f8")
    f8[(pos - 4) // 8], f8[(pos - 4) // 8 + 1] = lon, lat
    box = buf[:size // 8 * 8].view("<f8")                         # the bounding boxes start 0 mod 8
    for k, a in enumerate((np.minimum.reduceat(lon, first), np.minimum.reduceat(lat, first),
                           np.maximum.reduceat(lon, first), np.maximum.reduceat(lat, first))):
        box[(off + 12) // 8 + k] = a
    buf.tofile(base + ".shp")
    shx = np.zeros(100 + 8 * n, np.uint8)
    shx[:100] = head
    shx[24:28] = np.frombuffer(np.int32(shx.size // 2).byteswap().tobytes(), np.uint8)
    shx[100:].view(">i4").reshape(n, 2)[:] = np.stack([off // 2, clen // 2], 1)
    shx.tofile(base + ".shx")
    w = 12
    hdr = np.zeros(65, np.uint8)
    hdr[0] = 3
    hdr[4:12] = np.frombuffer(np.array([n], "<u4").tobytes() + np.array([65, 1 + w], "<u2").tobytes(), np.uint8)
    hdr[32:40] = np.frombuffer(b"UP_CELLS", np.uint8)
    hdr[43], hdr[48], hdr[64] = ord("N"), w, 0x0D
    recs = np.char.rjust(values.astype(str).astype("S"), w)
    body = np.full((n, 1 + w), ord(" "), np.uint8)
    body[:, 1:] = np.frombuffer(recs.tobytes(), np.uint8).reshape(n, w)
    with open(base + ".dbf", "wb") as f:
        f.write(hdr.tobytes() + body.tobytes() + b"\x1a")
    with open(base + ".prj", "w") as f:
        f.write(GEOG_PRJ)


def events(fn, reps=5, inner=5):
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


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 36000
    dev.require_cuda()
    lib = _lib.load()
    cx, cy = ow.tm_forward(-63.0, -37.0)
    grid = hw.Grid(float(cx) - n * 45.0, float(cy) + n * 45.0, 90.0, n, n)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    out_dst = dev.empty(n, n, _lib.F32, np.float32)
    for case, long_segments in (("network", 0), ("network_plus_8_long_segments", 8)):
        lon, lat, counts, values = network(long_segments=long_segments)
        res = {"case": case, "device": torch.cuda.get_device_name(),
               "nvidia_smi_name_power_limit_max_sm_clock": gpu[0] if gpu else None, "grid": [n, n], "res_m": 90.0,
               "features": int(counts.size), "vertices": int(lon.size), "segments": int(lon.size - counts.size)}
        with tempfile.TemporaryDirectory() as tmp:
            base = os.path.join(tmp, "rivers")
            write_network(base, lon, lat, counts, values)
            res["shp_MB"] = round(os.path.getsize(base + ".shp") / 1e6, 1)
            hr.read_lines(base + ".shp")                                             # warm the page cache
            t0 = time.perf_counter()
            lines = hr.read_lines(base + ".shp")
            res["read_lines_s"] = round(time.perf_counter() - t0, 3)
            assert lines.n_vertices == lon.size and lines.n_parts == counts.size
            hr.DeviceLines(lines)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dl = hr.DeviceLines(lines)
            torch.cuda.synchronize()
            res["upload_s"] = round(time.perf_counter() - t0, 3)
            ws = dev.scratch(lib.hd_rasterize_workspace_bytes(dl.n_vertices))
            p = lambda t: ctypes.c_void_p(t.data_ptr())                                  # noqa: E731

            def launch():
                _lib.check(lib.hd_rasterize_lines(p(dl.x), p(dl.y), dl.n_vertices, p(dl.part_start), p(dl.part_feature),
                                                  dl.n_parts, p(dl.values), dl.n_features, out_dst.ptr, out_dst.pitch, n, n,
                                                  hw._D4(grid.x0, grid.res, grid.y0, grid.res), 0, hw._D7(*lines.tm),
                                                  p(ws), ws.numel(), dev.stream_ptr()))

            res["kernels_ms"] = round(events(launch), 3)
            got = dev.download(out_dst)
            res["burned_cells"] = int((got > 0).sum())
            del got
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            hr.rasterize_rivers(base + ".shp", os.path.join(tmp, "rivers.tif"), grid)
            res["rasterize_rivers_file_to_file_s"] = round(time.perf_counter() - t0, 3)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()

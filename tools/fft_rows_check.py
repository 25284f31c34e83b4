"""Digests and per-launch times of the Fourier stage's row passes (fft_rows_kernel).

    python tools/fft_rows_check.py [--digests 36000 18000 10801] [--times 36000] [--reps 3]

--digests N...  SHA-256 of fshift, |F| and the float32 DetectApplyFourier output for a seeded N x N raster (the seed
                and the input are those of tests/test_gpu_fft_layout.py::digests).  The row passes promise the same
                bits from one version of the library to the next, so two builds are compared by these lines.
--times N       CUDA-side duration of each fft_rows_kernel launch of DetectApplyFourier on an N x N raster, from
                torch.profiler, in launch order, as the median over --reps runs.
One JSON line per result.
"""
import argparse
import hashlib
import json
import os
import statistics
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hydrodem_b200 import _lib, device as dev  # noqa: E402
from hydrodem_b200.filters import custom_filters as cf  # noqa: E402

CHUNK_ROWS = 1024


def raster_input(ny, nx):
    rng = np.random.default_rng(ny * 100003 + nx)
    src = dev.empty(ny, nx, _lib.F32)
    t = src.tensor()
    for r0 in range(0, ny, CHUNK_ROWS):          # row blocks: the same stream of normals as one (ny, nx) draw
        r1 = min(ny, r0 + CHUNK_ROWS)
        t[r0:r1] = torch.from_numpy((100 + 10 * rng.standard_normal((r1 - r0, nx))).astype(np.float32)).cuda()
    return src


def sha(raster):
    """SHA-256 of the raster's rows in row-major order (the bytes of np.ascontiguousarray of the whole raster)."""
    torch.cuda.synchronize()
    t = raster.tensor()
    h = hashlib.sha256()
    for r0 in range(0, t.shape[0], CHUNK_ROWS):
        h.update(np.ascontiguousarray(t[r0:r0 + CHUNK_ROWS].cpu().numpy()).tobytes())
    return h.hexdigest()


def digests(n):
    src = raster_input(n, n)
    daf = cf.DetectApplyFourier()
    out32 = daf.run_device(src)
    return {"size": n, "fshift": sha(daf.initial._fshift_dev), "fabs": sha(daf._fabs_dev),
            "detect_apply_f32": sha(out32)}


def row_pass_times(n, reps):
    src = raster_input(n, n)
    daf = cf.DetectApplyFourier()
    out = daf.run_device(src)                    # warm-up: plans, module load
    del out
    torch.cuda.synchronize()
    runs = []
    for _ in range(reps):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            out = daf.run_device(src)
            torch.cuda.synchronize()
        del out
        ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "fft_rows_kernel" in e.name]
        ev.sort(key=lambda e: e.time_range.start)
        runs.append([(e.name, e.time_range.elapsed_us() / 1000.0) for e in ev])
    names = [nm for nm, _ in runs[0]]
    ms = [statistics.median(r[i][1] for r in runs) for i in range(len(names))]
    return {"size": n, "reps": reps, "row_pass_ms": [round(v, 3) for v in ms], "total_ms": round(sum(ms), 3),
            "kernels": names}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--digests", type=int, nargs="*", default=[])
    ap.add_argument("--times", type=int, nargs="*", default=[])
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    for n in args.digests:
        print(json.dumps(digests(n)), flush=True)
    for n in args.times:
        print(json.dumps(row_pass_times(n, args.reps)), flush=True)


if __name__ == "__main__":
    main()

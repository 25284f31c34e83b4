"""CUDA-event times of the general scipy.ndimage paths (hd_correlate, hd_binary_morph_struct, hd_max_filter_rect) next to
the specialised kernels they generalise, on one N x N float32 raster (default 18000^2, 1.3 GB: far larger than L2).

    python tools/ndimage_args_time.py [--n 18000] [--reps 5] [--out results.json]

Each case is timed over `reps` calls after one warm-up call; the median is reported with the algorithmic bytes per cell
(each raster read or written once per launch), the share of the card's HBM bandwidth they imply (7.7 TB/s, the data sheet
figure of a 1000 W B200), and for the convolution the FP64 rate (one multiply and one add per tap and cell).  The card's
name and power limit are read in the same run."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from hydrodem_b200 import _lib, device as dev                                  # noqa: E402
from hydrodem_b200.filters import extension_filters as ef                     # noqa: E402

HBM = 7.7e12


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=18000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    dev.require_cuda()
    lib = _lib.load()
    n = args.n
    cells = n * n
    rng = torch.Generator(device="cuda").manual_seed(1)
    f32 = dev.empty(n, n, _lib.F32)
    f32.buf.uniform_(-100.0, 100.0, generator=rng)
    out32 = dev.empty(n, n, _lib.F32)
    u8 = dev.empty(n, n, _lib.U8)
    u8.tensor().copy_((f32.tensor() > -60.0).to(torch.uint8))
    mid8, out8 = dev.empty(n, n, _lib.U8), dev.empty(n, n, _lib.U8)
    work = dev.scratch(cells * 4)
    s = dev.stream_ptr()
    rows = []

    def add(name, fn, bytes_per_cell, flops_per_cell=None):
        ms = timed(fn, args.reps)
        row = {"case": name, "ms": round(ms, 3), "bytes_per_cell": bytes_per_cell,
               "hbm_share": round(bytes_per_cell * cells / (ms * 1e-3) / HBM, 3)}
        if flops_per_cell is not None:
            row["fp64_tflops"] = round(flops_per_cell * cells / (ms * 1e-3) / 1e12, 2)
        rows.append(row)
        print(json.dumps(row), flush=True)

    # ---- Convolve
    ones3 = (ctypes.c_double * 9)(*([1.0] * 9))
    add("convolve 3x3 hd_convolve3", lambda: _lib.check(lib.hd_convolve3(
        f32.ptr, f32.pitch, out32.ptr, out32.pitch, _lib.F32, n, n, ones3, 9.0, 0, None, 0, s)), 8, 18)
    for k in (3, 5, 15, 31):
        dy, dx, w = ef.convolve_taps(np.ones((k, k)))
        (dy, pdy), (dx, pdx) = ef._int_array(dy), ef._int_array(dx)
        w = np.ascontiguousarray(w)
        pw = w.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
        add(f"convolve {k}x{k} hd_correlate", lambda pdy=pdy, pdx=pdx, pw=pw, nt=len(w), kk=k: _lib.check(lib.hd_correlate(
            f32.ptr, f32.pitch, out32.ptr, out32.pitch, _lib.F32, n, n, nt, pdy, pdx, pw, float(kk * kk), s)), 8, 2 * k * k)

    # ---- BinaryClosing (U8 in, U8 out)
    add("closing cross hd_binary_morph", lambda: _lib.check(lib.hd_binary_morph(
        u8.ptr, _lib.U8, u8.pitch, out8.ptr, out8.pitch, n, n, _lib.MORPH_CLOSE, 0, 1, s)), 2)
    yy, xx = np.mgrid[-3:4, -3:4]
    for name, st in (("cross", None), ("disc 7x7", (yy ** 2 + xx ** 2) <= 9), ("square 31x31", np.ones((31, 31)))):
        dil, ero = ef.closing_taps(st)
        (dyd, pdyd), (dxd, pdxd) = ef._int_array(dil[0]), ef._int_array(dil[1])
        (dye, pdye), (dxe, pdxe) = ef._int_array(ero[0]), ef._int_array(ero[1])

        def run(pdyd=pdyd, pdxd=pdxd, pdye=pdye, pdxe=pdxe, nd=len(dyd), ne=len(dye)):
            _lib.check(lib.hd_binary_morph_struct(u8.ptr, _lib.U8, u8.pitch, mid8.ptr, mid8.pitch, n, n, 1, nd, pdyd, pdxd,
                                                  1, None, s))
            _lib.check(lib.hd_binary_morph_struct(mid8.ptr, _lib.U8, mid8.pitch, out8.ptr, out8.pitch, n, n, 0, ne, pdye,
                                                  pdxe, 1, None, s))
        add(f"closing {name} hd_binary_morph_struct", run, 4)

    # ---- BinaryErosion with the cross (U8 in, U8 out)
    add("erosion x8 hd_binary_morph", lambda: _lib.check(lib.hd_binary_morph(
        u8.ptr, _lib.U8, u8.pitch, out8.ptr, out8.pitch, n, n, _lib.MORPH_ERODE, 0, 8, s)), 2)

    def erode20():
        src = u8
        for i, k in enumerate((8, 8, 4)):
            dst = (mid8, out8, mid8)[i]
            _lib.check(lib.hd_binary_morph(src.ptr, _lib.U8, src.pitch, dst.ptr, dst.pitch, n, n, _lib.MORPH_ERODE, 0, k, s))
            src = dst
    add("erosion x20 hd_binary_morph x3", erode20, 6)

    # ---- GreyDilation (F32)
    add("grey 7x7 hd_max_filter", lambda: _lib.check(lib.hd_max_filter(
        f32.ptr, f32.pitch, out32.ptr, out32.pitch, _lib.F32, n, n, 7, s)), 8)
    for a, b in ((7, 7), (8, 8), (64, 3), (255, 255)):
        add(f"grey {a}x{b} hd_max_filter_rect", lambda a=a, b=b: _lib.check(lib.hd_max_filter_rect(
            f32.ptr, f32.pitch, out32.ptr, out32.pitch, _lib.F32, n, n, a, b, ctypes.c_void_p(work.data_ptr()), cells * 4,
            s)), 16)

    res = {"card": card(), "n": n, "reps": args.reps, "cases": rows}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print("card:", res["card"])


if __name__ == "__main__":
    main()

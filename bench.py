#!/usr/bin/env python
"""bench.py -- Mcells/s of the full HydroDEM conditioning chain on B200.

    python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR

--dump-outputs DIR writes what the last timed step computed -- final, filled and d8, in the dtypes a caller of
ConditioningChain receives them (float64 final, float32 filled, d8 widened to float32) -- as DIR/<name>.npy: the whole
rasters when they have at most DUMP_CELLS cells, else the cells at a fixed, seeded sample of positions (ascending
row-major order, the same at every N).  The inputs are a pure function of the seed, so two builds run with the same
arguments can be compared output for output.

Workload (BASELINE.json configs[4], the one both north-star targets are quoted on): the full conditioning chain --
Fourier stripe removal, groves correction x3, lagoon detection, recombination, 3x3 mean + round, sink-fill + D8 --
on ONE synthetic 36000 x 36000 mosaic (seed 1005, generated on the device, every cell a pure function of its
coordinates).  A "step" is one pass of the chain over the mosaic.  N = 1: `ConditioningChain` on one B200 (the mosaic
fits: ~100 GB).  N > 1: the SAME mosaic cut into N row bands, `sharding.Band.conditioning_chain` -- halo exchange and
the all-to-alls of the sharded Fourier stage over NCCL -- so scaling is STRONG, and the outputs are bit-identical to
the N = 1 run (the JSON line carries order-independent integer checksums of final DEM / filled DEM / D8).

Numbers on the JSON line
  value     whole-job Mcells/s with the inputs resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e       the same through the public API with HOST buffers: inputs uploaded from pinned host memory and the three
            results read back into host arrays inside the timed region
  roofline  dominant kernel of the step: algorithmic bytes per launch / average launch time, measured live with a
            CUDA event pair around every launch (hd_profile_*), against MEASURED_PEAKS.json hbm_gbs; `traffic` is the
            dram read + write per launch from the committed ncu capture (profiles/r2_ncu_traffic.json)
  cpu_baseline  the CPU oracle port (oracle/chain.py) timed on rank 0, one core, on a bounded sample tile; next to it
            the reference's OWN classes as timed in the build container (profiles/r2_reference_classes_cpu.json: the
            reference is pure Python and imports there, but /root/reference does not exist on the GPU box)
  secondary the 3601 x 3601 tile (configs[1], round 1's headline) and sink-fill + D8 on an 18000 x 18000 mosaic
            (configs[3]) at the same N
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

MOSAIC = 36000
SEED = 1005
METRIC = "Mcells/s, full conditioning chain"
UNIT = "Mcells/s"
DUMP_CELLS = 1 << 21            # cells per dumped output: 8 + 4 + 4 bytes each, 32 MB for the three outputs


def algo_bytes_per_cell(odd):
    """Algorithmic HBM bytes per cell and per launch of each kernel in this workload (DESIGN.md section 5).
    fft_rows: the four row passes of one forward + one masked inverse 2-D transform are real->c64 (4+8), c64->c64 on the
    Hermitian half (8+8)/2, masked c64->c64 (8+1+8; half the rows when odd x odd), c64 (pairs) ->|.| (8+4)."""
    return {
        "fft_rows_kernel": ((12 + 8 + 17 / 2 + 12) if odd else (12 + 8 + 17 + 12)) / 4.0,
        "transpose_kernel": 16.0, "transpose_real_kernel": 8.0, "quadratic_kernel": 9.0, "majority_kernel": 8.0,
        "fill_async_kernel": 12.0, "hollow_kernel": 9.0 * 0.25, "expand_kernel": 2.0, "morph_kernel": 2.0,
        "maxfilter_kernel": 8.0, "fix3_kernel": 8.0, "conv3_kernel": 20.0, "final_terms_kernel": 20.0,
        "elementwise_kernel": 9.0, "fill_finish_d8_kernel": 5.0, "tidy_lagoons_kernel": 8.0, "final_mean3_kernel": 16.0,
        "fill_init_kernel": 8.0,
    }


def env_int(name, default):
    return int(os.environ.get(name, default))


def workload_config(size, n_gpus):
    """The SAME dict for both arms (the driver compares them)."""
    return {"workload": f"full conditioning chain on ONE synthetic {size}x{size} mosaic (BASELINE.json configs[4]), "
                        f"{'one GPU' if n_gpus == 1 else f'row-band sharded over {n_gpus} GPUs, NCCL halo exchange + all-to-all'}",
            "stages": "fft2+peak mask+ifft2, groves x3 (quadratic 15), nanfix, majority 11, erode2, expand 7, max 7x7, combine, "
                      "mean3+round, sink-fill + D8 (fused last pass)",
            "mosaic": [size, size], "seed": SEED, "parallelism": "single GPU" if n_gpus == 1 else f"row bands x{n_gpus}",
            "l2": "inputs (11.7 GB) and every intermediate are far larger than the 126 MB L2: no flush needed"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines, self.first = index, None, [], 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        self.first = len(self.lines)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        last = len(self.lines)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in self.lines[self.first:last]:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons), "sampled": "during the timed steps"}


def measured_peak():
    try:
        with open(os.path.join(REPO, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback"          # /opt/skills/guides/B200_PROFILING.md


def load_json(rel):
    try:
        with open(os.path.join(REPO, rel)) as f:
            return json.load(f)
    except (OSError, ValueError):
        return None


# ---------------------------------------------------------------------------------------------------------
def cpu_chain_sample(size, seed):
    """One pass of the CPU oracle chain over a size x size sample tile -> seconds."""
    from hydrodem_b200.synth import SynthScene
    from oracle import chain
    sc = SynthScene(size, size, seed)
    a, g, h = sc.srtm(), sc.groves(), sc.hsheds()
    t0 = time.perf_counter()
    with np.errstate(all="ignore"):
        chain.conditioning_chain(a, g, h)
    return time.perf_counter() - t0


def _cpu_worker(args):
    return cpu_chain_sample(*args)


def reference_classes_record():
    rec = load_json("profiles/r2_reference_classes_cpu.json")
    if not rec:
        return None
    return {"value": rec.get("mcells_s"), "unit": UNIT, "cores": 1, "kind": "reference (recorded)",
            "sample": rec.get("sample"), "where": rec.get("where")}


def run_reference(args):
    """The reference arm: the CPU implementation of the path on all host cores.  The reference itself is pure Python
    (its filter layer imports wherever numpy / scipy exist), but /root/reference is not shipped to the GPU box, so what
    runs here is the oracle port -- a vectorised NumPy / SciPy restatement of the reference's filters, about 50x FASTER
    than the reference's own per-cell Python loops (their timing, taken in the build container, is reported beside it)."""
    if env_int("RANK", 0) != 0:
        return
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0)) or 1          # the cores this process may actually use
    size = args.cpu_sample
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(256, SEED + i) for i in range(cores)])          # warm-up (imports, page faults)
        for _ in range(args.warmup):
            pool.map(_cpu_worker, [(size, SEED + i) for i in range(cores)])
        steps = args.steps
        t0 = time.perf_counter()
        for _ in range(steps):
            pool.map(_cpu_worker, [(size, SEED + i) for i in range(cores)])     # one sample tile per core per step
        dt = time.perf_counter() - t0
    cells = size * size * cores * steps
    value = cells / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args.size, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "steps_run": steps,
                         "sample": f"oracle/chain.py on {cores} processes x {size}x{size} synthetic tiles per step "
                                   "(cost is linear in cells: fixed windows)",
                         "reference_classes": reference_classes_record()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from hydrodem_b200 import _lib, device as dev, sharding
    from hydrodem_b200.filters import new_filters as nf
    from hydrodem_b200.pipeline import ConditioningChain
    from hydrodem_b200.synth import DeviceMosaic, SynthScene

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the conditioning path has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL writes its banner and any NCCL_DEBUG output to stdout: stdout carries exactly one JSON line, so file
        # descriptor 1 points at stderr while the communicator is created and the first collective runs
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    lib = _lib.load()
    ny = nx = args.size
    cells = ny * nx

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [int(v) for v in t.tolist()]

    def checksums(raster, row0):
        """Order-independent integer checksums of an integer-valued raster: plain sum and a position-weighted sum."""
        t = raster.tensor()
        s0 = s1 = 0
        xs = torch.arange(t.shape[1], device=t.device, dtype=torch.int64)
        for a in range(0, t.shape[0], 2048):
            blk = torch.nan_to_num(t[a:a + 2048].to(torch.float64), nan=-1.0).to(torch.int64)
            ys = torch.arange(row0 + a, row0 + a + blk.shape[0], device=t.device, dtype=torch.int64)
            wgt = (ys[:, None] * 131 + xs[None, :] * 31) % 65521 + 1
            s0 += int(blk.sum().item())
            s1 += int((blk * wgt).sum().item())
        return s0, s1

    def dumped_outputs(res, row0):
        """final / filled / d8 of one step as --dump-outputs writes them (module docstring), gathered from all ranks."""
        whole = cells <= DUMP_CELLS
        idx = np.arange(cells) if whole else np.unique(np.random.default_rng(SEED).integers(0, cells, DUMP_CELLS))
        out = {}
        for name in ("final", "filled", "d8"):
            t = res[name].tensor()
            lo, hi = np.searchsorted(idx, [row0 * nx, (row0 + t.shape[0]) * nx])     # this rank's rows
            mine = torch.from_numpy(idx[lo:hi] - row0 * nx).to(t.device)
            vals = t[mine // nx, mine % nx].cpu().numpy()
            if world > 1:
                vals = np.concatenate(band.comm.gather_objects(vals))                 # bands in rank order
            vals = vals.astype(np.float64 if res[name].ref_dtype == np.float64 else np.float32)
            out[name] = vals.reshape(ny, nx) if whole else vals
        return out

    # ---- the mosaic: generated on the device, straight into the rasters the chain reads ---------------------------
    mosaic = DeviceMosaic(ny, nx, SEED)
    chain = ConditioningChain()
    if world == 1:
        band = None
        d_srtm = dev.DeviceRaster(torch.empty((ny, nx), dtype=torch.float32, device=dev.device()), ny, nx, _lib.F32, np.float32)
        d_gr, d_hs = dev.empty(ny, nx, _lib.U8, np.uint8), dev.empty(ny, nx, _lib.F32, np.float32)
        mosaic.band(0, ny, out={"srtm": d_srtm.tensor(), "groves": d_gr.tensor(), "hsheds": d_hs.tensor()})
        r0 = 0

        def step():
            return chain.run_device(d_srtm, d_gr, d_hs).rasters
    else:
        band = sharding.Band(sharding.DistComm(), ny, nx)
        r0 = band.r0
        d_srtm = dev.DeviceRaster(torch.empty((band.rows, nx), dtype=torch.float32, device=dev.device()), band.rows, nx,
                                  _lib.F32, np.float32)
        g_ext, h_ext = band.alloc_ext(_lib.U8, np.uint8), band.alloc_ext(_lib.F32, np.float32)
        mosaic.band(band.r0, band.r1, out={"srtm": d_srtm.tensor(), "groves": g_ext.owned().tensor(),
                                           "hsheds": h_ext.owned().tensor()})

        def step():
            return band.conditioning_chain(d_srtm, g_ext, h_ext)
    torch.cuda.synchronize()

    # ---- resident-input timing ------------------------------------------------------------------------
    sampler = ClockSampler(torch.cuda.current_device() if "CUDA_VISIBLE_DEVICES" not in os.environ else local)
    if rank == 0:
        sampler.start()                    # nvidia-smi needs ~0.5 s to start streaming: launch it before the warm-up
    res = None
    for _ in range(args.warmup):
        res = None
        res = step()
    barrier()
    if rank == 0:
        sampler.mark()                     # only samples taken from here on (the timed region) are reported
    lib.hd_reset_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for k in range(args.steps):
        res = None                                                         # the previous step's rasters go back to the pool
        ev[k][0].record()
        res = step()
        ev[k][1].record()
    barrier()
    launches = int(lib.hd_launch_count())
    clocks = sampler.stop() if rank == 0 else None
    total_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev))
    ms_per_step = total_ms / args.steps
    value = cells / (ms_per_step * 1e-3) / 1e6
    sums = []
    for name in ("final", "filled", "d8"):
        sums += list(checksums(res[name], r0))
    sums = sum_over_ranks(sums)
    if args.dump_outputs:
        dumped = dumped_outputs(res, r0)
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in dumped.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        del dumped
    fill_rounds = band.fill_rounds if band is not None else None
    fill_status = max_over_ranks(float(band.fill_status())) if band is not None else None

    # ---- per-kernel profile of one more step (event pair around every launch), rank 0's kernels ---------------------
    res = None
    lib.hd_profile_enable(1)
    res = step()
    cbuf = ctypes.create_string_buffer(1 << 16)
    lib.hd_profile_report(cbuf, 1 << 16)
    lib.hd_profile_enable(0)
    res = None
    kernels = {}
    for line in cbuf.value.decode().splitlines():
        name, cnt, ms = line.split()
        kernels[name] = {"launches": int(cnt), "total_ms": float(ms)}
    prof_total = sum(k["total_ms"] for k in kernels.values()) or 1.0
    top = max(kernels, key=lambda n: kernels[n]["total_ms"])
    peak, peak_kind = measured_peak()
    top_avg_ms = kernels[top]["total_ms"] / kernels[top]["launches"]
    local_cells = cells / world
    algo = algo_bytes_per_cell(bool((ny & 1) and (nx & 1)))
    algo_bytes = algo.get(top, 8.0) * local_cells
    achieved = algo_bytes / (top_avg_ms * 1e-3) / 1e9
    ncu = (load_json("profiles/r2_ncu_traffic.json") or {}).get(top)
    roofline = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
                "frac": achieved / peak, "traffic": ncu.get("dram_bytes_per_launch") if ncu else None,
                "traffic_source": ncu.get("source") if ncu else None, "launches_per_step": kernels[top]["launches"],
                "avg_launch_ms": top_avg_ms, "share_of_step": kernels[top]["total_ms"] / prof_total,
                "algorithmic_bytes_per_launch": algo_bytes}
    breakdown = {n: round(k["total_ms"], 3) for n, k in sorted(kernels.items(), key=lambda kv: -kv[1]["total_ms"])}
    stage_roofline = {n: round(algo[n] * local_cells * k["launches"] / (k["total_ms"] * 1e-3) / 1e9 / peak, 3)
                      for n, k in kernels.items() if n in algo and k["total_ms"] > 0}

    # ---- end to end through the public API, host buffers ---------------------------------------------------
    # every step uploads its three input rasters from pinned host memory and reads its three results back into
    # host arrays, all inside the timed region
    host = {}
    src = {"srtm": d_srtm, "groves": d_gr if world == 1 else None, "hsheds": d_hs if world == 1 else None}
    if world > 1:
        src["groves"], src["hsheds"] = g_ext.owned(), h_ext.owned()
    for name, r in src.items():
        pin = dev.pinned_empty(r.shape, dev._HD2NP[r.dtype])
        torch.from_numpy(pin).copy_(r.tensor())
        host[name] = pin
    torch.cuda.synchronize()
    if world == 1:
        del d_srtm, d_gr, d_hs
    else:
        del g_ext, h_ext
    del src
    torch.cuda.empty_cache()
    e2e_steps = max(1, args.e2e_steps)

    def e2e_step():
        if world == 1:
            out = chain.apply_to_host(host["srtm"], host["groves"], host["hsheds"])    # three streams, eager kernels
            got = (out["final"], out["filled"], out["d8"])                 # host arrays, copies complete
            assert got[0].dtype == np.float64 and got[0].shape == (ny, nx)
            return chain.last_transfer_bytes[1]                            # bytes that crossed PCIe (final as int16)
        else:
            out = band.apply_to_host(host["srtm"], host["groves"], host["hsheds"])
            got = (out["final"], out["filled"], out["d8"])
            assert got[0].dtype == np.float64 and got[0].shape == (band.rows, nx)
            return band.last_transfer_bytes[1]

    for _ in range(2):                                                     # warm-up: pinned result buffers get allocated,
        d2h = e2e_step()                                                   # the host side reaches its steady state
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        d2h = e2e_step()
    torch.cuda.synchronize()
    t_e2e = time.perf_counter() - t0
    barrier()
    h2d = sum(a.nbytes for a in host.values())
    e2e_ms = max_over_ranks(t_e2e / e2e_steps * 1e3)
    h2d_total, d2h_total = sum_over_ranks([h2d, d2h])
    host.clear()
    torch.cuda.empty_cache()

    # ---- secondary records ------------------------------------------------------------------------------------------
    secondary = {}
    if not args.no_secondary:
        # sink-fill + D8 on an 18000 x 18000 mosaic (BASELINE.json configs[3]) at this N
        n4 = 18000
        m4 = DeviceMosaic(n4, n4, 1004)
        if world == 1:
            z = dev.empty(n4, n4, _lib.F32, np.float32)
            m4.band(0, n4, out={"hsheds": z.tensor()})
            z.tensor()[z.tensor() < 0] = float("nan")                      # voids are nodata outlets
            f4 = nf.SinkFillD8()
            run4 = lambda: f4.run_device(z)                                # noqa: E731
            row4 = 0
        else:
            b4 = sharding.Band(band.comm, n4, n4)
            zx = b4.alloc_ext(_lib.F32, np.float32)
            m4.band(b4.r0, b4.r1, out={"hsheds": zx.owned().tensor()})
            t = zx.owned().tensor()
            t[t < 0] = float("nan")
            run4 = lambda: b4.sinkfill(zx)                                 # noqa: E731
            row4 = b4.r0
        out4 = run4()
        times4 = []
        for _ in range(3):
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); out4 = run4(); b.record()
            barrier()
            times4.append(max_over_ranks(a.elapsed_time(b)))
        c4 = sum_over_ranks(list(checksums(out4[0], row4)) + list(checksums(out4[1], row4)))
        secondary["c4_fill_d8_18000"] = {"workload": "sink-fill + D8 on a synthetic 18000x18000 mosaic (BASELINE.json configs[3])",
                                         "ms": min(times4), "mcells_s": n4 * n4 / min(times4) / 1e3, "checksums": c4,
                                         "fill_rounds": None if world == 1 else b4.fill_rounds}
        del out4
        torch.cuda.empty_cache()
        if world == 1:
            # the 3601 x 3601 tile (configs[1]): one CUDA graph per pass, L2 flushed between timed passes
            sc = SynthScene(3601, 3601, 1002)
            d_in = chain.upload_inputs(sc.srtm(), sc.groves(), sc.hsheds())
            cap = chain.capture(*d_in)
            flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
            for _ in range(3):
                cap.replay()
            ts = []
            for k in range(20):
                flush.fill_(k & 0xff)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); cap.replay(); b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            secondary["tile_3601"] = {"workload": "full chain, one synthetic 3601x3601 tile (BASELINE.json configs[1]), one "
                                                  f"CUDA graph of {cap.launches} kernels per pass",
                                      "ms_per_step": float(np.mean(ts)), "mcells_s": 3601 * 3601 / float(np.mean(ts)) / 1e3}

    if rank == 0:
        cfg = workload_config(args.size, world)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "e2e": {"value": cells / (e2e_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "h2d_bytes_per_step": int(h2d_total), "d2h_bytes_per_step": int(d2h_total),
                    "api": ("hydrodem_b200.pipeline.ConditioningChain().apply_to_host(srtm, groves, hsheds) -> final / filled / d8 ndarrays"
                            if world == 1 else
                            "hydrodem_b200.sharding.Band(comm, ny, nx).apply_to_host(srtm_rows, groves_rows, hsheds_rows)"),
                    "transport": ("inputs float32 / uint8 / float32 from pinned host arrays; final DEM (integer metres) down as "
                                  "int16 and widened to the reference's float64 by host threads inside the timed region, "
                                  "filled float32, d8 uint8"),
                    "host": {"cpus": len(os.sched_getaffinity(0)), "ranks_on_box": env_int("LOCAL_WORLD_SIZE", 1)}},
            "gpu_launches": launches, "launches_per_step": launches / args.steps,
            "checksums": {"final": sums[0:2], "filled": sums[2:4], "d8": sums[4:6],
                          "note": "integer sums over all ranks (plain, position weighted): equal at every N"},
            "fill": {"rounds": fill_rounds, "status": fill_status},
            "roofline": roofline, "kernel_ms": breakdown, "stage_hbm_frac": stage_roofline, "clocks": clocks,
            "secondary": secondary,
        }
        if world == 1 and not args.no_cpu_baseline:
            dt = cpu_chain_sample(args.cpu_sample, SEED)
            line["cpu_baseline"] = {"value": args.cpu_sample ** 2 / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
                                    "seconds": dt,
                                    "sample": f"oracle/chain.py (NumPy/SciPy restatement of the reference filters) on "
                                              f"one {args.cpu_sample}x{args.cpu_sample} synthetic tile, 1 process",
                                    "reference_classes": reference_classes_record()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=MOSAIC, help="mosaic edge (default 36000 = BASELINE.json configs[4])")
    ap.add_argument("--cpu-sample", type=int, default=1024, help="edge of the CPU baseline sample tile")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write final / filled / d8 of the last timed step to DIR/<name>.npy (GPU path only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm times sample tiles")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()

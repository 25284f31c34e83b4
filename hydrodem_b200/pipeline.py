"""The full conditioning chain, device resident.

Host-side mirror of ``HydroDEMProcess.start`` (hydro_dem_process.py:122-153)
with the GDAL file handling removed: the four rasters that ``image_srtm.py``
and ``image_hsheds.py`` read with ``gdal.Open(...).ReadAsArray()`` come in as
NumPy arrays, everything in between runs as CUDA kernels on device rasters,
and the results come back as NumPy arrays in the reference's dtypes.

    SRTM branch    DetectApplyFourier                       image_srtm.py:125-126
                   BinaryClosing(ones(3,3)) on the groves   image_srtm.py:177-178
                   GrovesCorrectionsIter(iterations=3)      image_srtm.py:199
    HSHEDS branch  LagoonsDetection                         image_hsheds.py:133-136
                   (river routing is out of scope: ``rivers`` is a given 0/1 raster, default none)
    combine        _prepare_final_terms + sum               hydro_dem_process.py:60-91, :148
                   PostProcessingFinal                      hydro_dem_process.py:149
    NEW            SinkFill + D8FlowDirection on the final DEM

Inside the chain rasters are stored as float32 / uint8 (the reference's
float64 intermediates hold float32-representable or tolerance-class values);
conversion to the reference dtype happens once, on download.
"""
import ctypes
import os

import numpy as np

from . import _lib, device as dev
from .exceptions import DeviceError, NumpyArrayExpectedError
from .filters import custom_filters as cf
from .filters import extension_filters as ef
from .filters import new_filters as nf


class ChainResult:
    """Device rasters of one run; ``.host(name)`` / attribute access copies to NumPy lazily."""

    def __init__(self, rasters, info):
        self.rasters = rasters
        self.info = info
        self._host = {}

    def host(self, name):
        if name not in self._host:
            self._host[name] = dev.download(self.rasters[name])
        return self._host[name]

    def __getattr__(self, name):
        rasters = self.__dict__.get("rasters", {})
        if name in rasters:
            return self.host(name)
        raise AttributeError(name)


class CapturedChain:
    """A CUDA graph of one pass of the chain (see ConditioningChain.capture)."""

    def __init__(self, graph, result, launches):
        self.graph, self.result, self.launches = graph, result, launches

    def replay(self):
        self.graph.replay()
        self.result._host.clear()
        return self.result


def copy_streams(owner):
    """The (upload, download) copy streams of ``owner`` (a chain or a band), created on first use and kept on it."""
    streams = owner.__dict__.get("_copy_streams")
    if streams is None:
        import torch
        streams = owner._copy_streams = (torch.cuda.Stream(), torch.cuda.Stream())
    return streams


def host_threads():
    """Host threads that widen int16 results: the cores this process may use, shared by the ranks of the box."""
    local = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    return max(1, min(16, len(os.sched_getaffinity(0)) // max(local, 1)))


def narrow_final_default():
    """Whether the eager host calls send the final DEM (integer metres) down as int16 (HD_NARROW_FINAL=0: float64)."""
    return os.environ.get("HD_NARROW_FINAL", "1") != "0"


def check_fill_status(status):
    """Raise DeviceError unless ``status`` (the sink-fill's sticky status word) says the fixed point was reached."""
    if status != 0:
        raise DeviceError(f"sink-fill did not reach its fixed point (status {status}): filled / d8 are invalid")


class _StreamSlot:
    """One pipeline slot of ConditioningChain.stream: static input rasters, the chain captured as CUDA-graph
    segments (split where an input is first needed / an output is complete) and the events that order the three
    streams (upload, compute, download)."""

    ORDER = ("srtm", "groves", "hsheds", "rivers")

    def __init__(self, chain, arrays, narrow_filled=True):
        import torch
        lib = _lib.load()
        self.chain = chain
        self.cur = torch.cuda.current_stream()
        self.up, self.down = copy_streams(chain)
        self.names = [n for n in self.ORDER if n in arrays]
        self.inputs = {n: dev.empty(*arrays[n].shape, dev.hd_dtype_of(arrays[n].dtype), arrays[n].dtype)
                       for n in self.names}
        if arrays["srtm"].dtype == np.float32:
            # the raw SRTM raster is only read by the row FFT (plain loads, any pitch): it lives densely and is the
            # direct target of its upload -- no staging copy, no re-pitch kernel
            ny, nx = arrays["srtm"].shape
            self.inputs["srtm"] = dev.DeviceRaster(torch.empty((ny, nx), dtype=torch.float32, device=dev.device()), ny, nx,
                                                   _lib.F32, np.float32)
        for r in self.inputs.values():
            r.buf.zero_()
        self.staging = {}
        st = {}
        inp = self.inputs
        stages = [("srtm", lambda: chain._stage_fourier(st, inp["srtm"])),
                  ("groves", lambda: chain._stage_groves(st, inp["groves"])),
                  ("hsheds", lambda: chain._stage_combine(st, inp["hsheds"], inp.get("rivers")))]
        if chain.with_hydrology:
            stages.append((None, lambda: chain._stage_hydrology(st)))
        for _, fn in stages:                                          # warm-up: FFT plans, function attributes
            fn()
        torch.cuda.synchronize()
        st.clear()
        n0 = lib.hd_launch_count()
        self.segments, pool = [], None
        for needs, fn in stages:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool, capture_error_mode="relaxed"):
                fn()
            pool = g.pool()
            self.segments.append((needs, g))
        self.launches = int(lib.hd_launch_count() - n0)
        self.st = st
        # what travels down: (result name, device raster, dtype the caller gets).  The final DEM goes as float32
        # (integer metres, |z| < 2**24: exact) and is widened to the reference's float64 on the host.
        # what travels down: (result name, device raster, dtype the caller gets, int16 transport?).  The final DEM and
        # the filled DEM hold integer metres: they cross PCIe as int16 (checked on the device: a tile with a NaN, a
        # fraction or |z| > 32767 falls back to float32) and are widened to the reference dtypes on the host.
        self.outputs = [("final", "final32", np.float64, True)]
        if chain.with_hydrology:
            self.outputs += [("filled", "filled", np.float32, bool(narrow_filled)), ("d8", "d8", np.uint8, False)]
        # Rasters travel as dense 1-D copies: with both PCIe directions busy, pitched 2-D copies reach 72 GB/s in total,
        # dense ones 95 GB/s (uint8 rows of 3601 bytes: half the rate even alone).  Re-pitching / packing is a small
        # device kernel on the COMPUTE stream, so the copy streams carry nothing but DMA -- a kernel there would have
        # to wait for a gap between the chain's kernels and hold up the copies queued behind it.
        self.dense_in = {n: (r.buf.view(-1) if r.pitch == r.nx else
                             torch.empty(r.ny * r.nx, dtype=r.buf.dtype, device=r.buf.device))
                         for n, r in self.inputs.items()}
        self.dense_out, self.flags = {}, {}
        for _, src, _, narrow in self.outputs:
            r = st[src]
            self.dense_out[src] = torch.empty(r.ny * r.nx, dtype=torch.int16 if narrow else r.buf.dtype, device=r.buf.device)
            if narrow:
                self.flags[src] = torch.zeros(1, dtype=torch.int32, device=r.buf.device)
        size = lambda t: t.numel() * t.element_size()
        self.transfer_bytes = (sum(size(t) for t in self.dense_in.values()), sum(size(t) for t in self.dense_out.values()))
        self.host_threads = host_threads()
        self.ev_compute = self.ev_down = None
        self.keep = None

    def submit(self, arrays):
        """Enqueue one tile; returns a function that waits for it and returns its host arrays."""
        import torch
        lib = _lib.load()
        cur, up, down = self.cur, self.up, self.down
        up.wait_stream(cur) if self.ev_compute is None else up.wait_event(self.ev_compute)
        ready, keep = {}, []
        for name in self.names:
            host = np.ascontiguousarray(arrays[name])
            if host.dtype == np.bool_:
                host = host.view(np.uint8)
            if not dev._is_pinned(host):
                pin = self.staging.get(name)
                if pin is None:
                    pin = self.staging[name] = dev.pinned_empty(host.shape, host.dtype)
                elif self.ev_compute is not None:
                    self.ev_compute.synchronize()                    # the previous upload from this buffer is over
                pin[...] = host
                host = pin
            keep.append(host)
            raster = self.inputs[name]
            es = host.dtype.itemsize
            dense = self.dense_in.get(name)
            if dense is None:                                         # (no staging buffer: pitched DMA into the raster)
                _lib.check(lib.hd_memcpy2d_h2d(raster.ptr, raster.pitch * es, ctypes.c_void_p(host.ctypes.data),
                                               raster.nx * es, raster.nx * es, raster.ny, ctypes.c_void_p(up.cuda_stream)))
            else:                                                     # dense DMA, re-pitched on the compute stream
                nbytes = dense.numel() * dense.element_size()
                _lib.check(lib.hd_memcpy2d_h2d(ctypes.c_void_p(dense.data_ptr()), nbytes, ctypes.c_void_p(host.ctypes.data),
                                               nbytes, nbytes, 1, ctypes.c_void_p(up.cuda_stream)))
            ready[name] = torch.cuda.Event()
            ready[name].record(up)
        if "rivers" in ready:
            ready["hsheds"] = ready["rivers"]                         # uploaded last: covers both
        if self.ev_down is not None:
            cur.wait_event(self.ev_down)                              # static outputs are free again
        pending = {}

        def send(name, src, np_dtype, narrow):
            raster = self.st[src]
            dense = self.dense_out[src]
            flag_host = None
            with torch.cuda.stream(cur):                              # pack on the compute stream, dense DMA
                if narrow:
                    _lib.check(lib.hd_pack_i16(raster.ptr, raster.pitch, ctypes.c_void_p(dense.data_ptr()), raster.ny,
                                               raster.nx, ctypes.c_void_p(self.flags[src].data_ptr()), dev.stream_ptr()))
                else:
                    dense.view(raster.ny, raster.nx).copy_(raster.tensor())
            ev = torch.cuda.Event()
            ev.record(cur)
            down.wait_event(ev)
            # plain pinned arrays + the library's copy: torch's host allocator then has no pending events on them
            # and hands the same blocks out again at once
            host = dev.pinned_empty(raster.shape, np.int16 if narrow else dev._HD2NP[raster.dtype])
            nbytes = dense.numel() * dense.element_size()
            _lib.check(lib.hd_memcpy2d_d2h(ctypes.c_void_p(host.ctypes.data), nbytes, ctypes.c_void_p(dense.data_ptr()),
                                           nbytes, nbytes, 1, ctypes.c_void_p(down.cuda_stream)))
            if narrow:
                flag_host = dev.pinned_empty((1,), np.int32)
                _lib.check(lib.hd_memcpy2d_d2h(ctypes.c_void_p(flag_host.ctypes.data), 4,
                                               ctypes.c_void_p(self.flags[src].data_ptr()), 4, 4, 1,
                                               ctypes.c_void_p(down.cuda_stream)))
            done = torch.cuda.Event()
            done.record(down)
            pending[name] = (host, done, np.dtype(np_dtype), flag_host, raster)

        def arrived(name):
            cur.wait_event(ready[name])
            for n in (("hsheds", "rivers") if name == "hsheds" else (name,)):
                r = self.inputs.get(n)
                if r is not None and n in ready and r.pitch != r.nx:
                    with torch.cuda.stream(cur):
                        r.tensor().copy_(self.dense_in[n].view(r.ny, r.nx))

        trace = getattr(self.chain, "_trace", None)                   # tools/e2e_prof.py: per-tile compute spans
        if trace is not None:
            t_begin = torch.cuda.Event(enable_timing=True)
            cur.wait_event(ready[self.segments[0][0]])
            t_begin.record(cur)
            marks = [t_begin]
        for needs, g in self.segments:
            if needs is not None:
                arrived(needs)
            g.replay()
            if trace is not None:
                marks.append(torch.cuda.Event(enable_timing=True))
                marks[-1].record(cur)
            if needs == "hsheds":
                send(*self.outputs[0])
        for spec in self.outputs[1:]:
            send(*spec)
        self.ev_compute = torch.cuda.Event(enable_timing=trace is not None)
        self.ev_compute.record(cur)
        if trace is not None:
            trace.append((t_begin, self.ev_compute, marks))
        self.ev_down = torch.cuda.Event()
        self.ev_down.record(down)
        self.keep = keep

        def collect():
            out = {}
            for name, (host, done, np_dtype, flag_host, raster) in pending.items():
                done.synchronize()
                arr = host
                if flag_host is not None and int(flag_host[0]) != 0:
                    # not int16-representable: fetch the float32 raster itself (still intact: the slot is not reused
                    # before this tile has been collected)
                    arr = dev.download(raster.with_ref(np_dtype))
                elif arr.dtype != np_dtype:                          # int16 -> float32 / float64 on host threads
                    wide = dev.pinned_empty(arr.shape, np_dtype)
                    _lib.check(lib.hd_host_widen_i16(ctypes.c_void_p(wide.ctypes.data), dev.hd_dtype_of(np_dtype),
                                                     ctypes.c_void_p(arr.ctypes.data), arr.size, self.host_threads))
                    arr = wide
                out[name] = arr
            return out
        return collect


class NarrowDownload:
    """The final DEM holds integer metres (hydro_dem_process.py:149 rounds it): it crosses PCIe as int16 (a quarter of the
    float64 bytes) in row chunks on the ``down`` stream, and a helper thread widens each chunk to float64 on the host's
    cores as it lands -- underneath the sink-fill and the download of the filled DEM.  hd_pack_i16 raises a device flag
    if any value is not an int16 integer; ``result()`` fetches the float64 raster itself then.  Same bits either way."""

    def __init__(self, raster, cur, down, chunks=8):
        import threading
        import torch
        lib = _lib.load()
        ny, nx = raster.shape
        self.raster = raster
        dense = torch.empty((ny, nx), dtype=torch.int16, device=dev.device())
        flag = torch.zeros(1, dtype=torch.int32, device=dev.device())
        with torch.cuda.stream(cur):
            _lib.check(lib.hd_pack_i16(raster.ptr, raster.pitch, ctypes.c_void_p(dense.data_ptr()), ny, nx,
                                       ctypes.c_void_p(flag.data_ptr()), dev.stream_ptr()))
        ev = torch.cuda.Event()
        ev.record(cur)
        down.wait_event(ev)
        dense.record_stream(down)
        flag.record_stream(down)
        flag_host = dev.pinned_empty((1,), np.int32)
        _lib.check(lib.hd_memcpy2d_d2h(ctypes.c_void_p(flag_host.ctypes.data), 4, ctypes.c_void_p(flag.data_ptr()), 4, 4, 1,
                                       ctypes.c_void_p(down.cuda_stream)))
        host16 = dev.pinned_empty((ny, nx), np.int16)
        self.wide = wide = dev.pinned_empty((ny, nx), np.float64)
        parts = []
        step = max(1, -(-ny // chunks))
        for a in range(0, ny, step):
            b = min(ny, a + step)
            nbytes = (b - a) * nx * 2
            _lib.check(lib.hd_memcpy2d_d2h(ctypes.c_void_p(host16[a:b].ctypes.data), nbytes,
                                           ctypes.c_void_p(dense.data_ptr() + a * nx * 2), nbytes, nbytes, 1,
                                           ctypes.c_void_p(down.cuda_stream)))
            done = torch.cuda.Event()
            done.record(down)
            parts.append((a, b, done))
        self.nbytes, self.extra_bytes = host16.nbytes + 4, 0
        self._last_copy, self._host16 = parts[-1][2], host16
        self.state = state = {"inexact": False, "error": None}
        device_index = torch.cuda.current_device()
        threads = host_threads()

        def widen():
            try:
                torch.cuda.set_device(device_index)
                for a, b, done in parts:
                    done.synchronize()
                    if int(flag_host[0]) != 0:                         # copied before the first chunk
                        state["inexact"] = True
                        return
                    _lib.check(lib.hd_host_widen_i16(ctypes.c_void_p(wide[a:b].ctypes.data), _lib.F64,
                                                     ctypes.c_void_p(host16[a:b].ctypes.data), (b - a) * nx, threads))
            except Exception as exc:     # noqa: BLE001  (re-raised on the calling thread)
                state["error"] = exc

        self.thread = threading.Thread(target=widen, name="hydrodem-widen")
        self.thread.start()

    def result(self):
        self.thread.join()
        if self.state["error"] is not None:
            raise self.state["error"]
        if self.state["inexact"]:
            self._last_copy.synchronize()                              # the int16 chunks still in flight own host16
            self.wide = dev.download(self.raster)                      # float64 over PCIe after all
            self.extra_bytes = self.wide.nbytes
        return self.wide


def overlapped_to_host(streams, inputs, run, narrow_final):
    """The eager ``apply_to_host`` of ConditioningChain and of Band: host arrays in and out, the PCIe traffic underneath
    the kernels.  ``inputs``: ``(name, host ndarray, destination raster or None)`` in the order the chain first needs
    them, uploaded on ``streams[0]`` (into a new raster without a destination).  ``run(rasters, ready, on_ready)``
    enqueues the chain (waiting for ``ready[name]`` where an input is first used, calling ``on_ready(name, raster)``
    when an output is enqueued) and returns a function that reads the sink-fill's status word, or None.  Outputs go down
    on ``streams[1]`` at once, the final DEM as int16 when ``narrow_final``.  Returns the ndarrays and the (H2D, D2H)
    bytes."""
    import torch
    cur = torch.cuda.current_stream()
    up, down = streams
    up.wait_stream(cur)                                   # recycled blocks: earlier work on them is over
    rasters, ready = {}, {}
    for name, host, into in inputs:
        if into is None:
            rasters[name], ready[name] = dev.upload_async(host, up)
        else:
            rasters[name], ready[name] = into, dev.upload_into(into, host, up)
        if not dev._is_pinned(host):
            up.synchronize()                              # a pageable source may be released by the caller
    pending, narrow = {}, {}

    def on_ready(name, raster):
        if narrow_final and raster.dtype == _lib.F32 and raster.ref_dtype == np.float64:
            narrow[name] = NarrowDownload(raster, cur, down)
            return
        conv = dev.convert(raster, dev.hd_dtype_of(raster.ref_dtype))
        ev = torch.cuda.Event()
        ev.record(cur)
        down.wait_event(ev)
        pending[name] = dev.download_async(conv, down) + (conv,)

    fill_status = run(rasters, ready, on_ready)
    out = {}
    for name, (host, ev, _conv) in pending.items():
        ev.synchronize()
        out[name] = host
    for name, nd in narrow.items():
        out[name] = nd.result()
    if fill_status is not None:
        check_fill_status(fill_status())
    transfer = (sum(host.nbytes for _, host, _ in inputs),
                sum(out[name].nbytes for name in pending) + sum(nd.nbytes + nd.extra_bytes for nd in narrow.values()))
    return {k: out[k] for k in ("final", "filled", "d8") if k in out}, transfer


class ConditioningChain:
    """Run the whole chain on the GPU.

    >>> out = ConditioningChain().apply(srtm, groves_class, hsheds)
    >>> out.final, out.filled, out.d8
    """

    def __init__(self, *, groves_iterations=3, with_hydrology=True, keep_intermediates=False, fill_stats=False,
                 keep_complete=False, fused_combine=True, sparse_groves=True, fused_lagoons=True):
        self.fused_lagoons = fused_lagoons    # False: TidyingLagoons as three kernels (tests compare both)
        # apply_to_host: rasters of at least this many cells run eagerly on three streams instead of captured slots
        self.eager_cells = int(os.environ.get("HD_EAGER_CELLS", str(64 << 20)))
        # ... and send the final DEM (integer metres) down as int16, widened to float64 by host threads as it lands
        self.narrow_final = narrow_final_default()
        self.sparse_groves = sparse_groves    # False: every groves iteration rewrites the whole raster (tests compare both)
        self.keep_complete = keep_complete    # also return / keep the float64 sum of the final terms ("dem_complete")
        self.fused_combine = fused_combine    # False: hd_final_terms + hd_convolve3 as two kernels (tests compare both)
        self.fill_stats = fill_stats          # True: SinkFill synchronises once to report its tile-visit count
        self.groves_iterations = groves_iterations
        self.with_hydrology = with_hydrology
        self.keep_intermediates = keep_intermediates

    # ---- device path --------------------------------------------------------------------------------
    # ---- the chain in four stages (each one is a CUDA-graph segment of ``stream``) --------------------
    def _stage_fourier(self, st, srtm):
        """DetectApplyFourier on the raw SRTM raster (image_srtm.py:125-126)."""
        st["daf"] = daf = cf.DetectApplyFourier()
        st["fourier"] = daf.run_device(srtm)                               # F32 storage, ref float64

    def _stage_groves(self, st, groves_class):
        """BinaryClosing of the groves class + GrovesCorrectionsIter (image_srtm.py:177-199)."""
        st["groves"] = groves = ef.BinaryClosing(structure=np.ones((3, 3))).run_device(groves_class)   # U8 0/1
        dem = st["fourier"]
        if self.sparse_groves and dem.dtype == _lib.F32 and not self.keep_intermediates and self.groves_iterations >= 1:
            # A cell outside the groves class leaves GrovesCorrection as it entered: after a full first pass (which also
            # flags the tiles that hold a groves cell) the later iterations ping-pong between the two rasters and only
            # load / store what can change (hd_groves_correction_tiles).  The stripe-free DEM's buffer is reused as the
            # second raster (it is dead after the first iteration unless the intermediates are kept).
            lib = _lib.load()
            import torch
            ny, nx = dem.shape
            flags = torch.empty(int(lib.hd_groves_tile_count(ny, nx)), dtype=torch.uint8, device=dev.device())
            g8 = dev.convert(groves, _lib.U8)
            src, dst = dem, dev.empty(ny, nx, _lib.F32, np.float64)
            for it in range(self.groves_iterations):
                _lib.check(lib.hd_groves_correction_tiles(src.ptr, src.pitch, g8.ptr, g8.pitch, dst.ptr, dst.pitch, ny, nx,
                                                          cf.GrovesCorrection.window_size, cf.GrovesCorrection.threshold,
                                                          ctypes.c_void_p(flags.data_ptr()), 1 if it else 0,
                                                          dev.stream_ptr()),
                           window_size=cf.GrovesCorrection.window_size, shape=dem.shape)
                src, dst = dst, src
            st["srtm"] = src.with_ref(np.float64)
            return
        gc = cf.GrovesCorrection(groves)
        for _ in range(self.groves_iterations):
            dem = gc.run_device(dem, out_dtype=_lib.F32)
        st["srtm"] = dem

    def _stage_combine(self, st, hsheds, rivers):
        """LagoonsDetection (custom_filters.py:633-661, float32 / uint8 intermediates), the sum of the final terms
        (hydro_dem_process.py:60-91, :148) and PostProcessingFinal (:149), float64 like the reference."""
        self._stage_lagoons(st, hsheds)
        self._stage_final(st, rivers)

    def _stage_lagoons(self, st, hsheds):
        """The HydroSHEDS branch up to the lagoon values: independent of the SRTM branch (run_device runs it before the
        groves stage, so that an overlapped upload can bring HydroSHEDS second and the groves mask last)."""
        lib = _lib.load()
        ny, nx = hsheds.shape
        st["hsheds_nan_fixed"] = fixed = cf.CorrectNANValues().run_device(hsheds)
        st["majority"] = majority = cf.MajorityFilter(window_size=11).run_device(fixed)
        if self.fused_lagoons and majority.dtype == _lib.F32:
            # TidyingLagoons as one kernel (erode x2 -> expand 7 -> x majority -> max 7x7): hd_tidy_lagoons
            tidy = dev.empty(ny, nx, _lib.F32, np.float64)
            _lib.check(lib.hd_tidy_lagoons(majority.ptr, majority.pitch, tidy.ptr, tidy.pitch, ny, nx, dev.stream_ptr()),
                       window_size=7, shape=(ny, nx))
            st["lagoons_values"] = tidy
        else:
            eroded = ef.BinaryErosion(iterations=2).run_device(majority)
            prod = dev.empty(ny, nx, _lib.F32, np.float64)                  # majority * expand(7): one fused kernel
            _lib.check(lib.hd_expand_select(eroded.ptr, eroded.dtype, eroded.pitch, majority.ptr, majority.pitch, prod.ptr,
                                            prod.pitch, ny, nx, 7, dev.stream_ptr()))
            st["lagoons_values"] = tidy = ef.GreyDilation(size=(7, 7)).run_device(prod)

    def _stage_final(self, st, rivers):
        lib = _lib.load()
        dem, fixed, tidy = st["srtm"], st["hsheds_nan_fixed"], st["lagoons_values"]
        ny, nx = dem.shape
        fixed32 = dev.convert(fixed, _lib.F32)
        final32 = dev.empty(ny, nx, _lib.F32, np.float32)                   # integer metres: exact in float32
        if rivers is None and dem.dtype == _lib.F32 and self.fused_combine:
            # no rivers: the sum of the final terms and PostProcessingFinal are ONE pass (hd_final_mean3, same bits as the
            # two separate kernels); the float64 `complete` raster is only written when somebody wants to look at it
            complete = dev.empty(ny, nx, _lib.F64, np.float64) if (self.keep_intermediates or self.keep_complete) else None
            _lib.check(lib.hd_final_mean3(dem.ptr, dem.pitch, tidy.ptr, tidy.pitch, fixed32.ptr, fixed32.pitch, final32.ptr,
                                          final32.pitch, complete.ptr if complete is not None else None,
                                          complete.pitch if complete is not None else 0, ny, nx, dev.stream_ptr()))
            if complete is not None:
                st["dem_complete"] = complete
            st["final"] = final32.with_ref(np.float64)                      # widened to the reference's float64 on download
            st["final32"] = final32
            return
        riv = dev.convert(rivers, _lib.F32) if rivers is not None else None
        st["dem_complete"] = complete = dev.empty(ny, nx, _lib.F64, np.float64)
        _lib.check(lib.hd_final_terms(dem.ptr, dem.dtype, dem.pitch, tidy.ptr, tidy.pitch, fixed32.ptr, fixed32.pitch,
                                      riv.ptr if riv is not None else None, riv.pitch if riv is not None else 0,
                                      complete.ptr, complete.dtype, complete.pitch, ny, nx, dev.stream_ptr()))
        st["final"] = cf.PostProcessingFinal().run_device(complete, copy32=final32)
        st["final32"] = final32

    def _stage_hydrology(self, st):
        """NEW stages: SinkFill + D8FlowDirection on the final DEM."""
        fill = nf.SinkFillD8(want_stats=self.fill_stats)             # fill + fused NaN restore / D8 pass
        st["filled"], st["d8"] = fill.run_device(st["final32"])
        st["fill"] = fill

    def _result(self, st):
        out = {"final": st["final"]}
        info = {}
        if self.with_hydrology:
            out.update(filled=st["filled"], d8=st["d8"])
            info["fill_sweeps"] = st["fill"].sweeps
            info["fill"] = st["fill"]
        if self.keep_complete and "dem_complete" in st:
            out["dem_complete"] = st["dem_complete"]
        if self.keep_intermediates:
            daf = st["daf"]
            out.update(fourier=st["fourier"], fourier_mask=daf._mask_dev, fabs=daf._fabs_dev,
                       **{k: st[k] for k in ("groves", "srtm", "hsheds_nan_fixed", "majority", "lagoons_values",
                                             "dem_complete")})
        return ChainResult(out, info)

    def run_device(self, srtm, groves_class, hsheds, rivers=None, ready=None, on_ready=None):
        """``ready``: optional {name: torch.cuda.Event} -- the compute stream waits for an input's upload only where
        that input is first used.  ``on_ready(name, raster)`` is called as soon as an output raster is enqueued."""
        import torch
        cur = torch.cuda.current_stream()

        def need(name):
            if ready and ready.get(name) is not None:
                cur.wait_event(ready[name])

        def emit(name):
            if on_ready:
                on_ready(name, st[name])

        st = {}
        need("srtm")
        self._stage_fourier(st, srtm)
        need("hsheds")
        self._stage_lagoons(st, hsheds)                       # independent of the SRTM branch
        need("groves")
        self._stage_groves(st, groves_class)
        if rivers is not None:
            need("rivers")
        self._stage_final(st, rivers)
        emit("final")
        if self.with_hydrology:
            self._stage_hydrology(st)
            emit("filled")
            emit("d8")
        return self._result(st)

    def capture(self, srtm, groves_class, hsheds, rivers=None):
        """Capture the whole device-resident chain for these (static) input rasters in ONE CUDA graph.

        The chain is ~40 short kernel launches; issued one by one from Python the host cannot keep a B200 busy
        (~4 ms of interpreter + ctypes time per pass).  A captured graph replays them with a single launch.  Returns a
        CapturedChain: ``replay()`` re-runs the chain on whatever the input rasters hold at that moment and returns
        the same ChainResult (its rasters are the graph's static output buffers)."""
        import torch
        self.run_device(srtm, groves_class, hsheds, rivers)          # warm-up: FFT plans, function attributes
        torch.cuda.synchronize()
        lib = _lib.load()
        n0 = lib.hd_launch_count()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            result = self.run_device(srtm, groves_class, hsheds, rivers)
        return CapturedChain(graph, result, int(lib.hd_launch_count() - n0))

    # ---- streaming host API: a sequence of tiles through double-buffered graph slots -------------------
    def stream(self, items, depth=2):
        """Run a sequence of tiles through the chain with the PCIe traffic of neighbouring tiles overlapped.

        ``items`` yields ``(srtm_raw, groves_class_raw, hsheds[, rivers])`` ndarray tuples (HydroDEMProcess handles one
        such tile per run, hydro_dem_process.py:122-153; a mosaic job is a sequence of them).  Yields, in order, one
        ``{"final", "filled", "d8"}`` dict of ndarrays per tile.  Each of the ``depth`` slots owns static input
        rasters and the chain captured as four CUDA-graph segments; tile i+1 uploads while tile i computes and tile
        i-1 downloads, so the steady-state cost per tile is max(kernels, H2D, D2H) instead of their sum."""
        import collections
        import torch
        rings = self.__dict__.setdefault("_slot_rings", {})
        # Waiting for a tile's downloads and widening its int16 results (2 ms of host threads per 3601^2 tile) happens on
        # a helper thread, so that this thread is free to enqueue the following tiles; both release the GIL.
        pool = self._collector(torch.cuda.current_device()) if depth > 1 else None
        inflight = collections.deque()

        def launch(slot, arrays):
            collect = slot.submit(arrays)
            return pool.submit(collect).result if pool is not None else collect

        for k, item in enumerate(items):
            arrays = self._check_inputs(*item)
            # one tile at a time (depth 1) is a latency call: the filled DEM then travels as float32, because widening it
            # on the host would sit at the very end of the critical path
            narrow_filled = depth > 1
            key = tuple((n, a.shape, a.dtype.str) for n, a in arrays.items()) + (narrow_filled,)
            ring = rings.setdefault(key, [])
            if k % depth >= len(ring):
                while inflight:                                      # capturing synchronises the device anyway
                    yield inflight.popleft()[1]()
                ring.append(_StreamSlot(self, arrays, narrow_filled))    # captured once per shape, kept for later calls
            slot = ring[min(k % depth, len(ring) - 1)]
            while any(s is slot for s, _ in inflight):               # the slot's previous tile must be collected first
                yield inflight.popleft()[1]()
            self.last_transfer_bytes = slot.transfer_bytes           # (H2D, D2H) PCIe bytes of one tile
            inflight.append((slot, launch(slot, arrays)))
            while len(inflight) >= depth:
                yield inflight.popleft()[1]()
        while inflight:
            yield inflight.popleft()[1]()

    def _collector(self, device_index):
        """One helper thread per chain (results come back in order), bound to this process's device."""
        pool = self.__dict__.get("_collect_pool")
        if pool is None:
            import concurrent.futures
            import torch
            pool = concurrent.futures.ThreadPoolExecutor(max_workers=1, thread_name_prefix="hydrodem-collect",
                                                         initializer=torch.cuda.set_device, initargs=(device_index,))
            self._collect_pool = pool
        return pool

    def release(self):
        """Drop the captured slots of ``stream`` / ``apply_to_host`` (their device memory returns to the allocator)."""
        self.__dict__.pop("_slot_rings", None)
        pool = self.__dict__.pop("_collect_pool", None)
        if pool is not None:
            pool.shutdown(wait=True)

    def _check_inputs(self, srtm_raw, groves_class_raw, hsheds, rivers=None):
        arrays = dict(srtm=srtm_raw, groves=groves_class_raw, hsheds=hsheds)
        if rivers is not None:
            arrays["rivers"] = rivers
        for a in arrays.values():
            if not isinstance(a, np.ndarray):
                raise NumpyArrayExpectedError(a)
        if not (srtm_raw.shape == groves_class_raw.shape == hsheds.shape):
            raise ValueError("srtm, groves_class and hsheds must have the same shape")
        dev.require_cuda()
        return arrays

    # ---- host API ---------------------------------------------------------------------------------
    def upload_inputs(self, srtm_raw, groves_class_raw, hsheds, rivers=None):
        self._check_inputs(srtm_raw, groves_class_raw, hsheds, rivers)
        return (dev.upload(srtm_raw), dev.upload(groves_class_raw), dev.upload(hsheds),
                dev.upload(rivers) if rivers is not None else None)

    def apply(self, srtm_raw, groves_class_raw, hsheds, rivers=None):
        """ndarrays in -> ChainResult (``final`` float64, ``filled`` float32, ``d8`` uint8); results are copied to
        the host lazily, on first access."""
        return self.run_device(*self.upload_inputs(srtm_raw, groves_class_raw, hsheds, rivers))

    def apply_to_host(self, srtm_raw, groves_class_raw, hsheds, rivers=None):
        """ndarrays in -> dict of ndarrays (``final``, ``filled``, ``d8``) with the PCIe traffic overlapped with the
        kernels: inputs go up on a copy stream (the Fourier stage starts as soon as the SRTM raster has landed,
        HydroSHEDS and groves follow underneath it), and each result starts its way down on a second copy stream
        the moment its last kernel is enqueued (the final DEM travels while the sink-fill runs).  Pageable inputs
        are staged through pinned buffers first.  One tile through ``stream``: the first call for a raster shape
        captures the chain's CUDA graphs, later calls replay them."""
        if srtm_raw.size >= self.eager_cells:
            return self._apply_overlapped(self._check_inputs(srtm_raw, groves_class_raw, hsheds, rivers))
        for out in self.stream([(srtm_raw, groves_class_raw, hsheds, rivers)], depth=1):
            return out

    def _apply_overlapped(self, arrays):
        """apply_to_host for a mosaic-sized raster: the same three streams, but the kernels are launched eagerly -- a
        captured slot would pin the whole working set of a 36000^2 mosaic in a private graph pool, and ~45 launches are
        nothing against 160 ms of kernels.  Timeline at 36000^2 on PCIe 5: SRTM up (94 ms) | Fourier stage under the
        HydroSHEDS upload (94 ms) | lagoon branch under the groves upload (24 ms) | groves, final terms | final DEM
        down as int16 (47 ms) over the sink-fill, widened on the host underneath | filled DEM + D8 down (118 ms)."""
        order = ("srtm", "hsheds", "groves", "rivers")                # the order run_device first needs them in
        inputs = [(n, np.ascontiguousarray(arrays[n]), None) for n in order if n in arrays]

        def run(rasters, ready, on_ready):
            res = self.run_device(rasters["srtm"], rasters["groves"], rasters["hsheds"], rasters.get("rivers"),
                                  ready=ready, on_ready=on_ready)
            fill = res.info.get("fill")
            return fill.status if fill is not None else None

        out, self.last_transfer_bytes = overlapped_to_host(copy_streams(self), inputs, run, self.narrow_final)
        return out

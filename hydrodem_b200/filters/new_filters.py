"""Stages named by the conditioning chain that the reference does not contain
(SURVEY.md section 0.3): median filter, sink-fill and D8 flow direction.

They follow the reference's filter idiom (keyword-only constructors,
``apply(ndarray) -> ndarray``).  Their parity oracle is this repository's own
definition (oracle/stencils.py:median, oracle/hydrology.py) -- "parity
unpinned" with respect to the reference.
"""
import ctypes

import numpy as np

from . import DeviceFilter
from .. import _lib, device as dev
from .custom_filters import WindowFilter, as_f32, check_window


class MedianFilter(WindowFilter):
    """np.nanmedian over a ws*ws (or corner-less "circular") window, ws in {3, 5};
    result in the input's dtype with the ws//2 border unchanged."""

    def __init__(self, *, window_size, circular=False):
        self.window_size = window_size
        self.circular = circular

    def run_device(self, raster):
        check_window(raster.shape, self.window_size)
        src = as_f32(raster)
        out = dev.empty(raster.ny, raster.nx, _lib.F32, raster.ref_dtype)
        _lib.check(_lib.load().hd_median(src.ptr, src.pitch, out.ptr, out.pitch, src.ny, src.nx, int(self.window_size),
                                         int(bool(self.circular)), dev.stream_ptr()),
                   window_size=self.window_size, shape=raster.shape)
        if raster.dtype != _lib.F32:
            # the border keeps the caller's exact values (dem.copy() convention)
            wide = dev.convert(out, raster.dtype, raster.ref_dtype)
            h = int(self.window_size) // 2
            ny, nx = raster.shape
            for (y0, y1, x0, x1) in ((0, h, 0, nx), (ny - h, ny, 0, nx), (h, ny - h, 0, h), (h, ny - h, nx - h, nx)):
                if y1 > y0 and x1 > x0:
                    dev.elementwise(_lib.OP_COPY, raster.sub(y0, y1, x0, x1), None, wide.sub(y0, y1, x0, x1))
            return wide
        return out


class SinkFill(DeviceFilter):
    """Depression filling: the Planchon-Darboux fixed point with eps = 0 and
    8-connectivity; frame cells and NaN cells are outlets.  float32 result.
    ``sweeps`` holds the number of tile visits of the finest level in the last call."""

    def __init__(self, *, want_stats=True):
        self.want_stats = want_stats      # False: no host synchronisation inside the call
        self.sweeps = None

    def run_device(self, raster):
        lib = _lib.load()
        src = as_f32(raster)
        out = dev.empty(raster.ny, raster.nx, _lib.F32, np.float32)
        nbytes = lib.hd_pdfill_workspace_bytes(raster.ny, raster.nx)
        work = dev.scratch(nbytes)
        import torch
        # statistics need a host synchronisation inside the call: impossible while a CUDA graph is being captured
        stats = self.want_stats and not torch.cuda.is_current_stream_capturing()
        visits = ctypes.c_int(-1)
        self._work = work
        _lib.check(lib.hd_pdfill(src.ptr, src.pitch, out.ptr, out.pitch, src.ny, src.nx, ctypes.c_void_p(work.data_ptr()),
                                 nbytes, ctypes.byref(visits) if stats else None, dev.stream_ptr()))
        self.sweeps = visits.value if stats else None
        return out


class SinkFillD8(DeviceFilter):
    """SinkFill followed by D8FlowDirection as ONE launch group: the fill, then a single pass that restores NaN at the
    nodata cells and writes the flow directions (``hd_pdfill_d8``).  ``run_device`` returns (filled, d8).
    ``status()`` reads the fill's sticky status word (0 = fixed point reached) -- it synchronises the stream."""

    def __init__(self, *, want_stats=False):
        self.want_stats = want_stats
        self.sweeps = None
        self._work = None

    def run_device(self, raster):
        import torch
        lib = _lib.load()
        src = as_f32(raster)
        filled = dev.empty(raster.ny, raster.nx, _lib.F32, np.float32)
        d8 = dev.empty(raster.ny, raster.nx, _lib.U8, np.uint8)
        nbytes = lib.hd_pdfill_workspace_bytes(raster.ny, raster.nx)
        self._work = work = dev.scratch(nbytes)
        # statistics need a host synchronisation inside the call: impossible while a CUDA graph is being captured
        stats = self.want_stats and not torch.cuda.is_current_stream_capturing()
        visits = ctypes.c_int(-1)
        _lib.check(lib.hd_pdfill_d8(src.ptr, src.pitch, filled.ptr, filled.pitch, d8.ptr, d8.pitch, src.ny, src.nx,
                                    ctypes.c_void_p(work.data_ptr()), nbytes, ctypes.byref(visits) if stats else None,
                                    dev.stream_ptr()))
        self.sweeps = visits.value if stats else None
        return filled, d8

    def status(self):
        st = ctypes.c_int(-1)
        _lib.check(_lib.load().hd_pdfill_status(ctypes.c_void_p(self._work.data_ptr()), ctypes.byref(st), dev.stream_ptr()))
        return st.value

    def apply(self, image_to_filter):
        from . import Filter
        Filter.apply(self, image_to_filter)
        filled, d8 = self.run_device(dev.upload(image_to_filter))
        return dev.download(filled), dev.download(d8)


class D8FlowDirection(DeviceFilter):
    """D8 flow direction (ESRI codes, uint8) of a filled surface."""

    def run_device(self, raster):
        src = as_f32(raster)
        out = dev.empty(raster.ny, raster.nx, _lib.U8, np.uint8)
        _lib.check(_lib.load().hd_d8(src.ptr, src.pitch, out.ptr, out.pitch, src.ny, src.nx, dev.stream_ptr()))
        return out

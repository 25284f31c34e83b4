"""Windowed and composed filters of the conditioning chain, CUDA backed.

Drop-in for ``cguerrero/hydrodem/filters/custom_filters.py``: same class
names, keyword-only constructors, result dtypes, border conventions and
aliasing (the in-place filters still return the caller's own array).  The
per-cell Python loops over ``SlidingWindow`` are gone: each class is one or a
few kernels of libhydrodem_b200 working on device rasters.
"""
import numpy as np

from . import ComposedFilter, ComposedFilterResults, DeviceFilter, Filter, LazyResults, run_stage
from .. import _lib, device as dev
from ..exceptions import (NumpyArrayExpectedError, WindowSizeEvenError, WindowSizeHighError)
from .extension_filters import (AbsoluteValues, Around, BinaryClosing, BinaryErosion, BitwiseXOR, Convolve,  # noqa: F401
                                GreyDilation)
from .simple_filters import (AdditionFilter, BooleanToInteger, GreaterThan, LowerThan, ProductFilter,     # noqa: F401
                             SubtractionFilter, binary_op)


def check_window(shape, window_size):
    """Guards of SlidingWindow.window_size (sliding_window.py:150-156): too large first, then even."""
    if any(window_size > n for n in shape):
        raise WindowSizeHighError(window_size, shape)
    if window_size % 2 != 1:
        raise WindowSizeEvenError(window_size)


def as_f32(raster):
    """The ``grid.astype('float32')`` every sliding window starts with (sliding_window.py:132)."""
    return dev.convert(raster, _lib.F32)


class WindowFilter(DeviceFilter):
    """A filter that builds SlidingWindow objects in the reference: the
    ndarray check comes from the grid setter (sliding_window.py:130-131)."""

    window_size = None

    def apply(self, image_to_filter):
        if not isinstance(image_to_filter, np.ndarray):
            raise NumpyArrayExpectedError(image_to_filter)
        check_window(image_to_filter.shape, self.window_size)
        return dev.download(self.run_device(dev.upload(image_to_filter)))


class MajorityFilter(WindowFilter):
    """Mode of the corner-less window if it fills more than 70 % of it
    (custom_filters.py:22-73).  float64 zeros elsewhere and on the border."""

    def __init__(self, *, window_size):
        self.window_size = window_size

    def run_device(self, raster):
        check_window(raster.shape, self.window_size)
        ws = int(self.window_size)
        min_count = int(np.floor((ws ** 2 - 1) * 0.7)) + 1        # count > (ws**2 - 1) * 0.7  (:71)
        src = as_f32(raster)
        out = dev.empty(raster.ny, raster.nx, _lib.F32, np.float64)
        _lib.check(_lib.load().hd_majority(src.ptr, src.pitch, out.ptr, out.dtype, out.pitch, src.ny, src.nx, ws,
                                           min_count, dev.stream_ptr()), window_size=ws, shape=raster.shape)
        return out


class ExpandFilter(WindowFilter):
    """1 where any cell of the corner-less window is > 0 (custom_filters.py:76-125)."""

    def __init__(self, *, window_size):
        self.window_size = window_size

    def run_device(self, raster):
        check_window(raster.shape, self.window_size)
        src = raster if raster.dtype in (_lib.U8, _lib.F32) else as_f32(raster)
        out = dev.empty(raster.ny, raster.nx, _lib.U8, np.float64)
        _lib.check(_lib.load().hd_expand(src.ptr, src.dtype, src.pitch, out.ptr, out.dtype, out.pitch, src.ny, src.nx,
                                         int(self.window_size), dev.stream_ptr()),
                   window_size=self.window_size, shape=raster.shape)
        return out


class _InPlace3(WindowFilter):
    """Shared plumbing of the two in-place 3x3 filters: Jacobi on the device
    (the reference reads a float32 snapshot, sliding_window.py:132), result
    copied back into the caller's array, which is returned."""

    _entry = None

    def run_device(self, raster):
        check_window(raster.shape, self.window_size)
        if int(self.window_size) != 3:
            raise dev.DeviceError(f"{type(self).__name__}: only window_size=3 is implemented on the device")
        if raster.dtype in (_lib.F32, _lib.F64):
            src = raster
        elif raster.dtype in (_lib.I16, _lib.U8):
            src = dev.convert(raster, _lib.F32)          # exact, and the windows are float32 anyway (sliding_window.py:132)
        else:
            src = dev.convert(raster, _lib.F64)
        out = dev.empty(raster.ny, raster.nx, src.dtype, raster.ref_dtype)
        fn = getattr(_lib.load(), self._entry)
        _lib.check(fn(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, src.ny, src.nx, dev.stream_ptr()))
        if np.dtype(raster.ref_dtype).kind in "iu":
            # the reference writes the float32 result into the caller's INTEGER array (dem[center] = mean, :316):
            # NumPy truncates toward zero on assignment, and the next stage (MajorityFilter) counts those integers
            dev.elementwise(_lib.OP_TRUNC, out, None, out)
        return out

    def apply(self, image_to_filter):
        if not isinstance(image_to_filter, np.ndarray):
            raise NumpyArrayExpectedError(image_to_filter)
        check_window(image_to_filter.shape, self.window_size)
        return dev.download(self.run_device(dev.upload(image_to_filter)), out=image_to_filter)


class CorrectNANValues(_InPlace3):
    """Voids (< 0) replaced by the float32 mean of their valid neighbours,
    in place (custom_filters.py:260-317)."""

    _entry = "hd_nanfix"

    def __init__(self, *, window_size=3):
        self.window_size = window_size


class IsolatedPoints(_InPlace3):
    """Mask cells without any positive neighbour cleared, in place
    (custom_filters.py:320-366)."""

    _entry = "hd_isolated"

    def __init__(self, *, window_size):
        self.window_size = window_size


class RouteRivers(WindowFilter):
    """Route / expand rivers along the low cells of a reference DEM (custom_filters.py:128-199): a raster scan over the
    mask cells with value 1 that marks the minima of each 3x3 DEM window and consumes them (10000) as it goes -- order
    dependent, run on the device as an order-preserving wavefront (csrc/rivers.cu).  Returns float64 zeros / ones."""

    def __init__(self, *, window_size, dem):
        import copy
        self.window_size = window_size
        self.dem = dem if isinstance(dem, dev.DeviceRaster) else copy.deepcopy(dem)      # (:163)

    def run_device(self, raster):
        import ctypes
        check_window(raster.shape, self.window_size)
        dem = self.dem if isinstance(self.dem, dev.DeviceRaster) else dev.upload(np.ascontiguousarray(self.dem))
        if dem.shape != raster.shape:
            raise ValueError(f"dem shape {dem.shape} does not match the rivers mask {raster.shape}")
        check_window(dem.shape, self.window_size)
        # the working copy the reference mutates: dem_sliding.grid = dem.astype('float32') (sliding_window.py:132)
        g = dev.empty(dem.ny, dem.nx, _lib.F32, np.float32)
        dev.elementwise(_lib.OP_COPY, dem, None, g)
        mask = as_f32(raster)
        out = dev.empty(raster.ny, raster.nx, _lib.U8, np.float64)
        nbytes = raster.ny * 4
        work = dev.scratch(nbytes)
        _lib.check(_lib.load().hd_route_rivers(mask.ptr, mask.pitch, g.ptr, g.pitch, out.ptr, out.pitch, raster.ny, raster.nx,
                                               int(self.window_size), ctypes.c_void_p(work.data_ptr()), nbytes,
                                               dev.stream_ptr()),
                   window_size=self.window_size, shape=raster.shape)
        return out


class ProcessRivers(ComposedFilter):
    """MaskPositives -> ExpandFilter(3) -> RouteRivers(3, dem=hsheds) -> BinaryClosing() (custom_filters.py:770-798)."""

    def __init__(self, hsheds):
        super().__init__()
        self.filters = [MaskPositives(), ExpandFilter(window_size=3), RouteRivers(window_size=3, dem=hsheds),
                        BinaryClosing()]


class ClipLagoonsRivers(ComposedFilter):
    """Rivers minus their intersection with the lagoons: ProductFilter(factor=mask_lagoons) ->
    BitwiseXOR(operand=rivers_routed_closing) (custom_filters.py:801-831)."""

    def __init__(self, mask_lagoons, rivers_routed_closing):
        super().__init__()
        self.filters = [ProductFilter(factor=mask_lagoons), BitwiseXOR(operand=rivers_routed_closing)]


class QuadraticFilter(WindowFilter):
    """Least-squares quadratic smoothing over a square window -- the "isotropic" filter
    (custom_filters.py:202-257).  Result in the input's dtype, ws//2 border unchanged."""

    def __init__(self, *, window_size):
        self.window_size = window_size

    def run_device(self, raster):
        check_window(raster.shape, self.window_size)
        ref = np.dtype(raster.ref_dtype)
        if raster.dtype == _lib.F32 and ref in (np.float32, np.float64):
            src = raster                                     # float32 storage (exact for the float32-cast windows)
        else:
            src = dev.convert(raster, _lib.F64)
        out = dev.empty(raster.ny, raster.nx, src.dtype, ref)
        _lib.check(_lib.load().hd_quadratic(src.ptr, src.pitch, out.ptr, out.pitch, src.dtype, src.ny, src.nx,
                                            int(self.window_size), dev.stream_ptr()),
                   window_size=self.window_size, shape=raster.shape)
        return out


class GrovesCorrection(DeviceFilter):
    """One groves-correction pass (custom_filters.py:664-732): QuadraticFilter(15) -> dem - smooth ->
    > 1.5 -> x groves_class -> 1 - . -> x (dem - smooth) -> + smooth, fused into ONE kernel.
    Returns float64 like the reference.  ``partial_results`` (the five intermediates the reference deep-copies, :728)
    is materialised lazily, with separate kernels, only when somebody reads it."""

    window_size = 15
    threshold = 1.5

    def __init__(self, groves_class):
        self._partials = []
        self._partials_pending = []
        self.groves_class = groves_class
        self._groves_dev = None

    @property
    def partial_results(self):
        """[smooth, dem - smooth, (> 1.5) * 1, x groves_class, 1 - .] per apply() call, in the reference's dtypes."""
        for src in self._partials_pending:
            smooth = QuadraticFilter(window_size=self.window_size).run_device(src)
            hi = binary_op(_lib.OP_RSUB, smooth, src, np.subtract)            # SubtractionFilter(minuend=dem)
            tall = MaskTallGroves().run_device(hi)
            g = self.groves_class if isinstance(self.groves_class, dev.DeviceRaster) else np.asarray(self.groves_class)
            prod = ProductFilter(factor=g).run_device(tall)
            keep = SubtractionFilter(minuend=1).run_device(prod)
            self._partials += [dev.download(r) for r in (smooth, hi, tall, prod, keep)]
        self._partials_pending = []
        return self._partials

    @partial_results.setter
    def partial_results(self, value):
        self._partials, self._partials_pending = list(value), []

    def _groves(self, shape):
        if self._groves_dev is None:
            g = self.groves_class
            if isinstance(g, dev.DeviceRaster):
                self._groves_dev = dev.convert(g, _lib.U8)
            else:
                g = np.asarray(g)
                if g.dtype != np.bool_ and not np.isin(g, (0, 1)).all():
                    raise dev.DeviceError("GrovesCorrection: groves_class must be a 0/1 mask on the device path")
                self._groves_dev = dev.upload(np.ascontiguousarray(g != 0))
        if self._groves_dev.shape != tuple(shape):
            raise ValueError(f"groves_class shape {self._groves_dev.shape} does not match the DEM {tuple(shape)}")
        return self._groves_dev

    def run_device(self, raster, out_dtype=None):
        check_window(raster.shape, self.window_size)
        src = raster if raster.dtype in (_lib.F32, _lib.F64) else dev.convert(raster, _lib.F64)
        if out_dtype is None:
            out_dtype = _lib.F64
        groves = self._groves(raster.shape)
        out = dev.empty(raster.ny, raster.nx, out_dtype, np.float64)
        _lib.check(_lib.load().hd_groves_correction(src.ptr, src.dtype, src.pitch, groves.ptr, groves.pitch, out.ptr,
                                                    out.dtype, out.pitch, src.ny, src.nx, self.window_size,
                                                    self.threshold, dev.stream_ptr()),
                   window_size=self.window_size, shape=raster.shape)
        return out

    def apply(self, image_to_filter):
        if not isinstance(image_to_filter, np.ndarray):
            raise NumpyArrayExpectedError(image_to_filter)
        check_window(image_to_filter.shape, self.window_size)
        src = dev.upload(image_to_filter)
        self._partials_pending.append(src)
        return dev.download(self.run_device(src))


class GrovesCorrectionsIter(ComposedFilter):
    """``iterations`` GrovesCorrection passes (custom_filters.py:735-767)."""

    def __init__(self, groves_class, iterations=3):
        super().__init__()
        shared = groves_class
        if not isinstance(groves_class, dev.DeviceRaster) and isinstance(groves_class, np.ndarray):
            first = GrovesCorrection(groves_class)
            self.filters = [first]
            for _ in range(iterations - 1):
                nxt = GrovesCorrection(groves_class)
                nxt._share = first                      # upload the mask once
                self.filters.append(nxt)
        else:
            self.filters = [GrovesCorrection(shared) for _ in range(iterations)]

    def run_device(self, raster):
        content = raster
        first = self.filters[0] if self.filters else None
        for f in self.filters:
            if isinstance(f, GrovesCorrection) and f is not first and getattr(f, "_share", None) is first:
                f._groves_dev = first._groves(content.shape)
            content = run_stage(f, content)
        return content

    def apply(self, image_to_filter):
        Filter.apply(self, image_to_filter)
        check_window(image_to_filter.shape, 15)
        return dev.download(self.run_device(dev.upload(image_to_filter)))


class MaskNegatives(ComposedFilter):
    """(image < 0) * 1 (custom_filters.py:465-486)."""

    def __init__(self):
        super().__init__()
        self.filters = [LowerThan(value=0.0), BooleanToInteger()]


class MaskPositives(ComposedFilter):
    """(image > 0) * 1 (custom_filters.py:489-510)."""

    def __init__(self):
        super().__init__()
        self.filters = [GreaterThan(value=0.0), BooleanToInteger()]


class MaskTallGroves(ComposedFilter):
    """(image > 1.5) * 1 (custom_filters.py:513-534)."""

    def __init__(self):
        super().__init__()
        self.filters = [GreaterThan(value=1.5), BooleanToInteger()]


class TidyingLagoons(ComposedFilter):
    """BinaryErosion(2) -> ExpandFilter(7) -> x majority image -> GreyDilation(7x7)
    (custom_filters.py:564-610)."""

    def __init__(self):
        super().__init__()
        self.filters = [BinaryErosion(iterations=2), ExpandFilter(window_size=7), ProductFilter(),
                        GreyDilation(size=(7, 7))]

    def run_device(self, raster):
        self.filters[2].factor = raster                     # the majority image is the factor (:607)
        return super().run_device(raster)

    def apply(self, image_to_filter):
        Filter.apply(self, image_to_filter)
        return dev.download(self.run_device(dev.upload(image_to_filter)))


class LagoonsDetection(ComposedFilterResults):
    """CorrectNANValues -> MajorityFilter(11) -> TidyingLagoons -> MaskPositives
    (custom_filters.py:613-661)."""

    def __init__(self):
        super().__init__()
        self.filters = [CorrectNANValues(), MajorityFilter(window_size=11), TidyingLagoons(), MaskPositives()]
        self.hsheds_nan_fixed = None
        self.mask_lagoons = None
        self.lagoons_values = None

    def apply(self, image_to_filter):
        Filter.apply(self, image_to_filter)
        check_window(image_to_filter.shape, 3)
        result = self._run(dev.upload(image_to_filter))
        # CorrectNANValues works in place: the caller's array is updated and IS results["CorrectNANValues"] (:658)
        fixed = dev.download(self.results.device("CorrectNANValues"), out=image_to_filter)
        self.results["CorrectNANValues"] = fixed
        self.hsheds_nan_fixed = fixed
        self.mask_lagoons = self.results["MaskPositives"]
        self.lagoons_values = self.results["TidyingLagoons"]
        return dev.download(result) if isinstance(result, dev.DeviceRaster) else result


class PostProcessingFinal(ComposedFilter):
    """Convolve() (3x3 mean, reflect) then Around() (custom_filters.py:1104-1125), fused in one kernel."""

    def __init__(self):
        super().__init__()
        self.filters = [Convolve(), Around()]

    def run_device(self, raster, copy32=None):
        conv, rnd = self.filters
        if type(conv) is Convolve and type(rnd) is Around:
            return conv.run_device(raster, do_round=True, copy32=copy32)
        return super().run_device(raster)

    def apply(self, image_to_filter):
        Filter.apply(self, image_to_filter)
        return dev.download(self.run_device(dev.upload(image_to_filter)))


# ---- Fourier stripe removal --------------------------------------------------------------------------------
from .extension_filters import FourierIShift, FourierITransform, FourierShift, FourierTransform  # noqa: E402,F401
import ctypes  # noqa: E402

FOURIER_MARGIN = 10            # FourierProcessQuarters._margin (custom_filters.py:911)
BLANKS_WINDOW = 55             # DetectBlanksFourier (custom_filters.py:457)
BLANKS_INNER = 5               # BlanksFourier (custom_filters.py:419)
BLANKS_FACTOR = 4.0            # centre > 4 * mean (custom_filters.py:424)


def _hollow_pass(src_f32, prev_mask, window_size, last=False, flags_out=None, flags_in=None):
    """One BlanksFourier pass on the device -> (accumulated mask, modified image F32).  ``last``: the mask is
    stored as float32 (what IsolatedPoints reads next) and the modified image is not written.  ``flags_out`` /
    ``flags_in``: per-tile hit flags (torch uint8) written by a first pass / restricting a second pass to the tiles
    where it can find anything (hd_hollow_mean_detect_tiles)."""
    mask = dev.empty(src_f32.ny, src_f32.nx, _lib.F32 if last else _lib.U8, np.float64)
    mod = None if last else dev.empty(src_f32.ny, src_f32.nx, _lib.F32, np.float64)
    pp, ppitch = (prev_mask.ptr, prev_mask.pitch) if prev_mask is not None else (None, 0)
    mp, mpitch = (mod.ptr, mod.pitch) if mod is not None else (None, 0)
    fo = ctypes.c_void_p(flags_out.data_ptr()) if flags_out is not None else None
    fi = ctypes.c_void_p(flags_in.data_ptr()) if flags_in is not None else None
    _lib.check(_lib.load().hd_hollow_mean_detect_tiles(src_f32.ptr, src_f32.pitch, pp, ppitch, mask.ptr, mask.dtype,
                                                       mask.pitch, mp, mpitch, src_f32.ny, src_f32.nx, int(window_size),
                                                       BLANKS_INNER, BLANKS_FACTOR, fo, fi, dev.stream_ptr()),
               window_size=window_size, shape=src_f32.shape)
    return mask, mod


class BlanksFourier(Filter):
    """Peak detector on a spectrum quarter (custom_filters.py:369-427): returns the TUPLE
    (mask float64, image * (1 - mask))."""

    def __init__(self, *, window_size):
        self.window_size = window_size

    def run_device(self, raster):
        check_window(raster.shape, self.window_size)
        return _hollow_pass(as_f32(raster), None, self.window_size)

    def apply(self, image_to_filter):
        if not isinstance(image_to_filter, np.ndarray):
            raise NumpyArrayExpectedError(image_to_filter)
        check_window(image_to_filter.shape, self.window_size)
        mask, mod = self.run_device(dev.upload(image_to_filter))
        return dev.download(mask), dev.download(mod)


class DetectBlanksFourier(WindowFilter):
    """Two BlanksFourier(55) passes, masks added (custom_filters.py:430-462)."""

    window_size = BLANKS_WINDOW

    def run_device(self, raster):
        check_window(raster.shape, BLANKS_WINDOW)
        import os
        import torch
        src = as_f32(raster)
        flags = None
        if os.environ.get("HD_HOLLOW_DENSE") != "1":               # (tests compare with the dense second pass)
            n = int(_lib.load().hd_hollow_tile_count(src.ny, src.nx))
            flags = torch.empty(n, dtype=torch.uint8, device=dev.device())
        mask, mod = _hollow_pass(src, None, BLANKS_WINDOW, flags_out=flags)
        mask, _ = _hollow_pass(mod, mask, BLANKS_WINDOW, last=True, flags_in=flags)
        return mask


class MaskFourier(ComposedFilter):
    """DetectBlanksFourier -> IsolatedPoints(3) -> ExpandFilter(13) (custom_filters.py:537-561)."""

    def __init__(self):
        super().__init__()
        self.filters = [DetectBlanksFourier(), IsolatedPoints(window_size=3), ExpandFilter(window_size=13)]

    def run_device(self, raster):
        mask = self.filters[0].run_device(raster)
        mask = self.filters[1].run_device(dev.convert(mask, _lib.F32))
        return self.filters[2].run_device(mask)

    def apply(self, image_to_filter):
        Filter.apply(self, image_to_filter)
        check_window(image_to_filter.shape, BLANKS_WINDOW)
        return dev.download(self.run_device(dev.upload(image_to_filter)))


class FourierInitial(ComposedFilterResults):
    """fft2 -> fftshift -> abs, keeping the shifted spectrum (custom_filters.py:834-877).
    One fused launch group: the shift and |.| are folded into the transform's last pass."""

    def __init__(self):
        super().__init__()
        self.filters = [FourierTransform(), FourierShift(), AbsoluteValues()]
        self._fshift_dev = None

    @property
    def fourier_shift(self):
        return self.results["FourierShift"] if "FourierShift" in self.results else None

    @fourier_shift.setter
    def fourier_shift(self, value):
        self.results["FourierShift"] = value

    def run_device(self, raster):
        lib = _lib.load()
        ref = np.dtype(raster.ref_dtype)
        src = as_f32(raster)
        cref = np.complex64 if ref == np.float32 else np.complex128
        fshift = dev.empty(raster.ny, raster.nx, _lib.C64, cref)
        fabs = dev.empty(raster.ny, raster.nx, _lib.F32, np.float32 if ref == np.float32 else np.float64)
        plan = dev.fft_plan(raster.ny, raster.nx)
        nbytes = lib.hd_fft2_workspace_bytes(raster.ny, raster.nx)
        work = dev.scratch(nbytes)
        _lib.check(lib.hd_fft2_forward_shift_abs(plan, src.ptr, src.pitch, fshift.ptr, fshift.pitch, fabs.ptr, fabs.pitch,
                                                 ctypes.c_void_p(work.data_ptr()), nbytes, dev.stream_ptr()))
        self._fshift_dev = fshift
        self.results["FourierShift"] = fshift
        self.results["AbsoluteValues"] = fabs
        return fabs

    def apply(self, image_to_filter):
        Filter.apply(self, image_to_filter)
        return dev.download(self.run_device(dev.upload(image_to_filter)))


class FourierProcessQuarters(Filter):
    """Quarter extraction, MaskFourier per quarter and point-symmetric mask assembly
    (custom_filters.py:880-1050).  ``apply`` ignores its argument like the reference."""

    def __init__(self, fft_transform_abs):
        self.fft_transform_abs = fft_transform_abs
        shape = fft_transform_abs.shape
        self._ny, self._nx = shape
        self._mid_y, self._y_odd = divmod(self._ny, 2)
        self._mid_x, self._x_odd = divmod(self._nx, 2)
        self.pair_mid = self._mid_y, self._mid_x
        self._margin = FOURIER_MARGIN

    def run_device(self, fabs=None, invert=False, out_dtype=None, mask_fn=None):
        """``mask_fn(quarter) -> U8 mask``: MaskFourier by default; the row-band sharded chain passes a version that
        computes each rank's rows of the quarter only (hydrodem_b200/sharding.py)."""
        fabs = fabs if fabs is not None else self.fft_transform_abs
        if isinstance(fabs, np.ndarray):
            fabs = dev.upload(fabs)
        fabs = as_f32(fabs)
        m = self._margin
        qh, qw = self._mid_y - m, self._mid_x - m
        if qh < 1 or qw < 1:
            raise WindowSizeHighError(BLANKS_WINDOW, (qh, qw))
        check_window((qh, qw), BLANKS_WINDOW)
        q1 = fabs.sub(0, qh, 0, qw)                                          # [:my-m, :mx-m]          (:942-943)
        x0 = self._mid_x + m + self._x_odd
        q2 = dev.empty(qh, qw, _lib.F32)                                     # [:my-m, mx+m+x_odd:nx]  (:945-947)
        dev.elementwise(_lib.OP_COPY, fabs.sub(0, qh, x0, self._nx), None, q2)
        mask_fn = mask_fn or MaskFourier().run_device
        m1 = mask_fn(q1)
        m2 = mask_fn(q2)
        out_dtype = _lib.U8 if out_dtype is None else out_dtype
        out = dev.empty(self._ny, self._nx, out_dtype, np.float64)
        _lib.check(_lib.load().hd_fourier_mask_assemble(m1.ptr, m1.pitch, m2.ptr, m2.pitch, out.ptr, out.dtype, out.pitch,
                                                        self._ny, self._nx, m, int(invert), dev.stream_ptr()))
        return out

    def apply(self, image_to_filter=None):
        return dev.download(self.run_device())


class DetectApplyFourier(ComposedFilter):
    """The whole stripe-removal stage (custom_filters.py:1053-1101): FourierInitial ->
    FourierProcessQuarters -> (1 - mask) * F_shift -> ifftshift -> ifft2 -> abs.  float64 result."""

    def __init__(self):
        super().__init__()
        self.initial = FourierInitial()
        self._fabs_dev = None
        self._mask_dev = None

    @property
    def fft_transform_abs(self):
        return dev.download(self._fabs_dev) if self._fabs_dev is not None else None

    @property
    def mask(self):
        """The assembled blanking mask (float64 0/1), for inspection and the parity tests."""
        return dev.download(self._mask_dev) if self._mask_dev is not None else None

    def run_device(self, raster, out_dtype=None):
        lib = _lib.load()
        fabs = self.initial.run_device(raster)
        fshift = self.initial._fshift_dev
        self._fabs_dev = fabs
        quarters = FourierProcessQuarters(fabs)
        mask = quarters.run_device(fabs)
        self._mask_dev = mask
        self.filters = [quarters, SubtractionFilter(minuend=1), ProductFilter(factor=fshift), FourierIShift(),
                        FourierITransform(), AbsoluteValues()]
        out = dev.empty(raster.ny, raster.nx, _lib.F32 if out_dtype is None else out_dtype, np.float64)
        plan = dev.fft_plan(raster.ny, raster.nx)
        nbytes = lib.hd_fft2_workspace_bytes(raster.ny, raster.nx)
        work = dev.scratch(nbytes)
        _lib.check(lib.hd_fft2_masked_inverse_abs(plan, fshift.ptr, fshift.pitch, mask.ptr, mask.pitch, out.ptr, out.dtype,
                                                  out.pitch, ctypes.c_void_p(work.data_ptr()), nbytes, dev.stream_ptr()))
        return out

    def apply(self, image_to_filter):
        Filter.apply(self, image_to_filter)
        return dev.download(self.run_device(dev.upload(image_to_filter)))

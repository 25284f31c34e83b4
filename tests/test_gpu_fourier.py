"""GPU parity of the Fourier stripe-removal stage and the quadratic / groves stage (tolerance class:
<= 1e-5 relative, written next to each check) plus the exact mask logic."""
import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200.filters import custom_filters as cf
    from hydrodem_b200.filters import extension_filters as ef
    from hydrodem_b200.synth import SynthScene
    from oracle import stencils, fourier

RTOL = 1e-5


def spectrum_close(got, want):
    """Spectral values: error measured against the RMS magnitude (single bins can be arbitrarily small)."""
    scale = np.sqrt(np.mean(np.abs(want).astype(np.float64) ** 2))
    err = np.abs(got.astype(np.complex128) - want.astype(np.complex128))
    # 1e-5 of the RMS magnitude plus 4 float32 ulps of the largest bin: the DC bin (~N * mean elevation) sets
    # the rounding floor of ANY single-precision transform, the reference's scipy.fftpack complex64 one included
    tol = RTOL * scale + 4 * np.finfo(np.float32).eps * np.abs(want).max()
    assert (err <= tol).all(), (float(err.max()), float(scale))


def test_quadratic_and_groves_fixtures():
    g = load_golden("run_stencils")
    q32 = cf.QuadraticFilter(window_size=15).apply(g["srtm"])
    assert q32.dtype == np.float32
    np.testing.assert_allclose(q32, g["quad32"], rtol=RTOL)
    q64 = cf.QuadraticFilter(window_size=15).apply(g["srtm64"])
    assert q64.dtype == np.float64
    np.testing.assert_allclose(q64, g["quad64"], rtol=RTOL)
    np.testing.assert_array_equal(q64[:7], g["srtm64"][:7])               # border untouched, exact float64
    np.testing.assert_array_equal(q64[:, -7:], g["srtm64"][:, -7:])
    g1 = cf.GrovesCorrection(g["groves_closed"]).apply(g["srtm64"])
    assert g1.dtype == np.float64
    np.testing.assert_allclose(g1, g["groves1"], rtol=RTOL)
    g3 = cf.GrovesCorrectionsIter(g["groves_closed"], iterations=3).apply(g["srtm64"])
    np.testing.assert_allclose(g3, g["groves3"], rtol=RTOL)
    assert np.abs(g["groves3"] - g["srtm64"]).max() > 1.0                 # the correction did something


@pytest.mark.parametrize("ws", [3, 5, 9, 15])
def test_quadratic_sizes_vs_oracle(ws):
    a = SynthScene(90, 301, 31).srtm()
    np.testing.assert_allclose(cf.QuadraticFilter(window_size=ws).apply(a), stencils.quadratic(a, ws), rtol=RTOL)


def test_blanks_and_mask_fixtures():
    g = load_golden("run_fourier")
    mask, mod = cf.BlanksFourier(window_size=55).apply(g["q1"])
    assert mask.dtype == np.float64 and mod.dtype == np.float64
    assert int((mask != g["blanks_mask"]).sum()) == 0                     # mask mismatches: expected 0
    np.testing.assert_array_equal(mod, g["blanks_mod"])
    np.testing.assert_array_equal(cf.DetectBlanksFourier().apply(g["q1"]), g["detect"])
    np.testing.assert_array_equal(cf.MaskFourier().apply(g["q1"]), g["mask_q1"])
    np.testing.assert_array_equal(cf.MaskFourier().apply(g["q2"]), g["mask_q2"])
    full = cf.FourierProcessQuarters(g["fabs"]).apply(None)
    assert full.dtype == np.float64
    np.testing.assert_array_equal(full, g["mask"])


def test_g4_clean_spectrum():
    g = load_golden("ref_mask_fourier")
    mask, _ = cf.BlanksFourier(window_size=55).apply(g["filtered_blank_expected_2"])
    assert mask.sum() == 0


@pytest.mark.parametrize("shape", [(131, 140), (140, 131), (131, 133), (134, 136)])
def test_mask_assembly_geometry(shape):
    """Odd / even sizes of FourierProcessQuarters' bookkeeping, against reference-generated layouts."""
    from hydrodem_b200 import _lib, device as dev
    g = load_golden("run_fourier")
    ny, nx = shape
    fake = g[f"geo_{ny}_{nx}_fake"]
    qa, qb = fourier.first_quarters(fake)
    m1 = dev.upload(np.ascontiguousarray(qa > 0.9))
    m2 = dev.upload(np.ascontiguousarray(qb > 0.8))
    out = dev.empty(ny, nx, _lib.F64)
    _lib.check(_lib.load().hd_fourier_mask_assemble(m1.ptr, m1.pitch, m2.ptr, m2.pitch, out.ptr, out.dtype, out.pitch, ny,
                                                    nx, 10, 0, dev.stream_ptr()))
    np.testing.assert_array_equal(dev.download(out), g[f"geo_{ny}_{nx}_full"])


def test_fft_forward_fixture():
    g = load_golden("run_fourier")
    init = cf.FourierInitial()
    fabs = init.apply(g["srtm"])
    assert fabs.dtype == np.float32 and init.fourier_shift.dtype == np.complex64
    spectrum_close(init.fourier_shift, g["fshift"])
    spectrum_close(fabs, g["fabs"])


def test_detect_apply_fourier_fixture():
    g = load_golden("run_fourier")
    daf = cf.DetectApplyFourier()
    out = daf.apply(g["srtm"])
    assert out.dtype == np.float64
    mism = int((daf.mask != g["mask"]).sum())
    assert mism == 0, f"{mism} mask cells differ from the reference"
    np.testing.assert_allclose(out, g["corrected"], rtol=RTOL)           # spatial domain: elementwise relative


@pytest.mark.parametrize("shape", [(64, 128), (150, 170), (131, 133), (256, 200), (519, 508)])
def test_fft_wrappers_vs_scipy(shape):
    from scipy import fftpack
    rng = np.random.default_rng(shape[0])
    a = (rng.normal(100, 10, shape)).astype(np.float32)
    f = ef.FourierTransform().apply(a)
    assert f.dtype == np.complex64
    want = fftpack.fft2(a)
    spectrum_close(f, want)
    back = ef.FourierITransform().apply(want)
    assert back.dtype == np.complex64
    np.testing.assert_allclose(back.real, a, rtol=RTOL)
    np.testing.assert_array_equal(ef.FourierShift().apply(want), fftpack.fftshift(want))
    np.testing.assert_array_equal(ef.FourierIShift().apply(want), fftpack.ifftshift(want))
    np.testing.assert_array_equal(ef.FourierShift().apply(a), fftpack.fftshift(a))


def test_fft_vs_cufft():
    """The hand-written transform against cuFFT (torch.fft) on the device."""
    a = torch.randn(300, 421, device="cuda", dtype=torch.float32) * 10 + 50
    want = torch.fft.fft2(a).cpu().numpy()
    got = ef.FourierTransform().apply(a.cpu().numpy())
    spectrum_close(got, want)


def test_stripe_removal_bundled_tile():
    """C1 tile (519 x 508, srtm_corrected.tif): GPU stage against the oracle run side by side.  On real SRTM a few
    spectral bins sit exactly on the detector's threshold (centre > 4 x hollow mean, float32): the mismatch count is
    reported and bounded, and the VALUES are compared in any case -- against the oracle's inverse transform applied to
    the mask the GPU found, so a borderline bin cannot hide an error elsewhere."""
    g = load_golden("ref_tiles")
    a = g["srtm_corrected"]
    want, mask, fabs = fourier.detect_apply_fourier(a)
    daf = cf.DetectApplyFourier()
    got = daf.apply(a)
    mism = int((daf.mask != mask).sum())
    print("bundled tile: mask cells that differ from the oracle:", mism)
    assert mism <= 4, f"{mism} mask cells differ"
    _, fshift = fourier.fourier_initial(a)
    np.testing.assert_allclose(got, fourier.apply_mask(daf.mask, fshift), rtol=RTOL)
    if mism == 0:
        np.testing.assert_allclose(got, want, rtol=RTOL)


def test_fft_size_limit_fails_loudly():
    """Rows above 8192 need a small factor (n = n1 * n2, n1 <= 16, n2 <= 8192): a large prime has none."""
    from hydrodem_b200.exceptions import DeviceError
    with pytest.raises(DeviceError):
        ef.FourierTransform().apply(np.zeros((16, 10007), dtype=np.float32))


@pytest.mark.parametrize("shape", [(40, 9000), (10801, 48), (33, 16384), (18000, 20), (150, 36000), (5, 32776), (28679, 3),
                                   (4, 49152), (20000, 6), (9, 7201), (7201, 9)])
def test_fft_long_rows_vs_scipy(shape):
    """Rows longer than one shared-memory transform: n = n1 * n2 split (9000 = 2 * 4500, 10801 = 7 * 1543,
    18000 = 3 * 6000, 36000 = 5 * 7200) and the 16384 power of two."""
    from scipy import fftpack
    rng = np.random.default_rng(shape[0])
    a = (rng.normal(100, 10, shape)).astype(np.float32)
    f = ef.FourierTransform().apply(a)
    want = fftpack.fft2(a)
    spectrum_close(f, want)
    back = ef.FourierITransform().apply(want)
    np.testing.assert_allclose(back.real, a, rtol=RTOL)


@pytest.mark.parametrize("n,radices", [(120, "2,3,4,5"), (432, "6,8,9"), (1800, "10,12,15"), (240, "16,15"), (7200, None),
                                       (6000, None), (3600, None), (4500, "9,10,10,5:31"), (3000, "5,10,10,6")])
def test_fft_mixed_radix_vs_scipy(n, radices, monkeypatch):
    """Lengths 2^a 3^b 5^c run as plain mixed-radix transforms (no Bluestein): every generated butterfly
    (tools/gen_fft_radix.py) and the planner's own choice for the mosaic sub-row lengths, against scipy."""
    from scipy import fftpack
    if radices:
        monkeypatch.setenv("HD_FFT_RADICES", radices)
    rows = 7 if radices else 5                      # (plans are cached per shape: each case has its own)
    rng = np.random.default_rng(n)
    a = (rng.normal(100, 10, (rows, n))).astype(np.float32)
    f = ef.FourierTransform().apply(a)
    want = fftpack.fft2(a)
    spectrum_close(f, want)
    back = ef.FourierITransform().apply(want)
    np.testing.assert_allclose(back.real, a, rtol=RTOL)


def test_stripe_removal_long_rows():
    """The fused forward / masked inverse passes on a raster whose rows need the n1 * n2 split."""
    sc = SynthScene(200, 9000, 17)
    a = sc.srtm()
    want, mask, _ = fourier.detect_apply_fourier(a)
    daf = cf.DetectApplyFourier()
    got = daf.apply(a)
    assert int((daf.mask != mask).sum()) == 0
    np.testing.assert_allclose(got, want, rtol=RTOL)


@pytest.mark.parametrize("shape", [(301, 333), (259, 10801), (333, 300), (131, 7201), (2025, 135), (10125, 131), (301, 256)])
def test_stripe_removal_odd_sizes_hermitian_path(shape, monkeypatch):
    """Odd x odd rasters take the Hermitian (real-output) inverse: half of the rows in the first pass, two output
    columns per transform in the second.  Must agree with the oracle, and with the plain complex path."""
    sc = SynthScene(*shape, 23)
    a = sc.srtm()
    want, mask, _ = fourier.detect_apply_fourier(a)
    daf = cf.DetectApplyFourier()
    got = daf.apply(a)
    assert int((daf.mask != mask).sum()) == 0
    np.testing.assert_allclose(got, want, rtol=RTOL)
    monkeypatch.setenv("HD_FFT_NO_HERMITIAN", "1")
    plain = cf.DetectApplyFourier().apply(a)
    np.testing.assert_allclose(got, plain, rtol=1e-6)



def test_c3_fourier_isotropic_median_at_10801():
    """BASELINE.json configs[2]: Fourier stripe removal + the isotropic (quadratic) filter + the median filter on a
    synthetic 10801 x 10801 tile.  The Fourier stage is compared on the WHOLE tile against scipy / the oracle (the
    rounding floor of a single-precision transform grows with N: this is where a complex64 inverse would show); the
    two window filters run on the whole tile on the GPU and are compared on a 700-row strip (windows are local; the
    oracle's per-cell cost is the same everywhere)."""
    import time
    from hydrodem_b200 import device as dev
    from hydrodem_b200.filters import new_filters as nf
    from hydrodem_b200.synth import DeviceMosaic
    n = 10801
    srtm_t, _, _ = DeviceMosaic(n, n, 1003).band(0, n)
    a = srtm_t.cpu().numpy()
    del srtm_t
    t0 = time.time()
    want, mask, _ = fourier.detect_apply_fourier(a)
    t_cpu = time.time() - t0
    daf = cf.DetectApplyFourier()
    d_in = dev.upload(a)
    d_out = daf.run_device(d_in)
    got = dev.download(d_out)
    mism = int((daf.mask != mask).sum())
    print(f"C3: oracle Fourier stage {t_cpu:.1f} s; mask cells that differ: {mism}; blanked bins: {int(mask.sum())}")
    assert mism == 0 and mask.sum() > 0
    np.testing.assert_allclose(got, want, rtol=RTOL)
    # isotropic + median on the stripe-free DEM, strip rows [r0, r1) (oracle fed with the halo it needs)
    r0, r1, h = 5000, 5700, 7
    smooth = dev.download(cf.QuadraticFilter(window_size=15).run_device(d_out))
    med = dev.download(nf.MedianFilter(window_size=5).run_device(d_out))
    strip = got[r0 - h:r1 + h]
    np.testing.assert_allclose(smooth[r0:r1], stencils.quadratic(strip, 15)[h:-h], rtol=RTOL)
    from oracle import clib
    np.testing.assert_array_equal(med[r0:r1], clib.median(strip, 5)[h:-h])


def test_int16_input_stripe_removal():
    """SRTM arrives as int16 (image_srtm.py:125-126): scipy.fftpack promotes it to float64 / complex128, the device path
    widens it to float32 (exact) and stays in single precision -- inside the stage's 1e-5 tolerance."""
    g = load_golden("run_int16")
    a = g["srtm_i16"]
    assert a.dtype == np.int16
    got = cf.DetectApplyFourier().apply(a)
    assert got.dtype == np.float64
    np.testing.assert_allclose(got, g["daf_i16"], rtol=RTOL)


def test_groves_partial_results_are_materialised_lazily():
    """GrovesCorrection.partial_results (custom_filters.py:728): the five intermediates, reference dtypes; computed by
    separate kernels only when read (the fused kernel never writes them)."""
    g = load_golden("run_stencils")
    dem, groves = g["srtm64"], g["groves_closed"]
    gc = cf.GrovesCorrection(groves)
    out = gc.apply(dem)
    assert gc._partials == [] and len(gc._partials_pending) == 1            # nothing computed yet
    pr = gc.partial_results
    assert len(pr) == 5 and gc.partial_results is pr
    smooth = stencils.quadratic(dem, 15)
    np.testing.assert_allclose(pr[0], smooth, rtol=RTOL)
    np.testing.assert_allclose(pr[1], dem - smooth, rtol=1e-3, atol=1e-4)
    assert pr[2].dtype == np.int64 and set(np.unique(pr[2])) <= {0, 1}
    np.testing.assert_array_equal(pr[3], groves * pr[2])
    np.testing.assert_array_equal(pr[4], 1 - pr[3])
    np.testing.assert_allclose(out, pr[4] * pr[1] + pr[0], rtol=RTOL)        # (:729-731)


def test_second_blanks_pass_only_near_first_hits(monkeypatch):
    """DetectBlanksFourier's second pass is restricted to the tiles whose 3 x 3 tile neighbourhood had a hit in the first
    (new hits can only appear within 27 cells of an old one): same mask as two dense passes, on a spectrum with isolated
    and clustered peaks, hits on tile corners and on the quarter's edges."""
    rng = np.random.default_rng(11)
    q = (rng.random((700, 833)).astype(np.float32) + 0.5) * 100
    for (y, x) in ((0, 0), (63, 63), (64, 64), (127, 500), (128, 501), (350, 400), (351, 430), (699, 832), (300, 0)):
        q[y, x] = 5000.0
    q[200:203, 600:603] = 900.0                                   # a cluster: second-pass hits next to first-pass hits
    q[201, 601] = 20000.0
    sparse = cf.DetectBlanksFourier().apply(q)
    monkeypatch.setenv("HD_HOLLOW_DENSE", "1")
    dense = cf.DetectBlanksFourier().apply(q)
    np.testing.assert_array_equal(sparse, dense)
    assert dense.sum() >= 10 and dense.max() >= 1
    want = stencils.detect_blanks_fourier(q)
    np.testing.assert_array_equal(sparse, want)

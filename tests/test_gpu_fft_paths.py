"""GPU: every path of the 1-D FFT against numpy's float64 FFT of the float32 / complex64 values the device read.

The planner (build1d in csrc/fft.cu) sends a row length to one of three algorithms -- radix-2^k, mixed radix
(2^a 3^b 5^c) or Bluestein (shared-memory transform of m = 16 ... 16384) -- and a length above 8192 to a thread-block
cluster of n1 = 2 ... 8 CTAs.  Each row pass then reads its input in one of four ways (real row pairs, complex rows,
(1 - mask) x the shifted spectrum, Hermitian row pairs).  The lengths below are chosen so that every combination runs;
each one asserts the plan it gets (hd_fft_plan_info), so a planner change that moves a length onto another path fails
here instead of silently dropping coverage.

Tolerance (DESIGN.md section 6), applied to every row on its own: max |dX| <= 1e-5 rms|X| + 4 eps32 max|X|.  The
normwise error |dX|_2 / |X|_2 of every row is also bounded by 3e-6, and the worst value per (algorithm, n1, load mode)
is printed by test_worst_normwise_errors."""
import contextlib
import ctypes

import numpy as np
import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

if torch.cuda.is_available():
    from hydrodem_b200 import _lib, device as dev
    from hydrodem_b200.filters import extension_filters as ef

POW2, BLUE, MIXED = 0, 1, 2
ALGO = {POW2: "radix-2^k", BLUE: "Bluestein", MIXED: "mixed"}
LOAD_REAL, LOAD_C64, LOAD_MASKED_SHIFTED, LOAD_C64_HPAIR = range(4)
LOAD = {LOAD_REAL: "real", LOAD_C64: "c64", LOAD_MASKED_SHIFTED: "masked", LOAD_C64_HPAIR: "hpair"}
EPS32 = float(np.finfo(np.float32).eps)
NORMWISE_BOUND = 3e-6

# length -> (n1, n, algorithm, m): n1 CTAs per row, inner length n = length / n1, shared-memory transform length m
PATHS = {
    # one transform per row
    4096: (1, 4096, POW2, 4096), 8192: (1, 8192, POW2, 8192), 16384: (1, 16384, POW2, 16384),
    243: (1, 243, MIXED, 243), 625: (1, 625, MIXED, 625), 2025: (1, 2025, MIXED, 2025), 6075: (1, 6075, MIXED, 6075),
    7: (1, 7, BLUE, 16), 11: (1, 11, BLUE, 32), 13: (1, 13, BLUE, 32), 14: (1, 14, BLUE, 32), 17: (1, 17, BLUE, 64),
    65: (1, 65, BLUE, 256), 3601: (1, 3601, BLUE, 8192),
    4097: (1, 4097, BLUE, 16384), 4801: (1, 4801, BLUE, 16384), 7201: (1, 7201, BLUE, 16384),
    8191: (1, 8191, BLUE, 16384),
    # long rows: a cluster of n1 CTAs
    8748: (2, 4374, MIXED, 4374), 8194: (2, 4097, BLUE, 16384),
    24576: (3, 8192, POW2, 8192), 10125: (3, 3375, MIXED, 3375), 8193: (3, 2731, BLUE, 8192),
    12291: (3, 4097, BLUE, 16384),
    32768: (4, 8192, POW2, 8192), 20000: (4, 5000, MIXED, 5000), 16388: (4, 4097, BLUE, 16384),
    40960: (5, 8192, POW2, 8192), 15625: (5, 3125, MIXED, 3125), 8195: (5, 1639, BLUE, 4096),
    20485: (5, 4097, BLUE, 16384),
    49152: (6, 8192, POW2, 8192), 34992: (6, 5832, MIXED, 5832), 24582: (6, 4097, BLUE, 16384),
    57344: (7, 8192, POW2, 8192), 42525: (7, 6075, MIXED, 6075), 8197: (7, 1171, BLUE, 4096),
    10801: (7, 1543, BLUE, 4096), 28679: (7, 4097, BLUE, 16384), 36001: (7, 5143, BLUE, 16384),
    65536: (8, 8192, POW2, 8192), 50000: (8, 6250, MIXED, 6250), 32776: (8, 4097, BLUE, 16384),
}


def _short_path(n):
    """The planner's rule for a length that fits one transform: powers of two as they are, 3/5-smooth lengths mixed
    radix, the rest Bluestein on the next power of two >= 2n - 1."""
    if n & (n - 1) == 0:
        return (1, n, POW2, n)
    r = n
    for p in (2, 3, 5):
        while r % p == 0:
            r //= p
    if r == 1:
        return (1, n, MIXED, n)
    return (1, n, BLUE, 1 << (2 * n - 2).bit_length())


for _n in range(1, 257):
    PATHS.setdefault(_n, _short_path(_n))

# one length per (algorithm, short / long) runs with more rows than the persistent grid holds, so that every CTA or
# cluster loops over rows
LOOPING = {16384, 625, 4801, 24576, 10125, 36001}

WORST = {}        # (algorithm, n1, load mode) -> worst normwise error seen by this run


@contextlib.contextmanager
def plan_1d(n):
    """A plan of a 1 x n raster, created for this test only (no cache, so HD_FFT_* settings of the test apply)."""
    lib = _lib.load()
    handle = ctypes.c_void_p()
    _lib.check(lib.hd_fft2_plan_create(1, n, ctypes.byref(handle)))
    try:
        yield handle
    finally:
        torch.cuda.synchronize()
        _lib.check(lib.hd_fft2_plan_destroy(handle))


def plan_info(plan, axis=0):
    """(n_total, n1, n, m, algorithm, k of the last radix-2^k pass)"""
    info = (ctypes.c_int64 * 6)()
    _lib.check(_lib.load().hd_fft_plan_info(plan, axis, info))
    return tuple(int(v) for v in info)


def _host(raster):
    torch.cuda.synchronize()
    return np.ascontiguousarray(raster.tensor().cpu().numpy())


def _empty_nan(ny, nx, dtype):
    out = dev.empty(ny, nx, dtype)
    out.buf.view(torch.float32).fill_(float("nan"))
    return out


def band_pass(plan, n, load, src, nrows, inverse=0, real_out=0, keep=0, mask=None, shift=0):
    """hd_fft_band_pass along axis 0; returns the (n x nrows) transposed result, NaN where nothing was written."""
    lib = _lib.load()
    out = _empty_nan(n, nrows, _lib.F32 if real_out else _lib.C64)
    nbytes = lib.hd_fft_band_workspace_bytes(nrows, n)
    work = dev.scratch(nbytes)
    _lib.check(lib.hd_fft_band_pass(plan, 0, load, src.ptr, src.pitch, nrows, mask.ptr if mask is not None else None,
                                    mask.pitch if mask is not None else 0, shift, inverse, real_out, out.ptr, out.pitch,
                                    keep, ctypes.c_void_p(work.data_ptr()), nbytes, dev.stream_ptr()))
    return _host(out)


def fft_rows(plan, n, src, nrows, inverse, transpose_out):
    """hd_fft_rows; returns the (nrows x n) result whichever layout the device wrote."""
    lib = _lib.load()
    out = _empty_nan(n, nrows, _lib.C64) if transpose_out else _empty_nan(nrows, n, _lib.C64)
    nbytes = lib.hd_fft2_workspace_bytes(nrows, n)
    work = dev.scratch(nbytes)
    _lib.check(lib.hd_fft_rows(plan, src.ptr, src.dtype, src.pitch, out.ptr, out.pitch, nrows, inverse, transpose_out,
                               ctypes.c_void_p(work.data_ptr()), nbytes, dev.stream_ptr()))
    got = _host(out)
    return got.T if transpose_out else got


def check_rows(got, want, what):
    """DESIGN.md section 6 per row; returns the worst normwise error of the rows."""
    got = got.astype(np.complex128)
    want = want.astype(np.complex128)
    err = np.abs(got - want)
    mag = np.abs(want)
    tol = 1e-5 * np.sqrt(np.mean(mag ** 2, axis=1)) + 4 * EPS32 * mag.max(axis=1)
    worst = err.max(axis=1)
    bad = np.flatnonzero(~(worst <= tol))                   # NaN fails
    assert bad.size == 0, (f"{what}: {bad.size} of {len(want)} rows out of tolerance, first rows {bad[:6].tolist()}: "
                           f"max |dX| {worst[bad[:6]].tolist()} > {tol[bad[:6]].tolist()}")
    norm_x = np.linalg.norm(want, axis=1)
    norm_e = np.linalg.norm(err, axis=1)
    rel = np.divide(norm_e, norm_x, out=np.zeros_like(norm_e), where=norm_x > 0)
    return float(rel.max())


def impulse_positions(n_total, n1, n):
    """0, N - 1, N / 2, and both sides of the long-row seams: the cluster ranks' column chunks r ceil(n / n1) and the
    n1-point DFT's segments a n."""
    pos = {0, n_total - 1, n_total // 2}
    chunk = -(-n // n1)
    for r in range(1, n1):
        pos |= {r * chunk - 1, r * chunk, r * chunk + 1, r * n - 1, r * n, r * n + 1}
    return sorted(p for p in pos if 0 <= p < n_total)


def make_rows(n_total, n1, n, nrows_min, rng, cplx):
    """Rows of length n_total: unit impulses (|X_k| = 1 in every bin, so a misplaced bin is an O(1) error), white noise,
    DEM-like rows (1000 + noise: DC dominates), single tones, and one more noise row at the end.  Rows of one kind come
    in pairs (two real rows share a transform, and a pair's rounding error scales with the larger of the two); the row
    count is odd, so the last row has no partner."""
    def noise(k):
        x = rng.standard_normal((k, n_total))
        return x + 1j * rng.standard_normal((k, n_total)) if cplx else x

    imp = impulse_positions(n_total, n1, n)
    if len(imp) % 2:
        imp.append(min(1, n_total - 1))
    rows = np.zeros((len(imp), n_total), dtype=np.complex128 if cplx else np.float64)
    rows[np.arange(len(imp)), imp] = 1.0
    n_noise = max(2, nrows_min - len(imp) - 5)
    n_noise += n_noise % 2
    t = np.arange(n_total)
    f = (n_total // 3 + 1) % n_total
    tone = np.exp(2j * np.pi * f * t / n_total + 0.3) if cplx else np.cos(2 * np.pi * f * t / n_total + 0.3)
    parts = [rows, noise(n_noise), 1000.0 + noise(2), np.stack([tone, 0.5 * tone]), noise(1)]
    return np.concatenate(parts).astype(np.complex64 if cplx else np.float32)


def hermitian_rows(real_rows):
    """complex64 spectra of real rows, made exactly Hermitian: X[N - k] = conj X[k], real X[0] (and X[N/2])."""
    n = real_rows.shape[1]
    h = np.fft.fft(real_rows.astype(np.float64), axis=1).astype(np.complex64)
    k = np.arange(1, (n + 1) // 2)
    h[:, n - k] = np.conj(h[:, k])
    h[:, 0] = h[:, 0].real
    if n % 2 == 0:
        h[:, n // 2] = h[:, n // 2].real
    return h


def looping_rows(info):
    """A row count for which every CTA (short rows, two rows per transform) or cluster (long rows) takes more than one
    row: more than the resident blocks an SM can hold with m complex64 of shared memory (228 KB per SM, at most 8 blocks
    of 256 threads), times the SMs."""
    _, n1, _, m, _, _ = info
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    per_sm = max(1, min(8, 228 * 1024 // ((m + 1) * 8)))
    return 2 * sms * per_sm + 1 if n1 == 1 else sms * per_sm // n1 + 1


@pytest.mark.parametrize("n_total", sorted(PATHS))
def test_fft_path_vs_float64(n_total):
    with plan_1d(n_total) as plan:
        info = plan_info(plan)
        assert info[0] == n_total
        assert (info[1], info[2], info[4], info[3]) == PATHS[n_total], f"plan {info}"
        _, n1, n, m, algo, _ = info
        nrows_min = looping_rows(info) if n_total in LOOPING else 0
        rng = np.random.default_rng(n_total)
        real = make_rows(n_total, n1, n, nrows_min, rng, cplx=False)
        cplx = make_rows(n_total, n1, n, nrows_min, rng, cplx=True)
        nrows = len(real)
        assert nrows % 2 == 1 and len(cplx) == nrows
        if n_total in LOOPING:
            assert nrows >= nrows_min
        d_real, d_cplx = dev.upload(real), dev.upload(cplx)
        r64, c64 = real.astype(np.complex128), cplx.astype(np.complex128)
        want = {(LOAD_REAL, 0): np.fft.fft(r64, axis=1), (LOAD_REAL, 1): np.fft.ifft(r64, axis=1),
                (LOAD_C64, 0): np.fft.fft(c64, axis=1), (LOAD_C64, 1): np.fft.ifft(c64, axis=1)}
        worst = {}

        def record(load, value):
            worst[load] = max(worst.get(load, 0.0), value)

        # real rows (two per transform on short rows): full and half spectrum, forward and inverse
        for inverse in (0, 1):
            for keep in sorted({n_total, n_total // 2 + 1}):
                got = band_pass(plan, n_total, LOAD_REAL, d_real, nrows, inverse=inverse, keep=keep)
                assert np.isnan(got[keep:]).all(), f"keep_cols={keep}: columns past the kept half were written"
                record(LOAD_REAL, check_rows(got[:keep].T, want[LOAD_REAL, inverse][:, :keep],
                                             f"band real inverse={inverse} keep={keep}"))
        # complex rows, forward and inverse, and |ifft| stored as float
        for inverse in (0, 1):
            got = band_pass(plan, n_total, LOAD_C64, d_cplx, nrows, inverse=inverse)
            record(LOAD_C64, check_rows(got.T, want[LOAD_C64, inverse], f"band c64 inverse={inverse}"))
        got = band_pass(plan, n_total, LOAD_C64, d_cplx, nrows, inverse=1, real_out=1)
        record(LOAD_C64, check_rows(got.T, np.abs(want[LOAD_C64, 1]), "band c64 |ifft|"))
        # (1 - mask) x the spectrum read with its columns shifted by N // 2, inverse
        mask = (rng.random((nrows, n_total)) < 0.5).astype(np.uint8)
        shift = n_total // 2
        got = band_pass(plan, n_total, LOAD_MASKED_SHIFTED, d_cplx, nrows, inverse=1, mask=dev.upload(mask), shift=shift)
        masked = np.roll(c64 * (1 - mask), -shift, axis=1)
        record(LOAD_MASKED_SHIFTED, check_rows(got.T, np.fft.ifft(masked, axis=1), "band masked inverse"))
        # two Hermitian rows per inverse transform, |re| and |im| stored as float
        herm = hermitian_rows(real)
        got = band_pass(plan, n_total, LOAD_C64_HPAIR, dev.upload(herm), nrows, inverse=1, real_out=1)
        record(LOAD_C64_HPAIR, check_rows(got.T, np.abs(np.fft.ifft(herm.astype(np.complex128), axis=1).real),
                                          "band hpair |ifft|"))
        # hd_fft_rows: rows written directly, or through the transposes (long rows: there and back)
        for load, src in ((LOAD_REAL, d_real), (LOAD_C64, d_cplx)):
            for inverse in (0, 1):
                for transpose_out in (0, 1):
                    got = fft_rows(plan, n_total, src, nrows, inverse, transpose_out)
                    record(load, check_rows(got, want[load, inverse],
                                            f"fft_rows {LOAD[load]} inverse={inverse} transpose_out={transpose_out}"))
    for load, value in worst.items():
        key = (ALGO[algo], n1, LOAD[load])
        WORST[key] = max(WORST.get(key, 0.0), value)
        assert value <= NORMWISE_BOUND, f"{key}: normwise error {value:.3g} at length {n_total}"


def test_planner_reaches_every_path():
    """The table reaches every (algorithm, n1) pair the planner can produce, Bluestein's 16384-point transform at every
    n1, and Bluestein's fused middle pass for k = 2, 3 and 4."""
    reached, blue_m16384, blue_k = set(), set(), set()
    for n_total, want in sorted(PATHS.items()):
        with plan_1d(n_total) as plan:
            info = plan_info(plan)
        assert info[0] == n_total and (info[1], info[2], info[4], info[3]) == want, (n_total, info)
        _, n1, _, m, algo, k_last = info
        reached.add((algo, n1))
        if algo == BLUE:
            blue_k.add(k_last)
            if m == 16384:
                blue_m16384.add(n1)
    # a power of two of 2 x 8192 is one 16384-point transform, so radix-2^k long rows start at n1 = 3
    want_pairs = {(POW2, n1) for n1 in (1, 3, 4, 5, 6, 7, 8)} | {(a, n1) for a in (MIXED, BLUE) for n1 in range(1, 9)}
    assert reached == want_pairs, sorted(want_pairs - reached)
    assert blue_m16384 == set(range(1, 9))
    assert blue_k == {2, 3, 4}


def test_fft_plan_info_arguments():
    lib = _lib.load()
    info = (ctypes.c_int64 * 6)()
    assert lib.hd_fft_plan_info(None, 0, info) == _lib.HD_ERR_NULL
    with plan_1d(3601) as plan:
        assert lib.hd_fft_plan_info(plan, 0, None) == _lib.HD_ERR_NULL
        assert lib.hd_fft_plan_info(plan, 2, info) == _lib.HD_ERR_ARG
        assert plan_info(plan, 1) == (1, 1, 1, 1, POW2, 0)           # the plan's column axis: length 1


@pytest.mark.parametrize("shape", [(1, 1), (1, 7), (7, 1), (2, 3), (3, 8193), (8193, 1)])
def test_fft2_wrappers_on_real_input(shape):
    """FourierTransform / FourierITransform (scipy.fftpack.fft2 / ifft2) of a float32 raster, the inverse included:
    its first pass runs the real-row pair split with the conjugate of the inverse."""
    from scipy import fftpack
    rng = np.random.default_rng(shape[0] * 10 + shape[1])
    a = (100 + 10 * rng.standard_normal(shape)).astype(np.float32)
    a64 = a.astype(np.float64)
    for filt, want in ((ef.FourierTransform(), fftpack.fft2(a64)), (ef.FourierITransform(), fftpack.ifft2(a64))):
        got = filt.apply(a)
        assert got.dtype == np.complex64 and got.shape == shape
        check_rows(got.reshape(1, -1), want.reshape(1, -1), type(filt).__name__)


def test_worst_normwise_errors():
    """Prints the worst normwise error of each (algorithm, n1, load mode) the sweep above met in this run."""
    if not WORST:
        pytest.skip("the length sweep did not run in this session")
    print("\nworst |dX|_2 / |X|_2 per row")
    print(f"{'algorithm':>10} {'n1':>3} {'load':>7} {'error':>10}")
    for (algo, n1, load), value in sorted(WORST.items()):
        print(f"{algo:>10} {n1:>3} {load:>7} {value:10.3e}")
    assert max(WORST.values()) <= NORMWISE_BOUND

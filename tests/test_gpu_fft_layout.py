"""GPU: the layout work of the 2-D Fourier stage (transposes, un-permuting of long rows, shifts, Hermitian mirrors) moves
values and never changes them -- the transposed row transforms are bitwise the row transforms, the mirrored half of the
shifted spectrum is bitwise the conjugate of the computed half, and the Fourier stage's outputs hash to the values
recorded before the transposes were rewritten as TMA pipelines."""
import ctypes
import hashlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200 import _lib, device as dev
    from hydrodem_b200.filters import custom_filters as cf


def _bits(a):
    """uint32 view of a float32 / complex64 array (bitwise comparisons: -0.0 != 0.0, NaN == NaN)."""
    return np.ascontiguousarray(a).view(np.uint32)


def _host(raster):
    torch.cuda.synchronize()
    return np.ascontiguousarray(raster.tensor().cpu().numpy())


def _sha(raster):
    return hashlib.sha256(_host(raster).tobytes()).hexdigest()


# partial tiles in both directions, long rows (18000 = 3 x 6000 mixed radix, stored digit-reversed; 10801 = 7 x 1543
# Bluestein), odd row lengths (scratch pitches padded for TMA)
@pytest.mark.parametrize("shape", [(37, 18000), (40, 10801), (1000, 1030), (4097, 33)])
@pytest.mark.parametrize("complex_in", [False, True])
def test_rows_transpose_out_is_the_transpose(shape, complex_in):
    nrows, nx = shape
    rng = np.random.default_rng(nrows * 7 + nx)
    a = rng.standard_normal((nrows, nx)).astype(np.float32)
    if complex_in:
        a = (a + 1j * rng.standard_normal((nrows, nx))).astype(np.complex64)
    lib = _lib.load()
    src = dev.upload(a)
    plan = dev.fft_plan(nrows, nx)
    nbytes = lib.hd_fft2_workspace_bytes(nrows, nx)
    work = dev.scratch(nbytes)
    rows_out = dev.empty(nrows, nx, _lib.C64)
    tr_out = dev.empty(nx, nrows, _lib.C64)
    for out, transpose_out in ((rows_out, 0), (tr_out, 1)):
        _lib.check(lib.hd_fft_rows(plan, src.ptr, src.dtype, src.pitch, out.ptr, out.pitch, nrows, 0, transpose_out,
                                   ctypes.c_void_p(work.data_ptr()), nbytes, dev.stream_ptr()))
    rows, tr = _host(rows_out), _host(tr_out)
    assert np.array_equal(_bits(rows.T), _bits(tr))
    want = np.fft.fft(a.astype(np.complex128), axis=1)                   # and it is the transform
    assert np.abs(rows - want).max() <= 1e-4 * np.sqrt(np.mean(np.abs(want) ** 2))


@pytest.mark.parametrize("shape", [(64, 100), (37, 41), (36, 45), (45, 36), (255, 18000)])
def test_fshift_mirror_half_is_exact_conjugate(shape):
    ny, nx = shape
    rng = np.random.default_rng(ny * 31 + nx)
    a = (100 + 10 * rng.standard_normal((ny, nx))).astype(np.float32)
    fi = cf.FourierInitial()
    fabs = fi.run_device(dev.upload(a))
    F = np.fft.ifftshift(_host(fi._fshift_dev))                          # F[ky][kx], unshifted
    A = np.fft.ifftshift(_host(fabs))
    nh = nx // 2 + 1
    ky = (-np.arange(ny)) % ny
    kx = np.arange(nh, nx)
    mirror = F[ky][:, nx - kx]
    assert np.array_equal(_bits(F[:, nh:]), _bits(np.conj(mirror)))
    assert np.array_equal(_bits(A[:, nh:]), _bits(A[ky][:, nx - kx]))
    np.testing.assert_allclose(F, np.fft.fft2(a.astype(np.float64)), rtol=0, atol=1e-4 * np.abs(F).max())


def digests(ny, nx):
    """SHA-256 of fshift, |F| and the DetectApplyFourier output (float32 and float64) for a seeded raster."""
    rng = np.random.default_rng(ny * 100003 + nx)
    a = (100 + 10 * rng.standard_normal((ny, nx))).astype(np.float32)
    src = dev.upload(a)
    daf = cf.DetectApplyFourier()
    out32 = daf.run_device(src)
    out = {"fshift": _sha(daf.initial._fshift_dev), "fabs": _sha(daf._fabs_dev), "detect_apply_f32": _sha(out32)}
    out["detect_apply_f64"] = _sha(cf.DetectApplyFourier().run_device(src, out_dtype=_lib.F64))
    return out


# recorded on a B200 (1000 W) with the library as it was before the transposes became TMA pipelines
RECORDED = {
    (512, 18000): {
        "fshift": "442e8740d08f18474f6b5790a204eb78ea66c443217dd46474199517dc00fab6",
        "fabs": "871e9e0ce4eb38fa3ac039b4a5827797debd41bbf598c43abf453cc53bc43d28",
        "detect_apply_f32": "abc61cd8c77dbc45fe26a3ff8dfe3433fead4e6f8022a1a29d5671ff61bd95f7",
        "detect_apply_f64": "f0ecfa862c6800f57db5ea583195972eeec33a82066a029508fab196d2025de4",
    },
    (3601, 3601): {
        "fshift": "0301b4e9cbd3a153f2c0cc15b60faa17cd544dc5c99fb5e210dc0372c0ed4153",
        "fabs": "721d604f1c26c84e08dd416e32fa2ca311c1b50ef92834cffd5c7811c9c4b8bd",
        "detect_apply_f32": "664bec01cc3ff9e6d212ee81f5963d380ab311fab8495899dc18f06ddfa411c6",
        "detect_apply_f64": "fce24c218bb437051a4e978ef3d5428c022f0cd2ba409f66e032e330a4de644f",
    },
    (1024, 1030): {
        "fshift": "fda817e1ea5831d7ab084b32c1dbfae32cafc61bbe70a24b017676ab98dcba41",
        "fabs": "4a9754ad13e71fc85716631685c06104b2f4bcbc2e8fbe3d6fe5cea79bc8cd99",
        "detect_apply_f32": "468cec92374f794700c72e6dc6bca76b8be98c3a7d6c601c71b7c73b79064f78",
        "detect_apply_f64": "5cb489e8ee5b7245e696780c10303ed0942175bb2b72edf7b0312955d262850f",
    },
}


@pytest.mark.parametrize("shape", sorted(RECORDED))
def test_fourier_outputs_unchanged(shape):
    assert digests(*shape) == RECORDED[shape]

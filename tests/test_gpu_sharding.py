"""GPU: row-band sharding emulated with ThreadComm (ranks = threads on one device).  Every banded result --
exact-class AND tolerance-class stages -- must equal the single-GPU result bit for bit (assert_array_equal)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200 import _lib, device as dev, sharding
    from hydrodem_b200.filters import custom_filters as cf, extension_filters as ef
    from hydrodem_b200.synth import SynthScene
    from oracle import hydrology


@pytest.mark.parametrize("world", [2, 3])
def test_banded_stencils_match_single_gpu(world):
    sc = SynthScene(301, 333, 51)
    hs, srtm = sc.hsheds(), sc.srtm()
    want_maj = cf.MajorityFilter(window_size=11).apply(hs)
    want_quad = cf.QuadraticFilter(window_size=15).apply(srtm)
    want_er = ef.BinaryErosion(iterations=2).apply(want_maj)

    def fn(comm):
        band = sharding.Band(comm, *hs.shape)
        maj = band.apply(cf.MajorityFilter(window_size=11), dev.upload(band.take(hs)), 5)
        quad = band.apply(cf.QuadraticFilter(window_size=15), dev.upload(band.take(srtm)), 7)
        er = band.apply(ef.BinaryErosion(iterations=2), maj, 2)
        return dev.download(maj), dev.download(quad), dev.download(er)

    res = sharding.ThreadComm.run(world, fn)
    np.testing.assert_array_equal(np.concatenate([r[0] for r in res]), want_maj)
    # tolerance class, but partition invariant: every cell's sums are a fixed sequence of double operations
    np.testing.assert_array_equal(np.concatenate([r[1] for r in res]), want_quad)
    np.testing.assert_array_equal(np.concatenate([r[2] for r in res]), want_er)


@pytest.mark.parametrize("world,ny", [(1, 400), (2, 400), (4, 400), (2, 512), (3, 386)])
def test_banded_sinkfill_matches_oracle(world, ny):
    # ny = 512 / world 2: the extended band has 257 rows, so the halo row sits alone in its tile row
    # world 1: the global coarse start and hd_pdfill_band_start on a band that is the whole mosaic, one round
    sc = SynthScene(ny, 390, 52)
    z = np.round(sc.srtm())
    z[100:103, 50:60] = np.nan
    z[200:260, 100:180] -= 9                                   # a pan that spans band boundaries
    want = hydrology.sinkfill(z)

    def fn(comm):
        band = sharding.Band(comm, *z.shape)
        w, d8 = band.sinkfill(dev.upload(band.take(z)))
        return dev.download(w), dev.download(d8), band.fill_rounds, band.fill_status()

    res = sharding.ThreadComm.run(world, fn)
    np.testing.assert_array_equal(np.concatenate([r[0] for r in res]), want)
    np.testing.assert_array_equal(np.concatenate([r[1] for r in res]), hydrology.d8(want))
    assert (res[0][2] == 1 if world == 1 else res[0][2] >= 2) and all(r[3] == 0 for r in res)


@pytest.mark.parametrize("direct", ["1", "0"])
@pytest.mark.parametrize("world,shape", [(2, (301, 333)), (3, (301, 333)), (2, (300, 334)), (3, (421, 300)), (4, (1300, 262))])
def test_banded_detect_apply_fourier_is_bit_identical(world, shape, direct, monkeypatch):
    """The stripe-removal stage on row bands (the same row transforms as on one GPU, transposes as all-to-alls,
    Hermitian completion in the K layout, banded peak detector): odd x odd takes the Hermitian inverse, the others the
    complex one; every output cell must carry the single-GPU bits -- with the exchanges as peer-memory stores from the
    transposes (direct) and as send / recv messages."""
    monkeypatch.setenv("HD_BAND_DIRECT", direct)
    sc = SynthScene(*shape, 71)
    srtm = sc.srtm()
    daf = cf.DetectApplyFourier()
    want = daf.apply(srtm)
    want_mask = daf.mask
    assert want_mask.sum() > 0

    def fn(comm):
        band = sharding.Band(comm, *srtm.shape)
        ext = band.detect_apply_fourier(dev.upload(band.take(srtm)))
        mask, kl = band._last_mask
        return dev.download(ext.owned()), dev.download(mask), kl

    res = sharding.ThreadComm.run(world, fn)
    got = np.concatenate([r[0] for r in res])
    assert got.dtype == np.float64 and got.shape == want.shape
    np.testing.assert_array_equal(got, want)
    # the assembled mask, row by row of every rank's K layout (spectrum row ky sits at shifted row (ky + ny/2) % ny)
    ny = shape[0]
    for _, m, kl in res:
        np.testing.assert_array_equal(m, want_mask[(kl["ky"] + ny // 2) % ny].astype(np.uint8))


@pytest.mark.parametrize("world,shape,direct", [(2, (420, 333), "1"), (3, (421, 333), "1"), (4, (640, 300), "1"),
                                                (3, (420, 334), "0")])
def test_banded_chain_is_bit_identical(world, shape, direct, monkeypatch):
    """The whole conditioning chain on row bands against the single-GPU chain: EVERY output identical -- with the
    exchanges of the Fourier stage as peer-memory stores from the transposes (direct) and as send / recv messages."""
    from hydrodem_b200.pipeline import ConditioningChain
    monkeypatch.setenv("HD_BAND_DIRECT", direct)
    sc = SynthScene(*shape, 81)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    hsheds[shape[0] // 2, 40] = -32768.0                       # a void right next to a cut
    ref = ConditioningChain(keep_intermediates=True).apply(srtm, groves, hsheds.copy())

    def fn(comm):
        band = sharding.Band(comm, *srtm.shape)
        out = band.conditioning_chain(dev.upload(band.take(srtm)), dev.upload(band.take(groves)),
                                      dev.upload(band.take(hsheds)), keep_complete=True)
        return {k: dev.download(v) for k, v in out.items()}

    res = sharding.ThreadComm.run(world, fn)
    got = {k: np.concatenate([r[k] for r in res]) for k in res[0]}
    np.testing.assert_array_equal(got["dem_complete"], ref.dem_complete)
    np.testing.assert_array_equal(got["final"], ref.final)
    np.testing.assert_array_equal(got["filled"], ref.filled)
    np.testing.assert_array_equal(got["d8"], ref.d8)
    np.testing.assert_array_equal(got["filled"], hydrology.sinkfill(got["final"]))
    np.testing.assert_array_equal(got["d8"], hydrology.d8(got["filled"]))


@pytest.mark.parametrize("world", [2, 3])
def test_banded_apply_to_host_is_bit_identical(world):
    """Band.apply_to_host (copies on their own streams, underneath the kernels) returns the single-GPU bits; pageable and
    pinned inputs, called twice (recycled buffers), the final DEM sent as int16 and as float64, and a final DEM outside
    int16 (the device flag makes the int16 transport fetch the float64 raster after all).  Every rank counts the PCIe
    bytes of its rows: the three inputs up; the final DEM (int16 + a 4-byte flag, or float64), filled (float32), d8
    down."""
    from hydrodem_b200.pipeline import ConditioningChain
    sc = SynthScene(420, 333, 83)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    ref = ConditioningChain().apply(srtm, groves, hsheds.copy())
    srtm_hi, hsheds_hi = srtm + np.float32(40000), hsheds + np.float32(40000)
    ref_hi = ConditioningChain().apply(srtm_hi, groves, hsheds_hi.copy())
    assert ref_hi.final.max() > 32767

    def fn(comm):
        band = sharding.Band(comm, *srtm.shape)
        rows = [np.ascontiguousarray(band.take(a)) for a in (srtm, groves.astype(np.uint8), hsheds)]
        pinned = []
        for a in rows:
            p = dev.pinned_empty(a.shape, a.dtype)
            p[...] = a
            pinned.append(p)
        out, sent = {}, {}
        out["pageable"] = band.apply_to_host(*rows)
        sent["pageable"] = band.last_transfer_bytes
        band.apply_to_host(*pinned)
        out["pinned"] = {k: v.copy() for k, v in band.apply_to_host(*pinned).items()}
        sent["pinned"] = band.last_transfer_bytes
        out["high"] = band.apply_to_host(band.take(srtm_hi), rows[1], band.take(hsheds_hi))
        sent["high"] = band.last_transfer_bytes
        band.narrow_final = False
        out["float64"] = band.apply_to_host(*pinned)
        sent["float64"] = band.last_transfer_bytes
        return out, sent, sum(a.nbytes for a in rows), band.rows * band.nx

    res = sharding.ThreadComm.run(world, fn)
    for which, want in (("pageable", ref), ("pinned", ref), ("high", ref_hi), ("float64", ref)):
        got = {k: np.concatenate([r[0][which][k] for r in res]) for k in ("final", "filled", "d8")}
        assert got["final"].dtype == np.float64 and got["filled"].dtype == np.float32 and got["d8"].dtype == np.uint8
        np.testing.assert_array_equal(got["final"], want.final)
        np.testing.assert_array_equal(got["filled"], want.filled)
        np.testing.assert_array_equal(got["d8"], want.d8)
    for _, sent, h2d, cells in res:
        assert sent["pageable"] == sent["pinned"] == (h2d, 2 * cells + 4 + 4 * cells + cells)
        assert sent["high"] == (h2d, 2 * cells + 4 + 8 * cells + 4 * cells + cells)     # int16 + flag, then float64
        assert sent["float64"] == (h2d, 8 * cells + 4 * cells + cells)


def test_banded_apply_to_host_raises_on_a_stalled_fill(monkeypatch):
    """A banded run whose sink-fill did not reach its fixed point raises DeviceError on every rank instead of returning
    the poisoned surface.  The status word is faked on the host: no fill is made to stall."""
    from hydrodem_b200.exceptions import DeviceError
    sc = SynthScene(420, 333, 83)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    monkeypatch.setattr(sharding.Band, "fill_status", lambda self: 1)

    def fn(comm):
        band = sharding.Band(comm, *srtm.shape)
        with pytest.raises(DeviceError, match="fixed point"):
            band.apply_to_host(band.take(srtm), band.take(groves), band.take(hsheds))
        return True

    assert sharding.ThreadComm.run(2, fn) == [True, True]

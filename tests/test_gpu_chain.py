"""GPU: the fused device-resident chain (hydrodem_b200.pipeline) against the oracle chain."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200.pipeline import ConditioningChain
    from hydrodem_b200.synth import SynthScene
    from oracle import chain as ochain, hydrology


@pytest.mark.parametrize("shape,seed", [((300, 420), 77), ((519, 508), 5)])
def test_chain_vs_oracle(shape, seed):
    sc = SynthScene(*shape, seed)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    res = ConditioningChain(keep_intermediates=True).apply(srtm, groves, hsheds.copy())
    with np.errstate(all="ignore"):
        want = ochain.conditioning_chain(srtm, groves, hsheds.copy())
    lag = want["lagoons"]
    # bit-exact class
    np.testing.assert_array_equal(res.hsheds_nan_fixed, lag["CorrectNANValues"])
    np.testing.assert_array_equal(res.majority, lag["MajorityFilter"])
    np.testing.assert_array_equal(res.lagoons_values, lag["TidyingLagoons"])
    np.testing.assert_array_equal(res.groves.astype(bool), want["groves"])
    assert int((res.fourier_mask != want["mask"]).sum()) == 0
    # tolerance class: <= 1e-5 relative
    np.testing.assert_allclose(res.fourier, want["fourier"], rtol=1e-5)
    np.testing.assert_allclose(res.srtm, want["srtm"], rtol=1e-5)
    np.testing.assert_allclose(res.dem_complete, want["dem_complete"], rtol=1e-5)
    # rounding: flips only where the 3x3 mean sits within 1e-3 of a half-integer
    assert res.final.dtype == np.float64
    from oracle import stencils
    mean = stencils.convolve_reflect(want["dem_complete"], np.ones((3, 3))) / 9
    flips = res.final != want["final"]
    frac = np.abs(mean - np.floor(mean) - 0.5)
    assert (frac[flips] < 1e-3).all() and np.abs(res.final - want["final"])[flips].max(initial=0) <= 1
    print("rounding flips:", int(flips.sum()), "of", flips.size)
    # hydrology on the chain's own final DEM
    np.testing.assert_array_equal(res.filled, hydrology.sinkfill(res.final))
    np.testing.assert_array_equal(res.d8, hydrology.d8(res.filled))


def test_c2_chain_vs_oracle_at_3601():
    """BASELINE.json configs[1] at its FULL size: the whole chain on a synthetic 3601 x 3601 tile against the CPU
    oracle (about a minute of CPU).  Exact stages must be identical, tolerance stages within 1e-5 relative; the rounded
    DEM may differ only where the 3x3 mean sits on a half-integer -- the number of such cells is printed."""
    import time
    from oracle import stencils
    sc = SynthScene(3601, 3601, 1002)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    res = ConditioningChain(keep_intermediates=True).apply(srtm, groves, hsheds.copy())
    t0 = time.time()
    with np.errstate(all="ignore"):
        want = ochain.conditioning_chain(srtm, groves, hsheds.copy(), with_hydrology=False)
    print(f"C2: oracle chain {time.time() - t0:.0f} s")
    lag = want["lagoons"]
    np.testing.assert_array_equal(res.hsheds_nan_fixed, lag["CorrectNANValues"])
    np.testing.assert_array_equal(res.majority, lag["MajorityFilter"])
    np.testing.assert_array_equal(res.lagoons_values, lag["TidyingLagoons"])
    np.testing.assert_array_equal(res.groves.astype(bool), want["groves"])
    mism = int((res.fourier_mask != want["mask"]).sum())
    print("C2: Fourier mask cells that differ:", mism, "of", int(want["mask"].sum()), "blanked")
    assert mism == 0
    np.testing.assert_allclose(res.fourier, want["fourier"], rtol=1e-5)
    # GrovesCorrection decides with a THRESHOLD (dem - smooth > 1.5, custom_filters.py:715-718): a groves cell whose
    # difference sits within float32 rounding of 1.5 m flips on any tolerance-class input difference, moves by ~1.5 m, and
    # nudges the smooth surface of the groves cells within 7 cells in the following iterations.  Those cells are located
    # from the ORACLE's own intermediate (|hi - 1.5| < 2e-3), counted, printed and excluded; everything else must agree.
    from scipy import ndimage
    border = np.zeros(srtm.shape, dtype=bool)
    for hi in want["groves_hi"]:
        border |= want["groves"] & (np.abs(hi - 1.5) < 2e-3)
    allowed = ndimage.binary_dilation(border, structure=np.ones((3, 3)), iterations=14)
    bad = ~np.isclose(res.srtm, want["srtm"], rtol=1e-5, atol=0)
    print("C2: groves cells on the 1.5 m threshold:", int(border.sum()), "-> cells that differ:", int(bad.sum()))
    assert border.sum() < 1e-4 * border.size and bad.sum() <= border.sum() and not (bad & ~allowed).any()
    ok = ~ndimage.binary_dilation(allowed, structure=np.ones((3, 3)))
    np.testing.assert_allclose(res.dem_complete[~allowed], want["dem_complete"][~allowed], rtol=1e-5)
    mean = stencils.convolve_reflect(want["dem_complete"], np.ones((3, 3))) / 9
    flips = (res.final != want["final"]) & ok
    frac = np.abs(mean - np.floor(mean) - 0.5)
    print("C2: rounding flips:", int(flips.sum()), "of", flips.size)
    assert flips.mean() < 1e-4 and (frac[flips] < 1e-3).all() and np.abs(res.final - want["final"])[flips].max(initial=0) <= 1
    # hydrology on the chain's own final DEM (C priority-flood oracle)
    np.testing.assert_array_equal(res.filled, hydrology.sinkfill(res.final))
    np.testing.assert_array_equal(res.d8, hydrology.d8(res.filled))


def test_fused_combine_equals_separate_kernels():
    """hd_final_mean3 (final terms + 3x3 mean + round in one pass, float32 staging) against hd_final_terms + hd_convolve3:
    same bits in every output, frame rows / columns (reflect) included; NaN and lagoon cells present."""
    sc = SynthScene(421, 517, 19)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    a = ConditioningChain(keep_complete=True).apply(srtm, groves, hsheds.copy())
    b = ConditioningChain(keep_complete=True, fused_combine=False).apply(srtm, groves, hsheds.copy())
    assert a.final.dtype == np.float64
    np.testing.assert_array_equal(a.final, b.final)
    np.testing.assert_array_equal(a.host("dem_complete"), b.host("dem_complete"))
    np.testing.assert_array_equal(a.filled, b.filled)
    np.testing.assert_array_equal(a.d8, b.d8)
    c = ConditioningChain().apply(srtm, groves, hsheds.copy())             # production: `complete` is never written
    np.testing.assert_array_equal(c.final, b.final)
    # groves iterations 2, 3 that only touch the tiles with groves cells (ping-pong rasters) against dense iterations
    d = ConditioningChain(keep_complete=True, sparse_groves=False).apply(srtm, groves, hsheds.copy())
    np.testing.assert_array_equal(a.host("dem_complete"), d.host("dem_complete"))
    np.testing.assert_array_equal(a.final, d.final)
    # TidyingLagoons as one kernel (hd_tidy_lagoons) against erosion + expand-select + max filter
    g = ConditioningChain(keep_intermediates=True, fused_lagoons=False).apply(srtm, groves, hsheds.copy())
    h = ConditioningChain(keep_intermediates=True).apply(srtm, groves, hsheds.copy())
    np.testing.assert_array_equal(h.host("lagoons_values"), g.host("lagoons_values"))
    assert np.count_nonzero(h.host("lagoons_values")) > 0
    np.testing.assert_array_equal(h.final, g.final)
    for iters in (1, 2, 4):
        e = ConditioningChain(keep_complete=True, groves_iterations=iters, with_hydrology=False).apply(srtm, groves, hsheds.copy())
        f = ConditioningChain(keep_complete=True, groves_iterations=iters, with_hydrology=False,
                              sparse_groves=False).apply(srtm, groves, hsheds.copy())
        np.testing.assert_array_equal(e.host("dem_complete"), f.host("dem_complete"))


def test_chain_with_rivers():
    sc = SynthScene(200, 260, 9)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    rivers = np.zeros(srtm.shape, dtype=np.float32)
    rivers[50, 20:200] = 1
    res = ConditioningChain(with_hydrology=False, keep_intermediates=True).apply(srtm, groves, hsheds.copy(), rivers)
    with np.errstate(all="ignore"):
        want = ochain.conditioning_chain(srtm, groves, hsheds.copy(), rivers=rivers, with_hydrology=False)
    np.testing.assert_allclose(res.dem_complete, want["dem_complete"], rtol=1e-5)


def test_apply_to_host_matches_lazy_path():
    """The overlapped host API returns exactly what the lazy ChainResult path returns."""
    sc = SynthScene(333, 401, 3)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    chain = ConditioningChain()
    a = chain.apply(srtm, groves, hsheds.copy())
    for _ in range(2):
        b = chain.apply_to_host(srtm, groves, hsheds.copy())
        assert b["final"].dtype == np.float64 and b["filled"].dtype == np.float32 and b["d8"].dtype == np.uint8
        np.testing.assert_array_equal(b["final"], a.final)
        np.testing.assert_array_equal(b["filled"], a.filled)
        np.testing.assert_array_equal(b["d8"], a.d8)
    # mosaic-sized rasters take the eager three-stream path (no captured slot): pageable and pinned inputs
    from hydrodem_b200 import device as dev
    chain.eager_cells = 0
    pinned = []
    for arr in (srtm, groves.astype(np.uint8), hsheds):
        p = dev.pinned_empty(arr.shape, arr.dtype)
        p[...] = arr
        pinned.append(p)
    for args in ((srtm, groves, hsheds.copy()), tuple(pinned), tuple(pinned)):
        b = chain.apply_to_host(*args)
        assert b["final"].dtype == np.float64 and b["filled"].dtype == np.float32 and b["d8"].dtype == np.uint8
        np.testing.assert_array_equal(b["final"], a.final)
        np.testing.assert_array_equal(b["filled"], a.filled)
        np.testing.assert_array_equal(b["d8"], a.d8)
    # the final DEM travels as int16 (+ a 4-byte flag) and is widened on the host
    assert chain.last_transfer_bytes == (srtm.nbytes + groves.size + hsheds.nbytes,
                                         2 * srtm.size + 4 + 4 * srtm.size + srtm.size)
    chain.narrow_final = False
    b = chain.apply_to_host(*pinned)
    np.testing.assert_array_equal(b["final"], a.final)
    assert chain.last_transfer_bytes[1] == 8 * srtm.size + 4 * srtm.size + srtm.size


def test_apply_to_host_raises_on_a_stalled_fill(monkeypatch):
    """The eager host call raises DeviceError when the sink-fill did not reach its fixed point.  The status word is
    faked on the host: no fill is made to stall."""
    from hydrodem_b200.exceptions import DeviceError
    from hydrodem_b200.filters import new_filters as nf
    sc = SynthScene(200, 260, 6)
    chain = ConditioningChain()
    chain.eager_cells = 0
    monkeypatch.setattr(nf.SinkFillD8, "status", lambda self: 1)
    with pytest.raises(DeviceError, match="fixed point"):
        chain.apply_to_host(sc.srtm(), sc.groves(), sc.hsheds())


def test_captured_graph_matches_eager():
    """Replaying the captured CUDA graph gives the same bits as eager launches, also after the inputs changed."""
    from hydrodem_b200 import device as dev
    sc = SynthScene(310, 387, 4)
    chain = ConditioningChain()
    d_in = chain.upload_inputs(sc.srtm(), sc.groves(), sc.hsheds())
    eager = chain.run_device(*d_in)
    want = (eager.final.copy(), eager.filled.copy(), eager.d8.copy())
    cap = chain.capture(*d_in)
    assert cap.launches > 20
    for _ in range(2):
        got = cap.replay()
        np.testing.assert_array_equal(got.final, want[0])
        np.testing.assert_array_equal(got.filled, want[1])
        np.testing.assert_array_equal(got.d8, want[2])
    # new data in the same buffers
    sc2 = SynthScene(310, 387, 5)
    for raster, arr in zip(d_in, (sc2.srtm(), sc2.groves(), sc2.hsheds())):
        raster.tensor().copy_(torch.from_numpy(arr).cuda())
    got = cap.replay()
    ref = chain.run_device(*d_in)
    np.testing.assert_array_equal(got.final, ref.final)
    np.testing.assert_array_equal(got.filled, ref.filled)


def test_stream_of_tiles_matches_single_calls():
    """ConditioningChain.stream: different tiles through the double-buffered graph slots, results in order and
    bit-identical to one-at-a-time runs (pageable inputs, slot reuse, a second shape in the same stream)."""
    scenes = [SynthScene(290, 333, s) for s in (11, 12, 13, 14, 15)] + [SynthScene(201, 260, 16)]
    chain = ConditioningChain()
    items = [(sc.srtm(), sc.groves(), sc.hsheds()) for sc in scenes]
    want = [chain.apply(a, b, c.copy()) for (a, b, c) in items]
    got = list(chain.stream(iter(items)))
    assert len(got) == len(items)
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g["final"], w.final)
        np.testing.assert_array_equal(g["filled"], w.filled)
        np.testing.assert_array_equal(g["d8"], w.d8)
    # the slots are kept: a second stream over the same shapes replays the captured graphs
    again = list(chain.stream(iter(items[:3]), depth=3))
    for g, w in zip(again, want):
        np.testing.assert_array_equal(g["final"], w.final)
    chain.release()


def test_stream_with_rivers_and_no_hydrology():
    sc = SynthScene(200, 260, 9)
    srtm, groves, hsheds = sc.srtm(), sc.groves(), sc.hsheds()
    rivers = np.zeros(srtm.shape, dtype=np.float32)
    rivers[50, 20:200] = 1
    chain = ConditioningChain(with_hydrology=False)
    want = chain.apply(srtm, groves, hsheds.copy(), rivers).final
    outs = list(chain.stream([(srtm, groves, hsheds, rivers)] * 3))
    for o in outs:
        assert set(o) == {"final"}
        np.testing.assert_array_equal(o["final"], want)


def test_stream_falls_back_to_float32_transport():
    """Elevations outside int16 (or NaN / fractional results) cannot use the int16 transport of the streaming API:
    the device-side check flags the tile and the float32 raster is fetched instead -- same bits as the plain path."""
    sc = SynthScene(210, 300, 21)
    srtm, groves, hsheds = sc.srtm() + np.float32(40000), sc.groves(), sc.hsheds() + np.float32(40000)
    chain = ConditioningChain()
    want = chain.apply(srtm, groves, hsheds.copy())
    assert want.final.max() > 32767
    ok = SynthScene(210, 300, 22)
    items = [(srtm, groves, hsheds), (ok.srtm(), ok.groves(), ok.hsheds()), (srtm, groves, hsheds)]
    got = list(chain.stream(items))
    for g in (got[0], got[2]):
        np.testing.assert_array_equal(g["final"], want.final)
        np.testing.assert_array_equal(g["filled"], want.filled)
        np.testing.assert_array_equal(g["d8"], want.d8)
    want_ok = chain.apply(ok.srtm(), ok.groves(), ok.hsheds())
    np.testing.assert_array_equal(got[1]["final"], want_ok.final)
    np.testing.assert_array_equal(got[1]["filled"], want_ok.filled)
    assert got[1]["final"].dtype == np.float64 and got[1]["filled"].dtype == np.float32
    # the eager three-stream path of mosaic-sized rasters: same flag, float64 fetched instead
    chain.eager_cells = 0
    for args, w in (((srtm, groves, hsheds.copy()), want), ((ok.srtm(), ok.groves(), ok.hsheds()), want_ok)):
        g = chain.apply_to_host(*args)
        assert g["final"].dtype == np.float64
        np.testing.assert_array_equal(g["final"], w.final)
        np.testing.assert_array_equal(g["filled"], w.filled)
        np.testing.assert_array_equal(g["d8"], w.d8)
    assert chain.last_transfer_bytes[1] == 2 * srtm.size + 4 + 4 * srtm.size + srtm.size


def test_stream_errors_propagate_and_chain_stays_usable():
    """A tile the Fourier stage cannot take (a spectrum quarter smaller than the 55-cell detector window,
    custom_filters.py:395-427 via sliding_window.py:151-156) raises the reference's WindowSizeHighError out of
    ``stream``; wrong argument types raise NumpyArrayExpectedError; the chain object keeps working afterwards."""
    from hydrodem_b200.exceptions import NumpyArrayExpectedError, WindowSizeHighError
    chain = ConditioningChain()
    small = SynthScene(120, 120, 5)
    with pytest.raises(WindowSizeHighError):
        list(chain.stream([(small.srtm(), small.groves(), small.hsheds())]))
    with pytest.raises(NumpyArrayExpectedError):
        list(chain.stream([(small.srtm().tolist(), small.groves(), small.hsheds())]))
    with pytest.raises(ValueError):
        list(chain.stream([(small.srtm()[:100], small.groves(), small.hsheds())]))
    ok = SynthScene(200, 260, 6)
    want = chain.apply(ok.srtm(), ok.groves(), ok.hsheds())
    got = list(chain.stream([(ok.srtm(), ok.groves(), ok.hsheds())] * 2))
    for g in got:
        np.testing.assert_array_equal(g["final"], want.final)
        np.testing.assert_array_equal(g["d8"], want.d8)

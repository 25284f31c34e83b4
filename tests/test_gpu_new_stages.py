"""GPU parity of the NEW stages (median, sink-fill, D8) against this repo's own oracle -- the reference has
no such code ("parity unpinned").  Bit-exact."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from hydrodem_b200.filters import new_filters as nf
    from hydrodem_b200.synth import SynthScene
    from oracle import stencils, hydrology, clib


def eq(a, b):
    assert a.dtype == b.dtype, (a.dtype, b.dtype)
    np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("ws,circ", [(3, False), (3, True), (5, False), (5, True)])
def test_median_vs_oracle(ws, circ):
    a = SynthScene(70, 261, 41).srtm()
    eq(nf.MedianFilter(window_size=ws, circular=circ).apply(a), stencils.median(a, ws, circ))
    b = a.copy()
    rng = np.random.default_rng(1)
    b[rng.random(a.shape) < 0.2] = np.nan
    b[10:17, 100:108] = np.nan
    b[30, 30] = np.inf
    b[31, 31] = -np.inf
    eq(nf.MedianFilter(window_size=ws, circular=circ).apply(b), stencils.median(b, ws, circ))
    c = a.astype(np.float64) * 1.0000001
    got = nf.MedianFilter(window_size=ws, circular=circ).apply(c)
    eq(got, stencils.median(c, ws, circ))


def test_median_full_tile_vs_c_oracle():
    a = SynthScene(3601, 3601, 1002).srtm()
    eq(nf.MedianFilter(window_size=5).apply(a), clib.median(a, 5, False))


def _terrain(ny, nx, seed):
    sc = SynthScene(ny, nx, seed)
    z = sc.srtm()
    rng = np.random.default_rng(seed)
    for _ in range(max(3, ny * nx // 20000)):                  # pits and pans
        y, x = int(rng.integers(2, ny - 2)), int(rng.integers(2, nx - 2))
        r = int(rng.integers(1, 12))
        z[max(0, y - r):y + r, max(0, x - r):x + r] -= np.float32(rng.uniform(1, 15))
    return z


@pytest.mark.parametrize("shape", [(60, 71), (64, 64), (65, 129), (200, 333), (700, 900)])
def test_sinkfill_d8_vs_oracle(shape):
    z = _terrain(*shape, seed=shape[0])
    z[5:8, 9:12] = np.nan
    fill = nf.SinkFill()
    w = fill.apply(z)
    want = hydrology.sinkfill(z)
    eq(w, want)
    assert fill.sweeps >= 1 and (want[~np.isnan(z)] > z[~np.isnan(z)]).sum() > 0
    eq(nf.D8FlowDirection().apply(w), hydrology.d8(want))
    # idempotence: a filled surface is a fixed point
    eq(nf.SinkFill().apply(w), w)


def _d8_ties(ny, nx, seed):
    """A surface whose D8 decisions hit every special case: exact ties between a straight and a diagonal drop
    (c = 1, straight neighbour 1 - q, diagonal neighbour 0 with q = float32(0.70710678): both drops are q), ties
    among straight and among diagonal drops, +-0.0, NaN, +inf and -inf cells, flats with no positive drop."""
    q = np.float32(0.70710678)
    vals = np.array([0.0, -0.0, 1.0, 2.0, np.float32(1) - q, np.float32(2) - 2 * q, 2 * q, q], dtype=np.float32)
    rng = np.random.default_rng(seed)
    w = vals[rng.integers(0, len(vals), (ny, nx))]
    special = rng.random((ny, nx))
    w[special < 0.03] = np.nan
    w[(special >= 0.03) & (special < 0.05)] = np.inf
    w[(special >= 0.05) & (special < 0.07)] = -np.inf
    return w


def test_d8_decision_special_cases():
    """hd_d8 against the strict-greater loop of the oracle on ties, signed zeros, NaN and infinities."""
    w = _d8_ties(61, 83, 7)
    want = hydrology.d8(w)
    # the input exercises what it claims: some cell's winner ties with a later straight or diagonal direction
    c = w[1:-1, 1:-1]
    drops = []
    with np.errstate(invalid="ignore"):
        for k, (dy, dx) in enumerate(zip(hydrology.D8_DY, hydrology.D8_DX)):
            d = (c - w[1 + dy:w.shape[0] - 1 + dy, 1 + dx:w.shape[1] - 1 + dx]).astype(np.float32)
            drops.append((d * hydrology.INV_SQRT2_F32).astype(np.float32) if k & 1 else d)
    drops = np.stack(drops)
    best = np.nanmax(np.where(drops > 0, drops, np.nan), axis=0, initial=0)
    attains = (drops == best) & (best > 0)
    assert (attains[0::2].any(axis=0) & attains[1::2].any(axis=0)).sum() > 100      # straight-diagonal ties
    assert (attains.sum(axis=0) > 1).sum() > 500 and (best == np.inf).sum() > 100
    assert (want[1:-1, 1:-1] == 0).sum() > 100
    eq(nf.D8FlowDirection().apply(w), want)


def test_sinkfill_modes_agree():
    """The worklist fill of an odd shape with a nodata block reaches the oracle's unique fixed point."""
    z = _terrain(515, 777, 12)
    z[100:104, 200:230] = np.nan
    eq(nf.SinkFill().apply(z), hydrology.sinkfill(z))


def test_sinkfill_small_against_iterative_pd():
    z = _terrain(48, 50, 3)
    it, _ = hydrology.sinkfill_iterative(z)
    eq(nf.SinkFill().apply(z), it)


def test_sinkfill_full_tile():
    """C2 size: 3601 x 3601 against the priority-flood oracle; D8 against the C oracle."""
    z = _terrain(3601, 3601, 1002)
    fill = nf.SinkFill()
    w = fill.apply(z)
    eq(w, clib.priority_flood(z))
    eq(nf.D8FlowDirection().apply(w), clib.d8(w))
    print("sweeps", fill.sweeps)


def test_fused_fill_d8_equals_separate_passes():
    """hd_pdfill_d8 (fill, then ONE pass restoring NaN and writing D8) against SinkFill -> D8FlowDirection and the
    oracle; the sticky status word reads 0."""
    from hydrodem_b200.filters import new_filters as nf
    from oracle import hydrology
    z = np.round(SynthScene(333, 517, 91).srtm())
    z[40:44, 100:130] = np.nan
    z[200, 0] = np.nan                                          # nodata on the frame
    z[150:220, 300:420] -= 7
    fused = nf.SinkFillD8(want_stats=True)
    filled, d8 = fused.apply(z)
    want = hydrology.sinkfill(z)
    np.testing.assert_array_equal(filled, want)
    np.testing.assert_array_equal(d8, hydrology.d8(want))
    np.testing.assert_array_equal(filled, nf.SinkFill().apply(z))
    np.testing.assert_array_equal(d8, nf.D8FlowDirection().apply(filled))
    assert fused.status() == 0 and fused.sweeps >= 1


@pytest.mark.parametrize("ctas_per_sm", ["1", "4"])
def test_fill_worklist_stress(ctas_per_sm, monkeypatch):
    """The inter-CTA polling protocol of fill_async_kernel (csrc/hydro.cu: poke / ticket / pending) under different
    amounts of concurrency, many odd shapes, NaN outlets on and off the frame, large flats: always the priority-flood
    fixed point, status word 0.  (compute-sanitizer racecheck is closed on the measurement pool.)"""
    from hydrodem_b200.filters import new_filters as nf
    from oracle import hydrology
    monkeypatch.setenv("HD_FILL_CTAS_PER_SM", ctas_per_sm)
    rng = np.random.default_rng(int(ctas_per_sm))
    for k in range(12):
        ny, nx = int(rng.integers(65, 700)), int(rng.integers(65, 900))
        z = np.round(SynthScene(ny, nx, 500 + k).srtm() * (1 + k % 3))
        if k % 2:
            z[ny // 3:ny // 3 + 3, nx // 4:nx // 4 + 9] = np.nan
            z[0, nx // 2] = np.nan
        if k % 4 == 0:
            z[ny // 2:ny // 2 + 40, 5:nx - 5] = z.min() - 3            # a long flat trench across tiles
        f = nf.SinkFillD8()
        filled, d8 = f.apply(z)
        want = hydrology.sinkfill(z)
        np.testing.assert_array_equal(filled, want)
        np.testing.assert_array_equal(d8, hydrology.d8(want))
        assert f.status() == 0

"""Float64 NumPy restatement of mosaics: several sources on one lattice sampled as one virtual raster (DESIGN.md §9c).

The reference hd_warp_mosaic is tested against; it is not on the product path.  ``mosaic`` materialises the virtual
raster (last listed source wins, nodata is transparent) with a "has sample" mask; ``sample`` is ``oracle.warp.sample``
restated with that mask and with (u, v) measured from another lattice point than the array's corner.  The projection
and the pixel coordinates are ``oracle.warp``'s.
"""
import numpy as np


def mosaic(sources):
    """The virtual raster of a mosaic, materialised: ``sources`` is a list of (array, (x0, dx, y0, dy), nodata or None)
    sharing the first source's pixel size and nodata.  Source i lies at the lattice offset (round((x0_i - x0_1) / dx),
    round((y0_1 - y0_i) / dy)) from the first listed source.  A pixel takes the value of the last listed source that
    covers it with a value that is not nodata; where there is none it has no sample and holds nodata (0 without).
    Returns (array in the sources' dtype, (x0, dx, y0, dy) of its top-left corner, has_sample bool mask)."""
    x0, dx, y0, dy = sources[0][1]
    nodata = sources[0][2]
    offs = [(int(round((g[0] - x0) / dx)), int(round((y0 - g[2]) / dy))) for _, g, _ in sources]
    u0 = min(u for u, _ in offs)
    v0 = min(v for _, v in offs)
    u1 = max(u + np.shape(a)[1] for (u, _), (a, _, _) in zip(offs, sources))
    v1 = max(v + np.shape(a)[0] for (_, v), (a, _, _) in zip(offs, sources))
    out = np.full((v1 - v0, u1 - u0), 0 if nodata is None else nodata, dtype=np.asarray(sources[0][0]).dtype)
    has = np.zeros(out.shape, bool)
    for (u, v), (a, _, nd) in zip(offs, sources):           # in list order: a later source overwrites
        a = np.asarray(a)
        ok = np.ones(a.shape, bool) if nd is None else ~((a == nd) | (np.isnan(nd) & np.isnan(a)))
        win = (slice(v - v0, v - v0 + a.shape[0]), slice(u - u0, u - u0 + a.shape[1]))
        out[win][ok] = a[ok]
        has[win] |= ok
    return out, (x0 + u0 * dx, dx, y0 - v0 * dy, dy), has


def sample(src, u, v, resample="nearest", nodata=None, valid=None, origin=(0, 0)):
    """Values at (u, v) as float64; cells with no sample get nodata (or 0 without one).  A pixel has no sample when it
    is outside src, equals nodata, or (``valid``, a bool mask of src) is marked False there.  ``origin``: the integer
    (u, v) of src's pixel (0, 0), for (u, v) measured from another lattice point (a mosaic's first listed source).
    Nearest: the pixel (floor u, floor v).  Bilinear: taps floor(u - 1/2), floor(v - 1/2) and their +1 neighbours,
    taps with no sample dropped and the remaining weights renormalised."""
    src = np.asarray(src)
    sny, snx = src.shape
    ou, ov = origin
    if valid is None:
        valid = np.ones(src.shape, bool)
    if nodata is not None:
        valid = valid & ~((src == nodata) | (np.isnan(nodata) & np.isnan(src)))

    def tap(tx, ty):
        """(has sample, value) of the taps at integer-valued (tx, ty) in the (u, v) frame."""
        ok = (tx >= ou) & (tx < ou + snx) & (ty >= ov) & (ty < ov + sny)
        iy, ix = ty[ok].astype(np.int64) - ov, tx[ok].astype(np.int64) - ou
        s = np.zeros(tx.shape)
        s[ok] = src[iy, ix]
        ok[ok] = valid[iy, ix]
        return ok, s

    fill = 0.0 if nodata is None else float(nodata)
    out = np.full(u.shape, fill)
    if resample == "nearest":
        ok, s = tap(np.floor(u), np.floor(v))
        out[ok] = s[ok]
        return out
    if resample != "bilinear":
        raise ValueError(resample)
    fu, fv = u - 0.5, v - 0.5
    x0, y0 = np.floor(fu), np.floor(fv)
    ax, ay = fu - x0, fv - y0
    acc = np.zeros(u.shape)
    wsum = np.zeros(u.shape)
    for ty, wy in ((y0, 1 - ay), (y0 + 1, ay)):                 # hd_warp's tap order and accumulation order
        for tx, wx in ((x0, 1 - ax), (x0 + 1, ax)):
            ok, s = tap(tx, ty)
            w = np.where(ok, wy * wx, 0.0)
            acc += np.where(ok, w * s, 0.0)
            wsum += w
    good = wsum > 0
    out[good] = acc[good] / wsum[good]
    return out

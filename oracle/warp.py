"""Float64 NumPy restatement of the reprojection onto the EPSG:22184 grid (utils_dem.resample_and_cut, utils_dem.py:65-84).

The reference the GPU warp is tested against; it is not on the product path.  Transverse Mercator by the Krueger series
to order n^6 (Karney 2011, "Transverse Mercator with an accuracy of a few nanometers", eqs. 35-36 and the coefficient
tables of his section 4), written term by term (no Clenshaw summation), with the conformal -> geodetic latitude step as
the classic fixed-point iteration (Snyder, "Map Projections -- A Working Manual", eq. 7-9) instead of a Newton step.
"""
import numpy as np

# EPSG:22184 POSGAR 94 / Argentina 4: WGS84 ellipsoid, lat0 = -90, lon0 = -63, k0 = 1, FE = 4 500 000 m, FN = 0
EPSG22184 = (6378137.0, 1.0 / 298.257223563, -90.0, -63.0, 1.0, 4500000.0, 0.0)


def _series(f):
    n = f / (2.0 - f)
    alpha = [n / 2 - 2 * n**2 / 3 + 5 * n**3 / 16 + 41 * n**4 / 180 - 127 * n**5 / 288 + 7891 * n**6 / 37800,
             13 * n**2 / 48 - 3 * n**3 / 5 + 557 * n**4 / 1440 + 281 * n**5 / 630 - 1983433 * n**6 / 1935360,
             61 * n**3 / 240 - 103 * n**4 / 140 + 15061 * n**5 / 26880 + 167603 * n**6 / 181440,
             49561 * n**4 / 161280 - 179 * n**5 / 168 + 6601661 * n**6 / 7257600,
             34729 * n**5 / 80640 - 3418889 * n**6 / 1995840,
             212378941 * n**6 / 319334400]
    beta = [n / 2 - 2 * n**2 / 3 + 37 * n**3 / 96 - n**4 / 360 - 81 * n**5 / 512 + 96199 * n**6 / 604800,
            n**2 / 48 + n**3 / 15 - 437 * n**4 / 1440 + 46 * n**5 / 105 - 1118711 * n**6 / 3870720,
            17 * n**3 / 480 - 37 * n**4 / 840 - 209 * n**5 / 4480 + 5569 * n**6 / 90720,
            4397 * n**4 / 161280 - 11 * n**5 / 504 - 830251 * n**6 / 7257600,
            4583 * n**5 / 161280 - 108847 * n**6 / 3991680,
            20648693 * n**6 / 638668800]
    A = 1.0 / (1 + n) * (1 + n**2 / 4 + n**4 / 64 + n**6 / 256)
    return n, A, alpha, beta


def _conformal(phi, e):
    """Geodetic -> conformal latitude (radians)."""
    s = np.sin(phi)
    with np.errstate(divide="ignore"):                  # the poles: atanh(+-1) = +-inf, tanh brings it back to +-1
        return np.arcsin(np.tanh(np.arctanh(s) - e * np.arctanh(e * s)))


def _xi_eta(phi, lam, e, alpha):
    chi = _conformal(phi, e)
    xip = np.arctan2(np.tan(chi), np.cos(lam))
    etap = np.arctanh(np.cos(chi) * np.sin(lam))
    xi, eta = xip.copy(), etap.copy()
    for j, a in enumerate(alpha, start=1):
        xi = xi + a * np.sin(2 * j * xip) * np.cosh(2 * j * etap)
        eta = eta + a * np.cos(2 * j * xip) * np.sinh(2 * j * etap)
    return xi, eta


def tm_forward(lon, lat, params=EPSG22184):
    """(lon, lat) degrees -> (easting, northing) metres."""
    a, f, lat0, lon0, k0, fe, fn = params
    _, A, alpha, _ = _series(f)
    e = np.sqrt(f * (2 - f))
    phi = np.radians(np.asarray(lat, dtype=np.float64))
    lam = np.radians(np.asarray(lon, dtype=np.float64) - lon0)
    xi, eta = _xi_eta(phi, lam, e, alpha)
    xi0, _ = _xi_eta(np.radians(np.float64(lat0)), np.float64(0.0), e, alpha)
    return fe + k0 * a * A * eta, fn + k0 * a * A * (xi - xi0)


def tm_inverse(x, y, params=EPSG22184):
    """(easting, northing) metres -> (lon, lat) degrees."""
    a, f, lat0, lon0, k0, fe, fn = params
    _, A, alpha, beta = _series(f)
    e = np.sqrt(f * (2 - f))
    xi0, _ = _xi_eta(np.radians(np.float64(lat0)), np.float64(0.0), e, alpha)
    xi = (np.asarray(y, dtype=np.float64) - fn) / (k0 * a * A) + xi0
    eta = (np.asarray(x, dtype=np.float64) - fe) / (k0 * a * A)
    xip, etap = xi.copy(), eta.copy()
    for j, b in enumerate(beta, start=1):
        xip = xip - b * np.sin(2 * j * xi) * np.cosh(2 * j * eta)
        etap = etap - b * np.cos(2 * j * xi) * np.sinh(2 * j * eta)
    chi = np.arcsin(np.sin(xip) / np.cosh(etap))
    lam = np.arctan2(np.sinh(etap), np.cos(xip))
    # conformal -> geodetic: phi = 2 atan(tan(pi/4 + chi/2) ((1 + e sin phi) / (1 - e sin phi))^(e/2)) - pi/2
    phi = chi.copy()
    t = np.tan(np.pi / 4 + chi / 2)
    for _ in range(60):
        s = e * np.sin(phi)
        nxt = 2 * np.arctan(t * ((1 + s) / (1 - s)) ** (e / 2)) - np.pi / 2
        done = np.all(np.abs(nxt - phi) <= 1e-16)
        phi = nxt
        if done:
            break
    return lon0 + np.degrees(lam), np.degrees(phi)


def pixel_coords(dst_geo, ny, nx, src_geo, tm=EPSG22184, row0=0):
    """Fractional source pixel coordinates (u, v), each (ny, nx), of the destination pixel centres.
    Grids are (x0, dx, y0, dy) of the top-left corner; tm None: the source is in the destination CRS."""
    x0, dx, y0, dy = dst_geo
    sx0, sdx, sy0, sdy = src_geo
    x = x0 + (np.arange(nx, dtype=np.float64) + 0.5) * dx
    y = y0 - (np.arange(row0, row0 + ny, dtype=np.float64) + 0.5) * dy
    X, Y = np.meshgrid(x, y)
    if tm is not None:
        X, Y = tm_inverse(X, Y, tm)
    return (X - sx0) / sdx, (sy0 - Y) / sdy


def sample(src, u, v, resample="nearest", nodata=None):
    """Values at (u, v) as float64; cells with no valid sample get nodata (or 0 without one)."""
    src = np.asarray(src)
    sny, snx = src.shape
    fill = 0.0 if nodata is None else float(nodata)
    out = np.full(u.shape, fill)
    if resample == "nearest":
        ok = (u >= 0) & (u < snx) & (v >= 0) & (v < sny)
        out[ok] = src[np.floor(v[ok]).astype(np.int64), np.floor(u[ok]).astype(np.int64)]
        return out
    if resample != "bilinear":
        raise ValueError(resample)
    fu, fv = u - 0.5, v - 0.5
    x0, y0 = np.floor(fu), np.floor(fv)
    ax, ay = fu - x0, fv - y0
    acc = np.zeros(u.shape)
    wsum = np.zeros(u.shape)
    for ty, wy in ((y0, 1 - ay), (y0 + 1, ay)):
        for tx, wx in ((x0, 1 - ax), (x0 + 1, ax)):
            ok = (tx >= 0) & (tx < snx) & (ty >= 0) & (ty < sny)
            s = np.zeros(u.shape)
            s[ok] = src[ty[ok].astype(np.int64), tx[ok].astype(np.int64)]
            if nodata is not None:
                ok &= ~((s == nodata) | (np.isnan(nodata) & np.isnan(s)))
            w = np.where(ok, wy * wx, 0.0)
            acc += np.where(ok, w * s, 0.0)
            wsum += w
    good = wsum > 0
    out[good] = acc[good] / wsum[good]
    return out


def warp(src, src_geo, dst_geo, ny, nx, resample="nearest", nodata=None, tm=EPSG22184, row0=0):
    """(u, v, float32 values) of the destination grid."""
    u, v = pixel_coords(dst_geo, ny, nx, src_geo, tm, row0)
    return u, v, sample(src, u, v, resample, nodata).astype(np.float32)

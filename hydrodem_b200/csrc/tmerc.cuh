// Transverse Mercator in float64, shared by the reprojection (warp.cu: inverse, per destination cell) and the line
// rasterizer (rasterize.cu: forward, per vertex).  Krueger series to order n^6 (Karney 2011, "Transverse Mercator with an
// accuracy of a few nanometers"; the formulation of PROJ's default tmerc), both directions summed by one Clenshaw routine.
// Every function is __host__ __device__ except tm_setup, so the host functions of the C ABI (hd_host_tm_inverse,
// hd_host_tm_forward) run the very same code on the CPU.  The build's --fmad=false keeps the device arithmetic unfused.
#pragma once
#include <cmath>

namespace {

// Everything both directions need, derived on the host from the (a, f, lat0, lon0, k0, FE, FN) block.
struct TmParams {
    double A;          // rectifying radius a / (1 + n) (1 + n^2/4 + n^4/64 + n^6/256)
    double k0, fe, fn;
    double xi0;        // rectifying latitude of lat0 (radians): M0 / A
    double lon0;       // degrees
    double e, e2m;     // eccentricity, 1 - e^2
    double alpha[6];   // Krueger forward coefficients
    double beta[6];    // Krueger inverse coefficients
};

// The series of one rectifying <-> conformal step evaluated on the complex angle zeta = xi + i eta:
// sum_j c[j] sin(2 j zeta), by Clenshaw's recurrence on 2 cos(2 zeta) (one sincos and one sinh / cosh per call).
__host__ __device__ inline void krueger_sum(const double c[6], double xi, double eta, double* re, double* im)
{
    const double s2 = sin(2.0 * xi), c2 = cos(2.0 * xi);
    const double sh2 = sinh(2.0 * eta), ch2 = cosh(2.0 * eta);
    const double ar = 2.0 * c2 * ch2, ai = -2.0 * s2 * sh2;          // 2 cos(2 zeta)
    double y1r = 0.0, y1i = 0.0, y2r = 0.0, y2i = 0.0;               // b_{k+1}, b_{k+2}
    for (int k = 5; k >= 0; --k) {
        const double yr = c[k] + (ar * y1r - ai * y1i) - y2r;
        const double yi = (ar * y1i + ai * y1r) - y2i;
        y2r = y1r; y2i = y1i;
        y1r = yr; y1i = yi;
    }
    const double sr = s2 * ch2, si = c2 * sh2;                       // sin(2 zeta)
    *re = y1r * sr - y1i * si;
    *im = y1r * si + y1i * sr;
}

// (lon, lat) degrees -> rectifying coordinates (xi, eta) on the unit-A sphere, before scale and false origin:
// geodetic -> conformal latitude as tau' = tau sqrt(1 + sigma^2) - sigma sqrt(1 + tau^2), sigma = sinh(e atanh(e sin phi)),
// then the Gauss-Schreiber (xi', eta') and the forward series.
__host__ __device__ inline void tm_xi_eta(const TmParams& p, double lon, double lat, double* xi, double* eta)
{
    const double d2r = 3.14159265358979323846 / 180.0;
    const double phi = lat * d2r, lam = (lon - p.lon0) * d2r;
    const double tau = tan(phi);
    const double sig = sinh(p.e * atanh(p.e * sin(phi)));
    const double taup = tau * sqrt(1.0 + sig * sig) - sig * sqrt(1.0 + tau * tau);
    const double cl = cos(lam), sl = sin(lam);
    const double xip = atan2(taup, cl);
    const double etap = asinh(sl / sqrt(taup * taup + cl * cl));
    double re, im;
    krueger_sum(p.alpha, xip, etap, &re, &im);
    *xi = xip + re;
    *eta = etap + im;
}

// (lon, lat) degrees -> projected (x, y) metres.
__host__ __device__ inline void tm_forward(const TmParams& p, double lon, double lat, double* x, double* y)
{
    double xi, eta;
    tm_xi_eta(p, lon, lat, &xi, &eta);
    *x = p.fe + p.k0 * p.A * eta;
    *y = p.fn + p.k0 * p.A * (xi - p.xi0);
}

// Projected (x, y) metres -> (lon, lat) degrees.
__host__ __device__ inline void tm_inverse(const TmParams& p, double x, double y, double* lon, double* lat)
{
    const double xi = ((y - p.fn) / p.k0 + p.xi0 * p.A) / p.A;
    const double eta = (x - p.fe) / (p.k0 * p.A);
    double sr, si;
    krueger_sum(p.beta, xi, eta, &sr, &si);
    const double xip = xi - sr, etap = eta - si;                     // conformal (Gauss-Schreiber) coordinates
    const double sxi = sin(xip), cxi = cos(xip), sheta = sinh(etap);
    const double taup = sxi / sqrt(sheta * sheta + cxi * cxi);       // tan of the conformal latitude
    const double lam = atan2(sheta, cxi);
    // conformal -> geodetic latitude: Newton on tau' (tau) = tau sqrt(1 + sigma^2) - sigma sqrt(1 + tau^2),
    // sigma = sinh(e atanh(e tau / sqrt(1 + tau^2))).  The start tau' / (1 - e^2) is O(e^4) off; three steps reach
    // the rounding floor.
    double tau = taup / p.e2m;
    for (int it = 0; it < 3; ++it) {
        const double t1 = sqrt(1.0 + tau * tau);
        const double sig = sinh(p.e * atanh(p.e * tau / t1));
        const double taupa = tau * sqrt(1.0 + sig * sig) - sig * t1;
        tau += (taup - taupa) * (1.0 + p.e2m * tau * tau) / (p.e2m * t1 * sqrt(1.0 + taupa * taupa));
    }
    const double r2d = 180.0 / 3.14159265358979323846;
    *lat = atan(tau) * r2d;
    *lon = p.lon0 + lam * r2d;
}

// Host: derive the projection constants.  Returns false for parameters that describe no ellipsoid.
inline bool tm_setup(const double* blk, TmParams* p)
{
    const double a = blk[0], f = blk[1], lat0 = blk[2], lon0 = blk[3], k0 = blk[4];
    if (!(a > 0.0) || !(f >= 0.0 && f < 1.0) || !(k0 > 0.0) || !std::isfinite(lat0) || !(std::fabs(lat0) <= 90.0) ||
        !std::isfinite(lon0) || !std::isfinite(blk[5]) || !std::isfinite(blk[6]))
        return false;
    const double n = f / (2.0 - f), n2 = n * n, n3 = n2 * n, n4 = n3 * n, n5 = n4 * n, n6 = n5 * n;
    const double e2 = f * (2.0 - f);
    p->A = a / (1.0 + n) * (1.0 + n2 / 4.0 + n4 / 64.0 + n6 / 256.0);
    p->k0 = k0; p->fe = blk[5]; p->fn = blk[6];
    p->lon0 = lon0;
    p->e = std::sqrt(e2); p->e2m = 1.0 - e2;
    p->beta[0] = n / 2.0 - 2.0 * n2 / 3.0 + 37.0 * n3 / 96.0 - n4 / 360.0 - 81.0 * n5 / 512.0 + 96199.0 * n6 / 604800.0;
    p->beta[1] = n2 / 48.0 + n3 / 15.0 - 437.0 * n4 / 1440.0 + 46.0 * n5 / 105.0 - 1118711.0 * n6 / 3870720.0;
    p->beta[2] = 17.0 * n3 / 480.0 - 37.0 * n4 / 840.0 - 209.0 * n5 / 4480.0 + 5569.0 * n6 / 90720.0;
    p->beta[3] = 4397.0 * n4 / 161280.0 - 11.0 * n5 / 504.0 - 830251.0 * n6 / 7257600.0;
    p->beta[4] = 4583.0 * n5 / 161280.0 - 108847.0 * n6 / 3991680.0;
    p->beta[5] = 20648693.0 * n6 / 638668800.0;
    p->alpha[0] = n / 2.0 - 2.0 * n2 / 3.0 + 5.0 * n3 / 16.0 + 41.0 * n4 / 180.0 - 127.0 * n5 / 288.0 + 7891.0 * n6 / 37800.0;
    p->alpha[1] = 13.0 * n2 / 48.0 - 3.0 * n3 / 5.0 + 557.0 * n4 / 1440.0 + 281.0 * n5 / 630.0 - 1983433.0 * n6 / 1935360.0;
    p->alpha[2] = 61.0 * n3 / 240.0 - 103.0 * n4 / 140.0 + 15061.0 * n5 / 26880.0 + 167603.0 * n6 / 181440.0;
    p->alpha[3] = 49561.0 * n4 / 161280.0 - 179.0 * n5 / 168.0 + 6601661.0 * n6 / 7257600.0;
    p->alpha[4] = 34729.0 * n5 / 80640.0 - 3418889.0 * n6 / 1995840.0;
    p->alpha[5] = 212378941.0 * n6 / 319334400.0;
    // rectifying latitude of lat0: the forward step on the central meridian (lam = 0, so eta' = 0 exactly)
    double eta0;
    tm_xi_eta(*p, lon0, lat0, &p->xi0, &eta0);
    return true;
}

}  // namespace

// Reprojection onto a fixed grid: utils_dem.resample_and_cut of the reference (utils_dem.py:65-84, gdal.Warp to EPSG:22184,
// 90 m Float32 pixels, cut to the area-of-interest envelope).  One output cell is independent of every other, so the kernel
// is a data-parallel map: destination pixel centre -> inverse Transverse Mercator (Krueger series to order n^6, Karney 2011,
// the formulation of PROJ's default tmerc) -> (lon, lat) -> source pixel coordinates -> nearest or bilinear sample.
// All coordinate arithmetic is float64 (the build's --fmad=false keeps it unfused).  The inverse projection is a
// __host__ __device__ function: hd_host_tm_inverse runs the very same code on the CPU for the host's footprint checks.
#include <cmath>

#include "common.cuh"

namespace {

// Everything the inverse projection needs, derived on the host from the (a, f, lat0, lon0, k0, FE, FN) block.
struct TmInv {
    double A;          // rectifying radius a / (1 + n) (1 + n^2/4 + n^4/64 + n^6/256)
    double k0, fe, fn;
    double xi0;        // rectifying latitude of lat0 (radians): M0 / A
    double lon0;       // degrees
    double e, e2m;     // eccentricity, 1 - e^2
    double beta[6];    // Krueger inverse coefficients
};

struct WarpGeo {
    double dx0, ddx, dy0, ddy;     // destination grid (top-left corner, pixel sizes)
    double sx0, sdx, sy0, sdy;     // source grid
    int64_t row0;                  // first destination row inside the grid dx0 / dy0 describe
    double nodata;
    int has_nodata;
    int project;                   // 0: the source is already in the destination CRS
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

// Projected (x, y) metres -> (lon, lat) degrees.
__host__ __device__ inline void tm_inverse(const TmInv& p, double x, double y, double* lon, double* lat)
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

// Host: derive the inverse-projection constants.  Returns false for parameters that describe no ellipsoid.
bool tm_setup(const double* blk, TmInv* p)
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
    // rectifying latitude of lat0 (forward series on the central meridian, eta' = 0)
    const double alpha[6] = {
        n / 2.0 - 2.0 * n2 / 3.0 + 5.0 * n3 / 16.0 + 41.0 * n4 / 180.0 - 127.0 * n5 / 288.0 + 7891.0 * n6 / 37800.0,
        13.0 * n2 / 48.0 - 3.0 * n3 / 5.0 + 557.0 * n4 / 1440.0 + 281.0 * n5 / 630.0 - 1983433.0 * n6 / 1935360.0,
        61.0 * n3 / 240.0 - 103.0 * n4 / 140.0 + 15061.0 * n5 / 26880.0 + 167603.0 * n6 / 181440.0,
        49561.0 * n4 / 161280.0 - 179.0 * n5 / 168.0 + 6601661.0 * n6 / 7257600.0,
        34729.0 * n5 / 80640.0 - 3418889.0 * n6 / 1995840.0,
        212378941.0 * n6 / 319334400.0};
    const double phi = lat0 * (3.14159265358979323846 / 180.0);
    const double tau = std::tan(phi);
    const double sig = std::sinh(p->e * std::atanh(p->e * std::sin(phi)));
    const double taup = tau * std::sqrt(1.0 + sig * sig) - sig * std::sqrt(1.0 + tau * tau);
    const double xip = std::atan2(taup, 1.0);
    double re, im;
    krueger_sum(alpha, xip, 0.0, &re, &im);
    p->xi0 = xip + re;
    return true;
}

template <typename S> __device__ __forceinline__ double load_src(const S* p) { return (double)__ldg(p); }

constexpr int WARP_THREADS = 128, WARP_CELLS = 4;                 // cells per thread, WARP_THREADS apart (coalesced stores)

template <typename S, bool BILINEAR>
__global__ void __launch_bounds__(WARP_THREADS) warp_kernel(const S* __restrict__ src, int64_t src_pitch, int64_t sny,
                                                            int64_t snx, float* __restrict__ dst, int64_t dst_pitch,
                                                            int64_t dny, int64_t dnx, const WarpGeo g, const TmInv tm)
{
    const double fill = g.has_nodata ? g.nodata : 0.0;
    const bool nd_nan = g.has_nodata && g.nodata != g.nodata;
    auto invalid = [&](double v) { return g.has_nodata && (v == g.nodata || (nd_nan && v != v)); };
    const int64_t xbase = (int64_t)blockIdx.x * (WARP_THREADS * WARP_CELLS) + threadIdx.x;
    for (int64_t j = blockIdx.y; j < dny; j += gridDim.y) {
        const double y = g.dy0 - ((double)(g.row0 + j) + 0.5) * g.ddy;
#pragma unroll
        for (int k = 0; k < WARP_CELLS; ++k) {
            const int64_t i = xbase + k * WARP_THREADS;
            if (i >= dnx) break;
            const double x = g.dx0 + ((double)i + 0.5) * g.ddx;
            double sx = x, sy = y;
            if (g.project) tm_inverse(tm, x, y, &sx, &sy);
            const double u = (sx - g.sx0) / g.sdx, v = (g.sy0 - sy) / g.sdy;
            double out = fill;
            if (!BILINEAR) {
                if (u >= 0.0 && u < (double)snx && v >= 0.0 && v < (double)sny)
                    out = load_src(src + (int64_t)floor(v) * src_pitch + (int64_t)floor(u));
            } else {
                const double fu = u - 0.5, fv = v - 0.5;
                const double x0 = floor(fu), y0 = floor(fv);
                const double ax = fu - x0, ay = fv - y0;
                double acc = 0.0, wsum = 0.0;
                // taps in the order (y0, x0), (y0, x0 + 1), (y0 + 1, x0), (y0 + 1, x0 + 1); NaN u / v fail every test
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const double tx = x0 + (double)(t & 1), ty = y0 + (double)(t >> 1);
                    if (!(tx >= 0.0 && tx < (double)snx && ty >= 0.0 && ty < (double)sny)) continue;
                    const double s = load_src(src + (int64_t)ty * src_pitch + (int64_t)tx);
                    if (invalid(s)) continue;
                    const double w = ((t >> 1) ? ay : 1.0 - ay) * ((t & 1) ? ax : 1.0 - ax);
                    acc += w * s;
                    wsum += w;
                }
                if (wsum > 0.0) out = acc / wsum;
            }
            dst[j * dst_pitch + i] = (float)out;
        }
    }
}

template <typename S>
int launch(const void* src, int64_t src_pitch, int64_t sny, int64_t snx, float* dst, int64_t dst_pitch, int64_t dny,
           int64_t dnx, const WarpGeo& g, const TmInv& tm, int resample, cudaStream_t s)
{
    const dim3 grid((unsigned)hd_cdiv(dnx, WARP_THREADS * WARP_CELLS), (unsigned)(dny < 65535 ? dny : 65535));
    if (resample == HD_WARP_NEAREST) {
        hd_prof_begin("warp_kernel_nearest", s);
        warp_kernel<S, false><<<grid, WARP_THREADS, 0, s>>>((const S*)src, src_pitch, sny, snx, dst, dst_pitch, dny, dnx, g, tm);
    } else {
        hd_prof_begin("warp_kernel_bilinear", s);
        warp_kernel<S, true><<<grid, WARP_THREADS, 0, s>>>((const S*)src, src_pitch, sny, snx, dst, dst_pitch, dny, dnx, g, tm);
    }
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

bool grid_ok(const double* geo)
{
    return std::isfinite(geo[0]) && std::isfinite(geo[2]) && geo[1] > 0.0 && geo[3] > 0.0 && std::isfinite(geo[1]) &&
           std::isfinite(geo[3]);
}

}  // namespace

extern "C" int hd_warp(const void* src, int src_dtype, int64_t src_pitch, int64_t src_ny, int64_t src_nx,
                       const double* src_geo, int has_nodata, double nodata, void* dst, int64_t dst_pitch, int64_t dst_ny,
                       int64_t dst_nx, const double* dst_geo, int64_t dst_row0, const double* tm, int resample, void* stream)
{
    if (!src || !dst || !src_geo || !dst_geo) return HD_ERR_NULL;
    if (src_ny < 1 || src_nx < 1 || dst_ny < 1 || dst_nx < 1 || src_pitch < src_nx || dst_pitch < dst_nx || dst_row0 < 0)
        return HD_ERR_ARG;
    if (!grid_ok(src_geo) || !grid_ok(dst_geo)) return HD_ERR_ARG;
    if (resample != HD_WARP_NEAREST && resample != HD_WARP_BILINEAR) return HD_ERR_ARG;
    WarpGeo g{dst_geo[0], dst_geo[1], dst_geo[2], dst_geo[3], src_geo[0], src_geo[1], src_geo[2], src_geo[3],
              dst_row0, nodata, has_nodata ? 1 : 0, tm ? 1 : 0};
    TmInv p{};
    if (tm && !tm_setup(tm, &p)) return HD_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    float* d = (float*)dst;
    switch (src_dtype) {
        case HD_U8: return launch<uint8_t>(src, src_pitch, src_ny, src_nx, d, dst_pitch, dst_ny, dst_nx, g, p, resample, s);
        case HD_I16: return launch<int16_t>(src, src_pitch, src_ny, src_nx, d, dst_pitch, dst_ny, dst_nx, g, p, resample, s);
        case HD_F32: return launch<float>(src, src_pitch, src_ny, src_nx, d, dst_pitch, dst_ny, dst_nx, g, p, resample, s);
        default: return HD_ERR_UNSUPPORTED;
    }
}

extern "C" int hd_host_tm_inverse(const double* tm, const double* x, const double* y, int64_t n, double* lon, double* lat)
{
    if (!tm || !x || !y || !lon || !lat) return HD_ERR_NULL;
    if (n < 0) return HD_ERR_ARG;
    TmInv p{};
    if (!tm_setup(tm, &p)) return HD_ERR_ARG;
    for (int64_t k = 0; k < n; ++k) tm_inverse(p, x[k], y[k], &lon[k], &lat[k]);
    return HD_OK;
}

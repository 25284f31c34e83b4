// Reprojection onto a fixed grid: utils_dem.resample_and_cut of the reference (utils_dem.py:65-84, gdal.Warp to EPSG:22184,
// 90 m Float32 pixels, cut to the area-of-interest envelope).  One output cell is independent of every other, so the kernel
// is a data-parallel map: destination pixel centre -> inverse Transverse Mercator (tmerc.cuh) -> (lon, lat) -> source
// pixel coordinates -> nearest or bilinear sample.  All coordinate arithmetic is float64.  hd_host_tm_inverse runs the
// same __host__ __device__ projection on the CPU for the host's footprint checks.
#include <cmath>

#include "common.cuh"
#include "tmerc.cuh"

namespace {

struct WarpGeo {
    double dx0, ddx, dy0, ddy;     // destination grid (top-left corner, pixel sizes)
    double sx0, sdx, sy0, sdy;     // source grid
    int64_t row0;                  // first destination row inside the grid dx0 / dy0 describe
    double nodata;
    int has_nodata;
    int project;                   // 0: the source is already in the destination CRS
};

template <typename S> __device__ __forceinline__ double load_src(const S* p) { return (double)__ldg(p); }

// nd_nan: the nodata value is NaN (computed once per thread, outside the cell loop)
__device__ __forceinline__ bool is_nodata(const WarpGeo& g, bool nd_nan, double v)
{
    return g.has_nodata && (v == g.nodata || (nd_nan && v != v));
}

constexpr int WARP_THREADS = 128, WARP_CELLS = 4;                 // cells per thread, WARP_THREADS apart (coalesced stores)

// A tap reader answers read(tx, ty, &s): does source pixel (tx, ty) (integer-valued doubles, or NaN / inf) hold a
// sample, and which.  warp_cell calls it for the nearest cell, or for each bilinear tap before its nodata test.

// One raster: inside its rectangle is a sample (a nodata value included; the bilinear path drops it).
template <typename S> struct RasterTaps {
    const S* __restrict__ src;
    int64_t pitch, ny, nx;
    __device__ __forceinline__ bool read(double tx, double ty, double& s) const
    {
        if (!(tx >= 0.0 && tx < (double)nx && ty >= 0.0 && ty < (double)ny)) return false;
        s = load_src(src + (int64_t)ty * pitch + (int64_t)tx);
        return true;
    }
};

// Mosaic index (hd_warp_mosaic): the bin grid of the selected sources' lattice extent, bins of bw x bh pixels from
// (iu0, iv0), and (u0, v0, u1, v1) the same extent in double for the range test that precedes every integer cast.
struct MosaicBins {
    double u0, v0, u1, v1;
    int64_t iu0, iv0, bw, bh, nbu;
};

// A virtual raster: the last listed source that contains the pixel and holds no nodata there.  Each bin lists the
// sources that meet it in descending list order, so the first hit of the walk is that source.
template <typename S> struct MosaicTaps {
    const int64_t* __restrict__ table;      // per source: device pointer, pitch, U, V, ny, nx
    const int64_t* __restrict__ start;      // CSR offsets, one per bin + 1
    const int64_t* __restrict__ list;       // source indices
    MosaicBins b;
    WarpGeo g;
    bool nd_nan;
    __device__ __forceinline__ bool read(double tx, double ty, double& s) const
    {
        if (!(tx >= b.u0 && tx < b.u1 && ty >= b.v0 && ty < b.v1)) return false;
        const int64_t U = (int64_t)tx, V = (int64_t)ty;
        const int64_t bin = (V - b.iv0) / b.bh * b.nbu + (U - b.iu0) / b.bw;
        const int64_t e = __ldg(start + bin + 1);
        for (int64_t k = __ldg(start + bin); k < e; ++k) {
            const int64_t* t = table + 6 * __ldg(list + k);
            const int64_t du = U - __ldg(t + 2), dv = V - __ldg(t + 3);
            if ((uint64_t)du >= (uint64_t)__ldg(t + 5) || (uint64_t)dv >= (uint64_t)__ldg(t + 4)) continue;
            const double v = load_src(reinterpret_cast<const S*>(__ldg(t)) + dv * __ldg(t + 1) + du);
            if (is_nodata(g, nd_nan, v)) continue;
            s = v;
            return true;
        }
        return false;
    }
};

// One destination cell, from its pixel centre (x, y): optional inverse projection -> source pixel coordinates (u, v) ->
// nearest cell or renormalised bilinear taps; no sample gives fill.  The only copy of the projection and the tap
// arithmetic; both kernels instantiate it.
template <bool BILINEAR, typename Taps>
__device__ __forceinline__ float warp_cell(const Taps& taps, const WarpGeo& g, const TmParams& tm, bool nd_nan,
                                           double fill, double x, double y)
{
    double sx = x, sy = y;
    if (g.project) tm_inverse(tm, x, y, &sx, &sy);
    const double u = (sx - g.sx0) / g.sdx, v = (g.sy0 - sy) / g.sdy;
    double out = fill;
    if (!BILINEAR) {
        double s;
        if (taps.read(floor(u), floor(v), s)) out = s;
    } else {
        const double fu = u - 0.5, fv = v - 0.5;
        const double x0 = floor(fu), y0 = floor(fv);
        const double ax = fu - x0, ay = fv - y0;
        double acc = 0.0, wsum = 0.0;
        // taps in the order (y0, x0), (y0, x0 + 1), (y0 + 1, x0), (y0 + 1, x0 + 1); NaN u / v fail every test
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const double tx = x0 + (double)(t & 1), ty = y0 + (double)(t >> 1);
            double s;
            if (!taps.read(tx, ty, s)) continue;
            if (is_nodata(g, nd_nan, s)) continue;
            const double w = ((t >> 1) ? ay : 1.0 - ay) * ((t & 1) ? ax : 1.0 - ax);
            acc += w * s;
            wsum += w;
        }
        if (wsum > 0.0) out = acc / wsum;
    }
    return (float)out;
}

// Destination cell (i, j) has centre (dx0 + (i + 1/2) ddx, dy0 - (row0 + j + 1/2) ddy).
template <bool BILINEAR, typename Taps>
__device__ __forceinline__ void warp_rows(const Taps& taps, bool nd_nan, float* __restrict__ dst, int64_t dst_pitch,
                                          int64_t dny, int64_t dnx, const WarpGeo& g, const TmParams& tm)
{
    const double fill = g.has_nodata ? g.nodata : 0.0;
    const int64_t xbase = (int64_t)blockIdx.x * (WARP_THREADS * WARP_CELLS) + threadIdx.x;
    for (int64_t j = blockIdx.y; j < dny; j += gridDim.y) {
        const double y = g.dy0 - ((double)(g.row0 + j) + 0.5) * g.ddy;
#pragma unroll
        for (int k = 0; k < WARP_CELLS; ++k) {
            const int64_t i = xbase + k * WARP_THREADS;
            if (i >= dnx) break;
            const double x = g.dx0 + ((double)i + 0.5) * g.ddx;
            dst[j * dst_pitch + i] = warp_cell<BILINEAR>(taps, g, tm, nd_nan, fill, x, y);
        }
    }
}

template <typename S, bool BILINEAR>
__global__ void __launch_bounds__(WARP_THREADS) warp_kernel(const S* __restrict__ src, int64_t src_pitch, int64_t sny,
                                                            int64_t snx, float* __restrict__ dst, int64_t dst_pitch,
                                                            int64_t dny, int64_t dnx, const WarpGeo g, const TmParams tm)
{
    const bool nd_nan = g.has_nodata && g.nodata != g.nodata;
    warp_rows<BILINEAR>(RasterTaps<S>{src, src_pitch, sny, snx}, nd_nan, dst, dst_pitch, dny, dnx, g, tm);
}

template <typename S, bool BILINEAR>
__global__ void __launch_bounds__(WARP_THREADS) warp_mosaic_kernel(const int64_t* __restrict__ table,
                                                                   const int64_t* __restrict__ start,
                                                                   const int64_t* __restrict__ list, const MosaicBins b,
                                                                   float* __restrict__ dst, int64_t dst_pitch,
                                                                   int64_t dny, int64_t dnx, const WarpGeo g,
                                                                   const TmParams tm)
{
    const bool nd_nan = g.has_nodata && g.nodata != g.nodata;
    warp_rows<BILINEAR>(MosaicTaps<S>{table, start, list, b, g, nd_nan}, nd_nan, dst, dst_pitch, dny, dnx, g, tm);
}

dim3 warp_grid(int64_t dny, int64_t dnx)
{
    return dim3((unsigned)hd_cdiv(dnx, WARP_THREADS * WARP_CELLS), (unsigned)(dny < 65535 ? dny : 65535));
}

template <typename S>
int launch(const void* src, int64_t src_pitch, int64_t sny, int64_t snx, float* dst, int64_t dst_pitch, int64_t dny,
           int64_t dnx, const WarpGeo& g, const TmParams& tm, int resample, cudaStream_t s)
{
    const dim3 grid = warp_grid(dny, dnx);
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

template <typename S>
int launch_mosaic(const int64_t* table, const int64_t* start, const int64_t* list, const MosaicBins& b, float* dst,
                  int64_t dst_pitch, int64_t dny, int64_t dnx, const WarpGeo& g, const TmParams& tm, int resample,
                  cudaStream_t s)
{
    const dim3 grid = warp_grid(dny, dnx);
    if (resample == HD_WARP_NEAREST) {
        hd_prof_begin("warp_mosaic_kernel_nearest", s);
        warp_mosaic_kernel<S, false><<<grid, WARP_THREADS, 0, s>>>(table, start, list, b, dst, dst_pitch, dny, dnx, g, tm);
    } else {
        hd_prof_begin("warp_mosaic_kernel_bilinear", s);
        warp_mosaic_kernel<S, true><<<grid, WARP_THREADS, 0, s>>>(table, start, list, b, dst, dst_pitch, dny, dnx, g, tm);
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
    TmParams p{};
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

extern "C" int hd_warp_mosaic(const int64_t* sources, int64_t n_sources, const int64_t* bin_start,
                              const int64_t* bin_list, const int64_t* bins, int src_dtype, const double* frame,
                              int has_nodata, double nodata, void* dst, int64_t dst_pitch, int64_t dst_ny, int64_t dst_nx,
                              const double* dst_geo, int64_t dst_row0, const double* tm, int resample, void* stream)
{
    if (!sources || !bin_start || !bin_list || !bins || !frame || !dst || !dst_geo) return HD_ERR_NULL;
    if (n_sources < 1 || dst_ny < 1 || dst_nx < 1 || dst_pitch < dst_nx || dst_row0 < 0) return HD_ERR_ARG;
    // bins: (iu0, iv0, bw, bh, nbu, nbv); the extent must stay exact in double for the range test
    constexpr int64_t lim = (int64_t)1 << 52;
    if (bins[2] < 1 || bins[3] < 1 || bins[4] < 1 || bins[5] < 1 || bins[4] > lim / bins[2] || bins[5] > lim / bins[3] ||
        bins[0] < -lim || bins[0] > lim || bins[1] < -lim || bins[1] > lim)
        return HD_ERR_ARG;
    if (!grid_ok(frame) || !grid_ok(dst_geo)) return HD_ERR_ARG;
    if (resample != HD_WARP_NEAREST && resample != HD_WARP_BILINEAR) return HD_ERR_ARG;
    WarpGeo g{dst_geo[0], dst_geo[1], dst_geo[2], dst_geo[3], frame[0], frame[1], frame[2], frame[3],
              dst_row0, nodata, has_nodata ? 1 : 0, tm ? 1 : 0};
    const MosaicBins b{(double)bins[0], (double)bins[1], (double)(bins[0] + bins[4] * bins[2]),
                       (double)(bins[1] + bins[5] * bins[3]), bins[0], bins[1], bins[2], bins[3], bins[4]};
    TmParams p{};
    if (tm && !tm_setup(tm, &p)) return HD_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    float* d = (float*)dst;
    switch (src_dtype) {
        case HD_U8: return launch_mosaic<uint8_t>(sources, bin_start, bin_list, b, d, dst_pitch, dst_ny, dst_nx, g, p, resample, s);
        case HD_I16: return launch_mosaic<int16_t>(sources, bin_start, bin_list, b, d, dst_pitch, dst_ny, dst_nx, g, p, resample, s);
        case HD_F32: return launch_mosaic<float>(sources, bin_start, bin_list, b, d, dst_pitch, dst_ny, dst_nx, g, p, resample, s);
        default: return HD_ERR_UNSUPPORTED;
    }
}

extern "C" int hd_host_tm_inverse(const double* tm, const double* x, const double* y, int64_t n, double* lon, double* lat)
{
    if (!tm || !x || !y || !lon || !lat) return HD_ERR_NULL;
    if (n < 0) return HD_ERR_ARG;
    TmParams p{};
    if (!tm_setup(tm, &p)) return HD_ERR_ARG;
    for (int64_t k = 0; k < n; ++k) tm_inverse(p, x[k], y[k], &lon[k], &lat[k]);
    return HD_OK;
}

extern "C" int hd_host_tm_forward(const double* tm, const double* lon, const double* lat, int64_t n, double* x, double* y)
{
    if (!tm || !lon || !lat || !x || !y) return HD_ERR_NULL;
    if (n < 0) return HD_ERR_ARG;
    TmParams p{};
    if (!tm_setup(tm, &p)) return HD_ERR_ARG;
    for (int64_t k = 0; k < n; ++k) tm_forward(p, lon[k], lat[k], &x[k], &y[k]);
    return HD_OK;
}

// Line rasterization onto a fixed grid: rasterize_rivers of the reference (utils_dem.py:183-191, gdal.RasterizeLayer of the
// HydroSHEDS river polylines with ATTRIBUTE=UP_CELLS), modelled on GDAL's default line burning (GDALdllImageLine, no
// ALL_TOUCHED, MERGE_ALG=REPLACE).  The contract is DESIGN.md §9b.
//
//   project_kernel   one thread per vertex: optional forward Transverse Mercator (tmerc.cuh), pixel coordinates
//                    ((X - x0) / dx, (y0 - Y) / dy) in the full grid's frame, floored to int32 (or "no vertex").
//   count_kernel     one thread per vertex i = the segment (i, i + 1) of its part: the interval of Bresenham steps whose
//                    pixel lies inside the destination rows, in closed form (no walk), and the tag feature + 1.
//   scan_*           a three-pass inclusive scan of those counts (block sums, scan of the block sums, block scans).
//   burn_kernel      persistent: every thread takes one in-grid step at a time, finds its segment by binary search over
//                    the scan, computes its pixel in closed form and atomicMax-es the tag into the destination viewed as
//                    uint32.  The largest tag is the last feature in file order: REPLACE, deterministic.
//   resolve_kernel   tag -> the feature's value (0 stays 0.0f), in place.
//
// Work per thread does not depend on segment length, the total step count stays on the device (no host sync), nothing is
// allocated: the call is capturable in a CUDA graph.
#include <climits>
#include <cmath>

#include "common.cuh"
#include "tmerc.cuh"

namespace {

constexpr double PIX_LIMIT = 536870912.0;        // 2^29: pixel coordinates at or beyond it count as no vertex
constexpr int32_t NO_PIX = INT32_MIN;
constexpr int THREADS = 256;
constexpr int SCAN_ITEMS = 8, SCAN_TILE = THREADS * SCAN_ITEMS;
constexpr int64_t MAX_VERTICES = int64_t(1) << 38;          // one thread per vertex: < 2^31 blocks

struct RasterGeo {
    double x0, dx, y0, dy;
    int64_t row0, ny, nx;
};

// One segment's Bresenham walk (GDALdllImageLine) between floored endpoints, on its major axis u and minor axis v:
// step k = 0 ... amaj is the pixel u0 + su k, v0 + sv m(k) with m(k) = floor((2 k amin + amaj - 1) / (2 amaj)).
struct Walk {
    int64_t u0, v0, amaj, amin;
    int su, sv;
    bool xmajor;
};

__device__ __forceinline__ Walk make_walk(int2 a, int2 b)
{
    const int64_t dx = (int64_t)b.x - a.x, dy = (int64_t)b.y - a.y;
    const int64_t adx = dx < 0 ? -dx : dx, ady = dy < 0 ? -dy : dy;
    Walk w;
    w.xmajor = adx >= ady;
    if (w.xmajor) { w.u0 = a.x; w.v0 = a.y; w.amaj = adx; w.amin = ady; w.su = dx < 0 ? -1 : 1; w.sv = dy < 0 ? -1 : 1; }
    else          { w.u0 = a.y; w.v0 = a.x; w.amaj = ady; w.amin = adx; w.su = dy < 0 ? -1 : 1; w.sv = dx < 0 ? -1 : 1; }
    return w;
}

__device__ __forceinline__ int64_t minor_offset(const Walk& w, int64_t k)
{
    return w.amaj ? (2 * k * w.amin + w.amaj - 1) / (2 * w.amaj) : 0;
}

// The first step k with m(k) >= M (amaj + 1 when there is none).  |coordinates| < 2^29 keeps every product below 2^62.
__device__ __forceinline__ int64_t first_step(const Walk& w, int64_t M)
{
    if (M <= 0) return 0;
    if (M > w.amin) return w.amaj + 1;
    const int64_t num = 2 * M * w.amaj - w.amaj + 1, den = 2 * w.amin;     // amin >= M >= 1
    return (num + den - 1) / den;
}

// The steps [k0, k1] whose pixel is inside columns [0, nx) and rows [row0, row0 + ny): u and m(k) are monotone in k, so
// the set is one interval.  False when it is empty.
__device__ __forceinline__ bool in_grid_steps(const Walk& w, const RasterGeo& g, int64_t* k0, int64_t* k1)
{
    const int64_t ulo = w.xmajor ? 0 : g.row0, uhi = w.xmajor ? g.nx - 1 : g.row0 + g.ny - 1;
    const int64_t vlo = w.xmajor ? g.row0 : 0, vhi = w.xmajor ? g.row0 + g.ny - 1 : g.nx - 1;
    int64_t a = w.su > 0 ? ulo - w.u0 : w.u0 - uhi, b = w.su > 0 ? uhi - w.u0 : w.u0 - ulo;
    const int64_t mlo = w.sv > 0 ? vlo - w.v0 : w.v0 - vhi, mhi = w.sv > 0 ? vhi - w.v0 : w.v0 - vlo;
    a = max(a, max((int64_t)0, first_step(w, mlo)));
    b = min(b, min(w.amaj, first_step(w, mhi + 1) - 1));
    *k0 = a; *k1 = b;
    return a <= b;
}

__global__ void __launch_bounds__(THREADS) project_kernel(const double* __restrict__ vx, const double* __restrict__ vy,
                                                          int64_t n, const RasterGeo g, const TmParams tm, int project,
                                                          int2* __restrict__ pix)
{
    const int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x;
    if (i < n) {
        double X = vx[i], Y = vy[i];
        if (project) {
            if (fabs(Y) <= 90.0) tm_forward(tm, X, Y, &X, &Y);
            else X = NAN;                                            // beyond a pole (or NaN): no vertex
        }
        const double px = (X - g.x0) / g.dx, py = (g.y0 - Y) / g.dy;
        int2 p = make_int2(NO_PIX, NO_PIX);
        if (fabs(px) < PIX_LIMIT && fabs(py) < PIX_LIMIT) p = make_int2((int)floor(px), (int)floor(py));
        pix[i] = p;
    }
}

// seg[i] = (first in-grid step, feature + 1) of the segment that starts at vertex i; count[i] = its in-grid steps.
__global__ void __launch_bounds__(THREADS) count_kernel(const int2* __restrict__ pix, int64_t n,
                                                        const int64_t* __restrict__ part_start, int64_t n_parts,
                                                        const int32_t* __restrict__ part_feature, int64_t n_features,
                                                        const RasterGeo g, int64_t* __restrict__ count, int2* __restrict__ seg)
{
    const int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x;
    if (i < n) {
        // the part of vertex i: the last p < n_parts with part_start[p] <= i (empty parts share a start with the next)
        int64_t lo = 0, hi = n_parts;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (part_start[mid] <= i) lo = mid + 1; else hi = mid;
        }
        const int64_t p = lo - 1;
        int64_t c = 0, k0 = 0, k1 = -1;
        uint32_t tag = 0;
        if (p >= 0 && i + 1 < n && i + 1 < part_start[p + 1]) {
            const int32_t f = part_feature[p];
            const int2 a = pix[i], b = pix[i + 1];
            if (f >= 0 && f < n_features && a.x != NO_PIX && b.x != NO_PIX && in_grid_steps(make_walk(a, b), g, &k0, &k1)) {
                c = k1 - k0 + 1;
                tag = (uint32_t)f + 1u;
            }
        }
        count[i] = c;
        seg[i] = make_int2((int)k0, (int)tag);
    }
}

// Exclusive scan of one value per thread over the block; *total = the block's sum.  Ends with a barrier (smem reusable).
__device__ __forceinline__ int64_t block_exclusive_scan(int64_t v, int64_t* warp_sums, int64_t* total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        int64_t s = lane < THREADS / 32 ? warp_sums[lane] : 0;
#pragma unroll
        for (int o = 1; o < THREADS / 32; o <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        if (lane < THREADS / 32) warp_sums[lane] = s;
    }
    __syncthreads();
    const int64_t out = (wid ? warp_sums[wid - 1] : 0) + x - v;
    *total = warp_sums[THREADS / 32 - 1];
    __syncthreads();
    return out;
}

// Pass 1: the sum of each SCAN_TILE-element tile.
__global__ void __launch_bounds__(THREADS) scan_tile_sums(const int64_t* __restrict__ count, int64_t n,
                                                          int64_t* __restrict__ tile_sum)
{
    __shared__ int64_t warp_sums[THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int64_t s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j)
        if (base + j < n) s += count[base + j];
    int64_t total;
    block_exclusive_scan(s, warp_sums, &total);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

// Pass 2 (one block): tile sums -> exclusive tile offsets, in place.
__global__ void __launch_bounds__(THREADS) scan_tile_offsets(int64_t* __restrict__ tile_sum, int64_t ntiles)
{
    __shared__ int64_t warp_sums[THREADS / 32];
    int64_t carry = 0;
    for (int64_t base = 0; base < ntiles; base += THREADS) {
        const int64_t i = base + threadIdx.x;
        const int64_t v = i < ntiles ? tile_sum[i] : 0;
        int64_t total;
        const int64_t ex = block_exclusive_scan(v, warp_sums, &total);
        if (i < ntiles) tile_sum[i] = carry + ex;
        carry += total;
    }
}

// Pass 3: counts -> inclusive ends, in place.
__global__ void __launch_bounds__(THREADS) scan_tiles(int64_t* __restrict__ count, int64_t n,
                                                      const int64_t* __restrict__ tile_off)
{
    __shared__ int64_t warp_sums[THREADS / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
    int64_t v[SCAN_ITEMS], s = 0;
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        v[j] = base + j < n ? count[base + j] : 0;
        s += v[j];
    }
    int64_t total;
    int64_t run = tile_off[blockIdx.x] + block_exclusive_scan(s, warp_sums, &total);
#pragma unroll
    for (int j = 0; j < SCAN_ITEMS; ++j) {
        run += v[j];
        if (base + j < n) count[base + j] = run;
    }
}

// The segment of global step t: the first i in [lo, hi] with ends[i] > t (one exists: ends[hi] > t).
__device__ __forceinline__ int64_t segment_of(const int64_t* __restrict__ ends, int64_t lo, int64_t hi, int64_t t)
{
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (ends[mid] > t) hi = mid; else lo = mid + 1;
    }
    return lo;
}

__global__ void __launch_bounds__(THREADS) burn_kernel(const int64_t* __restrict__ ends, int64_t n,
                                                       const int2* __restrict__ pix, const int2* __restrict__ seg,
                                                       const RasterGeo g, uint32_t* __restrict__ dst, int64_t pitch)
{
    __shared__ int64_t range[2];
    const int64_t total = ends[n - 1];
    // each block takes THREADS consecutive steps at a time; their segments lie in [range[0], range[1]]
    for (int64_t base = (int64_t)blockIdx.x * THREADS; base < total; base += (int64_t)gridDim.x * THREADS) {
        const int64_t last = min(base + THREADS, total) - 1;
        if (threadIdx.x == 0) range[0] = segment_of(ends, 0, n - 1, base);
        if (threadIdx.x == 32) range[1] = segment_of(ends, 0, n - 1, last);
        __syncthreads();
        const int64_t lo = range[0], hi = range[1];
        __syncthreads();
        const int64_t t = base + threadIdx.x;
        if (t > last) continue;
        const int64_t i = segment_of(ends, lo, hi, t);
        const int2 s = seg[i];
        const Walk w = make_walk(pix[i], pix[i + 1]);
        const int64_t k = t - (i ? ends[i - 1] : 0) + s.x;
        const int64_t u = w.u0 + w.su * k, v = w.v0 + w.sv * minor_offset(w, k);
        const int64_t x = w.xmajor ? u : v, y = w.xmajor ? v : u;
        atomicMax(dst + (y - g.row0) * pitch + x, (uint32_t)s.y);
    }
}

__global__ void __launch_bounds__(THREADS) resolve_kernel(float* __restrict__ dst, int64_t pitch, int64_t ny, int64_t nx,
                                                          const float* __restrict__ values)
{
    for (int64_t j = blockIdx.y; j < ny; j += gridDim.y)
        for (int64_t i = (int64_t)blockIdx.x * THREADS + threadIdx.x; i < nx; i += (int64_t)gridDim.x * THREADS) {
            float* p = dst + j * pitch + i;
            const uint32_t tag = __float_as_uint(*p);
            *p = tag ? __ldg(values + tag - 1) : 0.0f;
        }
}

constexpr int64_t align256(int64_t b) { return (b + 255) / 256 * 256; }

struct Layout {
    int64_t pix, ends, seg, tiles, total;
};

Layout layout(int64_t n)
{
    Layout l;
    l.pix = 0;
    l.ends = l.pix + align256(n * (int64_t)sizeof(int2));
    l.seg = l.ends + align256(n * (int64_t)sizeof(int64_t));
    l.tiles = l.seg + align256(n * (int64_t)sizeof(int2));
    l.total = l.tiles + align256((n + SCAN_TILE - 1) / SCAN_TILE * (int64_t)sizeof(int64_t));
    return l;
}

bool grid_ok(const double* geo)
{
    return std::isfinite(geo[0]) && std::isfinite(geo[2]) && geo[1] > 0.0 && geo[3] > 0.0 && std::isfinite(geo[1]) &&
           std::isfinite(geo[3]);
}

}  // namespace

extern "C" int64_t hd_rasterize_workspace_bytes(int64_t n_vertices)
{
    if (n_vertices < 0 || n_vertices > MAX_VERTICES) return 0;
    return layout(n_vertices).total;
}

extern "C" int hd_rasterize_lines(const void* vx, const void* vy, int64_t n_vertices, const void* part_start,
                                  const void* part_feature, int64_t n_parts, const void* values, int64_t n_features,
                                  void* dst, int64_t dst_pitch, int64_t dst_ny, int64_t dst_nx, const double* dst_geo,
                                  int64_t dst_row0, const double* tm, void* workspace, int64_t workspace_bytes, void* stream)
{
    if (!dst || !dst_geo || !part_start) return HD_ERR_NULL;
    if ((n_vertices > 0 && (!vx || !vy || !workspace)) || (n_parts > 0 && !part_feature) || (n_features > 0 && !values))
        return HD_ERR_NULL;
    if (n_vertices < 0 || n_vertices > MAX_VERTICES || n_parts < 0 || n_features < 0 || n_features > INT32_MAX)
        return HD_ERR_ARG;
    if (dst_ny < 1 || dst_nx < 1 || dst_pitch < dst_nx || dst_row0 < 0 || dst_nx > (int64_t)PIX_LIMIT ||
        dst_row0 + dst_ny > (int64_t)PIX_LIMIT || !grid_ok(dst_geo))
        return HD_ERR_ARG;
    TmParams p{};
    if (tm && !tm_setup(tm, &p)) return HD_ERR_ARG;
    const Layout l = layout(n_vertices);
    if (n_vertices > 0 && workspace_bytes < l.total) return HD_ERR_WORKSPACE;

    cudaStream_t s = (cudaStream_t)stream;
    HD_CUDA_OK(cudaMemset2DAsync(dst, dst_pitch * sizeof(float), 0, dst_nx * sizeof(float), dst_ny, s));
    if (n_vertices < 2 || n_parts == 0 || n_features == 0) return HD_OK;   // no segment: every cell 0

    const RasterGeo g{dst_geo[0], dst_geo[1], dst_geo[2], dst_geo[3], dst_row0, dst_ny, dst_nx};
    char* ws = (char*)workspace;
    int2* pix = (int2*)(ws + l.pix);
    int64_t* ends = (int64_t*)(ws + l.ends);
    int2* seg = (int2*)(ws + l.seg);
    int64_t* tiles = (int64_t*)(ws + l.tiles);
    const int64_t ntiles = (n_vertices + SCAN_TILE - 1) / SCAN_TILE;

    hd_prof_begin("rasterize_project", s);
    project_kernel<<<(unsigned)((n_vertices + THREADS - 1) / THREADS), THREADS, 0, s>>>((const double*)vx, (const double*)vy, n_vertices, g, p,
                                                           tm ? 1 : 0, pix);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    hd_prof_begin("rasterize_count", s);
    count_kernel<<<(unsigned)((n_vertices + THREADS - 1) / THREADS), THREADS, 0, s>>>(pix, n_vertices, (const int64_t*)part_start, n_parts,
                                                         (const int32_t*)part_feature, n_features, g, ends, seg);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    hd_prof_begin("rasterize_scan", s);
    scan_tile_sums<<<(unsigned)ntiles, THREADS, 0, s>>>(ends, n_vertices, tiles);
    HD_LAUNCH_CHECK();
    scan_tile_offsets<<<1, THREADS, 0, s>>>(tiles, ntiles);
    HD_LAUNCH_CHECK();
    scan_tiles<<<(unsigned)ntiles, THREADS, 0, s>>>(ends, n_vertices, tiles);
    HD_LAUNCH_CHECK();
    hd_count_launch(3);
    hd_prof_begin("rasterize_burn", s);
    burn_kernel<<<(unsigned)hd_num_sms() * 8, THREADS, 0, s>>>(ends, n_vertices, pix, seg, g, (uint32_t*)dst, dst_pitch);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    hd_prof_begin("rasterize_resolve", s);
    const dim3 rg((unsigned)hd_cdiv(dst_nx, THREADS * 4) , (unsigned)(dst_ny < 65535 ? dst_ny : 65535));
    resolve_kernel<<<rg, THREADS, 0, s>>>((float*)dst, dst_pitch, dst_ny, dst_nx, (const float*)values);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

// Shared pieces of the 32x128-tile stencil kernels: vector stores, reflect patching, launch helpers.
#pragma once
#include "common.cuh"

constexpr int TH = 32, TW = 128, NT = 256;

#ifdef __CUDACC__
template <typename T> __device__ __forceinline__ void store4(T* p, int64_t pitch, int64_t y, int64_t x, int64_t nx,
                                                             const float (&v)[4]);
template <> __device__ __forceinline__ void store4<float>(float* p, int64_t pitch, int64_t y, int64_t x, int64_t nx,
                                                          const float (&v)[4])
{
    float* q = p + y * pitch + x;
    if (x + 3 < nx && ((pitch & 3) == 0) && ((((uintptr_t)p) & 15) == 0)) {
        st_cs_f32x4(q, v[0], v[1], v[2], v[3]);
    } else {
        for (int j = 0; j < 4; ++j)
            if (x + j < nx) q[j] = v[j];
    }
}
template <> __device__ __forceinline__ void store4<double>(double* p, int64_t pitch, int64_t y, int64_t x, int64_t nx,
                                                           const float (&v)[4])
{
    double* q = p + y * pitch + x;
    if (x + 3 < nx && ((pitch & 1) == 0) && ((((uintptr_t)p) & 15) == 0)) {
        reinterpret_cast<double2*>(q)[0] = make_double2((double)v[0], (double)v[1]);
        reinterpret_cast<double2*>(q)[1] = make_double2((double)v[2], (double)v[3]);
    } else {
        for (int j = 0; j < 4; ++j)
            if (x + j < nx) q[j] = (double)v[j];
    }
}
template <> __device__ __forceinline__ void store4<uint8_t>(uint8_t* p, int64_t pitch, int64_t y, int64_t x, int64_t nx,
                                                            const float (&v)[4])
{
    uint8_t* q = p + y * pitch + x;
    if (x + 3 < nx && ((pitch & 3) == 0) && ((((uintptr_t)p) & 3) == 0)) {
        *reinterpret_cast<uchar4*>(q) = make_uchar4((uint8_t)v[0], (uint8_t)v[1], (uint8_t)v[2], (uint8_t)v[3]);
    } else {
        for (int j = 0; j < 4; ++j)
            if (x + j < nx) q[j] = (uint8_t)v[j];
    }
}

// same-dtype vector store of 4 consecutive cells
template <typename T> __device__ __forceinline__ void store4v(T* p, int64_t pitch, int64_t y, int64_t x, int64_t nx,
                                                              const T (&v)[4]);
template <> __device__ __forceinline__ void store4v<float>(float* p, int64_t pitch, int64_t y, int64_t x, int64_t nx,
                                                           const float (&v)[4])
{
    store4<float>(p, pitch, y, x, nx, v);
}
template <> __device__ __forceinline__ void store4v<double>(double* p, int64_t pitch, int64_t y, int64_t x, int64_t nx,
                                                            const double (&v)[4])
{
    double* q = p + y * pitch + x;
    if (x + 3 < nx && ((pitch & 1) == 0) && ((((uintptr_t)p) & 15) == 0)) {
        reinterpret_cast<double2*>(q)[0] = make_double2(v[0], v[1]);
        reinterpret_cast<double2*>(q)[1] = make_double2(v[2], v[3]);
    } else {
        for (int j = 0; j < 4; ++j)
            if (x + j < nx) q[j] = v[j];
    }
}

template <> __device__ __forceinline__ void store4v<uint8_t>(uint8_t* p, int64_t pitch, int64_t y, int64_t x, int64_t nx,
                                                             const uint8_t (&v)[4])
{
    uint8_t* q = p + y * pitch + x;
    if (x + 3 < nx && ((reinterpret_cast<uintptr_t>(q) & 3) == 0)) {
        *reinterpret_cast<uint32_t*>(q) = (uint32_t)v[0] | ((uint32_t)v[1] << 8) | ((uint32_t)v[2] << 16) | ((uint32_t)v[3] << 24);
    } else {
        for (int j = 0; j < 4; ++j)
            if (x + j < nx) q[j] = v[j];
    }
}

// four consecutive cells starting at p (column x of a row of nx cells) straight from global memory; cells past the
// end of the row read as 0.  One 16-byte load when the address allows it.
__device__ __forceinline__ void gload4(const float* p, int64_t x, int64_t nx, float (&v)[4])
{
    if (x + 3 < nx && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (x + j < nx) ? __ldg(p + j) : 0.f;
    }
}
__device__ __forceinline__ void gload4(const double* p, int64_t x, int64_t nx, double (&v)[4])
{
    if (x + 3 < nx && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
        const double2 a = __ldg(reinterpret_cast<const double2*>(p)), b = __ldg(reinterpret_cast<const double2*>(p) + 1);
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (x + j < nx) ? __ldg(p + j) : 0.0;
    }
}

__device__ __forceinline__ int reflect_idx(int64_t i, int64_t n)
{
    if (i < 0) i = -i - 1;
    if (i >= n) i = 2 * n - 1 - i;
    return (int)i;
}

// mode='reflect' for any distance from the raster (d c b a | a b c d | d c b a | a b ...): the extension repeats with
// period 2n, so windows wider than the raster wrap as often as they need.  reflect_idx is its first period only.
__device__ __forceinline__ int reflect_periodic_idx(int64_t i, int64_t n)
{
    int64_t m = i % (2 * n);
    if (m < 0) m += 2 * n;
    return (int)(m < n ? m : 2 * n - 1 - m);
}

// PERIODIC = false: one reflection (halo <= raster size); true: reflect_periodic_idx.  Every cell outside the raster is
// copied from a cell inside it, and that cell lies in the staged box whenever an output of the tile needs it.
template <typename T, bool PERIODIC = false>
__device__ __forceinline__ void patch_reflect(T* tile, int in_w, int in_h, int gy0, int gx0, int64_t ny, int64_t nx)
{
    const bool touches = gy0 < 0 || gx0 < 0 || gy0 + in_h > ny || gx0 + in_w > nx;
    if (!touches) return;
    for (int t = threadIdx.x; t < in_w * in_h; t += NT) {
        const int r = t / in_w, c = t - r * in_w;
        const int64_t gy = gy0 + r, gx = gx0 + c;
        if (gy >= 0 && gy < ny && gx >= 0 && gx < nx) continue;
        const int sy = (PERIODIC ? reflect_periodic_idx(gy, ny) : reflect_idx(gy, ny)) - gy0;
        const int sx = (PERIODIC ? reflect_periodic_idx(gx, nx) : reflect_idx(gx, nx)) - gx0;
        if (sy >= 0 && sy < in_h && sx >= 0 && sx < in_w) tile[t] = tile[sy * in_w + sx];
    }
    __syncthreads();
}

#endif  // __CUDACC__

static inline int grid_for(int ntiles, int ctas_per_sm)
{
    const int cap = hd_num_sms() * ctas_per_sm;
    return ntiles < cap ? ntiles : cap;
}

static inline int check_window(int64_t ny, int64_t nx, int ws)
{
    if (ws > ny || ws > nx) return HD_ERR_WINDOW_HIGH;   // sliding_window.py:152-153 (tested first)
    if (ws % 2 != 1) return HD_ERR_WINDOW_EVEN;          // :154-155
    return HD_OK;
}


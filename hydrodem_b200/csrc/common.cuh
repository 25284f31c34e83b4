// hydrodem_b200 -- shared device/host helpers for the sm_100a kernels.
//
// Tile staging: every windowed filter loads "tile + halo" boxes into shared
// memory with TMA (cp.async.bulk.tensor.2d, completion on an mbarrier) from a
// persistent grid, double buffered: while the CTA computes tile k the TMA unit
// is already filling the buffer for tile k+1.  Out-of-image box cells are
// filled by the TMA unit (zero, or NaN when the map asks for it), so kernels
// never branch on the image edge while loading.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/hydrodem_b200.h"

#define HD_CUDA_OK(expr)                                         \
    do {                                                         \
        cudaError_t _e = (expr);                                 \
        if (_e != cudaSuccess) { hd_set_last_cuda_error((int)_e); return HD_ERR_CUDA; } \
    } while (0)

#define HD_LAUNCH_CHECK()                                        \
    do {                                                         \
        cudaError_t _e = cudaGetLastError();                     \
        if (_e != cudaSuccess) { hd_set_last_cuda_error((int)_e); return HD_ERR_CUDA; } \
    } while (0)

void hd_set_last_cuda_error(int e);
void hd_count_launch(int n = 1);
// per-launch profiling hook: call right before a kernel launch; hd_count_launch() closes the record
void hd_prof_begin(const char* name, cudaStream_t stream);

// Host: encode a 2-D tiled tensor map over a pitched row-major raster.
// dtype: HD_U8 / HD_F32 / HD_F64 / HD_I32, or HD_C64 (encoded as 64-bit integers: the bits are moved, no NaN fill).
// swizzle128: CU_TENSOR_MAP_SWIZZLE_128B (box rows of at most 128 bytes; the shared-memory destination then wants
// 1024-byte alignment).
// Returns HD_OK or an error code (HD_ERR_ALIGN when base / pitch break the 16-byte TMA rules).
int hd_make_tmap_2d(CUtensorMap* out, const void* base, int dtype, int64_t ny, int64_t nx, int64_t pitch_elems,
                    int box_w, int box_h, bool nan_fill, bool swizzle128 = false);

int hd_num_sms();          // SMs persistent grids are sized for (HD_SM_RESERVE leaves some to communication kernels)
int hd_num_sms_total();
size_t hd_dtype_size(int dtype);

static inline int hd_cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }
// x halo rounded up to a 16-byte multiple for elements of `es` bytes
__host__ __device__ constexpr int hd_halo_x(int h, int es) { return (h * es + 15) / 16 * 16 / es; }

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------
// device side
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t done;
    const uint32_t addr = smem_u32(bar);
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}
// box whose top-left element is (x, y); coordinates may be negative / past the edge (OOB fill).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, int x, int y, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"((uint64_t)tm), "r"(smem_u32(bar)), "r"(x), "r"(y)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)tm) : "memory");
}

// One input plane of a staged tile.
// TMA rule (measured on B200, tools/probe/tma_probe.cu): the innermost box coordinate times the element size
// must be a multiple of 16 bytes, otherwise the load traps with "illegal instruction".  Row coordinates are
// free.  So the x halo of a plane is rounded up to 16 bytes (hd_halo_x) and kernels index the staged tile
// with the offset hd_halo_x(h) - h.
struct TilePlane {
    const CUtensorMap* tm;   // tensor map (kernel __grid_constant__ parameter)
    uint32_t smem_off;       // byte offset of this plane inside a stage (128-byte aligned)
    uint32_t bytes;          // box bytes (box_w * box_h * elem)
    int halo_x, halo_y;      // box origin = tile origin - halo
};

// Persistent TMA tile loop, NSTAGE = 2 (double buffered, default) or 1.  All threads of the CTA call it.
//   stage s of the ring lives at smem + s * stage_bytes; bars[0..1] are the "full" barriers.
//   body(stage_ptr, tile_y0, tile_x0) runs with the tile resident; it must not __syncthreads-diverge.
//   With NSTAGE = 1 (kernels whose scratch leaves no room for a second buffer) the next load is issued
//   after the body; latency is then hidden only by other resident CTAs.
template <int NPLANES, int NSTAGE = 2, class Body>
__device__ __forceinline__ void tile_loop(unsigned char* smem, uint32_t stage_bytes, uint64_t* bars,
                                          const TilePlane (&planes)[NPLANES], int tile_w, int tile_h, int tiles_x,
                                          int ntiles, Body&& body)
{
    static_assert(NSTAGE == 1 || NSTAGE == 2, "one or two stages");
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
#pragma unroll
        for (int p = 0; p < NPLANES; ++p) tma_prefetch_desc(planes[p].tm);
    }
    __syncthreads();
    uint32_t total = 0;
#pragma unroll
    for (int p = 0; p < NPLANES; ++p) total += planes[p].bytes;

    auto issue = [&](int tile, int s) {
        const int ty0 = (tile / tiles_x) * tile_h, tx0 = (tile % tiles_x) * tile_w;
        mbar_arrive_expect_tx(&bars[s], total);
#pragma unroll
        for (int p = 0; p < NPLANES; ++p)
            tma_load_2d(smem + s * stage_bytes + planes[p].smem_off, planes[p].tm, tx0 - planes[p].halo_x,
                        ty0 - planes[p].halo_y, &bars[s]);
    };
    int tile = blockIdx.x;
    if (threadIdx.x == 0 && tile < ntiles) issue(tile, 0);
    for (int k = 0; tile < ntiles; ++k, tile += gridDim.x) {
        const int s = NSTAGE == 2 ? (k & 1) : 0;
        const int next = tile + gridDim.x;
        // buffer s^1 was released by the __syncthreads that ended iteration k-1
        if (NSTAGE == 2 && threadIdx.x == 0 && next < ntiles) issue(next, s ^ 1);
        mbar_wait(&bars[s], NSTAGE == 2 ? ((k >> 1) & 1) : (k & 1));
        body(smem + s * stage_bytes, (tile / tiles_x) * tile_h, (tile % tiles_x) * tile_w);
        __syncthreads();
        if (NSTAGE == 1 && threadIdx.x == 0 && next < ntiles) issue(next, 0);
    }
}

// tile_loop over the tiles whose flag is set (flags[tile] != 0), same double-buffered TMA pipeline: a skipped tile costs one
// byte of flag traffic -- no tile load, no body, no store.  All threads walk the flag array identically.
template <int NPLANES, class Body>
__device__ __forceinline__ void tile_loop_flagged(unsigned char* smem, uint32_t stage_bytes, uint64_t* bars,
                                                  const TilePlane (&planes)[NPLANES], int tile_w, int tile_h, int tiles_x,
                                                  int ntiles, const uint8_t* __restrict__ flags, Body&& body)
{
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        mbar_fence_init();
#pragma unroll
        for (int p = 0; p < NPLANES; ++p) tma_prefetch_desc(planes[p].tm);
    }
    __syncthreads();
    uint32_t total = 0;
#pragma unroll
    for (int p = 0; p < NPLANES; ++p) total += planes[p].bytes;
    auto issue = [&](int tile, int s) {
        const int ty0 = (tile / tiles_x) * tile_h, tx0 = (tile % tiles_x) * tile_w;
        mbar_arrive_expect_tx(&bars[s], total);
#pragma unroll
        for (int p = 0; p < NPLANES; ++p)
            tma_load_2d(smem + s * stage_bytes + planes[p].smem_off, planes[p].tm, tx0 - planes[p].halo_x,
                        ty0 - planes[p].halo_y, &bars[s]);
    };
    auto next_flagged = [&](int tile) {                       // first flagged tile of this CTA's sequence at or after `tile`
        while (tile < ntiles && __ldg(flags + tile) == 0) tile += gridDim.x;
        return tile;
    };
    int tile = next_flagged(blockIdx.x);
    if (threadIdx.x == 0 && tile < ntiles) issue(tile, 0);
    for (int k = 0; tile < ntiles; ++k) {
        const int s = k & 1;
        const int next = next_flagged(tile + gridDim.x);
        if (threadIdx.x == 0 && next < ntiles) issue(next, s ^ 1);
        mbar_wait(&bars[s], (k >> 1) & 1);
        body(smem + s * stage_bytes, (tile / tiles_x) * tile_h, (tile % tiles_x) * tile_w, tile);
        __syncthreads();
        tile = next;
    }
}

__device__ __forceinline__ bool hd_isnan(float v) { return v != v; }

// streaming (evict-first) vector stores for outputs that are written once
__device__ __forceinline__ void st_cs_f32x4(float* p, float a, float b, float c, float d)
{
    asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Row-major walk over the cells of a raster for the 1-D grid-stride streaming kernels: the (row, column) pair is
// advanced by the grid stride with one compare instead of a 64-bit division per cell.
struct CellIter {
    int64_t y, x, sy, sx, nx;
    __device__ __forceinline__ explicit CellIter(int64_t nx_) : nx(nx_)
    {
        const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
        y = t0 / nx; x = t0 - y * nx;
        sy = stride / nx; sx = stride - sy * nx;
    }
    __device__ __forceinline__ void next()
    {
        x += sx; y += sy;
        if (x >= nx) { x -= nx; ++y; }
    }
};

#endif  // __CUDACC__

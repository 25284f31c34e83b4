// GeoTIFF block decode on the device (DESIGN §9d): compressed strips / tiles of one raster, uploaded as they are in the
// file, are decoded one warp per block (tiff_decode_kernel, the core of tiffcodec.cuh with a warp emitter) into a dense
// staging workspace, then tiff_store_kernel undoes the predictor and the byte order, crops and stores the rows into the
// pitched raster.  Both kernels are persistent, never wait for another warp or CTA, and check every table entry.
#include <cuda_runtime.h>

#include <type_traits>

#include "common.cuh"
#include "tiffcodec.cuh"

namespace {

constexpr int DEC_WARPS = 4;                                     // warps (= blocks in flight) per decode CTA
constexpr int STORE_WARPS = 8;
constexpr int64_t MAX_BLOCK_BYTES = (int64_t)1 << 31;            // LZW table offsets are 32-bit

// the core's emitter for one warp: the serial decode runs on every lane, copies are shared by the 32 lanes
struct WarpEmit {
    uint8_t* out;
    int ln;
    static constexpr int lanes = 32;
    __device__ __forceinline__ int lane() const { return ln; }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
    __device__ __forceinline__ uint64_t sum(uint64_t v) const
    {
#pragma unroll
        for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        return v;
    }
    __device__ __forceinline__ void put(int64_t op, uint8_t b) const
    {
        if (ln == 0) out[op] = b;
    }
    // out[op + i] = out[op - dist + i]: for an overlapping run (dist < len) byte i repeats byte i % dist of the period
    // that is already written, so the lanes never read what another lane of the same copy writes
    __device__ __forceinline__ void copy(int64_t op, int64_t dist, int64_t len) const
    {
        __syncwarp();                                            // earlier literals and copies are visible
        uint8_t* d = out + op;
        const uint8_t* s = d - dist;
        if (dist >= len) {
            for (int64_t i = ln; i < len; i += 32) d[i] = s[i];
        } else {
            const int p = (int)dist;
            for (int i = ln; i < (int)len; i += 32) d[i] = s[i % p];
        }
    }
    __device__ __forceinline__ void copy_in(int64_t op, const uint8_t* src, int64_t len) const
    {
        __syncwarp();
        for (int64_t i = ln; i < len; i += 32) out[op + i] = src[i];
    }
    __device__ __forceinline__ void zero(int64_t a, int64_t b) const
    {
        for (int64_t i = a + ln; i < b; i += 32) out[i] = 0;
    }
    __device__ __forceinline__ const uint8_t* data() const { return out; }
};

template <int CODEC>
using CodecTable = typename std::conditional<CODEC == 5, tiffcodec::LzwTable, tiffcodec::InflateTables>::type;

__host__ __device__ constexpr int64_t slot_bytes_of(int64_t bh, int64_t bw, int64_t es) { return (bh * bw * es + 15) / 16 * 16; }

// blocks: int64[n][5] = (src offset, nbytes, y0, x0, rows).  Block k decodes to stage + k * slot_bytes.
template <int CODEC>
__global__ void __launch_bounds__(DEC_WARPS * 32) tiff_decode_kernel(const uint8_t* __restrict__ src, int64_t src_bytes,
                                                                     const int64_t* __restrict__ blocks, int64_t n_blocks,
                                                                     uint8_t* stage, int64_t slot_bytes, int64_t row_bytes,
                                                                     int64_t ny, int64_t nx, int64_t bh, int* status)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int wid = threadIdx.x >> 5, ln = threadIdx.x & 31;
    CodecTable<CODEC>& t = reinterpret_cast<CodecTable<CODEC>*>(smem)[wid];
    for (int64_t k = (int64_t)blockIdx.x * DEC_WARPS + wid; k < n_blocks; k += (int64_t)gridDim.x * DEC_WARPS) {
        const int64_t off = blocks[5 * k], nb = blocks[5 * k + 1], y0 = blocks[5 * k + 2], x0 = blocks[5 * k + 3];
        const int64_t rows = blocks[5 * k + 4];
        int st = tiffcodec::CORRUPT;
        if (off >= 0 && nb >= 1 && off <= src_bytes && nb <= src_bytes - off && rows >= 1 && rows <= bh && y0 >= 0 &&
            y0 < ny && x0 >= 0 && x0 < nx) {
            const int64_t cap = rows * row_bytes;
            const WarpEmit em{stage + k * slot_bytes, ln};
            int64_t len = 0;
            __syncwarp();                                        // the previous block's table reads are done
            if constexpr (CODEC == 5) {
                st = tiffcodec::lzw(src + off, nb, em, cap, t, &len);
                if (st == tiffcodec::OK) em.zero(len, cap);      // short strips are zero-padded, as on the host
            } else {
                st = tiffcodec::inflate(src + off, nb, em, cap, t, &len);
                if (st == tiffcodec::OK && len < cap) st = tiffcodec::CORRUPT;
            }
        }
        if (ln == 0) status[k] = st;
    }
}

template <typename T>
__device__ __forceinline__ T bswap(T v)
{
    T r = 0;
#pragma unroll
    for (int b = 0; b < (int)sizeof(T); ++b) r = (T)((r << 8) | ((v >> (8 * b)) & 0xFF));
    return r;
}

template <typename U>
__device__ __forceinline__ U warp_scan(U v, int ln)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const U n = __shfl_up_sync(0xFFFFFFFFu, v, o);
        if (ln >= o) v += n;
    }
    return v;
}

// One warp per row of a block: predictor 2 (a prefix sum in sample arithmetic after the byte swap) or 3 (a byte-wise
// prefix sum over the row's byte planes) is undone in place in the staging row; then the row's cropped samples go to
// the raster in 16-byte aligned stores (partial ones at the two ends).
template <typename T>
__global__ void __launch_bounds__(STORE_WARPS * 32) tiff_store_kernel(uint8_t* stage, const int64_t* __restrict__ blocks,
                                                                      int64_t n_blocks, int64_t slot_bytes,
                                                                      const int* __restrict__ status, int predictor,
                                                                      int big_endian, uint8_t* out, int64_t out_pitch_bytes,
                                                                      int64_t ny, int64_t nx, int64_t bh, int64_t bw)
{
    constexpr int ES = sizeof(T), V = 16 / ES;
    using U = typename std::conditional<ES == 8, uint64_t, uint32_t>::type;
    const int ln = threadIdx.x & 31;
    const int64_t nw = (int64_t)gridDim.x * STORE_WARPS, ntask = n_blocks * bh;
    for (int64_t task = (int64_t)blockIdx.x * STORE_WARPS + (threadIdx.x >> 5); task < ntask; task += nw) {
        const int64_t k = task / bh, r = task - k * bh;
        if (status[k] != tiffcodec::OK) continue;               // the decode kernel vetted the entry
        const int64_t y0 = blocks[5 * k + 2], x0 = blocks[5 * k + 3], rows = blocks[5 * k + 4];
        const int64_t ys = rows < ny - y0 ? rows : ny - y0;
        if (r >= ys) continue;
        const int64_t xs = bw < nx - x0 ? bw : nx - x0;
        uint8_t* row = stage + k * slot_bytes + r * bw * ES;
        if (predictor == 2) {
            U carry = 0;
            for (int64_t base = 0; base < xs; base += 32) {
                const int64_t j = base + ln;
                U v = 0;
                if (j < xs) v = (U)(big_endian ? bswap(((const T*)row)[j]) : ((const T*)row)[j]);
                v = warp_scan(v, ln) + carry;
                if (j < xs) ((T*)row)[j] = (T)v;
                carry = __shfl_sync(0xFFFFFFFFu, v, 31);
            }
            __syncwarp();
        } else if (predictor == 3) {
            const int64_t L = bw * ES;
            uint32_t carry = 0;
            for (int64_t base = 0; base < L; base += 32) {
                const int64_t j = base + ln;
                uint32_t v = j < L ? row[j] : 0;
                v = warp_scan(v, ln) + carry;
                if (j < L) row[j] = (uint8_t)v;
                carry = __shfl_sync(0xFFFFFFFFu, v, 31);
            }
            __syncwarp();
        }
        auto sample = [&](int64_t j) -> T {
            if (predictor == 3) {                                // planes, most significant first: a big-endian float
                T v = 0;
#pragma unroll
                for (int b = 0; b < ES; ++b) v = (T)((v << 8) | row[b * bw + j]);
                return v;
            }
            const T v = ((const T*)row)[j];
            return predictor == 1 && big_endian ? bswap(v) : v;
        };
        uint8_t* d = out + (y0 + r) * out_pitch_bytes + x0 * ES;
        uint8_t* a0 = (uint8_t*)((uintptr_t)d & ~(uintptr_t)15);
        const int64_t nchunks = (d + xs * ES - a0 + 15) / 16;
        for (int64_t c = ln; c < nchunks; c += 32) {
            uint8_t* cb = a0 + 16 * c;
            const int64_t j0 = (cb - d) / ES;
            if (j0 >= 0 && j0 + V <= xs) {
                union { uint4 u; T v[V]; } pk;
#pragma unroll
                for (int v = 0; v < V; ++v) pk.v[v] = sample(j0 + v);
                *(uint4*)cb = pk.u;
            } else {
                for (int v = 0; v < V; ++v)
                    if (j0 + v >= 0 && j0 + v < xs) ((T*)cb)[v] = sample(j0 + v);
            }
        }
    }
}

bool dtype_ok(int dt) { return dt == HD_U8 || dt == HD_I16 || dt == HD_I32 || dt == HD_I64 || dt == HD_F32 || dt == HD_F64; }

template <int CODEC>
int launch_decode(const uint8_t* src, int64_t src_bytes, const int64_t* blocks, int64_t n_blocks, uint8_t* stage,
                  int64_t slot, int64_t row_bytes, int64_t ny, int64_t nx, int64_t bh, int* status, cudaStream_t s)
{
    const size_t smem = DEC_WARPS * sizeof(CodecTable<CODEC>);
    static int occ_of[64] = {};                                  // CTAs per SM, per device (the attribute is per device)
    int dev = 0;
    HD_CUDA_OK(cudaGetDevice(&dev));
    int& occ = occ_of[dev & 63];
    if (occ == 0) {
        HD_CUDA_OK(cudaFuncSetAttribute(tiff_decode_kernel<CODEC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HD_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, tiff_decode_kernel<CODEC>, DEC_WARPS * 32, smem));
        if (occ < 1) occ = 1;
    }
    const int64_t want = (n_blocks + DEC_WARPS - 1) / DEC_WARPS, cap = (int64_t)hd_num_sms() * occ;
    hd_prof_begin(CODEC == 5 ? "tiff_decode_lzw" : "tiff_decode_deflate", s);
    tiff_decode_kernel<CODEC><<<(unsigned)(want < cap ? want : cap), DEC_WARPS * 32, smem, s>>>(
        src, src_bytes, blocks, n_blocks, stage, slot, row_bytes, ny, nx, bh, status);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

template <typename T>
int launch_store(uint8_t* stage, const int64_t* blocks, int64_t n_blocks, int64_t slot, const int* status, int predictor,
                 int big_endian, uint8_t* out, int64_t out_pitch_bytes, int64_t ny, int64_t nx, int64_t bh, int64_t bw,
                 cudaStream_t s)
{
    const int64_t want = (n_blocks * bh + STORE_WARPS - 1) / STORE_WARPS, cap = (int64_t)hd_num_sms() * 8;
    hd_prof_begin("tiff_store", s);
    tiff_store_kernel<T><<<(unsigned)(want < cap ? want : cap), STORE_WARPS * 32, 0, s>>>(
        stage, blocks, n_blocks, slot, status, predictor, big_endian, out, out_pitch_bytes, ny, nx, bh, bw);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

}  // namespace

extern "C" int64_t hd_tiff_decode_workspace_bytes(int64_t n_blocks, int64_t block_h, int64_t block_w, int sample_dtype)
{
    if (n_blocks < 0 || n_blocks > ((int64_t)1 << 40) || block_h < 1 || block_w < 1 || !dtype_ok(sample_dtype)) return 0;
    const int64_t es = (int64_t)hd_dtype_size(sample_dtype);
    if (block_h > MAX_BLOCK_BYTES / block_w / es) return 0;
    const int64_t slot = slot_bytes_of(block_h, block_w, es);
    if (n_blocks > INT64_MAX / 2 / slot) return 0;
    return n_blocks * slot;
}

extern "C" int hd_tiff_decode(const void* src, int64_t src_bytes, const void* blocks, int64_t n_blocks, int compression,
                              int predictor, int sample_dtype, int big_endian, void* out, int64_t out_pitch, int64_t ny,
                              int64_t nx, int64_t block_h, int64_t block_w, void* status, void* workspace,
                              int64_t workspace_bytes, void* stream)
{
    if (!out || (n_blocks > 0 && (!src || !blocks || !status || !workspace))) return HD_ERR_NULL;
    if (compression != 5 && compression != 8 && compression != 32946) return HD_ERR_ARG;
    if (predictor < 1 || predictor > 3 || !dtype_ok(sample_dtype) || (big_endian != 0 && big_endian != 1)) return HD_ERR_ARG;
    const bool is_float = sample_dtype == HD_F32 || sample_dtype == HD_F64;
    if ((predictor == 3 && !is_float) || (predictor == 2 && is_float)) return HD_ERR_ARG;
    if (n_blocks < 0 || src_bytes < 0 || ny < 1 || nx < 1 || out_pitch < nx || block_h < 1 || block_w < 1) return HD_ERR_ARG;
    const int64_t need = hd_tiff_decode_workspace_bytes(n_blocks, block_h, block_w, sample_dtype);
    if (need == 0 && n_blocks > 0) return HD_ERR_ARG;            // a block above 2 GB or a table beyond 2^40 blocks
    if (workspace_bytes < need) return HD_ERR_WORKSPACE;
    const int64_t es = (int64_t)hd_dtype_size(sample_dtype);
    if (((uintptr_t)out & 15) || (out_pitch * es) % 16) return HD_ERR_ALIGN;
    if (n_blocks == 0) return HD_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t slot = slot_bytes_of(block_h, block_w, es);
    uint8_t* stage = (uint8_t*)workspace;
    const int64_t* tbl = (const int64_t*)blocks;
    int* st = (int*)status;
    int rc = compression == 5
                 ? launch_decode<5>((const uint8_t*)src, src_bytes, tbl, n_blocks, stage, slot, block_w * es, ny, nx, block_h, st, s)
                 : launch_decode<8>((const uint8_t*)src, src_bytes, tbl, n_blocks, stage, slot, block_w * es, ny, nx, block_h, st, s);
    if (rc != HD_OK) return rc;
    uint8_t* o = (uint8_t*)out;
    const int64_t opb = out_pitch * es;
    switch (es) {
    case 1: return launch_store<uint8_t>(stage, tbl, n_blocks, slot, st, predictor, big_endian, o, opb, ny, nx, block_h, block_w, s);
    case 2: return launch_store<uint16_t>(stage, tbl, n_blocks, slot, st, predictor, big_endian, o, opb, ny, nx, block_h, block_w, s);
    case 4: return launch_store<uint32_t>(stage, tbl, n_blocks, slot, st, predictor, big_endian, o, opb, ny, nx, block_h, block_w, s);
    default: return launch_store<uint64_t>(stage, tbl, n_blocks, slot, st, predictor, big_endian, o, opb, ny, nx, block_h, block_w, s);
    }
}

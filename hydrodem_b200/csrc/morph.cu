// Binary / flat morphology of the conditioning chain on bit-packed tiles.
//
//   hd_expand      ExpandFilter.apply                 custom_filters.py:102-125
//   hd_binary_morph BinaryErosion / BinaryClosing     extension_filters.py:218-235, :276-293 (scipy.ndimage)
//   hd_max_filter  GreyDilation(size=(s,s))           extension_filters.py:328-345 (scipy.ndimage.grey_dilation)
//   hd_binary_morph_struct  the same with any structure up to 31x31, several steps per launch, changed flag
//   hd_max_filter_rect      GreyDilation(size=(a, b)), any size 1 ... 255 per axis (van Herk / Gil-Werman)
//
// All three are HBM-bound: a 32x128 tile (+halo) is staged by TMA, thresholded to one bit per cell with
// warp ballots, and the window logic runs on 32-cell words (funnel shifts / ORs), a few hundred word
// operations per 4096-cell tile.  Output is written with 16-byte (or 4-byte for u8) coalesced stores.
#include "common.cuh"
#include "tile_common.cuh"

namespace {

constexpr int MAX_HALO = 8;
constexpr int MAX_IN_H = TH + 2 * MAX_HALO;            // 48
constexpr int MAX_IN_W = TW + 2 * 16;                  // 160: u8 planes need a 16-cell x halo
constexpr int NWORD = (MAX_IN_W + 31) / 32;            // 5
constexpr int STAGE_BYTES = MAX_IN_H * (TW + 2 * MAX_HALO) * 4;   // sized for f32 (x halo <= 8), u8 needs less

// threshold one staged tile to bits: bits[r * NWORD + k] bit i  <->  tile cell (r, 32k + i)
template <typename InT, int THREADS = NT, class Pred>
__device__ __forceinline__ void tile_to_bits(const InT* tile, int in_w, int in_h, uint32_t* bits, Pred pred)
{
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int r = warp; r < in_h; r += THREADS / 32) {
#pragma unroll
        for (int k = 0; k < NWORD; ++k) {
            const int c = 32 * k + lane;
            const bool p = (c < in_w) && pred(tile[r * in_w + c]);
            const uint32_t w = __ballot_sync(0xffffffffu, p);
            if (lane == 0) bits[r * NWORD + k] = w;
        }
    }
}

__device__ __forceinline__ uint64_t win64(const uint32_t* row, int k)
{
    const uint32_t lo = row[k], hi = (k + 1 < NWORD) ? row[k + 1] : 0u;
    return ((uint64_t)hi << 32) | lo;
}

// write a TH x TW tile of 0/1 results held as bit words res[ro * 4 + k]
template <typename OutT>
__device__ __forceinline__ void write_bits(const uint32_t* res, OutT* out, int64_t out_pitch, int ty0, int tx0,
                                           int64_t ny, int64_t nx, int border, const float* __restrict__ select = nullptr,
                                           int64_t sel_pitch = 0)
{
    // a tile that lies inside the frame [border, n - border) needs no per-cell edge tests (almost every tile)
    const bool inner = ty0 >= border && ty0 + TH <= ny - border && tx0 >= border && tx0 + TW <= nx - border;
#pragma unroll
    for (int rep = 0; rep < TH * TW / 4 / NT; ++rep) {
        const int idx = rep * NT + threadIdx.x;
        const int ro = idx >> 5, c4 = idx & 31;
        const int64_t y = ty0 + ro, x = tx0 + 4 * c4;
        if (y >= ny || x >= nx) continue;
        uint32_t nib = (res[ro * 4 + (c4 >> 3)] >> ((c4 & 7) * 4)) & 15u;
        if (!inner) {
            const bool yin = (y >= border) && (y < ny - border);
            uint32_t keep = 0u;
#pragma unroll
            for (int j = 0; j < 4; ++j) keep |= (yin && (x + j >= border) && (x + j < nx - border)) ? (1u << j) : 0u;
            nib &= keep;
        }
        if constexpr (sizeof(OutT) == 1) {
            if (!select) {
                // 0 / 1 bytes straight from the nibble: one 32-bit store
                const uint32_t word = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
                uint8_t* q = reinterpret_cast<uint8_t*>(out) + y * out_pitch + x;
                if (x + 3 < nx && ((reinterpret_cast<uintptr_t>(q) & 3) == 0)) {
                    *reinterpret_cast<uint32_t*>(q) = word;
                } else {
                    for (int j = 0; j < 4; ++j)
                        if (x + j < nx) q[j] = (uint8_t)((nib >> j) & 1u);
                }
                continue;
            }
        }
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = ((nib >> j) & 1u) ? 1.f : 0.f;
        if (select) {
            // fused ProductFilter(factor = select): factor * expanded  (TidyingLagoons, custom_filters.py:589-590, :607)
            float sv[4];
            gload4(select + y * sel_pitch + x, x, nx, sv);
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = __fmul_rn(sv[j], v[j]);
        }
        store4<OutT>(out, out_pitch, y, x, nx, v);
    }
}

// ------------------------------------------------------------------------------------------------ expand
template <typename InT, typename OutT>
__global__ void __launch_bounds__(NT) expand_kernel(const __grid_constant__ CUtensorMap tm_in, OutT* __restrict__ out,
                                                    int64_t out_pitch, int64_t ny, int64_t nx, int h, int in_w, int in_h,
                                                    int tiles_x, int ntiles, const float* __restrict__ select,
                                                    int64_t sel_pitch)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    __shared__ uint32_t bits[MAX_IN_H * NWORD];
    const int hx = hd_halo_x(h, sizeof(InT)), xoff = hx - h;
    __shared__ uint32_t hfull[MAX_IN_H * 4], hinner[MAX_IN_H * 4];
    __shared__ uint32_t res[TH * 4];
    const uint32_t stage_bytes = STAGE_BYTES;
    const TilePlane planes[1] = {{&tm_in, 0u, (uint32_t)(in_w * in_h * sizeof(InT)), hx, h}};
    tile_loop<1>(smem, stage_bytes, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        const InT* tile = reinterpret_cast<const InT*>(st);
        // window[~isnan(window)] > 0  (custom_filters.py:122-123): NaN > 0 is false
        tile_to_bits<InT>(tile, in_w, in_h, bits, [](InT v) { return (float)v > 0.f; });
        __syncthreads();
        // horizontal: output column xo looks at tile columns xoff+xo .. xoff+xo+2h (full) / xo+1 .. xo+2h-1 (top & bottom rows)
        for (int t = threadIdx.x; t < in_h * 4; t += NT) {
            const int r = t >> 2, k = t & 3;
            const uint64_t w = win64(&bits[r * NWORD], k);
            uint64_t f = 0, in = 0;
            for (int s = 0; s <= 2 * h; ++s) {
                f |= w >> (s + xoff);
                if (s >= 1 && s <= 2 * h - 1) in |= w >> (s + xoff);
            }
            hfull[t] = (uint32_t)f;
            hinner[t] = (uint32_t)in;
        }
        __syncthreads();
        if (threadIdx.x < TH * 4) {
            const int ro = threadIdx.x >> 2, k = threadIdx.x & 3;
            uint32_t acc = hinner[ro * 4 + k] | hinner[(ro + 2 * h) * 4 + k];   // corner-less top / bottom rows
            for (int r = ro + 1; r <= ro + 2 * h - 1; ++r) acc |= hfull[r * 4 + k];
            res[threadIdx.x] = acc;
        }
        __syncthreads();
        write_bits<OutT>(res, out, out_pitch, ty0, tx0, ny, nx, h, select, sel_pitch);
    });
}

// ------------------------------------------------------------------------------------------------ erosion / closing
struct MorphProgram {
    int nsteps;
    unsigned char dilate[MAX_HALO];   // 1 = dilation, 0 = erosion
    unsigned char full[MAX_HALO];     // 1 = 3x3 square, 0 = cross
};

template <typename InT>
__global__ void __launch_bounds__(NT) morph_kernel(const __grid_constant__ CUtensorMap tm_in, uint8_t* __restrict__ out,
                                                   int64_t out_pitch, int64_t ny, int64_t nx, MorphProgram prog, int in_w,
                                                   int in_h, int tiles_x, int ntiles)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    __shared__ uint32_t bufA[(MAX_IN_H + 2) * NWORD], bufB[(MAX_IN_H + 2) * NWORD];
    __shared__ uint32_t res[TH * 4];
    const int h = prog.nsteps, hx = hd_halo_x(h, sizeof(InT));
    const TilePlane planes[1] = {{&tm_in, 0u, (uint32_t)(in_w * in_h * sizeof(InT)), hx, h}};
    // rows 0 and in_h+1 of the bit buffers are zero guards
    for (int t = threadIdx.x; t < NWORD; t += NT) {
        bufA[t] = bufB[t] = 0u;
    }
    tile_loop<1>(smem, STAGE_BYTES, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        const InT* tile = reinterpret_cast<const InT*>(st);
        uint32_t* cur = bufA + NWORD;
        uint32_t* nxt = bufB + NWORD;
        // scipy: "non-zero elements are True" -- NaN != 0 is true; cells outside the image arrive as 0
        tile_to_bits<InT>(tile, in_w, in_h, cur, [](InT v) { return v != (InT)0; });
        if (threadIdx.x < NWORD) { cur[in_h * NWORD + threadIdx.x] = 0u; nxt[in_h * NWORD + threadIdx.x] = 0u; }
        __syncthreads();
        for (int s = 0; s < prog.nsteps; ++s) {
            const bool dil = prog.dilate[s], full = prog.full[s];
            for (int t = threadIdx.x; t < in_h * NWORD; t += NT) {
                const int r = t / NWORD, k = t - r * NWORD;
                auto hcomb = [&](const uint32_t* row) {       // centre | left | right (or &)
                    const uint32_t c = row[k];
                    const uint32_t lft = (c << 1) | (k > 0 ? row[k - 1] >> 31 : 0u);
                    const uint32_t rgt = (c >> 1) | (k + 1 < NWORD ? row[k + 1] << 31 : 0u);
                    return dil ? (c | lft | rgt) : (c & lft & rgt);
                };
                const uint32_t* rc = cur + r * NWORD;
                const uint32_t* ru = rc - NWORD;              // guard row is zero (outside = False)
                const uint32_t* rd = rc + NWORD;
                uint32_t v;
                if (full) {
                    const uint32_t a = hcomb(ru), b = hcomb(rc), c = hcomb(rd);
                    v = dil ? (a | b | c) : (a & b & c);
                } else {
                    const uint32_t b = hcomb(rc);
                    v = dil ? (b | ru[k] | rd[k]) : (b & ru[k] & rd[k]);
                }
                if (dil) {
                    // the dilated image only exists on the raster: outside stays border_value = 0
                    const int64_t gy = (int64_t)ty0 - h + r;
                    uint32_t m = 0u;
                    if (gy >= 0 && gy < ny) {
                        const int64_t gx0 = (int64_t)tx0 - hx + 32 * k;     // global x of bit 0
                        const int64_t lo = gx0 < 0 ? -gx0 : 0;
                        const int64_t hi = (nx - gx0) < 32 ? (nx - gx0) : 32;   // exclusive
                        if (hi > lo) m = (hi - lo >= 32 ? 0xffffffffu : ((1u << (hi - lo)) - 1u)) << lo;
                    }
                    v &= m;
                }
                nxt[t] = v;
            }
            __syncthreads();
            uint32_t* tmp = cur; cur = nxt; nxt = tmp;
        }
        // extract the TH x TW core (tile offset h) into output words
        if (threadIdx.x < TH * 4) {
            const int ro = threadIdx.x >> 2, k = threadIdx.x & 3;
            const uint64_t w = win64(cur + (ro + h) * NWORD, k);
            res[threadIdx.x] = (uint32_t)(w >> hx);
        }
        __syncthreads();
        write_bits<uint8_t>(res, out, out_pitch, ty0, tx0, ny, nx, 0);
    });
}

// ------------------------------------------------------------------------------------------------ max filter
// mode='reflect' (d c b a | a b c d | d c b a): OOB cells of frame tiles are patched in shared memory from
// their mirror cell, which always lies inside the same staged box (size <= min(ny, nx)).
template <typename T> __device__ __forceinline__ T tmax(T a, T b);
template <> __device__ __forceinline__ float tmax<float>(float a, float b) { return fmaxf(a, b); }
template <> __device__ __forceinline__ double tmax<double>(double a, double b) { return fmax(a, b); }

// HC > 0: half-window known at compile time (the chain's GreyDilation is 7x7): loops unroll and the horizontal pass
// shares its loads between four neighbouring outputs.  HC = 0: any half-window, plain loops.
template <typename T, int HC>
__global__ void __launch_bounds__(NT) maxfilter_kernel(const __grid_constant__ CUtensorMap tm_in, T* __restrict__ out,
                                                       int64_t out_pitch, int64_t ny, int64_t nx, int h_rt, int in_w, int in_h,
                                                       int tiles_x, int ntiles)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    constexpr uint32_t STAGE = MAX_IN_H * (TW + 2 * MAX_HALO) * sizeof(T);
    T* hmax = reinterpret_cast<T*>(smem + 2 * STAGE);          // [in_h][TW] horizontal maxima
    const int h = HC > 0 ? HC : h_rt;
    const int hx = hd_halo_x(h, sizeof(T)), xoff = hx - h;
    const TilePlane planes[1] = {{&tm_in, 0u, (uint32_t)(in_w * in_h * sizeof(T)), hx, h}};
    tile_loop<1>(smem, STAGE, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        T* tile = reinterpret_cast<T*>(st);
        patch_reflect<T>(tile, in_w, in_h, ty0 - h, tx0 - hx, ny, nx);
        if constexpr (HC > 0) {
            // horizontal: four consecutive outputs per thread from 4 + 2 HC loaded cells
            for (int t = threadIdx.x; t < in_h * (TW / 4); t += NT) {
                const int r = t / (TW / 4), c = 4 * (t - r * (TW / 4));
                const T* src = tile + r * in_w + c + xoff;
                T v[4 + 2 * HC];
#pragma unroll
                for (int k = 0; k < 4 + 2 * HC; ++k) v[k] = src[k];
                T mid = v[3];                                  // cells 3 .. 2 HC are shared by all four windows
#pragma unroll
                for (int k = 4; k <= 2 * HC; ++k) mid = tmax<T>(mid, v[k]);
                T o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    T m = mid;
#pragma unroll
                    for (int k = j; k < 3; ++k) m = tmax<T>(m, v[k]);
#pragma unroll
                    for (int k = 2 * HC + 1; k <= 2 * HC + j; ++k) m = tmax<T>(m, v[k]);
                    o[j] = m;
                }
                T* dst = hmax + r * TW + c;
#pragma unroll
                for (int j = 0; j < 4; ++j) dst[j] = o[j];
            }
        } else {
            for (int t = threadIdx.x; t < in_h * TW; t += NT) {
                const int r = t / TW, c = t - r * TW;
                T m = tile[r * in_w + c + xoff];
                for (int s = 1; s <= 2 * h; ++s) m = tmax<T>(m, tile[r * in_w + c + xoff + s]);
                hmax[t] = m;
            }
        }
        __syncthreads();
#pragma unroll
        for (int rep = 0; rep < TH * TW / 4 / NT; ++rep) {
            const int idx = rep * NT + threadIdx.x;
            const int ro = idx >> 5, c4 = idx & 31;
            const int64_t y = ty0 + ro, x = tx0 + 4 * c4;
            if (y >= ny || x >= nx) continue;
            T v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = hmax[ro * TW + 4 * c4 + j];
            if constexpr (HC > 0) {
#pragma unroll
                for (int s = 1; s <= 2 * HC; ++s) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = tmax<T>(v[j], hmax[(ro + s) * TW + 4 * c4 + j]);
                }
            } else {
                for (int s = 1; s <= 2 * h; ++s) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) v[j] = tmax<T>(v[j], hmax[(ro + s) * TW + 4 * c4 + j]);
                }
            }
            store4v<T>(out, out_pitch, y, x, nx, v);
        }
    });
}


// ------------------------------------------------------------------------------------------------ TidyingLagoons, fused
// custom_filters.py:587-610 as ONE kernel: BinaryErosion(iterations=2, cross) -> ExpandFilter(7) -> x majority image ->
// GreyDilation(7x7, reflect).  The majority tile is staged once with a halo of 2 + 3 + 3 = 8 cells; erosion and expansion
// run on bit rows in shared memory, the product and the separable 7x7 maximum on a 38 x 136 float array -- 4 B read +
// 4 B written per cell instead of three kernels with a uint8 and two float32 rasters in between.  Same bits as
// hd_binary_morph + hd_expand_select + hd_max_filter.
constexpr int TL_H = 8;                                   // halo
constexpr int TL_IN_W = TW + 2 * TL_H, TL_IN_H = TH + 2 * TL_H;      // 144 x 48
constexpr int TL_PW = TW + 8, TL_PH = TH + 6;             // product array: box columns 4 .. 139, box rows 5 .. 42
constexpr uint32_t TL_STAGE = TL_IN_W * TL_IN_H * 4;
constexpr int TL_NT = 512;                               // 2 CTAs x 16 warps per SM (the kernel is issue / latency bound)

__global__ void __launch_bounds__(TL_NT) tidy_lagoons_kernel(const __grid_constant__ CUtensorMap tm_in, float* __restrict__ out,
                                                          int64_t out_pitch, int64_t ny, int64_t nx, int tiles_x, int ntiles)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    __shared__ uint32_t bufA[(TL_IN_H + 2) * NWORD], bufB[(TL_IN_H + 2) * NWORD];
    __shared__ uint32_t hfull[TL_IN_H * NWORD], hinner[TL_IN_H * NWORD], ex[TL_PH * NWORD];
    float* prod = reinterpret_cast<float*>(smem + 2 * TL_STAGE);        // [TL_PH][TL_PW]
    float* hmax = prod + TL_PH * TL_PW;                                  // [TL_PH][TW]
    const TilePlane planes[1] = {{&tm_in, 0u, TL_STAGE, TL_H, TL_H}};
    for (int t = threadIdx.x; t < NWORD; t += TL_NT) bufA[t] = bufB[t] = 0u;                       // zero guard rows
    tile_loop<1>(smem, TL_STAGE, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        const float* tile = reinterpret_cast<const float*>(st);
        uint32_t* cur = bufA + NWORD;
        uint32_t* nxt = bufB + NWORD;
        // scipy: non-zero elements are True (NaN != 0 is true); cells outside the raster arrive as 0 = border_value
        tile_to_bits<float, TL_NT>(tile, TL_IN_W, TL_IN_H, cur, [](float v) { return v != 0.f; });
        if (threadIdx.x < NWORD) { cur[TL_IN_H * NWORD + threadIdx.x] = 0u; nxt[TL_IN_H * NWORD + threadIdx.x] = 0u; }
        __syncthreads();
        for (int step = 0; step < 2; ++step) {                           // BinaryErosion(iterations=2), cross
            for (int t = threadIdx.x; t < TL_IN_H * NWORD; t += TL_NT) {
                const int r = t / NWORD, k = t - r * NWORD;
                const uint32_t* rc = cur + r * NWORD;
                const uint32_t c = rc[k];
                const uint32_t lft = (c << 1) | (k > 0 ? rc[k - 1] >> 31 : 0u);
                const uint32_t rgt = (c >> 1) | (k + 1 < NWORD ? rc[k + 1] << 31 : 0u);
                nxt[t] = c & lft & rgt & rc[k - NWORD] & rc[k + NWORD];
            }
            __syncthreads();
            uint32_t* tmp = cur; cur = nxt; nxt = tmp;
        }
        // ExpandFilter(7): windows written by their FIRST column c' (output column c looks at bit c - 3)
        for (int t = threadIdx.x; t < TL_IN_H * NWORD; t += TL_NT) {
            const int r = t / NWORD, k = t - r * NWORD;
            const uint64_t w = win64(cur + r * NWORD, k);
            uint64_t f = w, in = 0;
#pragma unroll
            for (int sft = 1; sft <= 6; ++sft) {
                f |= w >> sft;
                if (sft <= 5) in |= w >> sft;
            }
            hfull[t] = (uint32_t)f;
            hinner[t] = (uint32_t)in;
        }
        __syncthreads();
        for (int t = threadIdx.x; t < TL_PH * NWORD; t += TL_NT) {
            const int pr = t / NWORD, k = t - pr * NWORD, r = pr + 5;    // box row
            uint32_t acc = hinner[(r - 3) * NWORD + k] | hinner[(r + 3) * NWORD + k];   // corner-less top / bottom rows
#pragma unroll
            for (int q = r - 2; q <= r + 2; ++q) acc |= hfull[q * NWORD + k];
            ex[t] = acc;
        }
        __syncthreads();
        // product with the majority image (ProductFilter(factor=majority), :607); ExpandFilter leaves its 3-cell frame at 0
        for (int t = threadIdx.x; t < TL_PH * TL_PW; t += TL_NT) {
            const int pr = t / TL_PW, pc = t - pr * TL_PW;
            const int r = pr + 5, c = pc + 4;                            // box coordinates
            const int64_t y = (int64_t)ty0 - TL_H + r, x = (int64_t)tx0 - TL_H + c;
            const int cb = c - 3;                                        // first column of the window
            const bool bit = cb >= 0 && ((ex[pr * NWORD + (cb >> 5)] >> (cb & 31)) & 1u);
            const bool inside = y >= 3 && y < ny - 3 && x >= 3 && x < nx - 3;
            prod[t] = __fmul_rn(tile[r * TL_IN_W + c], (bit && inside) ? 1.f : 0.f);
        }
        __syncthreads();
        // GreyDilation(size=(7, 7)), mode='reflect'
        patch_reflect<float>(prod, TL_PW, TL_PH, ty0 - 3, tx0 - 4, ny, nx);
        for (int t = threadIdx.x; t < TL_PH * (TW / 4); t += TL_NT) {
            const int r = t / (TW / 4), c = 4 * (t - r * (TW / 4));
            const float* src = prod + r * TL_PW + c + 1;                 // output column c looks at array columns c+1 .. c+7
            float v[10];
#pragma unroll
            for (int k = 0; k < 10; ++k) v[k] = src[k];
            float mid = v[3];
#pragma unroll
            for (int k = 4; k <= 6; ++k) mid = fmaxf(mid, v[k]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float mm = mid;
#pragma unroll
                for (int k = j; k < 3; ++k) mm = fmaxf(mm, v[k]);
#pragma unroll
                for (int k = 7; k <= 6 + j; ++k) mm = fmaxf(mm, v[k]);
                hmax[r * TW + c + j] = mm;
            }
        }
        __syncthreads();
#pragma unroll
        for (int rep = 0; rep < TH * TW / 4 / TL_NT; ++rep) {
            const int idx = rep * TL_NT + threadIdx.x;
            const int ro = idx >> 5, c4 = idx & 31;
            const int64_t y = ty0 + ro, x = tx0 + 4 * c4;
            if (y >= ny || x >= nx) continue;
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = hmax[ro * TW + 4 * c4 + j];
#pragma unroll
            for (int sft = 1; sft <= 6; ++sft)
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], hmax[(ro + sft) * TW + 4 * c4 + j]);
            store4v<float>(out, out_pitch, y, x, nx, v);
        }
    });
}

// ------------------------------------------------------------------------------------------------ any structure
// scipy.ndimage.binary_erosion / binary_dilation with a structure up to 31 x 31, border_value = 0.  The host passes the
// structure's True cells as offsets (dy, dx) from the output cell, reflected and origin-shifted for a dilation.  Erosion
// is the AND, dilation the OR of the bit rows shifted by each offset; cells outside the raster are False before and after
// every step.  `nsteps` repetitions run in the tile (halo = nsteps x reach); `changed` (may be NULL) is set when the
// result differs from the input anywhere.
constexpr int MS_MAX_REACH = 15;
constexpr int MS_MAX_TAPS = (2 * MS_MAX_REACH + 1) * (2 * MS_MAX_REACH + 1);
constexpr int MS_MAX_IN_H = TH + 2 * MS_MAX_REACH;                    // 62
constexpr uint32_t MS_STAGE = MS_MAX_IN_H * MAX_IN_W * 4;              // f32 box of 62 x 160

struct MorphTaps {
    int ntaps;
    signed char dy[MS_MAX_TAPS], dx[MS_MAX_TAPS];
};

// bits of columns 32k + dx ... 32k + 31 + dx of a bit row (columns outside the row's NWORD words read as 0)
__device__ __forceinline__ uint32_t shifted_word(const uint32_t* row, int k, int dx)
{
    if (dx >= 0) return __funnelshift_rc(row[k], k + 1 < NWORD ? row[k + 1] : 0u, (uint32_t)dx);
    return __funnelshift_lc(k > 0 ? row[k - 1] : 0u, row[k], (uint32_t)-dx);
}

template <typename InT>
__global__ void __launch_bounds__(NT) morph_struct_kernel(const __grid_constant__ CUtensorMap tm_in, uint8_t* __restrict__ out,
                                                          int64_t out_pitch, int64_t ny, int64_t nx,
                                                          const __grid_constant__ MorphTaps p, int dilate, int nsteps, int hy,
                                                          int hx, int in_w, int in_h, int tiles_x, int ntiles,
                                                          int* __restrict__ changed)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    __shared__ uint32_t src[MS_MAX_IN_H * NWORD], bufA[MS_MAX_IN_H * NWORD], bufB[MS_MAX_IN_H * NWORD];
    __shared__ uint32_t res[TH * 4];
    const TilePlane planes[1] = {{&tm_in, 0u, (uint32_t)(in_w * in_h * sizeof(InT)), hx, hy}};
    tile_loop<1>(smem, MS_STAGE, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        // scipy: non-zero elements are True (NaN != 0 is true); cells outside the raster arrive as 0 = border_value
        tile_to_bits<InT>(reinterpret_cast<const InT*>(st), in_w, in_h, src, [](InT v) { return v != (InT)0; });
        __syncthreads();
        const uint32_t* cur = src;
        for (int s = 0; s < nsteps; ++s) {
            uint32_t* nxt = (s & 1) ? bufB : bufA;
            for (int t = threadIdx.x; t < in_h * NWORD; t += NT) {
                const int r = t / NWORD, k = t - r * NWORD;
                uint32_t v = dilate ? 0u : 0xffffffffu;
                for (int j = 0; j < p.ntaps; ++j) {
                    const int rr = r + p.dy[j];
                    const uint32_t w = (rr >= 0 && rr < in_h) ? shifted_word(cur + rr * NWORD, k, p.dx[j]) : 0u;
                    v = dilate ? (v | w) : (v & w);
                }
                // the result only exists on the raster: outside stays border_value = 0
                const int64_t gy = (int64_t)ty0 - hy + r;
                uint32_t m = 0u;
                if (gy >= 0 && gy < ny) {
                    const int64_t gx0 = (int64_t)tx0 - hx + 32 * k;      // global x of bit 0
                    const int64_t lo = gx0 < 0 ? -gx0 : 0;
                    const int64_t hi = (nx - gx0) < 32 ? (nx - gx0) : 32;   // exclusive
                    if (hi > lo) m = (hi - lo >= 32 ? 0xffffffffu : ((1u << (hi - lo)) - 1u)) << lo;
                }
                nxt[t] = v & m;
            }
            __syncthreads();
            cur = nxt;
        }
        if (threadIdx.x < TH * 4) {
            const int ro = threadIdx.x >> 2, k = threadIdx.x & 3;
            const uint32_t w = (uint32_t)(win64(cur + (ro + hy) * NWORD, k) >> hx);
            res[threadIdx.x] = w;
            // both words are 0 on cells outside the raster
            if (changed && w != (uint32_t)(win64(src + (ro + hy) * NWORD, k) >> hx)) atomicOr(changed, 1);
        }
        __syncthreads();
        write_bits<uint8_t>(res, out, out_pitch, ty0, tx0, ny, nx, 0);
    });
}

// ------------------------------------------------------------------------------------------------ rectangular max
// One axis of scipy.ndimage.grey_dilation(size=(a, b)), mode='reflect' (any distance: periodic), as van Herk / Gil-Werman:
// the extended segment is cut into blocks of k cells; h = running max from each cell to the end of its block (backward),
// g = running max from the block start (forward); window [j, j + k - 1] = max(h[j], g[j + k - 1]).  Three maxima per cell
// for any k.  A CTA takes 32 lines x SG outputs; shared memory holds [position][line] with a 33-line pitch, so loads
// along either axis and the per-line scans (one lane per line) are conflict free.  NaN cells are skipped (fmax).
constexpr int ML_LINES = 32, ML_LP = ML_LINES + 1;
template <typename T> constexpr int ml_seg() { return sizeof(T) == 4 ? 256 : 128; }

template <typename T, int AXIS>   // AXIS 0: along columns (window rows), 1: along rows
__global__ void __launch_bounds__(NT) maxline_kernel(const T* __restrict__ in, int64_t in_pitch, T* __restrict__ out,
                                                     int64_t out_pitch, int64_t ny, int64_t nx, int k, int lo)
{
    constexpr int SG = ml_seg<T>();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int E = SG + k - 1;
    T* e = reinterpret_cast<T*>(smem_raw);                    // [E][ML_LP] the extended segment
    T* h = e + (size_t)E * ML_LP;                             // [E][ML_LP] backward maxima, then the result
    const int64_t n_along = AXIS == 0 ? ny : nx, n_lines = AXIS == 0 ? nx : ny;
    const int64_t segs = (n_along + SG - 1) / SG, lgroups = (n_lines + ML_LINES - 1) / ML_LINES;
    const int64_t ntiles = segs * lgroups;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t a0 = (tile % segs) * SG, l0 = (tile / segs) * ML_LINES;
        for (int idx = threadIdx.x; idx < E * ML_LINES; idx += NT) {
            const int p = AXIS == 0 ? idx / ML_LINES : idx % E, l = AXIS == 0 ? idx % ML_LINES : idx / E;
            const int64_t gl = l0 + l, raw = a0 - lo + p;
            const int64_t ga = (raw >= 0 && raw < n_along) ? raw : reflect_periodic_idx(raw, n_along);
            if (gl < n_lines) e[p * ML_LP + l] = AXIS == 0 ? in[ga * in_pitch + gl] : in[gl * in_pitch + ga];
        }
        __syncthreads();
        const int nb = (E + k - 1) / k;
        for (int b = warp; b * k < SG; b += NT / 32) {       // h over the blocks that hold outputs
            const int j0 = b * k, j1 = min(E, j0 + k) - 1;
            T m = e[j1 * ML_LP + lane];
            h[j1 * ML_LP + lane] = m;
            for (int j = j1 - 1; j >= j0; --j) {
                m = tmax<T>(m, e[j * ML_LP + lane]);
                h[j * ML_LP + lane] = m;
            }
        }
        __syncthreads();
        for (int b = warp; b < nb; b += NT / 32) {            // g, combined into h at the window's first cell
            const int i0 = b * k, i1 = min(E, i0 + k);
            T m = e[i0 * ML_LP + lane];
            for (int i = i0; i < i1; ++i) {
                m = tmax<T>(m, e[i * ML_LP + lane]);
                const int j = i - k + 1;
                if (j >= 0 && j < SG) h[j * ML_LP + lane] = tmax<T>(h[j * ML_LP + lane], m);
            }
        }
        __syncthreads();
        const int n_out = (int)min((int64_t)SG, n_along - a0);
        for (int idx = threadIdx.x; idx < SG * ML_LINES; idx += NT) {
            const int p = AXIS == 0 ? idx / ML_LINES : idx % SG, l = AXIS == 0 ? idx % ML_LINES : idx / SG;
            const int64_t gl = l0 + l;
            if (p >= n_out || gl >= n_lines) continue;
            const T v = h[p * ML_LP + l];
            if (AXIS == 0) out[(a0 + p) * out_pitch + gl] = v; else out[gl * out_pitch + a0 + p] = v;
        }
        __syncthreads();
    }
}

template <typename T>
int launch_max_rect(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int64_t ny, int64_t nx, int size_y,
                    int size_x, void* workspace, cudaStream_t s)
{
    constexpr int SG = ml_seg<T>();
    // grey_dilation: origin -1 on an even axis, so the window of output i is [i - (k/2 - 1), i + k/2]
    auto lo_of = [](int k) { return k / 2 - (k % 2 == 0 ? 1 : 0); };
    const size_t smem_y = 2 * (size_t)(SG + size_y - 1) * ML_LP * sizeof(T), smem_x = 2 * (size_t)(SG + size_x - 1) * ML_LP * sizeof(T);
    const int tiles_y = hd_cdiv(ny, SG) * hd_cdiv(nx, ML_LINES), tiles_x = hd_cdiv(nx, SG) * hd_cdiv(ny, ML_LINES);
    const int per_sm = sizeof(T) == 4 ? 2 : 1;
    T* ws = (T*)workspace;                                    // dense ny x nx
    HD_CUDA_OK(cudaFuncSetAttribute(maxline_kernel<T, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_y));
    HD_CUDA_OK(cudaFuncSetAttribute(maxline_kernel<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_x));
    hd_prof_begin("maxline_kernel", s);
    maxline_kernel<T, 0><<<grid_for(tiles_y, per_sm), NT, smem_y, s>>>((const T*)in, in_pitch, ws, nx, ny, nx, size_y,
                                                                       lo_of(size_y));
    HD_LAUNCH_CHECK();
    hd_count_launch();
    hd_prof_begin("maxline_kernel", s);
    maxline_kernel<T, 1><<<grid_for(tiles_x, per_sm), NT, smem_x, s>>>(ws, nx, (T*)out, out_pitch, ny, nx, size_x,
                                                                       lo_of(size_x));
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

template <typename InT, typename OutT>
int launch_expand(const CUtensorMap& tm, void* out, int64_t out_pitch, int64_t ny, int64_t nx, int h, int in_w, int in_h,
                  cudaStream_t stream, const float* select = nullptr, int64_t sel_pitch = 0)
{
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t smem = 2 * STAGE_BYTES;
    HD_CUDA_OK(cudaFuncSetAttribute(expand_kernel<InT, OutT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    hd_prof_begin("expand_kernel", stream);
    expand_kernel<InT, OutT><<<grid_for(ntiles, 3), NT, smem, stream>>>(tm, (OutT*)out, out_pitch, ny, nx, h, in_w, in_h,
                                                                        tiles_x, ntiles, select, sel_pitch);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

}  // namespace

extern "C" int hd_expand(const void* in, int in_dtype, int64_t in_pitch, void* out, int out_dtype, int64_t out_pitch,
                         int64_t ny, int64_t nx, int ws, void* stream)
{
    if (!in || !out) return HD_ERR_NULL;
    if (int e = check_window(ny, nx, ws)) return e;
    const int h = ws / 2;
    if (h < 1 || h > MAX_HALO - 1) return HD_ERR_UNSUPPORTED;
    if (in_pitch < nx || out_pitch < nx) return HD_ERR_ARG;
    if (in_dtype != HD_U8 && in_dtype != HD_F32) return HD_ERR_UNSUPPORTED;
    const int in_w = TW + 2 * hd_halo_x(h, (int)hd_dtype_size(in_dtype)), in_h = TH + 2 * h;
    if (in_w > MAX_IN_W) return HD_ERR_UNSUPPORTED;
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, in_dtype, ny, nx, in_pitch, in_w, in_h, false)) return e;
    cudaStream_t s = (cudaStream_t)stream;
#define HD_EXPAND_CASE(IT, ITAG, OT, OTAG) \
    if (in_dtype == ITAG && out_dtype == OTAG) return launch_expand<IT, OT>(tm, out, out_pitch, ny, nx, h, in_w, in_h, s);
    HD_EXPAND_CASE(float, HD_F32, uint8_t, HD_U8)
    HD_EXPAND_CASE(float, HD_F32, float, HD_F32)
    HD_EXPAND_CASE(float, HD_F32, double, HD_F64)
    HD_EXPAND_CASE(uint8_t, HD_U8, uint8_t, HD_U8)
    HD_EXPAND_CASE(uint8_t, HD_U8, float, HD_F32)
    HD_EXPAND_CASE(uint8_t, HD_U8, double, HD_F64)
#undef HD_EXPAND_CASE
    return HD_ERR_UNSUPPORTED;
}

extern "C" int hd_expand_select(const void* in, int in_dtype, int64_t in_pitch, const void* select, int64_t sel_pitch,
                                void* out, int64_t out_pitch, int64_t ny, int64_t nx, int ws, void* stream)
{
    if (!in || !out || !select) return HD_ERR_NULL;
    if (int e = check_window(ny, nx, ws)) return e;
    const int h = ws / 2;
    if (h < 1 || h > MAX_HALO - 1) return HD_ERR_UNSUPPORTED;
    if (in_pitch < nx || out_pitch < nx || sel_pitch < nx) return HD_ERR_ARG;
    if (in_dtype != HD_U8 && in_dtype != HD_F32) return HD_ERR_UNSUPPORTED;
    const int in_w = TW + 2 * hd_halo_x(h, (int)hd_dtype_size(in_dtype)), in_h = TH + 2 * h;
    if (in_w > MAX_IN_W) return HD_ERR_UNSUPPORTED;
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, in_dtype, ny, nx, in_pitch, in_w, in_h, false)) return e;
    cudaStream_t s = (cudaStream_t)stream;
    if (in_dtype == HD_U8)
        return launch_expand<uint8_t, float>(tm, out, out_pitch, ny, nx, h, in_w, in_h, s, (const float*)select, sel_pitch);
    return launch_expand<float, float>(tm, out, out_pitch, ny, nx, h, in_w, in_h, s, (const float*)select, sel_pitch);
}

extern "C" int hd_binary_morph(const void* in, int in_dtype, int64_t in_pitch, void* out, int64_t out_pitch, int64_t ny,
                               int64_t nx, int op, int full_structure, int iterations, void* stream)
{
    if (!in || !out) return HD_ERR_NULL;
    if (ny <= 0 || nx <= 0 || in_pitch < nx || out_pitch < nx || iterations < 1) return HD_ERR_ARG;
    MorphProgram prog{};
    if (op == HD_MORPH_ERODE || op == HD_MORPH_DILATE) {
        if (iterations > MAX_HALO) return HD_ERR_UNSUPPORTED;
        prog.nsteps = iterations;
        for (int i = 0; i < iterations; ++i) { prog.dilate[i] = (op == HD_MORPH_DILATE); prog.full[i] = full_structure != 0; }
    } else if (op == HD_MORPH_CLOSE || op == HD_MORPH_OPEN) {
        if (2 * iterations > MAX_HALO) return HD_ERR_UNSUPPORTED;
        prog.nsteps = 2 * iterations;
        for (int i = 0; i < 2 * iterations; ++i) {
            const bool first = i < iterations;
            prog.dilate[i] = (op == HD_MORPH_CLOSE) ? first : !first;
            prog.full[i] = full_structure != 0;
        }
    } else {
        return HD_ERR_ARG;
    }
    const int h = prog.nsteps;
    if (in_dtype != HD_U8 && in_dtype != HD_F32) return HD_ERR_UNSUPPORTED;
    const int in_w = TW + 2 * hd_halo_x(h, (int)hd_dtype_size(in_dtype)), in_h = TH + 2 * h;
    if (in_w > MAX_IN_W) return HD_ERR_UNSUPPORTED;
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, in_dtype, ny, nx, in_pitch, in_w, in_h, false)) return e;
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t smem = 2 * STAGE_BYTES;
    cudaStream_t s = (cudaStream_t)stream;
    if (in_dtype == HD_F32) {
        HD_CUDA_OK(cudaFuncSetAttribute(morph_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("morph_kernel", s);
        morph_kernel<float><<<grid_for(ntiles, 3), NT, smem, s>>>(tm, (uint8_t*)out, out_pitch, ny, nx, prog, in_w, in_h,
                                                                 tiles_x, ntiles);
    } else if (in_dtype == HD_U8) {
        HD_CUDA_OK(cudaFuncSetAttribute(morph_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("morph_kernel", s);
        morph_kernel<uint8_t><<<grid_for(ntiles, 3), NT, smem, s>>>(tm, (uint8_t*)out, out_pitch, ny, nx, prog, in_w, in_h,
                                                                   tiles_x, ntiles);
    } else {
        return HD_ERR_UNSUPPORTED;
    }
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

extern "C" int hd_max_filter(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny,
                             int64_t nx, int size, void* stream)
{
    if (!in || !out) return HD_ERR_NULL;
    if (size % 2 != 1 || size < 1) return HD_ERR_WINDOW_EVEN;
    if (size > ny || size > nx) return HD_ERR_WINDOW_HIGH;
    const int h = size / 2;
    if (h > MAX_HALO) return HD_ERR_UNSUPPORTED;
    if (in_pitch < nx || out_pitch < nx) return HD_ERR_ARG;
    if (dtype != HD_F32 && dtype != HD_F64) return HD_ERR_UNSUPPORTED;
    const size_t es = hd_dtype_size(dtype);
    const int in_w = TW + 2 * hd_halo_x(h, (int)es), in_h = TH + 2 * h;
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, dtype, ny, nx, in_pitch, in_w, in_h, false)) return e;
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t smem = 2 * MAX_IN_H * (TW + 2 * MAX_HALO) * es + MAX_IN_H * TW * es;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == HD_F32 && h == 3) {
        HD_CUDA_OK(cudaFuncSetAttribute(maxfilter_kernel<float, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("maxfilter_kernel", s);
        maxfilter_kernel<float, 3><<<grid_for(ntiles, 2), NT, smem, s>>>(tm, (float*)out, out_pitch, ny, nx, h, in_w, in_h,
                                                                        tiles_x, ntiles);
    } else if (dtype == HD_F32) {
        HD_CUDA_OK(cudaFuncSetAttribute(maxfilter_kernel<float, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("maxfilter_kernel", s);
        maxfilter_kernel<float, 0><<<grid_for(ntiles, 2), NT, smem, s>>>(tm, (float*)out, out_pitch, ny, nx, h, in_w, in_h,
                                                                        tiles_x, ntiles);
    } else {
        HD_CUDA_OK(cudaFuncSetAttribute(maxfilter_kernel<double, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("maxfilter_kernel", s);
        maxfilter_kernel<double, 0><<<grid_for(ntiles, 1), NT, smem, s>>>(tm, (double*)out, out_pitch, ny, nx, h, in_w, in_h,
                                                                         tiles_x, ntiles);
    }
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

extern "C" int hd_binary_morph_struct(const void* in, int in_dtype, int64_t in_pitch, void* out, int64_t out_pitch,
                                      int64_t ny, int64_t nx, int dilate, int ntaps, const int* tap_dy, const int* tap_dx,
                                      int iterations, int* changed, void* stream)
{
    if (!in || !out || (ntaps > 0 && (!tap_dy || !tap_dx))) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || in_pitch < nx || out_pitch < nx || ntaps < 0 || iterations < 1) return HD_ERR_ARG;
    if (in_dtype != HD_U8 && in_dtype != HD_F32) return HD_ERR_UNSUPPORTED;
    if (ntaps > MS_MAX_TAPS) return HD_ERR_UNSUPPORTED;
    MorphTaps p;
    p.ntaps = ntaps;
    int ry = 0, rx = 0;
    for (int t = 0; t < ntaps; ++t) {
        const int ay = tap_dy[t] < 0 ? -tap_dy[t] : tap_dy[t], ax = tap_dx[t] < 0 ? -tap_dx[t] : tap_dx[t];
        if (ay > MS_MAX_REACH || ax > MS_MAX_REACH) return HD_ERR_UNSUPPORTED;
        ry = ay > ry ? ay : ry;
        rx = ax > rx ? ax : rx;
        p.dy[t] = (signed char)tap_dy[t];
        p.dx[t] = (signed char)tap_dx[t];
    }
    if (iterations * ry > MS_MAX_REACH || iterations * rx > MS_MAX_REACH) return HD_ERR_UNSUPPORTED;
    const int hy = iterations * ry, hx = hd_halo_x(iterations * rx, (int)hd_dtype_size(in_dtype));
    const int in_w = TW + 2 * hx, in_h = TH + 2 * hy;
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, in_dtype, ny, nx, in_pitch, in_w, in_h, false)) return e;
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t smem = 2 * (size_t)MS_STAGE;
    cudaStream_t s = (cudaStream_t)stream;
    if (changed) HD_CUDA_OK(cudaMemsetAsync(changed, 0, sizeof(int), s));
    if (in_dtype == HD_F32) {
        HD_CUDA_OK(cudaFuncSetAttribute(morph_struct_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("morph_struct_kernel", s);
        morph_struct_kernel<float><<<grid_for(ntiles, 2), NT, smem, s>>>(tm, (uint8_t*)out, out_pitch, ny, nx, p, dilate != 0,
                                                                        iterations, hy, hx, in_w, in_h, tiles_x, ntiles, changed);
    } else {
        HD_CUDA_OK(cudaFuncSetAttribute(morph_struct_kernel<uint8_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("morph_struct_kernel", s);
        morph_struct_kernel<uint8_t><<<grid_for(ntiles, 2), NT, smem, s>>>(tm, (uint8_t*)out, out_pitch, ny, nx, p, dilate != 0,
                                                                          iterations, hy, hx, in_w, in_h, tiles_x, ntiles,
                                                                          changed);
    }
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

extern "C" int hd_max_filter_rect(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny,
                                  int64_t nx, int size_y, int size_x, void* workspace, int64_t workspace_bytes, void* stream)
{
    if (!in || !out || !workspace) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || in_pitch < nx || out_pitch < nx || size_y < 1 || size_x < 1) return HD_ERR_ARG;
    if (dtype != HD_F32 && dtype != HD_F64) return HD_ERR_UNSUPPORTED;
    if (size_y > 255 || size_x > 255) return HD_ERR_UNSUPPORTED;
    if (workspace_bytes < ny * nx * (int64_t)hd_dtype_size(dtype)) return HD_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == HD_F32) return launch_max_rect<float>(in, in_pitch, out, out_pitch, ny, nx, size_y, size_x, workspace, s);
    return launch_max_rect<double>(in, in_pitch, out, out_pitch, ny, nx, size_y, size_x, workspace, s);
}

// TidyingLagoons.apply (custom_filters.py:587-610) in one kernel: majority (F32) -> lagoon values (F32).
extern "C" int hd_tidy_lagoons(const void* majority, int64_t in_pitch, void* out, int64_t out_pitch, int64_t ny, int64_t nx,
                               void* stream)
{
    if (!majority || !out) return HD_ERR_NULL;
    if (int e = check_window(ny, nx, 7)) return e;
    if (in_pitch < nx || out_pitch < nx || majority == out) return HD_ERR_ARG;
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, majority, HD_F32, ny, nx, in_pitch, TL_IN_W, TL_IN_H, false)) return e;
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t smem = 2 * (size_t)TL_STAGE + (size_t)TL_PH * TL_PW * 4 + (size_t)TL_PH * TW * 4;
    HD_CUDA_OK(cudaFuncSetAttribute(tidy_lagoons_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    hd_prof_begin("tidy_lagoons_kernel", (cudaStream_t)stream);
    tidy_lagoons_kernel<<<grid_for(ntiles, 2), TL_NT, smem, (cudaStream_t)stream>>>(tm, (float*)out, out_pitch, ny, nx, tiles_x,
                                                                              ntiles);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

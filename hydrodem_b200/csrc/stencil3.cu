// 3x3 stencils of the conditioning chain.
//
//   hd_nanfix     CorrectNANValues.apply   custom_filters.py:286-317   (bit-exact float32 mean, numpy order)
//   hd_isolated   IsolatedPoints.apply     custom_filters.py:345-366
//   hd_convolve3  Convolve.apply + Around  extension_filters.py:166-184, :113-130 (PostProcessingFinal)
//   hd_correlate  Convolve.apply          extension_filters.py:166-184, any weights up to 31x31
//
// HBM-bound: 4 B read + 4 B written per cell (8 + 8 for float64 rasters).  A 32x128 tile with a one-cell
// halo is staged by TMA; each thread produces 4 consecutive cells of 4 rows and stores them as one
// 16-byte coalesced write.
#include "common.cuh"
#include "tile_common.cuh"

namespace {

constexpr int IN_H3 = TH + 2;

// ---- CorrectNANValues ----------------------------------------------------------------------------
// numpy float32 add.reduce over the compacted neighbour list (row-major, centre dropped, NaN and
// negatives dropped): n < 8 -> left-to-right from -0.0; n == 8 -> ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)).
__device__ __forceinline__ float nanfix_mean(const float (&v)[8])
{
    bool ok[8];
    int n = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) { ok[k] = v[k] >= 0.f; n += ok[k]; }   // NaN >= 0 is false  (:314-315)
    if (n == 0) return __int_as_float(0x7fc00000);                     // mean of empty slice
    float s;
    if (n == 8) {
        s = __fadd_rn(__fadd_rn(__fadd_rn(v[0], v[1]), __fadd_rn(v[2], v[3])),
                      __fadd_rn(__fadd_rn(v[4], v[5]), __fadd_rn(v[6], v[7])));
    } else {
        s = -0.0f;
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (ok[k]) s = __fadd_rn(s, v[k]);
    }
    return __fdiv_rn(s, (float)n);                                     // float32 sum / count  (:316)
}

// Four consecutive tile cells starting at a 16-byte aligned position, as ONE shared-memory access per lane
// (LDS.128 / 2 x LDS.128): lanes sit 16 (32) bytes apart, so a quarter-warp reads one contiguous 128-byte
// segment -- conflict free, where four scalar reads at a 4-cell lane stride are 4-way bank conflicts.
template <typename T> __device__ __forceinline__ void load_quad(const T* p, T (&q)[4]);
template <> __device__ __forceinline__ void load_quad<float>(const float* p, float (&q)[4])
{
    const float4 v = *reinterpret_cast<const float4*>(p);
    q[0] = v.x; q[1] = v.y; q[2] = v.z; q[3] = v.w;
}
template <> __device__ __forceinline__ void load_quad<double>(const double* p, double (&q)[4])
{
    const double2 a = reinterpret_cast<const double2*>(p)[0], b = reinterpret_cast<const double2*>(p)[1];
    q[0] = a.x; q[1] = a.y; q[2] = b.x; q[3] = b.y;
}

template <int MODE, typename T>   // MODE 0 = nanfix, 1 = isolated; T = raster dtype (windows are cast to float32)
__global__ void __launch_bounds__(NT) fix3_kernel(const __grid_constant__ CUtensorMap tm_in, T* __restrict__ out,
                                                  int64_t out_pitch, int64_t ny, int64_t nx, int in_w, int tiles_x,
                                                  int ntiles)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    const uint32_t stage_bytes = (uint32_t)((in_w * IN_H3 * sizeof(T) + 127) / 128 * 128);
    constexpr int HX = hd_halo_x(1, sizeof(T));
    const TilePlane planes[1] = {{&tm_in, 0u, (uint32_t)(in_w * IN_H3 * sizeof(T)), HX, 1}};
    tile_loop<1>(smem, stage_bytes, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        const T* tile = reinterpret_cast<const T*>(st);
#pragma unroll
        for (int rep = 0; rep < TH * TW / 4 / NT; ++rep) {
            const int idx = rep * NT + threadIdx.x;
            const int ro = idx >> 5, c4 = idx & 31;
            const int64_t y = ty0 + ro, x = tx0 + 4 * c4;
            if (y >= ny || x >= nx) continue;
            const T* c = tile + (ro + 1) * in_w + 4 * c4 + HX;
            T v[4], own[4];
            load_quad<T>(c, own);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float ctr = (float)own[j];               // grid.astype('float32'), sliding_window.py:132
                T r = own[j];
                const bool interior = y >= 1 && y < ny - 1 && x + j >= 1 && x + j < nx - 1;
                // iter_over_ones gate: int(v) == 1  (sliding_window.py:192)
                const bool gate = MODE == 0 ? (ctr < 0.f) : (ctr >= 1.f && ctr < 2.f);
                if (interior && gate) {
                    const float nb[8] = {(float)c[j - in_w - 1], (float)c[j - in_w],     (float)c[j - in_w + 1],
                                         (float)c[j - 1],        (float)c[j + 1],        (float)c[j + in_w - 1],
                                         (float)c[j + in_w],     (float)c[j + in_w + 1]};
                    if (MODE == 0) {
                        r = (T)nanfix_mean(nb);
                    } else {
                        bool any = false;
#pragma unroll
                        for (int k = 0; k < 8; ++k) any |= nb[k] > 0.f;     // NaN > 0 false (:364-365)
                        r = any ? (T)1 : (T)0;
                    }
                }
                v[j] = r;
            }
            store4v<T>(out, out_pitch, y, x, nx, v);
        }
    });
}

// ---- Convolve (3x3, reflect) + Around --------------------------------------------------------------
struct Conv3Params { double w[9]; double divisor; int do_round; };

template <typename T> __device__ __forceinline__ T div_round(T v, double divisor, int do_round);
template <> __device__ __forceinline__ float div_round<float>(float v, double divisor, int do_round)
{
    float r = __fdiv_rn(v, (float)divisor);
    return do_round ? rintf(r) : r;
}
template <> __device__ __forceinline__ double div_round<double>(double v, double divisor, int do_round)
{
    double r = __ddiv_rn(v, divisor);
    return do_round ? rint(r) : r;
}

template <typename T>
__global__ void __launch_bounds__(NT) conv3_kernel(const __grid_constant__ CUtensorMap tm_in, T* __restrict__ out,
                                                   int64_t out_pitch, float* __restrict__ out32, int64_t out32_pitch,
                                                   int64_t ny, int64_t nx, Conv3Params p, int in_w, int tiles_x, int ntiles)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    const uint32_t stage_bytes = (uint32_t)((in_w * IN_H3 * sizeof(T) + 127) / 128 * 128);
    constexpr int HX = hd_halo_x(1, sizeof(T));
    const TilePlane planes[1] = {{&tm_in, 0u, (uint32_t)(in_w * IN_H3 * sizeof(T)), HX, 1}};
    // V consecutive cells per thread = one 16-byte shared-memory read per window row: lanes 16 bytes apart are
    // conflict free (four float64 cells per thread, 32 bytes apart, made every LDS.128 a 2-way conflict)
    constexpr int V = 16 / (int)sizeof(T);
    constexpr int TPR = TW / V;                                  // threads per tile row
    tile_loop<1>(smem, stage_bytes, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        T* tile = reinterpret_cast<T*>(st);
        patch_reflect<T>(tile, in_w, IN_H3, ty0 - 1, tx0 - HX, ny, nx);
#pragma unroll
        for (int rep = 0; rep < TH * TW / V / NT; ++rep) {
            const int idx = rep * NT + threadIdx.x;
            const int ro = idx / TPR, cv = idx % TPR;
            const int64_t y = ty0 + ro, x = tx0 + V * cv;
            if (y >= ny || x >= nx) continue;
            const T* c = tile + ro * in_w + V * cv + HX;      // first of the V centre columns, top window row
            T win[3][V + 2];                                  // 3 window rows x (V centres + left and right neighbour)
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                const int4 raw = *reinterpret_cast<const int4*>(c + dy * in_w);
                const T* q = reinterpret_cast<const T*>(&raw);
                win[dy][0] = c[dy * in_w - 1];
#pragma unroll
                for (int j = 0; j < V; ++j) win[dy][j + 1] = q[j];
                win[dy][V + 1] = c[dy * in_w + V];
            }
            T v[V];
#pragma unroll
            for (int j = 0; j < V; ++j) {
                double acc = 0.0;                             // NI_Correlate: tmp = 0; tmp += in * w, row-major
#pragma unroll
                for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) {
                        const double w = p.w[dy * 3 + dx];
                        if (w != 0.0) acc = __dadd_rn(acc, __dmul_rn((double)win[dy][j + dx], w));
                    }
                v[j] = div_round<T>((T)acc, p.divisor, p.do_round);
            }
            T* po = out + y * out_pitch + x;
            if (x + V - 1 < nx && ((reinterpret_cast<uintptr_t>(po) & 15) == 0)) {
                int4 packed;
                T* pv = reinterpret_cast<T*>(&packed);
#pragma unroll
                for (int j = 0; j < V; ++j) pv[j] = v[j];
                *reinterpret_cast<int4*>(po) = packed;
            } else {
#pragma unroll
                for (int j = 0; j < V; ++j)
                    if (x + j < nx) po[j] = v[j];
            }
            if (out32) {                                      // optional float32 copy of the result (feeds the sink-fill)
                float* p32 = out32 + y * out32_pitch + x;
#pragma unroll
                for (int j = 0; j < V; ++j)
                    if (x + j < nx) p32[j] = (float)v[j];
            }
        }
    });
}

// ---- Convolve with any weights up to 31 x 31 (reflect) ----------------------------------------------------------------
// The host hands over NI_Correlate's footprint as a tap list: offsets (dy, dx) from the output cell, already flipped and
// origin-shifted for a convolution, with the weights |w| <= DBL_EPSILON left out, in the order the sum runs.  The list
// lives in kernel-parameter (constant) memory: every thread reads the same tap at the same time.
constexpr int CORR_MAX_REACH = 15;                       // 31 x 31 weights
constexpr int CORR_MAX_TAPS = (2 * CORR_MAX_REACH + 1) * (2 * CORR_MAX_REACH + 1);
constexpr int CORR_ROWS = TH * TW / NT;                  // output cells per thread, one column, every other row

struct CorrTaps {
    int ntaps;
    int off[CORR_MAX_TAPS];       // (hy + dy) * in_w + hx + dx: staged-box offset of the tap from the output cell's (ro, co)
    double w[CORR_MAX_TAPS];
};

template <typename T>
__global__ void __launch_bounds__(NT) correlate_kernel(const __grid_constant__ CUtensorMap tm_in, T* __restrict__ out,
                                                       int64_t out_pitch, int64_t ny, int64_t nx,
                                                       const __grid_constant__ CorrTaps p, double divisor, int hy, int hx,
                                                       int in_w, int in_h, int tiles_x, int ntiles)
{
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    const uint32_t stage_bytes = (uint32_t)((in_w * in_h * sizeof(T) + 127) / 128 * 128);
    const TilePlane planes[1] = {{&tm_in, 0u, (uint32_t)(in_w * in_h * sizeof(T)), hx, hy}};
    // lanes take consecutive columns (conflict-free shared-memory reads); rows rg, rg + 2, ... give each thread
    // CORR_ROWS independent accumulators for one weight read
    const int co = threadIdx.x % TW, rg = threadIdx.x / TW;
    constexpr int RSTEP = NT / TW;
    tile_loop<1>(smem, stage_bytes, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        T* tile = reinterpret_cast<T*>(st);
        patch_reflect<T, true>(tile, in_w, in_h, ty0 - hy, tx0 - hx, ny, nx);
        const T* base = tile + rg * in_w + co;
        double acc[CORR_ROWS];
#pragma unroll
        for (int i = 0; i < CORR_ROWS; ++i) acc[i] = 0.0;     // NI_Correlate: tmp = 0.0; tmp += in * w, footprint order
        for (int t = 0; t < p.ntaps; ++t) {
            const double w = p.w[t];
            const T* q = base + p.off[t];
#pragma unroll
            for (int i = 0; i < CORR_ROWS; ++i) acc[i] = __dadd_rn(acc[i], __dmul_rn((double)q[i * RSTEP * in_w], w));
        }
        const int64_t x = tx0 + co;
        if (x < nx) {
#pragma unroll
            for (int i = 0; i < CORR_ROWS; ++i) {
                const int64_t y = ty0 + rg + i * RSTEP;
                if (y < ny) out[y * out_pitch + x] = div_round<T>((T)acc[i], divisor, 0);   // cast, then / weights.size
            }
        }
    });
}

// ---- _prepare_final_terms + the three-term sum + PostProcessingFinal in ONE pass (no rivers) ----------------------------
// hydro_dem_process.py:60-91, :148-149 with rivers = 0:  complete = srtm * (1 - mask) + lagoon_values + hsheds * 0,
// mask = lagoon_values > 0, then Convolve(ones(3,3)) / 9 (mode='reflect') and Around.  With 0/1 masks `complete` is
// either the SRTM cell or the lagoon value (or NaN when a term is not finite) -- exactly a float32 -- so the staged
// 34 x 136 block of it lives in shared memory as float32 and the 3x3 mean accumulates it in double in scipy's order:
// the result is bit-identical to hd_final_terms + hd_convolve3, for 16 B/cell of HBM traffic instead of 40 (the float64
// `complete` raster and the float64 copy of the rounded DEM are never written unless asked for).
template <bool WITH_COMPLETE>
__global__ void __launch_bounds__(NT) final_mean3_kernel(const __grid_constant__ CUtensorMap tm_srtm,
                                                         const __grid_constant__ CUtensorMap tm_lag,
                                                         const __grid_constant__ CUtensorMap tm_hs, float* __restrict__ out32,
                                                         int64_t out32_pitch, double* __restrict__ complete,
                                                         int64_t complete_pitch, int64_t ny, int64_t nx, int tiles_x, int ntiles)
{
    constexpr int HX = hd_halo_x(1, 4);
    constexpr int IN_W = TW + 2 * HX;
    constexpr uint32_t PLANE = (uint32_t)((IN_W * IN_H3 * 4 + 127) / 128 * 128);
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bars[2];
    float* cplt = reinterpret_cast<float*>(smem + 3 * PLANE);            // [IN_H3][IN_W]
    const TilePlane planes[3] = {{&tm_srtm, 0u, (uint32_t)(IN_W * IN_H3 * 4), HX, 1},
                                 {&tm_lag, PLANE, (uint32_t)(IN_W * IN_H3 * 4), HX, 1},
                                 {&tm_hs, 2 * PLANE, (uint32_t)(IN_W * IN_H3 * 4), HX, 1}};
    tile_loop<3, 1>(smem, 3 * PLANE, bars, planes, TW, TH, tiles_x, ntiles, [&](unsigned char* st, int ty0, int tx0) {
        const float* ps = reinterpret_cast<const float*>(st);
        const float* pl = reinterpret_cast<const float*>(st + PLANE);
        const float* ph = reinterpret_cast<const float*>(st + 2 * PLANE);
        for (int t = threadIdx.x; t < IN_W * IN_H3; t += NT) {
            const double s = (double)ps[t], lv = (double)pl[t];
            const double mask = lv > 0.0 ? 1.0 : 0.0;
            const double first = __dmul_rn(s, 1.0 - (mask + 0.0));
            double acc = __dadd_rn(first, lv);
            acc = __dadd_rn(acc, 0.0 * (double)ph[t]);
            cplt[t] = (float)acc;
            if (WITH_COMPLETE) {
                const int r = t / IN_W, c = t - r * IN_W;
                const int64_t y = (int64_t)ty0 - 1 + r, x = (int64_t)tx0 - HX + c;
                if (r >= 1 && r <= TH && c >= HX && c < HX + TW && y < ny && x < nx) complete[y * complete_pitch + x] = acc;
            }
        }
        __syncthreads();
        patch_reflect<float>(cplt, IN_W, IN_H3, ty0 - 1, tx0 - HX, ny, nx);
#pragma unroll
        for (int rep = 0; rep < TH * TW / 4 / NT; ++rep) {
            const int idx = rep * NT + threadIdx.x;
            const int ro = idx >> 5, c4 = idx & 31;
            const int64_t y = ty0 + ro, x = tx0 + 4 * c4;
            if (y >= ny || x >= nx) continue;
            const float* c = cplt + ro * IN_W + 4 * c4 + HX;
            float win[3][6];
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                const float4 q = *reinterpret_cast<const float4*>(c + dy * IN_W);
                win[dy][0] = c[dy * IN_W - 1];
                win[dy][1] = q.x; win[dy][2] = q.y; win[dy][3] = q.z; win[dy][4] = q.w;
                win[dy][5] = c[dy * IN_W + 4];
            }
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                double acc = 0.0;                             // NI_Correlate: tmp = 0; tmp += in * w, row-major (w = 1)
#pragma unroll
                for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                    for (int dx = 0; dx < 3; ++dx) acc = __dadd_rn(acc, __dmul_rn((double)win[dy][j + dx], 1.0));
                v[j] = (float)rint(__ddiv_rn(acc, 9.0));      // / weights.size, np.around; integer metres: exact in float32
            }
            store4<float>(out32, out32_pitch, y, x, nx, v);
        }
    });
}

template <int MODE>
int launch_fix3(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
                void* stream)
{
    if (!in || !out) return HD_ERR_NULL;
    if (int e = check_window(ny, nx, 3)) return e;
    if (in_pitch < nx || out_pitch < nx) return HD_ERR_ARG;
    if (dtype != HD_F32 && dtype != HD_F64) return HD_ERR_UNSUPPORTED;
    const size_t es = hd_dtype_size(dtype);
    const int in_w = TW + 2 * hd_halo_x(1, (int)es);           // one-cell halo rounded up to 16 bytes per side
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, dtype, ny, nx, in_pitch, in_w, IN_H3, false)) return e;
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t smem = 2 * ((in_w * IN_H3 * es + 127) / 128 * 128);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == HD_F32) {
        hd_prof_begin("fix3_kernel", s);
        fix3_kernel<MODE, float><<<grid_for(ntiles, 4), NT, smem, s>>>(tm, (float*)out, out_pitch, ny, nx, in_w, tiles_x,
                                                                      ntiles);
    } else {
        HD_CUDA_OK(cudaFuncSetAttribute(fix3_kernel<MODE, double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("fix3_kernel", s);
        fix3_kernel<MODE, double><<<grid_for(ntiles, 3), NT, smem, s>>>(tm, (double*)out, out_pitch, ny, nx, in_w, tiles_x,
                                                                       ntiles);
    }
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

}  // namespace

extern "C" int hd_nanfix(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny,
                         int64_t nx, void* stream)
{
    return launch_fix3<0>(in, in_pitch, out, out_pitch, dtype, ny, nx, stream);
}

extern "C" int hd_isolated(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny,
                           int64_t nx, void* stream)
{
    return launch_fix3<1>(in, in_pitch, out, out_pitch, dtype, ny, nx, stream);
}

extern "C" int hd_convolve3(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny,
                            int64_t nx, const double* weights, double divisor, int do_round, void* out32,
                            int64_t out32_pitch, void* stream)
{
    if (!in || !out || !weights) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || in_pitch < nx || out_pitch < nx || (out32 && out32_pitch < nx)) return HD_ERR_ARG;
    if (dtype != HD_F32 && dtype != HD_F64) return HD_ERR_UNSUPPORTED;
    Conv3Params p;
    for (int k = 0; k < 9; ++k) p.w[k] = weights[k];
    p.divisor = divisor;
    p.do_round = do_round;
    const size_t es = hd_dtype_size(dtype);
    const int in_w = TW + 2 * hd_halo_x(1, (int)es);
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, dtype, ny, nx, in_pitch, in_w, IN_H3, false)) return e;
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t smem = 2 * ((in_w * IN_H3 * es + 127) / 128 * 128);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == HD_F32) {
        hd_prof_begin("conv3_kernel", s);
        conv3_kernel<float><<<grid_for(ntiles, 4), NT, smem, s>>>(tm, (float*)out, out_pitch, (float*)out32, out32_pitch, ny, nx, p,
                                                                 in_w, tiles_x, ntiles);
    } else {
        HD_CUDA_OK(cudaFuncSetAttribute(conv3_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("conv3_kernel", s);
        conv3_kernel<double><<<grid_for(ntiles, 3), NT, smem, s>>>(tm, (double*)out, out_pitch, (float*)out32, out32_pitch, ny, nx,
                                                                  p, in_w, tiles_x, ntiles);
    }
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

extern "C" int hd_correlate(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny,
                            int64_t nx, int ntaps, const int* tap_dy, const int* tap_dx, const double* tap_w, double divisor,
                            void* stream)
{
    if (!in || !out || (ntaps > 0 && (!tap_dy || !tap_dx || !tap_w))) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || in_pitch < nx || out_pitch < nx || ntaps < 0) return HD_ERR_ARG;
    if (dtype != HD_F32 && dtype != HD_F64) return HD_ERR_UNSUPPORTED;
    if (ntaps > CORR_MAX_TAPS) return HD_ERR_UNSUPPORTED;
    int ry = 0, rx = 0;
    for (int t = 0; t < ntaps; ++t) {
        const int ay = tap_dy[t] < 0 ? -tap_dy[t] : tap_dy[t], ax = tap_dx[t] < 0 ? -tap_dx[t] : tap_dx[t];
        if (ay > CORR_MAX_REACH || ax > CORR_MAX_REACH) return HD_ERR_UNSUPPORTED;
        ry = ay > ry ? ay : ry;
        rx = ax > rx ? ax : rx;
    }
    const size_t es = hd_dtype_size(dtype);
    const int hx = hd_halo_x(rx, (int)es), in_w = TW + 2 * hx, in_h = TH + 2 * ry;
    static thread_local CorrTaps q;                           // 11.5 KB: kept off the caller's stack
    static_assert(sizeof(CorrTaps) <= 32000, "kernel parameters are limited to 32 KB");
    q.ntaps = ntaps;
    for (int t = 0; t < ntaps; ++t) {
        q.off[t] = (ry + tap_dy[t]) * in_w + hx + tap_dx[t];
        q.w[t] = tap_w[t];
    }
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, dtype, ny, nx, in_pitch, in_w, in_h, false)) return e;
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t smem = 2 * ((in_w * in_h * es + 127) / 128 * 128);
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == HD_F32) {
        HD_CUDA_OK(cudaFuncSetAttribute(correlate_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("correlate_kernel", s);
        correlate_kernel<float><<<grid_for(ntiles, 2), NT, smem, s>>>(tm, (float*)out, out_pitch, ny, nx, q, divisor, ry, hx,
                                                                     in_w, in_h, tiles_x, ntiles);
    } else {
        HD_CUDA_OK(cudaFuncSetAttribute(correlate_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        hd_prof_begin("correlate_kernel", s);
        correlate_kernel<double><<<grid_for(ntiles, 1), NT, smem, s>>>(tm, (double*)out, out_pitch, ny, nx, q, divisor, ry, hx,
                                                                      in_w, in_h, tiles_x, ntiles);
    }
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

// srtm (groves-corrected DEM), lagoon_values, hsheds_fixed: F32 rasters.  final32 (F32): the rounded 3x3 mean of
// `complete` = srtm * (1 - (lagoon_values > 0)) + lagoon_values + hsheds_fixed * 0 (hydro_dem_process.py:60-91, :148-149,
// no rivers).  complete_out (F64, may be NULL): `complete` itself.  Same bits as hd_final_terms + hd_convolve3.
extern "C" int hd_final_mean3(const void* srtm, int64_t srtm_pitch, const void* lagoon_values, int64_t lag_pitch,
                              const void* hsheds_fixed, int64_t hs_pitch, void* final32, int64_t final32_pitch,
                              void* complete_out, int64_t complete_pitch, int64_t ny, int64_t nx, void* stream)
{
    if (!srtm || !lagoon_values || !hsheds_fixed || !final32) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || srtm_pitch < nx || lag_pitch < nx || hs_pitch < nx || final32_pitch < nx ||
        (complete_out && complete_pitch < nx))
        return HD_ERR_ARG;
    constexpr int IN_W = TW + 2 * hd_halo_x(1, 4);
    CUtensorMap tms, tml, tmh;
    if (int e = hd_make_tmap_2d(&tms, srtm, HD_F32, ny, nx, srtm_pitch, IN_W, IN_H3, false)) return e;
    if (int e = hd_make_tmap_2d(&tml, lagoon_values, HD_F32, ny, nx, lag_pitch, IN_W, IN_H3, false)) return e;
    if (int e = hd_make_tmap_2d(&tmh, hsheds_fixed, HD_F32, ny, nx, hs_pitch, IN_W, IN_H3, false)) return e;
    const int tiles_x = hd_cdiv(nx, TW), tiles_y = hd_cdiv(ny, TH), ntiles = tiles_x * tiles_y;
    const size_t plane = (IN_W * IN_H3 * 4 + 127) / 128 * 128, smem = 4 * plane;
    cudaStream_t s = (cudaStream_t)stream;
    hd_prof_begin("final_mean3_kernel", s);
    if (complete_out) {
        HD_CUDA_OK(cudaFuncSetAttribute(final_mean3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        final_mean3_kernel<true><<<grid_for(ntiles, 3), NT, smem, s>>>(tms, tml, tmh, (float*)final32, final32_pitch,
                                                                      (double*)complete_out, complete_pitch, ny, nx, tiles_x,
                                                                      ntiles);
    } else {
        HD_CUDA_OK(cudaFuncSetAttribute(final_mean3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        final_mean3_kernel<false><<<grid_for(ntiles, 3), NT, smem, s>>>(tms, tml, tmh, (float*)final32, final32_pitch, nullptr, 0,
                                                                       ny, nx, tiles_x, ntiles);
    }
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

// Elementwise filters of the reference (filters/simple_filters.py, extension_filters.py:12-130) as one
// dtype-generic kernel.  These are HBM-bound streaming ops; inside the fused chain they never run alone
// (they are folded into the neighbouring stencil kernels) -- this entry point exists so that each
// reference class has a device implementation behind the same Filter.apply() API.
#include <cstring>
#include <type_traits>

#include "common.cuh"
#include "tile_common.cuh"

namespace {

// Every op is evaluated in the dtype of NumPy's ufunc loop (the compute type C): both operands are converted to C
// as ndarray.astype would, the op runs in C with NumPy's semantics, and the result is converted to out_dtype.
struct cf { float re, im; };
struct cd { double re, im; };
template <typename T> constexpr bool is_cplx = std::is_same_v<T, cf> || std::is_same_v<T, cd>;
template <typename T> using part_t = std::conditional_t<std::is_same_v<T, cf>, float, double>;
// integer arithmetic wraps: done on unsigned words at least as wide as int, so no promotion overflows
template <typename T> using word_t = std::conditional_t<sizeof(T) == 8, uint64_t, uint32_t>;

template <typename S> __device__ __forceinline__ bool nonzero(S v)
{
    if constexpr (is_cplx<S>) return v.re != 0 || v.im != 0;
    else return v != 0;                                               // NaN is non-zero
}

// ndarray.astype(T): round to nearest between floats and from integers, truncate a float toward zero into an
// integer (then wrap into a narrower one), `!= 0` into bool, drop the imaginary part into a real type
template <typename T, typename S> __device__ __forceinline__ T cvt(S v)
{
    if constexpr (std::is_same_v<T, S>) return v;
    else if constexpr (std::is_same_v<T, bool>) return nonzero(v);
    else if constexpr (is_cplx<T> && is_cplx<S>) return T{(part_t<T>)v.re, (part_t<T>)v.im};
    else if constexpr (is_cplx<T>) return T{cvt<part_t<T>>(v), part_t<T>(0)};
    else if constexpr (is_cplx<S>) return cvt<T>(v.re);
    else if constexpr (std::is_integral_v<T> && std::is_floating_point_v<S>) return (T)(int64_t)v;
    else return (T)v;
}

template <typename C> __device__ __forceinline__ C load(const void* p, int dtype, int64_t i)
{
    switch (dtype) {
        case HD_BOOL: return cvt<C>(((const uint8_t*)p)[i] != 0);
        case HD_U8: return cvt<C>(((const uint8_t*)p)[i]);
        case HD_I16: return cvt<C>(((const int16_t*)p)[i]);
        case HD_I32: return cvt<C>(((const int32_t*)p)[i]);
        case HD_I64: return cvt<C>(((const int64_t*)p)[i]);
        case HD_F32: return cvt<C>(((const float*)p)[i]);
        case HD_F64: return cvt<C>(((const double*)p)[i]);
        case HD_C64: { const float2 v = ((const float2*)p)[i]; return cvt<C>(cf{v.x, v.y}); }
        default: { const double2 v = ((const double2*)p)[i]; return cvt<C>(cd{v.x, v.y}); }
    }
}

template <typename C> __device__ __forceinline__ void store(void* p, int dtype, int64_t i, C v)
{
    switch (dtype) {
        case HD_BOOL: ((uint8_t*)p)[i] = cvt<bool>(v); break;
        case HD_U8: ((uint8_t*)p)[i] = cvt<uint8_t>(v); break;
        case HD_I16: ((int16_t*)p)[i] = cvt<int16_t>(v); break;
        case HD_I32: ((int32_t*)p)[i] = cvt<int32_t>(v); break;
        case HD_I64: ((int64_t*)p)[i] = cvt<int64_t>(v); break;
        case HD_F32: ((float*)p)[i] = cvt<float>(v); break;
        case HD_F64: ((double*)p)[i] = cvt<double>(v); break;
        case HD_C64: { const cf c = cvt<cf>(v); ((float2*)p)[i] = make_float2(c.re, c.im); break; }
        default: { const cd c = cvt<cd>(v); ((double2*)p)[i] = make_double2(c.re, c.im); break; }
    }
}

// correctly rounded float ops of the part type, so that nothing is contracted or widened
__device__ __forceinline__ float add_rn(float x, float y) { return __fadd_rn(x, y); }
__device__ __forceinline__ double add_rn(double x, double y) { return __dadd_rn(x, y); }
__device__ __forceinline__ float sub_rn(float x, float y) { return __fsub_rn(x, y); }
__device__ __forceinline__ double sub_rn(double x, double y) { return __dsub_rn(x, y); }
__device__ __forceinline__ float mul_rn(float x, float y) { return __fmul_rn(x, y); }
__device__ __forceinline__ double mul_rn(double x, double y) { return __dmul_rn(x, y); }
__device__ __forceinline__ float div_rn(float x, float y) { return __fdiv_rn(x, y); }
__device__ __forceinline__ double div_rn(double x, double y) { return __ddiv_rn(x, y); }
__device__ __forceinline__ float fma_rn(float x, float y, float z) { return __fmaf_rn(x, y, z); }
__device__ __forceinline__ double fma_rn(double x, double y, double z) { return __fma_rn(x, y, z); }
__device__ __forceinline__ float sqrt_rn(float x) { return __fsqrt_rn(x); }
__device__ __forceinline__ double sqrt_rn(double x) { return __dsqrt_rn(x); }

// NumPy's complex loops (pinned against the host's NumPy in tests/test_gpu_elementwise.py):
//   x * y: re = fma(xr, yr, -(xi * yi)), im = fma(xr, yi, xi * yr)
//   |z|:   hi * sqrt(fma(r, r, 1)) with r = lo / hi (hi, lo = the larger and smaller of |re|, |im|);
//          inf if a part is infinite, else NaN if a part is NaN, and 0 when hi is 0
template <typename T> __device__ __forceinline__ T cmul(T x, T y)
{
    return T{fma_rn(x.re, y.re, -mul_rn(x.im, y.im)), fma_rn(x.re, y.im, mul_rn(x.im, y.re))};
}
template <typename T> __device__ __forceinline__ part_t<T> cabs(T z)
{
    using R = part_t<T>;
    const R a = fabs(z.re), b = fabs(z.im);
    if (isinf(a) || isinf(b)) return R(INFINITY);
    if (isnan(a) || isnan(b)) return R(NAN);
    const R hi = fmax(a, b), lo = fmin(a, b);
    if (hi == R(0)) return R(0);
    const R r = div_rn(lo, hi);
    return mul_rn(hi, sqrt_rn(fma_rn(r, r, R(1))));
}
// NumPy's complex ordering: by real part, then by imaginary part; a NaN part makes the real-part test false
template <typename T> __device__ __forceinline__ bool clt(T x, T y)
{
    return (x.re < y.re && x.im == x.im && y.im == y.im) || (x.re == y.re && x.im < y.im);
}

template <typename C> __device__ __forceinline__ C apply(int op, C a, C b)
{
    if constexpr (is_cplx<C>) {
        using R = part_t<C>;
        switch (op) {
            case HD_OP_MUL: return cmul(b, a);
            case HD_OP_ADD: return C{add_rn(b.re, a.re), add_rn(b.im, a.im)};
            case HD_OP_RSUB: return C{sub_rn(b.re, a.re), sub_rn(b.im, a.im)};
            case HD_OP_LT: return cvt<C>(clt(a, b));
            case HD_OP_GT: return cvt<C>(clt(b, a));
            case HD_OP_ABS: return C{cabs(a), R(0)};
            case HD_OP_RINT: return C{rint(a.re), rint(a.im)};
            default: return a;                                        // COPY
        }
    } else if constexpr (std::is_floating_point_v<C>) {
        switch (op) {
            case HD_OP_MUL: return mul_rn(b, a);
            case HD_OP_ADD: return add_rn(b, a);
            case HD_OP_RSUB: return sub_rn(b, a);
            case HD_OP_LT: return a < b;
            case HD_OP_GT: return a > b;
            case HD_OP_ABS: return fabs(a);
            case HD_OP_RINT: return rint(a);                          // half to even
            case HD_OP_TRUNC: return a == a ? trunc(a) : C(0);
            default: return a;
        }
    } else if constexpr (std::is_same_v<C, bool>) {
        switch (op) {
            case HD_OP_MUL: return a && b;
            case HD_OP_ADD: return a || b;
            case HD_OP_LT: return !a && b;
            case HD_OP_GT: return a && !b;
            case HD_OP_XOR: return a != b;
            default: return a;                                        // COPY, ABS, RINT, TRUNC
        }
    } else {
        using W = word_t<C>;
        switch (op) {
            case HD_OP_MUL: return (C)(W)((W)b * (W)a);
            case HD_OP_ADD: return (C)(W)((W)b + (W)a);
            case HD_OP_RSUB: return (C)(W)((W)b - (W)a);
            case HD_OP_LT: return a < b;
            case HD_OP_GT: return a > b;
            case HD_OP_ABS:                                           // the minimum stays the minimum
                if constexpr (std::is_signed_v<C>) return a < 0 ? (C)(W)(W(0) - (W)a) : a;
                else return a;
            case HD_OP_XOR: return a ^ b;
            default: return a;                                        // COPY, RINT, TRUNC
        }
    }
}

template <typename C>
__global__ void __launch_bounds__(256) elementwise_kernel(int op, const void* a, int a_dtype, int64_t a_pitch,
                                                          const void* b, int b_dtype, int64_t b_pitch, C b_scalar,
                                                          void* out, int out_dtype, int64_t out_pitch, int64_t ny,
                                                          int64_t nx)
{
    // `a` may be `out` (in-place TRUNC): each cell is read before it is written, by the same thread
    for (CellIter it(nx); it.y < ny; it.next()) {
        const int64_t y = it.y, x = it.x;
        const C va = load<C>(a, a_dtype, y * a_pitch + x);
        const C vb = b ? load<C>(b, b_dtype, y * b_pitch + x) : b_scalar;
        store(out, out_dtype, y * out_pitch + x, apply(op, va, vb));
    }
}

size_t dtype_size(int dtype) { return dtype == HD_BOOL ? 1 : hd_dtype_size(dtype); }

template <typename C>
int launch(int op, const void* a, int a_dtype, int64_t a_pitch, const void* b, int b_dtype, int64_t b_pitch,
           const void* b_scalar, void* out, int out_dtype, int64_t out_pitch, int64_t ny, int64_t nx, cudaStream_t s)
{
    C scalar{};
    if (b_scalar) {                                                   // read before the call returns
        if constexpr (std::is_same_v<C, bool>) scalar = *(const uint8_t*)b_scalar != 0;
        else memcpy(&scalar, b_scalar, sizeof(C));
    }
    const int64_t total = ny * nx;
    const int blocks = (int)((total + 255) / 256 < (int64_t)hd_num_sms() * 16 ? (total + 255) / 256 : hd_num_sms() * 16);
    hd_prof_begin("elementwise_kernel", s);
    elementwise_kernel<C><<<blocks, 256, 0, s>>>(op, a, a_dtype, a_pitch, b, b_dtype, b_pitch, scalar, out, out_dtype,
                                                 out_pitch, ny, nx);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

}  // namespace

extern "C" int hd_elementwise(int op, const void* a, int a_dtype, int64_t a_pitch, const void* b, int b_dtype,
                              int64_t b_pitch, const void* b_scalar, int compute_dtype, void* out, int out_dtype,
                              int64_t out_pitch, int64_t ny, int64_t nx, void* stream)
{
    if (!a || !out) return HD_ERR_NULL;
    if (op < HD_OP_COPY || op > HD_OP_TRUNC) return HD_ERR_ARG;
    if (!dtype_size(a_dtype) || !dtype_size(out_dtype) || !dtype_size(compute_dtype) || (b && !dtype_size(b_dtype)))
        return HD_ERR_ARG;
    const bool binary = op >= HD_OP_MUL && op <= HD_OP_GT || op == HD_OP_XOR;
    if (binary && !b && !b_scalar) return HD_ERR_NULL;
    if (ny < 0 || nx < 0 || a_pitch < nx || out_pitch < nx || (b && b_pitch < nx)) return HD_ERR_ARG;
    const bool is_float = compute_dtype == HD_F32 || compute_dtype == HD_F64;
    const bool is_cplx = compute_dtype == HD_C64 || compute_dtype == HD_C128;
    if ((op == HD_OP_XOR && (is_float || is_cplx)) || (op == HD_OP_RSUB && compute_dtype == HD_BOOL) ||
        (op == HD_OP_TRUNC && is_cplx))
        return HD_ERR_UNSUPPORTED;                                    // NumPy has no such loop either
    if (ny == 0 || nx == 0) return HD_OK;
    cudaStream_t s = (cudaStream_t)stream;
    switch (compute_dtype) {
#define HD_EW(T, TAG) \
    case TAG: return launch<T>(op, a, a_dtype, a_pitch, b, b_dtype, b_pitch, b_scalar, out, out_dtype, out_pitch, ny, nx, s);
        HD_EW(bool, HD_BOOL)
        HD_EW(uint8_t, HD_U8)
        HD_EW(int16_t, HD_I16)
        HD_EW(int32_t, HD_I32)
        HD_EW(int64_t, HD_I64)
        HD_EW(float, HD_F32)
        HD_EW(double, HD_F64)
        HD_EW(cf, HD_C64)
        HD_EW(cd, HD_C128)
#undef HD_EW
        default: return HD_ERR_ARG;
    }
}

// ---- HydroDEMProcess._prepare_final_terms + the three-term sum (hydro_dem_process.py:60-91, :148) ----------
//   mask   = lagoon_values > 0                         (LagoonsDetection.mask_lagoons, custom_filters.py:659)
//   first  = srtm * (1 - (mask + rivers))
//   third  = hsheds_fixed * rivers
//   out    = (first + lagoon_values) + third           float64 arithmetic, rounded once to the output dtype
namespace {
template <typename SrtmT, typename OutT>
__global__ void __launch_bounds__(256) final_terms_kernel(const SrtmT* __restrict__ srtm, int64_t srtm_pitch,
                                                          const float* __restrict__ lagoons, int64_t lag_pitch,
                                                          const float* __restrict__ hsheds, int64_t hs_pitch,
                                                          const float* __restrict__ rivers, int64_t riv_pitch,
                                                          OutT* __restrict__ out, int64_t out_pitch, int64_t ny, int64_t nx)
{
    // four consecutive cells per thread: 16-byte loads, enough of them in flight to cover the HBM latency
    const int64_t nxq = (nx + 3) / 4;
    for (CellIter it(nxq); it.y < ny; it.next()) {
        const int64_t y = it.y, x = 4 * it.x;
        SrtmT sv[4];
        float lv4[4], hv[4], rv[4] = {0.f, 0.f, 0.f, 0.f};
        gload4(srtm + y * srtm_pitch + x, x, nx, sv);
        gload4(lagoons + y * lag_pitch + x, x, nx, lv4);
        gload4(hsheds + y * hs_pitch + x, x, nx, hv);
        if (rivers) gload4(rivers + y * riv_pitch + x, x, nx, rv);
        OutT res[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double s = (double)sv[j];
            const double lv = (double)lv4[j];
            const double r = rivers ? (double)rv[j] : 0.0;
            const double mask = lv > 0.0 ? 1.0 : 0.0;
            const double first = __dmul_rn(s, 1.0 - (mask + r));
            double acc = __dadd_rn(first, lv);
            if (rivers) acc = __dadd_rn(acc, __dmul_rn((double)hv[j], r));
            else acc = __dadd_rn(acc, 0.0 * (double)hv[j]);
            res[j] = (OutT)acc;
        }
        store4v<OutT>(out, out_pitch, y, x, nx, res);
    }
}
}  // namespace

extern "C" int hd_final_terms(const void* srtm, int srtm_dtype, int64_t srtm_pitch, const void* lagoon_values,
                              int64_t lag_pitch, const void* hsheds_fixed, int64_t hs_pitch, const void* rivers,
                              int64_t riv_pitch, void* out, int out_dtype, int64_t out_pitch, int64_t ny, int64_t nx,
                              void* stream)
{
    if (!srtm || !lagoon_values || !hsheds_fixed || !out) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || srtm_pitch < nx || lag_pitch < nx || hs_pitch < nx || out_pitch < nx || (rivers && riv_pitch < nx))
        return HD_ERR_ARG;
    const int64_t total = ny * ((nx + 3) / 4);
    const int blocks = (int)((total + 255) / 256 < (int64_t)hd_num_sms() * 16 ? (total + 255) / 256 : hd_num_sms() * 16);
    cudaStream_t s = (cudaStream_t)stream;
#define HD_FT(ST, STAG, OT, OTAG)                                                                                      \
    if (srtm_dtype == STAG && out_dtype == OTAG) {                                                                     \
        hd_prof_begin("final_terms_kernel", s);                                                                        \
        final_terms_kernel<ST, OT><<<blocks, 256, 0, s>>>((const ST*)srtm, srtm_pitch, (const float*)lagoon_values,    \
                                                          lag_pitch, (const float*)hsheds_fixed, hs_pitch,             \
                                                          (const float*)rivers, riv_pitch, (OT*)out, out_pitch, ny, nx); \
        HD_LAUNCH_CHECK();                                                                                             \
        hd_count_launch();                                                                                             \
        return HD_OK;                                                                                                  \
    }
    HD_FT(float, HD_F32, float, HD_F32)
    HD_FT(float, HD_F32, double, HD_F64)
    HD_FT(double, HD_F64, double, HD_F64)
#undef HD_FT
    return HD_ERR_UNSUPPORTED;
}

// ---- lossless int16 transport of integer-valued float rasters (host API) -----------------------------------------------
namespace {
__global__ void __launch_bounds__(256) pack_i16_kernel(const float* __restrict__ src, int64_t src_pitch,
                                                       int16_t* __restrict__ dst, int64_t ny, int64_t nx,
                                                       int* __restrict__ inexact)
{
    const int64_t nxq = (nx + 3) / 4;
    bool bad = false;
    for (CellIter it(nxq); it.y < ny; it.next()) {
        const int64_t y = it.y, x = 4 * it.x;
        float v[4];
        gload4(src + y * src_pitch + x, x, nx, v);
        int16_t* q = dst + y * nx + x;                        // dense rows
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (x + j >= nx) break;
            const float r = rintf(v[j]);
            bad |= !(r == v[j] && r >= -32768.f && r <= 32767.f);      // NaN, fractions and out-of-range values
            q[j] = (int16_t)(int)fminf(fmaxf(r, -32768.f), 32767.f);
        }
    }
    if (__syncthreads_or(bad) && threadIdx.x == 0) *inexact = 1;
}
}  // namespace

extern "C" int hd_pack_i16(const void* src, int64_t src_pitch, void* dst_dense, int64_t ny, int64_t nx, int* inexact_flag,
                           void* stream)
{
    if (!src || !dst_dense || !inexact_flag) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || src_pitch < nx) return HD_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    HD_CUDA_OK(cudaMemsetAsync(inexact_flag, 0, sizeof(int), s));
    const int64_t total = ny * ((nx + 3) / 4);
    const int blocks = (int)((total + 255) / 256 < (int64_t)hd_num_sms() * 16 ? (total + 255) / 256 : hd_num_sms() * 16);
    hd_prof_begin("pack_i16_kernel", s);
    pack_i16_kernel<<<blocks, 256, 0, s>>>((const float*)src, src_pitch, (int16_t*)dst_dense, ny, nx, inexact_flag);
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

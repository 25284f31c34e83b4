// hydrodem_b200 runtime: status strings, launch counter, pitched copies, TMA tensor-map encoding.
#include <algorithm>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include <atomic>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

static thread_local int g_last_cuda_error = 0;
static std::atomic<int64_t> g_launches{0};

void hd_set_last_cuda_error(int e) { g_last_cuda_error = e; }

// ---- optional per-launch profiling (bench.py): an event pair around every kernel launch ------------------------
namespace {
struct ProfRecord { const char* name; cudaEvent_t start, stop; };
bool g_prof_on = false;
std::vector<ProfRecord> g_prof;
std::vector<cudaEvent_t> g_event_pool;
thread_local cudaStream_t g_prof_stream = nullptr;
thread_local int g_prof_open = -1;
constexpr size_t PROF_MAX_RECORDS = 200000;

cudaEvent_t prof_event()
{
    if (!g_event_pool.empty()) { cudaEvent_t e = g_event_pool.back(); g_event_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
}  // namespace

void hd_prof_begin(const char* name, cudaStream_t stream)
{
    if (!g_prof_on || g_prof.size() >= PROF_MAX_RECORDS) { g_prof_open = -1; return; }
    ProfRecord r{name, prof_event(), prof_event()};
    cudaEventRecord(r.start, stream);
    g_prof_stream = stream;
    g_prof.push_back(r);
    g_prof_open = (int)g_prof.size() - 1;
}

void hd_count_launch(int n)
{
    g_launches.fetch_add(n, std::memory_order_relaxed);
    if (g_prof_open >= 0) {
        cudaEventRecord(g_prof[g_prof_open].stop, g_prof_stream);
        g_prof_open = -1;
    }
}

size_t hd_dtype_size(int dtype)
{
    switch (dtype) {
        case HD_U8: return 1;
        case HD_F32: return 4;
        case HD_I32: return 4;
        case HD_I16: return 2;
        case HD_F64: return 8;
        case HD_I64: return 8;
        case HD_C64: return 8;
        case HD_C128: return 16;
        default: return 0;
    }
}

int hd_num_sms_total()
{
    static int total = 0;
    if (total == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&total, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || total <= 0) total = 148;
    }
    return total;
}

int hd_num_sms()
{
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        // HD_SM_RESERVE=k: persistent grids are sized for (SMs - k), leaving k SMs to the communication kernels that run
        // beside them in the row-band sharded chain (NCCL send / recv cannot start while every SM is full)
        if (const char* e = getenv("HD_SM_RESERVE")) {
            const int k = atoi(e);
            if (k > 0 && k < sms) sms -= k;
        }
    }
    return sms;
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode()
{
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    });
    return fn;
}

int hd_make_tmap_2d(CUtensorMap* out, const void* base, int dtype, int64_t ny, int64_t nx, int64_t pitch_elems,
                    int box_w, int box_h, bool nan_fill, bool swizzle128)
{
    PFN_encodeTiled enc = get_encode();
    if (!enc) { hd_set_last_cuda_error((int)cudaErrorNotSupported); return HD_ERR_CUDA; }
    CUtensorMapDataType dt;
    switch (dtype) {
        case HD_U8: dt = CU_TENSOR_MAP_DATA_TYPE_UINT8; break;
        case HD_F32: dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT32; break;
        case HD_F64: dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT64; break;
        case HD_I32: dt = CU_TENSOR_MAP_DATA_TYPE_INT32; break;
        case HD_C64: dt = CU_TENSOR_MAP_DATA_TYPE_INT64; break;      // moved as 8-byte words, bits untouched
        default: return HD_ERR_UNSUPPORTED;
    }
    const size_t es = hd_dtype_size(dtype);
    if (((uintptr_t)base & 15) || ((pitch_elems * es) & 15)) return HD_ERR_ALIGN;
    if (box_w > 256 || box_h > 256 || ((box_w * es) & 15)) return HD_ERR_UNSUPPORTED;
    if (swizzle128 && box_w * es > 128) return HD_ERR_UNSUPPORTED;
    if (nan_fill && dtype == HD_C64) return HD_ERR_UNSUPPORTED;
    cuuint64_t dims[2] = {(cuuint64_t)nx, (cuuint64_t)ny};
    cuuint64_t strides[1] = {(cuuint64_t)(pitch_elems * es)};
    cuuint32_t box[2] = {(cuuint32_t)box_w, (cuuint32_t)box_h};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     nan_fill ? CU_TENSOR_MAP_FLOAT_OOB_FILL_NAN_REQUEST_ZERO_FMA : CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { hd_set_last_cuda_error((int)cudaErrorInvalidValue); return HD_ERR_CUDA; }
    return HD_OK;
}

template <class Work>
static void host_parallel(int64_t n, int nthreads, Work work)
{
    nthreads = nthreads < 1 ? 1 : (nthreads > 64 ? 64 : nthreads);
    if (n < (int64_t)1 << 16) nthreads = 1;
    if (nthreads == 1) { work((int64_t)0, n); return; }
    std::vector<std::thread> pool;
    const int64_t chunk = ((n + nthreads - 1) / nthreads + 63) & ~(int64_t)63;
    for (int t = 1; t < nthreads; ++t) {
        const int64_t a = std::min(n, t * chunk), b = std::min(n, (t + 1) * chunk);
        if (a < b) pool.emplace_back(work, a, b);
    }
    work((int64_t)0, std::min(n, chunk));
    for (auto& th : pool) th.join();
}


extern "C" {

int hd_version(void) { return 100; }

const char* hd_status_string(int s)
{
    switch (s) {
        case HD_OK: return "ok";
        case HD_ERR_NULL: return "null pointer argument";
        case HD_ERR_WINDOW_HIGH: return "window size larger than the raster";
        case HD_ERR_WINDOW_EVEN: return "window size is even";
        case HD_ERR_ALIGN: return "pointer or pitch not 16-byte aligned";
        case HD_ERR_CUDA: return "CUDA error";
        case HD_ERR_UNSUPPORTED: return "unsupported parameter combination";
        case HD_ERR_ARG: return "invalid argument";
        case HD_ERR_WORKSPACE: return "workspace too small";
        default: return "unknown status";
    }
}

int hd_last_cuda_error(void) { return g_last_cuda_error; }
const char* hd_last_cuda_error_string(void) { return cudaGetErrorString((cudaError_t)g_last_cuda_error); }

int hd_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int hd_profile_enable(int on)
{
    g_prof_on = on != 0;
    return HD_OK;
}

// Synchronises the device, then writes one line per kernel: "<name> <launches> <total_ms>\n".  Clears the records.
int64_t hd_profile_report(char* buf, int64_t cap)
{
    if (cudaDeviceSynchronize() != cudaSuccess) return -1;
    std::map<std::string, std::pair<int64_t, double>> agg;
    for (auto& r : g_prof) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.start, r.stop) == cudaSuccess) {
            auto& a = agg[r.name];
            a.first += 1;
            a.second += ms;
        }
        g_event_pool.push_back(r.start);
        g_event_pool.push_back(r.stop);
    }
    g_prof.clear();
    std::string out;
    char line[256];
    for (auto& kv : agg) {
        snprintf(line, sizeof line, "%s %lld %.6f\n", kv.first.c_str(), (long long)kv.second.first, kv.second.second);
        out += line;
    }
    if (buf && cap > 0) {
        const size_t n = out.size() < (size_t)cap - 1 ? out.size() : (size_t)cap - 1;
        memcpy(buf, out.data(), n);
        buf[n] = 0;
    }
    return (int64_t)out.size();
}

int64_t hd_launch_count(void) { return g_launches.load(); }
void hd_reset_launch_count(void) { g_launches.store(0); }

int64_t hd_pitch_elems(int64_t nx, int dtype)
{
    const int64_t es = (int64_t)hd_dtype_size(dtype);
    if (es == 0) return -1;
    const int64_t q = 128 / es;  // 128-byte rows: every row starts on a cache line
    return (nx + q - 1) / q * q;
}

int hd_memcpy2d_h2d(void* dst, int64_t dp, const void* src, int64_t sp, int64_t w, int64_t rows, void* stream)
{
    if (!dst || !src) return HD_ERR_NULL;
    if (rows <= 0 || w <= 0) return HD_OK;
    if (rows == 1 || (dp == w && sp == w)) {  // dense on both sides: one linear copy (no 2-D pitch limits)
        HD_CUDA_OK(cudaMemcpyAsync(dst, src, (size_t)(w * rows), cudaMemcpyHostToDevice, (cudaStream_t)stream));
        return HD_OK;
    }
    HD_CUDA_OK(cudaMemcpy2DAsync(dst, (size_t)dp, src, (size_t)sp, (size_t)w, (size_t)rows, cudaMemcpyHostToDevice,
                                 (cudaStream_t)stream));
    return HD_OK;
}
int hd_memcpy2d_d2h(void* dst, int64_t dp, const void* src, int64_t sp, int64_t w, int64_t rows, void* stream)
{
    if (!dst || !src) return HD_ERR_NULL;
    if (rows <= 0 || w <= 0) return HD_OK;
    if (rows == 1 || (dp == w && sp == w)) {  // dense on both sides: one linear copy (no 2-D pitch limits)
        HD_CUDA_OK(cudaMemcpyAsync(dst, src, (size_t)(w * rows), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
        return HD_OK;
    }
    HD_CUDA_OK(cudaMemcpy2DAsync(dst, (size_t)dp, src, (size_t)sp, (size_t)w, (size_t)rows, cudaMemcpyDeviceToHost,
                                 (cudaStream_t)stream));
    return HD_OK;
}
// ---- host-side widening of results that crossed PCIe in a narrower type ----------------------------------------------
// The final DEM and the filled DEM hold integer metres: they travel as int16 (a quarter / half of the float64 /
// float32 bytes; the packing kernel verifies that every value is representable and the caller falls back to float32
// otherwise) and are widened here on nthreads host threads with streaming stores (the destination is written once
// and not read back, so the read-for-ownership of its cache lines is skipped).
int hd_host_widen_f32_f64(double* dst, const float* src, int64_t n, int nthreads)
{
    if (!dst || !src) return HD_ERR_NULL;
    if (n <= 0) return HD_OK;
    host_parallel(n, nthreads, [=](int64_t a, int64_t b) {
        int64_t i = a;
#if defined(__SSE2__)
        for (; i < b && ((uintptr_t)(dst + i) & 15); ++i) dst[i] = (double)src[i];
        for (; i + 4 <= b; i += 4) {
            const __m128 v = _mm_loadu_ps(src + i);
            _mm_stream_pd(dst + i, _mm_cvtps_pd(v));
            _mm_stream_pd(dst + i + 2, _mm_cvtps_pd(_mm_movehl_ps(v, v)));
        }
        _mm_sfence();
#endif
        for (; i < b; ++i) dst[i] = (double)src[i];
    });
    return HD_OK;
}

int hd_host_widen_i16(void* dst, int dst_dtype, const int16_t* src, int64_t n, int nthreads)
{
    if (!dst || !src) return HD_ERR_NULL;
    if (dst_dtype != HD_F32 && dst_dtype != HD_F64) return HD_ERR_UNSUPPORTED;
    if (n <= 0) return HD_OK;
    if (dst_dtype == HD_F32) {
        float* d = (float*)dst;
        host_parallel(n, nthreads, [=](int64_t a, int64_t b) {
            int64_t i = a;
#if defined(__SSE2__)
            for (; i < b && ((uintptr_t)(d + i) & 15); ++i) d[i] = (float)src[i];
            for (; i + 8 <= b; i += 8) {
                const __m128i v = _mm_loadu_si128((const __m128i*)(src + i));
                const __m128i lo = _mm_srai_epi32(_mm_unpacklo_epi16(v, v), 16), hi = _mm_srai_epi32(_mm_unpackhi_epi16(v, v), 16);
                _mm_stream_ps(d + i, _mm_cvtepi32_ps(lo));
                _mm_stream_ps(d + i + 4, _mm_cvtepi32_ps(hi));
            }
            _mm_sfence();
#endif
            for (; i < b; ++i) d[i] = (float)src[i];
        });
    } else {
        double* d = (double*)dst;
        host_parallel(n, nthreads, [=](int64_t a, int64_t b) {
            int64_t i = a;
#if defined(__SSE2__)
            for (; i < b && ((uintptr_t)(d + i) & 15); ++i) d[i] = (double)src[i];
            for (; i + 8 <= b; i += 8) {
                const __m128i v = _mm_loadu_si128((const __m128i*)(src + i));
                const __m128i lo = _mm_srai_epi32(_mm_unpacklo_epi16(v, v), 16), hi = _mm_srai_epi32(_mm_unpackhi_epi16(v, v), 16);
                _mm_stream_pd(d + i, _mm_cvtepi32_pd(lo));
                _mm_stream_pd(d + i + 2, _mm_cvtepi32_pd(_mm_shuffle_epi32(lo, 0xEE)));
                _mm_stream_pd(d + i + 4, _mm_cvtepi32_pd(hi));
                _mm_stream_pd(d + i + 6, _mm_cvtepi32_pd(_mm_shuffle_epi32(hi, 0xEE)));
            }
            _mm_sfence();
#endif
            for (; i < b; ++i) d[i] = (double)src[i];
        });
    }
    return HD_OK;
}

// ---- peer memory (row-band sharded chain: the transposes store straight into the other ranks' buffers) ---------------
// One process per GPU: a rank exports the allocation that holds its exchange buffers (CUDA IPC), the others open it
// once and keep the mapping.  handle64: 64 bytes (cudaIpcMemHandle_t); *offset = byte offset of ptr inside its
// allocation (the opened mapping starts at the allocation's base).
int hd_ipc_export(const void* ptr, void* handle64, int64_t* offset)
{
    if (!ptr || !handle64 || !offset) return HD_ERR_NULL;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t h;
    HD_CUDA_OK(cudaIpcGetMemHandle(&h, const_cast<void*>(ptr)));
    CUdeviceptr base = 0;
    size_t size = 0;
    typedef CUresult (*PFN_range)(CUdeviceptr*, size_t*, CUdeviceptr);
    static PFN_range fn = nullptr;
    if (!fn) {
        void* q = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &q, cudaEnableDefault, &qr) != cudaSuccess || !q) {
            hd_set_last_cuda_error((int)cudaErrorNotSupported);
            return HD_ERR_CUDA;
        }
        fn = (PFN_range)q;
    }
    if (fn(&base, &size, (CUdeviceptr)ptr) != CUDA_SUCCESS) { hd_set_last_cuda_error((int)cudaErrorInvalidValue); return HD_ERR_CUDA; }
    memcpy(handle64, &h, 64);
    *offset = (int64_t)((CUdeviceptr)ptr - base);
    return HD_OK;
}

int hd_ipc_import(const void* handle64, void** base)
{
    if (!handle64 || !base) return HD_ERR_NULL;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    HD_CUDA_OK(cudaIpcOpenMemHandle(base, h, cudaIpcMemLazyEnablePeerAccess));
    return HD_OK;
}

int hd_ipc_close(void* base)
{
    if (!base) return HD_OK;
    HD_CUDA_OK(cudaIpcCloseMemHandle(base));
    return HD_OK;
}

int hd_stream_synchronize(void* stream)
{
    HD_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    return HD_OK;
}

}  // extern "C"

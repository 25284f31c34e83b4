/*
 * hydrodem_b200 -- C ABI of the B200-native HydroDEM raster-conditioning hot path.
 *
 * This is the drop-in boundary.  The reference (CGuerreroCordova/HydroDEM) has no FFI: its hot
 * path is the Python protocol  Filter.apply(ndarray) -> ndarray  (filters/__init__.py:23-39).  The
 * entry points below are what a binding for that protocol calls, one per reference filter class;
 * each declaration cites the reference code it replaces (paths under cguerrero/hydrodem/).
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C, no torch / CUDA types in the signatures; `stream` is a cudaStream_t passed as void*
 *     (NULL = default stream).  All raster pointers are DEVICE pointers.
 *   - rasters are row-major; `*_pitch` is the row stride in ELEMENTS.  Windowed filters stage tiles
 *     with TMA, which needs the base pointer and the row stride in bytes to be multiples of 16
 *     (hd_pitch_elems gives a conforming pitch); otherwise HD_ERR_ALIGN is returned.
 *   - every function returns HD_OK (0) or a negative hd_status; nothing is allocated inside except
 *     where a workspace argument says so.  Kernels are launched asynchronously on `stream`.
 *   - there is no CPU fallback: without a CUDA device every compute call returns HD_ERR_CUDA.
 */
#ifndef HYDRODEM_B200_H
#define HYDRODEM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    HD_OK = 0,
    HD_ERR_NULL = -1,         /* null pointer argument */
    HD_ERR_WINDOW_HIGH = -2,  /* window larger than the raster: WindowSizeHighError, sliding_window.py:152-153 */
    HD_ERR_WINDOW_EVEN = -3,  /* even window: WindowSizeEvenError, sliding_window.py:154-155 */
    HD_ERR_ALIGN = -4,        /* base pointer / pitch not 16-byte aligned (TMA) */
    HD_ERR_CUDA = -5,         /* CUDA runtime error, see hd_last_cuda_error() */
    HD_ERR_UNSUPPORTED = -6,  /* parameter combination not implemented (e.g. window too large for the tile) */
    HD_ERR_ARG = -7,          /* invalid argument value */
    HD_ERR_WORKSPACE = -8     /* workspace too small */
} hd_status;

typedef enum {
    HD_U8 = 0,   /* also numpy bool */
    HD_F32 = 1,
    HD_F64 = 2,
    HD_I64 = 3,
    HD_C64 = 4,  /* interleaved float re, im  */
    HD_C128 = 5, /* interleaved double re, im */
    HD_I32 = 6,
    HD_I16 = 7,  /* SRTM / HydroSHEDS on disk: what gdal ReadAsArray hands the reference (image_srtm.py:125, image_hsheds.py:133) */
    HD_BOOL = 8  /* numpy bool, stored as one byte 0 / 1 like HD_U8; a dtype of hd_elementwise only, where it selects
                  * bool semantics: `!= 0` on conversion, OR / AND for add / multiply */
} hd_dtype;

/* ---- runtime --------------------------------------------------------------------------------- */
int hd_version(void);
const char* hd_status_string(int status);
int hd_last_cuda_error(void);
const char* hd_last_cuda_error_string(void);
int hd_device_count(void);
/* kernels launched by this library since the last reset (bench.py's gpu_launches) */
int64_t hd_launch_count(void);
void hd_reset_launch_count(void);
/* per-kernel timing for bench.py: while enabled, every launch is bracketed by a CUDA event pair on its own
 * stream; hd_profile_report synchronises the device and writes "<kernel> <launches> <total_ms>" lines. */
int hd_profile_enable(int on);
int64_t hd_profile_report(char* buf, int64_t cap);
/* smallest pitch (elements) >= nx that satisfies the alignment rules for `dtype` rasters */
int64_t hd_pitch_elems(int64_t nx, int dtype);
/* pitched host<->device copies (cudaMemcpy2DAsync); pitches and width in BYTES */
int hd_memcpy2d_h2d(void* dst, int64_t dst_pitch_bytes, const void* src, int64_t src_pitch_bytes, int64_t width_bytes,
                    int64_t rows, void* stream);
int hd_memcpy2d_d2h(void* dst, int64_t dst_pitch_bytes, const void* src, int64_t src_pitch_bytes, int64_t width_bytes,
                    int64_t rows, void* stream);
int hd_stream_synchronize(void* stream);
/* Stats._set_values / Stats._totals, stats.py:21-25, :63-86 (SURVEY.md 8(f) rank 4): confusion-matrix counts of a
 * simulated raster (F32 / F64; wet = value > threshold, compared in the raster's type) against a water mask (U8 / I16 /
 * F32), with NumPy's arithmetic per sample type (uint8 differences wrap, 0 * NaN counts as non-zero).
 * counts: DEVICE array of 6 uint64 -- TP, FN, FP, TN, total positives, total negatives; zeroed by the call. */
int hd_confusion_counts(const void* sim, int sim_dtype, int64_t sim_pitch, const void* truth, int truth_dtype,
                        int64_t truth_pitch, int64_t ny, int64_t nx, double threshold, void* counts, void* stream);

/* Narrow PCIe transport of integer-valued rasters (host API; the final DEM of hydro_dem_process.py:149 and the filled
 * DEM hold integer metres).  hd_pack_i16: F32 pitched raster -> dense int16 rows on the device; *inexact_flag (device
 * int) is set to 1 if any value is not an integer in [-32768, 32767] (NaN included) -- the caller then moves float32
 * instead.  hd_host_widen_*: HOST helpers, dst[i] = (T)src[i] on nthreads host threads with streaming stores. */
int hd_pack_i16(const void* src, int64_t src_pitch, void* dst_dense, int64_t ny, int64_t nx, int* inexact_flag, void* stream);
int hd_host_widen_f32_f64(double* dst, const float* src, int64_t n, int nthreads);
int hd_host_widen_i16(void* dst, int dst_dtype, const int16_t* src, int64_t n, int nthreads);
/* HOST helper of the GeoTIFF reader (hydrodem_b200/geotiff.py): TIFF 6.0 LZW (MSB-first codes, 9..12 bits, early change).
 * Returns the number of bytes written to dst (at most cap) or a negative hd_status for a corrupt stream. */
int64_t hd_host_lzw_decode(const uint8_t* src, int64_t nsrc, uint8_t* dst, int64_t cap);
/* HOST entries of the GPU block decoder's core (csrc/tiffcodec.cuh), for tests: hd_host_inflate decodes a zlib stream
 * (RFC 1950 header without preset dictionary, RFC 1951 blocks, Adler-32 verified, bytes after the stream ignored);
 * hd_host_tiff_lzw decodes TIFF LZW exactly as hd_host_lzw_decode.  Both return the number of bytes written to dst or a
 * negative hd_status: HD_ERR_ARG for a corrupt stream, and for hd_host_inflate HD_ERR_WORKSPACE when the stream decodes to
 * more than cap bytes. */
int64_t hd_host_inflate(const uint8_t* src, int64_t nsrc, uint8_t* dst, int64_t cap);
int64_t hd_host_tiff_lzw(const uint8_t* src, int64_t nsrc, uint8_t* dst, int64_t cap);

/* ---- elementwise filters (filters/simple_filters.py, extension_filters.py:12-130) -------------- */
typedef enum {
    HD_OP_COPY = 0, /* out = a          -- dtype conversion (ndarray.astype)                                   */
    HD_OP_MUL = 1,  /* out = b * a      ProductFilter.apply      simple_filters.py:165-180                 */
    HD_OP_ADD = 2,  /* out = b + a      AdditionFilter.apply     simple_filters.py:214-229                 */
    HD_OP_RSUB = 3, /* out = b - a      SubtractionFilter.apply  simple_filters.py:261-275 (b = minuend)   */
    HD_OP_LT = 4,   /* out = a < b      LowerThan.apply          simple_filters.py:35-50                   */
    HD_OP_GT = 5,   /* out = a > b      GreaterThan.apply        simple_filters.py:81-96                   */
    HD_OP_ABS = 6,  /* out = |a|        AbsoluteValues.apply     extension_filters.py:78-95 (C64 -> F32)   */
    HD_OP_RINT = 7, /* out = around(a)  Around.apply             extension_filters.py:113-130 (half-even)  */
    HD_OP_XOR = 8,  /* out = b ^ a      BitwiseXOR.apply         extension_filters.py:43-60                */
    HD_OP_TRUNC = 9 /* out = trunc(a), NaN -> 0: what NumPy's assignment of a float into an integer array does
                     * (CorrectNANValues on the int16 HydroSHEDS raster, custom_filters.py:316) */
} hd_elementwise_op;
/* Each op runs in `compute_dtype`, the dtype of NumPy's ufunc loop: `a` and `b` are converted to it as
 * ndarray.astype converts (round to nearest; a float truncated toward zero into an integer, then wrapped; `!= 0`
 * into HD_BOOL; the imaginary part dropped into a real dtype), the op is evaluated in it with NumPy's semantics
 * (integers wrap, float32 is not widened, complex multiply, |z| and ordering use NumPy's formulas, around rounds
 * both parts of a complex), and the result is converted the same way to `out_dtype`.  Comparisons give 0 / 1.
 * `b` may be NULL: then `b_scalar`, a host pointer to one value of compute_dtype (HD_BOOL: one byte), is the second
 * operand; it is read before the call returns.  `a` may be `out`.  XOR on float or complex, RSUB on HD_BOOL and
 * TRUNC on complex return HD_ERR_UNSUPPORTED, as NumPy has no such loop. */
int hd_elementwise(int op, const void* a, int a_dtype, int64_t a_pitch, const void* b, int b_dtype, int64_t b_pitch,
                   const void* b_scalar, int compute_dtype, void* out, int out_dtype, int64_t out_pitch, int64_t ny,
                   int64_t nx, void* stream);

/* HydroDEMProcess._prepare_final_terms and the three-term sum, hydro_dem_process.py:60-91, :148, fused:
 * out = srtm * (1 - ((lagoon_values > 0) + rivers)) + lagoon_values + hsheds_fixed * rivers, in float64
 * arithmetic.  srtm: F32 / F64; lagoon_values, hsheds_fixed, rivers (0/1, may be NULL = no rivers): F32;
 * out: F32 or F64. */
int hd_final_terms(const void* srtm, int srtm_dtype, int64_t srtm_pitch, const void* lagoon_values, int64_t lag_pitch,
                   const void* hsheds_fixed, int64_t hs_pitch, const void* rivers, int64_t riv_pitch, void* out, int out_dtype,
                   int64_t out_pitch, int64_t ny, int64_t nx, void* stream);
/* hd_final_terms (rivers = NULL) + hd_convolve3(ones(3,3), /9, round) in ONE pass: hydro_dem_process.py:60-91, :148-149.
 * All inputs F32; final32 (F32) = the rounded 3x3 mean (integer metres: exact); complete_out (F64, may be NULL) = the sum
 * of the final terms.  16 B/cell of HBM traffic instead of 40; same bits as the two separate calls. */
int hd_final_mean3(const void* srtm, int64_t srtm_pitch, const void* lagoon_values, int64_t lag_pitch,
                   const void* hsheds_fixed, int64_t hs_pitch, void* final32, int64_t final32_pitch, void* complete_out,
                   int64_t complete_pitch, int64_t ny, int64_t nx, void* stream);

/* ---- windowed filters (filters/custom_filters.py) ------------------------------------------------ */
/* ExpandFilter.apply, custom_filters.py:102-125.  in: F32 or U8; out: U8 / F32 / F64, every cell written
 * (1 where any non-NaN cell of the corner-less ws*ws window is > 0, else 0; ws/2 border = 0). */
int hd_expand(const void* in, int in_dtype, int64_t in_pitch, void* out, int out_dtype, int64_t out_pitch, int64_t ny,
              int64_t nx, int ws, void* stream);
/* ExpandFilter(ws) followed by ProductFilter(factor = select): the two middle stages of TidyingLagoons
 * (custom_filters.py:587-610) in one kernel.  in: F32 or U8; select, out: F32; out = select * expanded. */
int hd_expand_select(const void* in, int in_dtype, int64_t in_pitch, const void* select, int64_t sel_pitch, void* out,
                     int64_t out_pitch, int64_t ny, int64_t nx, int ws, void* stream);
/* MajorityFilter.apply, custom_filters.py:48-73.  in: F32; out: F32 / F64, every cell written (mode of the
 * corner-less window if its count >= min_count, else 0; border 0).  min_count = floor((ws*ws-1)*0.7)+1. */
int hd_majority(const void* in, int64_t in_pitch, void* out, int out_dtype, int64_t out_pitch, int64_t ny, int64_t nx,
                int ws, int min_count, void* stream);
/* CorrectNANValues.apply, custom_filters.py:286-317 (window 3).  dtype F32 or F64 (in and out alike),
 * out-of-place Jacobi: out = in except interior cells whose float32 cast is < 0, which get the float32 mean
 * (numpy summation order) of their non-NaN, >= 0 float32 neighbours; no such neighbour -> NaN. */
int hd_nanfix(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
              void* stream);
/* IsolatedPoints.apply, custom_filters.py:345-366 (window 3).  dtype F32 or F64, out-of-place: interior cells
 * with trunc(float32(v)) == 1 become 1 if any of the 8 neighbours is > 0 else 0; other cells are copied. */
int hd_isolated(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
                void* stream);

/* QuadraticFilter.apply, custom_filters.py:226-257 ("isotropic" least-squares quadratic smoother, ws <= 15).
 * dtype F32 or F64 (in and out alike): interior cells = ((s2+s3) r1 - s1 (r2+r3)) / (2 r1^2 - r0 (r2+r3)) over the
 * float32-cast window with the reference's half-pixel offsets; the ws/2 border is copied.  Tolerance class. */
int hd_quadratic(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx, int ws,
                 void* stream);
/* GrovesCorrection.apply, custom_filters.py:704-732, one iteration fused into the quadratic kernel:
 * smooth = Quadratic(dem); hi = dem - smooth; keep = 1 - groves * (hi > threshold); out = keep * hi + smooth.
 * in: F32 or F64; groves: U8 (0/1 class mask); out: F64 (the reference's dtype), or F32 for F32 input. */
int hd_groves_correction(const void* in, int in_dtype, int64_t in_pitch, const void* groves, int64_t groves_pitch, void* out,
                         int out_dtype, int64_t out_pitch, int64_t ny, int64_t nx, int ws, double threshold, void* stream);
/* GrovesCorrectionsIter (custom_filters.py:735-767) without re-copying the cells that cannot change: a cell outside the
 * groves class leaves GrovesCorrection as it entered.  sparse = 0 (first iteration): full pass, tile_flags[t] = "tile t
 * holds a groves cell"; sparse = 1 (later iterations): `out` must already hold the previous iteration's INPUT (ping-pong
 * between two rasters), only flagged tiles are loaded and only quads with a groves cell are stored.  F32 rasters;
 * tile_flags: hd_groves_tile_count(ny, nx) bytes.  Same bits as dense iterations. */
int64_t hd_groves_tile_count(int64_t ny, int64_t nx);
int hd_groves_correction_tiles(const void* in, int64_t in_pitch, const void* groves, int64_t groves_pitch, void* out,
                               int64_t out_pitch, int64_t ny, int64_t nx, int ws, double threshold, void* tile_flags,
                               int sparse, void* stream);

/* NEW stage (not in the reference, SURVEY.md 8a N1): median filter.  F32 -> F32; interior cells =
 * np.nanmedian of the float32 ws*ws window (ws 3 or 5; corner-less if `circular`), ws/2 border copied. */
int hd_median(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int64_t ny, int64_t nx, int ws, int circular,
              void* stream);

/* RouteRivers.apply, custom_filters.py:165-199 (window_size = 3 as used by ProcessRivers, :796): the order-dependent raster
 * scan, run as an order-preserving wavefront (one warp per row, pipelined on per-row progress counters).  mask: F32 (visits
 * where int(v) == 1); g: F32 working copy of the reference DEM, consumed cells are overwritten with 10000 IN PLACE like
 * dem_sliding.grid (:198); out: U8 (zeroed here), 1 = routed river.  workspace: ny ints. */
int hd_route_rivers(const void* mask, int64_t mask_pitch, void* g, int64_t g_pitch, void* out, int64_t out_pitch, int64_t ny,
                    int64_t nx, int ws, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- Fourier stripe removal (filters/custom_filters.py:369-462, :834-1101) ------------------------ */
/* BlanksFourier.apply, custom_filters.py:395-427 (ws = 55, inner = 5 as hard-coded there, :417-419, :457).
 * in: F32 spectrum quarter.  mask_out (U8 or F32, `mask_dtype`) = mask_prev (U8, may be NULL) + (centre > factor *
 * hollow mean); modified (F32, may be NULL) = in * (1 - hit).  The window is clipped to the raster; the centre 5x5
 * block is excluded. */
int hd_hollow_mean_detect(const void* in, int64_t in_pitch, const void* mask_prev, int64_t prev_pitch, void* mask_out,
                          int mask_dtype, int64_t mask_pitch, void* modified, int64_t mod_pitch, int64_t ny, int64_t nx,
                          int ws, int inner, double factor, void* stream);
/* The same with per-tile bookkeeping for DetectBlanksFourier's two passes (custom_filters.py:441-462): the second pass runs
 * on image * (1 - first mask), so it can only find new hits within 27 cells of an old one.  flags_out (pass 1): one byte per
 * 64 x 64 tile, "a hit in this tile"; flags_in (pass 2; modified must be NULL): only tiles whose 3 x 3 tile neighbourhood
 * was flagged are processed, everywhere else mask_out = mask_prev.  hd_hollow_tile_count(ny, nx) bytes per array. */
int64_t hd_hollow_tile_count(int64_t ny, int64_t nx);
int hd_hollow_mean_detect_tiles(const void* in, int64_t in_pitch, const void* mask_prev, int64_t prev_pitch, void* mask_out,
                                int mask_dtype, int64_t mask_pitch, void* modified, int64_t mod_pitch, int64_t ny, int64_t nx,
                                int ws, int inner, double factor, void* flags_out, const void* flags_in, void* stream);
/* FourierProcessQuarters._fill_complete_quarters / _getting_reversed_masks / _fill_complete_mask,
 * custom_filters.py:968-1050.  q1, q2: U8 masks of the two upper quarters, each (ny/2 - margin, nx/2 - margin);
 * out (U8 / F32 / F64, ny x nx) = assembled point-symmetric mask, or 1 - mask when `invert`. */
int hd_fourier_mask_assemble(const void* q1, int64_t q1_pitch, const void* q2, int64_t q2_pitch, void* out, int out_dtype,
                             int64_t out_pitch, int64_t ny, int64_t nx, int margin, int invert, void* stream);
/* FFT plans hold the twiddle / chirp tables of one (ny, nx) shape in device memory (allocated here).  Row
 * lengths up to 8192 (any factorisation: Bluestein in shared memory) or 16384 (powers of two) are one transform;
 * longer rows are split once as n = n1 * n2 with n1 <= 16, n2 <= 8192 (36000 = 5 * 7200, 10801 = 7 * 1543);
 * a length with no such factor (a prime above 8192) -> HD_ERR_UNSUPPORTED. */
int hd_fft2_plan_create(int64_t ny, int64_t nx, void** plan);
int hd_fft2_plan_destroy(void* plan);
/* Read-only description of the transform a plan runs along one axis (axis 0: rows of length nx, 1: columns of length
 * ny).  info[6] = n_total, n1 (cluster size of a long row, 1 = one transform), n (inner length, n_total = n1 * n),
 * m (shared-memory transform length), algorithm (0 radix-2^k, 1 Bluestein, 2 mixed radix), k of the last radix-2^k
 * pass (0 when there is none).  No plan or no info -> HD_ERR_NULL; an axis other than 0 or 1 -> HD_ERR_ARG. */
int hd_fft_plan_info(const void* plan, int axis, int64_t* info);
int64_t hd_fft2_workspace_bytes(int64_t ny, int64_t nx);
/* FourierInitial.apply, custom_filters.py:859-877: fft2 (complex64) -> fftshift -> abs.  in: F32 (ny x nx);
 * fshift: C64 out (may be NULL); fabs_out: F32 |F| in shifted layout. */
int hd_fft2_forward_shift_abs(void* plan, const void* in, int64_t in_pitch, void* fshift, int64_t fshift_pitch, void* fabs_out,
                              int64_t fabs_pitch, void* workspace, int64_t workspace_bytes, void* stream);
/* DetectApplyFourier tail, custom_filters.py:1097-1100: (1 - mask) * F_shift -> ifftshift -> ifft2 -> abs.
 * fshift: C64; mask: U8 (1 = blanked); out: F32 or F64.  Computed in complex64 (tolerance class). */
int hd_fft2_masked_inverse_abs(void* plan, const void* fshift, int64_t fshift_pitch, const void* mask, int64_t mask_pitch,
                               void* out, int out_dtype, int64_t out_pitch, void* workspace, int64_t workspace_bytes,
                               void* stream);
/* FourierTransform / FourierITransform.apply, extension_filters.py:363-379, :398-414 (scipy.fftpack.fft2 /
 * ifft2).  in: F32 or C64; out: C64 (may alias nothing). */
int hd_fft2_c2c(void* plan, const void* in, int in_dtype, int64_t in_pitch, void* out, int64_t out_pitch, int inverse,
                void* workspace, int64_t workspace_bytes, void* stream);
/* FourierShift / FourierIShift.apply, extension_filters.py:432-447, :465-480.  Any 4 / 8 / 16-byte dtype. */
/* Batched 1-D c2c transforms along the rows of an (nrows x nx) array, nx = the plan's row length (in: F32 or C64,
 * out: C64; transpose_out: out is (nx x nrows)).  Building block of the row-band distributed fft2
 * (extension_filters.py:363-480 on a mosaic sharded over several GPUs): local row transforms, all-to-all, local column
 * transforms.  Workspace: hd_fft2_workspace_bytes(nrows, nx). */
int hd_fft_rows(void* plan, const void* in, int in_dtype, int64_t in_pitch, void* out, int64_t out_pitch, int64_t nrows,
                int inverse, int transpose_out, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- row-band sharded Fourier stage (DetectApplyFourier, custom_filters.py:1053-1101, on a mosaic cut into row bands
 * over several GPUs: hydrodem_b200/sharding.py).  Every pass below runs EXACTLY the row transforms of the single-GPU
 * entry points above on a rank's local rows, so the sharded stage reproduces the single-GPU result bit for bit; the
 * transposes between the passes become all-to-all exchanges.
 * hd_fft_band_pass: batched 1-D transforms along the rows of a local (nrows x n) block (axis 0: n = plan nx, axis 1:
 * n = plan ny), then the local transpose into out_t (kept_cols x nrows, natural frequency order).  load: 0 real rows
 * (two per transform), 1 complex, 2 (1 - mask) * column-shifted spectrum (mask U8), 3 Hermitian row pairs.  real_out:
 * the pass stores |z| (load 1) or |re| / |im| (load 3) as F32.  keep_cols > 0: only the first keep_cols frequencies
 * are written (half spectrum of real rows).  Workspace: hd_fft_band_workspace_bytes(nrows, n) (nrows rows of n complex64
 * with 16-byte-aligned rows). */
int64_t hd_fft_band_workspace_bytes(int64_t nrows, int64_t n);
int hd_fft_band_pass(void* plan, int axis, int load, const void* in, int64_t in_pitch, int64_t nrows, const void* mask,
                     int64_t mask_pitch, int shift_cols, int inverse, int real_out, void* out_t, int64_t out_t_pitch,
                     int64_t keep_cols, void* workspace, int64_t workspace_bytes, void* stream);
/* The same pass with the all-to-all FUSED into the transpose: every element of the transposed result is stored straight
 * into the memory of the rank that owns it (peer pointers from hd_ipc_import), 256-byte row segments per warp over NVLink --
 * no send buffer, no NCCL call, no unpack copy.  Output row `orow` (a frequency / pixel index of the transposed axis) in
 * [row0, row1) of a segment lives at base[(orow - row0 + dst_row0) * pitch + column]; this rank's local row r lands at
 * column col_dst0[q] + (r - col_local0[q]).  The caller synchronises the ranks before (destinations free) and after.
 * Workspace: hd_fft_band_workspace_bytes(nrows, n), as for hd_fft_band_pass. */
#define HD_SCATTER_MAX_SEGS 16
typedef struct { int64_t row0, row1; void* base; int64_t pitch; int64_t dst_row0; } hd_scatter_seg;
typedef struct {
    int32_t nseg, ncolseg;
    hd_scatter_seg seg[HD_SCATTER_MAX_SEGS];
    int64_t col_local0[2], col_dst0[2], col_len[2];
} hd_scatter;
int hd_fft_band_pass_scatter(void* plan, int axis, int load, const void* in, int64_t in_pitch, int64_t nrows, const void* mask,
                             int64_t mask_pitch, int shift_cols, int inverse, int real_out, const hd_scatter* sc,
                             int64_t keep_cols, void* workspace, int64_t workspace_bytes, void* stream);
/* CUDA IPC plumbing for the peer pointers (one process per GPU): export the allocation that holds ptr (handle64: 64 bytes;
 * *offset = ptr's byte offset inside it), open it in another process (the mapping starts at the allocation base), close. */
int hd_ipc_export(const void* ptr, void* handle64, int64_t* offset);
int hd_ipc_import(const void* handle64, void** base);
int hd_ipc_close(void* base);
/* "K layout" of a rank's spectrum rows: ky in [a, b) (b <= ny/2 + 1) followed by their mirrors ny - ky in ascending
 * order -- closed under ky -> -ky, so the conjugate half of a real raster's spectrum is completed locally. */
int64_t hd_klayout_rows(int64_t a, int64_t b, int64_t ny);
int64_t hd_klayout_ky(int64_t a, int64_t b, int64_t ny, int64_t t);
/* half spectrum (rows x (nx/2 + 1), C64, rows in K layout) -> column-shifted full rows: fshift (C64, may be NULL) and
 * fabs (F32) = what FourierInitial leaves (custom_filters.py:859-877), for this rank's rows. */
int hd_hermitian_complete(const void* half, int64_t half_pitch, void* fshift, int64_t fshift_pitch, void* fabs_out,
                          int64_t fabs_pitch, int64_t a, int64_t b, int64_t ny, int64_t nx, void* stream);
/* bt (rows x ny, C64): columns ny/2+1 .. ny-1 = conjugates of columns ny-k (the Hermitian inverse's intermediate). */
int hd_conj_mirror_fill(void* bt, int64_t pitch, int64_t rows, int64_t ny, void* stream);
/* hd_fourier_mask_assemble for the rows of one K layout: q1 / q2 are slabs of the quarter masks starting at quarter row
 * q0 (q_rows rows); out: U8 (out_rows x nx). */
int hd_fourier_mask_assemble_rows(const void* q1, int64_t q1_pitch, const void* q2, int64_t q2_pitch, int64_t q0,
                                  int64_t q_rows, void* out, int64_t out_pitch, int64_t out_rows, int64_t a, int64_t b,
                                  int64_t ny, int64_t nx, int margin, void* stream);
int hd_fftshift2(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
                 int inverse, void* stream);

/* ---- morphology (filters/extension_filters.py, scipy.ndimage) ------------------------------------ */
typedef enum { HD_MORPH_ERODE = 0, HD_MORPH_DILATE = 1, HD_MORPH_CLOSE = 2, HD_MORPH_OPEN = 3 } hd_morph_op;
/* BinaryErosion.apply, extension_filters.py:218-235 (scipy.ndimage.binary_erosion(iterations=n)) and
 * BinaryClosing.apply, :276-293 (binary_closing(structure=None | ones((3,3)))).  in: F32 or U8, non-zero =
 * True (NaN is True); out: U8 0/1.  Structuring element: 3x3 cross (full_structure = 0, scipy default) or
 * 3x3 square; border_value = 0 throughout.  iterations <= 8 (erode/dilate) or <= 4 (close/open). */
int hd_binary_morph(const void* in, int in_dtype, int64_t in_pitch, void* out, int64_t out_pitch, int64_t ny, int64_t nx,
                    int op, int full_structure, int iterations, void* stream);
/* GreyDilation.apply, extension_filters.py:328-345 with size=(s, s), s odd <= 17: flat s*s maximum filter,
 * mode='reflect'.  dtype F32 or F64 (in and out alike).  NaN cells are skipped by the maximum (inputs are NaN-free in the chain). */
int hd_max_filter(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
                  int size, void* stream);
/* TidyingLagoons.apply, custom_filters.py:587-610, as ONE kernel: BinaryErosion(iterations=2) -> ExpandFilter(7) ->
 * x majority image -> GreyDilation(7x7).  majority, out: F32.  Same bits as hd_binary_morph + hd_expand_select +
 * hd_max_filter, 8 B/cell of HBM traffic instead of ~22. */
int hd_tidy_lagoons(const void* majority, int64_t in_pitch, void* out, int64_t out_pitch, int64_t ny, int64_t nx,
                    void* stream);
/* Convolve.apply + Around.apply = PostProcessingFinal, extension_filters.py:166-184, :113-130,
 * custom_filters.py:1124-1125.  3x3 correlation with `weights` (9 doubles, row-major, already reversed for
 * a convolution), mode='reflect', double accumulator in row-major order (scipy NI_Correlate), result cast
 * to the raster dtype, divided by `divisor` in that dtype, then rounded half-to-even if do_round.
 * dtype: F32 or F64 (in and out alike).  out32 (may be NULL): an additional F32 copy of the result. */
int hd_convolve3(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
                 const double* weights, double divisor, int do_round, void* out32, int64_t out32_pitch, void* stream);

/* ---- general scipy.ndimage footprints (the drop-in wrappers with any argument the reference accepts) ---------------- */
/* Convolve.apply, extension_filters.py:166-184, with any weights up to 31x31: out = (dtype) sum_t in[y + dy_t][x + dx_t] *
 * w_t / (dtype) divisor, mode='reflect' at any distance (the extension repeats with period 2n, so rasters smaller than the
 * weights work).  The taps (HOST arrays) are NI_Correlate's footprint: the flipped weights with scipy's origin shift on
 * even axes, entries with |w| <= DBL_EPSILON left out, in row-major order, which is the order of the double sum (from
 * +0.0, multiply then add, each rounded).  ntaps <= 961 (0: every cell 0), |dy|, |dx| <= 15, else HD_ERR_UNSUPPORTED.
 * dtype: F32 or F64 (in and out alike). */
int hd_correlate(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
                 int ntaps, const int* tap_dy, const int* tap_dx, const double* tap_w, double divisor, void* stream);
/* BinaryErosion / BinaryClosing.apply, extension_filters.py:218-235, :276-293, with any structure up to 31x31:
 * `iterations` erosions (dilate = 0: AND over the taps) or dilations (dilate = 1: OR) with border_value = 0.  The taps
 * (HOST arrays) are the structure's True cells as offsets from the output cell: as given for scipy.ndimage.binary_erosion,
 * reflected with the origin shift of even axes for binary_dilation.  ntaps = 0 gives all True (erosion) / all False
 * (dilation), as scipy does.  iterations x |dy| and iterations x |dx| <= 15, else HD_ERR_UNSUPPORTED.  in: F32 or U8,
 * non-zero = True (NaN is True); out: U8 0/1.  changed (DEVICE int, may be NULL): set to 1 if out differs from the input
 * anywhere, else 0 -- "until stable" reads it once per launch of several iterations. */
int hd_binary_morph_struct(const void* in, int in_dtype, int64_t in_pitch, void* out, int64_t out_pitch, int64_t ny,
                           int64_t nx, int dilate, int ntaps, const int* tap_dy, const int* tap_dx, int iterations,
                           int* changed, void* stream);
/* GreyDilation.apply, extension_filters.py:328-345, with size=(size_y, size_x), each 1 ... 255 (even sizes with scipy's
 * origin shift: the window of output i is [i - size/2 + 1, i + size/2]), mode='reflect' at any distance.  Two separable
 * passes with a van Herk / Gil-Werman running maximum (three maxima per cell for any size); NaN cells are skipped.
 * dtype: F32 or F64 (in and out alike).  workspace: DEVICE, at least ny * nx elements of dtype. */
int hd_max_filter_rect(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
                       int size_y, int size_x, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- NEW hydrology stages (not in the reference, SURVEY.md 8a N2 / N3) ----------------------------------- */
/* Sink-fill: Planchon-Darboux fixed point with eps = 0, 8-connectivity; frame cells and NaN cells are outlets.
 * z, w: F32.  Persistent worklist kernels with a multigrid start (coarse DEMs of 8x8 block maxima are filled first:
 * their fill is an upper bound of the answer and replaces +inf as the starting surface; the result is the same unique
 * fixed point); asynchronous and capturable in a CUDA graph unless visits_out is given (then the stream is
 * synchronised once and *visits_out = tile visits of the finest level). */
int64_t hd_pdfill_workspace_bytes(int64_t ny, int64_t nx);
int hd_pdfill(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, int64_t ny, int64_t nx, void* workspace,
              int64_t workspace_bytes, int* visits_out, void* stream);
/* Next round of the row-band fill of one band of a sharded mosaic (hydrodem_b200/sharding.py), after a halo exchange:
 * the raster passed in is [halo row | band | halo row] and W holds the previous round's result (the first round is
 * hd_pdfill_band_start); only the tile rows next to the halo rows are re-seeded.  flags: 2 / 4 = the top / bottom row
 * is a neighbour's halo row, not raster frame; any other bit is HD_ERR_ARG.  Nodata cells stay at -inf until
 * hd_pdfill_finish_d8 restores NaN.  *visits_out (may be NULL) = tile visits, synchronises once. */
int hd_pdfill_band(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, int64_t ny, int64_t nx, void* workspace,
                   int64_t workspace_bytes, int flags, int* visits_out, void* stream);
/* Fill + D8 fused: the fill, then ONE pass that restores NaN at the nodata cells and writes the D8 codes (W is not
 * re-read by a separate D8 launch).  Asynchronous and capturable; *visits_out (may be NULL) synchronises once. */
int hd_pdfill_d8(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, void* d8, int64_t d8_pitch, int64_t ny,
                 int64_t nx, void* workspace, int64_t workspace_bytes, int* visits_out, void* stream);
/* The fused last pass alone (row-band fill: after the last round), on the raster the fill ran on: z tells a nodata
 * cell (NaN) from a cell of height -inf, both -inf in W.  workspace: the fill's (status word), may be NULL. */
int hd_pdfill_finish_d8(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, void* d8, int64_t d8_pitch, int64_t ny,
                        int64_t nx, const void* workspace, void* stream);
/* Sticky status of the last fill run with this workspace (0 = fixed point reached; 1 worklist stalled, 2 in-tile
 * iteration cap, 4 work left).  The finish passes also poison W[0][0] = NaN when it is non-zero.  Synchronises. */
int hd_pdfill_status(const void* workspace, int* status_out, void* stream);
/* Row-band fill after a halo exchange: w_halo = min(w_halo, received); *lowered (device int) = 1 if a cell went down. */
int hd_halo_min_flag(void* w_halo, const void* received, int64_t nx, int* lowered, void* stream);
/* Row-band fill with a GLOBAL multigrid start (hydrodem_b200/sharding.py): every rank pools its band to 8x8 block maxima
 * (hd_fill_pool_band; the band's first row is a multiple of 8 in mosaic coordinates; flags 2 / 4 = top / bottom edge is an
 * interior cut; tile_flags_scratch: >= ceil(nyc/64) * ceil(nxc/64) ints), the coarse rows are all-gathered, each rank fills
 * the whole coarse mosaic (hd_pdfill_coarse: W carries the outlet marks on entry; workspace
 * hd_pdfill_workspace_bytes(nyc, nxc)) and starts its band from that upper bound (hd_pdfill_band_start: y_origin = mosaic
 * row of the extended band's row 0).  Same fixed point as hd_pdfill, far fewer exchange rounds. */
int hd_fill_pool_band(const void* z, int64_t z_pitch, int64_t ny, int64_t nx, void* zc, void* wc, int64_t c_pitch, int flags,
                      void* tile_flags_scratch, void* stream);
int hd_pdfill_coarse(const void* zc, void* wc, int64_t c_pitch, int64_t nyc, int64_t nxc, void* workspace,
                     int64_t workspace_bytes, void* stream);
int hd_pdfill_band_start(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, int64_t ny, int64_t nx, void* workspace,
                         int64_t workspace_bytes, int flags, const void* wc_global, int64_t c_pitch, int64_t y_origin,
                         void* stream);
/* D8 flow direction on a (filled) F32 surface -> U8 ESRI codes (E=1, SE=2, S=4, SW=8, W=16, NW=32, N=64, NE=128);
 * steepest positive drop, diagonals scaled by 0.70710678f, ties -> first in that order, frame / NaN / flat -> 0. */
int hd_d8(const void* w, int64_t w_pitch, void* out, int64_t out_pitch, int64_t ny, int64_t nx, void* stream);

/* ---- reprojection onto the EPSG:22184 grid: utils_dem.resample_and_cut, utils_dem.py:65-84 (gdal.Warp) ------------ */
typedef enum { HD_WARP_NEAREST = 0, HD_WARP_BILINEAR = 1 } hd_warp_resample;
/* Fill the F32 destination raster dst (dst_ny x dst_nx, rows dst_row0 ... of the grid dst_geo describes) from src
 * (U8 / I16 / F32).  Grids: HOST double[4] (x0, dx, y0, dy) of the top-left pixel corner, north up, dx, dy > 0.
 * Per destination cell: centre (x0 + (i + 1/2) dx, y0 - (dst_row0 + j + 1/2) dy); if tm (HOST double[7] a, f, lat0,
 * lon0, k0, FE, FN; degrees and metres) is not NULL, inverse Transverse Mercator (Krueger series to n^6, float64) to
 * (lon, lat) degrees; NULL: the source is in the destination CRS.  Source pixel coordinates u = (lon - sx0) / sdx,
 * v = (sy0 - lat) / sdy.  Nearest: the cell (floor u, floor v).  Bilinear: taps floor(u - 1/2), floor(v - 1/2) and their
 * +1 neighbours; taps outside the source or equal to nodata are dropped and the remaining weights renormalised.  A cell
 * with no valid sample gets nodata (has_nodata) or 0.  Allocates nothing; asynchronous and capturable.  Empty grids,
 * pitches below a row, dst_row0 < 0, non-positive pixel sizes, an unknown resampling code or a tm block that describes no
 * ellipsoid -> HD_ERR_ARG. */
int hd_warp(const void* src, int src_dtype, int64_t src_pitch, int64_t src_ny, int64_t src_nx, const double* src_geo,
            int has_nodata, double nodata, void* dst, int64_t dst_pitch, int64_t dst_ny, int64_t dst_nx, const double* dst_geo,
            int64_t dst_row0, const double* tm, int resample, void* stream);
/* hd_warp over a mosaic of sources sampled as one virtual raster (DESIGN §9c).  frame: HOST double[4] (x0, dx, y0, dy) of
 * the first listed source, the virtual raster's corner; u and v are computed from it exactly as in hd_warp.  Virtual pixel
 * (U, V) holds the value of the last listed source that contains it with a value that is not nodata; else it has no
 * sample, which nearest and bilinear treat as hd_warp treats a pixel outside its source.  DEVICE index built on the host:
 * sources = int64[n_sources][6] (device pointer, pitch in elements, U, V, ny, nx: the source's pixel (0, 0) is virtual
 * pixel (U, V)); bins = HOST int64[6] (iu0, iv0, bw, bh, nbu, nbv): a grid of nbu x nbv bins of bw x bh pixels from
 * (iu0, iv0); bin_start = int64[nbu * nbv + 1] and bin_list (int64) are the CSR lists, bin (bu, bv) = bv * nbu + bu, of
 * the sources whose rectangle meets the bin, in descending list order.  Every source has sample type src_dtype (U8 / I16
 * / F32).  Allocates nothing; asynchronous and capturable.  The checks of hd_warp, n_sources < 1, a bin size or count
 * below 1 or a bin grid beyond 2^52 pixels -> HD_ERR_ARG, before any device work. */
int hd_warp_mosaic(const int64_t* sources, int64_t n_sources, const int64_t* bin_start, const int64_t* bin_list,
                   const int64_t* bins, int src_dtype, const double* frame, int has_nodata, double nodata, void* dst,
                   int64_t dst_pitch, int64_t dst_ny, int64_t dst_nx, const double* dst_geo, int64_t dst_row0,
                   const double* tm, int resample, void* stream);
/* HOST: the same inverse Transverse Mercator as hd_warp, on n points (x, y metres -> lon, lat degrees); the host API uses it
 * to check that a destination grid overlaps its source before any device work. */
int hd_host_tm_inverse(const double* tm, const double* x, const double* y, int64_t n, double* lon, double* lat);
/* HOST: the forward Transverse Mercator hd_rasterize_lines applies to geographic vertices, on n points (lon, lat degrees ->
 * x, y metres): the Krueger series to n^6, summed by the same Clenshaw routine as the inverse. */
int hd_host_tm_forward(const double* tm, const double* lon, const double* lat, int64_t n, double* x, double* y);

/* ---- line rasterization onto the EPSG:22184 grid: rasterize_rivers, utils_dem.py:183-191 (gdal.RasterizeLayer) ------ */
/* DEVICE workspace bytes hd_rasterize_lines needs for n_vertices vertices (0 for n_vertices < 0 or above 2^38). */
int64_t hd_rasterize_workspace_bytes(int64_t n_vertices);
/* Burn polylines into the F32 destination dst (dst_ny x dst_nx, rows dst_row0 ... of the grid dst_geo describes; HOST
 * double[4] (x0, dx, y0, dy) as for hd_warp).  DEVICE inputs: vx, vy (double[n_vertices]; lon / lat degrees when tm, a
 * HOST double[7] as for hd_warp, is not NULL, else EPSG:22184 metres), part_start (int64[n_parts + 1], non-decreasing;
 * part p is vertices [part_start[p], part_start[p + 1])), part_feature (int32[n_parts], the feature of each part) and
 * values (float[n_features]).  A vertex has pixel (floor((X - x0) / dx), floor((y0 - Y) / dy)), rows in the full grid's
 * frame; a non-finite vertex, one with |latitude| > 90, or one whose pixel coordinate is 2^29 or more in magnitude burns no
 * segment.  Each segment of a part is walked by GDAL's integer Bresenham (GDALdllImageLine: major axis x when
 * |dx| >= |dy|, max(|dx|, |dy|) + 1 pixels, both ends burned, minor offset after k steps
 * floor((2 k |d_minor| + |d_major| - 1) / (2 |d_major|))); pixels outside dst are dropped.  A cell takes the value of the
 * last feature (largest index) whose walk touches it, 0 when none does.  Allocates nothing, never synchronises, capturable.
 * Workspace: hd_rasterize_workspace_bytes(n_vertices).  Counts < 0, n_vertices > 2^38, n_features > 2^31 - 1, an empty
 * grid, a pitch below a row, dst_row0 < 0, columns or rows at or beyond 2^29, non-positive pixel sizes or a tm block that
 * describes no ellipsoid -> HD_ERR_ARG. */
int hd_rasterize_lines(const void* vx, const void* vy, int64_t n_vertices, const void* part_start, const void* part_feature,
                       int64_t n_parts, const void* values, int64_t n_features, void* dst, int64_t dst_pitch, int64_t dst_ny,
                       int64_t dst_nx, const double* dst_geo, int64_t dst_row0, const double* tm, void* workspace,
                       int64_t workspace_bytes, void* stream);

/* ---- GeoTIFF block decode: geotiff.read_to_device of Deflate / LZW rasters (DESIGN §9d) ------------------------------ */
/* DEVICE workspace bytes hd_tiff_decode needs: one 16-byte aligned slot of block_h * block_w samples per block (0 for
 * invalid arguments, a block above 2 GB or more than 2^40 blocks). */
int64_t hd_tiff_decode_workspace_bytes(int64_t n_blocks, int64_t block_h, int64_t block_w, int sample_dtype);
/* Decode n_blocks compressed strips / tiles of one single-band TIFF into the pitched raster out (ny x nx, sample_dtype
 * U8 / I16 / I32 / I64 / F32 / F64, pitch in elements), as geotiff.read_array decodes them on the host.  DEVICE inputs:
 * src (src_bytes bytes of compressed data) and blocks = int64[n_blocks][5] (offset in src, byte count, y0, x0, rows): the
 * block decodes to rows x block_w samples (rows <= block_h; strips: min(block_h, ny - y0), tiles: block_h) and its
 * top-left sample is cell (y0, x0); what falls outside the raster is cropped.  compression 5 = TIFF LZW (short output is
 * zero-padded, output beyond the block is dropped), 8 / 32946 = zlib Deflate (Adler-32 verified; output shorter than the
 * block is corrupt).  predictor 1, 2 (horizontal, integer samples: a row-wise prefix sum modulo 2^bits after the byte
 * swap) or 3 (floating point, TIFF TN3: byte-wise prefix sum per row, planes most significant first); big_endian: the
 * file's byte order.  status = DEVICE int32[n_blocks], written per block: 0 decoded and stored, 1 corrupt (or a table
 * entry outside src or the raster), 2 a legal Deflate stream longer than the block: not stored, the caller re-decodes it
 * on the host.  One warp per block, persistent; no waiting between warps or CTAs.  Allocates nothing; asynchronous and
 * capturable.  Bad codes, a predictor the sample type does not allow, empty rasters or blocks, pitch < nx -> HD_ERR_ARG;
 * out or its row stride not 16-byte aligned -> HD_ERR_ALIGN; workspace below hd_tiff_decode_workspace_bytes ->
 * HD_ERR_WORKSPACE; all before any device work. */
int hd_tiff_decode(const void* src, int64_t src_bytes, const void* blocks, int64_t n_blocks, int compression, int predictor,
                   int sample_dtype, int big_endian, void* out, int64_t out_pitch, int64_t ny, int64_t nx, int64_t block_h,
                   int64_t block_w, void* status, void* workspace, int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HYDRODEM_B200_H */

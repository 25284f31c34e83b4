// 2-D Fourier stage: hand-written shared-memory FFT (no cuFFT in the product path; tests check it against
// cuFFT / scipy).
//
//   hd_fft2_forward_shift_abs   FourierInitial.apply         custom_filters.py:859-877
//                               (fftpack.fft2 -> fftshift -> abs, extension_filters.py:379, :447, :95)
//   hd_fft2_masked_inverse_abs  DetectApplyFourier tail      custom_filters.py:1097-1100
//                               ((1 - mask) * F_shift -> ifftshift -> ifft2 -> abs)
//   hd_fft2_c2c / hd_fftshift2  FourierTransform / FourierITransform / FourierShift / FourierIShift wrappers
//
// One CTA transforms one row held entirely in shared memory (complex64).  Power-of-two lengths use an
// iterative radix-2 FFT; every other length (3601 = 13 * 277, 519 = 3 * 173 ...) uses Bluestein's chirp-z
// identity  X[k] = w[k] * sum_n (x[n] w[n]) conj(w)[k - n],  w[n] = exp(-i pi n^2 / N),  evaluated as a
// circular convolution of length M = 2^ceil(log2(2N - 1)):  DIF FFT (natural -> bit-reversed), pointwise
// product with the pre-transformed chirp (stored bit-reversed, pre-scaled by 1/M), DIT inverse FFT
// (bit-reversed -> natural).  No bit-reversal pass is ever executed.  Chirp and twiddle tables are computed
// on the host in double precision (n^2 mod 2N in integers) and rounded once to float.
//
// The 2-D transform is rows -> tiled transpose -> rows -> tiled transpose; fftshift / ifftshift, |.|, and
// the (1 - mask) product are folded into the load / store index arithmetic of those passes, so the shifted
// spectrum is never materialised separately.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <complex>
#include <utility>
#include <vector>

#include "common.cuh"
#include "fft_radix.cuh"

namespace {

constexpr int FNT = 256;                 // threads per FFT CTA; two CTAs per SM overlap each other's barriers and global phases
constexpr int MAX_M = 16384;             // 136 KB of (padded) complex64 in shared memory
constexpr double PI = 3.14159265358979323846;

// Rows longer than one shared-memory transform are split once, Cooley-Tukey style: N = n1 * n2 with a SMALL n1
// (3, 5, 7 ... <= 8) and n2 <= 8192.  For each k1 < n1 one CTA of a thread-block cluster transforms the sequence
//     y_k1[j] = W_N^(j k1) * sum_a x[a n2 + j] W_n1^(a k1)          (n1-point DFT + twiddle: long_row_stage, via DSMEM)
// and X[k1 + n1 k2] = FFT_n2(y_k1)[k2].  The result is STORED as [k1][k2] (contiguous writes); the transposes
// that follow every row pass undo this permutation in their index arithmetic, so it costs no extra pass.
struct Plan1D {
    int n_total = 0, n1 = 1;             // n_total = n1 * n   (n = length transformed in shared memory)
    float2* d_wn = nullptr;              // [n1][n]    exp(-2 pi i j k1 / n_total)
    int n = 0, m = 0, log2m = 0;
    bool bluestein = false;
    int npass = 0, k[4] = {0, 0, 0, 0};  // radix-2^k passes (DIF order)
    float2* d_tw = nullptr;              // [m]    exp(-2 pi i k / m), full circle
    float2* d_w = nullptr;               // [n]    chirp exp(-i pi k^2 / n)                  (Bluestein only)
    float2* d_bhat = nullptr;            // [m]    FFT_m(conj chirp) / m, bit-reversed order (Bluestein only)
    // lengths 2^a 3^b 5^c that are not powers of two (6000, 7200: the sub-rows of the 18000 / 36000 mosaics) run as
    // plain mixed-radix transforms: no chirp, no padding to 2^k
    bool mixed = false;
    int nrad = 0, rad[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // DIF pass radices, first pass first
    int padsh = 4;                       // shared-memory index padding: i + (i >> padsh)   (31 = none)
    uint16_t* d_pos = nullptr;           // [n]    position of X[k] after the last DIF pass (digit reversal)
    uint16_t* d_ipos = nullptr;          // [n]    inverse: position p holds X[ipos[p]]
};

struct Plan2D {
    int64_t ny = 0, nx = 0;
    Plan1D px, py;                       // along x (length nx), along y (length ny)
};

// ---- host-side table construction ---------------------------------------------------------------------------
void host_fft(std::vector<std::complex<double>>& a)          // in-place radix-2, natural order in and out
{
    const size_t n = a.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) std::swap(a[i], a[j]);
    }
    for (size_t len = 2; len <= n; len <<= 1) {
        for (size_t i = 0; i < n; i += len)
            for (size_t k = 0; k < len / 2; ++k) {
                const double ang = -2.0 * PI * (double)k / (double)len;
                const std::complex<double> w(std::cos(ang), std::sin(ang));
                const std::complex<double> u = a[i + k], v = a[i + k + len / 2] * w;
                a[i + k] = u + v;
                a[i + k + len / 2] = u - v;
            }
    }
}

unsigned bitrev(unsigned v, int bits)
{
    unsigned r = 0;
    for (int i = 0; i < bits; ++i) r |= ((v >> i) & 1u) << (bits - 1 - i);
    return r;
}

int upload(float2** dst, const std::vector<float2>& src)
{
    HD_CUDA_OK(cudaMalloc((void**)dst, src.size() * sizeof(float2)));
    HD_CUDA_OK(cudaMemcpy(*dst, src.data(), src.size() * sizeof(float2), cudaMemcpyHostToDevice));
    return HD_OK;
}

void destroy1d(Plan1D& p)
{
    cudaFree(p.d_tw); cudaFree(p.d_w); cudaFree(p.d_bhat); cudaFree(p.d_wn); cudaFree(p.d_pos); cudaFree(p.d_ipos);
    p = Plan1D{};
}

constexpr int MAX_N1 = 8;              // = portable thread-block cluster size (one CTA per k1)
constexpr int MAX_INNER = 8192;
constexpr int FNT_HOST = 256;            // = FNT below (threads per FFT CTA)

// ---- mixed-radix planner ------------------------------------------------------------------------------------------
// Radices with a generated in-register butterfly (fft_radix.cuh).  The planner takes the factorisations of n with the
// fewest passes, every order of their radices and a few index paddings, and keeps the one whose shared-memory
// accesses need the fewest wavefronts under the bank model below (64-bit accesses are served per half-warp: 16 lanes,
// conflict-free iff their padded indices differ mod 16); ties go to the smaller SUM of radices (balanced passes: 7200 as
// 5 6 15 16 runs 6 % faster than as 2 15 15 16 -- a radix-2 pass is a full shared-memory round trip for one butterfly).
// Prototype + the same model in NumPy: tools/proto/fft_mixed.py.
constexpr int kRadices[] = {16, 15, 12, 10, 9, 8, 6, 5, 4, 3, 2};
constexpr int MAX_PASSES = 8;

bool smooth235(int64_t n)
{
    for (int p : {2, 3, 5}) while (n % p == 0) n /= p;
    return n == 1;
}

void enum_factorizations(int rem, int start, std::vector<int>& cur, std::vector<std::vector<int>>& out)
{
    if (rem == 1) { out.push_back(cur); return; }
    if ((int)cur.size() >= MAX_PASSES) return;
    for (int i = start; i < (int)(sizeof kRadices / sizeof kRadices[0]); ++i) {
        const int r = kRadices[i];
        if (rem % r == 0) {
            cur.push_back(r);
            enum_factorizations(rem / r, i, cur, out);
            cur.pop_back();
        }
    }
}

double dif_wavefronts(const std::vector<int>& order, int padsh, int n, int nthreads)
{
    double total = 0.0;
    int L = n;
    for (int r : order) {
        const int stride = L / r, ngroups = n / r, lanes = ngroups < nthreads ? ngroups : nthreads;
        long long tot = 0, cnt = 0;
        for (int q = 0; q < r; ++q)
            for (int w0 = 0; w0 < lanes; w0 += 16) {
                int words[16][16], nw[16] = {0};
                for (int l = w0; l < w0 + 16 && l < lanes; ++l) {
                    const int blk = l / stride, j = l - blk * stride;
                    const int a0 = blk * L + j + q * stride, a = a0 + (a0 >> padsh), b = a & 15;
                    bool seen = false;
                    for (int t = 0; t < nw[b]; ++t) seen |= words[b][t] == a;
                    if (!seen) words[b][nw[b]++] = a;
                }
                int worst = 0;
                for (int b = 0; b < 16; ++b) worst = nw[b] > worst ? nw[b] : worst;
                tot += worst; ++cnt;
            }
        total += 2.0 * (double)tot / (double)cnt;
        L = stride;
    }
    return total;
}

// position of X[k] after DIF passes with these radices (first pass first)
int dif_position(int k, const int* rad, int nrad, int L)
{
    int pos = 0;
    for (int s = 0; s < nrad; ++s) {
        const int stride = L / rad[s];
        pos += (k % rad[s]) * stride;
        k /= rad[s];
        L = stride;
    }
    return pos;
}

int plan_mixed(Plan1D& p, int n, int nthreads)
{
    std::vector<std::vector<int>> facs;
    std::vector<int> cur;
    enum_factorizations(n, 0, cur, facs);
    if (facs.empty()) return HD_ERR_UNSUPPORTED;
    size_t fewest = facs[0].size();
    for (auto& f : facs) fewest = f.size() < fewest ? f.size() : fewest;
    std::vector<int> best;
    int best_pad = 31, best_max = 1 << 30;             // best_max: sum of the radices of the best plan (tie-break)
    double best_cost = 1e30;
    if (const char* e = getenv("HD_FFT_RADICES")) {            // experiments: "8,9,10,10[:padsh]"
        std::vector<int> forced;
        int prod = 1, pad_forced = -1;
        for (const char* c = e; *c;) {
            if (*c == ':') { pad_forced = atoi(c + 1); break; }
            const int v = atoi(c);
            if (v > 1) { forced.push_back(v); prod *= v; }
            while (*c && *c != ',' && *c != ':') ++c;
            if (*c == ',') ++c;
        }
        if (prod == n && !forced.empty() && (int)forced.size() <= MAX_PASSES) {
            best = forced;
            best_pad = pad_forced > 0 ? pad_forced : 31;
            if (pad_forced <= 0) {
                for (int pad : {31, 3, 4, 5}) {
                    const double c = dif_wavefronts(forced, pad, n, nthreads);
                    if (c < best_cost) { best_cost = c; best_pad = pad; }
                }
            }
        }
    }
    if (best.empty()) {
        for (auto f : facs) {
            if (f.size() != fewest) continue;
            std::sort(f.begin(), f.end());
            do {
                int mx = 0;
                for (int r : f) mx += r;
                for (int pad : {31, 3, 4, 5}) {
                    const double c = dif_wavefronts(f, pad, n, nthreads);
                    if (c < best_cost - 1e-9 || (c < best_cost + 1e-9 && mx < best_max)) {
                        best_cost = c; best = f; best_pad = pad; best_max = mx;
                    }
                }
            } while (std::next_permutation(f.begin(), f.end()));
        }
    }
    p.mixed = true;
    p.nrad = (int)best.size();
    for (int i = 0; i < p.nrad; ++i) p.rad[i] = best[i];
    p.padsh = best_pad;
    std::vector<uint16_t> pos((size_t)n);
    for (int k = 0; k < n; ++k) pos[k] = (uint16_t)dif_position(k, p.rad, p.nrad, n);
    std::vector<uint16_t> ipos((size_t)n);
    for (int k = 0; k < n; ++k) ipos[pos[k]] = (uint16_t)k;
    HD_CUDA_OK(cudaMalloc((void**)&p.d_pos, pos.size() * sizeof(uint16_t)));
    HD_CUDA_OK(cudaMemcpy(p.d_pos, pos.data(), pos.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    HD_CUDA_OK(cudaMalloc((void**)&p.d_ipos, ipos.size() * sizeof(uint16_t)));
    HD_CUDA_OK(cudaMemcpy(p.d_ipos, ipos.data(), ipos.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    if (getenv("HD_FFT_TRACE")) {
        fprintf(stderr, "fft plan n=%d: mixed radix", n);
        for (int i = 0; i < p.nrad; ++i) fprintf(stderr, " %d", p.rad[i]);
        fprintf(stderr, "  pad i+(i>>%d)  %.2f wavefronts per element pair\n", p.padsh, best_cost);
    }
    return HD_OK;
}

int build1d(Plan1D& p, int64_t n_total)
{
    if (n_total < 1) return HD_ERR_ARG;
    int64_t n = n_total;
    p.n_total = (int)n_total;
    p.n1 = 1;
    const bool total_pow2 = (n_total & (n_total - 1)) == 0;
    if (n_total > MAX_INNER && !(total_pow2 && n_total <= MAX_M)) {
        int n1 = 0;
        for (int f = 2; f <= MAX_N1; ++f)
            if (n_total % f == 0 && n_total / f <= MAX_INNER) { n1 = f; break; }
        if (!n1) return HD_ERR_UNSUPPORTED;          // e.g. a prime length above 8192
        p.n1 = n1;
        n = n_total / n1;
        // wn[k1 * n + j] = W_N^(j k1): contiguous in j for each k1 (coalesced loads in long_row_stage)
        std::vector<float2> wn((size_t)n_total);
        for (int k1 = 0; k1 < n1; ++k1)
            for (int64_t j = 0; j < n; ++j) {
                const double ang = -2.0 * PI * (double)((j * k1) % n_total) / (double)n_total;
                wn[(size_t)k1 * n + j] = make_float2((float)std::cos(ang), (float)std::sin(ang));
            }
        if (int e = upload(&p.d_wn, wn)) return e;
    }
    const bool pow2 = (n & (n - 1)) == 0;
    const bool mixed = !pow2 && smooth235(n) && n <= MAX_INNER && !getenv("HD_FFT_NO_MIXED");
    int64_t m = 1;
    if (pow2 || mixed) m = n;
    else while (m < 2 * n - 1) m <<= 1;
    if (m > MAX_M) return HD_ERR_UNSUPPORTED;       // longer rows need a multi-pass (four-step) FFT: not built yet
    p.n = (int)n; p.m = (int)m; p.bluestein = !pow2 && !mixed;
    if (mixed)
        if (int e = plan_mixed(p, (int)n, FNT_HOST)) return e;
    p.log2m = 0;
    while ((1 << p.log2m) < m) ++p.log2m;
    p.npass = p.log2m ? (p.log2m + 3) / 4 : 0;
    for (int i = 0; i < p.npass; ++i) p.k[i] = p.log2m / p.npass + (i < p.log2m % p.npass ? 1 : 0);
    std::vector<float2> tw(m);
    for (int64_t k = 0; k < m; ++k) {
        const double ang = -2.0 * PI * (double)k / (double)m;
        tw[k] = make_float2((float)std::cos(ang), (float)std::sin(ang));
    }
    if (int e = upload(&p.d_tw, tw)) return e;
    if (p.bluestein) {
        std::vector<std::complex<double>> chirp(n);
        for (int64_t k = 0; k < n; ++k) {
            const int64_t q = (k * k) % (2 * n);                      // exact phase index
            const double ang = -PI * (double)q / (double)n;
            chirp[k] = std::complex<double>(std::cos(ang), std::sin(ang));
        }
        std::vector<std::complex<double>> b(m, std::complex<double>(0, 0));
        b[0] = std::conj(chirp[0]);
        for (int64_t k = 1; k < n; ++k) b[k] = b[m - k] = std::conj(chirp[k]);
        host_fft(b);
        std::vector<float2> w(n), bhat(m);
        for (int64_t k = 0; k < n; ++k) w[k] = make_float2((float)chirp[k].real(), (float)chirp[k].imag());
        for (int64_t i = 0; i < m; ++i) {
            const std::complex<double> v = b[bitrev((unsigned)i, p.log2m)] / (double)m;
            bhat[i] = make_float2((float)v.real(), (float)v.imag());
        }
        if (int e = upload(&p.d_w, w)) return e;
        if (int e = upload(&p.d_bhat, bhat)) return e;
    }
    return HD_OK;
}

// ---- device: complex helpers -----------------------------------------------------------------------------------
__device__ __forceinline__ float2 cmul(float2 a, float2 b)
{
    return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x));
}
__device__ __forceinline__ float2 cmul_conj(float2 a, float2 b)   // a * conj(b)
{
    return make_float2(fmaf(a.x, b.x, a.y * b.y), fmaf(a.y, b.x, -a.x * b.y));
}

// ---- register-blocked radix-2^K passes (prototype + proof of the index algebra: tools/proto/fft_passes.py) ------
// A pass of radix R = 2^K on sub-transforms of length L works on groups {base + r + q * (L/R)}, q = 0..R-1, held
// in registers by one thread:
//   DIF: y = DFT_R(x) by K constant-twiddle radix-2 stages (bit-reversed register order), y[p] *= W_L^(r * rev(p))
//   DIT: x[p] *= W_L^(+-r * rev(p)), then K constant-twiddle radix-2 stages (natural register order)
// so a length-8192 transform is 4 shared-memory round trips (radices 16, 8, 8, 8) instead of 13.
// Shared-memory index padding (one slot per 16) keeps the stride-R accesses of the last passes off the same banks.
__device__ __forceinline__ int pad(int i) { return i + (i >> 4); }

__host__ __device__ constexpr int rev_bits(int v, int bits)
{
    int r = 0;
    for (int i = 0; i < bits; ++i) r |= ((v >> i) & 1) << (bits - 1 - i);
    return r;
}

// d * W_16^E (CONJ: conjugate twiddle), E = 0..7
template <int E, bool CONJ>
__device__ __forceinline__ float2 mul_w16(float2 d)
{
    constexpr float C1 = 0.92387953251128674f, S1 = 0.38268343236508977f, H = 0.70710678118654752f;
    if constexpr (E == 0) return d;
    else if constexpr (E == 4) return CONJ ? make_float2(-d.y, d.x) : make_float2(d.y, -d.x);
    else {
        constexpr float c = (E == 1) ? C1 : (E == 2) ? H : (E == 3) ? S1 : (E == 5) ? -S1 : (E == 6) ? -H : -C1;
        constexpr float sn = (E == 1) ? S1 : (E == 2) ? H : (E == 3) ? C1 : (E == 5) ? C1 : (E == 6) ? H : S1;
        // W = c - i sn  (forward);  conj: c + i sn
        constexpr float si = CONJ ? sn : -sn;
        return make_float2(fmaf(d.x, c, -d.y * si), fmaf(d.x, si, d.y * c));
    }
}

template <int K, int T = 0>
__device__ __forceinline__ void dif_regs(float2 (&x)[1 << K])
{
    if constexpr (T < K) {
        constexpr int R = 1 << K, LT = R >> T, HALF = LT >> 1, STEP = 16 / LT;
#pragma unroll
        for (int blk = 0; blk < R; blk += LT) {
            auto bf = [&](auto jc) {
                constexpr int J = decltype(jc)::value;
                const float2 a = x[blk + J], b = x[blk + J + HALF];
                x[blk + J] = make_float2(a.x + b.x, a.y + b.y);
                x[blk + J + HALF] = mul_w16<J * STEP, false>(make_float2(a.x - b.x, a.y - b.y));
            };
            [&]<int... J>(std::integer_sequence<int, J...>) { (bf(std::integral_constant<int, J>{}), ...); }
            (std::make_integer_sequence<int, HALF>{});
        }
        dif_regs<K, T + 1>(x);
    }
}

template <int K, bool CONJ, int T = 0>
__device__ __forceinline__ void dit_regs(float2 (&x)[1 << K])
{
    if constexpr (T < K) {
        constexpr int R = 1 << K, HALF = 1 << T, LT = 2 * HALF, STEP = 16 / LT;
#pragma unroll
        for (int blk = 0; blk < R; blk += LT) {
            auto bf = [&](auto jc) {
                constexpr int J = decltype(jc)::value;
                const float2 a = x[blk + J];
                const float2 b = mul_w16<J * STEP, CONJ>(x[blk + J + HALF]);
                x[blk + J] = make_float2(a.x + b.x, a.y + b.y);
                x[blk + J + HALF] = make_float2(a.x - b.x, a.y - b.y);
            };
            [&]<int... J>(std::integer_sequence<int, J...>) { (bf(std::integral_constant<int, J>{}), ...); }
            (std::make_integer_sequence<int, HALF>{});
        }
        dit_regs<K, CONJ, T + 1>(x);
    }
}

// W_L^(r * mm), mm = 1 .. R-1: the powers of two are loaded from the table (correctly rounded), the others are products
// of at most three of them -- 4 loads instead of 15 for radix 16; the loads were the kernel's long-scoreboard stalls.
template <int K>
__device__ __forceinline__ void pass_twiddles(float2 (&w)[1 << K], const float2* __restrict__ tw, int r, int tshift)
{
    constexpr int R = 1 << K;
#pragma unroll
    for (int b = 1; b < R; b <<= 1) w[b] = __ldg(&tw[(r * b) << tshift]);
#pragma unroll
    for (int mm = 3; mm < R; ++mm) {
        constexpr int dummy = 0; (void)dummy;
        const int hi = 1 << (31 - __builtin_clz(mm));       // highest set bit (compile-time after unrolling)
        if (mm != hi) w[mm] = cmul(w[hi], w[mm - hi]);
    }
}

// Which group a thread takes.  With a group stride of 8 elements and radix 8 the 32 lanes of a warp touch four
// clusters of 8 consecutive elements, 64 elements (+4 of padding) apart: 8 banks.  The two clusters of a half-warp
// (64-bit accesses are served per half-warp) then overlap in 8 banks -- a 2-way conflict on two of the seven
// shared-memory sweeps.  Swapping lane bits 3 and 4 pairs clusters 0/2 and 1/3, which are 16 banks apart.
__device__ __forceinline__ int lane_group(int g, int lgst, int k)
{
    return (lgst == 3 && k == 3) ? ((g & ~24) | ((g & 8) << 1) | ((g & 16) >> 1)) : g;
}

// One DIF pass over sub-transforms of length L (log2 = lgL); tw = full-circle table exp(-2 pi i k / m).
// MULB: multiply the outputs by bhat[position] on the way out (the Bluestein pointwise product, fused).
template <int K, bool MULB>
__device__ __forceinline__ void dif_pass(float2* s, int m, int lgm, int lgL, const float2* __restrict__ tw,
                                         const float2* __restrict__ bhat)
{
    constexpr int R = 1 << K;
    const int lgst = lgL - K, st = 1 << lgst, tshift = lgm - lgL;
    for (int g0 = threadIdx.x; g0 < (m >> K); g0 += FNT) {
        const int g = lane_group(g0, lgst, K);
        const int r = g & (st - 1);
        const int base = ((g - r) << K) + r;
        float2 x[R];
#pragma unroll
        for (int q = 0; q < R; ++q) x[q] = s[pad(base + (q << lgst))];
        dif_regs<K>(x);
        float2 w[R];
        pass_twiddles<K>(w, tw, r, tshift);
#pragma unroll
        for (int p = 0; p < R; ++p) {
            const int mm = rev_bits(p, K);
            float2 v = x[p];
            if (p > 0) v = cmul(v, w[mm]);
            const int pos = base + (p << lgst);
            if (MULB) v = cmul(v, __ldg(&bhat[pos]));
            s[pad(pos)] = v;
        }
    }
    __syncthreads();
}

// One DIT pass producing sub-transforms of length L; CONJ selects exp(+2 pi i / m).
template <int K, bool CONJ>
__device__ __forceinline__ void dit_pass(float2* s, int m, int lgm, int lgL, const float2* __restrict__ tw)
{
    constexpr int R = 1 << K;
    const int lgst = lgL - K, st = 1 << lgst, tshift = lgm - lgL;
    for (int g0 = threadIdx.x; g0 < (m >> K); g0 += FNT) {
        const int g = lane_group(g0, lgst, K);
        const int r = g & (st - 1);
        const int base = ((g - r) << K) + r;
        float2 x[R], w[R];
        pass_twiddles<K>(w, tw, r, tshift);
#pragma unroll
        for (int p = 0; p < R; ++p) {
            const int mm = rev_bits(p, K);
            float2 v = s[pad(base + (p << lgst))];
            if (p > 0) v = CONJ ? cmul_conj(v, w[mm]) : cmul(v, w[mm]);
            x[p] = v;
        }
        dit_regs<K, CONJ>(x);
#pragma unroll
        for (int q = 0; q < R; ++q) s[pad(base + (q << lgst))] = x[q];
    }
    __syncthreads();
}

struct PassPlan { int npass; int k[4]; };

// Bluestein middle: the last DIF pass and the first inverse DIT pass work on the same 2^K contiguous elements with
// unit twiddles, so they run as one pass in registers: DIF butterflies, x bhat (the pointwise product with the
// transformed chirp), DIT butterflies -- one shared-memory round trip instead of two.
template <int K>
__device__ __forceinline__ void bluestein_mid_pass(float2* s, int m, const float2* __restrict__ bhat)
{
    constexpr int R = 1 << K;
    for (int g = threadIdx.x; g < (m >> K); g += FNT) {
        const int base = g << K;
        float2 x[R], b[R];
#pragma unroll
        for (int q = 0; q < R; ++q) b[q] = __ldg(&bhat[base + q]);
#pragma unroll
        for (int q = 0; q < R; ++q) x[q] = s[pad(base + q)];
        dif_regs<K>(x);
#pragma unroll
        for (int q = 0; q < R; ++q) x[q] = cmul(x[q], b[q]);
        dit_regs<K, true>(x);
#pragma unroll
        for (int q = 0; q < R; ++q) s[pad(base + q)] = x[q];
    }
    __syncthreads();
}

template <bool MULB_LAST>
__device__ __forceinline__ void fft_dif_all(float2* s, int m, int lgm, const PassPlan& pl, const float2* tw, const float2* bhat,
                                            int skip_last = 0)
{
    int lgL = lgm;
    for (int i = 0; i < pl.npass - skip_last; ++i) {
        const bool last = MULB_LAST && i == pl.npass - 1;
        switch (pl.k[i]) {
            case 1: last ? dif_pass<1, true>(s, m, lgm, lgL, tw, bhat) : dif_pass<1, false>(s, m, lgm, lgL, tw, bhat); break;
            case 2: last ? dif_pass<2, true>(s, m, lgm, lgL, tw, bhat) : dif_pass<2, false>(s, m, lgm, lgL, tw, bhat); break;
            case 3: last ? dif_pass<3, true>(s, m, lgm, lgL, tw, bhat) : dif_pass<3, false>(s, m, lgm, lgL, tw, bhat); break;
            default: last ? dif_pass<4, true>(s, m, lgm, lgL, tw, bhat) : dif_pass<4, false>(s, m, lgm, lgL, tw, bhat); break;
        }
        lgL -= pl.k[i];
    }
}

template <bool CONJ>
__device__ __forceinline__ void fft_dit_all(float2* s, int m, int lgm, const PassPlan& pl, const float2* tw, int skip_first = 0)
{
    int lgL = skip_first ? pl.k[pl.npass - 1] : 0;
    for (int i = pl.npass - 1 - skip_first; i >= 0; --i) {
        lgL += pl.k[i];
        switch (pl.k[i]) {
            case 1: dit_pass<1, CONJ>(s, m, lgm, lgL, tw); break;
            case 2: dit_pass<2, CONJ>(s, m, lgm, lgL, tw); break;
            case 3: dit_pass<3, CONJ>(s, m, lgm, lgL, tw); break;
            default: dit_pass<4, CONJ>(s, m, lgm, lgL, tw); break;
        }
    }
}


// ---- mixed-radix DIF passes (lengths 2^a 3^b 5^c) ----------------------------------------------------------------------
// In place, natural order in, digit-reversed order out (Plan1D::d_pos says where X[k] ends up).  A pass of radix R on
// sub-transforms of length L works on groups {base + j + q * (L/R)}, q = 0..R-1, held in registers by one thread:
//   y = DFT_R(x)   (generated straight-line butterflies, fft_radix.cuh),   y[q] *= W_L^(j q),   stored back in place.
struct MixPlan { int nrad; unsigned long long rad8; int padsh; const uint16_t* pos; };   // radices packed 8 bits each

__device__ __forceinline__ int padv(int i, int sh) { return i + (i >> sh); }

// W^(j q) for q = 1 .. R-1 from the table entries q = 1, 2, 4, 8 (correctly rounded) and at most three products
template <int R>
__device__ __forceinline__ void mix_twiddles(float2 (&w)[R], const float2* __restrict__ tw, int jt)
{
#pragma unroll
    for (int b = 1; b < R; b <<= 1) w[b] = __ldg(&tw[jt * b]);
#pragma unroll
    for (int q = 3; q < R; ++q) {
        const int hi = 1 << (31 - __builtin_clz(q));
        if (q != hi) w[q] = cmul(w[hi], w[q - hi]);
    }
}

// Group g = blk * stride + j.  Threads step through the groups FNT at a time, which moves (blk, j) on by the per-pass
// constants (FNT / stride, FNT % stride): no division per group.  The padded slot of element q of a group is
// padv(base, sh) + q * pst whenever that is exact, which holds for every pass of the planner's usual choices:
//   stride a multiple of 2^sh:  (base + q stride) >> sh = (base >> sh) + q (stride >> sh),  pst = padv(stride, sh);
//   stride 1, L a multiple of 2^sh and R <= 2^sh:  base = blk L, and base + q stays inside one padding period,  pst = 1.
// Other passes (pst = 0) pad each index on its own.
template <int R>
__device__ __forceinline__ void mix_dif_pass(float2* s, int n, int L, const float2* __restrict__ tw, int sh)
{
    const int stride = L / R, ngroups = n / R, tstep = n / L;
    const int dblk = FNT / stride, dj = FNT - dblk * stride;
    const int pmask = sh < 31 ? (1 << sh) - 1 : 0;
    const int pst = (stride & pmask) == 0 ? padv(stride, sh)
                  : (stride == 1 && (L & pmask) == 0 && R - 1 <= pmask) ? 1 : 0;
    int blk = (int)threadIdx.x / stride, j = (int)threadIdx.x - blk * stride;
    for (int g = threadIdx.x; g < ngroups; g += FNT) {
        const int base = blk * L + j;
        float2 x[R];
        if (pst) {
            const float2* p = s + padv(base, sh);
#pragma unroll
            for (int q = 0; q < R; ++q) x[q] = p[q * pst];
        } else {
#pragma unroll
            for (int q = 0; q < R; ++q) x[q] = s[padv(base + q * stride, sh)];
        }
        dft_fwd<R>(x);
        if (stride > 1) {
            float2 w[R];
            mix_twiddles<R>(w, tw, j * tstep);
#pragma unroll
            for (int q = 1; q < R; ++q) x[q] = cmul(x[q], w[q]);
        }
        if (pst) {
            float2* p = s + padv(base, sh);
#pragma unroll
            for (int q = 0; q < R; ++q) p[q * pst] = x[q];
        } else {
#pragma unroll
            for (int q = 0; q < R; ++q) s[padv(base + q * stride, sh)] = x[q];
        }
        blk += dblk;
        j += dj;
        if (j >= stride) { j -= stride; ++blk; }
    }
    __syncthreads();
}

__device__ __forceinline__ void fft_mixed_all(float2* s, int n, const MixPlan& mp, const float2* tw)
{
    int L = n;
    for (int i = 0; i < mp.nrad; ++i) {
        const int r = (int)((mp.rad8 >> (8 * i)) & 0xffull);
        switch (r) {
            case 2: mix_dif_pass<2>(s, n, L, tw, mp.padsh); break;
            case 3: mix_dif_pass<3>(s, n, L, tw, mp.padsh); break;
            case 4: mix_dif_pass<4>(s, n, L, tw, mp.padsh); break;
            case 5: mix_dif_pass<5>(s, n, L, tw, mp.padsh); break;
            case 6: mix_dif_pass<6>(s, n, L, tw, mp.padsh); break;
            case 8: mix_dif_pass<8>(s, n, L, tw, mp.padsh); break;
            case 9: mix_dif_pass<9>(s, n, L, tw, mp.padsh); break;
            case 10: mix_dif_pass<10>(s, n, L, tw, mp.padsh); break;
            case 12: mix_dif_pass<12>(s, n, L, tw, mp.padsh); break;
            case 15: mix_dif_pass<15>(s, n, L, tw, mp.padsh); break;
            default: mix_dif_pass<16>(s, n, L, tw, mp.padsh); break;
        }
        L /= r;
    }
}


enum LoadMode { LOAD_REAL = 0, LOAD_C64 = 1, LOAD_MASKED_SHIFTED = 2, LOAD_C64_HPAIR = 3 };
enum Algo { ALG_POW2 = 0, ALG_BLUESTEIN = 1, ALG_MIXED = 2 };

struct RowsArgs {
    const void* in;          // f32 (LOAD_REAL) or float2 rows
    int64_t in_pitch;        // elements
    float2* out;             // complex rows (may alias in for LOAD_C64) -- or float* when store_abs
    int64_t out_pitch;
    const uint8_t* mask;     // LOAD_MASKED_SHIFTED: 1 = blanked frequency, shifted layout
    int64_t mask_pitch;
    int nrows;
    int shift_rows, shift_cols;   // LOAD_MASKED_SHIFTED: source = ((row + shift_rows) % nrows, (col + shift_cols) % n)
    int inverse;             // conj in, conj out, scale 1/n
    int store_abs;           // write |z| as float instead of z
    int rows_total;          // LOAD_MASKED_SHIFTED: modulus of the row shift when only the first nrows rows are transformed
    int n1;                  // outer factor of a long row (1 = the whole row fits one transform)
    int n_total;             // n1 * n
    const float2* wn;        // [n1][n]  W_N^(j k1)
    int permuted;            // mixed radix: leave X in digit-reversed order (position p holds X[ipos[p]]); the transpose
                             // that consumes the rows un-permutes them in its index arithmetic
};

// one element of the (virtual) input row, natural column index `col`
template <int LOAD>
__device__ __forceinline__ float2 load_elem(const RowsArgs& a, int row, int col)
{
    float2 v = make_float2(0.f, 0.f);
    if (LOAD == LOAD_REAL) {
        v.x = reinterpret_cast<const float*>(a.in)[(int64_t)row * a.in_pitch + col];
    } else if (LOAD == LOAD_C64) {
        v = reinterpret_cast<const float2*>(a.in)[(int64_t)row * a.in_pitch + col];
    } else if (LOAD == LOAD_C64_HPAIR) {
        // two Hermitian rows (real inverse transforms) packed as a + i b: the real / imaginary parts of the result
        // are the two real output rows
        const float2* src = reinterpret_cast<const float2*>(a.in) + (int64_t)row * a.in_pitch + col;
        const float2 ra = src[0];
        v = ra;
        if (row + 1 < a.nrows) { const float2 rb = src[a.in_pitch]; v.x = ra.x - rb.y; v.y = ra.y + rb.x; }
    } else {
        int sr = row + a.shift_rows; if (sr >= a.rows_total) sr -= a.rows_total;
        int sc = col + a.shift_cols; if (sc >= a.n_total) sc -= a.n_total;
        v = reinterpret_cast<const float2*>(a.in)[(int64_t)sr * a.in_pitch + sc];
        const float keep = 1.0f - (float)a.mask[(int64_t)sr * a.mask_pitch + sc];   // SubtractionFilter(minuend=1)
        v.x *= keep; v.y *= keep;                                                     // ProductFilter(factor=F_shift)
    }
    if (a.inverse) v.y = -v.y;          // ifft(x) = conj(fft(conj x)) / N
    return v;
}

// ---- long rows: thread-block cluster + distributed shared memory ---------------------------------------------------
// A row longer than one shared-memory transform is split once, N = n1 * n (n1 <= 8 = the portable cluster size), and
// handled by a CLUSTER of n1 CTAs:
//   load      the cluster's threads share the columns j; the thread that owns j loads x[a n + j] for all a from global
//             memory (each element of the row is read exactly once, coalesced), takes the n1-point DFT in registers,
//             applies W_N^(j k1) and stores y_k1[j] into the shared memory of CTA k1 through DSMEM (long_row_load);
//   transform CTA k1 transforms y_k1 (length n) on its own and stores X[k1 + n1 k2] at position k1 * n + k2.
// Two cluster barriers per row: "all y have landed" and "my shared memory is free again" -- the second one is split
// (arrive after the store phase, wait under the next row's first global loads).
// Memory ordering of the two barriers:
//   1. "All y have landed" (cluster_sync_all after the load stage) orders the DSMEM stores of every CTA before the
//      shared-memory reads of the transform in the CTA that owns the memory: a writer-to-reader edge, so it is a
//      release arrive and an acquire wait.
//   2. "My shared memory is free" (cluster_arrive_relaxed after the store phase, waited for in long_row_load) only has
//      to keep the peers' DSMEM stores of the next row from landing before this CTA's reads of the current row.  Every
//      one of those reads has delivered its value into a register that the global store of the same iteration consumed
//      before the __syncthreads() that precedes the arrive, so a later write cannot change what was read; and nothing
//      in the cluster reads the global stores of the store phase (the next kernel does, ordered by the kernel
//      boundary).  A release arrive would add nothing here but a MEMBAR.ALL.GPU that makes every thread wait for its
//      global stores of the row to complete, so this arrive is relaxed.
__device__ __forceinline__ uint32_t cluster_rank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_arrive_relaxed()
{
    asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait()
{
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_sync_all() { cluster_arrive(); cluster_wait(); }
__device__ __forceinline__ uint32_t dsmem_addr(uint32_t local_addr, uint32_t rank)
{
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void dsmem_st(uint32_t addr, float2 v)
{
    asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(v.x), "f"(v.y) : "memory");
}

// Load stage of a long row for this CTA's share of the columns j: x[a n + j] for all a straight from global memory
// (n1 coalesced streams, every element of the row read once by the cluster), n1-point DFT in registers, W_N^(j k1)
// (and the Bluestein chirp), then y_k1[j] is stored into CTA k1's shared memory at slot(j) -- remote stores only, no
// remote loads.  The cluster barrier that says "everybody is done with the previous row's shared memory" is waited for
// after the first batch of global loads has been issued, i.e. under their latency.
// Inlined: the kernel is instantiated per n1 (fft_rows_kernel's N1), so each instantiation holds one case.
template <int N1, int LOAD, int ALG>
__device__ __forceinline__ void long_row_load(float2* s, int n, uint32_t rank, int row, const RowsArgs& a,
                                              const float2* __restrict__ chirp, int padsh)
{
    constexpr bool BLUE = ALG == ALG_BLUESTEIN;
    const float2* __restrict__ wn2 = a.wn;
    auto elem = [&](int r, int c) { return load_elem<LOAD>(a, r, c); };
    auto slot = [&](int k) { return ALG == ALG_MIXED ? padv(k, padsh) : pad(k); };
    const int chunk = (n + N1 - 1) / N1;
    const int j_end = min(n, (int)(rank + 1) * chunk);
    // the shared::cluster address of this CTA's s in CTA k1; slot offsets are added to it (the window of one CTA is
    // contiguous, so mapa(s + o, k1) = mapa(s, k1) + o)
    uint32_t dst[N1];
#pragma unroll
    for (int k1 = 0; k1 < N1; ++k1) dst[k1] = dsmem_addr(smem_u32(s), (uint32_t)k1);
    // software pipelined: the global loads of the next j are issued right after the remote stores of this one
    int j = (int)rank * chunk + (int)threadIdx.x;
    bool live = j < j_end;
    float2 x[N1];
    if (live) {
#pragma unroll
        for (int a = 0; a < N1; ++a) x[a] = elem(row, a * n + j);
    }
    cluster_wait();                                     // the previous row's shared memory is free everywhere
    while (live) {
        dft_fwd<N1>(x);
#pragma unroll
        for (int k1 = 1; k1 < N1; ++k1) x[k1] = cmul(x[k1], __ldg(&wn2[k1 * n + j]));     // W_N^(j k1)
        if (BLUE) {
            const float2 c = __ldg(&chirp[j]);
#pragma unroll
            for (int k1 = 0; k1 < N1; ++k1) x[k1] = cmul(x[k1], c);
        }
        const uint32_t off = (uint32_t)slot(j) * (uint32_t)sizeof(float2);
#pragma unroll
        for (int k1 = 0; k1 < N1; ++k1) dsmem_st(dst[k1] + off, x[k1]);
        j += FNT;
        live = j < j_end;
        if (live) {
#pragma unroll
            for (int a = 0; a < N1; ++a) x[a] = elem(row, a * n + j);
        }
    }
}

// N1 = the row's outer factor a.n1 (1: the whole row is one transform; 2..8: long rows on a cluster of N1 CTAs)
template <int LOAD, int ALG, int N1>
__global__ void __launch_bounds__(FNT, 3) fft_rows_kernel(RowsArgs a, int n, int m, int log2m, PassPlan plan,
                                                       const float2* __restrict__ tw, const float2* __restrict__ chirp,
                                                       const float2* __restrict__ bhat, MixPlan mix)
{
    constexpr bool LONG = N1 > 1;
    constexpr bool BLUE = ALG == ALG_BLUESTEIN;
    constexpr bool MIXED = ALG == ALG_MIXED;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* s = reinterpret_cast<float2*>(smem_raw);
    // Every variant takes its input in natural order (DIF passes) and finds X[k] in a permuted slot afterwards:
    // digit-reversed for the mixed-radix passes, bit-reversed for the radix-2^k ones; Bluestein ends in natural order.
    auto in_slot = [&](int k) -> int { return MIXED ? padv(k, mix.padsh) : pad(k); };
    auto out_slot = [&](int k) -> int {
        if (MIXED) return padv(a.permuted ? k : (int)__ldg(&mix.pos[k]), mix.padsh);
        if (BLUE) return pad(k);
        return pad(log2m ? (int)(__brev((unsigned)k) >> (32 - log2m)) : 0);
    };
    const float scale = a.inverse ? 1.0f / (float)a.n_total : 1.0f;
    const int n1 = N1;
    const uint32_t crank = LONG ? cluster_rank() : 0u;
    const int nworkers = LONG ? (int)gridDim.x / n1 : (int)gridDim.x;          // clusters (LONG) or CTAs
    const int worker = LONG ? (int)blockIdx.x / n1 : (int)blockIdx.x;
    // LOAD_REAL with n1 == 1 packs TWO real rows into one complex transform (x = row_a + i row_b) and separates the
    // two spectra afterwards: A[k] = (X[k] + conj X[n-k]) / 2, B[k] = (X[k] - conj X[n-k]) / 2i.
    const bool pair = (LOAD == LOAD_REAL) && !LONG;
    const bool hpair = (LOAD == LOAD_C64_HPAIR);
    const int nwork = (pair || hpair) ? (a.nrows + 1) / 2 : a.nrows;
    auto elem = [&](int row, int col) -> float2 { return load_elem<LOAD>(a, row, col); };
    if (LONG) cluster_arrive_relaxed();                 // "my shared memory is free" (matched by the wait in long_row_load)
    for (int item = worker; item < nwork; item += nworkers) {
        const int row = (pair || hpair) ? 2 * item : item;
        const int k1 = (int)crank;
        const bool has_b = pair && (row + 1 < a.nrows);
        // ---- load (+ chirp for Bluestein) ------------------------------------------------------------------------
        if constexpr (LONG) {
            if (BLUE)                                   // zero tail of the Bluestein buffer (own shared memory)
                for (int k = n + (int)threadIdx.x; k < m; k += FNT) s[in_slot(k)] = make_float2(0.f, 0.f);
            long_row_load<N1, LOAD, ALG>(s, n, crank, row, a, chirp, mix.padsh);
            cluster_sync_all();                         // every y_k1[j] of this row has landed
        } else {
            // batches of LB elements per thread: all global loads of a batch are issued before the first is used
            constexpr int LB = 8;
            for (int k0 = threadIdx.x; k0 < m; k0 += LB * FNT) {
                float2 v[LB], ch[LB];
#pragma unroll
                for (int j = 0; j < LB; ++j) {
                    const int k = k0 + j * FNT;
                    v[j] = make_float2(0.f, 0.f);
                    ch[j] = make_float2(1.f, 0.f);
                    if (k < n) {
                        if (pair) {
                            const float* src = reinterpret_cast<const float*>(a.in) + (int64_t)row * a.in_pitch + k;
                            v[j].x = src[0];
                            if (has_b) v[j].y = src[a.in_pitch];     // real rows: the inverse conj is applied after the split
                        } else {
                            v[j] = elem(row, k);
                        }
                        if (BLUE) ch[j] = __ldg(&chirp[k]);
                    }
                }
#pragma unroll
                for (int j = 0; j < LB; ++j) {
                    const int k = k0 + j * FNT;
                    if (k >= m) continue;
                    float2 u = v[j];
                    if (BLUE && k < n) u = cmul(u, ch[j]);
                    s[in_slot(k)] = u;
                }
            }
            __syncthreads();
        }
        if (BLUE) {
            // DIF passes, the fused middle (last DIF pass x FFT(conj chirp) / m x first inverse DIT pass), DIT passes
            fft_dif_all<false>(s, m, log2m, plan, tw, bhat, 1);
            switch (plan.k[plan.npass - 1]) {
                case 1: bluestein_mid_pass<1>(s, m, bhat); break;
                case 2: bluestein_mid_pass<2>(s, m, bhat); break;
                case 3: bluestein_mid_pass<3>(s, m, bhat); break;
                default: bluestein_mid_pass<4>(s, m, bhat); break;
            }
            fft_dit_all<true>(s, m, log2m, plan, tw, 1);
        } else if (MIXED) {
            fft_mixed_all(s, n, mix, tw);
        } else if (m > 1) {
            fft_dif_all<false>(s, m, log2m, plan, tw, bhat);
        }
        // ---- store: X[k1 + n1 * k] goes to position k1 * n + k (see Plan1D) ------------------------------------
        const int64_t obase = (int64_t)row * a.out_pitch + (int64_t)k1 * n;
#pragma unroll 4
        for (int k = threadIdx.x; k < n; k += FNT) {                       // unrolled: the chirp loads of four steps overlap
            float2 v = s[out_slot(k)];
            if (BLUE) v = cmul(v, __ldg(&chirp[k]));
            if (pair) {
                const int kn = k ? n - k : 0;
                float2 u = s[out_slot(kn)];
                if (BLUE) u = cmul(u, __ldg(&chirp[kn]));
                float2 fa = make_float2(0.5f * (v.x + u.x), 0.5f * (v.y - u.y));
                float2 fb = make_float2(0.5f * (v.y + u.y), 0.5f * (u.x - v.x));
                if (a.inverse) { fa.y = -fa.y; fb.y = -fb.y; }
                fa.x *= scale; fa.y *= scale; fb.x *= scale; fb.y *= scale;
                if (a.store_abs) {
                    float* dst = reinterpret_cast<float*>(a.out) + obase + k;
                    dst[0] = hypotf(fa.x, fa.y);
                    if (has_b) dst[a.out_pitch] = hypotf(fb.x, fb.y);
                } else {
                    float2* dst = a.out + obase + k;
                    dst[0] = fa;
                    if (has_b) dst[a.out_pitch] = fb;
                }
            } else if (hpair) {
                if (a.inverse) v.y = -v.y;
                float* dst = reinterpret_cast<float*>(a.out) + obase + k;           // store_abs layout (float rows)
                dst[0] = fabsf(v.x * scale);
                if (row + 1 < a.nrows) dst[a.out_pitch] = fabsf(v.y * scale);
            } else {
                if (a.inverse) v.y = -v.y;
                v.x *= scale; v.y *= scale;
                if (a.store_abs) reinterpret_cast<float*>(a.out)[obase + k] = hypotf(v.x, v.y);
                else a.out[obase + k] = v;
            }
        }
        __syncthreads();
        if (LONG) cluster_arrive_relaxed();             // this row is stored: my shared memory is free again
    }
    if (LONG) cluster_wait();                           // closes the last arrive; nobody writes to a CTA that has left
}

// ---- tiled transposes ---------------------------------------------------------------------------------------------
// out[(x + sx) % nx_out_rows ...]: generic "transpose + cyclic shift" of a (rows x cols) array into (cols x rows).
// Element in[r][c] lands at out[(c + shift_c) % cols][(r + shift_r) % rows].
// How the row pass that produced the input stored its columns: position c = k1 * n2 + p holds the frequency index
// k1 + n1 * k2, with k2 = p, or k2 = ipos[p] when the mixed-radix passes left their output digit-reversed.
struct RowPerm { int n1, n2; const uint16_t* ipos; };
__device__ __forceinline__ int unpermute(int c, const RowPerm& pm)
{
    if (pm.n1 == 1 && !pm.ipos) return c;
    const int k1 = c / pm.n2, p = c - k1 * pm.n2;
    const int k2 = pm.ipos ? (int)__ldg(&pm.ipos[p]) : p;
    return k1 + pm.n1 * k2;
}

// One TMA-pipelined kernel serves every transpose of the 2-D transform.  A tile is 64 input rows x 256 bytes of input
// columns (32 complex64 or 64 float), loaded as two 128-byte-wide boxes with the 128-byte swizzle: element (r, c) of a
// box sits at r * 128 + ((16-byte chunk of c) ^ (r & 7)) * 16, so the 16-byte reads of eight consecutive rows in one
// column group hit eight different chunks -- a tile column is read without bank conflicts.  A persistent grid walks
// the tiles through a TR_STAGES-deep ring: the loads of the next TR_STAGES - 1 tiles are in flight while a tile is
// stored.  What depends only on a tile column (un-permuting the row pass's storage order, the keep_max skip, the
// shifted output row, the Hermitian mirror row) is computed once per tile into a shared table, so the store phase
// does no division and no table load per element.  Stores: a warp writes 32 consecutive output columns of one
// output row (256 bytes of complex64).
//   in[r][c] lands at out[(kc + shift_c) % cols][(r + shift_r) % full_rows], kc = unpermute(c); out may be null.
//   WITH_ABS: |in[r][c]| (hypotf) also lands at the same place of out_abs.
//   keep_max >= 0: only input columns whose (unpermuted) index is <= keep_max are written (half spectrum of a real
//                  transform).
//   mirror_rows > 0: the input holds rows 0 .. rows-1 of a Hermitian spectrum whose full height is mirror_rows
//                  (X[mirror_rows - r][cols - c] = conj X[r][c]); the missing rows are written from their mirror.
//                  mirror_cols = 0: the symmetry is X[mirror_rows - r][c] = conj X[r][c] (second axis already real-space).
//                  full_rows = mirror_rows, otherwise rows.
//   OutT != T (float -> double only): the value is widened on the way out.
constexpr int TR_ROWS = 64;              // input rows per tile = output columns per tile
constexpr int TR_SWZ = 128;              // bytes per swizzled box row
constexpr int TR_BOX_BYTES = TR_ROWS * TR_SWZ;
constexpr int TR_STAGE_BYTES = 2 * TR_BOX_BYTES;
constexpr int TR_STAGES = 4;
constexpr int TR_THREADS = 256;
constexpr int TR_SMEM = TR_STAGES * TR_STAGE_BYTES + 1024;     // + alignment slack: the swizzle wants 1024-byte stages

struct TransArgs {
    void* out;               // OutT, may be null (then only out_abs is written)
    int64_t out_pitch;
    float* out_abs;          // WITH_ABS only
    int64_t abs_pitch;
    int rows, cols;          // input extent
    int tile_cols;           // input columns that can hold written values (cols, or keep_max + 1 when nothing is permuted)
    int shift_r, shift_c;
    RowPerm pm;
    int keep_max, mirror_rows, mirror_cols;
};

template <typename T, typename OutT, bool WITH_ABS>
__global__ void __launch_bounds__(TR_THREADS) transpose_tma_kernel(const __grid_constant__ CUtensorMap tm, TransArgs a)
{
    constexpr int ES = (int)sizeof(T);
    constexpr int BOXW = TR_SWZ / ES;            // elements per box row
    constexpr int TC = 2 * BOXW;                 // tile columns
    constexpr int V = 16 / ES;                   // elements per 16-byte shared-memory read
    constexpr int PER_THREAD = TR_ROWS * TC / V / TR_THREADS;
    static_assert(PER_THREAD * TR_THREADS * V == TR_ROWS * TC, "tile / thread mismatch");
    constexpr bool CPLX = sizeof(T) == 8;
    extern __shared__ unsigned char smem_raw[];
    __shared__ uint64_t full[TR_STAGES];
    __shared__ int orow_t[2][TC], mrow_t[2][TC];
    unsigned char* ring = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int tiles_c = (a.tile_cols + TC - 1) / TC;
    const int ntiles = tiles_c * ((a.rows + TR_ROWS - 1) / TR_ROWS);
    const int full_rows = a.mirror_rows > 0 ? a.mirror_rows : a.rows;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < TR_STAGES; ++s) mbar_init(&full[s], 1);
        mbar_fence_init();
        tma_prefetch_desc(&tm);
    }
    __syncthreads();
    auto issue = [&](int tile, int s) {
        const int r0 = (tile / tiles_c) * TR_ROWS, c0 = (tile % tiles_c) * TC;
        unsigned char* dst = ring + s * TR_STAGE_BYTES;
        mbar_arrive_expect_tx(&full[s], TR_STAGE_BYTES);      // out-of-range box cells are zero-filled and counted
        tma_load_2d(dst, &tm, c0, r0, &full[s]);
        tma_load_2d(dst + TR_BOX_BYTES, &tm, c0 + BOXW, r0, &full[s]);
    };
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < TR_STAGES - 1; ++k) {
            const int t = (int)blockIdx.x + k * (int)gridDim.x;
            if (t < ntiles) issue(t, k);
        }
    }
    int k = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++k) {
        const int s = k % TR_STAGES;
        const int r0 = (tile / tiles_c) * TR_ROWS, c0 = (tile % tiles_c) * TC;
        int* orow_tab = orow_t[k & 1];
        int* mrow_tab = mrow_t[k & 1];
        if (threadIdx.x < TC) {                                 // tile-column table (read two tiles ago: free again)
            const int c = c0 + (int)threadIdx.x;
            int orow = -1, mrow = -1;
            if (c < a.cols) {
                const int kc = unpermute(c, a.pm);
                if (a.keep_max < 0 || kc <= a.keep_max) {
                    orow = kc + a.shift_c; if (orow >= a.cols) orow -= a.cols;
                    mrow = (a.mirror_cols ? (kc ? a.cols - kc : 0) : kc) + a.shift_c; if (mrow >= a.cols) mrow -= a.cols;
                }
            }
            orow_tab[threadIdx.x] = orow;
            mrow_tab[threadIdx.x] = mrow;
        }
        __syncthreads();                                        // table visible; every thread is done with tile k - 1
        if (threadIdx.x == 0) {                                 // refill the stage tile k - 1 used
            const int t = tile + (TR_STAGES - 1) * (int)gridDim.x;
            if (t < ntiles) issue(t, (k + TR_STAGES - 1) % TR_STAGES);
        }
        mbar_wait(&full[s], (uint32_t)(k / TR_STAGES) & 1u);
        const unsigned char* st = ring + s * TR_STAGE_BYTES;
#pragma unroll
        for (int j = 0; j < PER_THREAD; ++j) {
            const int u = (int)threadIdx.x + j * TR_THREADS;
            const int r = u & (TR_ROWS - 1), cg = u / TR_ROWS;  // a warp: 32 consecutive rows of one 16-byte column group
            const int gr = r0 + r;
            if (gr >= a.rows) continue;
            const float4 raw = *reinterpret_cast<const float4*>(st + (cg >> 3) * TR_BOX_BYTES + r * TR_SWZ +
                                                                (((cg & 7) ^ (r & 7)) << 4));
            T vals[V];
            memcpy(vals, &raw, sizeof raw);
            int ocol = gr + a.shift_r; if (ocol >= full_rows) ocol -= full_rows;
            const bool mirror = a.mirror_rows > 0 && gr > 0 && 2 * gr != a.mirror_rows;
            int mcol = a.mirror_rows - gr + a.shift_r; if (mcol >= full_rows) mcol -= full_rows;
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const int orow = orow_tab[cg * V + v];
                if (orow < 0) continue;
                const T val = vals[v];
                if (a.out) reinterpret_cast<OutT*>(a.out)[(int64_t)orow * a.out_pitch + ocol] = (OutT)val;
                if constexpr (CPLX) {
                    const float2 z = *reinterpret_cast<const float2*>(&val);
                    float mag = 0.f;
                    if constexpr (WITH_ABS) {
                        mag = hypotf(z.x, z.y);                             // np.abs(complex64) -> float32
                        a.out_abs[(int64_t)orow * a.abs_pitch + ocol] = mag;
                    }
                    if (mirror) {                                           // conjugate partner
                        const int mrow = mrow_tab[cg * V + v];
                        if (a.out)
                            reinterpret_cast<float2*>(a.out)[(int64_t)mrow * a.out_pitch + mcol] = make_float2(z.x, -z.y);
                        if constexpr (WITH_ABS) a.out_abs[(int64_t)mrow * a.abs_pitch + mcol] = mag;
                    }
                }
            }
        }
    }
}

// ---- transpose fused with the all-to-all: remote stores over NVLink --------------------------------------------------------
// The sharded Fourier stage follows every row pass with "transpose, then send row range j of the result to rank j".
// Here the transpose writes each element STRAIGHT INTO THE MEMORY OF THE RANK THAT OWNS IT (peer pointers obtained once
// through CUDA IPC, hd_ipc_*): no send buffer, no NCCL call, no unpack copy -- the exchange is the transpose's own
// stores, 256-byte row segments per warp.  hd_scatter describes where output row `orow` lives (which peer, which row
// there) and at which column this rank's local rows land.
template <typename T>
__global__ void __launch_bounds__(256) transpose_scatter_kernel(const T* __restrict__ in, int64_t in_pitch, int rows, int cols,
                                                                RowPerm pm, int keep_max, hd_scatter sc)
{
    __shared__ T tile[32][33];
    const int tiles_c = (cols + 31) / 32, tiles_r = (rows + 31) / 32;
    const int ntiles = tiles_c * tiles_r;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int r0 = (t / tiles_c) * 32, c0 = (t % tiles_c) * 32;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r = r0 + ty + 8 * k, c = c0 + tx;
            if (r < rows && c < cols) tile[ty + 8 * k][tx] = in[(int64_t)r * in_pitch + c];
        }
        __syncthreads();
        // destination column of local row r (at most two segments: the K layout's lower / mirror rows)
        const int r = r0 + tx;
        int64_t ocol = -1;
#pragma unroll
        for (int q = 0; q < 2; ++q)
            if (q < sc.ncolseg && r >= sc.col_local0[q] && r < sc.col_local0[q] + sc.col_len[q])
                ocol = sc.col_dst0[q] + (r - sc.col_local0[q]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int c = c0 + ty + 8 * k;
            if (r < rows && c < cols && ocol >= 0) {
                const int orow = unpermute(c, pm);
                if (keep_max >= 0 && orow > keep_max) continue;
                for (int q = 0; q < sc.nseg; ++q) {
                    const hd_scatter_seg& sg = sc.seg[q];
                    if (orow >= sg.row0 && orow < sg.row1) {
                        reinterpret_cast<T*>(sg.base)[(orow - sg.row0 + sg.dst_row0) * sg.pitch + ocol] = tile[tx][ty + 8 * k];
                        break;
                    }
                }
            }
        }
        __syncthreads();
    }
}

// cyclic shift without transpose (FourierShift / FourierIShift wrappers): out[(r+sr)%rows][(c+sc)%cols] = in[r][c]
template <typename T>
__global__ void __launch_bounds__(256) shift_kernel(const T* __restrict__ in, int64_t in_pitch, T* __restrict__ out,
                                                    int64_t out_pitch, int rows, int cols, int sr, int sc)
{
    const int64_t total = (int64_t)rows * cols;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(t / cols), c = (int)(t - (int64_t)r * cols);
        int orow = r + sr; if (orow >= rows) orow -= rows;
        int ocol = c + sc; if (ocol >= cols) ocol -= cols;
        out[(int64_t)orow * out_pitch + ocol] = in[(int64_t)r * in_pitch + c];
    }
}


// ---- row-band building blocks (hydrodem_b200/sharding.py) ----------------------------------------------------------------
// "K layout": a rank of the sharded Fourier stage holds the spectrum rows ky in [a, b) (0 <= a < b <= ny/2 + 1) followed
// by their Hermitian mirrors {ny - ky} in ascending order -- a row set closed under ky -> -ky, so the conjugate half of
// the spectrum of a real raster can be completed without talking to another GPU.
struct KLayout {
    int a, b, ny, hlo, nhi;
    __host__ __device__ KLayout(int a_, int b_, int ny_) : a(a_), b(b_), ny(ny_)
    {
        const int kmin = a > 1 ? a : 1, kmax = (b - 1) < (ny - 1) / 2 ? (b - 1) : (ny - 1) / 2;
        nhi = kmax >= kmin ? kmax - kmin + 1 : 0;
        hlo = ny - kmax;
    }
    __host__ __device__ int rows() const { return (b - a) + nhi; }
    __host__ __device__ int ky(int t) const { return t < b - a ? a + t : hlo + (t - (b - a)); }
    __host__ __device__ int local(int k) const { return (k >= a && k < b) ? k - a : (b - a) + (k - hlo); }
};

// half (rows x nh) c64, rows in K layout  ->  fshift / fabs rows (rows x nx) with the COLUMNS fftshift-ed (the rows stay
// in K layout).  Same values as the last transpose of hd_fft2_forward_shift_abs: direct copy for kx <= nx/2, conjugate
// of the mirror row for the rest, |.| by hypotf.
__global__ void __launch_bounds__(256) hermitian_complete_kernel(const float2* __restrict__ half, int64_t half_pitch,
                                                                 float2* __restrict__ fshift, int64_t fs_pitch,
                                                                 float* __restrict__ fabs_out, int64_t fa_pitch, KLayout kl,
                                                                 int nx)
{
    const int nh = nx / 2 + 1, rows = kl.rows(), sx = nx / 2;
    for (CellIter it(nx); it.y < rows; it.next()) {
        const int t = (int)it.y, kx = (int)it.x;
        float2 v;
        if (kx < nh) {
            v = half[(int64_t)t * half_pitch + kx];
        } else {
            const int km = (kl.ny - kl.ky(t)) % kl.ny;
            v = half[(int64_t)kl.local(km) * half_pitch + (nx - kx)];
            v.y = -v.y;
        }
        int oc = kx + sx; if (oc >= nx) oc -= nx;
        if (fshift) fshift[(int64_t)t * fs_pitch + oc] = v;
        fabs_out[(int64_t)t * fa_pitch + oc] = hypotf(v.x, v.y);
    }
}

// bt (rows x ny) c64: bt[x][ny - k] = conj bt[x][k] for 0 < k, 2k != ny (what the Hermitian inverse's transpose writes)
__global__ void __launch_bounds__(256) conj_mirror_kernel(float2* __restrict__ bt, int64_t pitch, int rows, int ny)
{
    const int nlo = ny / 2 + 1, nm = ny - nlo;                  // columns nlo .. ny-1 are mirrors
    if (nm <= 0) return;
    for (CellIter it(nm); it.y < rows; it.next()) {
        const int k = nlo + (int)it.x;
        float2 v = bt[it.y * pitch + (ny - k)];
        v.y = -v.y;
        bt[it.y * pitch + k] = v;
    }
}

// ---- host launch helpers -----------------------------------------------------------------------------------------
// Does a row pass with this plan / load mode leave its output digit-reversed when the consumer allows it?  (Not when
// two real rows share a transform: separating their spectra needs X[k] and X[n-k] side by side.)
bool leaves_permuted(const Plan1D& p, int load) { return p.mixed && !(load == LOAD_REAL && p.n1 == 1); }
RowPerm perm_of(const Plan1D& p, int load, bool allow_permuted = true)
{
    return RowPerm{p.n1, p.n, (allow_permuted && leaves_permuted(p, load)) ? p.d_ipos : nullptr};
}

int launch_rows(const Plan1D& p, const RowsArgs& a_in, int load, cudaStream_t s, bool allow_permuted = true)
{
    RowsArgs a = a_in;
    a.permuted = (allow_permuted && leaves_permuted(p, load)) ? 1 : 0;
    a.n1 = p.n1;
    if (a.rows_total == 0) a.rows_total = a.nrows;
    a.n_total = p.n_total;
    a.wn = p.d_wn;
    const size_t smem = (size_t)(p.m + (p.m >> (p.mixed ? p.padsh : 4)) + 1) * sizeof(float2);
    PassPlan plan{p.npass, {p.k[0], p.k[1], p.k[2], p.k[3]}};
    unsigned long long rad8 = 0;
    for (int i = 0; i < p.nrad; ++i) rad8 |= (unsigned long long)p.rad[i] << (8 * i);
    MixPlan mix{p.nrad, rad8, p.padsh, p.d_pos};
    if (a.nrows < 1) return HD_OK;
#define HD_ROWS_L(LOADV, ALGV, N1V)                                                                     \
    {                                                                                                    \
        auto kern = fft_rows_kernel<LOADV, ALGV, N1V>;                                                   \
        HD_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   \
        const int nwork = ((LOADV == LOAD_REAL && N1V == 1) || LOADV == LOAD_C64_HPAIR) ? (a.nrows + 1) / 2 : a.nrows; \
        cudaLaunchConfig_t cfg = {};                                                                     \
        cfg.blockDim = dim3(FNT);                                                                        \
        cfg.dynamicSmemBytes = smem;                                                                     \
        cfg.stream = s;                                                                                  \
        cudaLaunchAttribute attr[1];                                                                     \
        int workers = 1;                                                                                 \
        if (N1V > 1) {                                                                                   \
            attr[0].id = cudaLaunchAttributeClusterDimension;                                            \
            attr[0].val.clusterDim.x = (unsigned)p.n1;                                                   \
            attr[0].val.clusterDim.y = 1;                                                                \
            attr[0].val.clusterDim.z = 1;                                                                \
            cfg.attrs = attr;                                                                            \
            cfg.numAttrs = 1;                                                                            \
            cfg.gridDim = dim3((unsigned)p.n1);                                                          \
            HD_CUDA_OK(cudaOccupancyMaxActiveClusters(&workers, kern, &cfg));   /* co-resident clusters */ \
            workers = (int)((int64_t)workers * hd_num_sms() / hd_num_sms_total());                       \
        } else {                                                                                         \
            int per_sm = 1;                                                                              \
            HD_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, FNT, smem));          \
            workers = hd_num_sms() * (per_sm < 1 ? 1 : per_sm);                                          \
        }                                                                                                \
        if (workers < 1) workers = 1;                                                                    \
        if (workers > nwork) workers = nwork;                                                            \
        cfg.gridDim = dim3((unsigned)(workers * (N1V > 1 ? p.n1 : 1)));                                    \
        hd_prof_begin("fft_rows_kernel", s);                                                             \
        HD_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, a, p.n, p.m, p.log2m, plan, (const float2*)p.d_tw,     \
                                      (const float2*)p.d_w, (const float2*)p.d_bhat, mix));              \
    }
#define HD_ROWS(LOADV, ALGV)                                        \
    {                                                               \
        switch (p.n1) {                                             \
            case 1: HD_ROWS_L(LOADV, ALGV, 1) break;                \
            case 2: HD_ROWS_L(LOADV, ALGV, 2) break;                \
            case 3: HD_ROWS_L(LOADV, ALGV, 3) break;                \
            case 4: HD_ROWS_L(LOADV, ALGV, 4) break;                \
            case 5: HD_ROWS_L(LOADV, ALGV, 5) break;                \
            case 6: HD_ROWS_L(LOADV, ALGV, 6) break;                \
            case 7: HD_ROWS_L(LOADV, ALGV, 7) break;                \
            default: HD_ROWS_L(LOADV, ALGV, 8) break;               \
        }                                                           \
    }
    if (p.bluestein) {
        if (load == LOAD_REAL) HD_ROWS(LOAD_REAL, ALG_BLUESTEIN)
        else if (load == LOAD_C64) HD_ROWS(LOAD_C64, ALG_BLUESTEIN)
        else if (load == LOAD_C64_HPAIR) HD_ROWS(LOAD_C64_HPAIR, ALG_BLUESTEIN)
        else HD_ROWS(LOAD_MASKED_SHIFTED, ALG_BLUESTEIN)
    } else if (p.mixed) {
        if (load == LOAD_REAL) HD_ROWS(LOAD_REAL, ALG_MIXED)
        else if (load == LOAD_C64) HD_ROWS(LOAD_C64, ALG_MIXED)
        else if (load == LOAD_C64_HPAIR) HD_ROWS(LOAD_C64_HPAIR, ALG_MIXED)
        else HD_ROWS(LOAD_MASKED_SHIFTED, ALG_MIXED)
    } else {
        if (load == LOAD_REAL) HD_ROWS(LOAD_REAL, ALG_POW2)
        else if (load == LOAD_C64) HD_ROWS(LOAD_C64, ALG_POW2)
        else if (load == LOAD_C64_HPAIR) HD_ROWS(LOAD_C64_HPAIR, ALG_POW2)
        else HD_ROWS(LOAD_MASKED_SHIFTED, ALG_POW2)
    }
#undef HD_ROWS_L
#undef HD_ROWS
    HD_LAUNCH_CHECK();
    hd_count_launch();
    return HD_OK;
}

int transpose_grid(int rows, int cols)
{
    const int64_t nt = (int64_t)((rows + 31) / 32) * ((cols + 31) / 32);
    const int64_t cap = (int64_t)hd_num_sms() * 8;
    return (int)(nt < cap ? nt : cap);
}

// Row pitch (elements) of the scratch arrays the transposes read: TMA wants 16-byte-aligned rows.
int64_t pitch_c64(int64_t n) { return (n + 1) & ~(int64_t)1; }
int64_t pitch_f32(int64_t n) { return (n + 3) & ~(int64_t)3; }

// in: (rows x cols) T with a 16-byte-aligned base and pitch (the scratch arrays of this file); name: profiler record
template <typename T, typename OutT, bool WITH_ABS>
int launch_transpose(const T* in, int64_t in_pitch, TransArgs a, cudaStream_t s, const char* name)
{
    constexpr int TC = 2 * TR_SWZ / (int)sizeof(T);
    if (a.rows < 1 || a.cols < 1) return HD_OK;
    // a half-spectrum consumer of rows in natural order only needs the columns up to keep_max
    a.tile_cols = (a.keep_max >= 0 && a.pm.n1 == 1 && !a.pm.ipos) ? std::min(a.cols, a.keep_max + 1) : a.cols;
    CUtensorMap tm;
    if (int e = hd_make_tmap_2d(&tm, in, sizeof(T) == 8 ? HD_C64 : HD_F32, a.rows, a.cols, in_pitch, TR_SWZ / (int)sizeof(T),
                                TR_ROWS, false, true))
        return e;
    auto kern = transpose_tma_kernel<T, OutT, WITH_ABS>;
    HD_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, TR_SMEM));
    int per_sm = 1;
    HD_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, TR_THREADS, TR_SMEM));
    const int64_t ntiles = (int64_t)hd_cdiv(a.tile_cols, TC) * hd_cdiv(a.rows, TR_ROWS);
    const int64_t cap = (int64_t)hd_num_sms() * (per_sm < 1 ? 1 : per_sm);
    hd_prof_begin(name, s);
    kern<<<(unsigned)(ntiles < cap ? ntiles : cap), TR_THREADS, TR_SMEM, s>>>(tm, a);
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

TransArgs trans_args(void* out, int64_t out_pitch, int rows, int cols, RowPerm pm)
{
    TransArgs a{};
    a.out = out; a.out_pitch = out_pitch;
    a.rows = rows; a.cols = cols;
    a.pm = pm;
    a.keep_max = -1; a.mirror_rows = 0; a.mirror_cols = 1;
    return a;
}

// The row pass of hd_fft_band_pass(_scatter): checks the arguments they share, then transforms the nrows local rows
// into the workspace, [nrows][*pitch] of complex64 (float when real_out) with 16-byte-aligned rows.  *pl: the plan of
// the transformed axis.
int band_rows(void* plan, int axis, int load, const void* in, int64_t in_pitch, int64_t nrows, const void* mask,
              int64_t mask_pitch, int shift_cols, int inverse, int real_out, void* workspace, int64_t workspace_bytes,
              cudaStream_t s, const Plan1D** pl, int64_t* pitch)
{
    if (!plan || !in || !workspace) return HD_ERR_NULL;
    Plan2D* p = (Plan2D*)plan;
    *pl = axis == 0 ? &p->px : &p->py;
    const int n = (*pl)->n_total;
    if (nrows < 1 || nrows > 0x7fffffff || axis < 0 || axis > 1 || load < 0 || load > 3) return HD_ERR_ARG;
    if (load == LOAD_MASKED_SHIFTED && !mask) return HD_ERR_NULL;
    if (load == LOAD_C64_HPAIR && !real_out) return HD_ERR_ARG;
    if (workspace_bytes < hd_fft_band_workspace_bytes(nrows, n)) return HD_ERR_WORKSPACE;
    if (in_pitch < n) return HD_ERR_ARG;
    *pitch = real_out ? pitch_f32(n) : pitch_c64(n);
    RowsArgs r{in, in_pitch, (float2*)workspace, *pitch, (const uint8_t*)mask, mask_pitch, (int)nrows, 0, shift_cols,
               inverse ? 1 : 0, real_out ? 1 : 0, (int)nrows};
    return launch_rows(**pl, r, load, s);
}

}  // namespace

extern "C" {

int hd_fft2_plan_create(int64_t ny, int64_t nx, void** plan)
{
    if (!plan) return HD_ERR_NULL;
    *plan = nullptr;
    if (ny < 1 || nx < 1) return HD_ERR_ARG;
    Plan2D* p = new Plan2D();
    p->ny = ny; p->nx = nx;
    int e = build1d(p->px, nx);
    if (!e) e = build1d(p->py, ny);
    if (e) { destroy1d(p->px); destroy1d(p->py); delete p; return e; }
    *plan = p;
    return HD_OK;
}

int hd_fft2_plan_destroy(void* plan)
{
    if (!plan) return HD_OK;
    Plan2D* p = (Plan2D*)plan;
    destroy1d(p->px); destroy1d(p->py);
    delete p;
    return HD_OK;
}

int hd_fft_plan_info(const void* plan, int axis, int64_t* info)
{
    if (!plan || !info) return HD_ERR_NULL;
    if (axis < 0 || axis > 1) return HD_ERR_ARG;
    const Plan2D* p = (const Plan2D*)plan;
    const Plan1D& pl = axis == 0 ? p->px : p->py;
    info[0] = pl.n_total;
    info[1] = pl.n1;
    info[2] = pl.n;
    info[3] = pl.m;
    info[4] = pl.bluestein ? ALG_BLUESTEIN : pl.mixed ? ALG_MIXED : ALG_POW2;
    info[5] = (!pl.mixed && pl.npass > 0) ? pl.k[pl.npass - 1] : 0;
    return HD_OK;
}

// two complex64 scratch arrays of ny x nx, each with room for 16-byte-aligned row pitches in either orientation
int64_t hd_fft2_workspace_bytes(int64_t ny, int64_t nx) { return 2 * pitch_c64(ny) * pitch_c64(nx) * (int64_t)sizeof(float2); }

int64_t hd_fft_band_workspace_bytes(int64_t nrows, int64_t n) { return nrows * pitch_c64(n) * (int64_t)sizeof(float2); }

int hd_fft2_forward_shift_abs(void* plan, const void* in, int64_t in_pitch, void* fshift, int64_t fshift_pitch, void* fabs_out,
                              int64_t fabs_pitch, void* workspace, int64_t workspace_bytes, void* stream)
{
    if (!plan || !in || !fabs_out || !workspace) return HD_ERR_NULL;
    Plan2D* p = (Plan2D*)plan;
    const int ny = (int)p->ny, nx = (int)p->nx;
    if (workspace_bytes < hd_fft2_workspace_bytes(ny, nx)) return HD_ERR_WORKSPACE;
    if (in_pitch < nx || fabs_pitch < nx || (fshift && fshift_pitch < nx)) return HD_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t pnx = pitch_c64(nx), pny = pitch_c64(ny);
    float2* A = (float2*)workspace;                 // [ny][pnx]
    float2* At = A + pny * pnx;                     // [nx][pny]
    // The input is real, so the spectrum is Hermitian: only columns kx = 0 .. nx/2 go through the second (column) pass,
    // the other half is written from its conjugate mirror by the last transpose.
    const int nh = nx / 2 + 1;
    RowsArgs r1{in, in_pitch, A, pnx, nullptr, 0, ny, 0, 0, 0, 0};
    if (int e = launch_rows(p->px, r1, LOAD_REAL, s)) return e;
    TransArgs t1 = trans_args(At, pny, ny, nx, perm_of(p->px, LOAD_REAL));
    t1.keep_max = nh - 1;
    if (int e = launch_transpose<float2, float2, false>(A, pnx, t1, s, "transpose_kernel")) return e;
    RowsArgs r2{At, pny, A, pny, nullptr, 0, nh, 0, 0, 0, 0};            // out of place: long rows read the whole row
    if (int e = launch_rows(p->py, r2, LOAD_C64, s)) return e;
    // A[kx][ky] = F[ky][kx] for kx < nh; transpose back with fftshift folded in:
    // F[ky][kx] -> Fs[(ky + ny/2) % ny][(kx + nx/2) % nx], plus the mirrored half
    TransArgs t2 = trans_args(fshift, fshift_pitch, nh, ny, perm_of(p->py, LOAD_C64));
    t2.out_abs = (float*)fabs_out; t2.abs_pitch = fabs_pitch;
    t2.shift_r = nx / 2; t2.shift_c = ny / 2;
    t2.mirror_rows = nx;
    return launch_transpose<float2, float2, true>(A, pny, t2, s, "transpose_kernel");
}

int hd_fft2_masked_inverse_abs(void* plan, const void* fshift, int64_t fshift_pitch, const void* mask, int64_t mask_pitch,
                               void* out, int out_dtype, int64_t out_pitch, void* workspace, int64_t workspace_bytes,
                               void* stream)
{
    if (!plan || !fshift || !mask || !out || !workspace) return HD_ERR_NULL;
    Plan2D* p = (Plan2D*)plan;
    const int ny = (int)p->ny, nx = (int)p->nx;
    if (workspace_bytes < hd_fft2_workspace_bytes(ny, nx)) return HD_ERR_WORKSPACE;
    if (fshift_pitch < nx || mask_pitch < nx || out_pitch < nx) return HD_ERR_ARG;
    if (out_dtype != HD_F32 && out_dtype != HD_F64) return HD_ERR_UNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t pnx = pitch_c64(nx), pny = pitch_c64(ny), pny_f = pitch_f32(ny);
    float2* A = (float2*)workspace;                 // [ny][pnx]
    float2* At = A + pny * pnx;                     // [nx][pny]
    // ifftshift: unshifted index k reads shifted index (k + n/2) % n
    float* absT = (float*)A;                        // [nx][pny_f] float, reuses A
    if ((ny & 1) && (nx & 1) && !getenv("HD_FFT_NO_HERMITIAN")) {
        // Odd x odd: the assembled mask is exactly point-symmetric about DC (custom_filters.py:1042-1049) and F is
        // the spectrum of a real raster, so (1 - mask) * F is Hermitian and the inverse is real.  Only rows
        // ky = 0 .. ny/2 go through the first pass; the other rows of the intermediate are conjugates
        // (c[ny - ky][x] = conj c[ky][x]) written by the transpose; the second pass packs two real-output columns
        // into one complex transform.  abs() of a real number: |re| (the reference's imaginary part is rounding noise).
        const int nyh = ny / 2 + 1;
        RowsArgs r1{fshift, fshift_pitch, A, pnx, (const uint8_t*)mask, mask_pitch, nyh, ny / 2, nx / 2, 1, 0, ny};
        if (int e = launch_rows(p->px, r1, LOAD_MASKED_SHIFTED, s)) return e;
        TransArgs t1 = trans_args(At, pny, nyh, nx, perm_of(p->px, LOAD_MASKED_SHIFTED));
        t1.mirror_rows = ny; t1.mirror_cols = 0;
        if (int e = launch_transpose<float2, float2, false>(A, pnx, t1, s, "transpose_kernel")) return e;
        RowsArgs r2{At, pny, (float2*)absT, pny_f, nullptr, 0, nx, 0, 0, 1, 1};
        if (int e = launch_rows(p->py, r2, LOAD_C64_HPAIR, s)) return e;
    } else {
        RowsArgs r1{fshift, fshift_pitch, A, pnx, (const uint8_t*)mask, mask_pitch, ny, ny / 2, nx / 2, 1, 0};
        if (int e = launch_rows(p->px, r1, LOAD_MASKED_SHIFTED, s)) return e;
        const TransArgs t1 = trans_args(At, pny, ny, nx, perm_of(p->px, LOAD_MASKED_SHIFTED));
        if (int e = launch_transpose<float2, float2, false>(A, pnx, t1, s, "transpose_kernel")) return e;
        RowsArgs r2{At, pny, (float2*)absT, pny_f, nullptr, 0, nx, 0, 0, 1, 1};
        if (int e = launch_rows(p->py, r2, LOAD_C64, s)) return e;
    }
    const RowPerm pm2 = perm_of(p->py, ((ny & 1) && (nx & 1) && !getenv("HD_FFT_NO_HERMITIAN")) ? LOAD_C64_HPAIR : LOAD_C64);
    const TransArgs t2 = trans_args(out, out_pitch, nx, ny, pm2);
    if (out_dtype == HD_F32) return launch_transpose<float, float, false>(absT, pny_f, t2, s, "transpose_real_kernel");
    return launch_transpose<float, double, false>(absT, pny_f, t2, s, "transpose_real_kernel");
}

int hd_fft2_c2c(void* plan, const void* in, int in_dtype, int64_t in_pitch, void* out, int64_t out_pitch, int inverse,
                void* workspace, int64_t workspace_bytes, void* stream)
{
    if (!plan || !in || !out || !workspace) return HD_ERR_NULL;
    Plan2D* p = (Plan2D*)plan;
    const int ny = (int)p->ny, nx = (int)p->nx;
    if (workspace_bytes < hd_fft2_workspace_bytes(ny, nx)) return HD_ERR_WORKSPACE;
    if (in_pitch < nx || out_pitch < nx) return HD_ERR_ARG;
    if (in_dtype != HD_F32 && in_dtype != HD_C64) return HD_ERR_UNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t pnx = pitch_c64(nx), pny = pitch_c64(ny);
    float2* A = (float2*)workspace;                 // [ny][pnx], then [nx][pny]
    float2* At = A + pny * pnx;                     // [nx][pny]
    RowsArgs r1{in, in_pitch, A, pnx, nullptr, 0, ny, 0, 0, inverse ? 1 : 0, 0};
    const int load1 = in_dtype == HD_F32 ? LOAD_REAL : LOAD_C64;
    if (int e = launch_rows(p->px, r1, load1, s)) return e;
    const TransArgs t1 = trans_args(At, pny, ny, nx, perm_of(p->px, load1));
    if (int e = launch_transpose<float2, float2, false>(A, pnx, t1, s, "transpose_kernel")) return e;
    RowsArgs r2{At, pny, A, pny, nullptr, 0, nx, 0, 0, inverse ? 1 : 0, 0};
    if (int e = launch_rows(p->py, r2, LOAD_C64, s)) return e;
    const TransArgs t2 = trans_args(out, out_pitch, nx, ny, perm_of(p->py, LOAD_C64));
    return launch_transpose<float2, float2, false>(A, pny, t2, s, "transpose_kernel");
}

// Batched 1-D transforms along the rows of an (nrows x nx) array (nx = the plan's row length): the building block of
// the row-band distributed fft2 (hydrodem_b200/sharding.py: local row transforms, all-to-all, local column transforms).
// transpose_out: out is (nx x nrows) -- the layout the all-to-all wants, and for free (the transpose also undoes the
// permuted storage of long rows).
int hd_fft_rows(void* plan, const void* in, int in_dtype, int64_t in_pitch, void* out, int64_t out_pitch, int64_t nrows,
                int inverse, int transpose_out, void* workspace, int64_t workspace_bytes, void* stream)
{
    if (!plan || !in || !out || !workspace) return HD_ERR_NULL;
    Plan2D* p = (Plan2D*)plan;
    const int nx = (int)p->nx;
    if (nrows < 1 || nrows > 0x7fffffff) return HD_ERR_ARG;
    if (workspace_bytes < hd_fft2_workspace_bytes(nrows, nx)) return HD_ERR_WORKSPACE;
    if (in_pitch < nx || out_pitch < (transpose_out ? nrows : nx)) return HD_ERR_ARG;
    if (in_dtype != HD_F32 && in_dtype != HD_C64) return HD_ERR_UNSUPPORTED;
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t pnx = pitch_c64(nx), pnr = pitch_c64(nrows);
    float2* A = (float2*)workspace;                 // [nrows][pnx]
    float2* At = A + pnr * pnx;                     // [nx][pnr]
    const bool direct = !transpose_out && p->px.n1 == 1;
    // LOAD_REAL would pack two real rows per transform and emit both spectra: fine here (full spectra are stored)
    RowsArgs r1{in, in_pitch, direct ? (float2*)out : A, direct ? out_pitch : pnx, nullptr, 0, (int)nrows, 0, 0,
                inverse ? 1 : 0, 0};
    const int load1 = in_dtype == HD_F32 ? LOAD_REAL : LOAD_C64;
    if (int e = launch_rows(p->px, r1, load1, s, !direct)) return e;
    if (direct) return HD_OK;
    const TransArgs t1 = trans_args(transpose_out ? out : (void*)At, transpose_out ? out_pitch : pnr, (int)nrows, nx,
                                    perm_of(p->px, load1));
    if (int e = launch_transpose<float2, float2, false>(A, pnx, t1, s, "transpose_kernel")) return e;
    if (transpose_out) return HD_OK;
    // long rows, row layout wanted: transpose back
    const TransArgs t2 = trans_args(out, out_pitch, nx, (int)nrows, RowPerm{1, nx, nullptr});
    return launch_transpose<float2, float2, false>(At, pnr, t2, s, "transpose_kernel");
}


// One pass of the sharded Fourier stage: batched 1-D transforms along the rows of a local (nrows x n) block (n = the
// plan's nx for axis 0, ny for axis 1), then the local transpose into out_t (kept_cols x nrows) in natural frequency
// order -- the layout the all-to-all sends from.  `load` selects exactly the row pass the single-GPU functions run
// (0 real rows [pairs], 1 complex, 2 (1 - mask) * shifted spectrum, 3 Hermitian row pairs), so every transform
// performs the same arithmetic as on one GPU.  real_out: the pass stores |z| (load 1) or |re|, |im| (load 3) as float.
int hd_fft_band_pass(void* plan, int axis, int load, const void* in, int64_t in_pitch, int64_t nrows, const void* mask,
                     int64_t mask_pitch, int shift_cols, int inverse, int real_out, void* out_t, int64_t out_t_pitch,
                     int64_t keep_cols, void* workspace, int64_t workspace_bytes, void* stream)
{
    if (!out_t) return HD_ERR_NULL;
    if (out_t_pitch < nrows) return HD_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const Plan1D* pl;
    int64_t pitch;
    if (int e = band_rows(plan, axis, load, in, in_pitch, nrows, mask, mask_pitch, shift_cols, inverse, real_out, workspace,
                          workspace_bytes, s, &pl, &pitch))
        return e;
    TransArgs t = trans_args(out_t, out_t_pitch, (int)nrows, pl->n_total, perm_of(*pl, load));
    if (real_out) return launch_transpose<float, float, false>((const float*)workspace, pitch, t, s, "transpose_real_kernel");
    t.keep_max = keep_cols > 0 ? (int)keep_cols - 1 : -1;
    return launch_transpose<float2, float2, false>((const float2*)workspace, pitch, t, s, "transpose_kernel");
}


// hd_fft_band_pass with the all-to-all fused into the transpose: the transposed result is scattered into peer memory as
// described by `sc` (see transpose_scatter_kernel).  The caller synchronises the ranks around it (all peers done with the
// destination buffers before, all writes landed after).
int hd_fft_band_pass_scatter(void* plan, int axis, int load, const void* in, int64_t in_pitch, int64_t nrows, const void* mask,
                             int64_t mask_pitch, int shift_cols, int inverse, int real_out, const hd_scatter* sc,
                             int64_t keep_cols, void* workspace, int64_t workspace_bytes, void* stream)
{
    if (!sc) return HD_ERR_NULL;
    if (sc->nseg < 0 || sc->nseg > HD_SCATTER_MAX_SEGS || sc->ncolseg < 0 || sc->ncolseg > 2) return HD_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    const Plan1D* pl;
    int64_t pitch;
    if (int e = band_rows(plan, axis, load, in, in_pitch, nrows, mask, mask_pitch, shift_cols, inverse, real_out, workspace,
                          workspace_bytes, s, &pl, &pitch))
        return e;
    const int n = pl->n_total, grid = transpose_grid((int)nrows, n), keep_max = keep_cols > 0 ? (int)keep_cols - 1 : -1;
    const RowPerm pm = perm_of(*pl, load);
    hd_prof_begin("transpose_scatter_kernel", s);
    if (real_out)
        transpose_scatter_kernel<float><<<grid, 256, 0, s>>>((const float*)workspace, pitch, (int)nrows, n, pm, -1, *sc);
    else
        transpose_scatter_kernel<float2><<<grid, 256, 0, s>>>((const float2*)workspace, pitch, (int)nrows, n, pm, keep_max, *sc);
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

int64_t hd_klayout_rows(int64_t a, int64_t b, int64_t ny) { return KLayout((int)a, (int)b, (int)ny).rows(); }
int64_t hd_klayout_ky(int64_t a, int64_t b, int64_t ny, int64_t t) { return KLayout((int)a, (int)b, (int)ny).ky((int)t); }

int hd_hermitian_complete(const void* half, int64_t half_pitch, void* fshift, int64_t fshift_pitch, void* fabs_out,
                          int64_t fabs_pitch, int64_t a, int64_t b, int64_t ny, int64_t nx, void* stream)
{
    if (!half || !fabs_out) return HD_ERR_NULL;
    if (a < 0 || b <= a || b > ny / 2 + 1 || nx < 2 || half_pitch < nx / 2 + 1 || fabs_pitch < nx || (fshift && fshift_pitch < nx))
        return HD_ERR_ARG;
    const KLayout kl((int)a, (int)b, (int)ny);
    const int64_t total = (int64_t)kl.rows() * nx;
    const int blocks = (int)((total + 255) / 256 < (int64_t)hd_num_sms() * 16 ? (total + 255) / 256 : hd_num_sms() * 16);
    hd_prof_begin("hermitian_complete_kernel", (cudaStream_t)stream);
    hermitian_complete_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const float2*)half, half_pitch, (float2*)fshift,
                                                                       fshift_pitch, (float*)fabs_out, fabs_pitch, kl, (int)nx);
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

int hd_conj_mirror_fill(void* bt, int64_t pitch, int64_t rows, int64_t ny, void* stream)
{
    if (!bt) return HD_ERR_NULL;
    if (rows < 1 || ny < 1 || pitch < ny) return HD_ERR_ARG;
    const int64_t total = rows * (ny - (ny / 2 + 1));
    if (total <= 0) return HD_OK;
    const int blocks = (int)((total + 255) / 256 < (int64_t)hd_num_sms() * 16 ? (total + 255) / 256 : hd_num_sms() * 16);
    hd_prof_begin("conj_mirror_kernel", (cudaStream_t)stream);
    conj_mirror_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((float2*)bt, pitch, (int)rows, (int)ny);
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

int hd_fftshift2(const void* in, int64_t in_pitch, void* out, int64_t out_pitch, int dtype, int64_t ny, int64_t nx,
                 int inverse, void* stream)
{
    if (!in || !out) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || ny > 0x7fffffff || nx > 0x7fffffff || in_pitch < nx || out_pitch < nx || in == out) return HD_ERR_ARG;
    // fftshift moves index k to (k + n/2) % n; ifftshift to (k + n - n/2) % n = (k + (n+1)/2) % n
    const int sr = (int)(inverse ? (ny + 1) / 2 : ny / 2) % (int)ny, sc = (int)(inverse ? (nx + 1) / 2 : nx / 2) % (int)nx;
    const int64_t total = ny * nx;
    const int blocks = (int)((total + 255) / 256 < (int64_t)hd_num_sms() * 16 ? (total + 255) / 256 : hd_num_sms() * 16);
    cudaStream_t s = (cudaStream_t)stream;
    switch (hd_dtype_size(dtype)) {
        case 4: hd_prof_begin("shift_kernel", s); shift_kernel<float><<<blocks, 256, 0, s>>>((const float*)in, in_pitch, (float*)out, out_pitch, (int)ny, (int)nx, sr, sc); break;
        case 8: hd_prof_begin("shift_kernel", s); shift_kernel<double><<<blocks, 256, 0, s>>>((const double*)in, in_pitch, (double*)out, out_pitch, (int)ny, (int)nx, sr, sc); break;
        case 16: hd_prof_begin("shift_kernel", s); shift_kernel<double2><<<blocks, 256, 0, s>>>((const double2*)in, in_pitch, (double2*)out, out_pitch, (int)ny, (int)nx, sr, sc); break;
        default: return HD_ERR_UNSUPPORTED;
    }
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

}  // extern "C"

// hydrodem_b200 -- the GeoTIFF block decoders (Deflate with its zlib wrapper, TIFF LZW), one __host__ __device__ core for
// the host entry points (hd_host_inflate, hd_host_tiff_lzw) and for one warp per block on the device (tiffdecode.cu).
//
// Both codecs decode one symbol at a time and then copy a run of earlier output.  The serial part runs identically on
// every lane of the caller (all lanes read the same input bytes and keep the same state in registers); the copy goes
// through an EMITTER: HostEmit copies byte by byte, the device emitter (tiffdecode.cu) with the 32 lanes of a warp.
// LZW table entries are (offset in the block's output, length): every LZW string is a substring of the output already
// written, so decoding a code is one copy as well.
//
// Safety on hostile input: every loop is bounded by the input's bit count or the output capacity, every back-reference is
// checked against the bytes already written and every write against the capacity, every Huffman code is checked for
// over-subscription / incompleteness as zlib's inftrees.c does.  Result: OK, CORRUPT, or HOST (a legal Deflate stream that
// decodes to more than `cap` bytes: writing stopped at `cap`, the caller re-decodes the block on the host).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define TC_HD __host__ __device__ __forceinline__
#else
#define TC_HD inline
#endif

namespace tiffcodec {

enum Status : int { OK = 0, CORRUPT = 1, HOST = 2 };

// ---- emitter of the host: one lane ------------------------------------------------------------------------------------
struct HostEmit {
    uint8_t* out;
    static constexpr int lanes = 1;
    TC_HD int lane() const { return 0; }
    TC_HD void sync() const {}
    TC_HD uint64_t sum(uint64_t v) const { return v; }
    TC_HD void put(int64_t op, uint8_t b) const { out[op] = b; }
    // out[op + i] = out[op - dist + i] for i < len, in order (so an overlapping run repeats its period)
    TC_HD void copy(int64_t op, int64_t dist, int64_t len) const
    {
        for (int64_t i = 0; i < len; ++i) out[op + i] = out[op - dist + i];
    }
    TC_HD void copy_in(int64_t op, const uint8_t* src, int64_t len) const
    {
        for (int64_t i = 0; i < len; ++i) out[op + i] = src[i];
    }
    TC_HD void zero(int64_t a, int64_t b) const
    {
        for (int64_t i = a; i < b; ++i) out[i] = 0;
    }
    TC_HD const uint8_t* data() const { return out; }
};

// ---- Adler-32 of out[0, n), lanes of the emitter in parallel -----------------------------------------------------------
template <class E>
TC_HD uint32_t adler32(const E& em, int64_t n)
{
    const uint8_t* p = em.data();
    uint64_t s1 = 0, s2 = 0;                                     // s2 = sum of (n - i) * p[i]; per lane < 2^63 for n < 2^38
    for (int64_t i = em.lane(); i < n; i += E::lanes) {
        const uint64_t d = p[i];
        s1 += d;
        s2 += (uint64_t)((n - i) % 65521) * d;
        if ((i / E::lanes & 0xFFFF) == 0xFFFF) { s1 %= 65521; s2 %= 65521; }
    }
    s1 = em.sum(s1 % 65521) % 65521;
    s2 = em.sum(s2 % 65521) % 65521;
    const uint32_t a = (uint32_t)((1 + s1) % 65521);
    const uint32_t b = (uint32_t)((s2 + (uint64_t)(n % 65521)) % 65521);
    return (b << 16) | a;
}

// ---- Deflate (RFC 1950 / 1951) ------------------------------------------------------------------------------------------
constexpr int LFAST = 10, DFAST = 8;                             // primary table bits; longer codes: canonical walk

struct Huff {                                                    // canonical code: count per length, symbols by code
    uint16_t count[16];
    uint16_t symbol[288];
};

struct InflateTables {                                           // per-decoder scratch (a warp's shared memory on the device)
    uint16_t lfast[1 << LFAST];                                  // (len << 9) | symbol, 0 = not resolved in LFAST bits
    uint16_t dfast[1 << DFAST];
    Huff lit, dist, codes;
    uint8_t lens[32 + 286 + 30];                                 // [0, 19): code lengths code; [32, ...): literal / distance
    int fixed;                                                   // the tables hold the fixed code
};

// LSB-first bit reader over src[0, n); past the end it reads zeros and overrun() tells
struct BitsLSB {
    const uint8_t* p;
    int64_t n, pos;
    uint64_t buf;
    int cnt;
    TC_HD void refill()
    {
        while (cnt <= 56) {
            const uint64_t b = pos < n ? p[pos] : 0;
            ++pos;
            buf |= b << cnt;
            cnt += 8;
        }
    }
    TC_HD uint32_t peek(int k) { if (cnt < k) refill(); return (uint32_t)(buf & ((1ull << k) - 1)); }
    TC_HD void drop(int k) { buf >>= k; cnt -= k; }
    TC_HD uint32_t get(int k) { const uint32_t v = peek(k); drop(k); return v; }
    TC_HD bool overrun() const { return pos * 8 - cnt > n * 8; }
    TC_HD int64_t byte_pos() const { return pos - cnt / 8; }      // after align(): the next unread byte
    TC_HD void align() { drop(cnt & 7); }
    TC_HD void seek(int64_t b) { pos = b; buf = 0; cnt = 0; }
};

// canonical walk of `bits` (next code bits, first bit in bit 0) up to maxlen bits: symbol | len << 9, or 0
TC_HD uint32_t huff_walk(const Huff& h, uint32_t bits, int maxlen)
{
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= maxlen; ++len) {
        code |= (bits >> (len - 1)) & 1;
        const int c = h.count[len];
        if (code - c < first) return (uint32_t)h.symbol[index + code - first] | ((uint32_t)len << 9);
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return 0;
}

enum HuffKind { CODES, LENS, DISTS };

// inftrees.c's rules: over-subscribed -> error; incomplete -> error unless a LENS / DISTS code with one code of length 1;
// no code at all -> an error for CODES (zlib then fails on the missing end-of-block), accepted for DISTS
template <class E>
TC_HD bool huff_build(const E& em, Huff& h, const uint8_t* lens, int n, HuffKind kind, uint16_t* fast, int fast_bits)
{
    bool ok = true;
    if (em.lane() == 0) {
        for (int l = 0; l < 16; ++l) h.count[l] = 0;
        for (int s = 0; s < n; ++s) h.count[lens[s]]++;
        h.count[0] = 0;
        int maxlen = 0;
        for (int l = 1; l < 16; ++l)
            if (h.count[l]) maxlen = l;
        if (maxlen == 0) {
            ok = kind == DISTS;
        } else {
            int left = 1;
            for (int l = 1; l < 16 && ok; ++l) {
                left = (left << 1) - h.count[l];
                if (left < 0) ok = false;
            }
            if (ok && left > 0 && (kind == CODES || maxlen != 1)) ok = false;
        }
        if (ok) {
            uint16_t offs[16];
            offs[1] = 0;
            for (int l = 1; l < 15; ++l) offs[l + 1] = (uint16_t)(offs[l] + h.count[l]);
            for (int s = 0; s < n; ++s)
                if (lens[s]) h.symbol[offs[lens[s]]++] = (uint16_t)s;
        }
    }
    em.sync();
    // every lane reaches the same verdict: lane 0 published it through the count of length 0
    if (em.lane() == 0) h.count[0] = ok ? 0 : 1;
    em.sync();
    ok = h.count[0] == 0;
    if (ok && fast)
        for (int e = em.lane(); e < (1 << fast_bits); e += E::lanes) fast[e] = (uint16_t)huff_walk(h, (uint32_t)e, fast_bits);
    em.sync();
    return ok;
}

// next symbol of the code (fast table, else the canonical walk over 15 bits); -1 for a code that is not in the table
TC_HD int huff_decode(BitsLSB& br, const Huff& h, const uint16_t* fast, int fast_bits)
{
    const uint32_t bits = br.peek(15);
    uint32_t e = fast ? fast[bits & ((1u << fast_bits) - 1)] : 0;
    if (!e) e = huff_walk(h, bits, 15);
    if (!e) return -1;
    br.drop((int)(e >> 9));
    return (int)(e & 511);
}

template <class E>
TC_HD int inflate(const uint8_t* src, int64_t n, const E& em, int64_t cap, InflateTables& t, int64_t* out_len)
{
    static constexpr uint16_t LBASE[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59,
                                           67, 83, 99, 115, 131, 163, 195, 227, 258};
    static constexpr uint8_t LEXT[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    static constexpr uint16_t DBASE[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                           1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
    static constexpr uint8_t DEXT[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11,
                                         12, 12, 13, 13};
    static constexpr uint8_t ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    int64_t op = 0;
    *out_len = 0;
    // zlib header: method 8, window <= 32 KB, FCHECK, no preset dictionary (zlib.decompress needs one it cannot have)
    if (n < 2) return CORRUPT;
    const uint32_t cmf = src[0], flg = src[1];
    if ((cmf * 256 + flg) % 31 != 0 || (cmf & 15) != 8 || (cmf >> 4) > 7 || (flg & 0x20)) return CORRUPT;
    BitsLSB br{src, n, 2, 0, 0};
    if (em.lane() == 0) t.fixed = 0;
    em.sync();
    int last = 0;
    while (!last) {
        last = (int)br.get(1);
        const uint32_t type = br.get(2);
        if (br.overrun()) return CORRUPT;
        if (type == 0) {                                         // stored
            br.align();
            const uint32_t len = br.get(16), nlen = br.get(16);
            if (br.overrun() || len != (~nlen & 0xFFFF)) return CORRUPT;
            const int64_t b = br.byte_pos();
            if (b + len > n) return CORRUPT;
            const int64_t w = len <= cap - op ? (int64_t)len : cap - op;
            em.copy_in(op, src + b, w);
            op += w;
            if (w < (int64_t)len) { *out_len = op; return HOST; }
            br.seek(b + len);
            continue;
        }
        if (type == 3) return CORRUPT;
        if (type == 1) {                                         // fixed code
            if (!t.fixed) {
                if (em.lane() == 0) {
                    for (int s = 0; s < 288; ++s) t.lens[s] = s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8;
                    for (int s = 0; s < 32; ++s) t.lens[288 + s] = 5;
                }
                em.sync();
                huff_build(em, t.lit, t.lens, 288, LENS, t.lfast, LFAST);
                huff_build(em, t.dist, t.lens + 288, 32, DISTS, t.dfast, DFAST);
                if (em.lane() == 0) t.fixed = 1;
                em.sync();
            }
        } else {                                                 // dynamic code
            const int nlen = (int)br.get(5) + 257, ndist = (int)br.get(5) + 1, ncode = (int)br.get(4) + 4;
            if (nlen > 286 || ndist > 30) return CORRUPT;
            if (em.lane() == 0)
                for (int i = 0; i < 19; ++i) t.lens[i] = 0;
            em.sync();
            for (int i = 0; i < ncode; ++i) {                    // every lane reads, lane 0 stores
                const uint8_t v = (uint8_t)br.get(3);
                if (em.lane() == 0) t.lens[ORDER[i]] = v;
            }
            em.sync();
            if (br.overrun()) return CORRUPT;
            if (!huff_build(em, t.codes, t.lens, 19, CODES, nullptr, 0)) return CORRUPT;
            if (em.lane() == 0) t.fixed = 0;
            em.sync();
            int i = 0;
            uint8_t lens_local_prev = 0;
            while (i < nlen + ndist) {
                const int sym = huff_decode(br, t.codes, nullptr, 0);
                if (sym < 0 || br.overrun()) return CORRUPT;
                int rep = 1;
                uint8_t val;
                if (sym < 16) {
                    val = (uint8_t)sym;
                } else if (sym == 16) {
                    if (i == 0) return CORRUPT;
                    val = lens_local_prev;
                    rep = 3 + (int)br.get(2);
                } else if (sym == 17) {
                    val = 0;
                    rep = 3 + (int)br.get(3);
                } else {
                    val = 0;
                    rep = 11 + (int)br.get(7);
                }
                if (i + rep > nlen + ndist) return CORRUPT;
                if (em.lane() == 0)
                    for (int r = 0; r < rep; ++r) t.lens[32 + i + r] = val;   // 32..: clear of the 19 code lengths
                i += rep;
                lens_local_prev = val;
            }
            if (br.overrun()) return CORRUPT;
            em.sync();
            if (t.lens[32 + 256] == 0) return CORRUPT;           // no end-of-block code
            if (!huff_build(em, t.lit, t.lens + 32, nlen, LENS, t.lfast, LFAST)) return CORRUPT;
            if (!huff_build(em, t.dist, t.lens + 32 + nlen, ndist, DISTS, t.dfast, DFAST)) return CORRUPT;
        }
        for (;;) {                                               // the block's symbols: each takes at least one bit
            const int sym = huff_decode(br, t.lit, t.lfast, LFAST);
            if (sym < 0 || br.overrun()) return CORRUPT;
            if (sym < 256) {
                if (op >= cap) { *out_len = op; return HOST; }
                em.put(op++, (uint8_t)sym);
                continue;
            }
            if (sym == 256) break;
            if (sym > 285) return CORRUPT;
            const int len = LBASE[sym - 257] + (int)br.get(LEXT[sym - 257]);
            const int ds = huff_decode(br, t.dist, t.dfast, DFAST);
            if (ds < 0 || ds > 29) return CORRUPT;
            const int64_t dist = DBASE[ds] + (int64_t)br.get(DEXT[ds]);
            if (br.overrun() || dist > op) return CORRUPT;
            const int64_t w = len <= cap - op ? (int64_t)len : cap - op;
            em.copy(op, dist, w);
            op += w;
            if (w < len) { *out_len = op; return HOST; }
        }
    }
    br.align();
    const int64_t b = br.byte_pos();
    if (br.overrun() || b + 4 > n) return CORRUPT;
    const uint32_t want = (uint32_t)src[b] << 24 | (uint32_t)src[b + 1] << 16 | (uint32_t)src[b + 2] << 8 | src[b + 3];
    em.sync();
    *out_len = op;
    return adler32(em, op) == want ? OK : CORRUPT;
}

// ---- TIFF LZW (TIFF 6.0 section 13, as hd_host_lzw_decode): MSB-first codes, 9..12 bits, early change --------------------
struct LzwTable {
    uint32_t off[4096];                                          // entry c >= 258: out[off, off + len)
    uint16_t len[4096];
};

// OK with *out_len bytes written (the stream ended at EOI, ran out of data, or filled `cap`), or CORRUPT
template <class E>
TC_HD int lzw(const uint8_t* src, int64_t n, const E& em, int64_t cap, LzwTable& t, int64_t* out_len)
{
    int nbits = 9, next = 258, old = -1;
    int64_t p_old = 0, l_old = 0;                                // where the previous string was written, its length
    uint64_t acc = 0;
    int have = 0;
    int64_t ip = 0, op = 0;
    *out_len = 0;
    for (;;) {
        while (have < nbits && ip < n) { acc = (acc << 8) | src[ip++]; have += 8; }
        if (have < nbits) break;                                 // data ran out without EOI
        const int code = (int)((acc >> (have - nbits)) & ((1u << nbits) - 1u));
        have -= nbits;
        if (code == 256) {                                       // entries are rewritten from here: no lane may lag behind
            nbits = 9; next = 258; old = -1;
            em.sync();
            continue;
        }
        if (code == 257) break;
        if (old < 0) {
            if (code > 255) return CORRUPT;
            if (op >= cap) break;
            em.put(op, (uint8_t)code);
            p_old = op++;
            l_old = 1;
            old = code;
            continue;
        }
        int64_t len;
        if (code < 256) {
            len = 1;
        } else if (code < next) {
            len = t.len[code];
        } else if (code == next) {
            len = l_old + 1;                                     // old's string + its first byte: an overlapping copy
        } else {
            return CORRUPT;
        }
        const int64_t w = len <= cap - op ? len : cap - op;
        if (code < 256) {
            if (w > 0) em.put(op, (uint8_t)code);
        } else {
            em.copy(op, op - (code == next ? p_old : (int64_t)t.off[code]), w);
        }
        if (next < 4096) {                                       // every lane writes the same entry: no wait before reads
            t.off[next] = (uint32_t)p_old;
            t.len[next] = (uint16_t)(l_old + 1);
            ++next;
            if (next == (1 << nbits) - 1 && nbits < 12) ++nbits;
        }
        p_old = op;
        l_old = len;
        op += w;
        old = code;
        if (op >= cap) break;
    }
    *out_len = op;
    return OK;
}

}  // namespace tiffcodec

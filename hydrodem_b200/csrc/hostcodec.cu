// HOST code of the C ABI (no kernel in this file): the TIFF flavour of LZW, for the GeoTIFF reader of the chain's callers
// (hydrodem_b200/geotiff.py; SURVEY.md section 8(f) rank 2: GDAL's COMPRESS=LZW rasters).  TIFF 6.0 section 13:
// codes are packed MSB first, start at 9 bits, 256 = ClearCode, 257 = EndOfInformation, first free code 258, and the code
// width grows one code EARLY (when the next free code reaches 2^width - 1), up to 12 bits.
#include <cstdint>
#include <cstring>

#include "../../include/hydrodem_b200.h"

extern "C" int64_t hd_host_lzw_decode(const uint8_t* src, int64_t nsrc, uint8_t* dst, int64_t cap)
{
    if (!src || !dst) return HD_ERR_NULL;
    if (nsrc < 0 || cap < 0) return HD_ERR_ARG;
    uint16_t prefix[4096];
    uint8_t suffix[4096], first[4096];
    uint16_t length[4096];
    for (int i = 0; i < 256; ++i) { prefix[i] = 0; suffix[i] = (uint8_t)i; first[i] = (uint8_t)i; length[i] = 1; }
    int nbits = 9, next = 258, old = -1;
    uint64_t acc = 0;
    int have = 0;
    int64_t ip = 0, op = 0;
    for (;;) {
        while (have < nbits && ip < nsrc) { acc = (acc << 8) | src[ip++]; have += 8; }
        if (have < nbits) break;                                  // data ran out without EOI: libtiff accepts that too
        const int code = (int)((acc >> (have - nbits)) & ((1u << nbits) - 1u));
        have -= nbits;
        if (code == 256) { nbits = 9; next = 258; old = -1; continue; }
        if (code == 257) break;
        if (old < 0) {
            if (code > 255) return HD_ERR_ARG;                    // a fresh table only holds the 256 roots
            if (op >= cap) break;
            dst[op++] = (uint8_t)code;
            old = code;
            continue;
        }
        int len;
        uint8_t head;
        if (code < next) {                                        // known string
            len = length[code];
            head = first[code];
        } else if (code == next) {                                // the string being defined: old + first(old)
            len = length[old] + 1;
            head = first[old];
        } else {
            return HD_ERR_ARG;                                    // corrupt stream
        }
        const int64_t room = cap - op;
        const int out = len <= room ? len : (int)room;
        {   // write the string back to front along the prefix chain (cut off at the capacity of dst)
            int c = code, k = len;
            if (code == next) {
                if (k <= out) dst[op + k - 1] = head;
                --k;
                c = old;
            }
            while (k > 0) {
                if (k <= out) dst[op + k - 1] = suffix[c];
                c = prefix[c];
                --k;
            }
        }
        op += out;
        if (next < 4096) {
            prefix[next] = (uint16_t)old;
            suffix[next] = head;
            first[next] = first[old];
            length[next] = (uint16_t)(length[old] + 1);
            ++next;
            if (next == (1 << nbits) - 1 && nbits < 12) ++nbits;  // "early change"
        }
        old = code;
        if (op >= cap) break;
    }
    return op;
}

// ---- the GPU decoder's core on the host (csrc/tiffcodec.cuh), for tests against zlib and hd_host_lzw_decode ------------
#include "tiffcodec.cuh"

extern "C" int64_t hd_host_inflate(const uint8_t* src, int64_t nsrc, uint8_t* dst, int64_t cap)
{
    if (!src || !dst) return HD_ERR_NULL;
    if (nsrc < 0 || cap < 0) return HD_ERR_ARG;
    tiffcodec::InflateTables t;
    int64_t n = 0;
    const int st = tiffcodec::inflate(src, nsrc, tiffcodec::HostEmit{dst}, cap, t, &n);
    return st == tiffcodec::OK ? n : st == tiffcodec::HOST ? (int64_t)HD_ERR_WORKSPACE : (int64_t)HD_ERR_ARG;
}

extern "C" int64_t hd_host_tiff_lzw(const uint8_t* src, int64_t nsrc, uint8_t* dst, int64_t cap)
{
    if (!src || !dst) return HD_ERR_NULL;
    if (nsrc < 0 || cap < 0) return HD_ERR_ARG;
    static thread_local tiffcodec::LzwTable t;
    int64_t n = 0;
    const int st = tiffcodec::lzw(src, nsrc, tiffcodec::HostEmit{dst}, cap, t, &n);
    return st == tiffcodec::OK ? n : (int64_t)HD_ERR_ARG;
}

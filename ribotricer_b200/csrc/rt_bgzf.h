// rt_bgzf.h -- BGZF members (SAM spec 4.1) as the BAM decoder (rt_bam.cpp) and the BGZF text inflate (rt_capi.cu,
// rt_bgzf_inflate) read them: the header walk and the host decoder of one member.  Internal to the library, like
// rt_host.h: everything here has internal linkage.
#pragma once

#include <zlib.h>

#include <cstdint>
#include <cstring>

bool rt_inflate_fast(const uint8_t* in, size_t in_n, uint8_t* out, size_t out_n);   // rt_inflate.cpp
uint32_t rt_crc32_fast(const uint8_t* p, size_t n);

namespace {

inline uint16_t bgzf_rd16(const uint8_t* p) { uint16_t v; memcpy(&v, p, 2); return v; }
inline uint32_t bgzf_rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }

struct Block { size_t in_off, in_len; size_t out_off; uint32_t out_len, crc; };

// One BGZF member: gzip header with a 'BC' extra subfield holding the block size (SAM spec 4.1).
bool parse_block(const uint8_t* base, size_t size, size_t off, Block& b, size_t& next) {
    if (off + 18 > size) return false;
    const uint8_t* p = base + off;
    if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return false;
    const uint16_t xlen = bgzf_rd16(p + 10);
    if (off + 12 + xlen > size) return false;
    int bsize = -1;
    for (size_t x = 12; x + 4 <= 12u + xlen;) {
        const uint16_t slen = bgzf_rd16(p + x + 2);
        if (p[x] == 'B' && p[x + 1] == 'C' && slen == 2) bsize = bgzf_rd16(p + x + 4);
        x += 4 + slen;
    }
    if (bsize < 0) return false;
    const size_t total = (size_t)bsize + 1;
    if (off + total > size || total < 12u + xlen + 8) return false;
    b.in_off = off + 12 + xlen;
    b.in_len = total - (12 + xlen) - 8;
    b.out_len = bgzf_rd32(p + total - 4);
    if (b.out_len > 65536u) return false;              // a BGZF block holds at most 64 KiB (SAM spec 4.1)
    b.crc = bgzf_rd32(p + total - 8);
    next = off + total;
    return true;
}

// Why parse_block refused the member at `off`: 1 = the file ends inside it (a gzip member header whose extra field or
// announced block size runs past the end), 2 = not a gzip member at all, 0 = a gzip member that is not a valid BGZF one.
int block_refusal(const uint8_t* base, size_t size, size_t off) {
    const uint8_t* p = base + off;
    const size_t rem = size - off;
    if (rem >= 1 && p[0] != 0x1f) return 2;
    if (rem >= 2 && p[1] != 0x8b) return 2;
    if (rem < 12) return 1;
    if (p[2] != 8 || !(p[3] & 4)) return 0;
    const uint16_t xlen = bgzf_rd16(p + 10);
    if (12u + xlen > rem) return 1;
    for (size_t x = 12; x + 4 <= 12u + xlen;) {
        const uint16_t slen = bgzf_rd16(p + x + 2);
        if (p[x] == 'B' && p[x + 1] == 'C' && slen == 2 && x + 6 <= 12u + xlen)
            return (size_t)bgzf_rd16(p + x + 4) + 1 > rem ? 1 : 0;
        x += 4 + slen;
    }
    return 0;
}

bool inflate_zlib(const uint8_t* src, size_t n, uint8_t* dst, uint32_t out_len) {
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) return false;
    zs.next_in = const_cast<Bytef*>(src);
    zs.avail_in = (uInt)n;
    zs.next_out = dst;
    zs.avail_out = out_len;
    const int rc = inflate(&zs, Z_FINISH);
    inflateEnd(&zs);
    return rc == Z_STREAM_END && zs.total_out == out_len;
}

// One BGZF block: the decoder of rt_inflate.cpp, checked against the CRC-32 of the block's footer; a block it refuses
// (or gets wrong) is decoded again by zlib, so the result never depends on the fast decoder alone.
bool inflate_block(const uint8_t* src, size_t n, uint8_t* dst, uint32_t out_len, uint32_t crc, bool zlib_only) {
    if (out_len == 0) return true;
    if (!zlib_only && rt_inflate_fast(src, n, dst, out_len) && rt_crc32_fast(dst, out_len) == crc) return true;
    return inflate_zlib(src, n, dst, out_len) && rt_crc32_fast(dst, out_len) == crc;
}

}  // namespace

// gcn10_b200/csrc/lzw_core.h -- the sequential half of the GPU decoder of LZW-compressed TIFF tiles.
//
// TIFF Compression 5 as libtiff writes and reads it (tif_lzw.c, LZWDecode; what GDAL's GTiff driver links): codes of
// 9 to 12 bits, most significant bit first, Clear = 256, EOI = 257, the first free entry 258, and the "early change" --
// the code width grows when the next free entry reaches 2^n - 1, one code before the table needs it.
//
// Every code >= 258 names a string that is an earlier piece of the output: entry e, made while decoding code i, is the
// output of code i - 1 followed by the first byte of code i's output -- i.e. the bytes that start where code i - 1's
// output starts, one longer.  So the decode lane keeps only (start, length) per entry and turns codes into LZ77-like
// (output position, source position) pairs, with no suffix chains; the bytes are produced by the writer warp
// (lzw_tiles.cuh).  Like inflate_core.h this header is plain C++ that tests/harness/lzw_host.cpp compiles for the host.
//
// Verdicts follow libtiff's LZWDecode: decoding stops when the tile is full (later codes are ignored, a string that
// crosses the end is cut); EOI or the end of the input before the tile is full is an error ("Not enough data"); so are
// a code above the next free entry, a first code after Clear that is not a literal, a code before the first Clear, and
// a code that would make entry 5119 (libtiff's table has 1023 spare entries behind code 4095: an encoder that misses
// its Clear by less than that still decodes).  Old-style (pre-TIFF 5.0, LSB-first) streams are refused.
#pragma once

#include "inflate_core.h"

namespace gcn10 {
namespace lzw {

constexpr int kCodes = 4096;            // entries a 12-bit code can name
constexpr uint32_t kTableLimit = 4096u + 1023u;     // libtiff's CSIZE: making entry kTableLimit is an error
constexpr int kBatch = 64;              // codes per batch
constexpr uint32_t kBatchBytes = 2048;  // a batch closes once its output reaches this: with strings of at most 3839
                                        // bytes a batch stays below 5887 bytes, so the batch plus the unflushed
                                        // piece before it (< inflate::kPiece) fits the 8 KB history ring
constexpr uint32_t kLit = 0x80000000u;  // queue source word: literal byte (else a source position in the tile)

// status codes behind inflate::kErrChecksum (10); kErrInput / kErrShort keep their meaning
enum {
    kErrOldStyle = 11,      // an old-style (pre-TIFF 5.0, LSB-first) LZW stream: not supported
    kErrCode = 12           // a code above the next free entry, a first code after Clear above 257, a code before the
                            // first Clear, or a table that overflows libtiff's without a Clear
};

struct Lane {
    uint64_t buf;           // bit buffer, MSB first: the next code is in the top bits
    int cnt;                // valid bits in buf
    uint32_t cons;          // byte offset (from the 16-byte aligned stream base) of the next ring word to load
    uint64_t bits_left;     // bits of the stream not consumed yet
    uint32_t out, out_end;  // output position / tile size
    uint32_t free_ent;      // next entry
    int nbits;              // code width
    int state;              // 0 = before the first Clear, 1 = right after a Clear, 2 = decoding
    uint32_t old_pos, old_len;  // output of the previous code
    int err;
};

GCN10_HD uint32_t bswap32(uint32_t v)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(v, 0u, 0x0123);
#else
    return (v >> 24) | ((v >> 8) & 0xFF00u) | ((v << 8) & 0xFF0000u) | (v << 24);
#endif
}

// cnt >= 32 afterwards
GCN10_HD void need32(Lane &s, const uint32_t *ring)
{
    if (s.cnt <= 32) {
        const uint32_t w = bswap32(ring[(s.cons >> 2) & (inflate::kRingWords - 1)]);
        s.buf |= (uint64_t)w << (32 - s.cnt);
        s.cnt += 32;
        s.cons += 4;
    }
}

// first_byte: offset of the stream from its 16-byte aligned base; the ring must hold its first word
GCN10_HD void lane_init(Lane &s, const uint32_t *ring, uint32_t first_byte, uint32_t size, uint32_t out_end)
{
    s.buf = 0;
    s.cnt = 0;
    s.cons = first_byte & ~3u;
    s.bits_left = 8ull * size;
    s.out = 0;
    s.out_end = out_end;
    s.free_ent = 258;
    s.nbits = 9;
    s.state = 0;
    s.old_pos = s.old_len = 0;
    s.err = 0;
    need32(s, ring);
    const int skip = 8 * (int)(first_byte & 3u);
    s.buf <<= skip;
    s.cnt -= skip;
    need32(s, ring);                    // a stream at offset 3 mod 4 has only its first byte in the first word
    // libtiff's test for an old-style stream: a first byte 0 with the low bit of the second set (the LSB-first Clear)
    if (size >= 2 && (s.buf >> 56) == 0u && ((s.buf >> 48) & 1u))
        s.err = kErrOldStyle;
}

// Up to kBatch codes read (Clear codes included: the caller stages the input ring between batches, and a batch reads
// at most kBatch * 12 bits of it), stopping early once kBatchBytes are queued.  Code j of the batch writes output
// [pos[j], pos[j + 1]) (the last one up to s.out); src[j] is kLit | byte or the position its bytes are copied from
// (src[j] < pos[j]; src[j] + length may reach pos[j] + 1: the KwKwK case, whose last byte is its own first).
// Returns the number queued; *event = kEvMore, kEvEnd (the tile is full) or kEvError (s.err says why).
GCN10_HD int decode_codes(Lane &s, const uint32_t *ring, uint32_t *tstart, uint16_t *tlen, uint32_t *pos, uint32_t *src,
                          int *event)
{
    using namespace inflate;
    *event = kEvMore;
    if (s.err) {
        *event = kEvError;
        return 0;
    }
    const uint32_t b0 = s.out;
    int n = 0;
    for (int reads = 0; reads < kBatch && s.out - b0 < kBatchBytes; reads++) {
        if (s.out >= s.out_end) {
            *event = kEvEnd;
            break;
        }
        if (s.bits_left < (uint64_t)s.nbits) {
            s.err = kErrInput;                  // input exhausted before the tile is full
            break;
        }
        need32(s, ring);
        const uint32_t code = (uint32_t)(s.buf >> (64 - s.nbits));
        s.buf <<= s.nbits;
        s.cnt -= s.nbits;
        s.bits_left -= (uint64_t)s.nbits;
        if (code == 256u) {
            s.free_ent = 258;
            s.nbits = 9;
            s.state = 1;
            continue;
        }
        if (code == 257u) {
            s.err = kErrShort;                  // EOI before the tile is full
            break;
        }
        uint32_t sw, len;
        if (s.state == 1) {
            if (code > 255u) {
                s.err = kErrCode;
                break;
            }
            sw = kLit | code;
            len = 1;
            s.state = 2;
        }
        else {
            if (s.state == 0 || s.free_ent >= kTableLimit || code > s.free_ent) {
                s.err = kErrCode;
                break;
            }
            // the new entry: the previous code's output plus one byte (the first of this code's output)
            if (s.free_ent < (uint32_t)kCodes) {
                tstart[s.free_ent] = s.old_pos;
                tlen[s.free_ent] = (uint16_t)(s.old_len + 1u);
            }
            s.free_ent++;
            if (s.free_ent >= (1u << s.nbits) - 1u && s.nbits < 12)
                s.nbits++;
            if (code < 256u) {
                sw = kLit | code;
                len = 1;
            }
            else {
                sw = tstart[code];
                len = tlen[code];
            }
        }
        pos[n] = s.out;
        src[n] = sw;
        n++;
        s.old_pos = s.out;
        s.old_len = len;
        const uint32_t room = s.out_end - s.out;
        s.out += len < room ? len : room;
    }
    if (s.err) {
        *event = kEvError;
        return 0;
    }
    return n;
}

// The writer's rule for byte p of a batch that starts at b0, in code k (pos[k] <= p < pos[k + 1]): follow the copy
// sources back until a literal or a byte before the batch.  Returns kLit | byte, or the position (< b0) to read.
// Every step moves to a strictly smaller position, so the loop ends.
GCN10_HD uint32_t resolve(const uint32_t *pos, const uint32_t *src, int n, uint32_t b0, uint32_t p, int k)
{
    for (;;) {
        const uint32_t sw = src[k];
        if (sw & kLit)
            return sw;
        p = sw + (p - pos[k]);
        if (p < b0)
            return p;
        int lo = 0, hi = k;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (pos[mid] <= p)
                lo = mid;
            else
                hi = mid - 1;
        }
        k = lo;
    }
}

}  // namespace lzw
}  // namespace gcn10

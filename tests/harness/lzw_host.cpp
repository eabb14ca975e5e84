// tests/harness/lzw_host.cpp -- TEST HARNESS, not product code.
//
// Compiles gcn10_b200/csrc/lzw_core.h (the decode-lane half of the GPU LZW tile decoder) for the host and drives it
// with a scalar emulation of the writer warp of lzw_tiles.cuh: the same 2 KB input ring and refill rule, the same
// batches, every byte of a batch resolved with lzw::resolve against the 8 KB history ring or -- for bytes older than
// the last flush -- the tile buffer the flushed 2 KB pieces went to.  tests/test_lzw_core.py compares the result with
// libtiff.  Built by the test itself (g++ -shared); nothing under gcn10_b200/ links or loads it.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../gcn10_b200/csrc/lzw_core.h"

using namespace gcn10;

// Returns the tile's status (0 or an inflate::kErr* / lzw::kErr* code), or a negative value when an invariant of
// lzw_core.h breaks; out[0, out_len) receives the tile's bytes as the flusher stores them.  stats: [codes, batches].
extern "C" int gcn10_test_lzw(const uint8_t *stream, uint32_t size, uint32_t misalign, uint8_t *out, uint32_t out_len,
                              uint64_t *stats)
{
    using namespace inflate;
    std::vector<uint8_t> padded((size_t)misalign + size + 4096 + 64, 0xA5);
    const uint32_t first = misalign & 15u;
    memcpy(padded.data() + first, stream, size);
    const uint8_t *base = padded.data();

    static uint32_t tstart[lzw::kCodes];
    static uint16_t tlen[lzw::kCodes];
    uint32_t ring[kRingWords];
    uint32_t qpos[lzw::kBatch], qsrc[lzw::kBatch];
    std::vector<uint8_t> window(kWindow, 0);
    uint32_t filled = 0;
    auto top_up = [&](uint32_t cons) {
        while (filled < cons + 1024u) {
            for (uint32_t k = 0; k < 512; k++)
                ((uint8_t *)ring)[(filled + k) & 2047u] = base[filled + k];
            filled += 512u;
        }
    };
    // the plane is the caller's buffer: flushed pieces go straight there, so a write past the tile hits the caller's
    // guard band; bytes not flushed yet keep the caller's fill value, which a wrong read-back would show
    uint8_t *plane = out;
    top_up(first & ~3u);
    lzw::Lane s;
    lzw::lane_init(s, ring, first, size, out_len);
    uint32_t b0 = 0, flushed = 0;
    uint64_t ncodes = 0, nbatches = 0;
    int err = 0;
    for (;;) {
        top_up(s.cons);
        int ev = kEvMore;
        const int n = lzw::decode_codes(s, ring, tstart, tlen, qpos, qsrc, &ev);
        if (ev == kEvError) {
            err = s.err;
            break;
        }
        const uint32_t b1 = s.out;
        if (b1 - flushed > (uint32_t)kWindow)
            return -1;                          // the ring bound of lzw_core.h does not hold
        if (b1 > out_len)
            return -3;                          // a batch runs past the tile
        // all bytes of the batch are resolved first, then stored: none of them depends on another
        std::vector<uint8_t> v(b1 - b0);
        int k = 0;
        for (uint32_t q = b0; q < b1; q++) {
            while (k + 1 < n && qpos[k + 1] <= q)
                k++;
            const uint32_t r = lzw::resolve(qpos, qsrc, n, b0, q, k);
            if (r & lzw::kLit)
                v[q - b0] = (uint8_t)r;
            else if (r >= b0)
                return -2;
            else
                v[q - b0] = r >= flushed ? window[r & (kWindow - 1)] : plane[r];
        }
        for (uint32_t q = b0; q < b1; q++)
            window[q & (kWindow - 1)] = v[q - b0];
        b0 = b1;
        while (flushed + (uint32_t)kPiece <= b0) {
            for (uint32_t i = 0; i < (uint32_t)kPiece; i++)
                plane[flushed + i] = window[(flushed + i) & (kWindow - 1)];
            flushed += (uint32_t)kPiece;
        }
        ncodes += (uint64_t)n;
        nbatches++;
        if (ev == kEvEnd)
            break;
    }
    if (!err)
        for (uint32_t i = flushed; i < out_len; i++)
            plane[i] = window[i & (kWindow - 1)];
    if (stats) {
        stats[0] = ncodes;
        stats[1] = nbatches;
    }
    return err;
}

// tests/harness/tile_code_host.cpp -- TEST HARNESS, not product code.
//
// A scalar reference of the two GPU tile encoders, byte for byte:
//   * cn_deflate_fused_kernel (cn_deflate_fused.cuh): one parse of the tile of value records, every selected plane's
//     stream written from it, with the tuned code of tile_code.h or RFC 1951's fixed code;
//   * deflate_tiles_kernel (deflate_tiles.cuh): one parse per plane tile, fixed code.
// Both parse each tile row greedily with two distances -- 256 (the pixel above) and 1 (the run of the left pixel) --
// in ONE function here, parse_tile(); the token statistics (tools/token_stats.py) use it too.  The code itself comes
// from build_tile_code() (tile_code.h, host code); everything else is restated from the rules in DESIGN.md section 4.5,
// not taken from the .cuh files.  tests/stream_ref.py wraps it; built by the tests with g++ -shared, nothing under
// gcn10_b200/ links it.
#include <stdint.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../gcn10_b200/csrc/tile_code.h"

using namespace gcn10;

namespace {

constexpr int T = 256;
constexpr int kPad = 256;                        // record id of the padding right of / below the raster (fused)
constexpr uint32_t kStored = 2 + 2 * 5 + T * T + 4;
constexpr uint32_t kFusedStoredAt = 31 * 1024 - 64;    // fused: stored when the stream would pass this (step 6)
constexpr uint32_t kPlainStoredAt = 40 * 1024;          // deflate_tiles_kernel: kEncCap
constexpr uint32_t kFusedOutCap = 31 * 1024;            // shared-memory staging of one round of planes

struct Out {
    std::vector<uint8_t> bytes;
    uint64_t acc = 0;
    int nacc = 0;
    void put(uint32_t v, int n)
    {
        acc |= (uint64_t)(v & (n == 32 ? 0xFFFFFFFFu : ((1u << n) - 1u))) << nacc;
        nacc += n;
        while (nacc >= 8) {
            bytes.push_back((uint8_t)acc);
            acc >>= 8;
            nacc -= 8;
        }
    }
    void flush()                                 // zero bits up to the next byte
    {
        if (nacc)
            bytes.push_back((uint8_t)acc);
        acc = 0;
        nacc = 0;
    }
};

// length symbol index (0..28 = symbols 257..285), extra bit count and value of a match length 3..258
void len_sym(int len, int &idx, int &e, int &extra)
{
    e = 0;
    extra = 0;
    if (len == 258) {
        idx = 28;
        return;
    }
    const int l = len - 3;
    if (l < 8) {
        idx = l;
        return;
    }
    e = 29 - __builtin_clz((unsigned)l);
    idx = 4 + 4 * e + ((l - (4 << e)) >> e);
    extra = (l - (4 << e)) & ((1 << e) - 1);
}

// One token of the parse: a literal (len == 1) of pixel p, or a match of len 3..258 at distance 256 (above) or 1.
struct Tok {
    int p, len;
    bool above;
};

// The greedy parse of a 256 x 256 tile of ids (equal ids = equal bytes in every plane the stream is written for).
// Per row: at pixel x, la = pixels equal to the pixel above (from x on), lr = pixels equal to pixel x - 1; the longer
// wins, a tie goes to the pixel above; a match is at least 3 long and stops at the row's end, else pixel x is a literal.
// row_runs (the fused kernel): a run of n >= 2 rows that each repeat the row above is 256 n bytes at distance 256,
// coded as matches of 258 across the rows plus the rest; a rest of 1 or 2 is split 129 + (129 + rest).  A single
// repeated row stays an ordinary row (one match of 256).
template <class F>
void parse_tile(const uint16_t *t, bool row_runs, F &&tok)
{
    auto row_eq = [&](int r) { return memcmp(t + T * r, t + T * (r - 1), T * sizeof(uint16_t)) == 0; };
    int r = 0;
    while (r < T) {
        const uint16_t *row = t + T * r;
        if (row_runs && r > 0 && row_eq(r)) {
            int n = 1;
            while (r + n < T && row_eq(r + n))
                n++;
            if (n >= 2) {
                const unsigned span = (unsigned)T * (unsigned)n;
                unsigned q = span / 258u;
                const unsigned rest = span - 258u * q;
                int tail[2] = { (int)rest, 0 };
                if (rest == 1u || rest == 2u) {
                    q--;
                    tail[0] = 129;
                    tail[1] = 129 + (int)rest;
                }
                for (unsigned i = 0; i < q; i++)
                    tok(Tok{ T * r, 258, true });
                for (int k = 0; k < 2; k++)
                    if (tail[k])
                        tok(Tok{ T * r, tail[k], true });
                r += n;
                continue;
            }
        }
        int x = 0;
        while (x < T) {
            int la = 0, lr = 0;
            if (r > 0)
                while (x + la < T && row[x + la] == row[x + la - T])
                    la++;
            if (x > 0)
                while (x + lr < T && row[x + lr] == row[x - 1])
                    lr++;
            const bool above = la >= lr;
            const int len = above ? la : lr;
            if (len >= 3) {
                tok(Tok{ T * r + x, len, above });
                x += len;
            }
            else {
                tok(Tok{ T * r + x, 1, false });
                x++;
            }
        }
        r++;
    }
}

void put_tuned_match(Out &o, const TileCode &tc, int len, bool above)
{
    int idx, e, extra;
    len_sym(len, idx, e, extra);
    o.put(tc.len_code[idx], tc.len_bits[idx]);
    o.put((uint32_t)extra, e);
    if (above) {
        o.put(tc.dist_code[1], tc.dist_bits[1]);
        o.put(63u, 6);                          // distance symbol 15 = 193..256, extra 63
    }
    else
        o.put(tc.dist_code[0], tc.dist_bits[0]);
}

void put_tuned_lit(Out &o, const TileCode &tc, uint8_t v)
{
    o.put(tile_code_detail::reverse_bits(tc.lit_first + tc.lit_rank[v], tc.lit_bits), tc.lit_bits);
}

// RFC 1951 3.2.6
void put_fixed_match(Out &o, int len, bool above)
{
    int idx, e, extra;
    len_sym(len, idx, e, extra);
    const int code = 257 + idx;
    if (code <= 279)
        o.put(tile_code_detail::reverse_bits((uint32_t)(code - 256), 7), 7);
    else
        o.put(tile_code_detail::reverse_bits((uint32_t)(0xC0 + code - 280), 8), 8);
    o.put((uint32_t)extra, e);
    if (above) {
        o.put(tile_code_detail::reverse_bits(15, 5), 5);
        o.put(63u, 6);
    }
    else
        o.put(0u, 5);
}

void put_fixed_lit(Out &o, uint8_t v)
{
    if (v < 144)
        o.put(tile_code_detail::reverse_bits(0x30u + v, 8), 8);
    else
        o.put(tile_code_detail::reverse_bits(0x190u + (v - 144u), 9), 9);
}

uint32_t adler32(const uint8_t *tile)
{
    uint32_t s1 = 1, s2 = 0;
    for (int i = 0; i < T * T; i++) {
        s1 = (s1 + tile[i]) % 65521u;
        s2 = (s2 + s1) % 65521u;
    }
    return (s2 << 16) | s1;
}

void put_adler(std::vector<uint8_t> &b, uint32_t ad)
{
    b.push_back((uint8_t)(ad >> 24));
    b.push_back((uint8_t)(ad >> 16));
    b.push_back((uint8_t)(ad >> 8));
    b.push_back((uint8_t)ad);
}

// zlib header, two stored blocks of 32768 bytes, Adler-32
uint32_t write_stored(const uint8_t *tile, uint8_t *out)
{
    static const uint8_t h1[7] = { 0x78, 0x9C, 0x00, 0x00, 0x80, 0xFF, 0x7F }, h2[5] = { 0x01, 0x00, 0x80, 0xFF, 0x7F };
    memcpy(out, h1, 7);
    memcpy(out + 7, tile, 32768);
    memcpy(out + 7 + 32768, h2, 5);
    memcpy(out + 12 + 32768, tile + 32768, 32768);
    const uint32_t ad = adler32(tile);
    uint8_t *a = out + kStored - 4;
    a[0] = (uint8_t)(ad >> 24); a[1] = (uint8_t)(ad >> 16); a[2] = (uint8_t)(ad >> 8); a[3] = (uint8_t)ad;
    return kStored;
}

// the tuned code's stream of a tile of bytes (no padding record: the ids are the bytes)
uint32_t tuned_stream(const TileCode &tc, const uint16_t *ids, const uint8_t *tile, std::vector<uint8_t> &b)
{
    Out o;
    for (int i = 0; i < tc.header_bits; i++)
        o.put((tc.header_words[i >> 5] >> (i & 31)) & 1u, 1);
    parse_tile(ids, true, [&](const Tok &k) {
        if (k.len == 1)
            put_tuned_lit(o, tc, tile[k.p]);
        else
            put_tuned_match(o, tc, k.len, k.above);
    });
    o.put(tc.eob_code, tc.eob_bits);
    o.flush();
    put_adler(o.bytes, adler32(tile));
    b.swap(o.bytes);
    return (uint32_t)b.size();
}

struct FusedRef {
    bool tuned;
    TileCode tc;
    int nsel;
    uint8_t cls[18];
};

// The mode step 6 of cn_deflate_fused_kernel picks for a tile (cn_deflate_fused.cuh:868-916), from the token list of
// the id tile and the stream sizes:
//   mode[0] stored planes   mode[1] bit mask of them   mode[2] template + overlays (1) or per-plane streams (0)
//   mode[3] rounds of the 31 KB staging area   mode[4] writing pass on checkpoint pieces (1), on the items (0), or
//   -1 when it cannot be (fixed code)   mode[5] pieces (fine) or items   mode[6] 9-bit-literal classes (0 = tuned
//   code)   mode[7] MAXP
void fused_mode(const FusedRef &f, const uint16_t *ids, const std::vector<Tok> &toks, const uint32_t *sizes, int *mode)
{
    const int nsel = f.nsel;
    bool stored[18];
    int nst = 0, smask = 0;
    for (int k = 0; k < nsel; k++) {
        stored[k] = sizes[k] == kStored;
        if (stored[k]) {
            nst++;
            smask |= 1 << k;
        }
    }
    bool clsz = true;
    int ncls = 0;
    for (int k = 0; k < nsel; k++) {
        clsz = clsz && f.cls[k] == 0;
        ncls = std::max(ncls, f.cls[k] + 1);
    }
    // (step 6) template when every stream has the same bit positions, plane 0 is compressed and two fit
    const uint32_t r16 = (sizes[0] + 15u) & ~15u;
    const bool tmpl = clsz && !stored[0] && 2u * r16 <= kFusedOutCap;
    uint32_t used = tmpl ? r16 : 0u;
    int nr = 0;
    for (int k = 0; k < nsel; k++) {
        if (stored[k])
            continue;
        const uint32_t a16 = (sizes[k] + 15u) & ~15u;
        if (used + a16 > kFusedOutCap) {
            nr++;
            used = tmpl ? r16 : 0u;
        }
        used += a16;
    }
    nr++;
    // items (step 2): rows cut at pixels that differ from the pixel above and from the pixel to their left, found in
    // the 4-pixel words that repeat neither the word above nor the left pixel; >= 8 pixels apart, <= 11 per row, and
    // at most 256 cuts per tile (beyond that every row that has cuts keeps 256 / rows of them)
    uint64_t above[T], left[T];
    bool rep[T];
    for (int r = 0; r < T; r++) {
        const uint16_t *row = ids + T * r;
        above[r] = left[r] = 0;
        for (int j = 0; j < 64; j++) {
            bool a = r > 0, l = j > 0;
            for (int b = 0; b < 4; b++) {
                a = a && row[4 * j + b] == row[4 * j + b - T];
                l = l && row[4 * j + b] == row[4 * j - 1];
            }
            above[r] |= (uint64_t)a << j;
            left[r] |= (uint64_t)l << j;
        }
        rep[r] = r > 0 && above[r] == ~0ull;
    }
    std::vector<std::vector<int>> cuts(T);
    int sum = 0, rows = 0;
    for (int r = 0; r < T; r++) {
        const uint64_t nw = ~(above[r] | left[r]);
        if (rep[r] || __builtin_popcountll(nw) < 2)
            continue;
        const uint16_t *row = ids + T * r;
        int last = 0;
        for (int j = 0; j < 64 && cuts[r].size() < 11; j++)
            if ((nw >> j) & 1u)
                for (int b = 0; b < 4 && cuts[r].size() < 11; b++) {
                    const int x = 4 * j + b;
                    if (x == 0 || (r > 0 && row[x] == row[x - T]) || row[x] == row[x - 1])
                        continue;
                    if (x - last >= 8) {
                        cuts[r].push_back(x);
                        last = x;
                    }
                }
        sum += (int)cuts[r].size();
        rows += cuts[r].empty() ? 0 : 1;
    }
    if (sum > 256)
        for (int r = 0; r < T; r++)
            if (cuts[r].size() > (size_t)(256 / rows))
                cuts[r].resize(256 / rows);
    int items = 0;
    for (int r = 0; r < T; r++)
        items += 1 + (int)cuts[r].size();
    // pieces (fine mode, tuned code): a row run's first row is one piece, its other rows none; an item of n tokens
    // leaves a checkpoint after tokens 2, 4, 6 ... (not after its last); when seven are taken every other one is
    // dropped and the step doubles
    int pieces = 0;
    {
        std::vector<int> ntok(T * 12, 0);
        std::vector<bool> run_row(T, false), inside(T, false);
        for (int r = 1; r < T; r++)
            if (rep[r]) {
                if (rep[r - 1])
                    inside[r] = true;
                else if (r + 1 < T && rep[r + 1])
                    run_row[r] = true;
            }
        for (const Tok &k : toks) {
            const int r = k.p / T, x = k.p % T;
            if (run_row[r] || inside[r])
                continue;
            int it = 0;
            while (it < (int)cuts[r].size() && cuts[r][it] <= x)
                it++;
            ntok[r * 12 + it]++;
        }
        for (int r = 0; r < T; r++) {
            if (inside[r])
                continue;
            if (run_row[r]) {
                pieces++;
                continue;
            }
            for (size_t it = 0; it <= cuts[r].size(); it++) {
                const int n = ntok[r * 12 + it];
                int count = 0, step = 2, next = 2;
                for (int t = 1; t <= n; t++)
                    if (t == next && t < n) {
                        if (count == 7) {
                            count = 3;
                            step *= 2;
                        }
                        count++;
                        next = t + step;
                    }
                pieces += 1 + count;
            }
        }
    }
    const bool fine = f.tuned && clsz;
    mode[0] = nst;
    mode[1] = smask;
    mode[2] = tmpl;
    mode[3] = nr;
    mode[4] = fine ? (pieces <= 1024 ? 1 : 0) : -1;
    mode[5] = fine && pieces <= 1024 ? pieces : items;
    mode[6] = f.tuned ? 0 : ncls;
    mode[7] = nsel <= 9 ? 9 : 18;
}

}  // namespace

extern "C" int gcn10_test_tile_code(const uint8_t *present, int *lit_bits, int *header_bits, int *len284_bits, int *eob_bits)
{
    bool p[256];
    for (int v = 0; v < 256; v++)
        p[v] = present[v] != 0;
    TileCode tc;
    if (!build_tile_code(p, tc))
        return 1;
    *lit_bits = tc.lit_bits;
    *header_bits = tc.header_bits;
    *len284_bits = tc.len_bits[27];
    *eob_bits = tc.eob_bits;
    return 0;
}

// tile: 256 x 256 bytes whose values are all `present`, encoded with the tuned code and the fused kernel's parse
// (the bytes are the ids); returns the stream length (0 = no code / overflow)
extern "C" uint32_t gcn10_test_tile_encode(const uint8_t *present, const uint8_t *tile, uint8_t *out, uint32_t cap)
{
    bool p[256];
    for (int v = 0; v < 256; v++)
        p[v] = present[v] != 0;
    TileCode tc;
    if (!build_tile_code(p, tc))
        return 0;
    std::vector<uint16_t> ids(tile, tile + T * T);
    std::vector<uint8_t> b;
    tuned_stream(tc, ids.data(), tile, b);
    if (b.size() > cap)
        return 0;
    memcpy(out, b.data(), b.size());
    return (uint32_t)b.size();
}

// Token statistics of the fused kernel's parse of one 256 x 256 tile of record ids.  hist: [0] literals,
// [1] end-of-block, [2..30] length symbols 257..285, [31] extra length bits, [32] matches at distance 256, [33] at
// distance 1.  tools/token_stats.py turns these into the model table of build_tile_code().
extern "C" void gcn10_test_tile_tokens(const uint8_t *tile, uint64_t *hist)
{
    std::vector<uint16_t> ids(tile, tile + T * T);
    parse_tile(ids.data(), true, [&](const Tok &k) {
        if (k.len == 1) {
            hist[0]++;
            return;
        }
        int idx, e, extra;
        len_sym(k.len, idx, e, extra);
        hist[2 + idx]++;
        hist[31] += (uint64_t)e;
        hist[k.above ? 32 : 33]++;
    });
    hist[1]++;
}

// the code build_tile_code() designs for `present`: bits of the 29 length symbols, end-of-block, literals, header
extern "C" int gcn10_test_tile_code_lengths(const uint8_t *present, int *len_bits /*[29]*/, int *eob_bits, int *lit_bits,
                                            int *header_bits)
{
    bool p[256];
    for (int v = 0; v < 256; v++)
        p[v] = present[v] != 0;
    TileCode tc;
    if (!build_tile_code(p, tc))
        return 1;
    for (int i = 0; i < 29; i++)
        len_bits[i] = tc.len_bits[i];
    *eob_bits = tc.eob_bits;
    *lit_bits = tc.lit_bits;
    *header_bits = tc.header_bits;
    return 0;
}

// ---- the fused encoder's reference ----------------------------------------------------------------------------

// present: the byte values the planes can hold (the code is designed for them); tuned = 0: RFC 1951's fixed code.
// cls[j]: 9-bit-literal class of the j-th selected plane (fixed code).  Returns null when the tuned code is asked
// for and cannot be built.
extern "C" void *gcn10_ref_fused_new(const uint8_t *present, int tuned, int nsel, const uint8_t *cls)
{
    FusedRef *f = new FusedRef();
    f->tuned = tuned != 0;
    f->nsel = nsel;
    for (int j = 0; j < 18; j++)
        f->cls[j] = j < nsel ? cls[j] : 0;
    if (f->tuned) {
        bool p[256];
        for (int v = 0; v < 256; v++)
            p[v] = present[v] != 0;
        if (!build_tile_code(p, f->tc)) {
            delete f;
            return nullptr;
        }
    }
    return f;
}

extern "C" void gcn10_ref_fused_free(void *f) { delete (FusedRef *)f; }

// One tile position through the fused encoder.  planes[j]: pixel (0, 0) of the tile in the j-th selected plane, rows
// `pitch` bytes apart; vw x vh pixels of it lie in the raster, the rest is padding -- zero bytes in every plane, and
// a record of its own in the parse (equal to no raster pixel, even one whose values are all zero).  Two raster
// pixels are the same record when they are equal in every selected plane.  out: nsel x 65552 bytes, the j-th stream
// at j * 65552; sizes[j] its length; mode[8]: see fused_mode().  Returns the number of tokens.
extern "C" int gcn10_ref_fused_tile(const void *handle, const uint8_t *const *planes, int64_t pitch, int vw, int vh,
                                    uint8_t *out, uint32_t *sizes, int *mode)
{
    const FusedRef &f = *(const FusedRef *)handle;
    const int nsel = f.nsel;
    std::vector<uint16_t> ids(T * T, (uint16_t)kPad);
    std::vector<uint8_t> tiles((size_t)nsel * T * T, 0);
    std::map<std::string, uint16_t> recs;
    std::string key(nsel, '\0'), prev;
    int prev_id = -1;
    for (int y = 0; y < vh; y++)
        for (int x = 0; x < vw; x++) {
            for (int j = 0; j < nsel; j++) {
                const uint8_t v = planes[j][(int64_t)y * pitch + x];
                key[j] = (char)v;
                tiles[(size_t)j * T * T + T * y + x] = v;
            }
            if (prev_id < 0 || key != prev) {
                auto it = recs.emplace(key, (uint16_t)recs.size()).first;
                prev_id = it->second;
                prev = key;
            }
            ids[T * y + x] = (uint16_t)prev_id;
        }
    std::vector<Tok> toks;
    parse_tile(ids.data(), true, [&](const Tok &k) { toks.push_back(k); });
    for (int j = 0; j < nsel; j++) {
        const uint8_t *tile = tiles.data() + (size_t)j * T * T;
        Out o;
        if (f.tuned)
            for (int i = 0; i < f.tc.header_bits; i++)
                o.put((f.tc.header_words[i >> 5] >> (i & 31)) & 1u, 1);
        else {
            o.put(0x9C78u, 16);
            o.put(3u, 3);                       // BFINAL = 1, BTYPE = 01
        }
        for (const Tok &k : toks) {
            if (k.len == 1) {
                if (f.tuned)
                    put_tuned_lit(o, f.tc, tile[k.p]);
                else
                    put_fixed_lit(o, tile[k.p]);
            }
            else if (f.tuned)
                put_tuned_match(o, f.tc, k.len, k.above);
            else
                put_fixed_match(o, k.len, k.above);
        }
        if (f.tuned)
            o.put(f.tc.eob_code, f.tc.eob_bits);
        else
            o.put(0u, 7);
        o.flush();
        uint8_t *dst = out + (size_t)j * kStored;
        if (o.bytes.size() + 4 > kFusedStoredAt)
            sizes[j] = write_stored(tile, dst);
        else {
            put_adler(o.bytes, adler32(tile));
            memcpy(dst, o.bytes.data(), o.bytes.size());
            sizes[j] = (uint32_t)o.bytes.size();
        }
    }
    fused_mode(f, ids.data(), toks, sizes, mode);
    return (int)toks.size();
}

// One plane tile through deflate_tiles_kernel: the same row parse on the plane's bytes (zero padding is the byte 0),
// no row runs, fixed code; stored when the stream would pass 40 KB.  out: 65552 bytes.  Returns the stream length.
extern "C" uint32_t gcn10_ref_plain_tile(const uint8_t *plane, int64_t pitch, int vw, int vh, uint8_t *out)
{
    std::vector<uint8_t> tile(T * T, 0);
    for (int y = 0; y < vh; y++)
        memcpy(tile.data() + T * y, plane + (int64_t)y * pitch, (size_t)vw);
    std::vector<uint16_t> ids(tile.begin(), tile.end());
    Out o;
    o.put(0x9C78u, 16);
    o.put(3u, 3);
    parse_tile(ids.data(), false, [&](const Tok &k) {
        if (k.len == 1)
            put_fixed_lit(o, tile[k.p]);
        else
            put_fixed_match(o, k.len, k.above);
    });
    o.put(0u, 7);
    o.flush();
    if (o.bytes.size() + 4 > kPlainStoredAt)
        return write_stored(tile.data(), out);
    put_adler(o.bytes, adler32(tile.data()));
    memcpy(out, o.bytes.data(), o.bytes.size());
    return (uint32_t)o.bytes.size();
}

// What-if model (tools/token_stats.py, DESIGN.md "Next"): the same two distances, but the greedy parse runs over the
// tile as ONE stream of 65536 bytes, so a match may run on from the end of a row into the next one (the kernel's
// matches stop at row ends; only whole repeated rows are chained).  Same histogram layout as gcn10_test_tile_tokens.
extern "C" void gcn10_test_tile_tokens_stream(const uint8_t *t, uint64_t *hist, int run_on_tie)
{
    const int n = 65536;
    int p = 0;
    while (p < n) {
        int la = 0, lr = 0;
        if (p >= 256)
            while (p + la < n && la < 258 && t[p + la] == t[p + la - 256])
                la++;
        if (p >= 1)
            while (p + lr < n && lr < 258 && t[p + lr] == t[p + lr - 1])
                lr++;
        const bool above = run_on_tie ? la > lr : la >= lr;
        const int len = above ? la : lr;
        if (len >= 3) {
            int idx, e, extra;
            len_sym(len, idx, e, extra);
            hist[2 + idx]++;
            hist[31] += (uint64_t)e;
            hist[above ? 32 : 33]++;
            p += len;
        }
        else {
            hist[0]++;
            p++;
        }
    }
    hist[1]++;
}

// gcn10_b200/csrc/cn_deflate_fused.cuh -- Curve Number + tile DEFLATE in one kernel (sm_100a).
//
// process_block() of the reference ends every raster with save_raster() (/root/reference/src/cn.c:363 ->
// raster.c:192-227: tiled DEFLATE GeoTIFF).  When the caller wants the compressed tiles and not the raw
// planes, writing 9..18 planes to HBM (cn_block_kernel) and reading them back (deflate_tiles_kernel, one CTA
// per tile per plane, two greedy parses each) is wasted work: all planes of a block are the SAME picture
// seen through different lookup tables.  A pixel's Curve Numbers in every plane are a function of its
// (land cover, soil code) pair (cn.c:88-131), so the host numbers the distinct value records (at most 256,
// 61 with the shipped tables) and this kernel works on the tile of record ids:
//
//   1. one CTA per 256 x 256 tile position: land cover (16-byte loads) + nearest-neighbour soil code
//      (fp64 index maps of cn.c:219-229, precomputed) -> record id per pixel, in shared memory;
//   2. ONE LZ77 parse of the id tile (distances 256 = pixel above and 1 = run, as deflate_tiles.cuh): equal
//      ids are equal bytes in every plane, so the token structure is valid for all planes at once;
//   3. per plane only the literal bytes differ (and, through the 8/9-bit fixed-Huffman literal codes, the
//      bit positions): a block scan of per-item (common bits, per-plane 9-bit-literal counts) places every
//      item in every plane's stream; the second parse writes all planes' streams in one go;
//   4. Adler-32 of every plane from per-id pixel counts and position-weight sums (run based).
//
// The parse of a row is serial, so how the rows are dealt out to the 256 threads decides the kernel's time.  Any
// token boundary of the greedy parse is a free place to cut (the parse has no state): rows are cut into items at
// pixels that no match can cross (step 2 of the kernel), and the sizing pass leaves checkpoints from which the
// writing pass runs on pieces of a few tokens each (FusedCkpt).  Neither changes a bit of the streams.
//
// HBM traffic per pixel: 1 byte read + the compressed bytes (~0.2) instead of 1 + 2 * 9.  The planes are
// never materialised.  The id parse cannot see matches between different records that happen to share a value in
// one plane, so a plane's stream can be a few bytes longer than deflate_tiles_kernel's for the same plane.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "deflate_tiles.cuh"

namespace gcn10 {

constexpr int kFusedOutCap = 31 * 1024;         // shared-memory staging for the streams of one round of planes
constexpr int kFusedIds = 256;
constexpr int kFusedPad = 255;                  // record id of the zero padding right / below the raster
constexpr int kFusedClasses = 3;                // distinct "which records need a 9-bit literal" patterns over the planes
#ifndef GCN10_FUSED_SPLIT_EST
#define GCN10_FUSED_SPLIT_EST 2
#endif
#ifndef GCN10_FUSED_CKPT_STEP
#define GCN10_FUSED_CKPT_STEP 2
#endif
#ifndef GCN10_FUSED_MIN_PIECE
#define GCN10_FUSED_MIN_PIECE 8
#endif
constexpr int kFusedSplitEst = GCN10_FUSED_SPLIT_EST;   // rows with at least this many "new" words are cut into items
constexpr int kFusedMinPiece = GCN10_FUSED_MIN_PIECE;   // ... of at least this many pixels
constexpr int kFusedMaxCuts = 11;               // per row (the row's spare bytes hold them)
constexpr int kFusedMaxItems = 512;             // two items per thread at most
constexpr int kFusedMaxExtra = kFusedMaxItems - kTile;  // items beyond one per row
constexpr int kFusedRowMeta = kTile;            // byte offset of a row's 16 spare bytes inside its 272-byte tile row:
                                                // u16 first item slot, u16 run length, u8 cuts, u8[11] cut pixels

template <int MAXP>
constexpr int fused_smem_bytes()
{
    // id tile | stream staging (+64) | value table (16 or 32 bytes per id) | row masks
    return kTile * kTileStride + kFusedOutCap + 64 + kFusedIds * (MAXP <= 9 ? 16 : 32) + kTile * 16;
}

// The Huffman code of the streams: the tuned code of tile_code.h (one dynamic block per tile, every literal
// lit_bits long), or RFC 1951's fixed code when header_bits == 0.
struct FusedCode {
    int header_bits;                // bits in front of the first token: zlib header + block header
    int lit_bits;
    uint32_t lit_first;             // literal v has the code word lit_first + lit_rank[v] (MSB first)
    uint16_t len_code[29];          // length symbols 257..285, bit-reversed
    uint8_t len_bits[29];
    uint16_t eob_code;
    uint8_t eob_bits;
    uint16_t dist_code[2];          // distance 1 / distance 256 (symbol 15, followed by 6 extra bits = 63)
    uint8_t dist_bits[2];
    const uint32_t *header_words;   // device: the header_bits bits, LSB first
    const uint8_t *lit_rank;        // device [256]
};

struct FusedParams {
    const uint8_t *esa;             // device land cover, row 0 = block row y_base
    size_t esa_pitch;
    int w, rows;                    // raster width, rows in this launch
    int y_base;
    const int32_t *col_idx;         // [roundup16(w)]
    const int32_t *row_idx;         // [block rows]
    const uint8_t *hsg;
    size_t hsg_pitch;
    const uint8_t *idmap;           // [16][256]: (soil class, land cover) -> record id
    const uint8_t *val;             // [256][16 or 32]: record id -> value in the j-th selected plane
    const unsigned long long *lit9; // [256]: 21-bit field c = 1 when the record needs a 9-bit literal in planes of class c
    uint8_t cls[18];                // 9-bit-literal class of the j-th selected plane (fixed code only)
    FusedCode code;
    int nsel;                       // selected planes (1..18)
    int tiles_x, tile_rows;
    uint8_t *blob;
    unsigned long long *cursor;
    unsigned long long *offsets;    // [nsel][tile_rows][tiles_x]
    uint32_t *sizes;
    unsigned long long *id_hist;    // [256] option "stats": raster pixels per record id, summed over the tiles (null = off)
};

// soil class of a raw HYSOGs byte: 0 = code 0, 1..4 = A..D, 5..8 = A/D..D/D (11..14), 9 = anything else
__device__ __forceinline__ uint32_t soil_class(uint32_t code)
{
    if (code <= 4u)
        return code;
    const uint32_t d = code - 11u;
    return d <= 3u ? 5u + d : 9u;
}

// all bits of a match token in the tuned code (<= 27 bits), LSB first
__device__ __forceinline__ void tuned_match_code(const FusedCode &c, int len, bool above, uint32_t &bits, int &n)
{
    int idx, e = 0, extra = 0;
    const int l = len - 3;
    if (len == 258)
        idx = 28;                               // symbol 285: only the row-run tokens are this long
    else if (l < 8)
        idx = l;
    else {
        e = 29 - __clz(l);
        idx = 4 + 4 * e + ((l - (4 << e)) >> e);
        extra = (l - (4 << e)) & ((1 << e) - 1);
    }
    int nb = c.len_bits[idx];
    uint32_t v = (uint32_t)c.len_code[idx] | ((uint32_t)extra << nb);
    nb += e;
    if (above) {
        v |= ((uint32_t)c.dist_code[1] | (63u << c.dist_bits[1])) << nb;
        nb += c.dist_bits[1] + 6;
    }
    else {
        v |= (uint32_t)c.dist_code[0] << nb;
        nb += c.dist_bits[0];
    }
    bits = v;
    n = nb;
}

__device__ __forceinline__ uint32_t field21(unsigned long long c, uint32_t f) { return (uint32_t)(c >> (21u * f)) & 0x1FFFFFu; }

// One match token into the streams of planes [lo, hi).  TMPL: all streams share positions AND bits, the token
// goes into the template stream once.  ONE: shared positions, one store per plane.  Otherwise every plane has the
// position of its literal class.  `at` = header bits + bits common to all planes in front of the token.
template <int MAXP, bool ONE, bool TMPL>
__device__ __forceinline__ void fused_emit_match(uint32_t *out, const uint32_t *obase, int lo, int hi,
                                                 unsigned long long clsbits, unsigned long long lit, uint32_t at,
                                                 uint32_t bits, int n)
{
    if (ONE && TMPL) {
        const uint32_t pp = at + (uint32_t)lit;
        const uint32_t sh = pp & 31u;
        uint32_t *o = out + (pp >> 5);
        atomicOr(o, bits << sh);
        if (sh + (uint32_t)n > 32u)
            atomicOr(o + 1, bits >> (32u - sh));
    }
    else if (ONE) {
        const uint32_t pp = at + (uint32_t)lit;
        const uint32_t sh = pp & 31u, w0 = bits << sh, w1 = sh ? bits >> (32u - sh) : 0u;
        const bool cross = sh + (uint32_t)n > 32u;
#pragma unroll
        for (int k = 0; k < MAXP; k++)
            if (k >= lo && k < hi) {
                uint32_t *o = out + (obase[k] >> 2) + (pp >> 5);
                atomicOr(o, w0);
                if (cross)
                    atomicOr(o + 1, w1);
            }
    }
    else {
        const uint32_t pc[3] = { at + field21(lit, 0), at + field21(lit, 1), at + field21(lit, 2) };
#pragma unroll
        for (int k = 0; k < MAXP; k++)
            if (k >= lo && k < hi) {
                const uint32_t c = (uint32_t)(clsbits >> (2 * k)) & 3u;
                put_bits(out + (obase[k] >> 2), c == 0u ? pc[0] : (c == 1u ? pc[1] : pc[2]), bits, n);
            }
    }
}

// A run of `nrows` >= 2 tile rows that all repeat the row above them: 256 * nrows bytes equal to the bytes 256
// back, coded as matches of length 258 (the longest DEFLATE has; they run across the tile rows) plus the rest.
template <bool WRITE, int MAXP, bool ONE, bool TMPL>
__device__ __forceinline__ uint32_t fused_row_run(int nrows, unsigned long long clsbits, unsigned long long lit,
                                                  uint32_t pos, uint32_t *out, const uint32_t *obase, int lo, int hi,
                                                  const FusedCode &code)
{
    const bool tuned = code.header_bits != 0;
    const uint32_t hdr = tuned ? (uint32_t)code.header_bits : 19u;
    const uint32_t span = (uint32_t)kTile * (uint32_t)nrows;
    uint32_t q = span / 258u, rest = span - 258u * q;
    int tail[2] = { (int)rest, 0 };
    if (rest == 1u || rest == 2u) {             // a match is at least 3 long: split 258 + rest in two
        q -= 1u;
        tail[0] = 129;
        tail[1] = 129 + (int)rest;
    }
    uint32_t bits;
    int n;
    if (tuned)
        tuned_match_code(code, 258, true, bits, n);
    else
        match_code(258, true, bits, n);
    if (WRITE) {
        for (uint32_t i = 0; i < q; i++)
            fused_emit_match<MAXP, ONE, TMPL>(out, obase, lo, hi, clsbits, lit, hdr + pos + i * (uint32_t)n, bits, n);
    }
    pos += q * (uint32_t)n;
#pragma unroll
    for (int t = 0; t < 2; t++)
        if (tail[t]) {
            if (tuned)
                tuned_match_code(code, tail[t], true, bits, n);
            else
                match_code(tail[t], true, bits, n);
            if (WRITE)
                fused_emit_match<MAXP, ONE, TMPL>(out, obase, lo, hi, clsbits, lit, hdr + pos, bits, n);
            pos += (uint32_t)n;
        }
    return pos;
}

// Checkpoints of the sizing pass.  The parse of an item is serial and the items are far from equal (a tile has some
// 750 tokens in 130 items, the longest has 17), so the pass that writes the streams -- the expensive one -- does not
// run on the items: the sizing pass notes, every `step` tokens, where the parse stands (pixel, bits so far), and the
// writing pass runs on the pieces between the notes, a few tokens each, dealt out evenly to the 256 threads.  A token
// boundary is a free place to cut: the greedy parse has no state, it goes on from there exactly as it would have.
// An item has room for kFusedCkpt notes; when they are used up every other one is dropped and the step doubles.
constexpr int kFusedCkpt = 7;
constexpr int kFusedCkptStep = GCN10_FUSED_CKPT_STEP;
constexpr int kFusedMaxSubs = 1024;             // pieces a tile may have (four per thread); more: the items are written

struct FusedCkpt {
    uint32_t *note;                             // [kFusedCkpt]: pixel | bits << 8
    uint32_t count, step, next, ntok;
};

// Greedy parse of pixels [xa, xb) of one row of the id tile (a whole row, or one 64-pixel item of a long row).
//   WRITE = false: returns the bits common to all planes; lit += 9-bit-literal counts per class
//   WRITE = true : emits planes [lo, hi) ; `pos` = common bits before this item, lit = class counts before
//                  it, obase[k] = byte offset of plane k's stream in `out` (16-byte aligned); the 19 header
//                  bits are added here.
//   CKPT  (sizing pass, pos = 0): notes the state of the parse in *ck as described above
template <bool WRITE, int MAXP, bool ONE = false, bool TMPL = false, bool CKPT = false>
__device__ __forceinline__ uint32_t fused_parse_row(const uint8_t *tile, int r, const RowMasks &m, const uint8_t *val,
                                                    const unsigned long long *lit9, unsigned long long clsbits,
                                                    unsigned long long &lit, uint32_t pos, uint32_t *out,
                                                    const uint32_t *obase, int lo, int hi, int xa, int xb,
                                                    const FusedCode &code, const uint8_t *rank, FusedCkpt *ck = nullptr)
{
    constexpr int VALB = MAXP <= 9 ? 16 : 32;
    const bool tuned = code.header_bits != 0;
    const uint32_t hdr = tuned ? (uint32_t)code.header_bits : 19u;
    const uint8_t *row = tile + r * kTileStride;
    int x = xa;
    while (x < xb) {
        const int la = r > 0 ? run_len<true>(row, m.above, 0, x) : 0;
        int lr = 0;
        if (x > 0)
            lr = run_len<false>(row, m.left, bcast_byte(row[x - 1]), x);
        int len = la >= lr ? la : lr;
        len = min(len, xb - x);                 // tokens do not cross the end of the item
        if (len >= 3) {
            uint32_t bits;
            int n;
            if (tuned)
                tuned_match_code(code, len, la >= lr, bits, n);
            else
                match_code(len, la >= lr, bits, n);
            if (WRITE)
                fused_emit_match<MAXP, ONE, TMPL>(out, obase, lo, hi, clsbits, lit, hdr + pos, bits, n);
            pos += n;
            x += len;
        }
        else {
            const uint32_t id = row[x];
            if (WRITE) {
                uint32_t vw[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
                const uint4 v0 = *reinterpret_cast<const uint4 *>(val + VALB * id);
                vw[0] = v0.x; vw[1] = v0.y; vw[2] = v0.z; vw[3] = v0.w;
                if constexpr (VALB == 32) {
                    const uint4 v1 = *reinterpret_cast<const uint4 *>(val + VALB * id + 16);
                    vw[4] = v1.x; vw[5] = v1.y; vw[6] = v1.z; vw[7] = v1.w;
                }
                const uint32_t pc[3] = { hdr + pos + field21(lit, 0), hdr + pos + field21(lit, 1), hdr + pos + field21(lit, 2) };
                const uint32_t sh = pc[0] & 31u;
#pragma unroll
                for (int k = 0; k < MAXP; k++)
                    if (k >= lo && k < hi) {
                        uint32_t bits;
                        int n;
                        const uint32_t v = (vw[k >> 2] >> (8 * (k & 3))) & 255u;
                        if (tuned) {
                            n = code.lit_bits;
                            bits = __brev(code.lit_first + rank[v]) >> (32 - n);
                        }
                        else
                            lit_code(v, bits, n);
                        if (ONE) {
                            uint32_t *o = out + (obase[k] >> 2) + (pc[0] >> 5);
                            atomicOr(o, bits << sh);
                            if (sh + (uint32_t)n > 32u)
                                atomicOr(o + 1, bits >> (32u - sh));
                        }
                        else {
                            const uint32_t c = (uint32_t)(clsbits >> (2 * k)) & 3u;
                            put_bits(out + (obase[k] >> 2), c == 0u ? pc[0] : (c == 1u ? pc[1] : pc[2]), bits, n);
                        }
                    }
            }
            lit += __ldg(lit9 + id);
            pos += tuned ? (uint32_t)code.lit_bits : 8u;
            x += 1;
        }
        if (CKPT) {
            if (++ck->ntok == ck->next && x < xb) {
                if (ck->count == (uint32_t)kFusedCkpt) {
                    ck->note[0] = ck->note[1];
                    ck->note[1] = ck->note[3];
                    ck->note[2] = ck->note[5];
                    ck->count = 3;
                    ck->step *= 2u;
                }
                ck->note[ck->count++] = (uint32_t)x | (pos << 8);
                ck->next = ck->ntok + ck->step;
            }
        }
    }
    return pos;
}

// pixels [xa, xb) of item `piece` of tile row r (see step 2 of the kernel)
__device__ __forceinline__ void fused_item_range(const uint8_t *tile, int r, uint32_t piece, int &xa, int &xb)
{
    const uint8_t *meta = tile + r * kTileStride + kFusedRowMeta + 4;
    const uint32_t ncut = meta[0];
    xa = piece ? (int)meta[piece] : 0;
    xb = piece < ncut ? (int)meta[1u + piece] : kTile;
}

// grid = (tiles_x, tile_rows), 256 threads, fused_smem_bytes<MAXP>() of dynamic shared memory
template <int MAXP>
__global__ void __maxnreg__(120)
cn_deflate_fused_kernel(const __grid_constant__ FusedParams p)
{
    constexpr int VALB = MAXP <= 9 ? 16 : 32;
    extern __shared__ __align__(16) uint8_t smem_fz[];
    uint8_t *tile = smem_fz;                                            // record ids, row stride 272 (16 spare bytes per row)
    uint8_t *outb = smem_fz + kTile * kTileStride;                      // stream staging / early scratch
    uint32_t *out = reinterpret_cast<uint32_t *>(outb);
    uint8_t *s_val = outb + kFusedOutCap + 64;                          // [256][VALB]
    RowMasks *s_masks = reinterpret_cast<RowMasks *>(s_val + kFusedIds * VALB);     // [256]
    // early scratch inside the staging area (dead before the first stream bit is written)
    uint8_t *s_idmap = outb;                                            // 4 KB  [16][256]
    int32_t *s_col = reinterpret_cast<int32_t *>(outb + 4096);          // 1 KB
    uint32_t *s_cnt = reinterpret_cast<uint32_t *>(outb + 5120);        // 1 KB  pixels per id
    uint32_t *s_w = reinterpret_cast<uint32_t *>(outb + 6144);          // 1 KB  sum of (N - i) per id (< 2^32 over a tile)
    uint16_t *s_perm = reinterpret_cast<uint16_t *>(outb + 8192);       // 1 KB  items in processing order: row | piece << 8
    uint32_t *s_ibits = reinterpret_cast<uint32_t *>(outb + 10240);     // 2 KB  per item slot (stream order): common bits
    unsigned long long *s_ilit = reinterpret_cast<unsigned long long *>(outb + 12288);   // 4 KB  ... 9-bit-literal counts
    uint8_t *s_nsub = outb + 9216;                                      // 512 B per item slot: pieces of the writing pass
    uint32_t *s_note = reinterpret_cast<uint32_t *>(outb + 16384);      // 14 KB per item slot: kFusedCkpt checkpoints
    uint2 *s_desc = reinterpret_cast<uint2 *>(outb);                    // 8 KB  the pieces (once s_cnt / s_w are dead)

    __shared__ unsigned long long s_scan[kTile / 32][2];
    __shared__ uint32_t s_adler[18], s_nbytes[18], s_obase[18], s_stored[18];
    __shared__ unsigned long long s_goff[18];
    __shared__ int s_round_hi[19], s_nrounds, s_use_tmpl;
    __shared__ uint32_t s_total_common;
    __shared__ unsigned long long s_total_lit;
    __shared__ uint32_t s_hist[66];
    __shared__ uint8_t s_cls[18];
    __shared__ uint8_t s_rank[256];                                     // literal value -> code word offset (tuned code)
    const bool tuned = p.code.header_bits != 0;
    __shared__ uint32_t s_nitems, s_rep[kTile / 32];
    unsigned long long clsbits = 0;
#pragma unroll
    for (int k = 0; k < 18; k++)
        clsbits |= (unsigned long long)(p.cls[k] & 3u) << (2 * k);
    // one bit position for all streams (see step 6): the writing pass can then run on checkpointed pieces
    const bool fine = tuned && clsbits == 0ull;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = blockIdx.x, ty = blockIdx.y;
    const int x0 = tx * kTile, y0 = ty * kTile;
    const int nsel = p.nsel;

    // ---- tables -> shared memory
    for (int i = tid; i < 4096 / 16; i += kTile)
        reinterpret_cast<uint4 *>(s_idmap)[i] = __ldg(reinterpret_cast<const uint4 *>(p.idmap) + i);
    for (int i = tid; i < kFusedIds * VALB / 16; i += kTile)
        reinterpret_cast<uint4 *>(s_val)[i] = __ldg(reinterpret_cast<const uint4 *>(p.val) + i);
    {
        const int gx = min(x0 + tid, p.w - 1);
        s_col[tid] = __ldg(p.col_idx + gx);
        s_cnt[tid] = 0;
        s_w[tid] = 0;
        if (tid < 66)
            s_hist[tid] = 0;
        if (tid < 18)
            s_cls[tid] = p.cls[tid];
        s_rank[tid] = tuned ? __ldg(p.code.lit_rank + tid) : (uint8_t)0;
    }
    __syncthreads();

    // ---- 1. record ids of the tile (zero padding beyond the raster = id kFusedPad)
    {
        const int g = tid & 15;
        const bool vec_ok = ((reinterpret_cast<uintptr_t>(p.esa) | p.esa_pitch) & 15) == 0;
        const int gx = x0 + 16 * g;
        const int nvalid = max(0, min(16, p.w - gx));
        // the soil cells under this thread's 16 pixel columns (the same for all its rows): at 25 pixels per cell
        // there are one or two; ksw = pixels that lie in the first one
        const int c0 = s_col[16 * g], c1 = s_col[16 * g + 15];
        // (the column map is monotone: the pixels of the first cell are the leading ones)
        int ksw = 0, n1 = 0;
#pragma unroll
        for (int k4 = 0; k4 < 4; k4++) {
            const int4 cc = *reinterpret_cast<const int4 *>(s_col + 16 * g + 4 * k4);
            ksw += (cc.x == c0) + (cc.y == c0) + (cc.z == c0) + (cc.w == c0);
            n1 += (cc.x == c1) + (cc.y == c1) + (cc.z == c1) + (cc.w == c1);
        }
        const bool two = c0 == c1 || ksw + n1 == 16;
        if (c0 == c1)
            ksw = 16;
        const uint32_t s_idmap32 = (uint32_t)__cvta_generic_to_shared(s_idmap);
        const uint32_t pad4 = 0x01010101u * kFusedPad;
#pragma unroll 1
        for (int half = 0; half < 2; half++) {
            // all loads of eight rows are in flight before the first dependent use
            int hr[8];
            uint32_t code0[8], code1[8];
            uint4 ev[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int gy = y0 + (tid >> 4) + 16 * (8 * half + j);
                hr[j] = gy < p.rows ? __ldg(p.row_idx + p.y_base + gy) : 0;
            }
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int gy = y0 + (tid >> 4) + 16 * (8 * half + j);
                const uint8_t *hrow = p.hsg + (size_t)hr[j] * p.hsg_pitch;
                code0[j] = __ldg(hrow + c0);
                code1[j] = __ldg(hrow + c1);
                ev[j] = make_uint4(0, 0, 0, 0);
                if (gy < p.rows && nvalid == 16 && vec_ok)
                    ev[j] = __ldcs(reinterpret_cast<const uint4 *>(p.esa + (size_t)gy * p.esa_pitch + gx));
            }
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int r = (tid >> 4) + 16 * (8 * half + j);
                const int gy = y0 + r;
                uint32_t idw[4] = { pad4, pad4, pad4, pad4 };
                if (gy < p.rows && nvalid > 0) {
                    uint32_t ew[4] = { ev[j].x, ev[j].y, ev[j].z, ev[j].w };
                    if (!(nvalid == 16 && vec_ok)) {
                        const uint8_t *e = p.esa + (size_t)gy * p.esa_pitch + gx;
#pragma unroll
                        for (int k = 0; k < 16; k++)
                            if (k < nvalid)
                                ew[k >> 2] |= (uint32_t)e[k] << (8 * (k & 3));
                    }
                    if (two && nvalid == 16) {
                        // interior fast path: per pixel one PRMT (class byte), one select of the cell's map, one add and
                        // one LDS.U8; four ids are packed with three PRMTs
                        const uint32_t a0 = s_idmap32 + 256u * soil_class(code0[j]);
                        const uint32_t a1 = s_idmap32 + 256u * soil_class(code1[j]);
#pragma unroll
                        for (int k4 = 0; k4 < 4; k4++) {
                            uint32_t b[4];
#pragma unroll
                            for (int q = 0; q < 4; q++) {
                                const uint32_t lc = __byte_perm(ew[k4], 0, 0x4440 | q);
                                asm("ld.shared.u8 %0, [%1];" : "=r"(b[q]) : "r"((4 * k4 + q < ksw ? a0 : a1) + lc));
                            }
                            idw[k4] = __byte_perm(__byte_perm(b[0], b[1], 0x0040), __byte_perm(b[2], b[3], 0x0040), 0x5410);
                        }
                    }
                    else if (two) {
                        const uint8_t *m0 = s_idmap + 256u * soil_class(code0[j]);
                        const uint8_t *m1 = s_idmap + 256u * soil_class(code1[j]);
#pragma unroll
                        for (int k = 0; k < 16; k++) {
                            const uint32_t lc = (ew[k >> 2] >> (8 * (k & 3))) & 255u;
                            const uint32_t id = k < nvalid ? (uint32_t)(k < ksw ? m0 : m1)[lc] : (uint32_t)kFusedPad;
                            idw[k >> 2] = (k & 3) == 0 ? id : (idw[k >> 2] | (id << (8 * (k & 3))));
                        }
                    }
                    else {
                        // more than two soil cells under 16 pixels (soil grid finer than 16 pixels): cell by cell
                        const uint8_t *hrow = p.hsg + (size_t)hr[j] * p.hsg_pitch;
                        int prev = -1;
                        const uint8_t *mrow = s_idmap;
#pragma unroll
                        for (int k = 0; k < 16; k++) {
                            const int ci = s_col[16 * g + k];
                            if (ci != prev) {
                                mrow = s_idmap + 256u * soil_class(__ldg(hrow + ci));
                                prev = ci;
                            }
                            const uint32_t lc = (ew[k >> 2] >> (8 * (k & 3))) & 255u;
                            const uint32_t id = k < nvalid ? (uint32_t)mrow[lc] : (uint32_t)kFusedPad;
                            idw[k >> 2] = (k & 3) == 0 ? id : (idw[k >> 2] | (id << (8 * (k & 3))));
                        }
                    }
                }
                *reinterpret_cast<uint4 *>(tile + r * kTileStride + 16 * g) = make_uint4(idw[0], idw[1], idw[2], idw[3]);
            }
        }
    }
    __syncthreads();

    // ---- 2. (thread r owns tile row r) word masks, per-id pixel counts / position-weight sums, work estimate
    {
        RowMasks m;
        const uint4 *rowv = reinterpret_cast<const uint4 *>(tile + tid * kTileStride);
        const uint4 *upv = rowv - kTileStride / 16;
        // (a) the two word masks, branch free: bit j of `above` = word j equals the word above it, bit j of `left` =
        // word j is four copies of the last byte of word j - 1
        {
            uint32_t ab[2] = { 0, 0 }, lf[2] = { 0, 0 };
            uint32_t last = 0;
#pragma unroll
            for (int i = 0; i < kTile / 16; i++) {
                const uint4 cv = rowv[i];
                const uint4 uv = tid > 0 ? upv[i] : make_uint4(~cv.x, ~cv.y, ~cv.z, ~cv.w);
                const uint32_t cw[4] = { cv.x, cv.y, cv.z, cv.w };
                const uint32_t uw[4] = { uv.x, uv.y, uv.z, uv.w };
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int j = 4 * i + k;
                    ab[j >> 5] |= (uint32_t)(cw[k] == uw[k]) << (j & 31);
                    if (j > 0)
                        lf[j >> 5] |= (uint32_t)(cw[k] == last * 0x01010101u) << (j & 31);
                    last = cw[k] >> 24;
                }
            }
            m.above = (unsigned long long)ab[0] | ((unsigned long long)ab[1] << 32);
            m.left = (unsigned long long)lf[0] | ((unsigned long long)lf[1] << 32);
        }
        // (b) per-id pixel counts and position-weight sums of the row, run by run.  Words that continue a run (the
        // `left` bits) are skipped in one step; only the words in which something changes are looked at byte by byte,
        // so that the 32 rows a warp handles in lockstep loop a dozen times instead of 64.
        {
            const uint32_t *roww = reinterpret_cast<const uint32_t *>(tile + tid * kTileStride);
            const uint32_t rowbase = (uint32_t)(kTileBytes - kTile * tid);      // N - i at x = 0
            uint32_t cur = roww[0] & 255u, n = 0, xs = 0;
            int j = 0;
            while (j < kTile / 4) {
                if ((m.left >> j) & 1ull) {
                    // (bit 0 is never set, so j > 0 here) c words equal to four copies of `cur`
                    const uint32_t c = (uint32_t)min(ones_from(m.left, j), kTile / 4 - j);
                    n += 4u * c;
                    xs += 16u * (c * (uint32_t)j + c * (c - 1u) / 2u) + 6u * c;
                    j += (int)c;
                }
                if (j < kTile / 4) {
                    const uint32_t wv = roww[j];
#pragma unroll
                    for (int b = 0; b < 4; b++) {
                        const uint32_t v = (wv >> (8 * b)) & 255u;
                        if (v != cur) {
                            if (n) {
                                atomicAdd(&s_cnt[cur], n);
                                atomicAdd(&s_w[cur], n * rowbase - xs);
                            }
                            cur = v;
                            n = 0;
                            xs = 0;
                        }
                        n += 1;
                        xs += 4u * (uint32_t)j + b;
                    }
                    j++;
                }
            }
            atomicAdd(&s_cnt[cur], n);
            atomicAdd(&s_w[cur], n * rowbase - xs);
        }
        s_masks[tid] = m;
        // Work items.  A row's parse is serial, so the longest row sets the latency of the whole CTA: rows with
        // several "new" words (neither a repeat of the row above nor the continuation of a run -- typically the first
        // row of a soil cell) are cut into items.  The cuts cost nothing: they are made at pixels that differ both from
        // the pixel above and from the pixel to their left -- no match can run through such a pixel, so the greedy
        // parse has a token boundary there anyway and goes on from it exactly as it would have.  Items are sorted by
        // expected work so that the 32 items a warp parses in lockstep are alike.
        // Runs of rows that all repeat the row above them (the inside of a soil cell) become ONE item: the first row
        // of the run codes all of them as length-258 matches that run across the tile rows (fused_row_run), the
        // other rows of the run contribute nothing.
        const uint32_t est = (uint32_t)__popcll(~(m.above | m.left));
        const bool rep = tid > 0 && m.above == ~0ull;
        const unsigned repbal = __ballot_sync(0xffffffffu, rep);
        uint8_t *meta = tile + tid * kTileStride + kFusedRowMeta;
        uint32_t ncut = 0;
        if (!rep && est >= (uint32_t)kFusedSplitEst) {
            const uint32_t *roww = reinterpret_cast<const uint32_t *>(tile + tid * kTileStride);
            const uint32_t *upw = roww - kTileStride / 4;
            unsigned long long newm = ~(m.above | m.left);      // only these words can hold such a pixel
            uint32_t lastcut = 0;
            while (newm && ncut < (uint32_t)kFusedMaxCuts) {
                const int j = __ffsll((long long)newm) - 1;
                newm &= newm - 1ull;
                const uint32_t cw = roww[j];
                const uint32_t uw = tid > 0 ? upw[j] : ~cw;
                const uint32_t prev = j ? roww[j - 1] >> 24 : (~cw & 255u);
                uint32_t nat = __vcmpne4(cw, uw) & __vcmpne4(cw, (cw << 8) | prev);     // 0xFF per pixel that qualifies
                if (j == 0)
                    nat &= 0xFFFFFF00u;                         // pixel 0 starts the row
                while (nat && ncut < (uint32_t)kFusedMaxCuts) {
                    const uint32_t b = (uint32_t)(__ffs((int)nat) - 1) >> 3;
                    nat &= ~(0xFFu << (8u * b));
                    const uint32_t x = 4u * (uint32_t)j + b;
                    if (x - lastcut >= (uint32_t)kFusedMinPiece) {
                        meta[5u + ncut++] = (uint8_t)x;
                        lastcut = x;
                    }
                }
            }
        }
        // at most kFusedMaxExtra items beyond one per row: if the rows want more, every row keeps its share
        {
            uint32_t sum = ncut, rows = ncut ? 1u : 0u;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                sum += __shfl_xor_sync(0xffffffffu, sum, o);
                rows += __shfl_xor_sync(0xffffffffu, rows, o);
            }
            if (lane == 0) {
                s_scan[warp][1] = ((unsigned long long)rows << 32) | sum;
                s_rep[warp] = repbal;
            }
        }
        __syncthreads();
        {
            uint32_t sum = 0, rows = 0;
            for (int wv = 0; wv < kTile / 32; wv++) {
                sum += (uint32_t)s_scan[wv][1];
                rows += (uint32_t)(s_scan[wv][1] >> 32);
            }
            if (sum > (uint32_t)kFusedMaxExtra)
                ncut = min(ncut, (uint32_t)kFusedMaxExtra / rows);
        }
        meta[4] = (uint8_t)ncut;
        uint32_t runlen = 0;                    // 0: ordinary row; 0xFFFF: inside a run; else rows in the run it starts
        if (rep) {
            const bool prev = lane ? ((repbal >> (lane - 1)) & 1u) != 0u : (s_rep[warp - 1] >> 31) != 0u;
            if (prev)
                runlen = 0xFFFFu;
            else {
                uint32_t bits = repbal >> lane, avail = 32u - lane, total = 0;
                int wv = warp;
                for (;;) {
                    uint32_t ones = bits == 0xFFFFFFFFu ? 32u : (uint32_t)__ffs((int)~bits) - 1u;
                    ones = min(ones, avail);
                    total += ones;
                    if (ones < avail || ++wv == kTile / 32)
                        break;
                    bits = s_rep[wv];
                    avail = 32u;
                }
                runlen = total >= 2u ? total : 0u;      // a single repeated row stays an ordinary row (one token)
            }
        }
        *reinterpret_cast<uint16_t *>(tile + tid * kTileStride + kFusedRowMeta + 2) = (uint16_t)runlen;
        const uint32_t nseg = ncut + 1u;
        const uint32_t key = runlen == 0xFFFFu ? 0u : runlen ? min(64u, 1u + runlen / 8u) : (est + ncut) / nseg;
        atomicAdd(&s_hist[64u - key], nseg);
        uint32_t inc = nseg;                    // first item slot of every row (stream order)
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o)
                inc += t;
        }
        if (lane == 31)
            s_scan[warp][0] = inc;
        __syncthreads();
        if (warp == 0) {
            // exclusive prefix of the 65 buckets (longest items first)
            const uint32_t a = s_hist[lane], b = s_hist[32 + lane];
            uint32_t ia = a, ib = b;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
                if (lane >= o) {
                    ia += ta;
                    ib += tb;
                }
            }
            const uint32_t tot_a = __shfl_sync(0xffffffffu, ia, 31), tot_b = __shfl_sync(0xffffffffu, ib, 31);
            s_hist[lane] = ia - a;
            s_hist[32 + lane] = tot_a + ib - b;
            if (lane == 0)
                s_hist[64] = tot_a + tot_b;
        }
        uint32_t slot0 = inc - nseg;
        for (int wv = 0; wv < warp; wv++)
            slot0 += (uint32_t)s_scan[wv][0];
        *reinterpret_cast<uint16_t *>(tile + tid * kTileStride + kFusedRowMeta) = (uint16_t)slot0;
        if (tid == kTile - 1)
            s_nitems = slot0 + nseg;
        __syncthreads();
        const uint32_t at = atomicAdd(&s_hist[64u - key], nseg);
        for (uint32_t q = 0; q < nseg; q++)
            s_perm[at + q] = (uint16_t)(tid | (q << 8));
    }
    __syncthreads();
    // option "stats": s_cnt is final and stays intact until step 6 reuses it for s_desc.  Id kFusedPad is the padding
    // beyond the raster, never a raster pixel.
    if (p.id_hist && tid != kFusedPad && s_cnt[tid])
        atomicAdd(p.id_hist + tid, (unsigned long long)s_cnt[tid]);

    // ---- 3. pass 1: thread t parses items perm[t] and perm[t + 256]; (common bits, 9-bit-literal counts) -> item slot
    const uint32_t n_items = s_nitems;
    uint32_t item0 = tid < (int)n_items ? s_perm[tid] : 0xFFFFu;
    uint32_t item1 = tid + kTile < (int)n_items ? s_perm[tid + kTile] : 0xFFFFu;
    uint32_t slot_a = 0, slot_b = 0;
#pragma unroll 1
    for (int q = 0; q < 2; q++) {
        const uint32_t item = q ? item1 : item0;
        if (item == 0xFFFFu)
            break;
        const int r = item & 255u, piece = item >> 8;
        int xa, xb;
        fused_item_range(tile, r, (uint32_t)piece, xa, xb);
        const RowMasks pm = s_masks[r];
        const uint32_t rl = *reinterpret_cast<const uint16_t *>(tile + r * kTileStride + kFusedRowMeta + 2);
        const uint32_t slot = *reinterpret_cast<const uint16_t *>(tile + r * kTileStride + kFusedRowMeta) + (uint32_t)piece;
        unsigned long long lit = 0;
        uint32_t bits = 0, nsub = rl == 0xFFFFu ? 0u : 1u;
        if (rl != 0u) {
            if (rl != 0xFFFFu)
                bits = fused_row_run<false, MAXP, false, false>((int)rl, clsbits, lit, 0u, nullptr, nullptr, 0, 0, p.code);
        }
        else if (fine) {
            FusedCkpt ck = { s_note + slot * kFusedCkpt, 0u, (uint32_t)kFusedCkptStep, (uint32_t)kFusedCkptStep, 0u };
            bits = fused_parse_row<false, MAXP, false, false, true>(tile, r, pm, s_val, p.lit9, clsbits, lit, 0u, nullptr, nullptr,
                                                                    0, 0, xa, xb, p.code, s_rank, &ck);
            nsub += ck.count;
        }
        else
            bits = fused_parse_row<false, MAXP>(tile, r, pm, s_val, p.lit9, clsbits, lit, 0u, nullptr, nullptr, 0, 0, xa, xb,
                                                p.code, s_rank);
        s_ibits[slot] = bits;
        s_ilit[slot] = lit;
        s_nsub[slot] = (uint8_t)nsub;
        if (q)
            slot_b = slot;
        else
            slot_a = slot;
    }
    __syncthreads();

    // ---- 4. exclusive scan over the item slots (thread t: slots 2t, 2t+1), in place
    {
        const uint32_t i0 = 2u * tid, i1 = 2u * tid + 1u;
        const uint32_t b0 = i0 < n_items ? s_ibits[i0] : 0u, b1 = i1 < n_items ? s_ibits[i1] : 0u;
        // (fine: the second scan counts the pieces of the writing pass instead of 9-bit literals, which the tuned
        // code does not have)
        const unsigned long long l0 = i0 < n_items ? (fine ? (unsigned long long)s_nsub[i0] : s_ilit[i0]) : 0ull;
        const unsigned long long l1 = i1 < n_items ? (fine ? (unsigned long long)s_nsub[i1] : s_ilit[i1]) : 0ull;
        unsigned long long inc0 = (unsigned long long)b0 + b1, inc1 = l0 + l1;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t0 = __shfl_up_sync(0xffffffffu, inc0, o), t1 = __shfl_up_sync(0xffffffffu, inc1, o);
            if (lane >= o) {
                inc0 += t0;
                inc1 += t1;
            }
        }
        if (lane == 31) {
            s_scan[warp][0] = inc0;
            s_scan[warp][1] = inc1;
        }
        __syncthreads();
        unsigned long long e0 = inc0 - b0 - b1, e1 = inc1 - l0 - l1;
        for (int wv = 0; wv < warp; wv++) {
            e0 += s_scan[wv][0];
            e1 += s_scan[wv][1];
        }
        if (i0 < n_items) {
            s_ibits[i0] = (uint32_t)e0;
            s_ilit[i0] = e1;
        }
        if (i1 < n_items) {
            s_ibits[i1] = (uint32_t)e0 + b0;
            s_ilit[i1] = e1 + l0;
        }
        if (tid == kTile - 1) {
            s_total_common = (uint32_t)e0 + b0 + b1;
            s_total_lit = e1 + l0 + l1;
        }
    }
    __syncthreads();
    // the items' stream positions move into registers: the staging area is about to be reused
    const uint32_t pos_a = s_ibits[slot_a], pos_b = s_ibits[slot_b];
    const unsigned long long lit_a = fine ? 0ull : s_ilit[slot_a], lit_b = fine ? 0ull : s_ilit[slot_b];
    // fine: the pieces of this thread's items -> (row | first pixel << 8 | last pixel << 16, bit position), in stream
    // order at the index the scan gave them; every thread then takes pieces t, t + 256, ... (below, after step 5)
    const bool use_fine = fine && s_total_lit <= (unsigned long long)kFusedMaxSubs;
    uint32_t sub_a = 0, sub_b = 0;
    if (use_fine) {
        sub_a = (uint32_t)s_ilit[slot_a];
        sub_b = (uint32_t)s_ilit[slot_b];
    }

    // ---- 5. Adler-32 per plane: s1 = 1 + sum cnt[id] val[id], s2 = N + sum w[id] val[id]  (mod 65521)
    for (int k = warp; k < nsel; k += kTile / 32) {
        unsigned long long a = 0, b = 0;
        for (int id = lane; id < kFusedIds; id += 32) {
            const unsigned long long v = s_val[VALB * id + k];
            a += (unsigned long long)s_cnt[id] * v;
            b += (unsigned long long)(s_w[id] % 65521u) * v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            a += __shfl_down_sync(0xffffffffu, a, o);
            b += __shfl_down_sync(0xffffffffu, b, o);
        }
        if (lane == 0) {
            const uint32_t s1 = (uint32_t)((1ull + a) % 65521ull);
            const uint32_t s2 = (uint32_t)(((unsigned long long)kTileBytes + b) % 65521ull);
            s_adler[k] = (s2 << 16) | s1;
        }
    }
    __syncthreads();
    uint32_t pc0[4] = { 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu }, pc1[4] = { 0, 0, 0, 0 };
    if (use_fine) {
        // (s_cnt / s_w are dead now: the descriptors may take their place)
#pragma unroll 1
        for (int q = 0; q < 2; q++) {
            const uint32_t item = q ? item1 : item0;
            if (item == 0xFFFFu)
                break;
            const uint32_t r = item & 255u, piece = item >> 8;
            int xai, xbi;
            fused_item_range(tile, (int)r, piece, xai, xbi);
            const uint32_t xa = (uint32_t)xai, xb = (uint32_t)xbi;
            const uint32_t slot = q ? slot_b : slot_a, base = q ? pos_b : pos_a, n = s_nsub[slot];
            const uint32_t *note = s_note + slot * kFusedCkpt;
            uint2 *d = s_desc + (q ? sub_b : sub_a);
            uint32_t a = xa, at = base;
            for (uint32_t j = 0; j < n; j++) {
                const uint32_t nt = j + 1u < n ? note[j] : 0u;
                const uint32_t b = j + 1u < n ? (nt & 255u) : xb;
                d[j] = make_uint2(r | (a << 8) | ((b - 1u) << 16), at);
                a = b;
                at = base + (nt >> 8);
            }
        }
        __syncthreads();
        const uint32_t nsubs = (uint32_t)s_total_lit;
#pragma unroll
        for (int mth = 0; mth < 4; mth++) {
            const uint32_t g = (uint32_t)tid + (uint32_t)kTile * mth;
            if (g < nsubs) {
                const uint2 d = s_desc[g];
                pc0[mth] = d.x;
                pc1[mth] = d.y;
            }
        }
        __syncthreads();
    }

    // ---- 6. sizes, stored fallbacks, arena allocation, rounds
    if (tid == 0) {
        unsigned long long need = 0;
        for (int k = 0; k < nsel; k++) {
            const uint32_t bits = tuned ? (uint32_t)p.code.header_bits + s_total_common + p.code.eob_bits
                                        : 19u + s_total_common + field21(s_total_lit, s_cls[k]) + 7u;
            const uint32_t deflate_end = (bits + 7u) >> 3;
            s_stored[k] = deflate_end + 4u > (uint32_t)kFusedOutCap - 64u;
            s_nbytes[k] = s_stored[k] ? (uint32_t)kStoredBytes : deflate_end + 4u;
        }
        // compressed planes first (contiguous per round, in the arena as in the staging area), stored ones behind
        int nr = 0;
        uint32_t used = 0;
        // With one bit position for all streams (tuned code, or one literal class) the streams differ only in
        // their literal bits: the staging area then holds ONE template stream (header, matches, end of block) in
        // front of per-plane overlays (literals, Adler-32), OR-ed together on the way out.
        const uint32_t r16 = (s_nbytes[0] + 15u) & ~15u;
        const int use_tmpl = clsbits == 0ull && !s_stored[0] && 2u * r16 <= (uint32_t)kFusedOutCap;
        s_use_tmpl = use_tmpl;
        if (use_tmpl)
            used = r16;
        for (int k = 0; k < nsel; k++) {
            if (s_stored[k])
                continue;
            const uint32_t a16 = (s_nbytes[k] + 15u) & ~15u;
            if (used + a16 > (uint32_t)kFusedOutCap) {
                s_round_hi[nr++] = k;
                used = use_tmpl ? r16 : 0u;
            }
            s_obase[k] = used;
            s_goff[k] = need;
            used += a16;
            need += a16;
        }
        s_round_hi[nr++] = nsel;
        s_nrounds = nr;
        for (int k = 0; k < nsel; k++)
            if (s_stored[k]) {
                s_goff[k] = need;
                need += ((unsigned long long)kStoredBytes + 15ull) & ~15ull;
            }
        const unsigned long long off = atomicAdd(p.cursor, need);
        for (int k = 0; k < nsel; k++) {
            s_goff[k] += off;
            const size_t ti = ((size_t)k * p.tile_rows + ty) * p.tiles_x + tx;
            p.offsets[ti] = s_goff[k];
            p.sizes[ti] = s_nbytes[k];
        }
    }
    __syncthreads();

    // ---- 7. rounds of planes: zero the staging area, second parse writes the streams, copy out
    const int nrounds = s_nrounds;
    const bool use_tmpl = s_use_tmpl != 0;
    int lo = 0;
    for (int rd = 0; rd < nrounds; rd++) {
        const int hi = s_round_hi[rd];
        // planes of this round that are compressed: [lo, hi) minus the stored ones
        uint32_t span = 0;
        int first = -1;
        for (int k = lo; k < hi; k++)
            if (!s_stored[k]) {
                if (first < 0)
                    first = k;
                span = s_obase[k] + ((s_nbytes[k] + 15u) & ~15u);
            }
        if (first >= 0 && use_tmpl) {
            // ---- template + overlays (see step 6); no stored planes in this mode
            const uint32_t r16 = s_obase[lo];                           // = size of the template = of every overlay
            for (uint32_t i = tid; i < span / 16 + 4; i += kTile)
                reinterpret_cast<uint4 *>(outb)[i] = make_uint4(0, 0, 0, 0);
            __syncthreads();
            if (use_fine) {
                uint32_t d0 = pc0[0], d1 = pc0[1], d2 = pc0[2], d3 = pc0[3];
                uint32_t e0 = pc1[0], e1 = pc1[1], e2 = pc1[2], e3 = pc1[3];
#pragma unroll 1
                for (int mth = 0; mth < 4 && d0 != 0xFFFFFFFFu; mth++) {
                    const int r = d0 & 255u, xa = (d0 >> 8) & 255u, xb = (int)((d0 >> 16) & 255u) + 1;
                    const RowMasks pm = s_masks[r];
                    unsigned long long lw = 0ull;
                    const uint32_t rl = *reinterpret_cast<const uint16_t *>(tile + r * kTileStride + kFusedRowMeta + 2);
                    if (rl)
                        fused_row_run<true, MAXP, true, true>((int)rl, clsbits, lw, e0, out, s_obase, lo, hi, p.code);
                    else
                        fused_parse_row<true, MAXP, true, true>(tile, r, pm, s_val, p.lit9, clsbits, lw, e0, out, s_obase, lo, hi,
                                                                xa, xb, p.code, s_rank);
                    d0 = d1; d1 = d2; d2 = d3; d3 = 0xFFFFFFFFu;
                    e0 = e1; e1 = e2; e2 = e3;
                }
            }
            else {
#pragma unroll 1
                for (int q = 0; q < 2; q++) {
                    const uint32_t item = q ? item1 : item0;
                    if (item == 0xFFFFu)
                        break;
                    const int r = item & 255u, piece = item >> 8;
                    int xa, xb;
                    fused_item_range(tile, r, (uint32_t)piece, xa, xb);
                    const RowMasks pm = s_masks[r];
                    unsigned long long lw = q ? lit_b : lit_a;
                    const uint32_t rl = *reinterpret_cast<const uint16_t *>(tile + r * kTileStride + kFusedRowMeta + 2);
                    if (rl == 0xFFFFu)
                        continue;
                    if (rl)
                        fused_row_run<true, MAXP, true, true>((int)rl, clsbits, lw, q ? pos_b : pos_a, out, s_obase, lo, hi, p.code);
                    else
                        fused_parse_row<true, MAXP, true, true>(tile, r, pm, s_val, p.lit9, clsbits, lw, q ? pos_b : pos_a, out,
                                                                s_obase, lo, hi, xa, xb, p.code, s_rank);
                }
            }
            if (tuned) {
                for (int i = tid; i < (p.code.header_bits + 31) >> 5; i += kTile)
                    atomicOr(out + i, __ldg(p.code.header_words + i));
                if (tid == 0)
                    put_bits(out, (uint32_t)p.code.header_bits + s_total_common, p.code.eob_code, p.code.eob_bits);
            }
            else if (tid == 0) {
                put_bits(out, 0, 0x9C78u, 16);
                put_bits(out, 16, 0x3u, 3);
            }
            __syncthreads();            // (the Adler bytes may share a word with the last literal bits: atomics first)
            if (tid < hi - lo) {
                uint8_t *ob = outb + s_obase[lo + tid] + s_nbytes[lo + tid] - 4;        // bytes behind the stream's last bit
                const uint32_t ad = s_adler[lo + tid];
                ob[0] = (uint8_t)(ad >> 24);
                ob[1] = (uint8_t)(ad >> 16);
                ob[2] = (uint8_t)(ad >> 8);
                ob[3] = (uint8_t)ad;
            }
            __syncthreads();
            uint4 *dst = reinterpret_cast<uint4 *>(p.blob + s_goff[lo]);
            const uint4 *tm = reinterpret_cast<const uint4 *>(outb);
            const uint4 *ov = reinterpret_cast<const uint4 *>(outb + r16);
            const uint32_t per = r16 / 16, n16 = per * (uint32_t)(hi - lo);
            for (uint32_t i = tid; i < n16; i += kTile) {
                const uint4 a = ov[i], b = tm[i % per];
                dst[i] = make_uint4(a.x | b.x, a.y | b.y, a.z | b.z, a.w | b.w);
            }
            __syncthreads();
        }
        else if (first >= 0) {
            for (uint32_t i = tid; i < span / 16 + 4; i += kTile)
                reinterpret_cast<uint4 *>(outb)[i] = make_uint4(0, 0, 0, 0);
            __syncthreads();
            // stored planes must not be written: hand the parse ranges of compressed planes only
            int a = lo;
            while (a < hi) {
                while (a < hi && s_stored[a])
                    a++;
                int b = a;
                while (b < hi && !s_stored[b])
                    b++;
                if (a < b && use_fine) {
                    uint32_t d0 = pc0[0], d1 = pc0[1], d2 = pc0[2], d3 = pc0[3];
                    uint32_t e0 = pc1[0], e1 = pc1[1], e2 = pc1[2], e3 = pc1[3];
#pragma unroll 1
                    for (int mth = 0; mth < 4 && d0 != 0xFFFFFFFFu; mth++) {
                        const int r = d0 & 255u, xa = (d0 >> 8) & 255u, xb = (int)((d0 >> 16) & 255u) + 1;
                        const RowMasks pm = s_masks[r];
                        unsigned long long lw = 0ull;
                        const uint32_t rl = *reinterpret_cast<const uint16_t *>(tile + r * kTileStride + kFusedRowMeta + 2);
                        if (rl)
                            fused_row_run<true, MAXP, true, false>((int)rl, clsbits, lw, e0, out, s_obase, a, b, p.code);
                        else
                            fused_parse_row<true, MAXP, true>(tile, r, pm, s_val, p.lit9, clsbits, lw, e0, out, s_obase, a, b, xa, xb,
                                                              p.code, s_rank);
                        d0 = d1; d1 = d2; d2 = d3; d3 = 0xFFFFFFFFu;
                        e0 = e1; e1 = e2; e2 = e3;
                    }
                }
                else if (a < b) {
#pragma unroll 1
                    for (int q = 0; q < 2; q++) {
                        const uint32_t item = q ? item1 : item0;
                        if (item == 0xFFFFu)
                            break;
                        const int r = item & 255u, piece = item >> 8;
                        int xa, xb;
                fused_item_range(tile, r, (uint32_t)piece, xa, xb);
                        const RowMasks pm = s_masks[r];
                        unsigned long long lw = q ? lit_b : lit_a;
                        const uint32_t pw = q ? pos_b : pos_a;
                        const uint32_t rl = *reinterpret_cast<const uint16_t *>(tile + r * kTileStride + kFusedRowMeta + 2);
                        if (rl == 0xFFFFu)
                            continue;
                        if (rl) {
                            if (clsbits == 0ull)
                                fused_row_run<true, MAXP, true, false>((int)rl, clsbits, lw, pw, out, s_obase, a, b, p.code);
                            else
                                fused_row_run<true, MAXP, false, false>((int)rl, clsbits, lw, pw, out, s_obase, a, b, p.code);
                        }
                        else if (clsbits == 0ull)
                            fused_parse_row<true, MAXP, true>(tile, r, pm, s_val, p.lit9, clsbits, lw, pw, out, s_obase, a, b, xa, xb, p.code, s_rank);
                        else
                            fused_parse_row<true, MAXP, false>(tile, r, pm, s_val, p.lit9, clsbits, lw, pw, out, s_obase, a, b, xa, xb, p.code, s_rank);
                    }
                }
                a = b;
            }
            if (tuned) {
                // zlib header + dynamic block header (the same words for every stream), then the end-of-block code
                const int hw = (p.code.header_bits + 31) >> 5;
                for (int i = tid; i < hw * (hi - lo); i += kTile) {
                    const int k = lo + i / hw;
                    if (!s_stored[k])
                        atomicOr(out + (s_obase[k] >> 2) + i % hw, __ldg(p.code.header_words + i % hw));
                }
                if (tid < hi - lo && !s_stored[lo + tid])
                    put_bits(out + (s_obase[lo + tid] >> 2), (uint32_t)p.code.header_bits + s_total_common, p.code.eob_code,
                             p.code.eob_bits);
            }
            else if (tid < hi - lo && !s_stored[lo + tid]) {
                const int k = lo + tid;
                put_bits(out + (s_obase[k] >> 2), 0, 0x9C78u, 16);      // CMF = 0x78, FLG = 0x9C
                put_bits(out + (s_obase[k] >> 2), 16, 0x3u, 3);         // BFINAL = 1, BTYPE = 01 (fixed Huffman)
            }
            __syncthreads();
            if (tid < hi - lo && !s_stored[lo + tid]) {
                // (fixed code: end-of-block = seven zero bits, already there); Adler-32 big endian after the padding
                const int k = lo + tid;
                uint8_t *ob = outb + s_obase[k] + s_nbytes[k] - 4;
                const uint32_t ad = s_adler[k];
                ob[0] = (uint8_t)(ad >> 24);
                ob[1] = (uint8_t)(ad >> 16);
                ob[2] = (uint8_t)(ad >> 8);
                ob[3] = (uint8_t)ad;
            }
            __syncthreads();
            uint4 *dst = reinterpret_cast<uint4 *>(p.blob + s_goff[first]);
            const uint4 *so = reinterpret_cast<const uint4 *>(outb + s_obase[first]);
            const uint32_t n16 = (span - s_obase[first]) / 16;
            for (uint32_t i = tid; i < n16; i += kTile)
                dst[i] = so[i];
            __syncthreads();
        }
        lo = hi;
    }

    // ---- 8. incompressible planes: zlib header, two stored blocks of 32768 bytes, Adler-32
    for (int k = 0; k < nsel; k++) {
        if (!s_stored[k])
            continue;
        uint8_t *dst = p.blob + s_goff[k];
        if (tid == 0) {
            dst[0] = 0x78; dst[1] = 0x9C;
            dst[2] = 0x00; dst[3] = 0x00; dst[4] = 0x80; dst[5] = 0xFF; dst[6] = 0x7F;
            uint8_t *b2 = dst + 7 + 32768;
            b2[0] = 0x01; b2[1] = 0x00; b2[2] = 0x80; b2[3] = 0xFF; b2[4] = 0x7F;
            const uint32_t ad = s_adler[k];
            uint8_t *t4 = dst + kStoredBytes - 4;
            t4[0] = (uint8_t)(ad >> 24); t4[1] = (uint8_t)(ad >> 16); t4[2] = (uint8_t)(ad >> 8); t4[3] = (uint8_t)ad;
        }
        for (int i = tid; i < kTileBytes; i += kTile) {
            const int r = i >> 8, c = i & 255;
            const int o = i < 32768 ? 7 + i : 7 + 5 + i;
            dst[o] = s_val[VALB * tile[r * kTileStride + c] + k];
        }
    }
}

}  // namespace gcn10

// fmx_device.cuh — device-side view of the index and the rank primitives every kernel shares.
//
// Rank block (64 B = one aligned 2-sector fetch): word 0 = number of 1-bits before the block,
// words 1..15 = 480 payload bits (bit j of the block lives in word 1 + j/32, bit j%32).
// rank1(pos) therefore touches exactly one block: block = pos / 480, offset = pos % 480.
//
// Two layouts are built from those blocks (SURVEY.md Appendix B; DESIGN.md §3):
//   WM     : wavelet matrix over the dense symbol codes, `levels` = ceil(log2 sigma) bitvectors, one
//            block per level per rank (the structure north_star names);
//   PLANES : one bitvector per symbol, one block per rank — trades HBM capacity (sigma*n/7.5 bytes)
//            for 1/levels of the random fetches.
//   WMX    : multi-ary wavelet matrix, 16-ary (4-ary for <= 4 symbols) levels of 128-byte blocks: a 128-byte request costs what a
//            64-byte one does, so a byte alphabet needs 2 requests per rank instead of 8 at about the same size.
// The '$' row (eof) is not a symbol: WM stores it under code 0 and subtracts it back out, PLANES never
// sets it; rank of byte 0 is (pos > eof).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/fmgpu.h"

namespace fmx {

constexpr uint32_t kBitsPerBlock = 480;
constexpr int kCodeAbsent = 0xFF;

struct DevIndex {
    const uint4   *blocks;      // [levels | sigma][stride] rank blocks
    uint64_t       stride;      // blocks per level / plane
    const uint8_t *bwt;         // n bytes, eof -> 0
    const uint32_t *C;          // 257: C[c] = cf(c), C[256] = n
    const uint32_t *base;       // 256: PLANES: C[c] ; WM: C[c] - start_final[code[c]] (mod 2^32)
    const uint8_t *code;        // 256: byte -> dense code, kCodeAbsent if the byte does not occur
    const uint4   *mark;        // sampled-row marker bitvector (rank blocks) or nullptr
    const uint32_t *samples;    // sa value of the k-th marked row
    const uint4   *bm;          // locate walk blocks: 56 BWT bytes + their 56 mark bits per 64 B (row r -> block r/56), or nullptr
    uint32_t n, eof;
    int32_t  layout, levels;
    uint32_t z[8];              // WM: zeros per level
    // multi-ary wavelet matrix (FMX_LAYOUT_WMX): wmx_b = bits per digit (4: 16-ary, 2: 4-ary; 0 = another layout), wmx_levels = digits per code.  Level l is an array of 128-BYTE blocks = one request: 2^b cumulative counts
    // (occurrences of every digit value before the block) + the digits of (128 - 4*2^b)*8/b rows.  zx[l][v] = rows whose digit at level l is < v.
    int32_t  wmx_b, wmx_levels;
    uint64_t wmx_stride;        // blocks per level
    uint32_t zx[2][16];
    // ---- optional accelerators (bit-exact shortcuts that spend HBM capacity; DESIGN.md §3) ----
    const uint2   *kmer;        // sigma^kmer_k entries: (sp,ep) after the first kmer_k backward steps, (0,0) if empty — or, when kmer_rows > 0,
                                // the same bytes as 64-byte k-mer group blocks (see kmer_group below)
    int32_t        kmer_k;
    uint32_t       kmer_sigma;
    int32_t        kmer_rows;   // 0 = plain table (first consumed symbol most significant); > 0 = group blocks in lexicographic k-mer order
                                // carrying the J-hop half of the row contexts of up to this many of their first rows
    const uint32_t *sa;         // full suffix array  sa[row]   (bwtFm2sa, util.scala:213-224)
    const uint4    *isat;       // per text position p: { isa[p], 96 bits of T'[p..] } — inverse SA and the text behind it in one 16-B fetch
    int32_t         isat_bits;  // bits per text symbol in isat: ceil(log2(sigma+1)); stored value = dense code + 1, 0 = '$' / past the end
    int32_t         isat_syms;  // symbols per entry = 96 / isat_bits  (bytes: 12, sigma <= 31: 19, DNA: 32)
    // row-indexed context: ctx[r] = { isa[sa[r]-j] for the five hop lengths j in ctx_S (ascending, ctx_S[4] = ctx_J), 96 bits = the ctx_J symbols
    // T'[sa[r]-ctx_J .. sa[r]-1] in the isat packing } — 32 B, one request.  A row whose text goes on (backwards) with the next j pattern
    // bytes HOPS to row isa[sa[r]-j] — j backward steps in one fetch — and a small interval is advanced by looking at each of its rows
    // (the rows whose text continues with those j bytes map onto exactly the next interval, contiguously).  ctx_plan picks, for every
    // remaining length, the hop that reaches the pattern's start in the fewest fetches (any length is a sum of hop lengths: 1 is one).
    const uint4    *ctx;        // 2 x uint4 per row, or nullptr
    int32_t         ctx_J;      // = isat_syms
    int32_t         ctx_raw;    // 1 (byte alphabets, 8-bit symbols): the 12 symbols are the raw text bytes, so pattern words compare directly
    const uint8_t  *ctx_plan;   // 256 bytes: [rem] = index into ctx_S of the hop to take with rem <= 127 symbols left, [128 + rem] = fetches per row to finish
    uint8_t         ctx_S[8];   // hop lengths (5 used)
    // compact row contexts for alphabets of <= 4 symbols on texts too large for the 32-byte form (4e9 rows: 32 GB instead of 128):
    // ctx8[r] = { isa[sa[r]-J], the J = 16 symbols T'[sa[r]-16 .. sa[r]-1] as 2-bit dense codes } — a hop of exactly J symbols, usable while
    // at least J bytes remain; rows with fewer than J text positions before them hold row 0xFFFFFFFF
    const uint2    *ctx8;
    int32_t         ctx8_J;
    // dictionary of WIDE intervals (FMX_ACCEL_DICT): for every depth d in kmer_k+1 .. dict_D, every d-mer whose interval holds more than
    // dict_min_rows rows — the intervals rank steps are slowest on (sp and ep in different blocks) and row contexts cannot help.  A hash
    // table of 32-byte buckets = 2 entries { key: 64 bits, sp, ep }; key = the d dense codes (dict_bits each, first consumed symbol lowest)
    // | (d-1) << 60; 0 = empty slot.  Linear probing over buckets, built at <= half load.  A prefix of a wide d-mer is wide, so the deepest
    // stored prefix of a pattern is found by bisection over the depth: one request when the whole prefix is wide.
    // CHAIN entries carry the same idea past depth D, where the symbols no longer fit a key: the interval after D + (t-1) Jc + j symbols
    // (tier t = 1.., j = 1 .. Jc) is stored under { sp of the interval after D + (t-1) Jc symbols (which identifies it at that depth), j, t,
    // the j symbols } — bits 0-31 sp, 32-34 j-1, 35-37 t, 38.. the symbols; Jc = min(8, 22 / dict_bits); top four bits 0 (a depth tag is >= 1).
    const uint4    *dict;
    uint64_t        dict_buckets;   // multiple of 4
    int32_t         dict_D, dict_bits;
    int32_t         dict_Dx, dict_Jc;   // deepest depth stored at all (= dict_D without chain entries); symbols per chain tier
    // text samples (fmx_opts.text_sample_rate): tsamp[k] = row of the suffix at T' position k * tsamp_rate, k = 0 .. (n-1) / tsamp_rate —
    // where an extract walk starts; sym[code] = the byte of a dense code (decodes the packed symbols of isat / ctx / ctx8)
    const uint32_t *tsamp;
    uint32_t        tsamp_rate;     // 0 = no samples
    const uint8_t  *sym;
};

// Pattern accessors handed to search_pattern: operator()(i) = byte i; word(w) = bytes 4w..4w+3 packed little-endian (bytes at or
// beyond `len` read as anything — callers mask them).
struct SmemPattern {                                   // pattern staged in shared memory
    const uint8_t *p;
    int len;
    bool aligned;                                      // p is 4-byte aligned: words are single LDS.32
    __device__ __forceinline__ uint32_t operator()(int i) const { return p[i]; }
    __device__ __forceinline__ uint32_t word(int w) const {
        if (aligned) return reinterpret_cast<const uint32_t *>(p)[w];
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) { const int i = 4 * w + b; if (i < len) v |= (uint32_t)p[i] << (8 * b); }
        return v;
    }
    // pattern bytes o .. o+11 as three little-endian words (bytes at or beyond `len` read as anything; the staging buffer is padded)
    __device__ __forceinline__ void bytes12(int o, uint32_t &w0, uint32_t &w1, uint32_t &w2) const {
        if (aligned) {
            const uint32_t *q = reinterpret_cast<const uint32_t *>(p) + (o >> 2);
            const uint32_t a = q[0], b = q[1], c = q[2], s = (uint32_t)(o & 3) * 8u;
            if (s == 0) { w0 = a; w1 = b; w2 = c; }
            else { const uint32_t d = q[3]; w0 = __funnelshift_r(a, b, s); w1 = __funnelshift_r(b, c, s); w2 = __funnelshift_r(c, d, s); }
        } else {
            uint32_t v[3] = {0, 0, 0};
#pragma unroll
            for (int b = 0; b < 12; ++b) { const int i = o + b; if (i < len) v[b >> 2] |= (uint32_t)p[i] << (8 * (b & 3)); }
            w0 = v[0]; w1 = v[1]; w2 = v[2];
        }
    }
};
struct GlobalPattern {                                 // pattern read from global memory (variable-length batches)
    const uint8_t *p;
    int len;
    __device__ __forceinline__ uint32_t operator()(int i) const { return (uint32_t)__ldg(p + i); }
    __device__ __forceinline__ uint32_t word(int w) const {
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) { const int i = 4 * w + b; if (i < len) v |= (uint32_t)__ldg(p + i) << (8 * b); }
        return v;
    }
    __device__ __forceinline__ void bytes12(int o, uint32_t &w0, uint32_t &w1, uint32_t &w2) const {
        uint32_t v[3] = {0, 0, 0};
#pragma unroll
        for (int b = 0; b < 12; ++b) { const int i = o + b; if (i < len) v[b >> 2] |= (uint32_t)__ldg(p + i) << (8 * (b & 3)); }
        w0 = v[0]; w1 = v[1]; w2 = v[2];
    }
};

constexpr uint32_t kCtxMaxRows = 8;    // intervals up to this many rows are advanced through ctx instead of rank steps
constexpr int      kCtxHops = 5;       // hop lengths per 32-byte entry
constexpr int      kCtxPlanMax = 127;  // remaining lengths covered by ctx_plan; longer ones take the full-depth hop

struct SharedTables {
    uint32_t C[257];
    uint32_t base[256];
    uint8_t  code[256];
    uint8_t  plan[256];         // DevIndex::ctx_plan (only when row contexts exist)
    uint8_t  hops[8];           // DevIndex::ctx_S
};

__device__ __forceinline__ void load_tables(SharedTables &s, const DevIndex &ix) {
    for (int i = threadIdx.x; i < 257; i += blockDim.x) s.C[i] = ix.C[i];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) { s.base[i] = ix.base[i]; s.code[i] = ix.code[i]; }
    if (ix.ctx != nullptr) {
        for (int i = threadIdx.x; i < 256; i += blockDim.x) s.plan[i] = ix.ctx_plan[i];
        if (threadIdx.x < 8) s.hops[threadIdx.x] = ix.ctx_S[threadIdx.x];
    }
}

// Index fetches.  Measured on B200 (tools/ldhint_bench.cu, profiles/r01_ldhint_*): what bounds random access is the number of
// load REQUESTS (one per load instruction and 128-B line), ~46-47 G/s from 4 B up to 128 B per request, as long as the touched
// footprint stays inside the ~64 GB TLB reach; a load without a prefetch-size hint makes the L2 pull 128 B from DRAM per miss,
// `.L2::64B` pulls the 64 B that are used.  Hence: one request per fetched block (the 256-bit load moves 32 B per lane), 64-B hint.
__device__ __forceinline__ uint4 ldg128(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::64B.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
// sm_100 256-bit load: 32 aligned bytes in one request
__device__ __forceinline__ void ldg256(const uint4 *p, uint4 &a, uint4 &b) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::64B.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}
__device__ __forceinline__ uint32_t ldg32(const uint32_t *p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::64B.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg64(const uint2 *p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::64B.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}

// popcount of the bits of a 64-bit lane word that lie below virtual bit `v` of the block, where this
// word covers virtual bits [first, first+64).  Virtual bit 32+j is payload bit j (bits 0..31 = header).
__device__ __forceinline__ uint32_t popc_below64(uint64_t w, int v, int first) {
    int t = v - first;
    t = t < 0 ? 0 : (t > 64 ? 64 : t);
    uint64_t mask = (t >= 64) ? ~0ull : ((1ull << t) - 1ull);
    return __popcll(w & mask);
}

// One lane's share of a block: WORDS = 16/G consecutive 32-bit words starting at word lane*WORDS.
template <int G> struct LaneBlock { uint4 v[4 / G]; };

template <int G>
__device__ __forceinline__ LaneBlock<G> load_block(const uint4 *bv, uint32_t blk, int lane) {
    LaneBlock<G> r;
    const uint4 *p = bv + (uint64_t)blk * 4 + lane * (4 / G);
    if constexpr (G == 4) r.v[0] = ldg128(p);                                   // four lanes x 16 B: one request
    else if constexpr (G == 2) ldg256(p, r.v[0], r.v[1]);                         // two lanes x 32 B: one request
    else { ldg256(p, r.v[0], r.v[1]); ldg256(p + 2, r.v[2], r.v[3]); }            // one lane: two requests
    return r;
}

// lane-local part of rank: ones among payload bits [0, off) that this lane holds
template <int G>
__device__ __forceinline__ uint32_t lane_rank(const LaneBlock<G> &b, uint32_t off, int lane) {
    const int v = (int)off + 32;
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < 4 / G; ++i) {
        int first = (lane * (4 / G) + i) * 128;
        uint64_t lo = ((uint64_t)b.v[i].y << 32) | b.v[i].x;
        uint64_t hi = ((uint64_t)b.v[i].w << 32) | b.v[i].z;
        if (first == 0) lo &= ~0xFFFFFFFFull;                      // header word is not payload
        s += popc_below64(lo, v, first) + popc_below64(hi, v, first + 64);
    }
    return s;
}

template <int G> __device__ __forceinline__ uint32_t group_mask() {
    if (G == 1) return 0xFFFFFFFFu;          // unused
    const uint32_t lane = threadIdx.x & 31;
    return ((1u << G) - 1u) << (lane & ~(G - 1));
}

template <int G> __device__ __forceinline__ uint32_t group_sum(uint32_t x, uint32_t mask) {
    if (G >= 2) x += __shfl_xor_sync(mask, x, 1);
    if (G >= 4) x += __shfl_xor_sync(mask, x, 2);
    return x;
}

// rank1 at two positions of the same bitvector; one block fetch when they share a block.
// All G lanes of the group call this together (group-uniform control flow).  `touched` counts
// distinct blocks for the roofline accounting when STATS.
template <int G, bool STATS>
__device__ __forceinline__ void rank_pair(const uint4 *bv, uint32_t pa, uint32_t pb, uint32_t &ra, uint32_t &rb,
                                          uint32_t &touched) {
    const int lane = (G == 1) ? 0 : (threadIdx.x & (G - 1));
    const uint32_t mask = group_mask<G>();
    const uint32_t ba = pa / kBitsPerBlock, oa = pa - ba * kBitsPerBlock;
    const uint32_t bb = pb / kBitsPerBlock, ob = pb - bb * kBitsPerBlock;
    LaneBlock<G> A = load_block<G>(bv, ba, lane);
    LaneBlock<G> B = A;
    if (bb != ba) B = load_block<G>(bv, bb, lane);
    if (STATS) touched += (bb != ba) ? 2u : 1u;
    uint32_t ha = A.v[0].x, hb = B.v[0].x;
    uint32_t sa = lane_rank<G>(A, oa, lane), sb = lane_rank<G>(B, ob, lane);
    if (G > 1) {
        sa = group_sum<G>(sa, mask);
        sb = group_sum<G>(sb, mask);
        ha = __shfl_sync(mask, ha, 0, G);
        hb = __shfl_sync(mask, hb, 0, G);
    }
    ra = ha + sa;
    rb = hb + sb;
}

// single-position rank (+ optionally the bit at that position) — used by LF walks
template <int G>
__device__ __forceinline__ uint32_t rank_one(const uint4 *bv, uint32_t p, uint32_t *bit_out) {
    const int lane = (G == 1) ? 0 : (threadIdx.x & (G - 1));
    const uint32_t mask = group_mask<G>();
    const uint32_t b = p / kBitsPerBlock, o = p - b * kBitsPerBlock;
    LaneBlock<G> A = load_block<G>(bv, b, lane);
    uint32_t h = A.v[0].x, s = lane_rank<G>(A, o, lane);
    uint32_t bit = 0;
    if (bit_out) {
        const int w = 1 + (int)(o >> 5);                   // word holding payload bit o
#pragma unroll
        for (int i = 0; i < 4 / G; ++i) {
            const int rel = w - (lane * (4 / G) + i) * 4;  // position inside this lane's i-th uint4
            if (rel >= 0 && rel < 4) {
                const uint4 q = A.v[i];
                const uint32_t word = rel == 0 ? q.x : rel == 1 ? q.y : rel == 2 ? q.z : q.w;
                bit = (word >> (o & 31)) & 1u;
            }
        }
    }
    if (G > 1) {
        s = group_sum<G>(s, mask);
        h = __shfl_sync(mask, h, 0, G);
        if (bit_out) bit = group_sum<G>(bit, mask);
    }
    if (bit_out) *bit_out = bit;
    return h + s;
}

// BWT byte and sampled-row mark of row r from the fused walk blocks: one 64-B fetch per LF step instead of two
constexpr uint32_t kRowsPerWalkBlock = 56;
template <int G>
__device__ __forceinline__ void walk_block(const uint4 *bm, uint32_t r, uint32_t &c, uint32_t &marked) {
    const int lane = (G == 1) ? 0 : (threadIdx.x & (G - 1));
    const uint32_t mask = group_mask<G>();
    const uint32_t b = r / kRowsPerWalkBlock, o = r - b * kRowsPerWalkBlock;
    LaneBlock<G> A = load_block<G>(bm, b, lane);
    uint32_t cc = 0, mm = 0;
    const uint32_t mbyte = 56 + (o >> 3);                       // byte holding the mark bit
#pragma unroll
    for (int i = 0; i < 4 / G; ++i) {
        const uint32_t first = (uint32_t)(lane * (4 / G) + i) * 16u;   // first byte of this uint4 inside the block
        const uint4 q = A.v[i];
        if (o >= first && o < first + 16) {
            const uint32_t rel = o - first, w = (rel >> 2) == 0 ? q.x : (rel >> 2) == 1 ? q.y : (rel >> 2) == 2 ? q.z : q.w;
            cc = (w >> (8 * (rel & 3))) & 0xFFu;
        }
        if (mbyte >= first && mbyte < first + 16) {
            const uint32_t rel = mbyte - first, w = (rel >> 2) == 0 ? q.x : (rel >> 2) == 1 ? q.y : (rel >> 2) == 2 ? q.z : q.w;
            mm = (w >> (8 * (rel & 3) + (o & 7))) & 1u;
        }
    }
    if (G > 1) { cc = group_sum<G>(cc, mask); mm = group_sum<G>(mm, mask); }   // exactly one lane holds each
    c = cc;
    marked = mm;
}

// ---- multi-ary wavelet-matrix blocks (128 B = 32 words, one request from four lanes x 256 bits) -------------------------------------
// rows per block: b = 4: 16 count words + 16 payload words x 8 digits = 128 ; b = 2: 4 count words + 28 payload words x 16 digits = 448
__device__ __forceinline__ uint32_t wmx_rows_per_block(int b) { return b == 4 ? 128u : 448u; }

template <int G> struct LaneBlockX { uint4 v[8 / G]; };          // a lane's 32/G consecutive words of the block

template <int G>
__device__ __forceinline__ LaneBlockX<G> load_block_x(const uint4 *lv, uint32_t blk, int lane) {
    LaneBlockX<G> r;
    const uint4 *p = lv + (uint64_t)blk * 8 + lane * (8 / G);
#pragma unroll
    for (int i = 0; i < 8 / G; i += 2) ldg256(p + i, r.v[i], r.v[i + 1]);       // G = 4: one 256-bit load per lane = one request per block
    return r;
}

// lane-local part of rank_d(off): the count word of digit d if this lane holds it, plus matches among this lane's payload digits < off
template <int G>
__device__ __forceinline__ uint32_t lane_rank_x(const LaneBlockX<G> &blkv, uint32_t off, uint32_t d, int b, int lane) {
    const int H = 1 << b, per = 32 / b;                           // header words, digits per payload word
    const uint32_t rep = b == 4 ? 0x11111111u : 0x55555555u;
    const uint32_t pat = d * rep;
    uint32_t s = 0;
#pragma unroll
    for (int i = 0; i < 8 / G; ++i) {
        const uint32_t w4[4] = {blkv.v[i].x, blkv.v[i].y, blkv.v[i].z, blkv.v[i].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int wi = (lane * (8 / G) + i) * 4 + k;          // word index inside the block
            if (wi < H) { if ((uint32_t)wi == d) s += w4[k]; continue; }
            const int first = (wi - H) * per;                     // first row of this payload word
            int t = (int)off - first;
            if (t <= 0) continue;
            const uint32_t x = w4[k] ^ pat;
            const uint32_t nz = b == 4 ? ((x | (x >> 1) | (x >> 2) | (x >> 3)) & rep) : ((x | (x >> 1)) & rep);   // low bit of every non-matching digit
            uint32_t eq = ~nz & rep;
            if (t < per) eq &= (1u << (t * b)) - 1u;
            s += __popc(eq);
        }
    }
    return s;
}

// rank_d at two positions of one level; one block fetch when they share a block
template <int G, bool STATS>
__device__ __forceinline__ void rank_pair_x(const uint4 *lv, int b, uint32_t d, uint32_t pa, uint32_t pb, uint32_t &ra, uint32_t &rb, uint32_t &touched) {
    const int lane = (G == 1) ? 0 : (threadIdx.x & (G - 1));
    const uint32_t mask = group_mask<G>();
    const uint32_t R = wmx_rows_per_block(b);
    const uint32_t ba = pa / R, oa = pa - ba * R, bb = pb / R, ob = pb - bb * R;
    LaneBlockX<G> A = load_block_x<G>(lv, ba, lane);
    LaneBlockX<G> B = A;
    if (bb != ba) B = load_block_x<G>(lv, bb, lane);
    if (STATS) touched += (bb != ba) ? 2u : 1u;
    uint32_t sa = lane_rank_x<G>(A, oa, d, b, lane), sb = lane_rank_x<G>(B, ob, d, b, lane);
    if (G > 1) { sa = group_sum<G>(sa, mask); sb = group_sum<G>(sb, mask); }
    ra = sa; rb = sb;
}
template <int G>
__device__ __forceinline__ uint32_t rank_one_x(const uint4 *lv, int b, uint32_t d, uint32_t p) {
    const int lane = (G == 1) ? 0 : (threadIdx.x & (G - 1));
    const uint32_t R = wmx_rows_per_block(b);
    const uint32_t blk = p / R, o = p - blk * R;
    uint32_t s = lane_rank_x<G>(load_block_x<G>(lv, blk, lane), o, d, b, lane);
    if (G > 1) s = group_sum<G>(s, group_mask<G>());
    return s;
}

// ---- one backward step: (sp,ep) -> (C[c]+rank_c(sp), C[c]+rank_c(ep))   findex.scala:32-36 ------------
template <int G, int LAYOUT, bool STATS>
__device__ __forceinline__ void backward_step(const DevIndex &ix, const SharedTables &t, uint32_t c, uint32_t &sp,
                                              uint32_t &ep, uint32_t &touched) {
    const uint32_t code = t.code[c];
    if (c == 0) {                                   // '$': occurs once, at row eof; C[0] = 0
        sp = sp > ix.eof ? 1u : 0u;
        ep = ep > ix.eof ? 1u : 0u;
        return;
    }
    if (code == kCodeAbsent) { sp = ep = t.C[c]; return; }
    if (LAYOUT == FMX_LAYOUT_PLANES) {
        uint32_t ra, rb;
        rank_pair<G, STATS>(ix.blocks + (uint64_t)code * ix.stride * 4, sp, ep, ra, rb, touched);
        sp = t.base[c] + ra;
        ep = t.base[c] + rb;
    } else if (LAYOUT == FMX_LAYOUT_WMX) {         // multi-ary wavelet matrix: one 128-byte request per digit
        uint32_t p = sp, q = ep;
        const int b = ix.wmx_b, L = ix.wmx_levels;
        for (int l = 0; l < L; ++l) {
            const uint32_t d = (code >> (b * (L - 1 - l))) & ((1u << b) - 1u);
            uint32_t ra, rb;
            rank_pair_x<G, STATS>(ix.blocks + (uint64_t)l * ix.wmx_stride * 8, b, d, p, q, ra, rb, touched);
            p = ix.zx[l][d] + ra;
            q = ix.zx[l][d] + rb;
        }
        if (code == 0) { p -= (sp > ix.eof); q -= (ep > ix.eof); }     // the '$' row is filed under code 0
        sp = t.base[c] + p;
        ep = t.base[c] + q;
    } else {
        uint32_t p = sp, q = ep;
        const int L = ix.levels;
        for (int l = 0; l < L; ++l) {
            uint32_t ra, rb;
            rank_pair<G, STATS>(ix.blocks + (uint64_t)l * ix.stride * 4, p, q, ra, rb, touched);
            if ((code >> (L - 1 - l)) & 1u) { p = ix.z[l] + ra; q = ix.z[l] + rb; }
            else { p -= ra; q -= rb; }
        }
        if (code == 0) { p -= (sp > ix.eof); q -= (ep > ix.eof); }     // the '$' row is filed under code 0
        sp = t.base[c] + p;
        ep = t.base[c] + q;
    }
}

// ---- wide-interval dictionary probe ----------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t dict_mix(uint64_t x) {
    x ^= x >> 31; x *= 0x9E3779B97F4A7C15ull; x ^= x >> 29; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 32;
    return x;
}
__device__ __forceinline__ uint64_t dict_home(uint64_t key, uint64_t buckets) { return __umul64hi(dict_mix(key), buckets); }

// key of the first d consumed symbols: their dense codes, `bits` each, the first one lowest, | (d-1) << 60
__device__ __forceinline__ uint64_t dict_key(uint64_t full, int d, uint32_t bits) {
    return (full & ((1ull << (bits * (uint32_t)d)) - 1ull)) | ((uint64_t)(d - 1) << 60);
}

constexpr int kDictMaxTiers = 7;
__host__ __device__ __forceinline__ uint64_t dict_chain_key(uint32_t parent_sp, int j, int tier, uint64_t syms) {
    return (uint64_t)parent_sp | ((uint64_t)(j - 1) << 32) | ((uint64_t)tier << 35) | (syms << 38);
}

// All G lanes of a group call this together with the same key.  Lane l looks at bucket (home rounded down to a multiple of G) + l, i.e.
// the group reads G consecutive 32-byte buckets = one request per round; a slot that is empty at or after the home bucket ends the search.
template <int G, bool STATS>
__device__ __forceinline__ bool dict_probe(const DevIndex &ix, uint64_t key, uint32_t &sp, uint32_t &ep, uint32_t &touched) {
    const int lane = (G == 1) ? 0 : (threadIdx.x & (G - 1));
    const uint32_t gmask = group_mask<G>();
    const uint64_t home = dict_home(key, ix.dict_buckets);
    uint64_t base = home & ~(uint64_t)(G - 1);
    bool first = true;
    for (int round = 0; round < 4096; ++round) {
        const uint64_t b = base + (uint64_t)lane;
        uint4 e0, e1;
        ldg256(ix.dict + b * 2, e0, e1);
        if (STATS && lane == 0) ++touched;
        const uint64_t k0 = ((uint64_t)e0.y << 32) | e0.x, k1 = ((uint64_t)e1.y << 32) | e1.x;
        const bool mine = !first || b >= home;             // buckets before the home bucket are not on this key's probe sequence
        uint32_t f = 0, s = 0, e = 0;
        if (mine && k0 == key) { f = 1; s = e0.z; e = e0.w; }
        else if (mine && k1 == key) { f = 1; s = e1.z; e = e1.w; }
        uint32_t stop = (mine && (k0 == 0ull || k1 == 0ull)) ? 1u : 0u;
        if (G > 1) { f = group_sum<G>(f, gmask); s = group_sum<G>(s, gmask); e = group_sum<G>(e, gmask); stop = group_sum<G>(stop, gmask); }
        if (f) { sp = s; ep = e; return true; }
        if (stop) return false;
        base += G;
        if (base >= ix.dict_buckets) base = 0;
        first = false;
    }
    return false;
}

// ---- the whole backward search of one pattern: SuffixAlgo.search, findex.scala:15-31 -----------------------
// pat(i) returns pattern byte i.  Every thread of the warp calls this together (inactive groups pass
// active=false); groups leave the loop individually, the warp leaves when all are done.
//   * k-mer table (optional): the first kmer_k steps are one lookup.
//   * first step from (0,n) otherwise: (C[c], C[c+1]) without touching memory.
//   * singleton shortcut (optional): once the interval is one row r and 3..isat_syms bytes remain, the remaining bytes
//     are compared with T' in front of position sa[r]; the answer row is isa[sa[r]-remaining].  Identical to
//     stepping: from a singleton, a step succeeds iff BWT[r] = T'[sa[r]-1] equals the byte, and lands on
//     LF(r) = isa[sa[r]-1].  Patterns containing byte 0 take the ordinary steps (the '$' row wraps the text).
// From the interval after dict_D symbols (found in the dictionary): go on through the chain entries while the pattern and the stored
// tiers last.  i = index of the next pattern byte to consume; leaves (sp, ep, i) at the deepest stored prefix reached this way (a miss
// just ends the chain: the caller goes on with ordinary steps).  Group-uniform.
// `depth` = symbols consumed so far (dict_D + whole tiers).  BISECT: when the probe with all j symbols of a tier misses, the deepest
// stored prefix inside the tier is found by bisection (stored = more than 8 rows, and a prefix of such a j-mer is one); without it the
// miss just ends the chain.  Returns false when the chain ended on a miss of the full-j probe and no bisection was done (the two-pass
// count's first pass: the bisection belongs to the second).
template <int G, bool STATS, bool BISECT, typename PatFn>
__device__ __forceinline__ bool dict_chain(const DevIndex &ix, const uint8_t *code, PatFn pat, int &i, uint32_t &sp, uint32_t &ep,
                                           uint32_t &touched, uint32_t &steps, int depth, bool top_known_missed = false) {
    const int Jc = ix.dict_Jc;
    const uint32_t bits = (uint32_t)ix.dict_bits;
    for (int t = (depth - ix.dict_D) / Jc + 1; t <= kDictMaxTiers && i >= 0 && depth < ix.dict_Dx; ++t) {
        const int j = (i + 1) < Jc ? (i + 1) : Jc;
        uint64_t syms = 0;
        bool ok = true;
        for (int k = 0; k < j; ++k) {
            const uint32_t c = pat(i - k), cd = code[c];
            ok = ok && (cd != (uint32_t)kCodeAbsent) && (c != 0);
            syms |= (uint64_t)cd << (bits * (uint32_t)k);
        }
        if (!ok) return true;
        uint32_t s, e;
        if (!top_known_missed && dict_probe<G, STATS>(ix, dict_chain_key(sp, j, t, syms), s, e, touched)) {
            sp = s; ep = e;
            i -= j;
            depth += j;
            if (STATS) steps += j;
            if (j < Jc) return true;
            continue;
        }
        if (!BISECT) return false;
        int lo = 0, hi = j - 1;
        uint32_t bs = 0, be = 0;
        const uint32_t psp = sp;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (dict_probe<G, STATS>(ix, dict_chain_key(psp, mid, t, syms & ((1ull << (bits * (uint32_t)mid)) - 1ull)), s, e, touched)) { lo = mid; bs = s; be = e; }
            else hi = mid - 1;
        }
        if (lo > 0) { sp = bs; ep = be; i -= lo; if (STATS) steps += lo; }
        return true;
    }
    return true;
}

// ---- row-context hops ------------------------------------------------------------------------------------------------------------
// The pattern side of a hop of j symbols that consumes pattern bytes o .. o+j-1, in the packing of the entries' 96-bit symbol field.
// zero: one of those bytes is 0 (the '$' row wraps the text: ordinary steps instead); absent: one does not occur in the text (nothing matches).
struct CtxQuery {
    unsigned long long qlo, qhi, mlo, mhi;
    uint32_t sh;
    bool zero, absent;
};
template <typename PatFn>
__device__ __forceinline__ CtxQuery ctx_query(const DevIndex &ix, const SharedTables &tb, PatFn pat, int j, int o) {
    CtxQuery q;
    const uint32_t bits = (uint32_t)ix.isat_bits;
    q.qlo = 0; q.qhi = 0;
    q.sh = (uint32_t)(ix.ctx_J - j) * bits;
    const uint32_t nb = (uint32_t)j * bits;                                          // nb >= 1
    q.mlo = nb >= 64 ? ~0ull : ((1ull << nb) - 1ull);
    q.mhi = nb <= 64 ? 0ull : ((1ull << (nb - 64)) - 1ull);
    q.zero = false; q.absent = false;
    if (ix.ctx_raw) {                                     // raw bytes: pattern words compare directly, no translation;
        uint32_t w0, w1, w2;                              // a byte that is absent from the text just never matches
        pat.bytes12(o, w0, w1, w2);
        q.qlo = ((unsigned long long)w1 << 32) | w0;
        q.qhi = w2;
        const unsigned long long l = q.qlo | ~q.mlo, h = (q.qhi & q.mhi) | ~q.mhi;   // bytes past the hop must not look like zeros
        q.zero = (((l - 0x0101010101010101ull) & ~l) | ((h - 0x0101010101010101ull) & ~h)) & 0x8080808080808080ull;
    } else {
        for (int k = 0; k < j; ++k) {
            const uint32_t pc = pat(o + k), cd = tb.code[pc];
            q.zero = q.zero || (pc == 0);
            q.absent = q.absent || (cd == (uint32_t)kCodeAbsent);
            const unsigned long long v = (unsigned long long)((cd + 1u) & ((1u << bits) - 1u));
            const uint32_t ob = (uint32_t)k * bits;
            if (ob < 64) { q.qlo |= v << ob; if (ob + bits > 64) q.qhi |= v >> (64 - ob); }
            else q.qhi |= v << (ob - 64);
        }
    }
    return q;
}
// does the row whose context's second half is `b` = ctx[2r+1] go on with the hop's bytes?
__device__ __forceinline__ bool ctx_match(const CtxQuery &q, const uint4 &b) {
    const unsigned long long elo = ((unsigned long long)b.z << 32) | b.y, ehi = b.w;
    unsigned long long lo, hi;
    if (q.sh == 0) { lo = elo; hi = ehi; }
    else if (q.sh < 64) { lo = (elo >> q.sh) | (ehi << (64 - q.sh)); hi = ehi >> q.sh; }
    else { lo = ehi >> (q.sh - 64); hi = 0; }
    return (((lo ^ q.qlo) & q.mlo) | ((hi ^ q.qhi) & q.mhi)) == 0ull;
}

// ---- k-mer group blocks (DevIndex::kmer_rows > 0; DESIGN.md §3) ------------------------------------------------------------------------
// One 64-byte block per kKmerGroup consecutive k-mers in lexicographic order, in the bytes the plain table gives them.  Byte 15 = kind.
//   narrow (kind 0..3 = inline rows): bytes 0-3 base row, bytes 4-11 eight cumulative u8 ends — entry e = [base + end[e-1], base + end[e]),
//     end[-1] = 0; bytes 16-63 = ctx[2r+1] (the J-hop half of the row context) of rows base .. base+kind-1.
//   wide (kind 0xFF: more than 255 rows, or a row of no k-mer — '$' or a suffix shorter than k — between two of the group's intervals):
//     bytes 0-3 base, bytes 16-47 eight u32 ends, bytes 48-55 eight u8 leading gaps — entry e = [end[e-1] + gap[e], end[e]), end[-1] = base.
// An empty entry decodes to (0,0), as in the plain table.
constexpr uint32_t kKmerGroup = 8, kKmerWide = 0xFFu, kKmerInlineRows = 3;

// The table lookup of a group-form index: one request per block at one lane per query (the count kernels' setting on such indexes; at 2
// and 4 lanes every lane of the group loads the whole block, two requests).  When the next hop the plan takes is the
// full-depth one (J symbols) and the interval is small enough for row contexts, the hop is resolved at once for the rows the block carries:
// all of them inline -> the hop is done here (i -= J); otherwise the partial (minimum, count) and the first row still to fetch are handed to
// the first row-context step of search_pattern, which looks only at the rest.  Group-uniform (every lane holds the whole block).
// Every thread of the warp calls this together; `fetch` = this lane's query looks its block up.
template <int G, bool STATS, typename PatFn>
__device__ __forceinline__ void kmer_group(const DevIndex &ix, const SharedTables &tb, PatFn pat, bool fetch, uint32_t idx, int &i,
                                           uint32_t &sp, uint32_t &ep, uint32_t &touched, uint32_t &steps, uint32_t &pre_from,
                                           uint32_t &pre_best, uint32_t &pre_cnt) {
    const uint4 *blk = reinterpret_cast<const uint4 *>(ix.kmer) + (uint64_t)(idx / kKmerGroup) * 4;
    uint4 q0, q1, q2, q3;
    if constexpr (G == 1) {
        // What a random load costs is one request per load instruction and line: one lane's two 256-bit loads of its block are two.  So
        // the lanes of a pair fetch each other's block halves — one instruction per block, two lanes x 32 B — and swap what the other needs.
        const uint32_t odd = threadIdx.x & 1u;
        const unsigned long long mine = reinterpret_cast<unsigned long long>(blk);
        const unsigned long long pe = __shfl_sync(0xFFFFFFFFu, mine, (threadIdx.x & 31u) & ~1u);
        const unsigned long long po = __shfl_sync(0xFFFFFFFFu, mine, (threadIdx.x & 31u) | 1u);
        const bool fe = __shfl_sync(0xFFFFFFFFu, fetch, (threadIdx.x & 31u) & ~1u), fo = __shfl_sync(0xFFFFFFFFu, fetch, (threadIdx.x & 31u) | 1u);
        uint4 x0 = make_uint4(0, 0, 0, 0), x1 = x0, y0 = x0, y1 = x0;
        if (fe) ldg256(reinterpret_cast<const uint4 *>(pe) + 2 * odd, x0, x1);     // half `odd` of the even lane's block
        if (fo) ldg256(reinterpret_cast<const uint4 *>(po) + 2 * odd, y0, y1);     // half `odd` of the odd lane's block
        uint4 s0 = odd ? x0 : y0, s1 = odd ? x1 : y1;                            // what the partner lacks of its own block
        s0.x = __shfl_xor_sync(0xFFFFFFFFu, s0.x, 1); s0.y = __shfl_xor_sync(0xFFFFFFFFu, s0.y, 1);
        s0.z = __shfl_xor_sync(0xFFFFFFFFu, s0.z, 1); s0.w = __shfl_xor_sync(0xFFFFFFFFu, s0.w, 1);
        s1.x = __shfl_xor_sync(0xFFFFFFFFu, s1.x, 1); s1.y = __shfl_xor_sync(0xFFFFFFFFu, s1.y, 1);
        s1.z = __shfl_xor_sync(0xFFFFFFFFu, s1.z, 1); s1.w = __shfl_xor_sync(0xFFFFFFFFu, s1.w, 1);
        if (odd) { q0 = s0; q1 = s1; q2 = y0; q3 = y1; } else { q0 = x0; q1 = x1; q2 = s0; q3 = s1; }
    } else {
        if (!fetch) return;
        ldg256(blk, q0, q1);
        ldg256(blk + 2, q2, q3);
    }
    if (!fetch) return;
    const uint32_t e = idx % kKmerGroup, kind = q0.w >> 24, base = q0.x;
    uint32_t lo, hi;
    if (kind != kKmerWide) {
        const unsigned long long ends = ((unsigned long long)q0.z << 32) | q0.y;
        hi = base + (uint32_t)((ends >> (8 * e)) & 0xFFu);
        lo = base + (e ? (uint32_t)((ends >> (8 * e - 8)) & 0xFFu) : 0u);
    } else {
        auto end_of = [&](uint32_t k) {
            return k < 4 ? (k < 2 ? (k == 0 ? q1.x : q1.y) : (k == 2 ? q1.z : q1.w)) : (k < 6 ? (k == 4 ? q2.x : q2.y) : (k == 6 ? q2.z : q2.w));
        };
        hi = end_of(e);
        lo = (e ? end_of(e - 1) : base) + (((e < 4 ? q3.x : q3.y) >> (8 * (e & 3))) & 0xFFu);
    }
    if (lo < hi) { sp = lo; ep = hi; } else { sp = 0; ep = 0; }
    if (STATS) { touched += 1; steps += ix.kmer_k; }
    if (kind == kKmerWide || kind == 0 || ix.ctx == nullptr || sp >= ep || i < 0) return;
    const int rem = i + 1;
    const uint32_t rows = ep - sp;
    const int t = rem <= kCtxPlanMax ? (int)tb.plan[rem] : kCtxHops - 1;
    const uint32_t need = rem <= kCtxPlanMax ? (uint32_t)tb.plan[128 + rem] : (uint32_t)(rem / ix.ctx_J + 3);
    // exactly the condition under which search_pattern's first step is this hop through the row contexts
    if (t != kCtxHops - 1 || rows > kCtxMaxRows || !(rows == 1u || rows * need <= (uint32_t)rem)) return;
    const int j = ix.ctx_J;
    const CtxQuery q = ctx_query(ix, tb, pat, j, rem - j);
    if (q.zero) return;
    uint32_t best = 0xFFFFFFFFu, cnt = 0;
#pragma unroll
    for (uint32_t k = 0; k < kKmerInlineRows; ++k) {
        const uint4 &pl = k == 0 ? q1 : k == 1 ? q2 : q3;
        if (k < kind && base + k >= sp && base + k < ep && !q.absent && ctx_match(q, pl)) { best = pl.x < best ? pl.x : best; ++cnt; }
    }
    if (ep <= base + kind) {
        if (cnt) { sp = best; ep = best + cnt; } else { sp = 0; ep = 0; }
        i -= j;
        if (STATS) steps += j;
    } else {
        const int lane = (G == 1) ? 0 : (threadIdx.x & (G - 1));
        pre_from = base + kind;
        pre_best = best;
        pre_cnt = lane == 0 ? cnt : 0u;                   // the lanes' counts are summed
    }
}

// `mode` — how the two-pass count (dictionary first, the rest compacted; fmx_kernels.cu) hands a query over: kSearchFresh = from the
// start; kSearchTopMissed = the dictionary probe at the deepest possible prefix has been done and missed (bisection goes on below it);
// kSearchResume = the dictionary has been followed as far as it goes, (rsp, rep) is the interval after `rconsumed` symbols;
// kSearchChainMissed = the same, and the chain probe with all the symbols of the next tier has missed (bisection inside the tier goes on).
constexpr int kSearchFresh = 0, kSearchTopMissed = 1, kSearchResume = 2, kSearchChainMissed = 3;
template <int G, int LAYOUT, bool STATS, typename PatFn>
__device__ __forceinline__ void search_pattern(const DevIndex &ix, const SharedTables &tb, PatFn pat, int len, bool active,
                                               uint32_t &sp, uint32_t &ep, uint32_t &touched, uint32_t &steps,
                                               int mode = kSearchFresh, uint32_t rsp = 0, uint32_t rep = 0, int rconsumed = 0) {
    const int lane = (G == 1) ? 0 : (threadIdx.x & (G - 1));
    const uint32_t gmask = group_mask<G>();
    sp = 0;
    ep = active ? ix.n : 0u;
    int i = len - 1;
    bool noshort = (ix.isat == nullptr);
    uint32_t pre_from = 0, pre_best = 0xFFFFFFFFu, pre_cnt = 0;      // rows of the first row-context hop already resolved by kmer_group
    bool kfetch = false;                                               // group-form table: this query's block is to be fetched (entry kidx)
    uint32_t kidx = 0;
    if (active && (mode == kSearchResume || mode == kSearchChainMissed)) {
        sp = rsp; ep = rep;
        i -= rconsumed;
        if (mode == kSearchChainMissed) dict_chain<G, STATS, true>(ix, tb.code, pat, i, sp, ep, touched, steps, rconsumed, true);
    } else if (active && i >= 0) {
        bool done = false;
        if (ix.dict != nullptr && len > ix.kmer_k) {
            // deepest stored prefix of the pattern (consumption order): first the longest the dictionary could hold, then bisection
            const int K = ix.kmer_k;
            const uint32_t bits = (uint32_t)ix.dict_bits;
            int hi = len < ix.dict_D ? len : ix.dict_D;
            uint64_t full = 0;
            bool ok = true;
            for (int j = 0; j < hi; ++j) {
                const uint32_t c = pat(len - 1 - j), code = tb.code[c];
                ok = ok && (code != (uint32_t)kCodeAbsent) && (c != 0);
                full |= (uint64_t)code << (bits * (uint32_t)j);
            }
            if (ok) {
                int lo = K, d = hi;
                uint32_t bsp = 0, bep = 0;
                if (mode == kSearchTopMissed) { --hi; d = (lo + hi + 1) >> 1; }
                while (lo < hi) {
                    uint32_t s, e;
                    if (dict_probe<G, STATS>(ix, dict_key(full, d, bits), s, e, touched)) { lo = d; bsp = s; bep = e; }
                    else hi = d - 1;
                    d = (lo + hi + 1) >> 1;
                }
                if (lo > K) {
                    sp = bsp; ep = bep;
                    i -= lo;
                    done = true;
                    if (STATS) steps += lo;
                    if (lo == ix.dict_D && ix.dict_Dx > ix.dict_D) dict_chain<G, STATS, true>(ix, tb.code, pat, i, sp, ep, touched, steps, lo);
                }
            }
        }
        if (!done && ix.kmer != nullptr && len >= ix.kmer_k) {
            const int K = ix.kmer_k;
            uint32_t idx = 0;
            bool ok = true;
            for (int j = 0; j < K; ++j) {                 // plain table: the last pattern byte most significant; groups: the k-mer's first
                const uint32_t c = pat(ix.kmer_rows ? len - K + j : len - 1 - j), code = tb.code[c];
                ok = ok && (code != (uint32_t)kCodeAbsent) && (c != 0);
                idx = idx * ix.kmer_sigma + code;
            }
            if (ok) {
                i -= K;
                done = true;
                if (ix.kmer_rows) { kfetch = true; kidx = idx; }     // the block is fetched below, where the whole warp is converged
                else {
                    const uint2 v = ldg64(ix.kmer + idx);
                    sp = v.x; ep = v.y;
                    if (STATS) { touched += 1; steps += K; }
                }
            }
        }
        if (!done) {
            const uint32_t c = pat(i);
            sp = tb.C[c];
            ep = tb.C[c + 1];
            --i;
            if (STATS) ++steps;
        }
    }
    if (ix.kmer != nullptr && ix.kmer_rows) kmer_group<G, STATS>(ix, tb, pat, kfetch, kidx, i, sp, ep, touched, steps, pre_from, pre_best, pre_cnt);
    bool noctx = (ix.ctx == nullptr && ix.ctx8 == nullptr);
    for (;;) {
        const bool go = (i >= 0) && (sp < ep);
        if (go) {
            bool stepped = false;
            const int rem = i + 1;
            if (!noctx && ix.ctx8 != nullptr && (ep - sp) <= kCtxMaxRows && rem >= ix.ctx8_J) {
                // compact form: 8 bytes per row, a hop of exactly ctx8_J symbols — the pattern bytes rem-J .. rem-1
                const int J = ix.ctx8_J, o = rem - J;
                uint32_t q = 0;
                bool zero = false, absent = false;
                for (int k = 0; k < J; ++k) {
                    const uint32_t pc = pat(o + k), cd = tb.code[pc];
                    zero = zero || (pc == 0);
                    absent = absent || (cd == (uint32_t)kCodeAbsent);
                    q |= (cd & 3u) << (2 * k);
                }
                if (zero) noctx = true;
                else {
                    uint32_t best = 0xFFFFFFFFu, cnt = 0;
                    if (!absent) {
                        for (uint32_t r = sp + (uint32_t)lane; r < ep; r += G) {
                            const uint2 e = ldg64(ix.ctx8 + r);
                            if (e.y == q && e.x != 0xFFFFFFFFu) { best = e.x < best ? e.x : best; ++cnt; }
                        }
                    }
                    if (STATS && lane == 0) { touched += absent ? 0u : ep - sp; steps += J; }
                    if (G >= 2) { best = min(best, __shfl_xor_sync(gmask, best, 1)); cnt += __shfl_xor_sync(gmask, cnt, 1); }
                    if (G >= 4) { best = min(best, __shfl_xor_sync(gmask, best, 2)); cnt += __shfl_xor_sync(gmask, cnt, 2); }
                    if (cnt) { sp = best; ep = best + cnt; } else { sp = 0; ep = 0; }
                    i -= J;
                    stepped = true;
                }
            }
            if (!stepped && !noctx && ix.ctx != nullptr && (ep - sp) <= kCtxMaxRows) {
                // every row of the interval is looked at through its 32-byte context entry: the rows whose text goes on with the next
                // j pattern bytes map onto exactly the next interval (their targets isa[sa[r]-j] are its rows, contiguous) — j backward
                // steps for one fetch per row.  The plan table names the hop that finishes `rem` symbols in the fewest fetches; rank
                // steps are kept when they are cheaper (a wide interval with a few symbols left).
                const uint32_t rows = ep - sp;
                const int t = rem <= kCtxPlanMax ? (int)tb.plan[rem] : kCtxHops - 1;
                const uint32_t need = rem <= kCtxPlanMax ? (uint32_t)tb.plan[128 + rem] : (uint32_t)(rem / ix.ctx_J + 3);
                if (rows == 1u || rows * need <= (uint32_t)rem) {
                    const int j = (int)tb.hops[t];                       // this hop consumes pattern bytes rem-j .. rem-1
                    const CtxQuery q = ctx_query(ix, tb, pat, j, rem - j);
                    if (q.zero) noctx = true;                             // byte 0: the '$' row wraps the text, take the ordinary steps
                    else {
                        // rows before pre_from were resolved from the k-mer group block (their minimum and count carried in)
                        const uint32_t from = sp > pre_from ? sp : pre_from;
                        uint32_t best = pre_best, cnt = pre_cnt;
                        if (!q.absent) {
                            for (uint32_t r = from + (uint32_t)lane; r < ep; r += G) {
                                uint4 a, b;
                                ldg256(ix.ctx + (uint64_t)r * 2, a, b);
                                if (ctx_match(q, b)) {
                                    const uint32_t row = t == 0 ? a.x : t == 1 ? a.y : t == 2 ? a.z : t == 3 ? a.w : b.x;
                                    best = row < best ? row : best;
                                    ++cnt;
                                }
                            }
                        }
                        pre_from = 0; pre_best = 0xFFFFFFFFu; pre_cnt = 0;
                        if (STATS && lane == 0) { touched += q.absent ? 0u : ep - from; steps += j; }
                        if (G >= 2) { best = min(best, __shfl_xor_sync(gmask, best, 1)); cnt += __shfl_xor_sync(gmask, cnt, 1); }
                        if (G >= 4) { best = min(best, __shfl_xor_sync(gmask, best, 2)); cnt += __shfl_xor_sync(gmask, cnt, 2); }
                        if (cnt) { sp = best; ep = best + cnt; } else { sp = 0; ep = 0; }
                        i -= j;
                        stepped = true;
                    }
                }
            }
            if (!stepped && !noshort && (ep - sp) == 1u && i >= 2 && i < ix.isat_syms) {
                // one 16-byte entry holds isa[p] and the next isat_syms symbols of T': the whole shortcut is sa[row] -> isat[sa[row]-rem]
                const uint32_t q = ldg32(ix.sa + sp);
                const bool fits = q >= (uint32_t)rem;
                const uint32_t b0 = fits ? q - (uint32_t)rem : 0u;
                const uint4 e = ldg128(ix.isat + b0);
                const uint32_t bits = (uint32_t)ix.isat_bits, fmask = (1u << bits) - 1u;
                bool eq = fits, zero = false;
                for (int k = lane; k < rem; k += G) {
                    const uint32_t pc = pat(k);
                    const uint32_t o = (uint32_t)k * bits, w = o >> 5;
                    const uint32_t lo = w == 0 ? e.y : w == 1 ? e.z : e.w, hi = w == 0 ? e.z : w == 1 ? e.w : 0u;
                    const uint32_t sym = __funnelshift_r(lo, hi, o & 31u) & fmask;      // dense code + 1 of T'[b0 + k]
                    zero = zero || (pc == 0);
                    eq = eq && (sym == (uint32_t)tb.code[pc] + 1u);                     // an absent byte (code 0xFF) never matches
                }
                if (G > 1) { eq = __all_sync(gmask, eq); zero = __any_sync(gmask, zero); }
                if (zero) noshort = true;
                else {
                    if (eq) { sp = e.x; ep = e.x + 1; } else { sp = 0; ep = 0; }
                    i = -1;
                    stepped = true;
                    if (STATS) { touched += 2; steps += rem; }
                }
            }
            if (!stepped) {
                backward_step<G, LAYOUT, STATS>(ix, tb, pat(i), sp, ep, touched);
                --i;
                if (STATS) ++steps;
            }
        }
        if (__all_sync(0xFFFFFFFFu, !go)) break;
    }
}

// rank_c(pos) for a single position (occ / LF).  Returns C[c] + rank.
template <int G, int LAYOUT>
__device__ __forceinline__ uint32_t lf_value(const DevIndex &ix, const SharedTables &t, uint32_t c, uint32_t pos) {
    const uint32_t code = t.code[c];
    if (c == 0) return pos > ix.eof ? 1u : 0u;
    if (code == kCodeAbsent) return t.C[c];
    if (LAYOUT == FMX_LAYOUT_PLANES) {
        return t.base[c] + rank_one<G>(ix.blocks + (uint64_t)code * ix.stride * 4, pos, nullptr);
    } else if (LAYOUT == FMX_LAYOUT_WMX) {
        uint32_t p = pos;
        const int b = ix.wmx_b, L = ix.wmx_levels;
        for (int l = 0; l < L; ++l) {
            const uint32_t d = (code >> (b * (L - 1 - l))) & ((1u << b) - 1u);
            p = ix.zx[l][d] + rank_one_x<G>(ix.blocks + (uint64_t)l * ix.wmx_stride * 8, b, d, p);
        }
        if (code == 0) p -= (pos > ix.eof);
        return t.base[c] + p;
    } else {
        uint32_t p = pos;
        const int L = ix.levels;
        for (int l = 0; l < L; ++l) {
            uint32_t r = rank_one<G>(ix.blocks + (uint64_t)l * ix.stride * 4, p, nullptr);
            if ((code >> (L - 1 - l)) & 1u) p = ix.z[l] + r; else p -= r;
        }
        if (code == 0) p -= (pos > ix.eof);
        return t.base[c] + p;
    }
}

}  // namespace fmx

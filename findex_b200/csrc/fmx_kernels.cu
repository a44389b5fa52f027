// fmx_kernels.cu — the search kernels of libfmgpu (sm_100a).
//
//   K1 count         : SuffixAlgo.search            src/main/scala/org/fmindex/findex.scala:15-31
//      prev_range    : SuffixAlgo.getPrevRange      findex.scala:32-36
//      interval      : getIntervalPrevRange         findex.scala:37-51
//      occ           : NaiveFMSearcher.occ          bwtmerger.scala:354-375
//      lf/prev_substr: getPrevI / prevSubstr        bwtmerger.scala:386-389, 409-419
//   K2 locate        : sa[] of bwtFm2sa             util.scala:213-224, via sampled rows + LF walk
//   K3 regex         : ReTree._matchSA              re2/retree.scala:618-653 — fmx_regex_kernel.cu
//   K4 gather bench  : the random-64-B-gather roofline denominator (SURVEY.md §8d)
//
// All of them are bound by the rate of random HBM requests (DESIGN.md §5): G (1, 2 or 4) lanes cooperate on one
// query so that a 64-byte rank block arrives as ONE request (256-bit loads at G <= 2); the two ends of the interval are
// fetched together (two independent loads in flight per lane) and share the fetch when they fall into the
// same block.  Nothing here is GEMM-shaped, so no tensor-core path exists by design.
#include "fmx_kernels.cuh"

#include <algorithm>

namespace fmx {

// =====================================================================================================
// K1: count
// =====================================================================================================
// resident CTAs per SM the count kernel is compiled for: 8 (32 registers) for the bitvector layouts at 2/4 lanes, 6 at one lane; the
// multi-ary blocks hold twice the words per lane and get 5 (48 registers, no spills)
template <int G, int LAYOUT, bool STATS, typename OutT, int MINB = (LAYOUT == FMX_LAYOUT_WMX ? 5 : (G == 1) ? 6 : 8)>
__global__ void __launch_bounds__(kThreads, MINB)
count_fixed_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ pat, int len, long long m,
                   OutT *__restrict__ sp_out, OutT *__restrict__ ep_out, unsigned long long *stats, const __grid_constant__ PeerSinks sinks) {
    __shared__ SharedTables tb;
    extern __shared__ __align__(16) uint8_t spat[];
    constexpr int QPB = kThreads / G;                     // queries per CTA
    load_tables(tb, ix);

    const long long q0 = (long long)blockIdx.x * QPB;
    const int nq = (int)((m - q0) < (long long)QPB ? (m - q0) : (long long)QPB);
    {   // stage this CTA's patterns (contiguous bytes) into shared memory, 16 B per thread when aligned
        const uint8_t *src = pat + q0 * len;
        const int nbytes = nq * len;
        if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
            const int nvec = nbytes >> 4;
            for (int i = threadIdx.x; i < nvec; i += kThreads)
                reinterpret_cast<uint4 *>(spat)[i] = ldg128(reinterpret_cast<const uint4 *>(src) + i);
            for (int i = (nvec << 4) + threadIdx.x; i < nbytes; i += kThreads) spat[i] = src[i];
        } else {
            for (int i = threadIdx.x; i < nbytes; i += kThreads) spat[i] = src[i];
        }
    }
    __syncthreads();

    const int g = threadIdx.x / G;
    const bool active = g < nq;
    uint32_t sp, ep, touched = 0, steps = 0;
    search_pattern<G, LAYOUT, STATS>(ix, tb, SmemPattern{spat + g * len, len, (len & 3) == 0}, len, active, sp, ep, touched, steps);
    const bool hit = sp < ep;
    const uint32_t cnt = hit ? ep - sp : 0u;
    if (active && (threadIdx.x % G) == 0) {
        sp_out[q0 + g] = hit ? (OutT)sp : (OutT)0;
        ep_out[q0 + g] = hit ? (OutT)ep : (OutT)0;
        if (sinks.n == 1) sinks.p[0][sinks.offset + q0 + g] = cnt;          // count-only host call: one local sink
    }
    // fused exchange: the CTA's hit counts go straight into every rank's gathered buffer (peer-mapped memory over NVLink/NVSwitch).
    // They are transposed through shared memory so that a warp stores 512 contiguous bytes (32 lanes x 16 B) to ONE peer: per CTA
    // 2 store instructions per peer instead of one 128-byte store per warp and peer (each remote store instruction costs the kernel
    // about as much as a local request; measured +1.6 % of the step per peer before).
    if (sinks.n > 1) {                                                       // grid-uniform
        __shared__ __align__(16) uint32_t scnt[kThreads];
        if ((threadIdx.x % G) == 0) scnt[g] = active ? cnt : 0u;
        __syncthreads();
        const long long base = sinks.offset + q0;
        if (nq == QPB && (base & 3) == 0) {
            constexpr int V = QPB / 4;                                       // 16-byte pieces per peer
            for (int w = threadIdx.x; w < sinks.n * V; w += kThreads) {
                const int j = w / V, k = w - j * V;
                reinterpret_cast<uint4 *>(sinks.p[j] + base)[k] = reinterpret_cast<const uint4 *>(scnt)[k];
            }
        } else {
            for (int w = threadIdx.x; w < sinks.n * nq; w += kThreads) {
                const int j = w / nq, k = w - j * nq;
                sinks.p[j][base + k] = scnt[k];
            }
        }
    }
    if (STATS) {
        if ((threadIdx.x % G) != 0) { touched = 0; steps = 0; }
        for (int o = 16; o; o >>= 1) {
            touched += __shfl_xor_sync(0xFFFFFFFFu, touched, o);
            steps += __shfl_xor_sync(0xFFFFFFFFu, steps, o);
        }
        if ((threadIdx.x & 31) == 0) { atomicAdd(&stats[0], (unsigned long long)touched); atomicAdd(&stats[1], (unsigned long long)steps); }
    }
}

// Fixed-length patterns too long to stage a CTA's worth of them in shared memory: read from global memory, same outputs
template <int G, int LAYOUT, typename OutT>
__global__ void __launch_bounds__(kThreads)
count_fixed_gmem_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ pat, int len, long long m, OutT *__restrict__ sp_out,
                        OutT *__restrict__ ep_out, const __grid_constant__ PeerSinks sinks) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    constexpr int QPB = kThreads / G;
    const long long q = (long long)blockIdx.x * QPB + threadIdx.x / G;
    const bool active = q < m;
    uint32_t sp, ep, touched = 0, steps = 0;
    search_pattern<G, LAYOUT, false>(ix, tb, GlobalPattern{pat + (active ? q : 0) * len, len}, len, active, sp, ep, touched, steps);
    if (active && (threadIdx.x % G) == 0) {
        const bool hit = sp < ep;
        sp_out[q] = hit ? (OutT)sp : (OutT)0;
        ep_out[q] = hit ? (OutT)ep : (OutT)0;
        for (int j = 0; j < sinks.n; ++j) sinks.p[j][sinks.offset + q] = hit ? ep - sp : 0u;
    }
}

// ---- two-pass count for indexes with a dictionary of wide intervals --------------------------------------------------------------------
// With a dictionary most queries are ONE request (the probe at their deepest possible prefix) while the rest walk a chain of a dozen; in
// one kernel a warp waits for its slowest query and the request rate collapses (measured: 17 G requests/s instead of 46).  So the work is
// split by cost.  Pass 1, one thread per query: that single probe; a hit covering the whole pattern is the answer, everything else is
// appended to a work list (warp-aggregated) with what is known: the probe missed / the probe hit and (sp, ep) after D symbols is in the
// output arrays / not probed (absent symbol, byte 0).  Pass 2: the general search over the compacted list, patterns from global memory.
constexpr uint32_t kListModeShift = 30, kListIdMask = (1u << kListModeShift) - 1u;

template <typename OutT>
__global__ void __launch_bounds__(kThreads)
count_dict_first_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ pat, int len, long long m, OutT *__restrict__ sp_out,
                        OutT *__restrict__ ep_out, uint2 *__restrict__ list, unsigned long long *__restrict__ list_count,
                        const __grid_constant__ PeerSinks sinks) {
    __shared__ uint8_t scode[256];
    extern __shared__ __align__(16) uint8_t spat[];
    for (int i = threadIdx.x; i < 256; i += kThreads) scode[i] = ix.code[i];
    const int d0 = len < ix.dict_D ? len : ix.dict_D;         // symbols the probe covers: the last d0 bytes of the pattern
    const long long q0 = (long long)blockIdx.x * kThreads;
    const int nq = (int)((m - q0) < (long long)kThreads ? (m - q0) : (long long)kThreads);
    {
        const uint8_t *src = pat + q0 * len;
        const int nbytes = nq * len;
        if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
            const int nvec = nbytes >> 4;
            for (int i = threadIdx.x; i < nvec; i += kThreads)
                reinterpret_cast<uint4 *>(spat)[i] = ldg128(reinterpret_cast<const uint4 *>(src) + i);
            for (int i = (nvec << 4) + threadIdx.x; i < nbytes; i += kThreads) spat[i] = src[i];
        } else {
            for (int i = threadIdx.x; i < nbytes; i += kThreads) spat[i] = src[i];
        }
    }
    __syncthreads();
    const bool active = (int)threadIdx.x < nq;
    const long long q = q0 + threadIdx.x;
    uint32_t entry = 0xFFFFFFFFu, consumed = 0;                // 0xFFFFFFFF = finished here
    if (active) {
        const uint8_t *p = spat + (size_t)threadIdx.x * len;
        const uint32_t bits = (uint32_t)ix.dict_bits;
        uint64_t full = 0;
        bool ok = true;
        for (int j = 0; j < d0; ++j) {
            const uint32_t c = p[len - 1 - j], code = scode[c];
            ok = ok && (code != (uint32_t)kCodeAbsent) && (c != 0);
            full |= (uint64_t)code << (bits * (uint32_t)j);
        }
        entry = (uint32_t)threadIdx.x | ((uint32_t)kSearchFresh << kListModeShift);
        if (ok) {
            uint32_t s = 0, e = 0, touched = 0;
            if (dict_probe<1, false>(ix, dict_key(full, d0, bits), s, e, touched)) {
                int i = len - 1 - d0;
                bool chain_open = true;                          // false: the next tier's full probe missed, its bisection is left to pass 2
                if (i >= 0 && ix.dict_Dx > ix.dict_D) {          // d0 = dict_D: on through the chain entries
                    uint32_t steps = 0;
                    chain_open = dict_chain<1, false, false>(ix, scode, SmemPattern{p, len, false}, i, s, e, touched, steps, d0);
                }
                consumed = (uint32_t)(len - 1 - i);
                sp_out[q] = (OutT)s;
                ep_out[q] = (OutT)e;
                if (i < 0) {
                    entry = 0xFFFFFFFFu;
                    for (int j = 0; j < sinks.n; ++j) sinks.p[j][sinks.offset + q] = e - s;
                } else entry = (uint32_t)threadIdx.x | ((uint32_t)(chain_open ? kSearchResume : kSearchChainMissed) << kListModeShift);
            } else entry = (uint32_t)threadIdx.x | ((uint32_t)kSearchTopMissed << kListModeShift);
        }
    }
    // append the CTA's unfinished queries with ONE atomic (125 k same-address atomics per 4 M queries, one per warp, cost more than the probes)
    __shared__ uint32_t wcount[kThreads / 32];
    __shared__ unsigned long long cta_base;
    const uint32_t need = __ballot_sync(0xFFFFFFFFu, entry != 0xFFFFFFFFu);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) wcount[warp] = (uint32_t)__popc(need);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t total = 0;
        for (int w = 0; w < kThreads / 32; ++w) { const uint32_t c = wcount[w]; wcount[w] = total; total += c; }
        cta_base = total ? atomicAdd(list_count, (unsigned long long)total) : 0ull;
    }
    __syncthreads();
    if (entry != 0xFFFFFFFFu) {
        const uint32_t mode = entry >> kListModeShift;
        list[cta_base + wcount[warp] + __popc(need & ((1u << lane) - 1u))] = make_uint2((uint32_t)(q0 + (entry & kListIdMask)) | (mode << kListModeShift), consumed);
    }
}

template <int G, int LAYOUT, typename OutT>
__global__ void __launch_bounds__(kThreads)
count_list_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ pat, int len, OutT *__restrict__ sp_out, OutT *__restrict__ ep_out,
                  const uint2 *__restrict__ list, const unsigned long long *__restrict__ list_count, const __grid_constant__ PeerSinks sinks) {
    __shared__ SharedTables tb;
    extern __shared__ __align__(16) uint8_t spat[];
    constexpr int QPB = kThreads / G;
    const unsigned long long count = *list_count;
    if ((unsigned long long)blockIdx.x * QPB >= count) return;
    load_tables(tb, ix);
    const int g = threadIdx.x / G, lane = threadIdx.x % G;
    const int stride = (len + 3) & ~3;                      // every staged pattern starts on a word
    {   // one chunk of the list per CTA (CTAs beyond the list's end have left above): the block scheduler balances the chains
        const unsigned long long t = (unsigned long long)blockIdx.x * QPB + g;
        const bool active = t < count;
        const uint2 le = active ? list[t] : make_uint2(0u, 0u);
        const uint32_t entry = le.x;
        const long long q = (long long)(entry & kListIdMask);
        const int mode = (int)(entry >> kListModeShift);
        __syncthreads();                                    // tables loaded / the previous round is done with spat
        if (active) {                                       // the group stages its own pattern
            const uint8_t *src = pat + q * len;
            uint8_t *dst = spat + (size_t)g * stride;
            if ((len & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 3) == 0)
                for (int w = lane; w < (len >> 2); w += G) reinterpret_cast<uint32_t *>(dst)[w] = __ldg(reinterpret_cast<const uint32_t *>(src) + w);
            else
                for (int b = lane; b < len; b += G) dst[b] = __ldg(src + b);
        }
        __syncthreads();
        uint32_t rsp = 0, rep = 0;
        if (active && (mode == kSearchResume || mode == kSearchChainMissed)) { rsp = (uint32_t)sp_out[q]; rep = (uint32_t)ep_out[q]; }
        uint32_t sp, ep, touched = 0, steps = 0;
        search_pattern<G, LAYOUT, false>(ix, tb, SmemPattern{spat + (size_t)g * stride, len, true}, len, active, sp, ep, touched, steps, mode, rsp, rep, (int)le.y);
        if (active && (threadIdx.x % G) == 0) {
            const bool hit = sp < ep;
            sp_out[q] = hit ? (OutT)sp : (OutT)0;
            ep_out[q] = hit ? (OutT)ep : (OutT)0;
            for (int j = 0; j < sinks.n; ++j) sinks.p[j][sinks.offset + q] = hit ? ep - sp : 0u;
        }
    }
}

template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
count_var_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ pat, const long long *__restrict__ off,
                 long long m, long long *__restrict__ sp_out, long long *__restrict__ ep_out) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    constexpr int QPB = kThreads / G;
    const long long q = (long long)blockIdx.x * QPB + threadIdx.x / G;
    const bool active = q < m;
    long long lo = 0, hi = 0;
    if (active) { lo = off[q]; hi = off[q + 1]; }
    uint32_t sp, ep, touched = 0, steps = 0;
    search_pattern<G, LAYOUT, false>(ix, tb, GlobalPattern{pat + lo, (int)(hi - lo)}, (int)(hi - lo), active, sp, ep, touched, steps);
    if (active && (threadIdx.x % G) == 0) {
        const bool hit = sp < ep;
        sp_out[q] = hit ? (long long)sp : 0;
        ep_out[q] = hit ? (long long)ep : 0;
    }
}

// ---- matching statistics (fmx_match_stats_batch / fmx_smem_*; include/fmgpu.h) -----------------------------------------------------
// One query per group, left to right (file order), state (l, sp, ep) = the longest suffix S of the query so far that occurs and the
// interval of reverse(S).  A symbol extends S by one backward step; when the step comes back empty, the interval is widened to its LCP
// parent (lcp_widen) and the step retried, until it succeeds or l = 0 (from (0, n) the step is (C[c], C[c+1]), no request).  Each retry
// lowers l, so a query of length L takes at most 2L steps and L widenings.  Outputs by text position off[q] + j: ms_len, and the interval
// when ms_sp != nullptr; flag != nullptr: flag = 1 where an SMEM of at least min_len symbols ends (ms_len[j] >= min_len and j is the last
// position or ms_len[j+1] <= ms_len[j]).  STATS: stats[0..2] += rank blocks, lcp8 blocks + record / lcpx reads, minima lines.
template <int G, int LAYOUT, bool STATS>
__global__ void __launch_bounds__(kThreads)
match_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ pat, const long long *__restrict__ off, long long m,
             int *__restrict__ ms_len, uint32_t *__restrict__ ms_sp, uint32_t *__restrict__ ms_ep, uint32_t *__restrict__ flag, int min_len,
             unsigned long long *__restrict__ stats) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const long long q = (long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (q >= m) return;                                                   // group-uniform; only group shuffles follow
    const bool lead = (threadIdx.x % G) == 0;
    const long long lo = off[q], hi = off[q + 1];
    uint32_t l = 0, sp = 0, ep = ix.n, prev = 0, rank_req = 0, lcp_req = 0, min_req = 0;
    for (long long i = lo; i < hi; ++i) {
        const uint32_t c = __ldg(pat + i);
        for (;;) {
            if (l == 0) {
                sp = tb.C[c]; ep = tb.C[c + 1];
                if (sp < ep) l = 1; else { sp = 0; ep = ix.n; }
                break;
            }
            uint32_t s = sp, e = ep;
            backward_step<G, LAYOUT, STATS>(ix, tb, c, s, e, rank_req);
            if (s < e) { sp = s; ep = e; ++l; break; }
            lcp_widen<G, STATS>(ix, sp, ep, l, lcp_req, min_req);
        }
        if (lead) {
            ms_len[i] = (int)l;
            if (ms_sp) { ms_sp[i] = sp; ms_ep[i] = ep; }
            if (flag && i > lo) flag[i - 1] = (prev >= (uint32_t)min_len && l <= prev) ? 1u : 0u;
        }
        prev = l;
    }
    if (lead && flag && hi > lo) flag[hi - 1] = prev >= (uint32_t)min_len ? 1u : 0u;
    if (STATS && lead) {
        atomicAdd(&stats[0], (unsigned long long)rank_req);
        atomicAdd(&stats[1], (unsigned long long)lcp_req);
        atomicAdd(&stats[2], (unsigned long long)min_req);
    }
}

// SMEM offsets per query: out_off[q] = the exclusive scan of the flags at the query's first position (q = m: the total)
__global__ void smem_offsets_kernel(const uint32_t *__restrict__ scan, const long long *__restrict__ off, long long m, long long *__restrict__ out_off) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q <= m) out_off[q] = (long long)scan[off[q]];
}

// every flagged position i -> its SMEM (start inside the query, length, interval) at slot scan[i]
__global__ void smem_compact_kernel(const uint32_t *__restrict__ flag, const uint32_t *__restrict__ scan, const int *__restrict__ ms_len,
                                    const uint32_t *__restrict__ ms_sp, const uint32_t *__restrict__ ms_ep, const long long *__restrict__ off,
                                    long long m, long long T, int *__restrict__ start, int *__restrict__ len, uint32_t *__restrict__ sp,
                                    uint32_t *__restrict__ ep) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= T || !flag[i]) return;
    long long a = 0, b = m;                                               // the query: last q < m with off[q] <= i
    while (b - a > 1) { const long long mid = (a + b) >> 1; if (off[mid] <= i) a = mid; else b = mid; }
    const uint32_t k = scan[i];
    const int l = ms_len[i];
    start[k] = (int)(i - off[a]) - l + 1;
    len[k] = l;
    sp[k] = ms_sp[i];
    ep[k] = ms_ep[i];
}

// ---- k-mer census (fmx_kmer_spectrum / fmx_kmer_list_*; include/fmgpu.h) --------------------------------------------------------------
// Row r < n-1 ends a run of rows that share their first k symbols when LCP[r] < k; row n-1 always does (its LCP is 0).  The run from the
// row after the previous end to an end row e is the interval [start, e+1) of one k-mer, or one of the k single rows whose suffix is
// shorter than k + 1 ('$' within its first k symbols).  One streaming pass over lcp8: a warp owns a tile of kCensusTile consecutive
// 64-row blocks and walks it 32 blocks (one per lane, two 32-byte loads) at a time; each lane turns its block into the 64-bit mask of its
// end rows.  The run open at a lane's first row comes from the lanes before it (a warp max scan of "row after the last end", 0 = none),
// at a tile's first row from the tiles before it (census_last_kernel, then inclusive_max_u32 over the tiles), so a run may span any
// number of lanes and tiles.
constexpr uint32_t kCensusTile = 256, kCensusBuckets = 1024;

__device__ __forceinline__ void ldg256_stream(const uint4 *p, uint4 &a, uint4 &b) {
    asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w) : "l"(p));
}

// end rows of block blk (bit o = row 64 blk + o), 0 past the last block.  For k > 255 the rows with lcp8 = 255 compare their exact LCP,
// read from lcpx, where a block's escaped values are consecutive from its record's first escape.
__device__ __forceinline__ unsigned long long census_mask(const DevIndex &ix, uint32_t blk, uint32_t nb, uint32_t k) {
    if (blk >= nb) return 0ull;
    uint4 v[4];
    ldg256_stream(ix.lcp8 + (uint64_t)blk * 4, v[0], v[1]);
    ldg256_stream(ix.lcp8 + (uint64_t)blk * 4 + 2, v[2], v[3]);
    const uint32_t dup = (k < kLcpEsc ? k : kLcpEsc) * 0x01010101u;
    unsigned long long m = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t w[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) m |= (unsigned long long)byte_flags4(__vcmpltu4(w[j], dup)) << (16 * i + 4 * j);
    }
    const uint32_t rows = ix.n - blk * kLcpRows;
    const unsigned long long valid = rows < kLcpRows ? (1ull << rows) - 1ull : ~0ull;      // rows >= n pad the last block
    m &= valid;
    if (k > kLcpEsc) {
        unsigned long long esc = ~m & valid;
        if (esc) {
            uint32_t x = ldg64(ix.lcp_rec + blk).y;
            for (; esc; esc &= esc - 1ull, ++x)
                if (ldg32(ix.lcpx + x) < k) m |= esc & (0ull - esc);
        }
    }
    return m;
}

// the row after the last end row before this lane's block (lanes before it, else `carry`); carry becomes the warp's last end + 1
__device__ __forceinline__ uint32_t census_open(unsigned long long m, uint32_t r0, uint32_t &carry) {
    const int lane = threadIdx.x & 31;
    uint32_t incl = m ? r0 + 64u - (uint32_t)__clzll((long long)m) : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl = max(incl, o);
    }
    uint32_t excl = __shfl_up_sync(0xFFFFFFFFu, incl, 1);
    excl = lane == 0 ? 0u : excl;
    const uint32_t open = max(carry, excl);
    carry = max(carry, __shfl_sync(0xFFFFFFFFu, incl, 31));
    return open;
}

// the start row of the run that ends at bit e of a lane's mask m (block rows from r0; `open` = the start of the lane's first run)
__device__ __forceinline__ uint32_t census_start(unsigned long long m, int e, uint32_t r0, uint32_t open) {
    const unsigned long long below = m & ((1ull << e) - 1ull);
    return below ? r0 + 64u - (uint32_t)__clzll((long long)below) : open;
}

// tile_last[t] = the row after the last end row of tile t, 0 when it has none; the warp reads its tile backwards and stops at the first
// 32 blocks that hold an end row (for most k the tile's last ones)
__global__ void __launch_bounds__(kThreads)
census_last_kernel(const __grid_constant__ DevIndex ix, uint32_t nb, uint32_t ntiles, uint32_t k, uint32_t *__restrict__ tile_last) {
    const int lane = threadIdx.x & 31;
    for (uint32_t t = blockIdx.x * (kThreads / 32) + threadIdx.x / 32; t < ntiles; t += gridDim.x * (kThreads / 32)) {
        uint32_t after = 0;
        for (int c = (int)(kCensusTile / 32) - 1; c >= 0; --c) {
            const uint32_t blk = t * kCensusTile + (uint32_t)c * 32u + (uint32_t)lane;
            const unsigned long long m = census_mask(ix, blk, nb, k);
            const uint32_t bal = __ballot_sync(0xFFFFFFFFu, m != 0ull);
            if (bal) {
                const int hl = 31 - __clz(bal);
                after = __shfl_sync(0xFFFFFFFFu, m ? blk * kLcpRows + 64u - (uint32_t)__clzll((long long)m) : 0u, hl);
                break;
            }
        }
        if (lane == 0) tile_last[t] = after;
    }
}

// MODE kCensusSpectrum: hist[min(count, buckets) - 1] += 1 and max_occ = max count over every run (the short-suffix rows included; the
// host takes them out).  Runs of one row (an end row after an end row) are counted by popcount; the others go to a shared histogram of
// the first kCensusBuckets buckets (one global atomic per non-empty bucket and CTA) or straight to the global one.
// MODE kCensusCount: tile_cnt[t] = the runs of tile t with min_count <= count <= max_count (0 = no bound) — single rows only when
// min_count = 1, and then not those in ex[0 .. nex) (sorted: the short-suffix rows).  MODE kCensusEmit: the same runs, (start, end + 1)
// to sp / ep from slot tile_off[t] on, in row order.
enum { kCensusSpectrum = 0, kCensusCount = 1, kCensusEmit = 2 };
template <int MODE>
__global__ void __launch_bounds__(kThreads)
census_kernel(const __grid_constant__ DevIndex ix, uint32_t nb, uint32_t ntiles, uint32_t k, const uint32_t *__restrict__ tile_incl,
              uint32_t buckets, unsigned long long *__restrict__ hist, unsigned long long *__restrict__ max_occ, uint32_t min_count,
              uint32_t max_count, const uint32_t *__restrict__ ex, uint32_t nex, uint32_t *__restrict__ tile_cnt,
              const uint32_t *__restrict__ tile_off, uint32_t *__restrict__ sp, uint32_t *__restrict__ ep) {
    __shared__ uint32_t sh[MODE == kCensusSpectrum ? kCensusBuckets : 1];
    __shared__ uint32_t sh_max;
    const int lane = threadIdx.x & 31;
    const uint32_t nsh = buckets < kCensusBuckets ? buckets : kCensusBuckets;
    if (MODE == kCensusSpectrum) {
        for (uint32_t i = threadIdx.x; i < nsh; i += blockDim.x) sh[i] = 0;
        if (threadIdx.x == 0) sh_max = 0;
        __syncthreads();
    }
    uint32_t ones = 0, mx = 0;
    for (uint32_t t = blockIdx.x * (kThreads / 32) + threadIdx.x / 32; t < ntiles; t += gridDim.x * (kThreads / 32)) {
        uint32_t carry = t ? tile_incl[t - 1] : 0u;
        uint32_t lo = 0, hi = 0, slot = 0;
        if (MODE != kCensusSpectrum && min_count == 1 && nex) {                // short-suffix rows of this tile: ex[lo .. hi)
            const uint64_t a = (uint64_t)t * kCensusTile * kLcpRows, b = a + kCensusTile * kLcpRows;
            uint32_t l = 0, h = nex;
            while (l < h) { const uint32_t md = (l + h) >> 1; if ((uint64_t)ex[md] < a) l = md + 1; else h = md; }
            lo = l; h = nex;
            while (l < h) { const uint32_t md = (l + h) >> 1; if ((uint64_t)ex[md] < b) l = md + 1; else h = md; }
            hi = l;
        }
        if (MODE == kCensusEmit) slot = tile_off[t];
        uint32_t tcount = 0;
        for (uint32_t c = 0; c < kCensusTile / 32; ++c) {
            const uint32_t blk = t * kCensusTile + c * 32u + (uint32_t)lane, r0 = blk * kLcpRows;
            const unsigned long long m = census_mask(ix, blk, nb, k);
            if (__all_sync(0xFFFFFFFFu, m == 0ull)) { if (t * kCensusTile + c * 32u >= nb) break; continue; }
            const uint32_t open = census_open(m, r0, carry);
            const unsigned long long prev = (m << 1) | (open == r0 ? 1ull : 0ull);   // rows whose previous row ends a run
            if (MODE == kCensusSpectrum) {
                ones += (uint32_t)__popcll(m & prev);
                for (unsigned long long R = m & ~prev; R; R &= R - 1ull) {
                    const int e = __ffsll((long long)R) - 1;
                    const uint32_t cnt = r0 + (uint32_t)e + 1u - census_start(m, e, r0, open);
                    const uint32_t bk = (cnt < buckets ? cnt : buckets) - 1u;
                    if (bk < kCensusBuckets) atomicAdd(&sh[bk], 1u); else atomicAdd(&hist[bk], 1ull);
                    mx = max(mx, cnt);
                }
                if (m & prev) mx = max(mx, 1u);
            } else {
                unsigned long long X = 0;                                    // short-suffix rows of this block
                if (hi > lo) {
                    uint32_t l = lo, h = hi;
                    while (l < h) { const uint32_t md = (l + h) >> 1; if (ex[md] < r0) l = md + 1; else h = md; }
                    for (; l < hi && ex[l] - r0 < 64u && ex[l] >= r0; ++l) X |= 1ull << (ex[l] - r0);
                }
                auto keep = [&](uint32_t cnt) { return cnt >= min_count && (max_count == 0 || cnt <= max_count); };
                uint32_t cl = min_count == 1 ? (uint32_t)__popcll(m & prev & ~X) : 0u;
                if (max_count != 1)
                    for (unsigned long long R = m & ~prev; R; R &= R - 1ull) {
                        const int e = __ffsll((long long)R) - 1;
                        cl += keep(r0 + (uint32_t)e + 1u - census_start(m, e, r0, open)) ? 1u : 0u;
                    }
                if (MODE == kCensusCount) tcount += cl;
                else {
                    uint32_t pre = cl;                                           // exclusive warp scan of the lanes' counts
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) { const uint32_t o = __shfl_up_sync(0xFFFFFFFFu, pre, d); if (lane >= d) pre += o; }
                    const uint32_t total = __shfl_sync(0xFFFFFFFFu, pre, 31);
                    uint32_t s = slot + pre - cl;
                    for (unsigned long long R = cl ? (min_count == 1 ? m & ~X : m & ~prev) : 0ull; R; R &= R - 1ull) {
                        const int e = __ffsll((long long)R) - 1;
                        const uint32_t st = census_start(m, e, r0, open), end = r0 + (uint32_t)e + 1u;
                        if (keep(end - st)) { sp[s] = st; ep[s] = end; ++s; }
                    }
                    slot += total;
                }
            }
        }
        if (MODE == kCensusCount) {
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) tcount += __shfl_xor_sync(0xFFFFFFFFu, tcount, d);
            if (lane == 0) tile_cnt[t] = tcount;
        }
    }
    if (MODE == kCensusSpectrum) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) { ones += __shfl_xor_sync(0xFFFFFFFFu, ones, d); mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, d)); }
        if (lane == 0) { if (ones) atomicAdd(&sh[0], ones); atomicMax(&sh_max, mx); }
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < nsh; i += blockDim.x)
            if (sh[i]) atomicAdd(&hist[i], (unsigned long long)sh[i]);
        if (threadIdx.x == 0 && sh_max) atomicMax(max_occ, (unsigned long long)sh_max);
    }
}

// rows[0 .. steps] = row 0 and the rows of the LF walk from it: the rows of T' positions n-1, n-2, .. n-1-steps (one group)
template <int G, int LAYOUT>
__global__ void census_walk_kernel(const __grid_constant__ DevIndex ix, uint32_t steps, uint32_t *__restrict__ rows) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    uint32_t r = 0;
    if (threadIdx.x == 0) rows[0] = 0;
    for (uint32_t i = 1; i <= steps; ++i) {
        r = lf_value<G, LAYOUT>(ix, tb, ix.bwt[r], r);
        if (threadIdx.x == 0) rows[i] = r;
    }
}

// =====================================================================================================
// element-wise operator calls
// =====================================================================================================
template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
occ_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ c, const long long *__restrict__ key, long long m,
           long long *__restrict__ out) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const long long q = (long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (q >= m) return;                                   // group-uniform
    long long k = key[q] + 1;                             // occ(c,key) = rank_c(key+1)
    k = k < 0 ? 0 : (k > (long long)ix.n ? (long long)ix.n : k);
    const uint32_t cc = c[q];
    const uint32_t v = lf_value<G, LAYOUT>(ix, tb, cc, (uint32_t)k);
    if ((threadIdx.x % G) == 0) out[q] = (long long)(v - tb.C[cc]);
}

template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
prev_range_kernel(const __grid_constant__ DevIndex ix, const long long *__restrict__ sp, const long long *__restrict__ ep,
                  const uint8_t *__restrict__ c, long long m, long long *__restrict__ sp1, long long *__restrict__ ep1) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const long long q = (long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (q >= m) return;
    uint32_t a = (uint32_t)sp[q], b = (uint32_t)ep[q], touched = 0;
    backward_step<G, LAYOUT, false>(ix, tb, c[q], a, b, touched);
    if ((threadIdx.x % G) == 0) { sp1[q] = a; ep1[q] = b; }
}

template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
interval_prev_range_kernel(const __grid_constant__ DevIndex ix, uint32_t sp, uint32_t ep, int cstart, int cend,
                           long long *__restrict__ sp1, long long *__restrict__ ep1) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const int q = blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (q > cend - cstart) return;
    uint32_t a = sp, b = ep, touched = 0;
    backward_step<G, LAYOUT, false>(ix, tb, (uint32_t)(cstart + q), a, b, touched);
    if ((threadIdx.x % G) == 0) { sp1[q] = a; ep1[q] = b; }
}

template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
lf_kernel(const __grid_constant__ DevIndex ix, const long long *__restrict__ row, long long m, long long *__restrict__ out) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const long long q = (long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (q >= m) return;
    const uint32_t r = (uint32_t)row[q];
    const uint32_t c = ix.bwt[r];                          // bwt[eof] is stored as 0
    const uint32_t v = lf_value<G, LAYOUT>(ix, tb, c, r);
    if ((threadIdx.x % G) == 0) out[q] = v;
}

template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
prev_substr_kernel(const __grid_constant__ DevIndex ix, const long long *__restrict__ row, long long m, int len,
                   uint8_t *__restrict__ out) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const long long q = (long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (q >= m) return;
    uint32_t r = (uint32_t)row[q];
    for (int k = 0; k < len; ++k) {
        const uint32_t c = ix.bwt[r];
        if ((threadIdx.x % G) == 0) out[q * len + k] = (uint8_t)c;
        r = lf_value<G, LAYOUT>(ix, tb, c, r);
    }
}

// ---- extract: the file bytes F[f .. f+len) = T'[q-1], T'[q-2], ... with q = n-1-f (fmx_text_batch / fmx_text_dev) --------------------
// One work item per segment of at most kTextSegment output bytes: output bytes [a, b) of request j are T' positions [q-b, q-a), reached
// from the sample at the first multiple of the sample rate at or above q-a (position n-1 = row 0 when that is past the text).  A step
// from position x (row r) emits T'[x-1], T'[x-2], ... and keeps those inside the segment's positions:
//   TEXT_ISAT: no walk — isat[p] holds T'[p .. p+isat_syms), independent loads from p = q-b on;
//   TEXT_CTX : ctx[2r+1] = { isa[x-J], T'[x-J .. x-1] } — J symbols and the row J positions back in one 16-byte request;
//   TEXT_CTX8: ctx8[r] = { isa[x-16], T'[x-16 .. x-1] as 2-bit codes }, LF steps for the last x < 16 positions (no hop there);
//   TEXT_LF  : one LF step per symbol (BWT byte + rank), as prevSubstr.
// STATS: *requests += the index requests the walks make (the sample, each entry / BWT byte / rank block).
enum { kTextIsat = 0, kTextCtx = 1, kTextCtx8 = 2, kTextLf = 3 };
constexpr int kTextSegment = 512;

// the byte of packed symbol k of a 96-bit isat / ctx field (e.y, e.z, e.w): dense code + 1 -> byte, or the byte itself (raw contexts)
__device__ __forceinline__ uint32_t text_sym(const uint4 &e, uint32_t k, uint32_t bits, bool raw, const uint8_t *sym) {
    const uint32_t o = k * bits, w = o >> 5;
    const uint32_t lo = w == 0 ? e.y : w == 1 ? e.z : e.w, hi = w == 0 ? e.z : w == 1 ? e.w : 0u;
    const uint32_t v = __funnelshift_r(lo, hi, o & 31u) & ((1u << bits) - 1u);
    return raw ? v : (uint32_t)sym[(v - 1u) & 0xFFu];
}

template <int G, int LAYOUT, int PATH, bool STATS>
__global__ void __launch_bounds__(kThreads)
text_kernel(const __grid_constant__ DevIndex ix, const uint32_t *__restrict__ off, long long m, int len, int nseg, uint8_t *__restrict__ out,
            int *__restrict__ out_len, unsigned long long *__restrict__ requests) {
    __shared__ SharedTables tb;
    __shared__ uint8_t sym[256];
    load_tables(tb, ix);
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sym[i] = ix.sym[i];
    __syncthreads();
    const uint32_t t = blockIdx.x * (kThreads / G) + threadIdx.x / G;     // < 2^31: the launcher slices larger batches
    if ((long long)t >= m * nseg) return;
    const bool lead = (threadIdx.x % G) == 0;
    const uint32_t j = t / (uint32_t)nseg;
    const int s = (int)(t - j * (uint32_t)nseg);
    const uint32_t f = off[j], last = ix.n - 1u;                  // |F| = n - 1
    if (f > last) {                                              // only the device form gets here unchecked
        if (s == 0 && lead) out_len[j] = -1;
        return;
    }
    const uint32_t q = last - f;
    const int olen = (int)min((uint32_t)len, q);
    if (s == 0 && lead) out_len[j] = olen;
    const int a = s * kTextSegment, b = min(a + kTextSegment, olen);
    if (a >= b) return;
    const uint32_t lo = q - (uint32_t)b, hi = q - (uint32_t)a;   // T' positions of this segment: [lo, hi)
    uint8_t *row = out + (long long)j * len;
#define FMX_PUT(P, V) (row[q - 1u - (P)] = (uint8_t)(V))            // T' position P is output byte q-1-P
    uint64_t req = 0;
    if constexpr (PATH == kTextIsat) {
        const uint32_t bits = (uint32_t)ix.isat_bits, syms = (uint32_t)ix.isat_syms;
        for (uint32_t p = lo; p < hi; p += syms) {
            const uint4 e = ldg128(ix.isat + p);
            const uint32_t cnt = min(syms, hi - p);
            for (uint32_t k = 0; k < cnt; ++k) FMX_PUT(p + k, text_sym(e, k, bits, false, sym));
            if (STATS) ++req;
        }
    } else {
        const uint32_t rate = ix.tsamp_rate;
        const uint64_t k0 = ((uint64_t)hi + rate - 1) / rate;
        uint64_t x64 = k0 * rate;                                // 64-bit: near n = 2^32 - 2 the multiple overflows uint32
        uint32_t r = 0;
        if (x64 > last) x64 = last;                              // position n-1 (the '$' suffix) is row 0
        else { r = ldg32(ix.tsamp + k0); if (STATS) ++req; }
        uint32_t x = (uint32_t)x64;
        if constexpr (PATH == kTextCtx) {
            const uint32_t J = (uint32_t)ix.ctx_J, bits = (uint32_t)ix.isat_bits;
            const bool raw = ix.ctx_raw != 0;
            while (x > lo) {
                const uint4 e = ldg128(ix.ctx + (uint64_t)r * 2 + 1);
                if (STATS) ++req;
                // symbol k of the entry is T'[x-J+k]; keep positions inside [lo, hi)
                const uint32_t kmin = x >= J ? (lo > x - J ? lo - (x - J) : 0u) : J - x + lo;
                const uint32_t kend = x <= hi ? J : x - hi >= J ? 0u : J - (x - hi);
                for (uint32_t k = kmin; k < kend; ++k) FMX_PUT(x - J + k, text_sym(e, k, bits, raw, sym));
                r = e.x;
                x = x > J ? x - J : 0u;
            }
        } else if constexpr (PATH == kTextCtx8) {
            constexpr uint32_t J = 16;
            while (x > lo && x >= J) {
                const uint2 e = ldg64(ix.ctx8 + r);
                if (STATS) ++req;
                const uint32_t kmin = lo > x - J ? lo - (x - J) : 0u, kend = x <= hi ? J : x - hi >= J ? 0u : J - (x - hi);
                for (uint32_t k = kmin; k < kend; ++k) FMX_PUT(x - J + k, sym[(e.y >> (2 * k)) & 3u]);
                r = e.x;
                x -= J;
            }
        }
        // LF steps: the whole walk (TEXT_LF), or the last x < 16 positions of a compact-context walk
        const uint32_t per_step = 1u + (LAYOUT == FMX_LAYOUT_WM ? (uint32_t)ix.levels : LAYOUT == FMX_LAYOUT_WMX ? (uint32_t)ix.wmx_levels : 1u);
        while (x > lo) {
            const uint32_t c = ix.bwt[r];
            if (x - 1u < hi && lead) FMX_PUT(x - 1u, c);
            if (--x > lo) { r = lf_value<G, LAYOUT>(ix, tb, c, r); if (STATS) req += per_step; }
            else if (STATS) ++req;
        }
    }
#undef FMX_PUT
    if (STATS && lead) atomicAdd(requests, (unsigned long long)req);
}

// FL step (getNextI, bwtmerger.scala:390-392: fm[i]) without the 4n-byte .fm array: the F-column symbol of row i
// is the c with C[c] <= i < C[c+1]; the answer is the row of its (i-C[c])-th occurrence in the BWT, found by
// binary search on rank_c.
template <int G, int LAYOUT>
__device__ __forceinline__ uint32_t fl_step(const DevIndex &ix, const SharedTables &tb, uint32_t i) {
    int lo = 0, hi = 255;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (tb.C[mid] <= i) lo = mid; else hi = mid - 1; }
    const uint32_t c = (uint32_t)lo;
    if (c == 0) return ix.eof;
    const uint32_t want = i - tb.C[c] + 1;
    uint32_t a = 0, b = ix.n - 1;
    while (a < b) {
        const uint32_t mid = a + ((b - a) >> 1);
        const uint32_t r = lf_value<G, LAYOUT>(ix, tb, c, mid + 1) - tb.C[c];
        if (r >= want) b = mid; else a = mid + 1;
    }
    return a;
}

template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
fl_kernel(const __grid_constant__ DevIndex ix, const long long *__restrict__ row, long long m, long long *__restrict__ out) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const long long q = (long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (q >= m) return;
    const uint32_t v = fl_step<G, LAYOUT>(ix, tb, (uint32_t)row[q]);
    if ((threadIdx.x % G) == 0) out[q] = v;
}

// nextSubstr (bwtmerger.scala:394-405): bytes in walk order (the host reverses them), stops after the '\0'
template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
next_substr_kernel(const __grid_constant__ DevIndex ix, const long long *__restrict__ row, long long m, int len,
                   uint8_t *__restrict__ out, int *__restrict__ out_len) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const long long q = (long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (q >= m) return;
    uint32_t cp = fl_step<G, LAYOUT>(ix, tb, (uint32_t)row[q]);
    int k = 0;
    for (; k < len; ++k) {
        const uint32_t b = ix.bwt[cp];
        if ((threadIdx.x % G) == 0) out[q * len + k] = (uint8_t)b;
        if (b == 0) { ++k; break; }
        cp = fl_step<G, LAYOUT>(ix, tb, cp);
    }
    if ((threadIdx.x % G) == 0) out_len[q] = k;
}

// =====================================================================================================
// K2: locate — one group per occurrence, LF-walk to the nearest sampled row
// =====================================================================================================
// One lane group per occurrence.  (Round 2 also tried a persistent form — a warp owning a chunk of occurrences, groups refilling as their
// walks end, the sample fetch deferred so that every round costs two dependent fetches: 334 ms instead of 286 ms for 4.9e8 occurrences.
// The walks are bound by the request rate, not by idle lanes: adjacent lanes start on adjacent rows and share walk / mark blocks,
// which the refill order gives up.)
template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
locate_kernel(const __grid_constant__ DevIndex ix, const uint32_t *__restrict__ sp, const long long *__restrict__ off,
              long long q0, long long q1, long long t0, long long count, uint32_t *__restrict__ pos, unsigned long long *__restrict__ key,
              unsigned long long *steps_out) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const long long t = (long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;      // slab-local occurrence
    if (t >= count) return;
    const long long T = t0 + t;                                                          // its place in the whole batch
    // owning query: last q in [q0, q1) with off[q] <= T (queries without occurrences share their offset with the next one)
    long long lo = q0, hi = q1;
    while (hi - lo > 1) { const long long mid = (lo + hi) >> 1; if (off[mid] <= T) lo = mid; else hi = mid; }
    uint32_t r = sp[lo] + (uint32_t)(T - off[lo]);
    // output: the position alone (a slab that is one query), or the sort key (query index inside the slab, position) of the per-query ordering
    const unsigned long long seg = (unsigned long long)(lo - q0) << 32;
#define FMX_EMIT(P) do { if ((threadIdx.x % G) == 0) { if (key) key[t] = seg | (unsigned long long)(P); else pos[t] = (P); } } while (0)
    if (ix.sa != nullptr) {                                    // full suffix array resident: one load per occurrence
        FMX_EMIT(ix.sa[r]);
        return;
    }
    uint32_t k = 0;
    if (ix.bm != nullptr) {                                    // fused walk blocks: BWT byte + mark bit in one fetch per step
        for (;;) {
            uint32_t c, marked;
            walk_block<G>(ix.bm, r, c, marked);
            if (marked) {
                const uint32_t mr = rank_one<G>(ix.mark, r, nullptr);
                FMX_EMIT(ix.samples[mr] + k);
                if ((threadIdx.x % G) == 0 && steps_out) atomicAdd(steps_out, (unsigned long long)k);
                return;
            }
            r = lf_value<G, LAYOUT>(ix, tb, c, r);
            if (++k > ix.n) { FMX_EMIT(0xFFFFFFFFu); return; }      // cannot happen on a consistent index (fmx_open checks)
        }
    }
    for (;;) {
        uint32_t bit;
        const uint32_t mr = rank_one<G>(ix.mark, r, &bit);
        if (bit) {                                         // row eof (sa = 0) is always sampled, so '$' is never stepped over
            FMX_EMIT(ix.samples[mr] + k);
            if ((threadIdx.x % G) == 0 && steps_out) atomicAdd(steps_out, (unsigned long long)k);
            return;
        }
        r = lf_value<G, LAYOUT>(ix, tb, ix.bwt[r], r);
        if (++k > ix.n) { FMX_EMIT(0xFFFFFFFFu); return; }
    }
#undef FMX_EMIT
}

// low words of the sorted (query, position) keys: the positions, ascending inside each query — as uint32 (device callers) or widened
// to the ABI's int64 (host callers)
template <typename OutT>
__global__ void key_positions_kernel(const unsigned long long *__restrict__ key, long long n, OutT *__restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (OutT)(key[i] & 0xFFFFFFFFull);
}
cudaError_t launch_key_positions(const uint64_t *d_key, int64_t n, uint32_t *d_out32, int64_t *d_out64, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)((n + 255) / 256);
    if (d_out32) key_positions_kernel<uint32_t><<<grid, 256, 0, st>>>((const unsigned long long *)d_key, n, d_out32);
    else key_positions_kernel<long long><<<grid, 256, 0, st>>>((const unsigned long long *)d_key, n, (long long *)d_out64);
    return cudaGetLastError();
}

// 2-bit symbol codes -> pattern bytes: thread t writes four consecutive bytes of one pattern (its packed byte t % ceil(len/4))
__global__ void unpack2_kernel(const uint8_t *__restrict__ codes, int len, long long m, uint32_t alpha4, uint8_t *__restrict__ out) {
    const int pb = (len + 3) >> 2;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m * pb) return;
    const long long q = t / pb;
    const int b = (int)(t - q * pb);
    const uint32_t c = codes[t];
    uint8_t *dst = out + q * len + 4 * b;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        if (4 * b + j < len) dst[j] = (uint8_t)(alpha4 >> (8 * ((c >> (2 * j)) & 3u)));
}
cudaError_t launch_unpack2(const uint8_t *d_codes, int len, int64_t m, uint32_t alpha4, uint8_t *d_out, cudaStream_t st) {
    const int64_t total = m * ((len + 3) / 4);
    if (total > 0) unpack2_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_codes, len, m, alpha4, d_out);
    return cudaGetLastError();
}

// occurrences per query (0 for an empty interval), as the scan input of the locate offsets; element m is 0
__global__ void interval_len_kernel(const uint32_t *__restrict__ sp, const uint32_t *__restrict__ ep, long long m, long long *__restrict__ out) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (q > m) return;
    out[q] = (q < m && ep[q] > sp[q]) ? (long long)(ep[q] - sp[q]) : 0ll;
}
cudaError_t launch_interval_len(const uint32_t *d_sp, const uint32_t *d_ep, int64_t m, int64_t *d_out, cudaStream_t st) {
    interval_len_kernel<<<(unsigned)((m + 1 + 255) / 256), 256, 0, st>>>(d_sp, d_ep, m, (long long *)d_out);
    return cudaGetLastError();
}

// Exchange step of the variable-length results (located positions, regex triples): this rank's slab of `count` 4-byte words goes
// straight into every rank's gathered buffer (peer-mapped memory over NVLink/NVSwitch) at word offset *d_dst_off — the scanned
// offset of this rank's first result, read on the device so no host round trip sits between the scan and the stores.
__global__ void __launch_bounds__(256)
scatter_words_kernel(const uint32_t *__restrict__ src, long long count, const __grid_constant__ PeerSinks sinks, const long long *__restrict__ d_dst_off,
                     long long dst_scale) {
    const long long dst0 = sinks.offset + (d_dst_off ? *d_dst_off * dst_scale : 0ll);
    const long long stride = (long long)gridDim.x * blockDim.x, tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (((reinterpret_cast<uintptr_t>(src) | (uintptr_t)(dst0 * 4)) & 15) == 0) {       // 16-byte pieces (peer buffers are cudaMalloc-aligned)
        const long long nv = count >> 2;
        for (long long i = tid; i < nv; i += stride) {
            const uint4 v = reinterpret_cast<const uint4 *>(src)[i];
            for (int j = 0; j < sinks.n; ++j) reinterpret_cast<uint4 *>(sinks.p[j] + dst0)[i] = v;
        }
        for (long long i = (nv << 2) + tid; i < count; i += stride) { const uint32_t v = src[i]; for (int j = 0; j < sinks.n; ++j) sinks.p[j][dst0 + i] = v; }
    } else {
        for (long long i = tid; i < count; i += stride) { const uint32_t v = src[i]; for (int j = 0; j < sinks.n; ++j) sinks.p[j][dst0 + i] = v; }
    }
}
cudaError_t launch_scatter_words(const uint32_t *d_src, int64_t count, const PeerSinks &sinks, const int64_t *d_dst_off, int64_t dst_scale, cudaStream_t st) {
    if (count <= 0 || sinks.n <= 0) return cudaSuccess;
    const unsigned grid = (unsigned)std::min<int64_t>((count / 4 + 255) / 256 + 1, 148 * 8);
    scatter_words_kernel<<<grid, 256, 0, st>>>(d_src, count, sinks, (const long long *)d_dst_off, dst_scale);
    return cudaGetLastError();
}

// =====================================================================================================
// K4: random gather microbenchmark (pointer-chase of `chain` dependent gathers per group)
// =====================================================================================================
template <int LANES, int VEC>     // VEC uint4 per lane; bytes per gather = LANES*VEC*16
__global__ void __launch_bounds__(kThreads)
gather_kernel(const uint4 *__restrict__ base, unsigned long long n_units, long long gathers, int chain, uint32_t seed,
              unsigned long long *sink) {
    const long long gid = ((long long)blockIdx.x * kThreads + threadIdx.x) / LANES;
    const int lane = threadIdx.x % LANES;
    if (gid >= gathers) return;
    unsigned long long x = (unsigned long long)gid * 0x9E3779B97F4A7C15ull + seed;
    uint32_t acc = 0;
    for (int s = 0; s < chain; ++s) {
        x ^= x >> 33; x *= 0xFF51AFD7ED558CCDull; x ^= x >> 33; x *= 0xC4CEB9FE1A85EC53ull; x ^= x >> 33;
        const unsigned long long unit = __umul64hi(x, n_units);          // unit = one gather-sized aligned chunk
        const uint4 *p = base + unit * (LANES * VEC) + lane * VEC;
        uint32_t v = 0;
#pragma unroll
        for (int i = 0; i < VEC; ++i) { const uint4 q = ldg128(p + i); v ^= q.x ^ q.y ^ q.z ^ q.w; }
        if (LANES > 1) {
            const uint32_t mask = ((LANES == 32) ? 0xFFFFFFFFu : ((1u << LANES) - 1u)) << ((threadIdx.x & 31) & ~(LANES - 1));
            for (int o = 1; o < LANES; o <<= 1) v ^= __shfl_xor_sync(mask, v, o);
        }
        acc ^= v;
        x += v;                                                       // next address depends on the loaded data
    }
    if (acc == 0x12345678u && lane == 0) atomicAdd(sink, 1ull);
}

// =====================================================================================================
// launchers
// =====================================================================================================
static inline unsigned grid_for(int64_t items, int lanes) {
    const int64_t per = kThreads / lanes;
    return (unsigned)((items + per - 1) / per);
}

cudaError_t launch_count_fixed(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_pat, int len, int64_t m, void *d_sp,
                               void *d_ep, bool out64, unsigned long long *d_stats, cudaStream_t st, const PeerSinks *sinks_or_null) {
    if (m <= 0) return cudaSuccess;
    if (cfg.count_lanes) cfg.lanes = cfg.count_lanes;
    PeerSinks sinks{};
    if (sinks_or_null) sinks = *sinks_or_null;
    // + 16: the 12-byte pattern windows of the row-context hops are read as whole words and may run past the last pattern
    const size_t smem = (size_t)(kThreads / cfg.lanes) * (size_t)(len > 0 ? len : 1) + 16;
    const bool too_long = smem > 160 * 1024;             // patterns of more than ~640 bytes per lane: read them from global memory
    if (ix.dict != nullptr && len > ix.kmer_k && len <= ix.dict_Dx && !d_stats && m < (1ll << kListModeShift) && (size_t)kThreads * (size_t)len <= 160 * 1024) {
        // two passes: the dictionary probe for everybody, the general search for what it leaves (compacted).  Only where the probe can
        // finish a query (len <= the deepest stored depth): longer patterns all go on with rank steps and the single kernel is balanced enough
        unsigned long long *cnt = nullptr;                     // [0] = list length, the list behind it
        cudaError_t e = cudaMallocAsync(&cnt, 16 + (size_t)m * 8, st);
        if (e != cudaSuccess) return e;
        uint2 *list = reinterpret_cast<uint2 *>(cnt + 2);
        cudaMemsetAsync(cnt, 0, 8, st);
        const size_t smem1 = (size_t)kThreads * (size_t)len;
        const unsigned grid1 = grid_for(m, 1);
        if (out64) {
            auto k = count_dict_first_kernel<long long>;
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1);
            k<<<grid1, kThreads, smem1, st>>>(ix, d_pat, len, m, (long long *)d_sp, (long long *)d_ep, list, cnt, sinks);
        } else {
            auto k = count_dict_first_kernel<uint32_t>;
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1);
            k<<<grid1, kThreads, smem1, st>>>(ix, d_pat, len, m, (uint32_t *)d_sp, (uint32_t *)d_ep, list, cnt, sinks);
        }
        const unsigned grid2 = grid_for(m, cfg.lanes);
        dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
            const size_t smem2 = (size_t)(kThreads / g) * (size_t)((len + 3) & ~3) + 16;
            if (out64) count_list_kernel<g, lay, long long><<<grid2, kThreads, smem2, st>>>(ix, d_pat, len, (long long *)d_sp, (long long *)d_ep, list, cnt, sinks);
            else count_list_kernel<g, lay, uint32_t><<<grid2, kThreads, smem2, st>>>(ix, d_pat, len, (uint32_t *)d_sp, (uint32_t *)d_ep, list, cnt, sinks);
        });
        cudaFreeAsync(cnt, st);
        return cudaGetLastError();
    }
    if (too_long && d_stats) return cudaErrorInvalidValue;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        if (too_long) {
            if (out64) count_fixed_gmem_kernel<g, lay, long long><<<grid_for(m, g), kThreads, 0, st>>>(ix, d_pat, len, m, (long long *)d_sp, (long long *)d_ep, sinks);
            else count_fixed_gmem_kernel<g, lay, uint32_t><<<grid_for(m, g), kThreads, 0, st>>>(ix, d_pat, len, m, (uint32_t *)d_sp, (uint32_t *)d_ep, sinks);
        } else if (d_stats) {
            auto k = count_fixed_kernel<g, lay, true, uint32_t>;
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k<<<grid_for(m, g), kThreads, smem, st>>>(ix, d_pat, len, m, (uint32_t *)d_sp, (uint32_t *)d_ep, d_stats, sinks);
        } else if (out64) {
            auto k = count_fixed_kernel<g, lay, false, long long>;
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k<<<grid_for(m, g), kThreads, smem, st>>>(ix, d_pat, len, m, (long long *)d_sp, (long long *)d_ep, nullptr, sinks);
        } else {
            auto k = count_fixed_kernel<g, lay, false, uint32_t>;
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k<<<grid_for(m, g), kThreads, smem, st>>>(ix, d_pat, len, m, (uint32_t *)d_sp, (uint32_t *)d_ep, nullptr, sinks);
        }
    });
    return cudaGetLastError();
}

cudaError_t launch_count_var(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_pat, const int64_t *d_off, int64_t m,
                             int64_t *d_sp, int64_t *d_ep, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    if (cfg.count_lanes) cfg.lanes = cfg.count_lanes;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        count_var_kernel<g, lay><<<grid_for(m, g), kThreads, 0, st>>>(ix, d_pat, (const long long *)d_off, m, (long long *)d_sp, (long long *)d_ep);
    });
    return cudaGetLastError();
}

cudaError_t launch_match(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_pat, const int64_t *d_off, int64_t m, int32_t *d_len,
                         uint32_t *d_sp, uint32_t *d_ep, uint32_t *d_flag, int min_len, unsigned long long *d_stats, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    if (ix.lcp8 == nullptr) return cudaErrorInvalidValue;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        if (d_stats) match_kernel<g, lay, true><<<grid_for(m, g), kThreads, 0, st>>>(ix, d_pat, (const long long *)d_off, m, d_len, d_sp, d_ep, d_flag, min_len, d_stats);
        else match_kernel<g, lay, false><<<grid_for(m, g), kThreads, 0, st>>>(ix, d_pat, (const long long *)d_off, m, d_len, d_sp, d_ep, d_flag, min_len, nullptr);
    });
    return cudaGetLastError();
}

cudaError_t launch_smem_offsets(const uint32_t *d_scan, const int64_t *d_off, int64_t m, int64_t *d_out_off, cudaStream_t st) {
    smem_offsets_kernel<<<(unsigned)((m + 1 + 255) / 256), 256, 0, st>>>(d_scan, (const long long *)d_off, m, (long long *)d_out_off);
    return cudaGetLastError();
}

cudaError_t launch_smem_compact(const uint32_t *d_flag, const uint32_t *d_scan, const int32_t *d_ms_len, const uint32_t *d_ms_sp,
                                const uint32_t *d_ms_ep, const int64_t *d_off, int64_t m, int64_t T, int32_t *d_start, int32_t *d_len,
                                uint32_t *d_sp, uint32_t *d_ep, cudaStream_t st) {
    if (T <= 0 || m <= 0) return cudaSuccess;
    smem_compact_kernel<<<(unsigned)((T + 255) / 256), 256, 0, st>>>(d_flag, d_scan, d_ms_len, d_ms_sp, d_ms_ep, (const long long *)d_off, m, T,
                                                                     d_start, d_len, d_sp, d_ep);
    return cudaGetLastError();
}

int64_t census_tiles(int64_t n) { return ((n + kLcpRows - 1) / kLcpRows + kCensusTile - 1) / kCensusTile; }

// a grid-stride grid of at most what is resident at once, so that the spectrum's shared histogram is flushed once per resident CTA
template <typename K> static unsigned census_grid(K kernel, int64_t ntiles) {
    int dev = 0, sms = 148, per_sm = 1;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kThreads, 0);
    const int64_t want = (ntiles + kThreads / 32 - 1) / (kThreads / 32);
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sms * std::max(per_sm, 1)));
}

cudaError_t launch_census_last(const DevIndex &ix, uint32_t k, uint32_t *d_tile_last, cudaStream_t st) {
    if (ix.lcp8 == nullptr) return cudaErrorInvalidValue;
    const int64_t ntiles = census_tiles(ix.n);
    census_last_kernel<<<census_grid(census_last_kernel, ntiles), kThreads, 0, st>>>(ix, (uint32_t)((ix.n + kLcpRows - 1) / kLcpRows),
                                                                                  (uint32_t)ntiles, k, d_tile_last);
    return cudaGetLastError();
}

cudaError_t launch_census_spectrum(const DevIndex &ix, uint32_t k, const uint32_t *d_tile_incl, uint32_t buckets, unsigned long long *d_hist,
                                   unsigned long long *d_max, cudaStream_t st) {
    if (ix.lcp8 == nullptr) return cudaErrorInvalidValue;
    const int64_t ntiles = census_tiles(ix.n);
    auto kern = census_kernel<kCensusSpectrum>;
    kern<<<census_grid(kern, ntiles), kThreads, 0, st>>>(ix, (uint32_t)((ix.n + kLcpRows - 1) / kLcpRows), (uint32_t)ntiles, k, d_tile_incl,
                                                         buckets, d_hist, d_max, 0, 0, nullptr, 0, nullptr, nullptr, nullptr, nullptr);
    return cudaGetLastError();
}

cudaError_t launch_census_list(const DevIndex &ix, uint32_t k, const uint32_t *d_tile_incl, uint32_t min_count, uint32_t max_count,
                               const uint32_t *d_ex, uint32_t nex, uint32_t *d_tile_cnt, const uint32_t *d_tile_off, uint32_t *d_sp,
                               uint32_t *d_ep, cudaStream_t st) {
    if (ix.lcp8 == nullptr) return cudaErrorInvalidValue;
    const int64_t ntiles = census_tiles(ix.n);
    const uint32_t nb = (uint32_t)((ix.n + kLcpRows - 1) / kLcpRows);
    auto kern = d_tile_off ? census_kernel<kCensusEmit> : census_kernel<kCensusCount>;
    kern<<<census_grid(kern, ntiles), kThreads, 0, st>>>(ix, nb, (uint32_t)ntiles, k, d_tile_incl, 1, nullptr, nullptr, min_count, max_count,
                                                         d_ex, nex, d_tile_cnt, d_tile_off, d_sp, d_ep);
    return cudaGetLastError();
}

cudaError_t launch_census_walk(const DevIndex &ix, LaunchCfg cfg, uint32_t steps, uint32_t *d_rows, cudaStream_t st) {
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) { census_walk_kernel<g, lay><<<1, (unsigned)g, 0, st>>>(ix, steps, d_rows); });
    return cudaGetLastError();
}

cudaError_t launch_occ(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_c, const int64_t *d_key, int64_t m, int64_t *d_out,
                       cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        occ_kernel<g, lay><<<grid_for(m, g), kThreads, 0, st>>>(ix, d_c, (const long long *)d_key, m, (long long *)d_out);
    });
    return cudaGetLastError();
}

cudaError_t launch_prev_range(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_sp, const int64_t *d_ep, const uint8_t *d_c,
                              int64_t m, int64_t *d_sp1, int64_t *d_ep1, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        prev_range_kernel<g, lay><<<grid_for(m, g), kThreads, 0, st>>>(ix, (const long long *)d_sp, (const long long *)d_ep, d_c, m, (long long *)d_sp1, (long long *)d_ep1);
    });
    return cudaGetLastError();
}

cudaError_t launch_interval_prev_range(const DevIndex &ix, LaunchCfg cfg, int64_t sp, int64_t ep, int cstart, int cend,
                                       int64_t *d_sp1, int64_t *d_ep1, cudaStream_t st) {
    const int64_t m = cend - cstart + 1;
    if (m <= 0) return cudaSuccess;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        interval_prev_range_kernel<g, lay><<<grid_for(m, g), kThreads, 0, st>>>(ix, (uint32_t)sp, (uint32_t)ep, cstart, cend, (long long *)d_sp1, (long long *)d_ep1);
    });
    return cudaGetLastError();
}

cudaError_t launch_lf(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_row, int64_t m, int64_t *d_out, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        lf_kernel<g, lay><<<grid_for(m, g), kThreads, 0, st>>>(ix, (const long long *)d_row, m, (long long *)d_out);
    });
    return cudaGetLastError();
}

cudaError_t launch_prev_substr(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_row, int64_t m, int len, uint8_t *d_out,
                               cudaStream_t st) {
    if (m <= 0 || len <= 0) return cudaSuccess;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        prev_substr_kernel<g, lay><<<grid_for(m, g), kThreads, 0, st>>>(ix, (const long long *)d_row, m, len, d_out);
    });
    return cudaGetLastError();
}

int text_path(const DevIndex &ix) {
    return ix.isat != nullptr ? kTextIsat : ix.tsamp == nullptr ? -1 : ix.ctx != nullptr ? kTextCtx : ix.ctx8 != nullptr ? kTextCtx8 : kTextLf;
}

cudaError_t launch_text(const DevIndex &ix, LaunchCfg cfg, const uint32_t *d_off, int64_t m, int len, uint8_t *d_out, int *d_out_len,
                        unsigned long long *d_requests, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    const int path = text_path(ix);
    if (path < 0) return cudaErrorInvalidValue;
    const int nseg = len > 0 ? (len + kTextSegment - 1) / kTextSegment : 1;
    const int64_t slice = (1ll << 30) / nseg;                     // requests per launch: the kernel's work-item indices stay 32-bit
    for (int64_t j0 = 0; j0 < m; j0 += slice) {
        const int64_t mj = std::min(slice, m - j0);
        auto text = [&](auto g, auto lay, auto p) {
            if (d_requests) text_kernel<g, lay, p, true><<<grid_for(mj * nseg, g), kThreads, 0, st>>>(ix, d_off + j0, mj, len, nseg, d_out + j0 * len, d_out_len + j0, d_requests);
            else text_kernel<g, lay, p, false><<<grid_for(mj * nseg, g), kThreads, 0, st>>>(ix, d_off + j0, mj, len, nseg, d_out + j0 * len, d_out_len + j0, nullptr);
        };
        // the hop paths are one lane per segment (one request per entry); the LF walk shares each rank block among cfg.lanes lanes
        using One = std::integral_constant<int, 1>;
        using Planes = std::integral_constant<int, FMX_LAYOUT_PLANES>;
        if (path == kTextIsat) text(One{}, Planes{}, std::integral_constant<int, kTextIsat>{});
        else if (path == kTextCtx) text(One{}, Planes{}, std::integral_constant<int, kTextCtx>{});
        else if (path == kTextCtx8) dispatch_layout(cfg.layout, [&](auto lay) { text(One{}, lay, std::integral_constant<int, kTextCtx8>{}); });
        else dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) { text(g, lay, std::integral_constant<int, kTextLf>{}); });
    }
    return cudaGetLastError();
}

cudaError_t launch_fl(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_row, int64_t m, int64_t *d_out, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        fl_kernel<g, lay><<<grid_for(m, g), kThreads, 0, st>>>(ix, (const long long *)d_row, m, (long long *)d_out);
    });
    return cudaGetLastError();
}

cudaError_t launch_next_substr(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_row, int64_t m, int len, uint8_t *d_out,
                               int *d_out_len, cudaStream_t st) {
    if (m <= 0) return cudaSuccess;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        next_substr_kernel<g, lay><<<grid_for(m, g), kThreads, 0, st>>>(ix, (const long long *)d_row, m, len, d_out, d_out_len);
    });
    return cudaGetLastError();
}

cudaError_t launch_locate(const DevIndex &ix, LaunchCfg cfg, const uint32_t *d_sp, const int64_t *d_off, int64_t q0, int64_t q1,
                          int64_t t0, int64_t count, uint32_t *d_pos, uint64_t *d_key, unsigned long long *d_steps, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        locate_kernel<g, lay><<<grid_for(count, g), kThreads, 0, st>>>(ix, d_sp, (const long long *)d_off, q0, q1, t0, count, d_pos, (unsigned long long *)d_key, d_steps);
    });
    return cudaGetLastError();
}

cudaError_t launch_gather_bench(const uint4 *base, uint64_t n_blocks64, int bytes, int lanes, int64_t gathers, int chain,
                                uint32_t seed, unsigned long long *d_sink, cudaStream_t st) {
    const int per_lane = bytes / lanes;                    // bytes each lane loads
    if (per_lane < 16 || per_lane % 16 || (per_lane / 16) > 8 || lanes < 1 || lanes > 32 || (lanes & (lanes - 1))) return cudaErrorInvalidValue;
    const int vec = per_lane / 16;
    const unsigned long long units = n_blocks64 * 64ull / (unsigned long long)bytes;
    const unsigned grid = (unsigned)((gathers * lanes + kThreads - 1) / kThreads);
#define GK(L, V) gather_kernel<L, V><<<grid, kThreads, 0, st>>>(base, units, gathers, chain, seed, d_sink)
    if (vec == 1) { switch (lanes) { case 1: GK(1, 1); break; case 2: GK(2, 1); break; case 4: GK(4, 1); break; case 8: GK(8, 1); break; case 16: GK(16, 1); break; default: GK(32, 1); } }
    else if (vec == 2) { switch (lanes) { case 1: GK(1, 2); break; case 2: GK(2, 2); break; case 4: GK(4, 2); break; case 8: GK(8, 2); break; default: return cudaErrorInvalidValue; } }
    else if (vec == 4) { switch (lanes) { case 1: GK(1, 4); break; case 2: GK(2, 4); break; case 4: GK(4, 4); break; default: return cudaErrorInvalidValue; } }
    else if (vec == 8) { switch (lanes) { case 1: GK(1, 8); break; case 2: GK(2, 8); break; default: return cudaErrorInvalidValue; } }
    else return cudaErrorInvalidValue;
#undef GK
    return cudaGetLastError();
}

}  // namespace fmx

// fmx_regex_kernel.cu — K3: traversal of the position automata over SA intervals.
//
//   ReTree._matchSA      re2/retree.scala:618-653   (StatePoint :562-567, start items :576)
//   REParser.matchSA     re2/re2.scala:568-693      (Thompson positions: emit and go on)
//   DFA.matchSA          dfa.scala:261-289
//
// The reference pops (len, sp, ep, state) items from a priority queue, takes one getPrevRange step (findex.scala:32-36) with the
// state's character and either emits a result or pushes the state's follow positions.  With the caps off the result is a multiset
// that does not depend on the order in which items are taken, so nothing here is level-synchronous:
//
//   * every warp keeps a stack of items in shared memory: children go there (no atomics, nobody else sees them) and idle lanes pop it
//     first; only what does not fit spills to the global ring, and only a warp whose stack is empty takes work from it.  The balance
//     of births and deaths a warp has not reported to `pending` is flushed whenever it turns positive (before a child could become
//     visible to others) and when the warp runs dry, so `pending` never undercounts and most iterations touch no global counter.
//   * a persistent grid of workers (G lanes per item) owns a global RING of items in HBM (start items, overflow of the stacks): a
//     bounded MPMC queue with a sequence word per slot.  Consumers take tickets from `head` with one
//     warp-aggregated atomic and wait for their slot to be filled; producers reserve tickets from `tail` the same way, write the
//     payload and publish it with a release exchange on the slot's state word (an occupied slot = the ring is too small: the run is
//     abandoned and the host reruns it with a larger ring).  `pending` counts live items; the worker that brings it to zero raises `done`.
//   * depth first where it is free: an item whose state has 1..3 follow positions goes on with the first one in its own registers
//     (a literal run never touches the ring) and pushes only the others; the per-state record (character, flags, follow list) is one
//     16-byte load, and the record of the first follow is fetched together with the rank blocks of the step.
//   * wide follow lists (classes, '.', big alternations) are expanded by the whole warp, one parent at a time, and filtered: a follow
//     position with character c survives its backward step iff c occurs in BWT[sp..ep), so for an interval of <= 32 rows only the
//     positions whose character is there are pushed — identical results, and a '.' after a one-row interval costs 1 item, not 253.
//   * matches are appended to the result array with one atomic per warp; the caller sorts them by (regex, len, sp, ep).
//
// There is no grid barrier and no cooperative launch; a lane that runs out of work refills from the ring while its neighbours go on.
#include "fmx_kernels.cuh"

#include <algorithm>
#include <atomic>

namespace fmx {

namespace {

// The ring is a bounded multi-producer / multi-consumer queue with one sequence word per slot (Vyukov): slot i starts at seq = i; the
// producer of ticket t may write slot t & mask only while seq == t, and publishes with seq = t + 1; the consumer of ticket t waits for
// seq == t + 1, reads the item and frees the slot for the next lap with seq = t + capacity.  Tickets that alias a slot (t and
// t + capacity) can therefore never see each other's item, however many consumers wait; a producer that finds its slot not yet freed
// reports the ring as too small.
__device__ __forceinline__ uint32_t ld_acquire(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ld_relaxed(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(uint32_t *p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint4 ld_cg(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.cg.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    return r;
}
__device__ __forceinline__ unsigned long long ld_volatile_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// publish one item at ticket `t`.  Returns false if the slot has not been freed by the consumer of the previous lap (ring too small).
__device__ __forceinline__ bool ring_publish(FrontierItem *ring, uint32_t *seq, unsigned long long mask, unsigned long long t, uint32_t state,
                                             uint32_t len, uint32_t sp, uint32_t ep) {
    const unsigned long long i = t & mask;
    if (ld_acquire(seq + i) != (uint32_t)t) return false;
    *reinterpret_cast<uint4 *>(ring + i) = make_uint4(state, len, sp, ep);
    st_release(seq + i, (uint32_t)t + 1u);
    return true;
}

}  // namespace

// ctrl (8 x u64, zeroed by the caller): see RegexCtrl in fmx_kernels.cuh
__global__ void regex_seed_kernel(const uint32_t *__restrict__ first, long long n_first, uint32_t n, FrontierItem *ring, uint32_t *seq, long long cap,
                                  unsigned long long *ctrl) {
    // level-0 items: StatePoint(0, 0, sa.n, state) for every first position  (retree.scala:576) = tickets 0 .. n_first-1, already published
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (long long)gridDim.x * blockDim.x) {
        if (i < n_first) ring[i] = FrontierItem{first[i], 0u, 0u, n};
        seq[i] = (uint32_t)i + (i < n_first ? 1u : 0u);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        ctrl[kRxHead] = 0; ctrl[kRxTail] = (unsigned long long)n_first; ctrl[kRxPending] = (unsigned long long)n_first;
        ctrl[kRxMatches] = 0; ctrl[kRxStatus] = 0; ctrl[kRxDone] = n_first == 0 ? 1ull : 0ull; ctrl[kRxMaxLen] = 0; ctrl[kRxSteps] = 0;
    }
}

constexpr int kLocalSlots = 256;           // per-warp stack of items in shared memory (one '.' expansion = 253 children fits)

template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
regex_queue_kernel(const __grid_constant__ DevIndex ix, const __grid_constant__ RegexTables rt, FrontierItem *ring, uint32_t *seq, unsigned long long ring_mask,
                   RegexResult *__restrict__ res, long long cap_res, unsigned long long *ctrl, uint32_t len_cap, uint32_t local_keep) {
    __shared__ SharedTables tb;
    __shared__ __align__(16) FrontierItem lstack[kThreads / 32][kLocalSlots];
    load_tables(tb, ix);
    __syncthreads();
    const uint32_t lane = threadIdx.x & 31;
    const bool leader = (threadIdx.x % G) == 0;
    const int lead_lane = (int)(lane & ~(uint32_t)(G - 1));
    FrontierItem *mine = lstack[threadIdx.x >> 5];
    constexpr uint32_t kWide = 4, kFilterRows = 32;
    constexpr unsigned long long kNoTicket = ~0ull;

    bool have = false, have_rec = false;                   // an item in registers / its state record already loaded
    unsigned long long ticket = kNoTicket;
    FrontierItem it = {0, 0, 0, 0};
    uint4 rec = {0, 0, 0, 0};
    uint32_t max_len = 0, idle_rounds = 0, nsteps = 0;
    uint32_t ltop = 0;                                     // items on this warp's stack (warp-uniform)
    long long ldelta = 0;                                  // births - deaths this warp has not told `pending` about yet (never left > 0)
    bool ring_ok = true;

    // children of this iteration go to the warp's own stack while it has room (no atomics, nobody else sees them) and to the global ring
    // beyond that; `idx` = position of the child among the `total` children pushed together
    auto place = [&](uint32_t idx, unsigned long long tbase, uint32_t room, uint32_t state, uint32_t len, uint32_t sp, uint32_t ep) {
        if (idx < room) mine[ltop + idx] = FrontierItem{state, len, sp, ep};
        else ring_ok = ring_publish(ring, seq, ring_mask, tbase + (idx - room), state, len, sp, ep) && ring_ok;
    };

    for (;;) {
        // ---- refill: (1) a lane that holds a ticket of the global ring looks at its slot; (2) lanes still without an item pop the warp's
        // own stack (a ticket holder too — its ring item, should it arrive meanwhile, waits for the lane's next refill); (3) lanes
        // without item and ticket take tickets (one atomic per warp) once the stack is empty
        auto poll = [&]() {
            if (leader && !have && ticket != kNoTicket) {
                const unsigned long long i = ticket & ring_mask;
                // waiting costs a relaxed load per round (no fence); the acquire is paid once, when the slot has been filled
                if (ld_relaxed(seq + i) == (uint32_t)ticket + 1u) {
                    (void)ld_acquire(seq + i);
                    const uint4 raw = ld_cg(reinterpret_cast<const uint4 *>(ring + i));
                    it = FrontierItem{raw.x, raw.y, raw.z, raw.w};
                    st_release(seq + i, (uint32_t)ticket + (uint32_t)(ring_mask + 1ull));      // the slot is free for the next lap (after the read above)
                    have = true;
                    have_rec = false;
                    ticket = kNoTicket;
                }
            }
        };
        poll();
        {
            const uint32_t want = __ballot_sync(0xFFFFFFFFu, leader && !have);
            if (want && ltop) {
                const uint32_t rank = __popc(want & ((1u << lane) - 1u));
                const uint32_t take = min((uint32_t)__popc(want), ltop);
                if (leader && !have && rank < take) { it = mine[ltop - 1 - rank]; have = true; have_rec = false; }
                ltop -= take;
            }
        }
        if (ltop == 0) {
            const uint32_t want = __ballot_sync(0xFFFFFFFFu, leader && !have && ticket == kNoTicket);
            if (want) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(&ctrl[kRxHead], (unsigned long long)__popc(want));
                base = __shfl_sync(0xFFFFFFFFu, base, 0);
                if (leader && !have && ticket == kNoTicket) ticket = base + __popc(want & ((1u << lane) - 1u));
                poll();
            }
        }
        if (G > 1) {                                       // the group works on its leader's item
            have = __shfl_sync(0xFFFFFFFFu, (int)have, lead_lane) != 0;
            it.state = __shfl_sync(0xFFFFFFFFu, it.state, lead_lane); it.len = __shfl_sync(0xFFFFFFFFu, it.len, lead_lane);
            it.sp = __shfl_sync(0xFFFFFFFFu, it.sp, lead_lane); it.ep = __shfl_sync(0xFFFFFFFFu, it.ep, lead_lane);
            have_rec = __shfl_sync(0xFFFFFFFFu, (int)have_rec, lead_lane) != 0;
        }
        if (!__any_sync(0xFFFFFFFFu, have)) {              // nothing to do in this warp (its stack is empty too): report, then done or wait
            if (ldelta != 0) {
                if (lane == 0) {
                    const unsigned long long old = atomicAdd(&ctrl[kRxPending], (unsigned long long)ldelta);
                    if (old + (unsigned long long)ldelta == 0ull) atomicExch(&ctrl[kRxDone], 1ull);      // the last live item ended here
                }
                ldelta = 0;
            }
            if (ld_volatile_u64(&ctrl[kRxDone]) != 0) break;
            if (++idle_rounds > 4) __nanosleep(idle_rounds > 64 ? 400 : 100);
            continue;
        }
        idle_rounds = 0;

        // ---- one backward step per item: getPrevRange(sp, ep, c)
        if (have && !have_rec) rec = ldg128(rt.rec + it.state);
        const uint32_t c = rec.x & 0xFFu, flags = (rec.x >> 8) & 0xFFu, fo = rec.y, nf_all = rec.z, f0 = rec.w;
        uint4 nrec = {0, 0, 0, 0};
        if (have && nf_all >= 1 && nf_all < kWide) nrec = ldg128(rt.rec + f0);      // in flight together with the rank blocks
        bool alive = have;
        if (have && leader) ++nsteps;
        if (have) {
            uint32_t touched = 0;
            backward_step<G, LAYOUT, false>(ix, tb, c, it.sp, it.ep, touched);
            alive = it.sp < it.ep;
        }
        const uint32_t nlen = it.len + 1;
        const bool emits = alive && (flags & 1u);
        const bool stop = emits && (flags & 2u);            // Glushkov: a last position emits and is not expanded (retree.scala:640-643)
        const bool too_deep = alive && nlen > ix.n;         // cannot happen for a match inside the text; guards runaway automata
        // REParser.matchSA's maxLength (re2.scala:636-641): follow positions are enqueued only while their len stays below it
        const uint32_t nf = (alive && !stop && !too_deep && (len_cap == 0u || nlen < len_cap)) ? nf_all : 0u;
        if (too_deep && leader) atomicMax(&ctrl[kRxStatus], 2ull);
        if (alive && nlen > max_len) max_len = nlen;

        // matches: ballot + one atomic per warp
        const uint32_t mm = __ballot_sync(0xFFFFFFFFu, emits && leader);
        if (mm) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(&ctrl[kRxMatches], (unsigned long long)__popc(mm));
            base = __shfl_sync(0xFFFFFFFFu, base, 0);
            if (emits && leader) {
                const unsigned long long idx = base + __popc(mm & ((1u << lane) - 1u));
                if (idx < (unsigned long long)cap_res) res[idx] = RegexResult{rt.st_regex[it.state], nlen, it.sp, it.ep};
            }
        }

        // deaths of this iteration: items that neither go on in their lane nor were expanded (wide parents end after their expansion)
        const bool narrow = leader && nf >= 1 && nf < kWide;
        const uint32_t np = narrow ? nf - 1 : 0u;            // children this group pushes (its first follow stays in the lane)
        uint32_t incl = np;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o); if (lane >= (uint32_t)o) incl += v; }
        const uint32_t pushes = __shfl_sync(0xFFFFFFFFu, incl, 31);
        const uint32_t finished = __popc(__ballot_sync(0xFFFFFFFFu, leader && have && !(nf >= 1 && nf < kWide)));
        uint32_t wide = __ballot_sync(0xFFFFFFFFu, leader && nf >= kWide);

        // ---- wide follow lists: the whole warp expands one parent at a time, filtered by the bytes present in BWT[sp..ep)
        while (wide) {
            const int src = __ffs(wide) - 1;
            wide &= wide - 1;
            const uint32_t cnt = __shfl_sync(0xFFFFFFFFu, nf, src), fs = __shfl_sync(0xFFFFFFFFu, fo, src);
            const uint32_t a = __shfl_sync(0xFFFFFFFFu, it.sp, src), e = __shfl_sync(0xFFFFFFFFu, it.ep, src), ln = __shfl_sync(0xFFFFFFFFu, nlen, src);
            const bool filt = (e - a) <= kFilterRows;
            uint32_t present = 0;                           // lane w (0..7) holds bits 32w..32w+31 of the set of bytes in BWT[a..e)
            if (filt) {
                const bool has = lane < (e - a);
                const uint32_t ch = has ? (uint32_t)ix.bwt[a + lane] : 0u;
#pragma unroll
                for (uint32_t w = 0; w < 8; ++w) {
                    const uint32_t r = __reduce_or_sync(0xFFFFFFFFu, (has && (ch >> 5) == w) ? (1u << (ch & 31u)) : 0u);
                    if (lane == w) present = r;
                }
            }
            uint32_t kept_total = cnt;
            if (filt) {
                kept_total = 0;
                for (uint32_t j0 = 0; j0 < cnt; j0 += 32) {
                    const uint32_t j = j0 + lane;
                    const uint32_t ch = j < cnt ? (ldg128(rt.rec + rt.fol[fs + j]).x & 0xFFu) : 0u;
                    const uint32_t word = __shfl_sync(0xFFFFFFFFu, present, ch >> 5);
                    kept_total += __popc(__ballot_sync(0xFFFFFFFFu, j < cnt && ((word >> (ch & 31u)) & 1u)));
                }
            }
            if (kept_total == 0) continue;                  // warp-uniform
            // births are counted before anybody else can see them: the running balance is flushed whenever it turns positive
            ldelta += kept_total;
            const uint32_t room = min(local_keep > ltop ? local_keep - ltop : 0u, kept_total);
            unsigned long long tb0 = 0;
            if (lane == 0) {
                if (ldelta > 0) atomicAdd(&ctrl[kRxPending], (unsigned long long)ldelta);
                if (kept_total > room) tb0 = atomicAdd(&ctrl[kRxTail], (unsigned long long)(kept_total - room));
            }
            if (ldelta > 0) ldelta = 0;
            tb0 = __shfl_sync(0xFFFFFFFFu, tb0, 0);
            uint32_t done_cnt = 0;
            for (uint32_t j0 = 0; j0 < cnt; j0 += 32) {
                const uint32_t j = j0 + lane;
                const uint32_t fstate = j < cnt ? rt.fol[fs + j] : 0u;
                bool keep = j < cnt;
                if (filt) {
                    const uint32_t ch = j < cnt ? (ldg128(rt.rec + fstate).x & 0xFFu) : 0u;
                    const uint32_t word = __shfl_sync(0xFFFFFFFFu, present, ch >> 5);
                    keep = keep && ((word >> (ch & 31u)) & 1u);
                }
                const uint32_t km = __ballot_sync(0xFFFFFFFFu, keep);
                if (keep) place(done_cnt + __popc(km & ((1u << lane) - 1u)), tb0, room, fstate, ln, a, e);
                done_cnt += __popc(km);
            }
            ltop += room;
            __syncwarp();
        }

        // ---- short follow lists: go on with the first follow in registers, push the others; settle the balance
        ldelta += (long long)pushes - (long long)finished;
        {
            const uint32_t room = min(local_keep > ltop ? local_keep - ltop : 0u, pushes);
            unsigned long long tb0 = 0;
            if (lane == 0) {
                if (ldelta > 0) atomicAdd(&ctrl[kRxPending], (unsigned long long)ldelta);
                if (pushes > room) tb0 = atomicAdd(&ctrl[kRxTail], (unsigned long long)(pushes - room));
            }
            if (ldelta > 0) ldelta = 0;
            if (pushes) {
                tb0 = __shfl_sync(0xFFFFFFFFu, tb0, 0);
                for (uint32_t j = 0; j < np; ++j) place(incl - np + j, tb0, room, rt.fol[fo + 1 + j], nlen, it.sp, it.ep);
                ltop += room;
                __syncwarp();
            }
        }
        if (have) {
            if (nf >= 1 && nf < kWide) { it.state = f0; it.len = nlen; rec = nrec; have_rec = true; }
            else have = false;
        }
        if (!__all_sync(0xFFFFFFFFu, ring_ok)) {             // an unread slot was overwritten: abandon the run, the host regrows the ring
            if (lane == 0) { atomicMax(&ctrl[kRxStatus], 1ull); atomicExch(&ctrl[kRxDone], 1ull); }
            break;
        }
    }
    for (int o = 16; o; o >>= 1) max_len = max(max_len, __shfl_xor_sync(0xFFFFFFFFu, max_len, o));
    for (int o = 16; o; o >>= 1) nsteps += __shfl_xor_sync(0xFFFFFFFFu, nsteps, o);
    if (lane == 0 && max_len) atomicMax(&ctrl[kRxMaxLen], (unsigned long long)max_len);
    if (lane == 0 && nsteps) atomicAdd(&ctrl[kRxSteps], (unsigned long long)nsteps);       // backward steps taken = items processed
}

std::atomic<int> g_regex_local_keep{kLocalSlots};          // measured on 100 k cfg-4 regexes: 0 -> 1.02 ms, 64 -> 0.84, 256 (everything local) -> 0.72
void set_regex_local_keep(int v) { g_regex_local_keep = v; }

cudaError_t launch_regex_search(const DevIndex &ix, LaunchCfg cfg, const RegexTables &rt, const uint32_t *d_first, int64_t n_first,
                                FrontierItem *d_ring, uint32_t *d_seq, int64_t ring_cap, RegexResult *d_res, int64_t cap_res,
                                unsigned long long *d_ctrl, uint32_t max_len, cudaStream_t st) {
    if (ring_cap < n_first || (ring_cap & (ring_cap - 1))) return cudaErrorInvalidValue;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    regex_seed_kernel<<<(unsigned)std::min<int64_t>((ring_cap + 255) / 256, sms * 8), 256, 0, st>>>(d_first, n_first, ix.n, d_ring, d_seq, ring_cap, d_ctrl);
    if (n_first <= 0) return cudaGetLastError();
    // children a warp keeps on its own stack; what exceeds it goes to the global ring where idle warps find it (a '.' expansion is 253
    // children: all-local leaves the other warps idle, all-global pays an atomic round trip per child)
    const uint32_t local_keep = (uint32_t)std::min(std::max(g_regex_local_keep.load(), 0), kLocalSlots);
    dispatch_layout_lanes(cfg.layout, cfg.lanes, [&](auto g, auto lay) {
        auto k = regex_queue_kernel<g, lay>;
        int per_sm = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, kThreads, 0);
        if (e == cudaSuccess) {
            if (per_sm <= 0) e = cudaErrorLaunchOutOfResources;
            else k<<<(unsigned)(sms * per_sm), kThreads, 0, st>>>(ix, rt, d_ring, d_seq, (unsigned long long)(ring_cap - 1), d_res, cap_res, d_ctrl, max_len, local_keep);
        }
    });
    return e != cudaSuccess ? e : cudaGetLastError();
}

// ---- result ordering and per-regex offsets on the device -------------------------------------------------------------------------
__device__ __forceinline__ bool res_less(const RegexResult &a, const RegexResult &b) {
    if (a.regex != b.regex) return a.regex < b.regex;
    if (a.len != b.len) return a.len < b.len;
    if (a.sp != b.sp) return a.sp < b.sp;
    return a.ep < b.ep;
}

// up to kSmallSort results: one CTA, bitonic network in shared memory (a handful of results does not pay for device-wide radix passes)
__global__ void __launch_bounds__(1024)
sort_results_small_kernel(RegexResult *res, int n) {
    extern __shared__ __align__(16) uint8_t raw[];
    RegexResult *s = reinterpret_cast<RegexResult *>(raw);
    int p = 1;
    while (p < n) p <<= 1;
    for (int i = threadIdx.x; i < p; i += blockDim.x) s[i] = i < n ? res[i] : RegexResult{0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu};
    __syncthreads();
    for (int k = 2; k <= p; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < p; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const bool up = (i & k) == 0;
                    const RegexResult x = s[i], y = s[l];
                    if (res_less(y, x) == up) { s[i] = y; s[l] = x; }
                }
            }
            __syncthreads();
        }
    for (int i = threadIdx.x; i < n; i += blockDim.x) res[i] = s[i];
}
cudaError_t sort_results_small(RegexResult *d_res, int64_t n, cudaStream_t st) {
    if (n <= 1) return cudaSuccess;
    if (n > kSmallSort) return cudaErrorInvalidValue;
    int p = 1;
    while (p < n) p <<= 1;
    const size_t smem = (size_t)p * sizeof(RegexResult);
    cudaError_t e = cudaFuncSetAttribute(sort_results_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    sort_results_small_kernel<<<1, (unsigned)std::min<int>(1024, std::max(32, p / 2)), smem, st>>>(d_res, (int)n);
    return cudaGetLastError();
}

// off[r] = index of the first result of regex r in the sorted results (lower bound), off[m] = n
__global__ void result_offsets_kernel(const RegexResult *__restrict__ res, long long n, long long m, long long *__restrict__ off) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > m) return;
    long long lo = 0, hi = n;
    while (lo < hi) { const long long mid = (lo + hi) >> 1; if ((long long)res[mid].regex < r) lo = mid + 1; else hi = mid; }
    off[r] = lo;
}
__global__ void split_results_kernel(const RegexResult *__restrict__ res, long long n, int *__restrict__ len, long long *__restrict__ sp, long long *__restrict__ ep) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const RegexResult r = res[i];
    len[i] = (int)r.len; sp[i] = (long long)r.sp; ep[i] = (long long)r.ep;
}
cudaError_t launch_result_offsets(const RegexResult *d_res, int64_t n, int64_t m, int64_t *d_off, cudaStream_t st) {
    result_offsets_kernel<<<(unsigned)((m + 1 + 255) / 256), 256, 0, st>>>(d_res, n, m, (long long *)d_off);
    return cudaGetLastError();
}
cudaError_t launch_split_results(const RegexResult *d_res, int64_t n, int32_t *d_len, int64_t *d_sp, int64_t *d_ep, cudaStream_t st) {
    if (n > 0) split_results_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_res, n, d_len, (long long *)d_sp, (long long *)d_ep);
    return cudaGetLastError();
}

}  // namespace fmx

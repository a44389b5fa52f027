// fmx_kernels.cuh — host-callable launchers of the search kernels (definitions in fmx_kernels.cu).
#pragma once
#include "fmx_device.cuh"

namespace fmx {

constexpr int kThreads = 256;

struct LaunchCfg {
    int layout;          // FMX_LAYOUT_WM / FMX_LAYOUT_PLANES
    int lanes;           // 1, 2 or 4 lanes per query
    int count_lanes = 0;       // > 0: lanes per query of the count kernels only (one lane once row contexts answer most queries in a
                               // single 32-byte request each: twice the queries in flight, half the instructions per query)
    int min_blocks = 0;        // 4 or 6: the device-pointer count kernel compiled for that many resident CTAs per SM (0 = default: 8, 6 at one lane)
};

// fused exchange: up to 8 gathered buffers (one per rank, peer-mapped) that receive this shard's hit counts
struct PeerSinks {
    uint32_t *p[8];
    int32_t   n;
    long long offset;            // element offset of this shard inside each gathered buffer
};

// count: fixed-length patterns (device pointers).  out64 selects int64 vs uint32 outputs.
cudaError_t launch_count_fixed(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_pat, int len, int64_t m,
                               void *d_sp, void *d_ep, bool out64, unsigned long long *d_stats, cudaStream_t st,
                               const PeerSinks *sinks_or_null = nullptr);
// count: variable-length patterns with int64 offsets.
cudaError_t launch_count_var(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_pat, const int64_t *d_off, int64_t m,
                             int64_t *d_sp, int64_t *d_ep, cudaStream_t st);
cudaError_t launch_occ(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_c, const int64_t *d_key, int64_t m,
                       int64_t *d_out, cudaStream_t st);
cudaError_t launch_prev_range(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_sp, const int64_t *d_ep,
                              const uint8_t *d_c, int64_t m, int64_t *d_sp1, int64_t *d_ep1, cudaStream_t st);
// getIntervalPrevRange: one interval, chars cstart..cend; outputs indexed by (c - cstart)
cudaError_t launch_interval_prev_range(const DevIndex &ix, LaunchCfg cfg, int64_t sp, int64_t ep, int cstart, int cend,
                                       int64_t *d_sp1, int64_t *d_ep1, cudaStream_t st);
// LF step for rows (getPrevI)
cudaError_t launch_lf(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_row, int64_t m, int64_t *d_out, cudaStream_t st);
// FL step for rows (getNextI) and nextSubstr
cudaError_t launch_fl(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_row, int64_t m, int64_t *d_out, cudaStream_t st);
cudaError_t launch_next_substr(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_row, int64_t m, int len, uint8_t *d_out,
                               int *d_out_len, cudaStream_t st);
// prevSubstr: len LF steps per row, emitting the BWT byte at each visited row
cudaError_t launch_prev_substr(const DevIndex &ix, LaunchCfg cfg, const int64_t *d_row, int64_t m, int len,
                               uint8_t *d_out, cudaStream_t st);
// extract: d_out row j (len bytes) = file bytes F[off[j] .. off[j] + out_len[j]), out_len[j] = min(len, n-1-off[j]) (-1 for off[j] > n-1).
// The path follows what `ix` shows: isat, else (with text samples) ctx, ctx8 or LF steps; text_path = that choice (-1: neither isat nor
// samples, the launch fails).  d_requests != nullptr: += the index requests of the walks (the counting instance of the kernel).
int text_path(const DevIndex &ix);
cudaError_t launch_text(const DevIndex &ix, LaunchCfg cfg, const uint32_t *d_off, int64_t m, int len, uint8_t *d_out, int *d_out_len,
                        unsigned long long *d_requests, cudaStream_t st);
// locate: one work item per occurrence of the queries [q0, q1) — occurrences [t0, t0 + count) of the batch, d_off[m+1] = exclusive
// offsets over the whole batch; writes the unsorted sa values of the slab to d_pos[0 .. count), or — d_key != nullptr — the sort keys
// ((query - q0) << 32 | sa value) of the per-query ordering to d_key[0 .. count)
cudaError_t launch_locate(const DevIndex &ix, LaunchCfg cfg, const uint32_t *d_sp, const int64_t *d_off, int64_t q0, int64_t q1,
                          int64_t t0, int64_t count, uint32_t *d_pos, uint64_t *d_key, unsigned long long *d_steps_or_null, cudaStream_t st);
// low 32 bits of n sorted keys -> uint32 (d_out32) or int64 (d_out64)
cudaError_t launch_key_positions(const uint64_t *d_key, int64_t n, uint32_t *d_out32, int64_t *d_out64, cudaStream_t st);
// m patterns of `len` 2-bit codes ((len+3)/4 bytes each) -> m x len bytes; alpha4 = the four symbols, symbol i in byte i
cudaError_t launch_unpack2(const uint8_t *d_codes, int len, int64_t m, uint32_t alpha4, uint8_t *d_out, cudaStream_t st);
// d_out[q] = ep[q] - sp[q] (0 when empty) for q < m, d_out[m] = 0
cudaError_t launch_interval_len(const uint32_t *d_sp, const uint32_t *d_ep, int64_t m, int64_t *d_out, cudaStream_t st);
// copies `count` 4-byte words to every sink at word offset sinks.offset + (*d_dst_off) * dst_scale (d_dst_off may be null)
cudaError_t launch_scatter_words(const uint32_t *d_src, int64_t count, const PeerSinks &sinks, const int64_t *d_dst_off, int64_t dst_scale, cudaStream_t st);

// regex traversal (fmx_regex_kernel.cu)
struct RegexTables {
    const uint4    *rec;         // per global state: { c | flags << 8, first index into fol, number of follows, first follow state };
                                 // flags bit0 = emits a result, bit1 = stops after emitting (Glushkov last position)
    const uint32_t *st_regex;    // owning regex index in the batch
    const uint32_t *fol;         // follow lists, global state ids
};
struct FrontierItem { uint32_t state, len, sp, ep; };   // a ring slot / stack entry
struct RegexResult  { uint32_t regex, len, sp, ep; };
// control words of one traversal (8 x u64 on the device, initialised by the seed kernel)
enum { kRxHead = 0, kRxTail = 1, kRxPending = 2, kRxMatches = 3, kRxStatus = 4, kRxDone = 5, kRxMaxLen = 6, kRxSteps = 7 };
// The whole traversal: seed kernel (initialises the ring's sequence words and the start items) + one persistent work-queue kernel.
// d_ring / d_seq: ring_cap (power of two, >= n_first) slots and their sequence words.  d_ctrl[kRxMatches] = matches found (may exceed cap_res: writes are dropped, the count
// keeps growing), [kRxStatus] = 0 ok, 1 = the ring was too small (rerun with a larger, re-emptied ring), 2 = an item grew longer than the
// text, [kRxMaxLen] = longest item, [kRxSteps] = items processed (one backward step each).
cudaError_t launch_regex_search(const DevIndex &ix, LaunchCfg cfg, const RegexTables &rt, const uint32_t *d_first, int64_t n_first,
                                FrontierItem *d_ring, uint32_t *d_seq, int64_t ring_cap, RegexResult *d_res, int64_t cap_res,
                                unsigned long long *d_ctrl, uint32_t max_len, cudaStream_t st);
void set_regex_local_keep(int items);                    // children a warp keeps on its own stack before spilling to the ring (default: all 256)
constexpr int64_t kSmallSort = 4096;                    // results ordered by one CTA in shared memory up to here
cudaError_t sort_results_small(RegexResult *d_res, int64_t n, cudaStream_t st);
cudaError_t launch_result_offsets(const RegexResult *d_res, int64_t n, int64_t m, int64_t *d_off, cudaStream_t st);
cudaError_t launch_split_results(const RegexResult *d_res, int64_t n, int32_t *d_len, int64_t *d_sp, int64_t *d_ep, cudaStream_t st);

// K4 random gather microbenchmark
cudaError_t launch_gather_bench(const uint4 *base, uint64_t n_blocks64, int bytes_per_gather, int lanes, int64_t gathers,
                                int chain, uint32_t seed, unsigned long long *d_sink, cudaStream_t st);

}  // namespace fmx

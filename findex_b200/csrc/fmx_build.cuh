// fmx_build.cuh — device-side construction entry points (definitions in fmx_build.cu)
#pragma once
#include <string>
#include <vector>

#include "fmx_kernels.cuh"

namespace fmx {

// wavelet matrix: d_blocks holds levels*nblk rank blocks (64 B each), nblk = n/480 + 1
cudaError_t build_wm(const uint8_t *d_bwt, int64_t n, uint32_t eof, const uint8_t *d_code, int levels, uint32_t *d_blocks,
                     int64_t nblk, cudaStream_t st);
// multi-ary wavelet matrix: b bits per digit (2 or 4), `levels` digits per code; d_blocks holds levels*nblk 128-byte blocks,
// nblk = n / rows_per_block + 1 with rows_per_block = 128 (b = 4) or 448 (b = 2)
cudaError_t build_wmx(const uint8_t *d_bwt, int64_t n, uint32_t eof, const uint8_t *d_code, int b, int levels, uint32_t *d_blocks, int64_t nblk,
                      cudaStream_t st);
// per-symbol planes: d_blocks holds sigma*nblk rank blocks; d_sym[code] = byte value
cudaError_t build_planes(const uint8_t *d_bwt, int64_t n, uint32_t eof, const uint8_t *d_sym, int sigma, uint32_t *d_blocks,
                         int64_t nblk, cudaStream_t st);
// sampled SA: marks rows with sa % rate == 0 (rank blocks, nblk) and stores their sa values in mark-rank order.  In the same chain walk,
// d_tsamp != nullptr receives the text samples d_tsamp[v / text_rate] = row of T' position v for every v % text_rate == 0; rate = 0 walks
// for the text samples alone (no marks, no samples)
cudaError_t build_sa_samples(const DevIndex &ix, int layout, int rate, uint32_t *d_mark_blocks, int64_t nblk, uint32_t *d_samples,
                             int64_t n_samples, cudaStream_t st, std::string &err, int text_rate = 0, uint32_t *d_tsamp = nullptr);
// locate walk blocks (56 BWT bytes + 56 mark bits per 64 B); nwb = n/56 + 1
cudaError_t build_walk_blocks(const uint8_t *d_bwt, const uint32_t *d_mark_blocks, int64_t n, uint8_t *d_bm, int64_t nwb, cudaStream_t st);
// full suffix array, its inverse and T' (text[n-1] = 0) by the same chain walks
cudaError_t build_full_sa(const DevIndex &ix, int layout, uint32_t *d_sa, uint32_t *d_isa, uint8_t *d_text, cudaStream_t st, std::string &err);
cudaError_t build_isat(const uint32_t *d_isa, const uint8_t *d_text, const uint8_t *d_code, int64_t n, int bits, int syms, uint4 *d_isat, cudaStream_t st);
// row-indexed 32-byte context entries (DevIndex::ctx): hop lengths + plan table for a context depth J (host), then the entries
struct CtxHops { int h[8]; };
void ctx_hop_plan(int J, CtxHops &hops, uint8_t plan[256]);
cudaError_t build_ctx(const uint32_t *d_sa, const uint32_t *d_isa, const uint8_t *d_text, const uint8_t *d_code, int64_t n, int bits, int J,
                      int raw, const CtxHops &hops, uint4 *d_ctx, cudaStream_t st);
cudaError_t build_ctx8(const uint32_t *d_sa, const uint32_t *d_isa, const uint8_t *d_text, const uint8_t *d_code, int64_t n, int J,
                       uint2 *d_ctx8, cudaStream_t st);
// d_lcp[r] = lcp(suffix of row r, suffix of row r+1), d_lcp[n-1] = 0   (bwtFm2LCP, util.scala:153-212)
cudaError_t build_lcp(const uint32_t *d_sa, const uint32_t *d_isa, const uint8_t *d_text, int64_t n, int32_t *d_lcp, cudaStream_t st);
// the resident LCP structure (DevIndex::lcp8 ...; fmx_device.cuh lcp_widen) in one allocation: lcp8 | records | minima levels | lcpx, each
// part 128-byte aligned; fixed_bytes = everything but the 4 bytes per escaped row (LCP >= 255)
struct LcpLayout {
    int64_t nb, rec_off, tree_off, x_off, fixed_bytes;
    int64_t lvl[6], lvl_count[6];      // level t+1: u32 offset from tree_off / 4, entries before padding
    int top;                           // levels above the records
};
LcpLayout lcp_layout(int64_t n);
// from the int32 LCP array: *d_out = cudaMalloc'ed structure of *bytes_out bytes
cudaError_t build_lcp_struct(const int32_t *d_lcp, int64_t n, const LcpLayout &L, void **d_out, int64_t *bytes_out, cudaStream_t st);
// (sp,ep) after the first K backward steps for every K-mer over the sigma occurring symbols; lex = false: the first consumed (last) pattern
// byte is the most significant digit of the entry index, lex = true: lexicographic order of the K-mer (its first byte most significant)
cudaError_t build_kmer_table(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_sym, uint32_t sigma, int K, uint2 *d_table, cudaStream_t st,
                             bool lex = false);
// converts a lexicographic table of `entries` (sp,ep) in place into k-mer group blocks (fmx_device.cuh kmer_group) that carry ctx[2r+1] of
// up to kKmerInlineRows of their first rows; the buffer must hold ceil(entries / 8) * 64 bytes
cudaError_t pack_kmer_groups(uint2 *d_table, uint64_t entries, const uint4 *d_ctx, cudaStream_t st);
// dictionary of wide intervals (DevIndex::dict) grown from the dense k-mer table of `ix`: depths kmer_k+1 .. <= Dmax, intervals of more than
// min_rows rows, at most max_entries entries; *d_table_out = nullptr when there is nothing to store (cudaMalloc'ed otherwise, 32 * buckets bytes)
// (the deepest level, d = Dmax, keeps intervals of more than min_rows_top rows when those fit)
cudaError_t build_dict(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_sym, uint32_t sigma, int bits, int Dmax, uint32_t min_rows, uint32_t min_rows_top,
                       int64_t max_entries, void **d_table_out, int64_t *buckets_out, int *depth_out, int *depth_x_out, int *jc_out, int64_t *entries_out,
                       cudaStream_t st);
// suffix sort of t+'$' (t has no zero bytes) -> BWT, eof row, byte counts; optionally the suffix array
cudaError_t suffix_sort_bwt(const uint8_t *d_t, int64_t len, uint8_t *d_bwt, int64_t *eof_out, int64_t counts_out[256],
                            uint32_t *d_sa_out, int *rounds_out, cudaStream_t st);
// counts_out[c] = number of bytes of value c among d_bytes[0..n)
cudaError_t byte_histogram(const uint8_t *d_bytes, int64_t n, int64_t counts_out[256], cudaStream_t st);
cudaError_t reverse_bytes(const uint8_t *d_src, int64_t len, uint8_t *d_dst, cudaStream_t st);
cudaError_t build_fm_array(const uint8_t *d_bwt, int64_t n, uint32_t *d_fm, cudaStream_t st);

}  // namespace fmx

/*
 * fmgpu.h — C ABI of libfmgpu.so: the B200-native FM-index search path behind findex's operator API.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference (martende/findex, Scala) has no FFI
 * layer; its operator interface for the path is the trait pair SuffixAlgo / SuffixWalkingAlgo
 * (src/main/scala/org/fmindex/findex.scala:9-57, "M/findex.scala") implemented on disk by
 * NaiveFMSearcher (M/bwtmerger.scala:335-421) and consumed by ReTree.matchSA (M/re2/retree.scala:570).
 * Every entry point below cites the reference member it replaces.  A JVM host binds these with JNA
 * direct mapping (see INTEGRATION.md for the Scala shim); tests bind them with ctypes.
 *
 * Conventions
 *   - every function returns FMX_OK (0) or a negative FMX_E_* code; nothing throws across the ABI;
 *     fmx_last_error() returns a thread-local message for the last failure on the calling thread.
 *   - rows / positions are int64 at the ABI (the device works in uint32; n must be < 2^32).
 *   - intervals are half-open [sp,ep) exactly as in the reference; "None" is reported as sp=ep=0
 *     by the *_count_* calls and as sp1>=ep1 by the prev-range calls.
 *   - the caller owns every input and output buffer.  "_batch" calls take HOST pointers and do the
 *     H2D/D2H copies themselves; "_dev" calls take DEVICE pointers valid on the index's device and a
 *     cudaStream_t (passed as void*; NULL = the legacy default stream) and are asynchronous.
 *   - there is no CPU fallback: without a usable CUDA device every compute call returns FMX_E_CUDA.
 */
#ifndef FMGPU_H
#define FMGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FMX_OK              0
#define FMX_E_IO           -1   /* file missing / unreadable                                            */
#define FMX_E_FORMAT       -2   /* "File %s bad size" / bad elSize (M/bwtmerger.scala:153, :261-262)     */
#define FMX_E_CUDA         -3   /* no device, out of memory, launch failure                             */
#define FMX_E_ARG          -4   /* null pointer, negative size, row out of range                        */
#define FMX_E_CAPACITY     -5   /* output buffer too small; required size is reported                   */
#define FMX_E_SYNTAX       -6   /* Exception("re2post syntax") (M/re2/re2.scala:86-110, :134-182)        */
#define FMX_E_UNSUPPORTED  -7   /* MatchError / NoSuchElementException of ReTree.apply (Q3), n >= 2^32   */
#define FMX_E_LIMIT        -8   /* regex traversal exceeded the configured frontier / length limits     */

/* Rank-structure layouts (fmx_opts.layout) */
#define FMX_LAYOUT_AUTO     0   /* planes if it fits fmx_opts.max_index_bytes (default 64 GiB) and max_total_bytes, else WMX, else WM */
#define FMX_LAYOUT_WM       1   /* byte-alphabet wavelet matrix, ceil(log2 sigma) levels, 64-B rank blocks */
#define FMX_LAYOUT_PLANES   2   /* one 64-B-rank-block bitvector per symbol (1 block fetch per rank)     */
#define FMX_LAYOUT_WMX      3   /* multi-ary wavelet matrix: 16-ary digits (4-ary for <= 4 symbols) in 128-byte blocks = one request per digit:
                                   2 requests per rank for a byte alphabet (1 for <= 16 symbols) at ~2n bytes (0.29n for DNA)        */

/* Bit-exact accelerators of the count path (fmx_opts.accel); they spend HBM capacity, never change results */
#define FMX_ACCEL_AUTO      0
#define FMX_ACCEL_KMER      1   /* table of (sp,ep) after the first k steps, k = max with sigma^k*8 B <= kmer_table_bytes */
#define FMX_ACCEL_TEXT      2   /* full SA + {inverse SA, 96 bits of text} entries (20n bytes): singleton intervals finish in 2 fetches; locate is 1 fetch */
#define FMX_ACCEL_CTX       4   /* 32-byte row contexts { isa[sa[r]-j] for five hop lengths j (1 .. J) ; the J symbols before sa[r] } (32n bytes): an interval
                                   of <= 8 rows advances j symbols in one fetch per row, any remaining length is a sum of hops — a pattern costs about
                                   1 + ceil((len-k)/J) fetches (J = 12 for byte alphabets, 19 for sigma <= 31, 32 for DNA)                       */
#define FMX_ACCEL_CTX8     16   /* (alphabets of <= 4 symbols) compact 8-byte row contexts { isa[sa[r]-16], 16 two-bit symbols }: hops of exactly 16 symbols,
                                   the last < 16 by rank steps; chosen automatically when the 32-byte form does not fit (4e9-row DNA index)         */
#define FMX_ACCEL_DICT     64   /* dictionary of WIDE intervals on top of the k-mer table: a hash table of (sp,ep) for every d-mer, k < d <= D (D = min(16, 60 / bits
                                   per symbol): 12 for sigma <= 32), whose interval holds more than dict_min_rows (2) rows — where rank steps cost two requests
                                   each and row contexts do not apply.  The deepest stored prefix of a pattern is found by bisection over d (a prefix of a wide
                                   d-mer is wide): one request when the whole prefix is wide.  Deeper prefixes hang off depth D as chain entries keyed by
                                   { sp of the interval a tier starts from, up to 22 / bits further symbols }.  Texts with frequent k-mers (natural language) get one;
                                   uniform texts have no wide k-mers beyond the table and get none                                        */
#define FMX_ACCEL_NONE      8   /* plain backward search only                                                */
#define FMX_ACCEL_NO_SA    32   /* count-only deployment: do not keep the full suffix array (4n bytes) that the context/shortcut construction produces;
                                   without it locate needs sa_sample_rate > 0                                                         */

typedef struct fmx_index fmx_index;     /* opaque; library-owned until fmx_close  */
typedef struct fmx_regex fmx_regex;     /* opaque; library-owned until fmx_regex_free */

typedef struct fmx_opts {
    int32_t  device;            /* CUDA device ordinal; -1 = current device                              */
    int32_t  layout;            /* FMX_LAYOUT_*                                                          */
    int32_t  sa_sample_rate;    /* 0 = no locate support; k>=1: rows with sa%k==0 are sampled (32 = cfg3) */
    int32_t  require_fm;        /* 1 = fail like the reference when <base>.fm is absent                  */
    int64_t  max_index_bytes;   /* budget for FMX_LAYOUT_AUTO; 0 = default                               */
    int32_t  lanes_per_query;   /* 0 = default; 1, 2 or 4 lanes cooperate on one 64-B rank block         */
    int32_t  accel;             /* FMX_ACCEL_* bit mask; 0 = auto (all that fit the memory budget)          */
    int64_t  kmer_table_bytes;  /* budget of the k-mer table; 0 = auto: the deepest table that keeps what a count query touches inside
                                   the ~64 GB TLB reach (DESIGN.md §5), else 256 MiB .. 16 GiB (a sixteenth of free memory)     */
    int64_t  max_total_bytes;   /* cap on EVERYTHING resident for this index (rank structure + BWT + sampled SA + accelerators); 0 = no cap.
                                   FMX_LAYOUT_AUTO / FMX_ACCEL_AUTO pick the fastest combination under it; fmx_info reports what was built  */
    int64_t  dict_bytes;        /* budget of the wide-interval dictionary (FMX_ACCEL_DICT); 0 = auto: 12 GiB or an eighth of the free memory    */
    int32_t  dict_min_rows;     /* intervals of more than this many rows are stored; 0 = 2.  (Chain entries past depth D always need more than
                                   max(this, 8) rows: narrower ones are what the row contexts take in one fetch per row)                      */
    int32_t  dict_top_min_rows; /* threshold of the deepest keyed level D (where every pattern at least that long probes first); 0 = 1:
                                   everything that occurs twice, when it fits the budget, else dict_min_rows                                   */
    int32_t  text_sample_rate;  /* 0 = none; s in 1..65536: the row of every s-th text position is kept (4 * ((n-1)/s + 1) bytes), which
                                   fmx_text_batch / fmx_text_dev start their walks from                                                   */
} fmx_opts;

void        fmx_opts_default(fmx_opts *o);
const char *fmx_last_error(void);
const char *fmx_version(void);

/* ---- load: new NaiveFMSearcher(filename, bigEndian)  M/bwtmerger.scala:335-350 ----------------------
 * `path` may carry any extension; it is stripped like BWTTempStorage.gen*Filename (:10-48) and
 * .bwt/.aux(/.fm) are opened.  Validates BWTLoader (:153) and FMLoader (:261-262) size rules.  The
 * occurrence structure is repacked into the GPU rank structure on the device.                         */
int fmx_open(const char *path, int big_endian, const fmx_opts *opts, fmx_index **out);
/* Same, from memory: bwt[n] (byte at eof ignored), eof row, counts[256] as stored in .aux.            */
int fmx_open_mem(const uint8_t *bwt, int64_t n, int64_t eof, const int64_t counts[256],
                 const fmx_opts *opts, fmx_index **out);
int fmx_close(fmx_index *ix);

int64_t fmx_n(const fmx_index *ix);                          /* SuffixAlgo.n          M/findex.scala:10  */
int64_t fmx_eof(const fmx_index *ix);                        /* BWTLoader.eof         M/bwtmerger.scala:151 */
int     fmx_ctable(const fmx_index *ix, int64_t C[256]);     /* cf(c) for all c       M/bwtmerger.scala:352 */
int     fmx_info(const fmx_index *ix, int32_t *layout, int32_t *levels, int32_t *sigma,
                 int64_t *index_bytes, int32_t *sa_sample_rate);

int     fmx_accel_info(const fmx_index *ix, int32_t *kmer_k, int32_t *text_shortcut);   /* accelerators in effect */
/* wide-interval dictionary in effect (0 = none): depth = deepest d-mer stored under its own symbols, chain_depth = deepest prefix reachable
 * through the chain entries behind it (>= depth)                                                                                     */
int     fmx_dict_info(const fmx_index *ix, int32_t *depth, int32_t *chain_depth, int64_t *entries, int64_t *bytes);
int     fmx_ctx_depth(const fmx_index *ix);                  /* J of the row contexts (FMX_ACCEL_CTX / _CTX8), 0 = not built */
/* rows whose row-context J-hop the k-mer table's 64-byte group blocks carry inline (0 = plain table of (sp,ep) entries).  Built under
 * FMX_ACCEL_AUTO with 32-byte row contexts, a saturating table and no dictionary; FMX_KMER_ROWS=0 in the environment at open keeps the plain table */
int     fmx_kmer_rows(const fmx_index *ix);
int     fmx_ctx_entry_bytes(const fmx_index *ix);            /* 32, 8 or 0 */

/* ---- occ(c,key)  M/bwtmerger.scala:354-375  (number of c in BWT[0..key], key=-1 -> 0) --------------- */
int fmx_occ_batch(fmx_index *ix, const uint8_t *c, const int64_t *key, int64_t m, int64_t *out);

/* ---- getPrevRange(sp,ep,c)  M/findex.scala:32-36 ; empty <=> sp1>=ep1 ------------------------------- */
int fmx_prev_range_batch(fmx_index *ix, const int64_t *sp, const int64_t *ep, const uint8_t *c, int64_t m,
                         int64_t *sp1, int64_t *ep1);

/* ---- getIntervalPrevRange(sp,ep,cstart,cend)  M/findex.scala:37-51 ---------------------------------
 * One interval, every c in [cstart,cend]; non-empty results in the reference's order (descending c).
 * out arrays must hold cend-cstart+1 entries; *n_out receives the number written.                      */
int fmx_interval_prev_range(fmx_index *ix, int64_t sp, int64_t ep, int cstart, int cend,
                            int32_t *out_c, int64_t *out_sp, int64_t *out_ep, int64_t *n_out);

/* ---- search(in)  M/findex.scala:15-31 — batched count ----------------------------------------------
 * pat = concatenated pattern bytes, off[m+1] = offsets; pattern q is pat[off[q]..off[q+1]).
 * The pattern is consumed last byte first, with the reference's early exit.  Some((sp,ep)) -> sp<ep;
 * None -> sp=ep=0.  Empty pattern -> (0,n).                                                            */
int fmx_count_batch(fmx_index *ix, const uint8_t *pat, const int64_t *off, int64_t m, int64_t *sp, int64_t *ep);
/* Fixed-length fast path: m patterns of `len` bytes, back to back.                                     */
int fmx_count_fixed(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m, int64_t *sp, int64_t *ep);
/* Same with the reference's own result width, Option[(Int, Int)]: 32-bit rows (n must be < 2^31, else FMX_E_UNSUPPORTED).   */
int fmx_count_fixed_i32(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m, int32_t *sp, int32_t *ep);
/* Alphabets of <= 4 symbols (DNA): the patterns cross PCIe as 2-bit codes — pattern q occupies ceil(len/4) bytes, symbol j =
 * alphabet[(byte[j/4] >> 2(j%4)) & 3] — and are expanded on the device; rows come back as uint32 (row_bytes = 4; n < 2^32) or int64
 * (row_bytes = 8).  Results equal fmx_count_fixed on the expanded patterns.  A len-32 read costs 8 + 8 bytes of PCIe instead of 32 + 16. */
int fmx_count_fixed_packed2(fmx_index *ix, const uint8_t *codes, const uint8_t alphabet[4], int32_t len, int64_t m, void *sp, void *ep, int32_t row_bytes);
/* Count only: counts[q] = ep - sp (0 for None), uint32 — the number of occurrences without the interval.    */
int fmx_count_only_fixed(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m, uint32_t *counts);
/* Device-pointer variant (asynchronous on `stream`): d_pat holds m*len bytes, d_sp/d_ep are uint32[m]. */
int fmx_count_fixed_dev(fmx_index *ix, const void *d_pat, int32_t len, int64_t m,
                        void *d_sp_u32, void *d_ep_u32, void *stream);

/* Fused count + exchange for the multi-GPU path (index replicated, batch sharded): besides d_sp/d_ep, the hit
 * count (ep-sp, uint32) of local query q is stored to sinks[j][offset+q] for each of the n_sinks (<= 8) gathered
 * buffers — this rank's and, via CUDA IPC, its peers' — so the all-gather of counts happens inside the kernel over
 * NVLink/NVSwitch peer memory instead of in a separate collective.
 * Protocol the caller owns (bench.py::FusedExchange is the reference form): after the kernel, a cross-rank barrier on the stream (a
 * 4-byte all-reduce) makes every rank's stores of the step visible everywhere; consumers of step s read the gathered buffer behind
 * that barrier.  A buffer set may be written again only after every rank's consumers of its previous use have finished: rotate THREE
 * sets and launch kernel s (set s mod 3) behind the barrier of step s-2 — every rank enqueued the consumers of step s-3 ahead of its
 * kernel s-2, so that barrier's completion proves they are done.  Two sets with only the same-set barrier are not enough.        */
int fmx_count_fixed_dev_gather(fmx_index *ix, const void *d_pat, int32_t len, int64_t m, void *d_sp_u32, void *d_ep_u32,
                               void *const *sinks, int32_t n_sinks, int64_t offset, void *stream);
/* cudaMalloc'ed, zeroed buffers that the ranks of one node can map into each other (cudaIpc*); sizes are rounded up to 2 MiB so that
 * no two buffers share an underlying block (CUDA IPC maps whole blocks).  Keep the mappings open for the life of the process group:
 * closing the last mapping of a peer takes the lazily enabled peer access down with it, which NCCL in the same process relies on.  */
int fmx_dev_alloc(void **p, int64_t bytes);
int fmx_dev_free(void *p);
int fmx_ipc_export(void *p, uint8_t handle[64]);
int fmx_ipc_import(const uint8_t handle[64], void **p);
int fmx_ipc_close(void *p);
int fmx_memcpy_d2h(void *dst, const void *src, int64_t bytes);

/* ---- locate: sorted { sa[r] : r in [sp,ep) }, sa as bwtFm2sa  M/util.scala:213-224 -----------------
 * (== SACreator.create M/bwtmerger.scala:541-555).  Positions are in T' = reverse(file)+'$' coordinates;
 * file offset of a length-k match = (n-1) - pos - k.  out_off[m+1] receives the per-query offsets;
 * if the total exceeds cap_total, FMX_E_CAPACITY is returned and out_off[m] holds the required total.  */
int fmx_locate_batch(fmx_index *ix, const int64_t *sp, const int64_t *ep, int64_t m, int64_t cap_total,
                     int64_t *out_off, int64_t *pos);

/* Device-resident locate (asynchronous pieces on `stream`, one synchronisation to learn the total): d_sp/d_ep = uint32 rows of m
 * intervals exactly as fmx_count_fixed_dev leaves them (None = (0,0)); d_off (int64[m+1]) receives the exclusive offsets, d_pos
 * (uint32[cap]) the positions, ascending inside each query, T' coordinates.  FMX_E_CAPACITY with *total_out set when cap is small.   */
int fmx_locate_dev(fmx_index *ix, const void *d_sp_u32, const void *d_ep_u32, int64_t m, void *d_off_i64, void *d_pos_u32, int64_t cap,
                   int64_t *total_out, void *stream);
/* Occurrences per internal slab of the locate calls (default 2^30; 0 restores it).  A batch may hold any number of occurrences; it is
 * processed slab by slab.  Exposed so that tests can exercise the slab seams on small inputs.                                       */
int fmx_set_locate_slab(int64_t occurrences);
/* Roofline accounting: fmx_set_stats(ix, 1) makes locate calls count the LF steps of their walks and text calls the index requests of
 * theirs (untimed runs only); regex searches always count the items they process (one backward step each).  fmx_last_steps = that
 * count for the last locate / text / regex call.                                                                                      */
int     fmx_set_stats(fmx_index *ix, int32_t on);
int64_t fmx_last_steps(const fmx_index *ix);
/* Split of the last locate call's device time: LF walks vs the per-query sort.                              */
int fmx_last_locate_ms(const fmx_index *ix, double *walk_ms, double *sort_ms);
/* Exchange step of the variable-length results on the multi-GPU path (located positions, regex triples): this rank's slab of `count`
 * 4-byte words is stored into each of the n_sinks (<= 8) gathered buffers — this rank's and, via CUDA IPC, its peers' — at word offset
 * `offset` + (*d_dst_off) * dst_scale, where d_dst_off is a DEVICE int64 (the scanned offset of this rank's first result; no host
 * round trip between the scan and the stores) or NULL.  Asynchronous on `stream`.                              */
int fmx_scatter_dev(const void *d_src, int64_t count, void *const *sinks, int32_t n_sinks, int64_t offset, const void *d_dst_off,
                    int64_t dst_scale, void *stream);

/* ---- LF / FL steps and extraction  M/bwtmerger.scala:376-419 --------------------------------------- */
int fmx_get_prev_i_batch(fmx_index *ix, const int64_t *row, int64_t m, int64_t *out);   /* getPrevI :386 */
int fmx_get_next_i_batch(fmx_index *ix, const int64_t *row, int64_t m, int64_t *out);   /* getNextI :390 */
int fmx_pos2char(const fmx_index *ix, int64_t key, int32_t *c);                         /* pos2char :376 */
/* prevSubstr(sp,len) :409-419 and nextSubstr(sp,len) :394-405; out is m*len bytes (row-major),
 * out_len[m] the bytes written per row (nextSubstr stops after the '\0').                              */
int fmx_prev_substr_batch(fmx_index *ix, const int64_t *row, int64_t m, int32_t len, uint8_t *out, int32_t *out_len);
int fmx_next_substr_batch(fmx_index *ix, const int64_t *row, int64_t m, int32_t len, uint8_t *out, int32_t *out_len);
/* Both walks under one name: direction > 0 = nextSubstr, else prevSubstr.                              */
int fmx_extract_batch(fmx_index *ix, const int64_t *row, int64_t m, int32_t len, int32_t direction, uint8_t *out, int32_t *out_len);

/* ---- extract: the indexed text at any file offset ------------------------------------------------------
 * F = the indexed file bytes (0x00 dropped, as FileBWTReader reads them) = reverse(T'[0 .. n-2]), |F| = n-1.  Out row q (len bytes,
 * row-major) = F[off[q] .. off[q] + out_len[q]), out_len[q] = min(len, n-1-off[q]).  From a located position: patterns are matched
 * in T', so a length-k match at T' position p (fmx_locate_*) is reverse(pattern) at file offset (n-1) - p - k.
 * A walk starts at the text sample at or after the request's end (fmx_opts.text_sample_rate) and goes backwards through T' by the row
 * contexts' J-hops (FMX_ACCEL_CTX: J symbols per 16-byte request; FMX_ACCEL_CTX8: 16), else by LF steps; with the singleton shortcut
 * (FMX_ACCEL_TEXT) the text is read directly, without samples.  What fmx_set_accel_mask hides is not used.
 * FMX_E_UNSUPPORTED when the index has neither text samples nor a visible singleton shortcut; FMX_E_ARG for an offset outside
 * [0, n-1], len < 0 or null pointers.  With fmx_set_stats(ix, 1), fmx_last_steps = the index requests of the last call's walks.      */
int fmx_text_sample_rate(const fmx_index *ix);              /* 0 = no samples */
int fmx_text_batch(fmx_index *ix, const int64_t *off, int64_t m, int32_t len, uint8_t *out, int32_t *out_len);
/* device-resident, asynchronous on `stream`: d_off uint32[m] file offsets, d_out uint8[m*len], d_out_len int32[m]; an offset above
 * n-1 is not checked on the host and yields out_len = -1                                                                               */
int fmx_text_dev(fmx_index *ix, const void *d_off_u32, int64_t m, int32_t len, void *d_out, void *d_out_len, void *stream);

/* ---- regex: REParser.re2post M/re2/re2.scala:50-185 + ReTree.apply M/re2/retree.scala:156-370 -------
 * Compiles on the host to the reference's Glushkov position automaton, quirks included (SURVEY Q1-Q5);
 * FMX_E_SYNTAX / FMX_E_UNSUPPORTED exactly where the reference throws.                                  */
int  fmx_regex_compile(const uint8_t *re, int64_t re_len, int line_only, fmx_regex **out);
/* Same front-end, choice of automaton: FMX_ENGINE_GLUSHKOV = ReTree (above); FMX_ENGINE_THOMPSON = REParser.createNFA
 * M/re2/re2.scala:264-334, whose search is REParser.matchSA :568-693 with maxIterations = maxLength = 0 (a position that
 * reaches the MatchState emits and is still expanded; no border trimming; `[..]` sets, nullable regexes and epsilon cycles
 * are FMX_E_UNSUPPORTED exactly where the reference throws).  fmx_regex_search_batch accepts both kinds, also mixed.   */
#define FMX_ENGINE_GLUSHKOV 0
#define FMX_ENGINE_THOMPSON 1
int  fmx_regex_compile_engine(const uint8_t *re, int64_t re_len, int line_only, int engine, fmx_regex **out);
void fmx_regex_free(fmx_regex *rx);
/* Introspection (used by the parity tests; mirrors CharNode.c/.num, isLast, follows, root.firsts).
 * follows_off has n_states+1 entries.  Pass NULL to skip an output.                                    */
int  fmx_regex_tables(const fmx_regex *rx, int32_t *n_states, int32_t *n_follows, int32_t *n_firsts,
                      uint8_t *c, uint8_t *is_last, int32_t *num, int32_t *follows_off, int32_t *follows,
                      int32_t *firsts);
/* ReTree.matchSA M/re2/retree.scala:570-653 with the caps disabled (maxBranching=Int.MaxValue,
 * maxIterations=0): per regex the sorted multiset of SAResult (len,sp,ep) M/re2/re2.scala:9-19.
 * out_off[m+1]; FMX_E_CAPACITY with the required total in out_off[m] when cap_total is too small.      */
int  fmx_regex_search_batch(fmx_index *ix, fmx_regex *const *rx, int64_t m, int64_t cap_total,
                            int64_t *out_off, int32_t *len, int64_t *sp, int64_t *ep);

/* ---- DFA engine  M/dfa.scala --------------------------------------------------------------------------
 * fmx_dfa_create = DFA.processLinkList(startState) (:391-407) + compileBuckets (:198-223) for an automaton the caller built from
 * StartState / State / FinishState objects and link(to, chr) calls (:291-336).  kind[i] = 0 start (exactly one), 1 state, 2 finish;
 * state i's links are link_to/link_chr[link_off[i] .. link_off[i+1]) in the reference's LIST order (link() prepends: most recently
 * added first).  Unreachable states are dropped; reachable ones are numbered as the reference's `visited` set grows (start = 0).
 * The handle is an fmx_regex: fmx_regex_search_batch / fmx_regex_set_* run DFA.matchSA (:261-289) with the 500-iteration cap off —
 * per automaton the sorted multiset of DFAResult (len, sp, ep); only DFAChar actions are followed (a DFABucket, i.e. two or more
 * consecutive characters with one target, is never traversed: StatePoint.expand :238-256), and a finish state emits and is still
 * expanded.  Free with fmx_regex_free.                                                                                   */
int fmx_dfa_create(int32_t n_states, const uint8_t *kind, const int32_t *link_off, const int32_t *link_to,
                   const int32_t *link_chr, fmx_regex **out);
/* DFA.fromNFA(initialState)  M/dfa.scala:343-389: subset construction over an NFA of NfaBaseState objects (:5-37) — state i's links are
 * link_to/link_chr[link_off[i] .. link_off[i+1]), link_chr = -1 for an EpsilonLink; is_finish[i] marks the NfaFinishState(s).  The set of
 * the initial state becomes the StartState and never accepts, also when it holds a finish state or is reached again (:353-359); every
 * other set with a finish state is a FinishState.  Then as fmx_dfa_create.  FMX_E_LIMIT beyond 100000 DFA states.                    */
int fmx_dfa_from_nfa(int32_t n_states, const uint8_t *is_finish, int32_t initial, const int32_t *link_off, const int32_t *link_to,
                     const int32_t *link_chr, fmx_regex **out);
/* moves (n_states x 256, -1 = none), finishStates, and number[i] = DFA index of the caller's state i (-1 = unreachable).    */
int fmx_dfa_info(const fmx_regex *dfa, int32_t *n_states, int32_t *moves, uint8_t *finish, int32_t *number, int32_t n_number);
/* buckets(state).mkString(",") with the reference's toString, e.g. "DFABucket('c-d' ->1),DFAChar('f'->1)"  (:190-196)        */
int fmx_dfa_buckets(const fmx_regex *dfa, int32_t state, char *buf, int64_t cap, int64_t *needed);
/* DFA.matchString (:160-171), bytes unsigned                                                                               */
int fmx_dfa_match_string(const fmx_regex *dfa, const uint8_t *s, int64_t len, int32_t *matched);

/* Compile once, search many times: a regex set keeps the concatenated automata of a batch resident on the index's device
 * (the batched form of `val t = ReTree(post)` ... `t.matchSA(sa)` ... `t.matchSA(sa2)`).  fmx_regex_search_batch is
 * create + search + free.  Follow positions whose byte does not occur in `ix`'s text are pruned at creation (they cannot survive their
 * step; results are unchanged), so a set may be searched against an index on the same device whose symbols all occur in `ix`'s text.                          */
typedef struct fmx_regex_set fmx_regex_set;
int  fmx_regex_set_create(fmx_index *ix, fmx_regex *const *rx, int64_t m, fmx_regex_set **out);
int  fmx_regex_set_search(fmx_index *ix, fmx_regex_set *set, int64_t cap_total, int64_t *out_off, int32_t *len, int64_t *sp, int64_t *ep);
/* Device-resident form: the results stay on the index's device as {regex, len, sp, ep} records (4 x uint32) ordered by (regex, len, sp, ep)
 * in d_res[cap]; d_off (int64[m+1], may be NULL) receives the index of every regex's first result; *total_out the number of results
 * (FMX_E_CAPACITY when it exceeds cap).  What a multi-GPU caller exchanges, and what fmx_regex_set_search copies out.
 * Stream contract: the search runs on a stream of the library and the call returns when d_res/d_off are complete; it does NOT order
 * itself after work the caller still has in flight on d_res/d_off (a fill, a previous step's readers) — synchronise that first.   */
int  fmx_regex_set_search_dev(fmx_index *ix, fmx_regex_set *set, void *d_res, int64_t cap, void *d_off_i64, int64_t *total_out);
/* Length cap of later searches of the set: max_len = the maxLength argument of REParser.matchSA (M/re2/re2.scala:568, applied at :636-641) —
 * an item's follow positions are enqueued only while their len stays below max_len, matches are emitted whatever their length; 0 = off.
 * Order-independent, so the result is still a well-defined multiset (for the Glushkov engine, whose matchSA has no such argument, it is
 * an extension with the same meaning).  The reference's order-dependent caps (maxIterations; ReTree.matchSA's maxBranching = 1024,
 * maxIterations = 1000 defaults, retree.scala:570, :628) are not offered: what survives them depends on Scala's PriorityQueue tie order. */
int  fmx_regex_set_limits(fmx_regex_set *set, int64_t max_len);
/* Tuning hook of the traversal kernel: children a warp keeps on its own shared-memory stack (0..256, default 256) before spilling to
 * the global ring where idle warps find them.  Results never change.                                                                 */
int  fmx_set_regex_local_keep(int32_t items);
/* Sizes the set's device work ring to `slots` items (power of two, >= the number of start positions; default: 4x the start positions,
 * at least 2^20).  A traversal that overflows its ring is abandoned and rerun with a 4x larger one — results never change.            */
int  fmx_regex_set_ring(fmx_regex_set *set, int64_t slots);
void fmx_regex_set_free(fmx_regex_set *set);

/* ---- instrumentation for the roofline accounting (not on the timed path) ---------------------------
 * Runs the same count kernel with block-touch counting: *blocks = number of distinct 64-B rank blocks
 * the batch reads (a level whose sp and ep probes share a block counts once), *steps = executed
 * backward steps.                                                                                      */
int fmx_count_fixed_stats(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m,
                          int64_t *blocks, int64_t *steps);
/* K4: random 64-B-aligned gather microbenchmark over the index's own rank-block array.
 * bytes_per_gather in {32,64,128}; returns achieved GB/s of useful bytes in *gbs.                       */
int fmx_gather_bench(fmx_index *ix, int32_t bytes_per_gather, int32_t lanes, int64_t gathers, int32_t chain,
                     int32_t iters, double *gbs, double *ms);
/* Time of the last *_batch call's kernel section in ms (CUDA events on the library's stream).          */
/* Page-locked host buffers: batch calls given such buffers copy by asynchronous DMA and overlap the copies
 * with the kernels (a JVM host wraps the pointer as a direct ByteBuffer).  Any host pointer is accepted by the
 * batch calls; pageable memory just copies slower.                                                      */
int fmx_host_alloc(void **p, int64_t bytes);
int fmx_host_free(void *p);
/* cudaLimitMaxL2FetchGranularity of the current device (32/64/128; 0 = only query).  Random 64-B block fetches
 * over-fetch from DRAM when the L2 promotes misses to 128 B; see DESIGN.md §5.                              */
int fmx_set_l2_fetch_granularity(int32_t bytes, int32_t *effective);
/* Hides accelerators that were built from subsequent calls: `mask` = FMX_ACCEL_* bits to keep (FMX_ACCEL_NONE = plain backward
 * search over the rank structure; FMX_ACCEL_AUTO = all that were built).  Results never change; for measuring one index both ways. */
int fmx_set_accel_mask(fmx_index *ix, int32_t mask);
/* Queries per pipeline chunk of the host-buffer count calls (0 = default 2^20).                          */
int fmx_set_chunk(fmx_index *ix, int64_t queries_per_chunk);
/* Re-selects how many lanes (1, 2 or 4) cooperate on one 64-B rank block for subsequent calls.           */
int fmx_set_lanes(fmx_index *ix, int32_t lanes_per_query);
int fmx_get_lanes(const fmx_index *ix);                      /* lanes per query of the count kernels (may differ from the other kernels' by default) */
double fmx_last_kernel_ms(const fmx_index *ix);
int64_t fmx_last_kernel_launches(const fmx_index *ix);
/* Length of the longest (len, sp, ep) item the last regex search produced (the depth of the traversal).  */
int64_t fmx_last_regex_levels(const fmx_index *ix);

/* ---- index construction on the device (SURVEY §8f rank 1; tooling for synthetic configs) -----------
 * text = FILE bytes (forward order).  Reproduces FileBWTReader (M/bwtreader.scala:196-211: 0x00 dropped,
 * text reversed), suffix-sorts reverse(text)+'$' on the GPU and writes <base>.bwt/.aux in the
 * reference's layout (BWTTempStorage :75-98, writeAuxFile :841-856); write_fm also writes <base>.fm
 * (FMCreator.create :452-532).                                                                          */
int fmx_build_index_files(const uint8_t *text, int64_t len, const char *base, int big_endian, int write_fm,
                          int device);
/* Same, to memory: bwt_out[n], *eof_out, counts_out[256]; n = (number of non-zero bytes) + 1.          */
int fmx_build_bwt(const uint8_t *text, int64_t len, uint8_t *bwt_out, int64_t *n_out, int64_t *eof_out,
                  int64_t counts_out[256], int device);

/* SACreator(filename).create()  M/bwtmerger.scala:535-556: writes <base>.sa (n x int32 big-endian, no header; SALoader :214-249 reads it),
 * sa[r] as bwtFm2sa (M/util.scala:213-224).  Uses the resident suffix array when the index has one, else builds it for the call.      */
int fmx_write_sa_file(fmx_index *ix, const char *path);

/* LCPCreator(filename).create()  M/bwtmerger.scala:558-652 == Util.bwtstring.bwtFm2LCP  M/util.scala:153-212 (the consistency the reference's
 * LCPLoaderTest asserts, T/Indexer.scala:1017-1042): lcp[r] = longest common prefix of the suffixes of rows r and r+1, computed on the device.
 * fmx_build_lcp fills lcp_out[n] (lcp[n-1] = 0, never written by the reference); fmx_write_lcp_file writes <base>.lcp as the reference does —
 * big-endian int32, no header, the first max(n-1, 1) entries (LCPLoader :176-211; LCPSearcher.getLCP(i) :328 reads entry i).           */
int fmx_build_lcp(fmx_index *ix, int32_t *lcp_out);
int fmx_write_lcp_file(fmx_index *ix, const char *path);

#ifdef __cplusplus
}
#endif
#endif /* FMGPU_H */

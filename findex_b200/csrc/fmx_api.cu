// fmx_api.cu — the C ABI of libfmgpu.so (include/fmgpu.h): index upload, batched operator calls, regex
// frontier driver, locate, device-side index construction.  Host buffers in, host buffers out; every
// compute call runs on the index's CUDA stream and fails with FMX_E_CUDA when no device is usable —
// there is no CPU path in this library.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <vector>

#include "fmx_build.cuh"
#include "fmx_cub.cuh"
#include "fmx_internal.h"
#include "fmx_kernels.cuh"

using namespace fmx;

struct fmx_index {
    int device = 0;
    cudaStream_t stream = nullptr, h2d = nullptr, d2h = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_alloc = nullptr;
    int64_t chunk_queries = 0;
    bool accel_text = false;
    int kmer_k = 0;
    DevIndex d{};                      // what the kernels see (fmx_set_accel_mask may hide accelerators)
    DevIndex d_full{};                 // everything that was built
    int count_lanes_full = 0;
    LaunchCfg cfg{FMX_LAYOUT_WM, 4};
    int64_t n = 0, eof = 0;
    int64_t C[257] = {0};
    int64_t counts0[256] = {0};        // raw counts (bucketStarts0 / pos2char)
    int sigma = 0, levels = 0, sample_rate = 0, text_rate = 0;
    int64_t nblk = 0, index_bytes = 0, n_samples = 0, rank_units64 = 0, dict_entries = 0;
    int api_layout = FMX_LAYOUT_WM;    // what fmx_info reports
    std::vector<void *> owned;         // device allocations freed at close
    std::atomic<double> last_ms{0.0}, locate_walk_ms{0.0}, locate_sort_ms{0.0};      // diagnostics of the most recent call
    bool stats = false;                // fmx_set_stats: the next locate / regex calls also count their LF steps / items
    std::atomic<int64_t> last_steps{0}, last_launches{0}, total_launches{0}, last_levels{0};
    std::mutex mu;                     // guards cfg / d / chunk_queries / stats and the pool below; never held across GPU work
    // Batch calls run concurrently: each takes one of kCallSets private stream sets for its duration (copies and kernels of different
    // host threads overlap; the index itself is read-only).  `stream`/`h2d`/`d2h` above belong to fmx_open and the rare whole-index calls.
    struct StreamSet { cudaStream_t stream = nullptr, h2d = nullptr, d2h = nullptr; cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_alloc = nullptr; bool busy = false; };
    static constexpr int kCallSets = 4;
    StreamSet sets[kCallSets];
    std::condition_variable cv;
};

namespace {

#define CU(x)                                                                                         \
    do {                                                                                              \
        cudaError_t e_ = (x);                                                                         \
        if (e_ != cudaSuccess) return fail(FMX_E_CUDA, "CUDA error %s at %s:%d (%s)", cudaGetErrorName(e_), __FILE__, __LINE__, cudaGetErrorString(e_)); \
    } while (0)

// RAII stream-ordered device buffer
struct DBuf {
    void *p = nullptr;
    cudaStream_t st;
    explicit DBuf(cudaStream_t s) : st(s) {}
    ~DBuf() { if (p) cudaFreeAsync(p, st); }
    cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes ? bytes : 1, st); }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};

struct Events {                                                 // per-chunk events of a pipelined call, destroyed on every exit path
    std::vector<cudaEvent_t> v;
    ~Events() { for (cudaEvent_t e : v) if (e) cudaEventDestroy(e); }
    cudaError_t make(size_t k) { v.assign(k, nullptr); for (auto &e : v) { cudaError_t r = cudaEventCreateWithFlags(&e, cudaEventDisableTiming); if (r != cudaSuccess) return r; } return cudaSuccess; }
};

struct SaBuf {
    void *p = nullptr;
    ~SaBuf() { if (p) cudaFree(p); }
    template <typename T> T *as() { return reinterpret_cast<T *>(p); }
};

// One batch call's view of the index: a private stream set (taken from the pool for the call's duration) and a snapshot of the
// settings, so that calls of different host threads neither serialise nor race with fmx_set_*.
struct CallCtx {
    fmx_index *ix;
    fmx_index::StreamSet *set = nullptr;
    cudaStream_t stream = nullptr, h2d = nullptr, d2h = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_alloc = nullptr;
    DevIndex d;
    LaunchCfg cfg;
    int64_t chunk_queries;
    bool stats, ok = true;
    explicit CallCtx(fmx_index *i) : ix(i) {
        std::unique_lock<std::mutex> lk(ix->mu);
        for (;;) {
            for (auto &s : ix->sets) if (!s.busy) { set = &s; break; }
            if (set) break;
            ix->cv.wait(lk);
        }
        set->busy = true;
        d = ix->d; cfg = ix->cfg; chunk_queries = ix->chunk_queries; stats = ix->stats;
        if (!set->stream) {                                  // first use of this set
            int prev = -1;
            cudaGetDevice(&prev);
            if (prev != ix->device) cudaSetDevice(ix->device);
            ok = cudaStreamCreateWithFlags(&set->stream, cudaStreamNonBlocking) == cudaSuccess &&
                 cudaStreamCreateWithFlags(&set->h2d, cudaStreamNonBlocking) == cudaSuccess &&
                 cudaStreamCreateWithFlags(&set->d2h, cudaStreamNonBlocking) == cudaSuccess && cudaEventCreate(&set->ev0) == cudaSuccess &&
                 cudaEventCreate(&set->ev1) == cudaSuccess && cudaEventCreateWithFlags(&set->ev_alloc, cudaEventDisableTiming) == cudaSuccess;
            if (prev >= 0 && prev != ix->device) cudaSetDevice(prev);
        }
        stream = set->stream; h2d = set->h2d; d2h = set->d2h; ev0 = set->ev0; ev1 = set->ev1; ev_alloc = set->ev_alloc;
    }
    ~CallCtx() {
        { std::lock_guard<std::mutex> lk(ix->mu); set->busy = false; }
        ix->cv.notify_one();
    }
    CallCtx(const CallCtx &) = delete;
    CallCtx &operator=(const CallCtx &) = delete;
};
#define CHECK_CC(cc) do { if (!(cc).ok) return fail(FMX_E_CUDA, "cannot create CUDA streams/events for the call"); } while (0)

struct Timed {
    fmx_index *ix;
    CallCtx &cc;
    Timed(fmx_index *i, CallCtx &c) : ix(i), cc(c) { cudaEventRecord(cc.ev0, cc.stream); ix->last_launches = 0; }
    void stop() { cudaEventRecord(cc.ev1, cc.stream); }
    void collect() { float ms = 0; if (cudaEventElapsedTime(&ms, cc.ev0, cc.ev1) == cudaSuccess) ix->last_ms = ms; }
};

int ensure_device(int device, int *chosen) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(FMX_E_CUDA, "no usable CUDA device (%s): libfmgpu has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    int dev = device;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
    if (dev >= count) return fail(FMX_E_ARG, "device %d out of range (%d devices)", dev, count);
    CU(cudaSetDevice(dev));
    *chosen = dev;
    return FMX_OK;
}

template <typename T> T *dev_upload(fmx_index *ix, const T *host, size_t count, cudaError_t *err) {
    void *p = nullptr;
    *err = cudaMalloc(&p, count ? count * sizeof(T) : 1);
    if (*err != cudaSuccess) return nullptr;
    ix->owned.push_back(p);
    if (count) *err = cudaMemcpyAsync(p, host, count * sizeof(T), cudaMemcpyHostToDevice, ix->stream);
    return reinterpret_cast<T *>(p);
}

// The stream-ordered pool keeps freed blocks cached (release threshold = max) so that batch calls do not re-map memory;
// after the large one-off constructions the cache is handed back.
void trim_pool(int dev) {
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
}

int bitrev(int v, int bits) { int r = 0; for (int i = 0; i < bits; ++i) r |= ((v >> i) & 1) << (bits - 1 - i); return r; }

// ---- index upload (K0): tables on the host, rank structures on the device -------------------------------
int upload_index(fmx_index *ix, const uint8_t *bwt, int64_t n, int64_t eof, const int64_t counts[256], const fmx_opts &o) {
    if (n < 1 || eof < 0 || eof >= n) return fail(FMX_E_ARG, "bad n/eof");
    if (n >= (1ll << 32) - 1) return fail(FMX_E_UNSUPPORTED, "n = %lld needs 64-bit rows; this build indexes n < 2^32-1", (long long)n);
    if (o.text_sample_rate < 0 || o.text_sample_rate > 65536) return fail(FMX_E_ARG, "text_sample_rate = %d: 0 (none) or 1 .. 65536", o.text_sample_rate);
    ix->n = n; ix->eof = eof;
    // C table: bucketStarts with counts[0] := 1   (bwtmerger.scala:346-350, util.scala:109-119)
    int64_t tot = 0;
    for (int c = 0; c < 256; ++c) { ix->C[c] = tot; tot += (c == 0) ? 1 : counts[c]; ix->counts0[c] = counts[c]; }
    ix->C[256] = n;
    if (tot != n) return fail(FMX_E_FORMAT, "aux counts sum %lld != n-1 = %lld", (long long)(tot - 1), (long long)(n - 1));

    // dense symbol codes over the bytes that occur ('$' is not a symbol)
    uint8_t code[256], sym[256];
    int sigma = 0;
    code[0] = kCodeAbsent;
    for (int c = 1; c < 256; ++c) { if (counts[c] > 0) { code[c] = (uint8_t)sigma; sym[sigma++] = (uint8_t)c; } else code[c] = kCodeAbsent; }
    if (sigma > 254) {           // 255 distinct bytes: code 0xFF collides with the "absent" marker only if sigma == 256
        // codes run 0..254 here, 0xFF stays free because byte 0 never occurs in the text
    }
    int levels = 1;
    while ((1 << levels) < sigma) ++levels;
    ix->sigma = sigma; ix->levels = levels;
    const int64_t nblk = n / kBitsPerBlock + 1;
    ix->nblk = nblk;

    int layout = o.layout;
    const int64_t planes_bytes = (int64_t)std::max(sigma, 1) * nblk * 64, wm_bytes = (int64_t)levels * nblk * 64;
    const int64_t budget = o.max_index_bytes > 0 ? o.max_index_bytes : (64ll << 30);
    // max_total_bytes bounds EVERYTHING resident for this index (rank structure, BWT, sampled SA, accelerators); 0 = what the device holds
    const int64_t total_cap = o.max_total_bytes > 0 ? o.max_total_bytes : (1ll << 62);
    if (o.max_total_bytes > 0 && wm_bytes + n > total_cap && layout != FMX_LAYOUT_PLANES && layout != FMX_LAYOUT_WMX)
        return fail(FMX_E_ARG, "max_total_bytes = %lld is below the smallest index of this text (%lld bytes: wavelet matrix + BWT)", (long long)total_cap, (long long)(wm_bytes + n));
    // multi-ary wavelet matrix: 16-ary digits (4-ary when at most 4 symbols occur), 128-byte blocks
    const int xb = sigma <= 4 ? 2 : 4, xlevels = sigma <= (1 << xb) ? 1 : 2;
    const int64_t xrows = xb == 4 ? 128 : 448, nblkx = n / xrows + 1, wmx_bytes = (int64_t)xlevels * nblkx * 128;
    if (layout == FMX_LAYOUT_AUTO) {
        size_t fr = 0, to = 0;
        cudaMemGetInfo(&fr, &to);
        const int64_t sampled = (o.sa_sample_rate > 0 ? nblk * 64 + (n / o.sa_sample_rate + 1) * 4 + (n / kRowsPerWalkBlock + 1) * 64 : 0) +
                                (o.text_sample_rate > 0 ? ((n - 1) / o.text_sample_rate + 1) * 4 : 0);
        layout = (planes_bytes <= budget && planes_bytes + n + sampled <= total_cap && planes_bytes + (6ll << 30) + 2 * n < (int64_t)fr) ? FMX_LAYOUT_PLANES
                 : (wmx_bytes + n + sampled <= total_cap ? FMX_LAYOUT_WMX : FMX_LAYOUT_WM);
    }
    if (layout != FMX_LAYOUT_WM && layout != FMX_LAYOUT_PLANES && layout != FMX_LAYOUT_WMX) return fail(FMX_E_ARG, "bad layout %d", layout);
    const bool wmx = layout == FMX_LAYOUT_WMX;
    ix->api_layout = layout;
    int lanes = o.lanes_per_query ? o.lanes_per_query : (wmx ? 4 : 2);      // re-tuned below once the accelerators are known
    if (lanes != 1 && lanes != 2 && lanes != 4) return fail(FMX_E_ARG, "lanes_per_query must be 1, 2 or 4");
    ix->cfg = LaunchCfg{layout, lanes};
    if (const char *mb = std::getenv("FMX_MINB")) ix->cfg.min_blocks = std::atoi(mb);      // occupancy experiment (profiles/r01_count_design_sweep.jsonl)
    ix->index_bytes = (layout == FMX_LAYOUT_PLANES ? planes_bytes : wmx ? wmx_bytes : wm_bytes) + n;

    // base[c]: PLANES: C[c].  WM: C[c] - start_final[code], where after `levels` stable bit partitions the
    // symbols are ordered by bit-reversed code; the '$' row travels with code 0.
    uint32_t C32[257], base[256], z[8] = {0}, zx[2][16] = {{0}};
    for (int c = 0; c <= 256; ++c) C32[c] = (uint32_t)ix->C[c];
    for (int c = 0; c < 256; ++c) base[c] = C32[c];
    if (wmx) {
        // after the stable partitions by digit 0 (most significant), then digit 1, ... the codes are ordered by their digits read in
        // reverse; zx[l][v] = rows whose digit at level l is below v
        const int ncodes = 1 << (xb * xlevels), dm = (1 << xb) - 1;
        std::vector<int64_t> cc((size_t)ncodes, 0);
        for (int s = 0; s < sigma; ++s) cc[(size_t)s] = counts[sym[s]];
        cc[0] += 1;                                              // the '$' row is filed under code 0
        for (int l = 0; l < xlevels; ++l) {
            int64_t per[16] = {0};
            for (int s = 0; s < ncodes; ++s) per[(s >> (xb * (xlevels - 1 - l))) & dm] += cc[(size_t)s];
            int64_t acc = 0;
            for (int v = 0; v <= dm; ++v) { zx[l][v] = (uint32_t)acc; acc += per[v]; }
        }
        auto rev = [&](int s) { int r = 0; for (int l = 0; l < xlevels; ++l) r = (r << xb) | ((s >> (xb * l)) & dm); return r; };
        std::vector<int> order((size_t)ncodes);
        for (int s = 0; s < ncodes; ++s) order[(size_t)s] = s;
        std::sort(order.begin(), order.end(), [&](int a, int b) { return rev(a) < rev(b); });
        std::vector<int64_t> start((size_t)ncodes, 0);
        int64_t acc = 0;
        for (int s : order) { start[(size_t)s] = acc; acc += cc[(size_t)s]; }
        for (int s = 0; s < sigma; ++s) base[sym[s]] = (uint32_t)(ix->C[sym[s]] - start[(size_t)s]);
    } else if (layout == FMX_LAYOUT_WM) {
        std::vector<int64_t> cc(1 << levels, 0);                 // occurrences per code ('$' under code 0)
        for (int s = 0; s < sigma; ++s) cc[s] = counts[sym[s]];
        cc[0] += 1;
        for (int l = 0; l < levels; ++l) {
            int64_t zeros = 0;
            for (int s = 0; s < (1 << levels); ++s) if (!((s >> (levels - 1 - l)) & 1)) zeros += cc[s];
            z[l] = (uint32_t)zeros;
        }
        std::vector<int> order(1 << levels);
        for (int s = 0; s < (1 << levels); ++s) order[s] = s;
        std::sort(order.begin(), order.end(), [&](int a, int b) { return bitrev(a, levels) < bitrev(b, levels); });
        std::vector<int64_t> start(1 << levels, 0);
        int64_t acc = 0;
        for (int s : order) { start[s] = acc; acc += cc[s]; }
        for (int s = 0; s < sigma; ++s) base[sym[s]] = (uint32_t)(ix->C[sym[s]] - start[s]);
    }

    cudaError_t e;
    uint8_t *d_bwt = dev_upload(ix, bwt, (size_t)n, &e); CU(e);
    CU(cudaMemsetAsync(d_bwt + eof, 0, 1, ix->stream));
    {   // the BWT must hold exactly the .aux counts (and one '$'): otherwise LF is not a permutation of the rows and the chain walks,
        // locate walks and table fills below would run off the index (a corrupt or mismatched .bwt/.aux pair)
        int64_t hist[256];
        CU(byte_histogram(d_bwt, n, hist, ix->stream));
        for (int c = 0; c < 256; ++c)
            if (hist[c] != (c == 0 ? 1 : counts[c]))
                return fail(FMX_E_FORMAT, "the BWT holds %lld bytes of value %d, the .aux counts say %lld: .bwt and .aux do not belong together", (long long)hist[c], c, (long long)(c == 0 ? 1 : counts[c]));
    }
    uint32_t *d_C = dev_upload(ix, C32, 257, &e); CU(e);
    uint32_t *d_base = dev_upload(ix, base, 256, &e); CU(e);
    uint8_t *d_code = dev_upload(ix, code, 256, &e); CU(e);
    uint8_t *d_sym = dev_upload(ix, sym, 256, &e); CU(e);
    void *blocks = nullptr;
    const int64_t nplanes = layout == FMX_LAYOUT_PLANES ? std::max(sigma, 1) : levels;
    const int64_t rank_alloc = wmx ? wmx_bytes : nplanes * nblk * 64;
    ix->rank_units64 = rank_alloc / 64;
    e = cudaMalloc(&blocks, (size_t)rank_alloc);
    if (e != cudaSuccess) return fail(FMX_E_CUDA, "cannot allocate %lld bytes for the rank structure: %s", (long long)rank_alloc, cudaGetErrorString(e));
    ix->owned.push_back(blocks);
    CU(cudaMemsetAsync(blocks, 0, (size_t)rank_alloc, ix->stream));
    if (layout == FMX_LAYOUT_PLANES) CU(build_planes(d_bwt, n, (uint32_t)eof, d_sym, sigma, (uint32_t *)blocks, nblk, ix->stream));
    else if (wmx) CU(build_wmx(d_bwt, n, (uint32_t)eof, d_code, xb, xlevels, (uint32_t *)blocks, nblkx, ix->stream));
    else CU(build_wm(d_bwt, n, (uint32_t)eof, d_code, levels, (uint32_t *)blocks, nblk, ix->stream));

    DevIndex &d = ix->d;
    d.blocks = (const uint4 *)blocks; d.stride = (uint64_t)nblk; d.bwt = d_bwt; d.C = d_C; d.base = d_base; d.code = d_code;
    d.bm = nullptr;
    d.kmer = nullptr; d.kmer_k = 0; d.kmer_sigma = 0; d.kmer_rows = 0; d.sa = nullptr; d.isat = nullptr; d.isat_bits = 8; d.isat_syms = 12; d.ctx = nullptr; d.ctx_J = 0; d.ctx_raw = 0; d.ctx_plan = nullptr; d.ctx8 = nullptr; d.ctx8_J = 0;
    d.dict = nullptr; d.dict_buckets = 0; d.dict_D = 0; d.dict_bits = 0; d.dict_Dx = 0; d.dict_Jc = 1;
    for (int t = 0; t < 8; ++t) d.ctx_S[t] = 0;
    d.tsamp = nullptr; d.tsamp_rate = 0; d.sym = d_sym;
    d.mark = nullptr; d.samples = nullptr; d.n = (uint32_t)n; d.eof = (uint32_t)eof; d.layout = layout; d.levels = levels;
    for (int l = 0; l < 8; ++l) d.z[l] = z[l];
    d.wmx_b = wmx ? xb : 0; d.wmx_levels = wmx ? xlevels : 0; d.wmx_stride = (uint64_t)nblkx;
    for (int l = 0; l < 2; ++l) for (int v = 0; v < 16; ++v) d.zx[l][v] = zx[l][v];

    ix->sample_rate = o.sa_sample_rate;
    // text samples (extract): the row of every text_rate-th T' position, recorded by the same chain walk as the sampled SA (or by that walk
    // alone without a sampled SA)
    uint32_t *tsamp = nullptr;
    if (o.text_sample_rate > 0) {
        const int64_t nt = (n - 1) / o.text_sample_rate + 1;
        if (ix->index_bytes + nt * 4 > total_cap)
            return fail(FMX_E_ARG, "max_total_bytes = %lld leaves no room for the %lld bytes of text samples", (long long)total_cap, (long long)nt * 4);
        e = cudaMalloc((void **)&tsamp, (size_t)nt * 4); CU(e); ix->owned.push_back(tsamp);
        ix->index_bytes += nt * 4;
        ix->text_rate = o.text_sample_rate;
        if (o.sa_sample_rate <= 0) {
            std::string err;
            e = build_sa_samples(d, layout, 0, nullptr, nblk, nullptr, 0, ix->stream, err, o.text_sample_rate, tsamp);
            if (e != cudaSuccess) return fail(err.empty() ? FMX_E_CUDA : FMX_E_FORMAT, "text sample construction failed: %s", err.empty() ? cudaGetErrorString(e) : err.c_str());
        }
        d.tsamp = tsamp; d.tsamp_rate = (uint32_t)o.text_sample_rate;
    }
    if (o.sa_sample_rate > 0) {
        const int64_t ns = (n + o.sa_sample_rate - 1) / o.sa_sample_rate;
        void *mark = nullptr, *samples = nullptr;
        e = cudaMalloc(&mark, (size_t)nblk * 64); CU(e); ix->owned.push_back(mark);
        e = cudaMalloc(&samples, (size_t)ns * 4); CU(e); ix->owned.push_back(samples);
        std::string err;
        e = build_sa_samples(d, layout, o.sa_sample_rate, (uint32_t *)mark, nblk, (uint32_t *)samples, ns, ix->stream, err, o.text_sample_rate, tsamp);
        if (e != cudaSuccess) return fail(err.empty() ? FMX_E_CUDA : FMX_E_FORMAT, "sampled SA construction failed: %s", err.empty() ? cudaGetErrorString(e) : err.c_str());
        d.mark = (const uint4 *)mark; d.samples = (const uint32_t *)samples;
        ix->n_samples = ns;
        ix->index_bytes += nblk * 64 + ns * 4;
        if (o.sa_sample_rate > 1) {                              // fused BWT+mark blocks: one fetch per LF step of the locate walk
            const int64_t nwb = n / kRowsPerWalkBlock + 1;
            void *bm = nullptr;
            e = cudaMalloc(&bm, (size_t)nwb * 64); CU(e); ix->owned.push_back(bm);
            CU(build_walk_blocks(d_bwt, (const uint32_t *)mark, n, (uint8_t *)bm, nwb, ix->stream));
            d.bm = (const uint4 *)bm;
            ix->index_bytes += nwb * 64;
        }
    }
    // ---- optional accelerators ---------------------------------------------------------------------------
    // Sizing rule (measured, tools/ldhint_bench.cu): random fetches run at ~46 G requests/s while the footprint a kernel touches stays
    // inside the ~64 GB TLB reach and fall off a cliff beyond (36 G/s at 80 GB, 19 G/s at 100 GB).  So the structures the count
    // kernel touches per query — k-mer table, row contexts, and the rank structure unless the table is deep enough that intervals
    // are down to a few rows when it has been consulted — are kept inside `reach`; everything else may fill the rest of the HBM.
    // fmx_opts.max_total_bytes caps the sum of everything resident.
    int accel = o.accel;
    if (accel & FMX_ACCEL_NONE) accel = FMX_ACCEL_NONE;
    size_t fr = 0, to = 0;
    CU(cudaStreamSynchronize(ix->stream));
    trim_pool(ix->device);
    cudaMemGetInfo(&fr, &to);
    double reach = 68e9;
    if (const char *env = std::getenv("FMX_TLB_REACH_GB")) { const double v = std::atof(env); if (v > 0) reach = v * 1e9; }
    const int64_t rank_bytes = (layout == FMX_LAYOUT_PLANES ? planes_bytes : wmx ? wmx_bytes : wm_bytes);
    if ((accel & FMX_ACCEL_CTX8) && accel != FMX_ACCEL_NONE && sigma > 4)
        return fail(FMX_E_UNSUPPORTED, "FMX_ACCEL_CTX8 stores 2-bit symbols: the text has %d distinct symbols (at most 4 fit)", sigma);
    auto room = [&]() { return total_cap - ix->index_bytes; };          // bytes the cap still allows
    const bool is_auto = accel == FMX_ACCEL_AUTO;
    // row contexts: the 32-byte form when it fits the reach (and leaves a quarter of the cap to the table); for alphabets of <= 4
    // symbols on larger texts the compact 8-byte form.  Construction needs sa + isa + text (9n) next to the entries.
    const bool fits32 = 32.0 * n + 4e9 <= reach && 41 * n + (8ll << 30) < (int64_t)fr && 32 * n <= room() - room() / 4;
    const bool fits8 = sigma <= 4 && 8.0 * n + 4e9 <= reach && 17 * n + (8ll << 30) < (int64_t)fr && 8 * n <= room() - room() / 4;
    const bool want_ctx = n > 2 && ((accel & FMX_ACCEL_CTX) || (is_auto && fits32));
    const bool want_ctx8 = n > 2 && sigma <= 4 && !want_ctx && ((accel & FMX_ACCEL_CTX8) || (is_auto && fits8));
    // isat (16n bytes, the singleton shortcut) only where no row contexts exist: a context entry does the same in one fetch
    const bool want_isat = n > 2 && ((accel & FMX_ACCEL_TEXT) || (is_auto && !want_ctx && !want_ctx8 && 25 * n + (2ll << 30) < (int64_t)fr &&
                                                                 ix->index_bytes + 20 * n <= budget + (24ll << 30) && 20 * n <= room() / 2));
    const bool build_sa = want_isat || want_ctx || want_ctx8;
    const bool want_kmer = (accel & (FMX_ACCEL_KMER | FMX_ACCEL_DICT)) || is_auto;
    if (build_sa) {
        // isa and the text are scratch that is folded into the isat / context entries; sa stays when it is wanted for locate
        SaBuf sa;                                                 // plain cudaMalloc: it may become a resident part of the index
        DBuf isa(ix->stream), text(ix->stream);
        CU(cudaMalloc(&sa.p, (size_t)n * 4)); CU(isa.alloc((size_t)n * 4)); CU(text.alloc((size_t)n + 16));
        std::string err;
        e = build_full_sa(d, layout, sa.as<uint32_t>(), isa.as<uint32_t>(), text.as<uint8_t>(), ix->stream, err);
        if (e != cudaSuccess) return fail(err.empty() ? FMX_E_CUDA : FMX_E_FORMAT, "suffix array construction failed: %s", err.empty() ? cudaGetErrorString(e) : err.c_str());
        int ibits = 1;
        while ((1 << ibits) < sigma + 1) ++ibits;                 // values 0..sigma: dense code + 1, 0 = '$'
        const int isyms = 96 / ibits;
        d.isat_bits = ibits; d.isat_syms = isyms;
        if (want_isat) {
            void *isat = nullptr;
            e = cudaMalloc(&isat, (size_t)n * 16); CU(e); ix->owned.push_back(isat);
            CU(build_isat(isa.as<uint32_t>(), text.as<uint8_t>(), d_code, n, ibits, isyms, (uint4 *)isat, ix->stream));
            d.isat = (const uint4 *)isat;
            ix->index_bytes += 16 * n;
        }
        if (want_ctx) {
            void *ctx = nullptr;
            e = cudaMalloc(&ctx, (size_t)n * 32);
            if (e != cudaSuccess) { cudaGetLastError(); if (accel & FMX_ACCEL_CTX) return fail(FMX_E_CUDA, "cannot allocate %lld bytes for the row contexts", (long long)n * 32); }
            else {
                ix->owned.push_back(ctx);
                const int raw = ibits == 8 ? 1 : 0;
                CtxHops hops;
                uint8_t plan[256];
                ctx_hop_plan(isyms, hops, plan);
                uint8_t *d_plan = dev_upload(ix, plan, 256, &e); CU(e);
                CU(build_ctx(sa.as<uint32_t>(), isa.as<uint32_t>(), text.as<uint8_t>(), d_code, n, ibits, isyms, raw, hops, (uint4 *)ctx, ix->stream));
                CU(cudaStreamSynchronize(ix->stream));             // `plan` is a local
                d.ctx = (const uint4 *)ctx; d.ctx_J = isyms; d.ctx_raw = raw; d.ctx_plan = d_plan;
                for (int t = 0; t < 8; ++t) d.ctx_S[t] = (uint8_t)hops.h[t];
                ix->index_bytes += 32 * n;
            }
        }
        if (want_ctx8) {
            void *ctx8 = nullptr;
            e = cudaMalloc(&ctx8, (size_t)n * 8);
            if (e != cudaSuccess) { cudaGetLastError(); if (accel & FMX_ACCEL_CTX8) return fail(FMX_E_CUDA, "cannot allocate %lld bytes for the compact row contexts", (long long)n * 8); }
            else {
                ix->owned.push_back(ctx8);
                CU(build_ctx8(sa.as<uint32_t>(), isa.as<uint32_t>(), text.as<uint8_t>(), d_code, n, 16, (uint2 *)ctx8, ix->stream));
                d.ctx8 = (const uint2 *)ctx8; d.ctx8_J = 16;
                ix->index_bytes += 8 * n;
            }
        }
        // the full suffix array stays resident (locate = one load per occurrence) when the singleton shortcut needs it, or when no sampled
        // SA was asked for and neither the cap nor FMX_ACCEL_NO_SA forbids it; otherwise it was scratch
        const bool keep_sa = want_isat || (o.sa_sample_rate == 0 && !(accel & FMX_ACCEL_NO_SA) && 4 * n <= room() - (want_kmer ? room() / 4 : 0));
        CU(cudaStreamSynchronize(ix->stream));
        if (keep_sa) {
            ix->owned.push_back(sa.p);
            d.sa = (const uint32_t *)sa.p;
            sa.p = nullptr;
            ix->index_bytes += 4 * n;
        }
    }
    trim_pool(ix->device);
    if (want_kmer && sigma >= 1) {
        size_t fr2 = 0, to2 = 0;
        cudaMemGetInfo(&fr2, &to2);
        const int64_t max_entries = std::min<int64_t>(1ll << 32, std::max<int64_t>(8 * n, 1 << 16));   // no point in far more entries than rows
        auto entries_of = [&](int k) { int64_t v = 1; for (int j = 0; j < k; ++j) { if (v > max_entries) return max_entries + 1; v *= sigma; } return v; };
        int K = 0;
        if (o.kmer_table_bytes > 0) {                                   // explicit budget
            while (K < 16 && entries_of(K + 1) <= max_entries && entries_of(K + 1) * 8 <= o.kmer_table_bytes && entries_of(K + 1) * 8 <= room()) ++K;
        } else {
            // the deepest table whose working set stays inside the TLB reach, a third of the free memory and the cap ...
            for (int k = 16; k >= 2 && K == 0; --k) {
                const int64_t en = entries_of(k);
                if (en > max_entries || en * 8 > (int64_t)(fr2 / 3) || en * 8 > room()) continue;
                const bool have_ctx = d.ctx != nullptr || d.ctx8 != nullptr;
                const bool saturating = have_ctx && en >= n / 2;            // intervals are a few rows once the table has been consulted
                const double ws = en * 8.0 + (d.ctx ? 32.0 * n : 0.0) + (d.ctx8 ? 8.0 * n : 0.0) +
                                  (saturating ? 0.0 : (double)rank_bytes + (d.isat && !have_ctx ? 20.0 * n : 0.0));
                if (ws <= reach) K = k;
            }
            // ... else (the rest of the index is already beyond the reach) 256 MiB .. 16 GiB scaled to a sixteenth of the free memory
            if (K == 0) {
                const int64_t table_budget = std::min<int64_t>(std::min<int64_t>(std::max<int64_t>(256ll << 20, (int64_t)(fr2 / 16)), 16ll << 30), room());
                while (K < 16 && entries_of(K + 1) <= std::min<int64_t>(max_entries, std::max<int64_t>(4 * n, 1 << 16)) && entries_of(K + 1) * 8 <= table_budget) ++K;
            }
        }
        if (sigma == 1) K = std::min(K, 16);
        if (K >= 2) {
            const int64_t entries = entries_of(K);
            void *tab = nullptr;
            e = cudaMalloc(&tab, (size_t)((entries + kKmerGroup - 1) / kKmerGroup) * kKmerGroup * 8); CU(e); ix->owned.push_back(tab);   // whole groups
            CU(build_kmer_table(d, ix->cfg, d_sym, (uint32_t)sigma, K, (uint2 *)tab, ix->stream));
            CU(cudaStreamSynchronize(ix->stream));
            d.kmer = (const uint2 *)tab; d.kmer_k = K; d.kmer_sigma = (uint32_t)sigma;
            ix->index_bytes += entries * 8;
        }
    }
    // dictionary of wide intervals on top of the dense table: only texts whose k-mers stay frequent beyond the table's depth (natural
    // language, repeats) have any; the level-wise construction finds out
    const bool want_dict = d.kmer != nullptr && sigma >= 2 && accel != FMX_ACCEL_NONE && ((accel & FMX_ACCEL_DICT) || is_auto);
    if (want_dict) {
        int dbits = 1;
        while ((1 << dbits) < sigma) ++dbits;
        const int Dmax = std::min(16, 60 / dbits);
        size_t fr3 = 0, to3 = 0;
        cudaMemGetInfo(&fr3, &to3);
        int64_t dict_budget = o.dict_bytes > 0 ? o.dict_bytes : std::min<int64_t>(12ll << 30, (int64_t)(fr3 / 8));
        dict_budget = std::min<int64_t>(dict_budget, room());
        const uint32_t min_rows = o.dict_min_rows > 0 ? (uint32_t)o.dict_min_rows : 2u;
        if (Dmax > d.kmer_k && dict_budget >= 4096) {
            void *table = nullptr;
            int64_t buckets = 0, entries = 0;
            int depth = 0, depth_x = 0, jc = 1;
            const uint32_t min_rows_top = o.dict_top_min_rows > 0 ? (uint32_t)o.dict_top_min_rows : 1u;
            e = build_dict(d, ix->cfg, d_sym, (uint32_t)sigma, dbits, Dmax, min_rows, min_rows_top, dict_budget / 32, &table, &buckets, &depth, &depth_x, &jc, &entries, ix->stream);
            if (e != cudaSuccess) { cudaGetLastError(); if (accel & FMX_ACCEL_DICT) return fail(FMX_E_CUDA, "dictionary construction failed: %s", cudaGetErrorString(e)); }
            else if (table) {
                ix->owned.push_back(table);
                d.dict = (const uint4 *)table; d.dict_buckets = (uint64_t)buckets; d.dict_D = depth; d.dict_bits = dbits; d.dict_Dx = depth_x; d.dict_Jc = jc;
                ix->dict_entries = entries;
                ix->index_bytes += buckets * 32;
            }
        }
        trim_pool(ix->device);
    }
    // k-mer group blocks: with a saturating table (intervals of about one row) most queries that go on with a full-depth hop through the row
    // contexts find the rows' contexts in the table's own 64-byte block — one request instead of two (DESIGN.md §3/§5).  The group form needs
    // the lexicographic order, so the table is built again in that order (same bytes, no more memory); the dictionary is grown from the
    // plain order and is not combined with it.  FMX_KMER_ROWS=0 keeps the plain table (the A/B switch of the measurement).
    const char *kr_env = std::getenv("FMX_KMER_ROWS");
    const bool want_groups = !(kr_env && std::atoi(kr_env) == 0);
    if (want_groups && is_auto && d.kmer != nullptr && d.ctx != nullptr && d.dict == nullptr && std::pow((double)sigma, d.kmer_k) >= n / 2.0) {
        uint64_t entries = 1;
        for (int j = 0; j < d.kmer_k; ++j) entries *= (uint64_t)sigma;
        uint2 *tab = const_cast<uint2 *>(d.kmer);
        CU(build_kmer_table(d, ix->cfg, d_sym, (uint32_t)sigma, d.kmer_k, tab, ix->stream, true));
        CU(pack_kmer_groups(tab, entries, d.ctx, ix->stream));
        CU(cudaStreamSynchronize(ix->stream));
        d.kmer_rows = (int32_t)kKmerInlineRows;
    }
    // two lanes per query: with the 256-bit load a 64-B rank block is one request from two lanes (as from four lanes with 128-bit
    // loads), and twice as many queries are in flight per SM
    if (!o.lanes_per_query) {
        ix->cfg.lanes = wmx ? 4 : 2;                        // a 128-byte multi-ary block is one request from four lanes x 256 bits
        // count kernels: one lane per query once a deep table + row contexts answer most queries in two single-lane requests
        // (measured on cfg 2: 19.96 vs 18.69 G q/s; the kernel at two lanes is issue-bound, 80 % of the issue slots)
        const bool saturating = (d.ctx != nullptr || d.ctx8 != nullptr) && d.kmer != nullptr && std::pow((double)sigma, d.kmer_k) >= n / 2.0;
        ix->cfg.count_lanes = saturating ? 1 : 0;
    }
    ix->accel_text = d.isat != nullptr;
    ix->kmer_k = d.kmer ? d.kmer_k : 0;
    ix->d_full = d;
    ix->count_lanes_full = ix->cfg.count_lanes;
    CU(cudaStreamSynchronize(ix->stream));
    trim_pool(ix->device);                              // construction scratch goes back to the device
    return FMX_OK;
}

int new_index(const fmx_opts *opts, fmx_index **out, fmx_opts *resolved) {
    fmx_opts o;
    fmx_opts_default(&o);
    if (opts) o = *opts;
    int dev = 0;
    int rc = ensure_device(o.device, &dev);
    if (rc) return rc;
    fmx_index *ix = new fmx_index();
    ix->device = dev;
    if (cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ix->h2d, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ix->d2h, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&ix->ev0) != cudaSuccess ||
        cudaEventCreate(&ix->ev1) != cudaSuccess || cudaEventCreateWithFlags(&ix->ev_alloc, cudaEventDisableTiming) != cudaSuccess) {
        delete ix;
        return fail(FMX_E_CUDA, "cannot create CUDA stream/events");
    }
    {   // keep freed stream-ordered allocations cached in the pool: batch calls reuse them instead of re-mapping
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    *out = ix;
    *resolved = o;
    return FMX_OK;
}

// FMX_TRACE=1: host-side phase times of the batch calls on stderr (where does an end-to-end call spend its time)
struct Phases {
    bool on = std::getenv("FMX_TRACE") != nullptr;
    const char *what;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    explicit Phases(const char *w) : what(w) {}
    void mark(const char *phase) {
        if (!on) return;
        auto t1 = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[fmx trace] %s: %-22s %8.3f ms\n", what, phase, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define CHECK_IX(ix) do { if (!(ix)) return fail(FMX_E_ARG, "null index"); } while (0)

}  // namespace

// =========================================================================================================
extern "C" {

void fmx_opts_default(fmx_opts *o) {
    if (!o) return;
    std::memset(o, 0, sizeof *o);
    o->device = -1;
    o->layout = FMX_LAYOUT_AUTO;
    o->sa_sample_rate = 0;
}

const char *fmx_version(void) { return "fmgpu 0.1 (sm_100a)"; }

int fmx_open(const char *path, int big_endian, const fmx_opts *opts, fmx_index **out) {
    if (!path || !out) return fail(FMX_E_ARG, "null argument");
    *out = nullptr;
    fmx_opts o;
    fmx_opts_default(&o);
    if (opts) o = *opts;
    IndexFiles f;
    int rc = load_index_files(strip_extension(path), big_endian != 0, o.require_fm != 0, f);   // validate before touching the GPU
    if (rc) return rc;
    fmx_index *ix = nullptr;
    rc = new_index(&o, &ix, &o);
    if (rc) return rc;
    rc = upload_index(ix, f.bwt.data(), f.n, f.eof, f.counts, o);
    if (rc) { fmx_close(ix); return rc; }
    *out = ix;
    return FMX_OK;
}

int fmx_open_mem(const uint8_t *bwt, int64_t n, int64_t eof, const int64_t counts[256], const fmx_opts *opts, fmx_index **out) {
    if (!bwt || !counts || !out) return fail(FMX_E_ARG, "null argument");
    *out = nullptr;
    fmx_opts o;
    fmx_index *ix = nullptr;
    int rc = new_index(opts, &ix, &o);
    if (rc) return rc;
    rc = upload_index(ix, bwt, n, eof, counts, o);
    if (rc) { fmx_close(ix); return rc; }
    *out = ix;
    return FMX_OK;
}

int fmx_close(fmx_index *ix) {
    if (!ix) return FMX_OK;
    cudaSetDevice(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    for (void *p : ix->owned) cudaFree(p);
    trim_pool(ix->device);                                     // hand the cached stream-ordered scratch back: the next open (or suffix sort) may need all of it
    for (auto &st : ix->sets) {
        if (st.stream) { cudaStreamSynchronize(st.stream); cudaStreamDestroy(st.stream); }
        if (st.h2d) cudaStreamDestroy(st.h2d);
        if (st.d2h) cudaStreamDestroy(st.d2h);
        if (st.ev0) cudaEventDestroy(st.ev0);
        if (st.ev1) cudaEventDestroy(st.ev1);
        if (st.ev_alloc) cudaEventDestroy(st.ev_alloc);
    }
    if (ix->ev0) cudaEventDestroy(ix->ev0);
    if (ix->ev1) cudaEventDestroy(ix->ev1);
    if (ix->ev_alloc) cudaEventDestroy(ix->ev_alloc);
    if (ix->h2d) cudaStreamDestroy(ix->h2d);
    if (ix->d2h) cudaStreamDestroy(ix->d2h);
    if (ix->stream) cudaStreamDestroy(ix->stream);
    delete ix;
    return FMX_OK;
}

int64_t fmx_n(const fmx_index *ix) { return ix ? ix->n : -1; }
int64_t fmx_eof(const fmx_index *ix) { return ix ? ix->eof : -1; }
int fmx_ctable(const fmx_index *ix, int64_t C[256]) {
    CHECK_IX(ix);
    if (!C) return fail(FMX_E_ARG, "null argument");
    for (int c = 0; c < 256; ++c) C[c] = ix->C[c];
    return FMX_OK;
}
int fmx_accel_info(const fmx_index *ix, int32_t *kmer_k, int32_t *text_shortcut) {
    CHECK_IX(ix);
    if (kmer_k) *kmer_k = ix->kmer_k;
    if (text_shortcut) *text_shortcut = ix->accel_text ? 1 : 0;
    return FMX_OK;
}
int fmx_dict_info(const fmx_index *ix, int32_t *depth, int32_t *chain_depth, int64_t *entries, int64_t *bytes) {
    if (!ix) return fail(FMX_E_ARG, "null index");
    if (depth) *depth = ix->d.dict ? ix->d.dict_D : 0;
    if (chain_depth) *chain_depth = ix->d.dict ? ix->d.dict_Dx : 0;
    if (entries) *entries = ix->d.dict ? ix->dict_entries : 0;
    if (bytes) *bytes = ix->d.dict ? (int64_t)ix->d.dict_buckets * 32 : 0;
    return FMX_OK;
}
int fmx_kmer_rows(const fmx_index *ix) { return ix && ix->d.kmer ? ix->d.kmer_rows : 0; }
int fmx_ctx_depth(const fmx_index *ix) { return !ix ? 0 : ix->d.ctx ? ix->d.ctx_J : ix->d.ctx8 ? ix->d.ctx8_J : 0; }
int fmx_ctx_entry_bytes(const fmx_index *ix) { return !ix ? 0 : ix->d.ctx ? 32 : ix->d.ctx8 ? 8 : 0; }
int fmx_info(const fmx_index *ix, int32_t *layout, int32_t *levels, int32_t *sigma, int64_t *index_bytes, int32_t *rate) {
    CHECK_IX(ix);
    if (layout) *layout = ix->api_layout;
    if (levels) *levels = ix->api_layout == FMX_LAYOUT_WM ? ix->levels : ix->api_layout == FMX_LAYOUT_WMX ? ix->d_full.wmx_levels : 1;
    if (sigma) *sigma = ix->sigma;
    if (index_bytes) *index_bytes = ix->index_bytes;
    if (rate) *rate = ix->sample_rate;
    return FMX_OK;
}
int fmx_set_lanes(fmx_index *ix, int32_t lanes) {
    CHECK_IX(ix);
    if (lanes != 1 && lanes != 2 && lanes != 4) return fail(FMX_E_ARG, "lanes_per_query must be 1, 2 or 4");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->cfg.lanes = lanes;
    ix->cfg.count_lanes = 0;
    return FMX_OK;
}
// Hides built accelerators from subsequent calls (FMX_ACCEL_* bits to keep; FMX_ACCEL_NONE = plain backward search over the rank
// structure, FMX_ACCEL_AUTO = everything that was built): measures the same index with and without them, without a second open.
int fmx_set_accel_mask(fmx_index *ix, int32_t mask) {
    CHECK_IX(ix);
    std::lock_guard<std::mutex> lk(ix->mu);
    DevIndex d = ix->d_full;
    if (mask != FMX_ACCEL_AUTO) {
        if ((mask & FMX_ACCEL_NONE) || !(mask & FMX_ACCEL_KMER)) { d.kmer = nullptr; d.kmer_k = 0; }
        if ((mask & FMX_ACCEL_NONE) || !(mask & FMX_ACCEL_TEXT)) d.isat = nullptr;
        if ((mask & FMX_ACCEL_NONE) || !(mask & FMX_ACCEL_CTX)) d.ctx = nullptr;
        if ((mask & FMX_ACCEL_NONE) || !(mask & FMX_ACCEL_CTX8)) d.ctx8 = nullptr;
        if ((mask & FMX_ACCEL_NONE) || !(mask & FMX_ACCEL_DICT) || !d.kmer) d.dict = nullptr;
    }
    ix->d = d;
    ix->cfg.count_lanes = (d.kmer && (d.ctx || d.ctx8)) ? ix->count_lanes_full : 0;
    ix->accel_text = d.isat != nullptr;
    ix->kmer_k = d.kmer ? d.kmer_k : 0;
    return FMX_OK;
}
int fmx_set_chunk(fmx_index *ix, int64_t queries_per_chunk) {
    CHECK_IX(ix);
    if (queries_per_chunk < 0) return fail(FMX_E_ARG, "bad chunk");
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->chunk_queries = queries_per_chunk;
    return FMX_OK;
}
int fmx_set_l2_fetch_granularity(int32_t bytes, int32_t *effective) {
    int dev = 0;
    int rc = ensure_device(-1, &dev);
    if (rc) return rc;
    if (bytes > 0) CU(cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)bytes));
    size_t v = 0;
    CU(cudaDeviceGetLimit(&v, cudaLimitMaxL2FetchGranularity));
    if (effective) *effective = (int32_t)v;
    return FMX_OK;
}
int fmx_host_alloc(void **p, int64_t bytes) {
    if (!p || bytes < 0) return fail(FMX_E_ARG, "bad argument");
    int dev = 0;
    int rc = ensure_device(-1, &dev);
    if (rc) return rc;
    CU(cudaHostAlloc(p, (size_t)(bytes ? bytes : 1), cudaHostAllocPortable));
    return FMX_OK;
}
int fmx_host_free(void *p) {
    if (p) CU(cudaFreeHost(p));
    return FMX_OK;
}
int fmx_get_lanes(const fmx_index *ix) { return ix ? (ix->cfg.count_lanes ? ix->cfg.count_lanes : ix->cfg.lanes) : 0; }
double fmx_last_kernel_ms(const fmx_index *ix) { return ix ? ix->last_ms.load() : 0.0; }
int64_t fmx_last_kernel_launches(const fmx_index *ix) { return ix ? ix->last_launches.load() : 0; }
int64_t fmx_last_regex_levels(const fmx_index *ix) { return ix ? ix->last_levels.load() : 0; }

// pos2char: bwtmerger.scala:376-385 (bucketStarts0 = prefix sums of the raw counts)
int fmx_pos2char(const fmx_index *ix, int64_t key, int32_t *c) {
    CHECK_IX(ix);
    if (!c) return fail(FMX_E_ARG, "null argument");
    int64_t bs0[256], tot = 0;
    for (int i = 0; i < 256; ++i) { bs0[i] = tot; tot += ix->counts0[i]; }
    int i = 255;
    if (bs0[i] > key) { while (bs0[i] > key && i > 0) --i; }
    else { while (bs0[i - 1] == bs0[i] && i > 1) --i; --i; }
    *c = i;
    return FMX_OK;
}

// ---- element-wise operator batches -----------------------------------------------------------------------
int fmx_occ_batch(fmx_index *ix, const uint8_t *c, const int64_t *key, int64_t m, int64_t *out) {
    CHECK_IX(ix);
    if (m < 0 || (m && (!c || !key || !out))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dc(st), dk(st), dout(st);
    CU(dc.alloc(m)); CU(dk.alloc(m * 8)); CU(dout.alloc(m * 8));
    CU(cudaMemcpyAsync(dc.p, c, m, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dk.p, key, m * 8, cudaMemcpyHostToDevice, st));
    Timed t(ix, cc);
    CU(launch_occ(cc.d, cc.cfg, dc.as<uint8_t>(), dk.as<int64_t>(), m, dout.as<int64_t>(), st));
    ix->last_launches = 1; ix->total_launches += 1;
    t.stop();
    CU(cudaMemcpyAsync(out, dout.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    t.collect();
    return FMX_OK;
}

int fmx_prev_range_batch(fmx_index *ix, const int64_t *sp, const int64_t *ep, const uint8_t *c, int64_t m, int64_t *sp1, int64_t *ep1) {
    CHECK_IX(ix);
    if (m < 0 || (m && (!sp || !ep || !c || !sp1 || !ep1))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    for (int64_t i = 0; i < m; ++i)
        if (sp[i] < 0 || ep[i] < 0 || sp[i] > ix->n || ep[i] > ix->n) return fail(FMX_E_ARG, "row out of range at %lld", (long long)i);
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dsp(st), dep(st), dc(st), o1(st), o2(st);
    CU(dsp.alloc(m * 8)); CU(dep.alloc(m * 8)); CU(dc.alloc(m)); CU(o1.alloc(m * 8)); CU(o2.alloc(m * 8));
    CU(cudaMemcpyAsync(dsp.p, sp, m * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dep.p, ep, m * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dc.p, c, m, cudaMemcpyHostToDevice, st));
    Timed t(ix, cc);
    CU(launch_prev_range(cc.d, cc.cfg, dsp.as<int64_t>(), dep.as<int64_t>(), dc.as<uint8_t>(), m, o1.as<int64_t>(), o2.as<int64_t>(), st));
    ix->last_launches = 1; ix->total_launches += 1;
    t.stop();
    CU(cudaMemcpyAsync(sp1, o1.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(ep1, o2.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    t.collect();
    return FMX_OK;
}

int fmx_interval_prev_range(fmx_index *ix, int64_t sp, int64_t ep, int cstart, int cend, int32_t *out_c, int64_t *out_sp,
                            int64_t *out_ep, int64_t *n_out) {
    CHECK_IX(ix);
    if (!n_out) return fail(FMX_E_ARG, "null argument");
    *n_out = 0;
    if (cstart < 0 || cend > 255 || sp < 0 || ep < 0 || sp > ix->n || ep > ix->n) return fail(FMX_E_ARG, "bad argument");
    const int m = cend - cstart + 1;
    if (m <= 0) return FMX_OK;
    if (!out_c || !out_sp || !out_ep) return fail(FMX_E_ARG, "null argument");
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf o1(st), o2(st);
    CU(o1.alloc(m * 8)); CU(o2.alloc(m * 8));
    Timed t(ix, cc);
    CU(launch_interval_prev_range(cc.d, cc.cfg, sp, ep, cstart, cend, o1.as<int64_t>(), o2.as<int64_t>(), st));
    ix->last_launches = 1; ix->total_launches += 1;
    t.stop();
    std::vector<int64_t> a(m), b(m);
    CU(cudaMemcpyAsync(a.data(), o1.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(b.data(), o2.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    t.collect();
    int64_t k = 0;
    for (int c = cend; c >= cstart; --c)                       // the reference prepends while c ascends
        if (a[c - cstart] < b[c - cstart]) { out_c[k] = c; out_sp[k] = a[c - cstart]; out_ep[k] = b[c - cstart]; ++k; }
    *n_out = k;
    return FMX_OK;
}

// ---- count -------------------------------------------------------------------------------------------------
int fmx_count_fixed_dev(fmx_index *ix, const void *d_pat, int32_t len, int64_t m, void *d_sp, void *d_ep, void *stream) {
    CHECK_IX(ix);
    if (len < 0 || m < 0 || (m && (!d_sp || !d_ep || (len && !d_pat)))) return fail(FMX_E_ARG, "bad argument");
    CallCtx cc(ix);
    CHECK_CC(cc);                    // cfg and the launch counters are shared with the host-buffer calls; the launch is asynchronous
    DeviceGuard g(ix->device);
    CU(launch_count_fixed(cc.d, cc.cfg, (const uint8_t *)d_pat, len, m, d_sp, d_ep, false, nullptr, (cudaStream_t)stream));
    ix->last_launches = 1; ix->total_launches += 1;
    return FMX_OK;
}

// Host-buffer count: the batch is cut into chunks that flow through three streams — H2D of chunk k+1, the count
// kernel on chunk k and the D2H of chunk k-1 overlap (PCIe is full duplex).  With pinned (fmx_host_alloc'ed or
// cudaHostRegister'ed) caller buffers every copy is an asynchronous DMA; with pageable buffers the driver stages
// the copies and the pipeline degrades gracefully to copy-then-compute.
// Fused count + all-gather: every hit count is also stored into n_sinks gathered buffers (this rank's own and its peers',
// opened with fmx_ipc_import) at element offset `offset`.  The caller orders the consumers behind the producers
// (stream order on this GPU plus one tiny cross-rank barrier per step).
int fmx_count_fixed_dev_gather(fmx_index *ix, const void *d_pat, int32_t len, int64_t m, void *d_sp, void *d_ep,
                               void *const *sinks, int32_t n_sinks, int64_t offset, void *stream) {
    CHECK_IX(ix);
    if (len < 0 || m < 0 || n_sinks < 0 || n_sinks > 8 || offset < 0 || (n_sinks && !sinks) || (m && (!d_sp || !d_ep || (len && !d_pat))))
        return fail(FMX_E_ARG, "bad argument");
    PeerSinks ps{};
    ps.n = n_sinks;
    ps.offset = offset;
    for (int j = 0; j < n_sinks; ++j) { if (!sinks[j]) return fail(FMX_E_ARG, "null sink %d", j); ps.p[j] = (uint32_t *)sinks[j]; }
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    CU(launch_count_fixed(cc.d, cc.cfg, (const uint8_t *)d_pat, len, m, d_sp, d_ep, false, nullptr, (cudaStream_t)stream, &ps));
    ix->last_launches = 1; ix->total_launches += 1;
    return FMX_OK;
}

// ---- raw device buffers that can be shared between the ranks of one node (CUDA IPC) -----------------------------------
int fmx_dev_alloc(void **p, int64_t bytes) {
    if (!p || bytes < 0) return fail(FMX_E_ARG, "bad argument");
    // Sizes are rounded up to 2 MiB: cudaMalloc packs smaller requests into shared 2 MiB blocks, and CUDA IPC shares (and maps) the
    // whole underlying block — a peer that opened the handle of the second buffer of a block got the block's base, i.e. the first
    // buffer (seen on 2 x B200: one exchange's counts landing in an earlier exchange's buffer).
    const size_t gran = 2u << 20, sz = ((size_t)(bytes ? bytes : 1) + gran - 1) / gran * gran;
    CU(cudaMalloc(p, sz));
    CU(cudaMemset(*p, 0, sz));
    return FMX_OK;
}
int fmx_dev_free(void *p) { if (p) CU(cudaFree(p)); return FMX_OK; }
int fmx_ipc_export(void *p, uint8_t handle[64]) {
    if (!p || !handle) return fail(FMX_E_ARG, "bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, p));
    std::memcpy(handle, &h, 64);
    return FMX_OK;
}
int fmx_ipc_import(const uint8_t handle[64], void **p) {
    if (!p || !handle) return fail(FMX_E_ARG, "bad argument");
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    CU(cudaIpcOpenMemHandle(p, h, cudaIpcMemLazyEnablePeerAccess));
    return FMX_OK;
}
int fmx_ipc_close(void *p) { if (p) CU(cudaIpcCloseMemHandle(p)); return FMX_OK; }
int fmx_memcpy_d2h(void *dst, const void *src, int64_t bytes) {
    if (bytes < 0 || (bytes && (!dst || !src))) return fail(FMX_E_ARG, "bad argument");
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost));
    return FMX_OK;
}

// packed2_alphabet != nullptr: `pat` holds 2-bit symbol codes, (len+3)/4 bytes per pattern (symbol j = bits 2(j%4) of byte j/4), which are
// expanded to the alphabet's bytes on the device after crossing PCIe at a quarter of the size
static int count_fixed_pipeline(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m, int64_t *sp, int64_t *ep, uint32_t *counts,
                                int32_t *sp32 = nullptr, int32_t *ep32 = nullptr, const uint8_t *packed2_alphabet = nullptr) {
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    const bool only_counts = counts != nullptr, narrow = sp32 != nullptr;     // narrow: 32-bit rows out (the reference's Int / uint32 rows)
    const bool packed = packed2_alphabet != nullptr;
    const int64_t wire_len = packed ? (len + 3) / 4 : len;                    // bytes per pattern on the wire
    uint32_t alpha4 = 0;
    if (packed) alpha4 = (uint32_t)packed2_alphabet[0] | ((uint32_t)packed2_alphabet[1] << 8) | ((uint32_t)packed2_alphabet[2] << 16) | ((uint32_t)packed2_alphabet[3] << 24);
    DBuf dp(st), dsp(st), dep(st), dcnt(st), dwire(st);
    CU(dp.alloc((size_t)m * len + 16));
    if (packed) CU(dwire.alloc((size_t)m * wire_len));
    CU(dsp.alloc(m * ((only_counts || narrow) ? 4 : 8))); CU(dep.alloc(m * ((only_counts || narrow) ? 4 : 8)));
    if (only_counts) CU(dcnt.alloc(m * 4));
    const int64_t chunk = cc.chunk_queries > 0 ? cc.chunk_queries : (1 << 20);
    const int64_t nchunks = (m + chunk - 1) / chunk;
    Events evs_in, evs_k;
    CU(evs_in.make((size_t)nchunks)); CU(evs_k.make((size_t)nchunks));
    std::vector<cudaEvent_t> &ev_in = evs_in.v, &ev_k = evs_k.v;
    // the copy streams may touch the stream-ordered allocations only after the allocating stream reached this point
    CU(cudaEventRecord(cc.ev_alloc, st));
    CU(cudaStreamWaitEvent(cc.h2d, cc.ev_alloc, 0));
    CU(cudaStreamWaitEvent(cc.d2h, cc.ev_alloc, 0));
    Timed t(ix, cc);
    int rc = FMX_OK;
    for (int64_t k = 0; k < nchunks && rc == FMX_OK; ++k) {
        const int64_t q0 = k * chunk, nq = std::min(chunk, m - q0);
        cudaError_t e = cudaSuccess;
        uint8_t *wire_dst = packed ? dwire.as<uint8_t>() + q0 * wire_len : dp.as<uint8_t>() + q0 * len;
        if (len) e = cudaMemcpyAsync(wire_dst, pat + q0 * wire_len, (size_t)nq * wire_len, cudaMemcpyHostToDevice, cc.h2d);
        if (e == cudaSuccess) e = cudaEventRecord(ev_in[(size_t)k], cc.h2d);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(st, ev_in[(size_t)k], 0);
        if (e == cudaSuccess && packed && len) e = launch_unpack2(wire_dst, len, nq, alpha4, dp.as<uint8_t>() + q0 * len, st);
        if (e == cudaSuccess) {
            if (only_counts) {                       // ep-sp lands in dcnt through the kernel's fused-exchange sink; only that goes back
                PeerSinks ps{};
                ps.n = 1; ps.offset = q0; ps.p[0] = dcnt.as<uint32_t>();
                e = launch_count_fixed(cc.d, cc.cfg, dp.as<uint8_t>() + q0 * len, len, nq, dsp.as<uint32_t>() + q0, dep.as<uint32_t>() + q0, false, nullptr, st, &ps);
            } else if (narrow) {
                e = launch_count_fixed(cc.d, cc.cfg, dp.as<uint8_t>() + q0 * len, len, nq, dsp.as<uint32_t>() + q0, dep.as<uint32_t>() + q0, false, nullptr, st);
            } else {
                e = launch_count_fixed(cc.d, cc.cfg, dp.as<uint8_t>() + q0 * len, len, nq, dsp.as<int64_t>() + q0, dep.as<int64_t>() + q0, true, nullptr, st);
            }
        }
        if (e == cudaSuccess) e = cudaEventRecord(ev_k[(size_t)k], st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(cc.d2h, ev_k[(size_t)k], 0);
        if (only_counts) {
            if (e == cudaSuccess) e = cudaMemcpyAsync(counts + q0, dcnt.as<uint32_t>() + q0, (size_t)nq * 4, cudaMemcpyDeviceToHost, cc.d2h);
        } else if (narrow) {
            if (e == cudaSuccess) e = cudaMemcpyAsync(sp32 + q0, dsp.as<uint32_t>() + q0, (size_t)nq * 4, cudaMemcpyDeviceToHost, cc.d2h);
            if (e == cudaSuccess) e = cudaMemcpyAsync(ep32 + q0, dep.as<uint32_t>() + q0, (size_t)nq * 4, cudaMemcpyDeviceToHost, cc.d2h);
        } else {
            if (e == cudaSuccess) e = cudaMemcpyAsync(sp + q0, dsp.as<int64_t>() + q0, (size_t)nq * 8, cudaMemcpyDeviceToHost, cc.d2h);
            if (e == cudaSuccess) e = cudaMemcpyAsync(ep + q0, dep.as<int64_t>() + q0, (size_t)nq * 8, cudaMemcpyDeviceToHost, cc.d2h);
        }
        if (e != cudaSuccess) rc = fail(FMX_E_CUDA, "CUDA error %s in the count pipeline (%s)", cudaGetErrorName(e), cudaGetErrorString(e));
    }
    ix->last_launches = nchunks * (packed ? 2 : 1); ix->total_launches += nchunks * (packed ? 2 : 1);
    t.stop();
    cudaError_t e1 = cudaStreamSynchronize(cc.h2d), e2 = cudaStreamSynchronize(st), e3 = cudaStreamSynchronize(cc.d2h);
    if (rc == FMX_OK && (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess))
        rc = fail(FMX_E_CUDA, "CUDA error while draining the count pipeline");
    t.collect();
    return rc;
}

int fmx_count_fixed(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m, int64_t *sp, int64_t *ep) {
    CHECK_IX(ix);
    if (len < 0 || m < 0 || (m && (!sp || !ep || (len && !pat)))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    return count_fixed_pipeline(ix, pat, len, m, sp, ep, nullptr);
}

// The reference's own result width: Option[(Int, Int)] (findex.scala:15-31) — 32-bit rows, half the result bytes over PCIe.
int fmx_count_fixed_i32(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m, int32_t *sp, int32_t *ep) {
    CHECK_IX(ix);
    if (len < 0 || m < 0 || (m && (!sp || !ep || (len && !pat)))) return fail(FMX_E_ARG, "bad argument");
    if (ix->n > 0x7FFFFFFFll) return fail(FMX_E_UNSUPPORTED, "n = %lld does not fit the reference's Int rows; use fmx_count_fixed", (long long)ix->n);
    if (m == 0) return FMX_OK;
    return count_fixed_pipeline(ix, pat, len, m, nullptr, nullptr, nullptr, sp, ep);
}

// Count only: counts[q] = ep - sp of search(pattern q) (0 for None) — for callers that want the number of occurrences and not
// the interval; moves 4 instead of 16 result bytes per query over PCIe.
int fmx_count_only_fixed(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m, uint32_t *counts) {
    CHECK_IX(ix);
    if (len < 0 || m < 0 || (m && (!counts || (len && !pat)))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    return count_fixed_pipeline(ix, pat, len, m, nullptr, nullptr, counts);
}

// Patterns over an alphabet of <= 4 symbols as 2-bit codes on the wire (a DNA read of 32 bases = 8 bytes instead of 32): pattern q occupies
// bytes [q * ceil(len/4), (q+1) * ceil(len/4)), symbol j = alphabet[(byte[j/4] >> 2(j%4)) & 3].  Rows come back as uint32 (n < 2^32 always
// holds on this build) when row_bytes = 4, as int64 when 8.  Same (sp, ep) as fmx_count_fixed on the expanded patterns.
int fmx_count_fixed_packed2(fmx_index *ix, const uint8_t *codes, const uint8_t alphabet[4], int32_t len, int64_t m, void *sp, void *ep, int32_t row_bytes) {
    CHECK_IX(ix);
    if (len < 0 || m < 0 || !alphabet || (row_bytes != 4 && row_bytes != 8) || (m && (!sp || !ep || (len && !codes)))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    if (row_bytes == 4) return count_fixed_pipeline(ix, codes, len, m, nullptr, nullptr, nullptr, (int32_t *)sp, (int32_t *)ep, alphabet);
    return count_fixed_pipeline(ix, codes, len, m, (int64_t *)sp, (int64_t *)ep, nullptr, nullptr, nullptr, alphabet);
}

int fmx_count_batch(fmx_index *ix, const uint8_t *pat, const int64_t *off, int64_t m, int64_t *sp, int64_t *ep) {
    CHECK_IX(ix);
    if (m < 0 || (m && (!off || !sp || !ep))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    for (int64_t i = 0; i < m; ++i) if (off[i + 1] < off[i] || off[i] < 0) return fail(FMX_E_ARG, "offsets must be non-decreasing");
    const int64_t nbytes = off[m];
    if (nbytes && !pat) return fail(FMX_E_ARG, "null pattern buffer");
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dp(st), doff(st), dsp(st), dep(st);
    CU(dp.alloc(nbytes)); CU(doff.alloc((m + 1) * 8)); CU(dsp.alloc(m * 8)); CU(dep.alloc(m * 8));
    if (nbytes) CU(cudaMemcpyAsync(dp.p, pat, nbytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(doff.p, off, (m + 1) * 8, cudaMemcpyHostToDevice, st));
    Timed t(ix, cc);
    CU(launch_count_var(cc.d, cc.cfg, dp.as<uint8_t>(), doff.as<int64_t>(), m, dsp.as<int64_t>(), dep.as<int64_t>(), st));
    ix->last_launches = 1; ix->total_launches += 1;
    t.stop();
    CU(cudaMemcpyAsync(sp, dsp.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(ep, dep.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    t.collect();
    return FMX_OK;
}

int fmx_count_fixed_stats(fmx_index *ix, const uint8_t *pat, int32_t len, int64_t m, int64_t *blocks, int64_t *steps) {
    CHECK_IX(ix);
    if (len < 0 || m < 0 || (m && len && !pat)) return fail(FMX_E_ARG, "bad argument");
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dp(st), dsp(st), dep(st), ds(st);
    CU(dp.alloc((size_t)m * len)); CU(dsp.alloc(m * 4)); CU(dep.alloc(m * 4)); CU(ds.alloc(16));
    if (m && len) CU(cudaMemcpyAsync(dp.p, pat, (size_t)m * len, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(ds.p, 0, 16, st));
    CU(launch_count_fixed(cc.d, cc.cfg, dp.as<uint8_t>(), len, m, dsp.p, dep.p, false, ds.as<unsigned long long>(), st));
    unsigned long long h[2] = {0, 0};
    CU(cudaMemcpyAsync(h, ds.p, 16, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (blocks) *blocks = (int64_t)h[0];
    if (steps) *steps = (int64_t)h[1];
    return FMX_OK;
}

// ---- LF / FL / extraction -----------------------------------------------------------------------------------
int fmx_get_prev_i_batch(fmx_index *ix, const int64_t *row, int64_t m, int64_t *out) {
    CHECK_IX(ix);
    if (m < 0 || (m && (!row || !out))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    for (int64_t i = 0; i < m; ++i) if (row[i] < 0 || row[i] >= ix->n) return fail(FMX_E_ARG, "row out of range at %lld", (long long)i);
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dr(st), dout(st);
    CU(dr.alloc(m * 8)); CU(dout.alloc(m * 8));
    CU(cudaMemcpyAsync(dr.p, row, m * 8, cudaMemcpyHostToDevice, st));
    Timed t(ix, cc);
    CU(launch_lf(cc.d, cc.cfg, dr.as<int64_t>(), m, dout.as<int64_t>(), st));
    ix->last_launches = 1; ix->total_launches += 1;
    t.stop();
    CU(cudaMemcpyAsync(out, dout.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    t.collect();
    return FMX_OK;
}

int fmx_prev_substr_batch(fmx_index *ix, const int64_t *row, int64_t m, int32_t len, uint8_t *out, int32_t *out_len) {
    CHECK_IX(ix);
    if (m < 0 || len < 0 || (m && (!row || (len && !out)))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    for (int64_t i = 0; i < m; ++i) if (row[i] < 0 || row[i] >= ix->n) return fail(FMX_E_ARG, "row out of range at %lld", (long long)i);
    if (out_len) for (int64_t i = 0; i < m; ++i) out_len[i] = len;      // prevSubstr never stops early (its eof flag is never set)
    if (len == 0) return FMX_OK;
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dr(st), dout(st);
    CU(dr.alloc(m * 8)); CU(dout.alloc((size_t)m * len));
    CU(cudaMemcpyAsync(dr.p, row, m * 8, cudaMemcpyHostToDevice, st));
    Timed t(ix, cc);
    CU(launch_prev_substr(cc.d, cc.cfg, dr.as<int64_t>(), m, len, dout.as<uint8_t>(), st));
    ix->last_launches = 1; ix->total_launches += 1;
    t.stop();
    CU(cudaMemcpyAsync(out, dout.p, (size_t)m * len, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    t.collect();
    return FMX_OK;
}

int fmx_get_next_i_batch(fmx_index *ix, const int64_t *row, int64_t m, int64_t *out) {
    CHECK_IX(ix);
    if (m < 0 || (m && (!row || !out))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    for (int64_t i = 0; i < m; ++i) if (row[i] < 0 || row[i] >= ix->n) return fail(FMX_E_ARG, "row out of range at %lld", (long long)i);
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dr(st), dout(st);
    CU(dr.alloc(m * 8)); CU(dout.alloc(m * 8));
    CU(cudaMemcpyAsync(dr.p, row, m * 8, cudaMemcpyHostToDevice, st));
    Timed t(ix, cc);
    CU(launch_fl(cc.d, cc.cfg, dr.as<int64_t>(), m, dout.as<int64_t>(), st));
    ix->last_launches = 1; ix->total_launches += 1;
    t.stop();
    CU(cudaMemcpyAsync(out, dout.p, m * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    t.collect();
    return FMX_OK;
}

int fmx_next_substr_batch(fmx_index *ix, const int64_t *row, int64_t m, int32_t len, uint8_t *out, int32_t *out_len) {
    CHECK_IX(ix);
    if (m < 0 || len < 0 || (m && (!row || !out_len || (len && !out)))) return fail(FMX_E_ARG, "bad argument");
    if (m == 0) return FMX_OK;
    for (int64_t i = 0; i < m; ++i) if (row[i] < 0 || row[i] >= ix->n) return fail(FMX_E_ARG, "row out of range at %lld", (long long)i);
    if (len == 0) { for (int64_t i = 0; i < m; ++i) out_len[i] = 0; return FMX_OK; }
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dr(st), dout(st), dlen(st);
    CU(dr.alloc(m * 8)); CU(dout.alloc((size_t)m * len)); CU(dlen.alloc(m * 4));
    CU(cudaMemcpyAsync(dr.p, row, m * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(dout.p, 0, (size_t)m * len, st));
    Timed t(ix, cc);
    CU(launch_next_substr(cc.d, cc.cfg, dr.as<int64_t>(), m, len, dout.as<uint8_t>(), dlen.as<int>(), st));
    ix->last_launches = 1; ix->total_launches += 1;
    t.stop();
    CU(cudaMemcpyAsync(out, dout.p, (size_t)m * len, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(out_len, dlen.p, m * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    t.collect();
    for (int64_t i = 0; i < m; ++i) std::reverse(out + i * len, out + i * len + out_len[i]);     // ret.reverse.toString
    return FMX_OK;
}

// One name for both walks (the sketch of SURVEY §8b): direction > 0 = nextSubstr, else prevSubstr.
int fmx_extract_batch(fmx_index *ix, const int64_t *row, int64_t m, int32_t len, int32_t direction, uint8_t *out, int32_t *out_len) {
    return direction > 0 ? fmx_next_substr_batch(ix, row, m, len, out, out_len) : fmx_prev_substr_batch(ix, row, m, len, out, out_len);
}

// ---- extract: file bytes at file offsets (include/fmgpu.h) -----------------------------------------------------
int fmx_text_sample_rate(const fmx_index *ix) { return ix ? ix->text_rate : 0; }

// Host-buffer form: the requests flow through the call's three streams in chunks, as in the count pipeline (H2D of the offsets of chunk
// k+1, the walks of chunk k and the D2H of chunk k-1 overlap).
int fmx_text_batch(fmx_index *ix, const int64_t *off, int64_t m, int32_t len, uint8_t *out, int32_t *out_len) {
    CHECK_IX(ix);
    if (m < 0 || len < 0 || (m && (!off || !out_len || (len && !out)))) return fail(FMX_E_ARG, "bad argument");
    for (int64_t i = 0; i < m; ++i)
        if (off[i] < 0 || off[i] > ix->n - 1) return fail(FMX_E_ARG, "file offset %lld at %lld is outside [0, %lld]", (long long)off[i], (long long)i, (long long)(ix->n - 1));
    CallCtx cc(ix);
    CHECK_CC(cc);
    if (text_path(cc.d) < 0) return fail(FMX_E_UNSUPPORTED, "extract needs text samples (fmx_opts.text_sample_rate) or the singleton shortcut (FMX_ACCEL_TEXT)");
    if (m == 0) return FMX_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    std::vector<uint32_t> off32((size_t)m);
    for (int64_t i = 0; i < m; ++i) off32[(size_t)i] = (uint32_t)off[i];
    DBuf doff(st), dout(st), dlen(st), dreq(st);
    CU(doff.alloc((size_t)m * 4)); CU(dout.alloc((size_t)m * len)); CU(dlen.alloc((size_t)m * 4));
    if (cc.stats) { CU(dreq.alloc(8)); CU(cudaMemsetAsync(dreq.p, 0, 8, st)); }
    // chunks of about 64 MiB of output (at least 2^12 requests), or the caller's fmx_set_chunk
    const int64_t chunk = cc.chunk_queries > 0 ? cc.chunk_queries : std::max<int64_t>(1 << 12, (64ll << 20) / std::max<int32_t>(len, 1));
    const int64_t nchunks = (m + chunk - 1) / chunk;
    Events evs_in, evs_k;
    CU(evs_in.make((size_t)nchunks)); CU(evs_k.make((size_t)nchunks));
    CU(cudaEventRecord(cc.ev_alloc, st));
    CU(cudaStreamWaitEvent(cc.h2d, cc.ev_alloc, 0));
    CU(cudaStreamWaitEvent(cc.d2h, cc.ev_alloc, 0));
    Timed t(ix, cc);
    int rc = FMX_OK;
    for (int64_t k = 0; k < nchunks && rc == FMX_OK; ++k) {
        const int64_t q0 = k * chunk, nq = std::min(chunk, m - q0);
        cudaError_t e = cudaMemcpyAsync(doff.as<uint32_t>() + q0, off32.data() + q0, (size_t)nq * 4, cudaMemcpyHostToDevice, cc.h2d);
        if (e == cudaSuccess) e = cudaEventRecord(evs_in.v[(size_t)k], cc.h2d);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(st, evs_in.v[(size_t)k], 0);
        if (e == cudaSuccess) e = launch_text(cc.d, cc.cfg, doff.as<uint32_t>() + q0, nq, len, dout.as<uint8_t>() + q0 * len, dlen.as<int>() + q0,
                                              cc.stats ? dreq.as<unsigned long long>() : nullptr, st);
        if (e == cudaSuccess) e = cudaEventRecord(evs_k.v[(size_t)k], st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(cc.d2h, evs_k.v[(size_t)k], 0);
        if (e == cudaSuccess && len) e = cudaMemcpyAsync(out + q0 * len, dout.as<uint8_t>() + q0 * len, (size_t)nq * len, cudaMemcpyDeviceToHost, cc.d2h);
        if (e == cudaSuccess) e = cudaMemcpyAsync(out_len + q0, dlen.as<int>() + q0, (size_t)nq * 4, cudaMemcpyDeviceToHost, cc.d2h);
        if (e != cudaSuccess) rc = fail(FMX_E_CUDA, "CUDA error %s in the extract pipeline (%s)", cudaGetErrorName(e), cudaGetErrorString(e));
    }
    ix->last_launches = nchunks; ix->total_launches += nchunks;
    t.stop();
    cudaError_t e1 = cudaStreamSynchronize(cc.h2d), e2 = cudaStreamSynchronize(st), e3 = cudaStreamSynchronize(cc.d2h);
    if (rc == FMX_OK && (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)) rc = fail(FMX_E_CUDA, "CUDA error while draining the extract pipeline");
    t.collect();
    if (rc == FMX_OK && cc.stats) {
        unsigned long long h = 0;
        CU(cudaMemcpy(&h, dreq.p, 8, cudaMemcpyDeviceToHost));
        ix->last_steps = (int64_t)h;
    }
    return rc;
}

int fmx_text_dev(fmx_index *ix, const void *d_off, int64_t m, int32_t len, void *d_out, void *d_out_len, void *stream) {
    CHECK_IX(ix);
    if (m < 0 || len < 0 || (m && (!d_off || !d_out_len || (len && !d_out)))) return fail(FMX_E_ARG, "bad argument");
    CallCtx cc(ix);
    CHECK_CC(cc);
    if (text_path(cc.d) < 0) return fail(FMX_E_UNSUPPORTED, "extract needs text samples (fmx_opts.text_sample_rate) or the singleton shortcut (FMX_ACCEL_TEXT)");
    if (m == 0) return FMX_OK;
    DeviceGuard g(ix->device);
    cudaStream_t st = (cudaStream_t)stream;
    DBuf dreq(st);
    if (cc.stats) { CU(dreq.alloc(8)); CU(cudaMemsetAsync(dreq.p, 0, 8, st)); }
    CU(launch_text(cc.d, cc.cfg, (const uint32_t *)d_off, m, len, (uint8_t *)d_out, (int *)d_out_len, cc.stats ? dreq.as<unsigned long long>() : nullptr, st));
    ix->last_launches = 1; ix->total_launches += 1;
    if (cc.stats) {                                            // counting runs are untimed: wait for the count
        unsigned long long h = 0;
        CU(cudaMemcpyAsync(&h, dreq.p, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        ix->last_steps = (int64_t)h;
    }
    return FMX_OK;
}

// ---- locate ---------------------------------------------------------------------------------------------------
namespace {
bool debug_sync() { static const bool on = std::getenv("FMX_DEBUG_SYNC") != nullptr; return on; }     // synchronise + check after each stage
// Occurrences are processed in slabs of whole queries (<= 2^27 occurrences each, or one query of any size): the LF walks emit
// (query, position) sort keys into slab-sized scratch, one radix sort orders the slab — ascending positions inside every query,
// whatever the spread of the query sizes (English-like text: from 1 to millions of occurrences per pattern) — and the slab is handed
// to the caller's sink.  A batch may hold any number of occurrences; device memory is bounded by the slab, not by the batch.
std::atomic<int64_t> g_locate_slab{1ll << 27};
int64_t locate_slab() { return g_locate_slab.load(); }

// sink(t0, cnt, d_keys): the cnt sorted keys of the occurrences [t0, t0 + cnt) of the batch (low 32 bits = position); is_u32 = the slab
// was a single query and d_keys holds plain uint32 positions instead
using SlabSink = std::function<int(int64_t, int64_t, const void *, bool)>;
int locate_core(fmx_index *ix, CallCtx &cc, const uint32_t *d_sp, const int64_t *d_off, const int64_t *h_off, int64_t m, int64_t total, cudaStream_t st, const SlabSink &sink) {
    ix->locate_walk_ms = 0.0; ix->locate_sort_ms = 0.0;
    double walk_ms = 0.0, sort_ms = 0.0;
    if (total <= 0) return FMX_OK;
    const int64_t slab = locate_slab();
    std::vector<int64_t> cuts{0};                              // query indices where slabs begin
    if (total > slab) {
        for (int64_t q = 0, t0 = 0; q < m; ++q)
            if (h_off[q + 1] - t0 > slab && q > cuts.back()) { cuts.push_back(q); t0 = h_off[q]; }
    }
    cuts.push_back(m);
    int64_t largest = 0;
    std::vector<int64_t> hb(cuts.size());
    for (size_t k = 0; k < cuts.size(); ++k) hb[k] = (total > slab) ? h_off[cuts[k]] : (k == 0 ? 0 : total);
    for (size_t k = 0; k + 1 < cuts.size(); ++k) largest = std::max(largest, hb[k + 1] - hb[k]);
    DBuf ka(st), kb(st), dsteps(st);
    CU(ka.alloc((size_t)largest * 8)); CU(kb.alloc((size_t)largest * 8));
    if (cc.stats) { CU(dsteps.alloc(8)); CU(cudaMemsetAsync(dsteps.p, 0, 8, st)); }
    unsigned long long *steps = cc.stats ? dsteps.as<unsigned long long>() : nullptr;
    cudaEvent_t ev[3];
    for (auto &e : ev) CU(cudaEventCreate(&e));
    struct EvGuard { cudaEvent_t *e; ~EvGuard() { for (int i = 0; i < 3; ++i) cudaEventDestroy(e[i]); } } eg{ev};
    for (size_t k = 0; k + 1 < cuts.size(); ++k) {
        const int64_t q0 = cuts[k], q1 = cuts[k + 1], t0 = hb[k], cnt = hb[k + 1] - t0;
        if (cnt <= 0) continue;
        const bool single = (q1 - q0 == 1);                    // one query: plain 32-bit positions
        CU(cudaEventRecord(ev[0], st));
        CU(launch_locate(cc.d, cc.cfg, d_sp, d_off, q0, q1, t0, cnt, single ? ka.as<uint32_t>() : nullptr, single ? nullptr : ka.as<uint64_t>(), steps, st));
        CU(cudaEventRecord(ev[1], st));
        if (debug_sync()) { cudaError_t de = cudaStreamSynchronize(st); if (de != cudaSuccess) return fail(FMX_E_CUDA, "locate walk kernel failed: %s (slab %zu, queries %lld..%lld, %lld occurrences)", cudaGetErrorString(de), k, (long long)q0, (long long)q1, (long long)cnt); }
        if (single) CU(radix_sort_u32(ka.as<uint32_t>(), kb.as<uint32_t>(), cnt, st));
        else {
            int seg_bits = 1;
            while ((1ll << seg_bits) < q1 - q0) ++seg_bits;
            CU(radix_sort_u64(ka.as<uint64_t>(), kb.as<uint64_t>(), cnt, 32 + seg_bits, st));
        }
        CU(cudaEventRecord(ev[2], st));
        int rc = sink(t0, cnt, kb.p, single);
        if (rc) return rc;
        CU(cudaStreamSynchronize(st));                         // the scratch is reused by the next slab
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, ev[0], ev[1]); cudaEventElapsedTime(&b, ev[1], ev[2]);
        walk_ms += a; sort_ms += b;
        ix->last_launches += 1; ix->total_launches += 1;
    }
    ix->locate_walk_ms = walk_ms; ix->locate_sort_ms = sort_ms;
    ix->last_ms = walk_ms + sort_ms;
    if (cc.stats) {
        unsigned long long hs = 0;
        CU(cudaMemcpyAsync(&hs, dsteps.p, 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        ix->last_steps = (int64_t)hs;
    }
    return FMX_OK;
}
}  // namespace

// Device-resident locate: d_sp/d_ep = uint32 rows of m intervals (as fmx_count_fixed_dev leaves them; an empty interval has sp >= ep),
// d_off[m+1] receives the exclusive offsets, d_pos[cap] the positions (uint32, ascending inside each query).  Synchronises `stream`
// to learn the total (and once per slab).  FMX_E_CAPACITY with *total_out set when cap is too small.
int fmx_locate_dev(fmx_index *ix, const void *d_sp, const void *d_ep, int64_t m, void *d_off, void *d_pos, int64_t cap, int64_t *total_out, void *stream) {
    CHECK_IX(ix);
    if (m < 0 || !d_off || !total_out || (m && (!d_sp || !d_ep))) return fail(FMX_E_ARG, "bad argument");
    if (ix->sample_rate <= 0 && ix->d_full.sa == nullptr) return fail(FMX_E_ARG, "index was opened without sa_sample_rate (and without a resident suffix array); locate unavailable");
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = (cudaStream_t)stream;
    ix->last_launches = 0;
    DBuf len(st);
    CU(len.alloc((size_t)(m + 1) * 8));
    CU(launch_interval_len((const uint32_t *)d_sp, (const uint32_t *)d_ep, m, len.as<int64_t>(), st));
    CU(exclusive_sum_i64(len.as<int64_t>(), (int64_t *)d_off, m + 1, st));
    int64_t total = 0;
    CU(cudaMemcpyAsync(&total, (const int64_t *)d_off + m, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *total_out = total;
    if (total > cap) return fail(FMX_E_CAPACITY, "locate needs %lld output slots, capacity %lld", (long long)total, (long long)cap);
    if (total == 0) return FMX_OK;
    if (!d_pos) return fail(FMX_E_ARG, "null output");
    std::vector<int64_t> h_off;
    if (total > locate_slab()) {
        h_off.resize((size_t)m + 1);
        CU(cudaMemcpyAsync(h_off.data(), d_off, (size_t)(m + 1) * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    uint32_t *out = (uint32_t *)d_pos;
    return locate_core(ix, cc, (const uint32_t *)d_sp, (const int64_t *)d_off, h_off.empty() ? nullptr : h_off.data(), m, total, st,
                       [&](int64_t t0, int64_t cnt, const void *keys, bool is_u32) -> int {
                           if (is_u32) CU(cudaMemcpyAsync(out + t0, keys, (size_t)cnt * 4, cudaMemcpyDeviceToDevice, st));
                           else CU(launch_key_positions((const uint64_t *)keys, cnt, out + t0, nullptr, st));
                           return FMX_OK;
                       });
}

// Instrumentation for the roofline accounting: with stats on, locate calls also count the LF steps of their walks (one atomic per
// occurrence — not for timed runs); regex searches always count their items.  fmx_last_steps returns the count of the last such call.
int fmx_set_stats(fmx_index *ix, int32_t on) { CHECK_IX(ix); std::lock_guard<std::mutex> lk(ix->mu); ix->stats = on != 0; return FMX_OK; }
int64_t fmx_last_steps(const fmx_index *ix) { return ix ? ix->last_steps.load() : 0; }

int fmx_set_locate_slab(int64_t occurrences) {
    g_locate_slab = occurrences > 0 ? occurrences : (1ll << 27);
    return FMX_OK;
}

int fmx_last_locate_ms(const fmx_index *ix, double *walk_ms, double *sort_ms) {
    CHECK_IX(ix);
    if (walk_ms) *walk_ms = ix->locate_walk_ms.load();
    if (sort_ms) *sort_ms = ix->locate_sort_ms.load();
    return FMX_OK;
}

int fmx_locate_batch(fmx_index *ix, const int64_t *sp, const int64_t *ep, int64_t m, int64_t cap_total, int64_t *out_off, int64_t *pos) {
    CHECK_IX(ix);
    if (m < 0 || !out_off || (m && (!sp || !ep))) return fail(FMX_E_ARG, "bad argument");
    if (ix->sample_rate <= 0 && ix->d_full.sa == nullptr) return fail(FMX_E_ARG, "index was opened without sa_sample_rate (and without a resident suffix array); locate unavailable");
    int64_t total = 0;
    std::vector<uint32_t> sp32((size_t)m);
    for (int64_t i = 0; i < m; ++i) {
        if (sp[i] < 0 || ep[i] > ix->n || (ep[i] < sp[i])) return fail(FMX_E_ARG, "bad interval at %lld", (long long)i);
        out_off[i] = total;
        total += ep[i] - sp[i];
        sp32[(size_t)i] = (uint32_t)sp[i];
    }
    out_off[m] = total;
    if (total > cap_total) return fail(FMX_E_CAPACITY, "locate needs %lld output slots, capacity %lld", (long long)total, (long long)cap_total);
    if (total == 0) return FMX_OK;
    if (!pos) return fail(FMX_E_ARG, "null output");
    CallCtx cc(ix);
    CHECK_CC(cc);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    ix->last_launches = 0;
    DBuf dsp(st), doff(st), w0(st), w1(st);
    CU(dsp.alloc(m * 4)); CU(doff.alloc((m + 1) * 8));
    CU(cudaMemcpyAsync(dsp.p, sp32.data(), m * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(doff.p, out_off, (m + 1) * 8, cudaMemcpyHostToDevice, st));
    // every sorted slab is widened to the ABI's int64 on the device, in pieces that stream straight into the caller's buffer: the
    // widening of piece k+1 overlaps the D2H of piece k (asynchronous DMA when `pos` is page-locked), and the copies of a slab overlap
    // the LF walks of the next one
    const int64_t piece = 32ll << 20;
    CU(w0.alloc((size_t)std::min(piece, total) * 8)); CU(w1.alloc((size_t)std::min(piece, total) * 8));
    CU(cudaEventRecord(cc.ev_alloc, st));
    CU(cudaStreamWaitEvent(cc.d2h, cc.ev_alloc, 0));
    cudaEvent_t done[2];
    CU(cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming)); CU(cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming));
    struct Ev2 { cudaEvent_t *e; ~Ev2() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } ev2{done};
    int64_t pieces = 0;
    int rc = locate_core(ix, cc, dsp.as<uint32_t>(), doff.as<int64_t>(), out_off, m, total, st,
                         [&](int64_t t0, int64_t cnt, const void *keys, bool is_u32) -> int {
                             for (int64_t o = 0; o < cnt; o += piece, ++pieces) {
                                 const int64_t c = std::min(piece, cnt - o);
                                 int64_t *w = (pieces & 1) ? w1.as<int64_t>() : w0.as<int64_t>();
                                 if (pieces >= 2) CU(cudaStreamWaitEvent(st, done[pieces & 1], 0));          // the piece buffer is free again
                                 if (is_u32) CU(widen_u32_i64((const uint32_t *)keys + o, w, c, st));
                                 else CU(launch_key_positions((const uint64_t *)keys + o, c, nullptr, w, st));
                                 CU(cudaEventRecord(cc.ev1, st));
                                 CU(cudaStreamWaitEvent(cc.d2h, cc.ev1, 0));
                                 CU(cudaMemcpyAsync(pos + t0 + o, w, (size_t)c * 8, cudaMemcpyDeviceToHost, cc.d2h));
                                 CU(cudaEventRecord(done[pieces & 1], cc.d2h));
                             }
                             return FMX_OK;
                         });
    cudaError_t e1 = cudaStreamSynchronize(st), e2 = cudaStreamSynchronize(cc.d2h);
    if (rc == FMX_OK && (e1 != cudaSuccess || e2 != cudaSuccess)) rc = fail(FMX_E_CUDA, "CUDA error while draining the locate copy-out");
    return rc;
}

// Exchange step for variable-length results: `count` 4-byte words of this rank go into every sink (this rank's and, via CUDA IPC, its
// peers' gathered buffers) at word offset `offset` + (*d_dst_off) * dst_scale; d_dst_off is a DEVICE int64 (e.g. the scanned offset of
// this rank's first result) or NULL.  Asynchronous on `stream`.
int fmx_scatter_dev(const void *d_src, int64_t count, void *const *sinks, int32_t n_sinks, int64_t offset, const void *d_dst_off, int64_t dst_scale, void *stream) {
    if (count < 0 || n_sinks < 0 || n_sinks > 8 || (n_sinks && !sinks) || (count && !d_src)) return fail(FMX_E_ARG, "bad argument");
    PeerSinks ps{};
    ps.n = n_sinks; ps.offset = offset;
    for (int j = 0; j < n_sinks; ++j) { if (!sinks[j]) return fail(FMX_E_ARG, "null sink %d", j); ps.p[j] = (uint32_t *)sinks[j]; }
    CU(launch_scatter_words((const uint32_t *)d_src, count, ps, (const int64_t *)d_dst_off, dst_scale, (cudaStream_t)stream));
    return FMX_OK;
}

// ---- regex ------------------------------------------------------------------------------------------------------
int fmx_regex_compile(const uint8_t *re, int64_t re_len, int line_only, fmx_regex **out) {
    if (!out || re_len < 0 || (re_len && !re)) return fail(FMX_E_ARG, "bad argument");
    *out = nullptr;
    fmx_regex *rx = new fmx_regex();
    std::string err;
    int rc = compile_regex(re, re_len, line_only != 0, rx->a, err);
    if (rc) { delete rx; return fail(rc, "%s", err.c_str()); }
    *out = rx;
    return FMX_OK;
}
int fmx_regex_compile_engine(const uint8_t *re, int64_t re_len, int line_only, int engine, fmx_regex **out) {
    if (engine == FMX_ENGINE_GLUSHKOV) return fmx_regex_compile(re, re_len, line_only, out);
    if (engine != FMX_ENGINE_THOMPSON) return fail(FMX_E_ARG, "unknown regex engine %d", engine);
    if (!out || re_len < 0 || (re_len && !re)) return fail(FMX_E_ARG, "bad argument");
    *out = nullptr;
    fmx_regex *rx = new fmx_regex();
    std::string err;
    int rc = compile_thompson(re, re_len, line_only != 0, rx->a, err);
    if (rc) { delete rx; return fail(rc, "%s", err.c_str()); }
    *out = rx;
    return FMX_OK;
}
void fmx_regex_free(fmx_regex *rx) { delete rx; }

// ---- DFA engine (dfa.scala) ---------------------------------------------------------------------------------------------
int fmx_dfa_create(int32_t n_states, const uint8_t *kind, const int32_t *link_off, const int32_t *link_to, const int32_t *link_chr, fmx_regex **out) {
    if (!out) return fail(FMX_E_ARG, "null output");
    *out = nullptr;
    if (n_states > 0 && link_off && link_off[n_states] > 0 && (!link_to || !link_chr)) return fail(FMX_E_ARG, "null link arrays");
    fmx_regex *rx = new fmx_regex();
    std::string err;
    int rc = compile_dfa(n_states, kind, link_off, link_to, link_chr, rx->dfa, rx->a, err);
    if (rc) { delete rx; return fail(rc, "%s", err.c_str()); }
    *out = rx;
    return FMX_OK;
}
int fmx_dfa_from_nfa(int32_t n_states, const uint8_t *is_finish, int32_t initial, const int32_t *link_off, const int32_t *link_to,
                     const int32_t *link_chr, fmx_regex **out) {
    if (!out) return fail(FMX_E_ARG, "null output");
    *out = nullptr;
    if (n_states > 0 && link_off && link_off[n_states] > 0 && (!link_to || !link_chr)) return fail(FMX_E_ARG, "null link arrays");
    std::vector<uint8_t> kind;
    std::vector<int32_t> off, to, chr;
    std::string err;
    int rc = dfa_from_nfa(n_states, is_finish, initial, link_off, link_to, link_chr, kind, off, to, chr, err);
    if (rc) return fail(rc, "%s", err.c_str());
    if (to.empty()) { to.push_back(0); chr.push_back(0); }
    return fmx_dfa_create((int32_t)kind.size(), kind.data(), off.data(), to.data(), chr.data(), out);
}
int fmx_dfa_info(const fmx_regex *dfa, int32_t *n_states, int32_t *moves, uint8_t *finish, int32_t *number, int32_t n_number) {
    if (!dfa || dfa->dfa.n_states == 0) return fail(FMX_E_ARG, "not a DFA handle");
    const CompiledDfa &d = dfa->dfa;
    if (n_states) *n_states = d.n_states;
    if (moves) std::copy(d.moves.begin(), d.moves.end(), moves);
    if (finish) std::copy(d.finish.begin(), d.finish.end(), finish);
    if (number) std::copy(d.number.begin(), d.number.begin() + std::min<size_t>(d.number.size(), (size_t)std::max(n_number, 0)), number);
    return FMX_OK;
}
int fmx_dfa_buckets(const fmx_regex *dfa, int32_t state, char *buf, int64_t cap, int64_t *needed) {
    if (!dfa || dfa->dfa.n_states == 0) return fail(FMX_E_ARG, "not a DFA handle");
    if (state < 0 || state >= dfa->dfa.n_states) return fail(FMX_E_ARG, "state %d out of range", state);
    const std::string s = dfa_bucket_string(dfa->dfa, state);
    if (needed) *needed = (int64_t)s.size() + 1;
    if (!buf || cap < (int64_t)s.size() + 1) return fail(FMX_E_CAPACITY, "bucket string needs %lld bytes", (long long)s.size() + 1);
    std::memcpy(buf, s.c_str(), s.size() + 1);
    return FMX_OK;
}
int fmx_dfa_match_string(const fmx_regex *dfa, const uint8_t *s, int64_t len, int32_t *matched) {
    if (!dfa || dfa->dfa.n_states == 0 || !matched || len < 0 || (len && !s)) return fail(FMX_E_ARG, "bad argument");
    const CompiledDfa &d = dfa->dfa;
    int cur = 0;
    for (int64_t i = 0; i < len && cur >= 0; ++i) cur = d.moves[(size_t)cur * 256 + s[i]];
    *matched = (cur >= 0 && d.finish[(size_t)cur]) ? 1 : 0;
    return FMX_OK;
}

int fmx_regex_tables(const fmx_regex *rx, int32_t *n_states, int32_t *n_follows, int32_t *n_firsts, uint8_t *c, uint8_t *is_last,
                     int32_t *num, int32_t *follows_off, int32_t *follows, int32_t *firsts) {
    if (!rx) return fail(FMX_E_ARG, "null regex");
    const CompiledRegex &a = rx->a;
    if (n_states) *n_states = (int32_t)a.c.size();
    if (n_follows) *n_follows = (int32_t)a.follows.size();
    if (n_firsts) *n_firsts = (int32_t)a.firsts.size();
    if (c) std::copy(a.c.begin(), a.c.end(), c);
    if (is_last) std::copy(a.is_last.begin(), a.is_last.end(), is_last);
    if (num) std::copy(a.num.begin(), a.num.end(), num);
    if (follows_off) std::copy(a.follows_off.begin(), a.follows_off.end(), follows_off);
    if (follows) std::copy(a.follows.begin(), a.follows.end(), follows);
    if (firsts) std::copy(a.firsts.begin(), a.firsts.end(), firsts);
    return FMX_OK;
}

// A regex set = the automata of a batch concatenated (global state ids, 16-byte state records, follow lists, owning regex) and resident
// on the device together with the work ring of its traversals: compile once, search many times — the batched form of
// `val t = ReTree(post); t.matchSA(sa)`.
struct fmx_regex_set {
    int device = 0;
    int64_t m = 0;
    size_t n_states = 0, n_fol = 0, n_first = 0;
    void *d_rec = nullptr, *d_rx = nullptr, *d_f = nullptr, *d_first = nullptr;
    void *d_ring = nullptr, *d_seq = nullptr, *d_ctrl = nullptr;     // work ring, its per-slot sequence words, the traversal's control words
    int64_t ring_cap = 0;
    uint32_t max_len = 0;                          // fmx_regex_set_limits
    bool present[256] = {false};                   // the alphabet the follow lists were pruned for
    std::mutex mu;                                 // one traversal at a time per set (they share the ring)
};

void fmx_regex_set_free(fmx_regex_set *s) {
    if (!s) return;
    cudaSetDevice(s->device);
    cudaFree(s->d_rec); cudaFree(s->d_rx); cudaFree(s->d_f); cudaFree(s->d_first); cudaFree(s->d_ring); cudaFree(s->d_seq); cudaFree(s->d_ctrl);
    delete s;
}

int fmx_regex_set_create(fmx_index *ix, fmx_regex *const *rx, int64_t m, fmx_regex_set **out) {
    CHECK_IX(ix);
    if (m < 0 || !out || (m && !rx)) return fail(FMX_E_ARG, "bad argument");
    *out = nullptr;
    if (m >= (1ll << 32)) return fail(FMX_E_LIMIT, "too many regexes in one batch");
    Phases ph("regex_set_create");
    size_t n_states = 0, n_fol = 0, n_first = 0;
    for (int64_t r = 0; r < m; ++r) {
        if (!rx[r]) return fail(FMX_E_ARG, "null regex at %lld", (long long)r);
        n_states += rx[r]->a.c.size(); n_fol += rx[r]->a.follows.size(); n_first += rx[r]->a.firsts.size();
    }
    if (n_states >= (1ull << 32) - 1 || n_fol >= (1ull << 32)) return fail(FMX_E_LIMIT, "regex batch has too many states; split the batch");
    // A follow position whose character does not occur in the indexed text can never survive its backward step (getPrevRange of an
    // absent byte is None), so it is left out of the device follow lists: '.' = 253 positions in the reference costs sigma items here
    // (28 on English text), '\\d' over a text without digits none.  Results are unchanged; the set remembers the alphabet it was pruned
    // for and refuses an index that has other symbols.
    bool present[256];
    present[0] = true;                                        // a step with byte 0 is defined (the '$' row), keep it
    for (int c = 1; c < 256; ++c) present[c] = ix->counts0[c] > 0;
    std::vector<uint4> rec(n_states);
    std::vector<uint32_t> st_regex(n_states), fol, first(n_first);
    fol.reserve(n_fol);
    {
        size_t so = 0, io = 0;
        for (int64_t r = 0; r < m; ++r) {
            const CompiledRegex &a = rx[r]->a;
            const uint32_t base = (uint32_t)so;
            const size_t ns = a.c.size();
            const uint32_t stop = a.stop_on_emit ? 2u : 0u;
            for (size_t s = 0; s < ns; ++s) {
                const uint32_t f0 = (uint32_t)fol.size();
                for (int32_t k = a.follows_off[s]; k < a.follows_off[s + 1]; ++k)
                    if (present[a.c[(size_t)a.follows[(size_t)k]]]) fol.push_back(base + (uint32_t)a.follows[(size_t)k]);
                const uint32_t nf = (uint32_t)fol.size() - f0;
                rec[so + s] = make_uint4((uint32_t)a.c[s] | (((uint32_t)a.is_last[s] | stop) << 8), f0, nf, nf ? fol[f0] : 0u);
                st_regex[so + s] = (uint32_t)r;
            }
            for (int32_t f : a.firsts) first[io++] = base + (uint32_t)f;
            so += ns;
        }
    }
    n_fol = fol.size();
    if (fol.empty()) fol.push_back(0);
    ph.mark("concatenate tables");
    DeviceGuard g(ix->device);
    fmx_regex_set *s = new fmx_regex_set();
    s->device = ix->device; s->m = m; s->n_states = n_states; s->n_fol = n_fol; s->n_first = n_first;
    for (int c = 0; c < 256; ++c) s->present[c] = present[c];
    auto up = [&](void **d, const void *h, size_t bytes) -> cudaError_t {
        cudaError_t e = cudaMalloc(d, bytes ? bytes : 16);
        if (e == cudaSuccess && bytes) e = cudaMemcpy(*d, h, bytes, cudaMemcpyHostToDevice);
        return e;
    };
    cudaError_t e = up(&s->d_rec, rec.data(), n_states * sizeof(uint4));
    if (e == cudaSuccess) e = up(&s->d_rx, st_regex.data(), n_states * 4);
    if (e == cudaSuccess) e = up(&s->d_f, fol.data(), fol.size() * 4);
    if (e == cudaSuccess) e = up(&s->d_first, first.data(), n_first * 4);
    if (e == cudaSuccess) e = cudaMalloc(&s->d_ctrl, 64);
    if (e != cudaSuccess) { fmx_regex_set_free(s); return fail(FMX_E_CUDA, "regex set upload failed: %s", cudaGetErrorString(e)); }
    ph.mark("upload tables");
    *out = s;
    return FMX_OK;
}

// max_len = the maxLength of REParser.matchSA (re2.scala:568, :636-641): an item's follow positions are enqueued only while their len stays
// below it; matches are emitted whatever their length; 0 = no limit.  Does not depend on the order in which items are taken, so the result
// is still a well-defined multiset.  (The order-dependent caps — maxIterations, ReTree.matchSA's maxBranching — are not offered: which
// results survive them depends on the reference's priority-queue tie order.)
int fmx_regex_set_limits(fmx_regex_set *set, int64_t max_len) {
    if (!set || max_len < 0 || max_len > 0xFFFFFFFFll) return fail(FMX_E_ARG, "bad argument");
    std::lock_guard<std::mutex> lk(set->mu);
    set->max_len = (uint32_t)max_len;
    return FMX_OK;
}

// Tuning hook of the traversal kernel: how many children a warp keeps on its own shared-memory stack (0..256, default 256) before the
// rest goes to the global ring, where idle warps pick it up.  Results never change.
int fmx_set_regex_local_keep(int32_t items) { set_regex_local_keep(items); return FMX_OK; }

// Pre-sizes (or shrinks) the set's work ring to `slots` (rounded up to a power of two, at least the number of start items): a ring that
// turns out too small is abandoned and the traversal rerun with a 4x larger one, which this lets tests and memory-tight callers provoke.
int fmx_regex_set_ring(fmx_regex_set *set, int64_t slots) {
    if (!set || slots < 0) return fail(FMX_E_ARG, "bad argument");
    std::lock_guard<std::mutex> lk(set->mu);
    cudaSetDevice(set->device);
    int64_t cap = 1024;
    while (cap < slots || cap < (int64_t)set->n_first) cap <<= 1;
    if (set->d_ring) { CU(cudaDeviceSynchronize()); CU(cudaFree(set->d_ring)); CU(cudaFree(set->d_seq)); set->d_ring = set->d_seq = nullptr; set->ring_cap = 0; }
    CU(cudaMalloc(&set->d_ring, (size_t)cap * sizeof(FrontierItem)));
    CU(cudaMalloc(&set->d_seq, (size_t)cap * 4));
    set->ring_cap = cap;
    return FMX_OK;
}

namespace {
// Runs the traversal of a set and leaves its results, ordered by (regex, len, sp, ep), in d_res (capacity cap_res).  *total_out = number of
// results (also when it exceeds cap_res: then nothing is ordered and FMX_E_CAPACITY is returned).  Caller holds a CallCtx and set->mu.
int regex_search_core(fmx_index *ix, CallCtx &cc, fmx_regex_set *set, RegexResult *d_res, int64_t cap_res, int64_t *total_out, cudaStream_t st) {
    const int64_t n_first = (int64_t)set->n_first;
    *total_out = 0;
    if (set->m == 0 || n_first == 0) return FMX_OK;
    for (int c = 1; c < 256; ++c)
        if (ix->counts0[c] > 0 && !set->present[c])
            return fail(FMX_E_ARG, "the regex set was created for an index without byte %d, which this index contains; create the set against this index", c);
    size_t fr = 0, to = 0;
    RegexTables rt{(const uint4 *)set->d_rec, (const uint32_t *)set->d_rx, (const uint32_t *)set->d_f};
    auto grow_ring = [&](int64_t want) -> int {
        int64_t cap = 1 << 20;
        while (cap < want) cap <<= 1;
        cudaMemGetInfo(&fr, &to);
        if (cap > set->ring_cap && (size_t)cap * sizeof(FrontierItem) > fr / 2 + (size_t)set->ring_cap * sizeof(FrontierItem))
            return fail(FMX_E_LIMIT, "regex traversal needs a work ring of %lld items, more than half of the free device memory; split the batch", (long long)cap);
        if (cap > set->ring_cap) {
            if (set->d_ring) { CU(cudaStreamSynchronize(st)); CU(cudaFree(set->d_ring)); CU(cudaFree(set->d_seq)); set->d_ring = set->d_seq = nullptr; set->ring_cap = 0; }
            CU(cudaMalloc(&set->d_ring, (size_t)cap * sizeof(FrontierItem)));
            CU(cudaMalloc(&set->d_seq, (size_t)cap * 4));
            set->ring_cap = cap;
        }
        return FMX_OK;                                      // the seed kernel of every traversal initialises the sequence words
    };
    if (set->ring_cap < n_first || set->d_ring == nullptr) { int rc = grow_ring(4 * n_first); if (rc) return rc; }
    Timed t(ix, cc);
    int64_t launches = 0;
    unsigned long long h[8] = {0};
    for (;;) {
        if (debug_sync()) { cudaError_t de = cudaDeviceSynchronize(); if (de != cudaSuccess) return fail(FMX_E_CUDA, "an earlier asynchronous error surfaced before the regex traversal: %s", cudaGetErrorString(de)); }
        CU(launch_regex_search(cc.d, cc.cfg, rt, (const uint32_t *)set->d_first, n_first, (FrontierItem *)set->d_ring, (uint32_t *)set->d_seq, set->ring_cap, d_res, cap_res,
                               (unsigned long long *)set->d_ctrl, set->max_len, st));
        launches += 2;
        if (debug_sync()) { cudaError_t de = cudaStreamSynchronize(st); if (de != cudaSuccess) return fail(FMX_E_CUDA, "regex traversal kernels failed: %s (ring %lld slots, %lld start items, device %d)", cudaGetErrorString(de), (long long)set->ring_cap, (long long)n_first, ix->device); }
        CU(cudaMemcpyAsync(h, set->d_ctrl, 64, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (h[kRxStatus] == 0) break;
        if (h[kRxStatus] == 2) return fail(FMX_E_LIMIT, "regex traversal deeper than the text");
        int rc = grow_ring(set->ring_cap * 4);              // the ring overflowed: abandon, re-empty a larger one, rerun
        if (rc) return rc;
    }
    ix->last_levels = (int64_t)h[kRxMaxLen];
    ix->last_steps = (int64_t)h[kRxSteps];
    const int64_t total = (int64_t)h[kRxMatches];
    *total_out = total;
    ix->last_launches = launches; ix->total_launches += launches;
    if (total > cap_res) { t.stop(); return fail(FMX_E_CAPACITY, "regex search needs %lld result slots, capacity %lld", (long long)total, (long long)cap_res); }
    // result order = (regex, len, sp, ep), on the device: one CTA's bitonic network for a handful, radix passes beyond
    if (total > kSmallSort) {
        DBuf tmp(st);
        CU(tmp.alloc(total * sizeof(RegexResult)));
        CU(sort_regex_results(d_res, tmp.as<RegexResult>(), total, (uint32_t)set->m, (uint32_t)h[kRxMaxLen], st));
        ix->last_launches += 6; ix->total_launches += 6;
    } else if (total > 1) {
        CU(sort_results_small(d_res, total, st));
        ix->last_launches += 1; ix->total_launches += 1;
    }
    t.stop();
    CU(cudaStreamSynchronize(st));
    t.collect();
    return FMX_OK;
}
}  // namespace

// Device-resident search: results stay on the device as RegexResult {regex, len, sp, ep} (4 x uint32) ordered by (regex, len, sp, ep),
// d_off (int64[m+1], may be NULL) = first result of every regex.
int fmx_regex_set_search_dev(fmx_index *ix, fmx_regex_set *set, void *d_res, int64_t cap, void *d_off, int64_t *total_out) {
    CHECK_IX(ix);
    if (!set || !total_out || cap < 0 || (cap && !d_res)) return fail(FMX_E_ARG, "bad argument");
    if (set->device != ix->device) return fail(FMX_E_ARG, "regex set lives on device %d, index on device %d", set->device, ix->device);
    CallCtx cc(ix);
    CHECK_CC(cc);
    std::lock_guard<std::mutex> lk2(set->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    DBuf dummy(st);
    RegexResult *res = (RegexResult *)d_res;
    if (!res) { CU(dummy.alloc(sizeof(RegexResult))); res = dummy.as<RegexResult>(); }
    int rc = regex_search_core(ix, cc, set, res, cap, total_out, st);
    if (rc) return rc;
    if (d_off) {
        CU(launch_result_offsets(res, *total_out, set->m, (int64_t *)d_off, st));
        CU(cudaStreamSynchronize(st));
    }
    return FMX_OK;
}

int fmx_regex_set_search(fmx_index *ix, fmx_regex_set *set, int64_t cap_total, int64_t *out_off, int32_t *len, int64_t *sp, int64_t *ep) {
    CHECK_IX(ix);
    if (!set || !out_off || cap_total < 0) return fail(FMX_E_ARG, "bad argument");
    if (set->device != ix->device) return fail(FMX_E_ARG, "regex set lives on device %d, index on device %d", set->device, ix->device);
    const int64_t m = set->m;
    if (m == 0 || set->n_first == 0) { for (int64_t i = 0; i <= m; ++i) out_off[i] = 0; return FMX_OK; }
    Phases ph("regex_set_search");
    CallCtx cc(ix);
    CHECK_CC(cc);
    std::lock_guard<std::mutex> lk2(set->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = cc.stream;
    const int64_t cap_res = std::max<int64_t>(cap_total, 1 << 16);
    DBuf d_res(st), d_off(st), d_len(st), d_sp(st), d_ep(st);
    CU(d_res.alloc(cap_res * sizeof(RegexResult))); CU(d_off.alloc((m + 1) * 8));
    int64_t total = 0;
    int rc = regex_search_core(ix, cc, set, d_res.as<RegexResult>(), cap_res, &total, st);
    ph.mark("traversal + order");
    if (rc == FMX_E_CAPACITY || total > cap_total) {
        for (int64_t i = 0; i < m; ++i) out_off[i] = 0;
        out_off[m] = total;
        return fail(FMX_E_CAPACITY, "regex search needs %lld result slots, capacity %lld", (long long)total, (long long)cap_total);
    }
    if (rc) return rc;
    if (total && (!len || !sp || !ep)) return fail(FMX_E_ARG, "null output");
    // offsets and the three output columns are produced on the device and copied straight into the caller's buffers
    CU(launch_result_offsets(d_res.as<RegexResult>(), total, m, d_off.as<int64_t>(), st));
    CU(cudaMemcpyAsync(out_off, d_off.p, (m + 1) * 8, cudaMemcpyDeviceToHost, st));
    if (total) {
        CU(d_len.alloc(total * 4)); CU(d_sp.alloc(total * 8)); CU(d_ep.alloc(total * 8));
        CU(launch_split_results(d_res.as<RegexResult>(), total, d_len.as<int32_t>(), d_sp.as<int64_t>(), d_ep.as<int64_t>(), st));
        CU(cudaMemcpyAsync(len, d_len.p, total * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(sp, d_sp.p, total * 8, cudaMemcpyDeviceToHost, st));
        CU(cudaMemcpyAsync(ep, d_ep.p, total * 8, cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    ph.mark("offsets + copy out");
    return FMX_OK;
}

int fmx_regex_search_batch(fmx_index *ix, fmx_regex *const *rx, int64_t m, int64_t cap_total, int64_t *out_off, int32_t *len,
                           int64_t *sp, int64_t *ep) {
    CHECK_IX(ix);
    if (m < 0 || !out_off || (m && !rx)) return fail(FMX_E_ARG, "bad argument");
    for (int64_t i = 0; i <= m; ++i) out_off[i] = 0;
    if (m == 0) return FMX_OK;
    fmx_regex_set *set = nullptr;
    int rc = fmx_regex_set_create(ix, rx, m, &set);
    if (rc) return rc;
    rc = fmx_regex_set_search(ix, set, cap_total, out_off, len, sp, ep);
    fmx_regex_set_free(set);
    return rc;
}

// ---- K4 gather microbenchmark -------------------------------------------------------------------------------------
int fmx_gather_bench(fmx_index *ix, int32_t bytes, int32_t lanes, int64_t gathers, int32_t chain, int32_t iters, double *gbs, double *ms_out) {
    CHECK_IX(ix);
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = ix->stream;
    DBuf sink(st);
    CU(sink.alloc(8));
    CU(cudaMemsetAsync(sink.p, 0, 8, st));
    const uint64_t nb = (uint64_t)ix->rank_units64;
    CU(launch_gather_bench(ix->d.blocks, nb, bytes, lanes, gathers, chain, 1u, sink.as<unsigned long long>(), st));   // warm-up
    float best = 1e30f;
    for (int it = 0; it < std::max(iters, 1); ++it) {
        CU(cudaEventRecord(ix->ev0, st));
        CU(launch_gather_bench(ix->d.blocks, nb, bytes, lanes, gathers, chain, 1000u + it, sink.as<unsigned long long>(), st));
        CU(cudaEventRecord(ix->ev1, st));
        CU(cudaStreamSynchronize(st));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, ix->ev0, ix->ev1));
        best = std::min(best, ms);
    }
    if (ms_out) *ms_out = best;
    if (gbs) *gbs = (double)gathers * chain * bytes / (best * 1e-3) / 1e9;
    return FMX_OK;
}

// ---- index construction on the device -----------------------------------------------------------------------------
static int build_bwt_impl(const uint8_t *text, int64_t len, int device, std::vector<uint8_t> &bwt, int64_t *eof, int64_t counts[256],
                          std::vector<uint32_t> *fm) {
    if (len < 0 || (len && !text)) return fail(FMX_E_ARG, "bad argument");
    int dev = 0;
    int rc = ensure_device(device, &dev);
    if (rc) return rc;
    // FileBWTReader.copyReverse (bwtreader.scala:196-211): 0x00 bytes are dropped, the text is reversed
    std::vector<uint8_t> filtered;
    const uint8_t *src = text;
    int64_t flen = len;
    if (len && std::memchr(text, 0, (size_t)len)) {
        filtered.reserve((size_t)len);
        for (int64_t i = 0; i < len; ++i) if (text[i]) filtered.push_back(text[i]);
        src = filtered.data(); flen = (int64_t)filtered.size();
    }
    const int64_t n = flen + 1;
    if (n >= (1ll << 32) - 1) return fail(FMX_E_UNSUPPORTED, "text too long for 32-bit rows");
    cudaStream_t st;
    CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CU(cudaDeviceSynchronize());
    trim_pool(dev);                                            // the prefix-doubling sort wants ~35 bytes of scratch per text byte
    uint8_t *d_fwd = nullptr, *d_rev = nullptr, *d_bwt = nullptr;
    CU(cudaMalloc(&d_fwd, flen + 16)); CU(cudaMalloc(&d_rev, flen + 16)); CU(cudaMalloc(&d_bwt, n));
    if (flen) CU(cudaMemcpyAsync(d_fwd, src, flen, cudaMemcpyHostToDevice, st));
    CU(reverse_bytes(d_fwd, flen, d_rev, st));
    cudaError_t e = suffix_sort_bwt(d_rev, flen, d_bwt, eof, counts, nullptr, nullptr, st);
    if (e != cudaSuccess) { cudaFree(d_fwd); cudaFree(d_rev); cudaFree(d_bwt); cudaStreamDestroy(st); return fail(FMX_E_CUDA, "suffix sort failed: %s", cudaGetErrorString(e)); }
    bwt.resize((size_t)n);
    CU(cudaMemcpyAsync(bwt.data(), d_bwt, n, cudaMemcpyDeviceToHost, st));
    if (fm) {
        uint32_t *d_fm = nullptr;
        CU(cudaMalloc(&d_fm, n * 4));
        CU(build_fm_array(d_bwt, n, d_fm, st));
        fm->resize((size_t)n);
        CU(cudaMemcpyAsync(fm->data(), d_fm, n * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        cudaFree(d_fm);
    }
    CU(cudaStreamSynchronize(st));
    cudaFree(d_fwd); cudaFree(d_rev); cudaFree(d_bwt);
    cudaStreamDestroy(st);
    trim_pool(dev);
    return FMX_OK;
}

int fmx_build_bwt(const uint8_t *text, int64_t len, uint8_t *bwt_out, int64_t *n_out, int64_t *eof_out, int64_t counts_out[256], int device) {
    if (!bwt_out || !n_out || !eof_out || !counts_out) return fail(FMX_E_ARG, "null argument");
    std::vector<uint8_t> bwt;
    int rc = build_bwt_impl(text, len, device, bwt, eof_out, counts_out, nullptr);
    if (rc) return rc;
    std::memcpy(bwt_out, bwt.data(), bwt.size());
    *n_out = (int64_t)bwt.size();
    return FMX_OK;
}

int fmx_build_index_files(const uint8_t *text, int64_t len, const char *base, int big_endian, int write_fm, int device) {
    if (!base) return fail(FMX_E_ARG, "null argument");
    std::vector<uint8_t> bwt; std::vector<uint32_t> fm;
    int64_t eof = 0, counts[256];
    int rc = build_bwt_impl(text, len, device, bwt, &eof, counts, write_fm ? &fm : nullptr);
    if (rc) return rc;
    return write_index_files(strip_extension(base), bwt.data(), (int64_t)bwt.size(), eof, counts, big_endian != 0, write_fm ? fm.data() : nullptr);
}

// bwtFm2LCP (util.scala:153-212): lcp[r] = longest common prefix of the suffixes of rows r and r+1 (lcp[n-1] = 0), computed on the device
// from the suffix array, its inverse and T' (built for the call by the parallel LF chain walks).
int fmx_build_lcp(fmx_index *ix, int32_t *lcp_out) {
    CHECK_IX(ix);
    if (!lcp_out) return fail(FMX_E_ARG, "null argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = ix->stream;
    const int64_t n = ix->n;
    if (n <= 2) { for (int64_t r = 0; r < n; ++r) lcp_out[r] = 0; return FMX_OK; }
    DBuf sa(st), isa(st), text(st), lcp(st);
    CU(sa.alloc((size_t)n * 4)); CU(isa.alloc((size_t)n * 4)); CU(text.alloc((size_t)n + 16)); CU(lcp.alloc((size_t)n * 4));
    std::string err;
    cudaError_t e = build_full_sa(ix->d_full, ix->cfg.layout, sa.as<uint32_t>(), isa.as<uint32_t>(), text.as<uint8_t>(), st, err);
    if (e != cudaSuccess) return fail(err.empty() ? FMX_E_CUDA : FMX_E_FORMAT, "suffix array construction failed: %s", err.empty() ? cudaGetErrorString(e) : err.c_str());
    CU(build_lcp(sa.as<uint32_t>(), isa.as<uint32_t>(), text.as<uint8_t>(), n, lcp.as<int32_t>(), st));
    CU(cudaMemcpyAsync(lcp_out, lcp.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return FMX_OK;
}

// LCPCreator(filename).create()  (bwtmerger.scala:558-652): <base>.lcp = big-endian int32, no header; entry k-1 is written for every row
// k >= 1 (and entry 0 for row 0), so the file holds max(n-1, 1) entries — LCPLoader (:176-211) reads them back.
int fmx_write_lcp_file(fmx_index *ix, const char *path) {
    CHECK_IX(ix);
    if (!path) return fail(FMX_E_ARG, "null argument");
    std::vector<int32_t> h((size_t)ix->n);
    int rc = fmx_build_lcp(ix, h.data());
    if (rc) return rc;
    const int64_t entries = std::max<int64_t>(ix->n - 1, 1);
    const std::string file = strip_extension(path) + ".lcp";
    FILE *f = std::fopen(file.c_str(), "wb");
    if (!f) return fail(FMX_E_IO, "cannot create %s", file.c_str());
    std::vector<uint8_t> buf(1 << 20);
    bool ok = true;
    for (int64_t i = 0; ok && i < entries;) {
        size_t k = 0;
        for (; k + 4 <= buf.size() && i < entries; ++i, k += 4) {
            const uint32_t v = (uint32_t)h[(size_t)i];
            buf[k] = (uint8_t)(v >> 24); buf[k + 1] = (uint8_t)(v >> 16); buf[k + 2] = (uint8_t)(v >> 8); buf[k + 3] = (uint8_t)v;
        }
        ok = std::fwrite(buf.data(), 1, k, f) == k;
    }
    std::fclose(f);
    if (!ok) return fail(FMX_E_IO, "short write %s", file.c_str());
    return FMX_OK;
}

// SACreator.create (bwtmerger.scala:535-556): <base>.sa = n x 32-bit big-endian, no header, sa[r] as bwtFm2sa (util.scala:213-224).
// The words are unsigned: positions at or beyond 2^31 (n < 2^32 - 1) are written as they are.
// The reference walks the .fm array with one seek+write per row; here the suffix array the index already holds (or one built for
// the occasion by the parallel LF chain walks) is copied out.
int fmx_write_sa_file(fmx_index *ix, const char *path) {
    CHECK_IX(ix);
    if (!path) return fail(FMX_E_ARG, "null argument");
    std::lock_guard<std::mutex> lk(ix->mu);
    DeviceGuard g(ix->device);
    cudaStream_t st = ix->stream;
    const int64_t n = ix->n;
    std::vector<uint32_t> h((size_t)n);
    if (ix->d.sa != nullptr) {
        CU(cudaMemcpyAsync(h.data(), ix->d.sa, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    } else if (n <= 2) {
        for (int64_t r = 0; r < n; ++r) h[(size_t)r] = (uint32_t)(r == ix->eof ? 0 : n - 1);      // n = 1: sa = [0]; n = 2: sa[eof] = 0, sa[0] = 1
    } else {
        DBuf sa(st), isa(st), text(st);
        CU(sa.alloc((size_t)n * 4)); CU(isa.alloc((size_t)n * 4)); CU(text.alloc((size_t)n + 16));
        std::string err;
        cudaError_t e = build_full_sa(ix->d, ix->cfg.layout, sa.as<uint32_t>(), isa.as<uint32_t>(), text.as<uint8_t>(), st, err);
        if (e != cudaSuccess) return fail(err.empty() ? FMX_E_CUDA : FMX_E_FORMAT, "suffix array construction failed: %s", err.empty() ? cudaGetErrorString(e) : err.c_str());
        CU(cudaMemcpyAsync(h.data(), sa.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    const std::string file = strip_extension(path) + ".sa";
    FILE *f = std::fopen(file.c_str(), "wb");
    if (!f) return fail(FMX_E_IO, "cannot create %s", file.c_str());
    std::vector<uint8_t> buf(1 << 20);
    bool ok = true;
    for (int64_t i = 0; ok && i < n;) {
        size_t k = 0;
        for (; k + 4 <= buf.size() && i < n; ++i, k += 4) {
            const uint32_t v = h[(size_t)i];
            buf[k] = (uint8_t)(v >> 24); buf[k + 1] = (uint8_t)(v >> 16); buf[k + 2] = (uint8_t)(v >> 8); buf[k + 3] = (uint8_t)v;
        }
        ok = std::fwrite(buf.data(), 1, k, f) == k;
    }
    std::fclose(f);
    if (!ok) return fail(FMX_E_IO, "short write %s", file.c_str());
    return FMX_OK;
}

}  // extern "C"

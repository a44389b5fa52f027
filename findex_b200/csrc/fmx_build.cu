// fmx_build.cu — device-side construction: (a) the GPU rank structures from the BWT ("index upload", K0),
// (b) sampled-suffix-array marks/samples by parallel LF chain walks, (c) suffix sorting of a text by prefix
// doubling to produce .bwt/.aux for synthetic configs (SURVEY.md §8f rank 1; replaces BWTMerger2.merge,
// src/main/scala/org/fmindex/bwtmerger.scala:1085-1260, for texts that fit in HBM — any correct suffix
// sorter yields the same, unique BWT).
#include "fmx_build.cuh"

#include "fmx_cub.cuh"

namespace fmx {

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return e_; } while (0)

// ======================================================================================================
// (a) rank structures
// ======================================================================================================
__global__ void map_codes_kernel(const uint8_t *__restrict__ bwt, int64_t n, uint32_t eof, const uint8_t *__restrict__ code,
                                 uint8_t *__restrict__ out) {
    __shared__ uint8_t sc[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sc[i] = code[i];
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = (i == eof) ? (uint8_t)0 : sc[bwt[i]];
}

// one thread per payload word of one bitvector: bit j of word w = (codes[32w + j] >> bit) & 1
__global__ void pack_level_kernel(const uint8_t *__restrict__ codes, int64_t n, int bit, uint32_t *__restrict__ blocks,
                                  int64_t nblk) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nblk * 15) return;
    const int64_t p0 = w * 32;
    uint32_t word = 0;
    if (p0 + 32 <= n) {
        const uint4 a = reinterpret_cast<const uint4 *>(codes + p0)[0], b = reinterpret_cast<const uint4 *>(codes + p0)[1];
        const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t m = (v[k] >> bit) & 0x01010101u;                  // bit of each of 4 codes, at bit 0 of each byte
            word |= (((m & 0x01u) | ((m >> 7) & 0x02u) | ((m >> 14) & 0x04u) | ((m >> 21) & 0x08u))) << (4 * k);
        }
    } else {
        for (int j = 0; j < 32 && p0 + j < n; ++j) word |= (uint32_t)((codes[p0 + j] >> bit) & 1u) << j;
    }
    blocks[(w / 15) * 16 + 1 + (w % 15)] = word;
}

// PLANES: a CTA stages TB blocks' worth of BWT bytes in shared memory and emits that column of every plane
template <int TB>
__global__ void __launch_bounds__(256)
pack_planes_kernel(const uint8_t *__restrict__ bwt, int64_t n, uint32_t eof, const uint8_t *__restrict__ sym, int sigma,
                   uint32_t *__restrict__ blocks, int64_t nblk) {
    __shared__ __align__(16) uint8_t tile[TB * 480];
    const int64_t b0 = (int64_t)blockIdx.x * TB, pos0 = b0 * 480;
    for (int i = threadIdx.x; i < TB * 480; i += 256) {
        const int64_t p = pos0 + i;
        tile[i] = (p < n && p != (int64_t)eof) ? bwt[p] : (uint8_t)0;       // 0 never equals a real symbol
    }
    __syncthreads();
    constexpr int W = TB * 15;
    for (int idx = threadIdx.x; idx < sigma * W; idx += 256) {
        const int code = idx / W, w = idx % W;
        const uint32_t pat = (uint32_t)sym[code] * 0x01010101u;
        const uint4 a = reinterpret_cast<const uint4 *>(tile + w * 32)[0], b = reinterpret_cast<const uint4 *>(tile + w * 32)[1];
        const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t word = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t eq = __vcmpeq4(v[k], pat);                           // 0xFF per equal byte
            word |= (((eq & 0x08040201u) * 0x01010101u) >> 24) << (4 * k);
        }
        const int64_t blk = b0 + w / 15;
        if (blk < nblk) blocks[((int64_t)code * nblk + blk) * 16 + 1 + (w % 15)] = word;
    }
}

__global__ void block_popc_kernel(const uint32_t *__restrict__ blocks, int64_t nblk_total, uint32_t *__restrict__ cnt) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk_total) return;
    const uint4 *p = reinterpret_cast<const uint4 *>(blocks + b * 16);
    const uint4 q0 = p[0], q1 = p[1], q2 = p[2], q3 = p[3];
    cnt[b] = __popc(q0.y) + __popc(q0.z) + __popc(q0.w) + __popc(q1.x) + __popc(q1.y) + __popc(q1.z) + __popc(q1.w) +
             __popc(q2.x) + __popc(q2.y) + __popc(q2.z) + __popc(q2.w) + __popc(q3.x) + __popc(q3.y) + __popc(q3.z) + __popc(q3.w);
}

// header of block b of plane p = ones before it inside plane p = pre[p*nblk+b] - pre[p*nblk]
__global__ void write_headers_kernel(uint32_t *__restrict__ blocks, const uint32_t *__restrict__ pre, int64_t nblk, int64_t nplanes) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblk * nplanes) return;
    blocks[b * 16] = pre[b] - pre[(b / nblk) * nblk];
}

static cudaError_t finish_headers(uint32_t *d_blocks, int64_t nblk, int64_t nplanes, cudaStream_t st) {
    const int64_t tot = nblk * nplanes;
    uint32_t *cnt = nullptr, *pre = nullptr;
    CK(cudaMallocAsync(&cnt, tot * 4, st));
    CK(cudaMallocAsync(&pre, tot * 4, st));
    block_popc_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(d_blocks, tot, cnt);
    CK(exclusive_sum_u32(cnt, pre, tot, st));          // total ones over all planes <= n < 2^32: no overflow
    write_headers_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(d_blocks, pre, nblk, nplanes);
    cudaFreeAsync(cnt, st);
    cudaFreeAsync(pre, st);
    return cudaGetLastError();
}

cudaError_t build_wm(const uint8_t *d_bwt, int64_t n, uint32_t eof, const uint8_t *d_code, int levels, uint32_t *d_blocks,
                     int64_t nblk, cudaStream_t st) {
    uint8_t *cur = nullptr, *nxt = nullptr;
    CK(cudaMallocAsync(&cur, n + 64, st));
    CK(cudaMallocAsync(&nxt, n + 64, st));
    map_codes_kernel<<<148 * 8, 256, 0, st>>>(d_bwt, n, eof, d_code, cur);
    for (int l = 0; l < levels; ++l) {
        const int bit = levels - 1 - l;
        pack_level_kernel<<<(unsigned)((nblk * 15 + 255) / 256), 256, 0, st>>>(cur, n, bit, d_blocks + (int64_t)l * nblk * 16, nblk);
        if (l + 1 < levels) {
            CK(stable_partition_bit_u8(cur, nxt, n, bit, st));
            uint8_t *t = cur; cur = nxt; nxt = t;
        }
    }
    CK(finish_headers(d_blocks, nblk, levels, st));
    cudaFreeAsync(cur, st);
    cudaFreeAsync(nxt, st);
    return cudaGetLastError();
}

// ---- multi-ary wavelet matrix (FMX_LAYOUT_WMX) ---------------------------------------------------------------------------------------
// one thread per payload word of one level: digit j of the word = (codes[first + j] >> shift) & (2^b - 1)
__global__ void pack_digits_kernel(const uint8_t *__restrict__ codes, int64_t n, int shift, int b, uint32_t *__restrict__ blocks, int64_t nblk) {
    const int H = 1 << b, per = 32 / b, pw = 32 - H;            // header words, digits per word, payload words per block
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= nblk * pw) return;
    const int64_t blk = w / pw;
    const int k = (int)(w - blk * pw);
    const int64_t p0 = (blk * pw + k) * per;
    uint32_t word = 0;
    const uint32_t m = (1u << b) - 1u;
    for (int j = 0; j < per && p0 + j < n; ++j) word |= (((uint32_t)codes[p0 + j] >> shift) & m) << (j * b);
    blocks[blk * 32 + H + k] = word;
}
// cnt[v * nblk + blk] = occurrences of digit v among the rows of block blk (rows beyond n do not count)
__global__ void digit_counts_kernel(const uint8_t *__restrict__ codes, int64_t n, int shift, int b, uint32_t *__restrict__ cnt, int64_t nblk) {
    const int H = 1 << b, R = (32 - H) * (32 / b);
    const int64_t blk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (blk >= nblk) return;
    uint32_t c[16];
#pragma unroll
    for (int v = 0; v < 16; ++v) c[v] = 0;
    const uint32_t m = (1u << b) - 1u;
    const int64_t p0 = blk * R;
    for (int j = 0; j < R && p0 + j < n; ++j) {
        const uint32_t d = ((uint32_t)codes[p0 + j] >> shift) & m;
#pragma unroll
        for (int v = 0; v < 16; ++v) c[v] += (d == (uint32_t)v);
    }
    for (int v = 0; v < H; ++v) cnt[(int64_t)v * nblk + blk] = c[v];
}
__global__ void write_headers_x_kernel(uint32_t *__restrict__ blocks, const uint32_t *__restrict__ pre, int64_t nblk, int H) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nblk * H) return;
    const int64_t v = t / nblk, blk = t - v * nblk;
    blocks[blk * 32 + v] = pre[t] - pre[v * nblk];
}
cudaError_t build_wmx(const uint8_t *d_bwt, int64_t n, uint32_t eof, const uint8_t *d_code, int b, int levels, uint32_t *d_blocks, int64_t nblk,
                      cudaStream_t st) {
    const int H = 1 << b;
    uint8_t *cur = nullptr, *nxt = nullptr;
    uint32_t *cnt = nullptr, *pre = nullptr;
    CK(cudaMallocAsync(&cur, n + 64, st));
    CK(cudaMallocAsync(&nxt, n + 64, st));
    CK(cudaMallocAsync(&cnt, (size_t)nblk * H * 4, st));
    CK(cudaMallocAsync(&pre, (size_t)nblk * H * 4, st));
    map_codes_kernel<<<148 * 8, 256, 0, st>>>(d_bwt, n, eof, d_code, cur);
    for (int l = 0; l < levels; ++l) {
        const int shift = b * (levels - 1 - l);
        uint32_t *lv = d_blocks + (int64_t)l * nblk * 32;
        pack_digits_kernel<<<(unsigned)((nblk * (32 - H) + 255) / 256), 256, 0, st>>>(cur, n, shift, b, lv, nblk);
        digit_counts_kernel<<<(unsigned)((nblk + 127) / 128), 128, 0, st>>>(cur, n, shift, b, cnt, nblk);
        CK(exclusive_sum_u32(cnt, pre, nblk * H, st));          // total digits = n < 2^32: no overflow
        write_headers_x_kernel<<<(unsigned)((nblk * H + 255) / 256), 256, 0, st>>>(lv, pre, nblk, H);
        if (l + 1 < levels) {
            CK(stable_partition_digit_u8(cur, nxt, n, shift, shift + b, st));
            uint8_t *t = cur; cur = nxt; nxt = t;
        }
    }
    cudaFreeAsync(cur, st); cudaFreeAsync(nxt, st); cudaFreeAsync(cnt, st); cudaFreeAsync(pre, st);
    return cudaGetLastError();
}

cudaError_t build_planes(const uint8_t *d_bwt, int64_t n, uint32_t eof, const uint8_t *d_sym, int sigma, uint32_t *d_blocks,
                         int64_t nblk, cudaStream_t st) {
    constexpr int TB = 8;
    if (sigma > 0) pack_planes_kernel<TB><<<(unsigned)((nblk + TB - 1) / TB), 256, 0, st>>>(d_bwt, n, eof, d_sym, sigma, d_blocks, nblk);
    CK(finish_headers(d_blocks, nblk, sigma > 0 ? sigma : 1, st));       // an empty text still owns one (all-zero) plane
    return cudaGetLastError();
}

// ======================================================================================================
// (b) sampled suffix array by parallel LF chain walks
// ======================================================================================================
// Rows k*S (and the eof row) are chain starts.  LF is one n-cycle, so walking from every start to the next
// start partitions it; the host links the chains from sa[eof] = 0 (util.scala:213-224: sa[eof]=0, and
// sa[LF(r)] = sa[r]-1 mod n), and a second walk stamps every row whose sa is a multiple of `rate`.
template <int LAYOUT>
__global__ void __launch_bounds__(kThreads)
chain_len_kernel(const __grid_constant__ DevIndex ix, uint32_t S, uint32_t nchains, uint32_t eof_chain, uint32_t *__restrict__ next,
                 uint32_t *__restrict__ len) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const uint32_t j = blockIdx.x * kThreads + threadIdx.x;
    if (j >= nchains) return;
    uint32_t r = (j == eof_chain) ? ix.eof : j * S, steps = 0;
    for (;;) {
        r = lf_value<1, LAYOUT>(ix, tb, ix.bwt[r], r);
        ++steps;
        if (r == ix.eof) { next[j] = eof_chain; break; }
        if (r % S == 0) { next[j] = r / S; break; }
        // LF of a consistent index is one n-cycle: a walk that leaves the rows or outlives n steps is on a corrupt index.  The chain is
        // closed on itself with an impossible length, which fails the host's single-cycle check (prepare_chains) instead of hanging.
        if (r >= ix.n || steps > ix.n) { next[j] = j; steps = 0xFFFFFFFFu; break; }
    }
    len[j] = steps;
}

template <int LAYOUT>
__global__ void __launch_bounds__(kThreads)
chain_mark_kernel(const __grid_constant__ DevIndex ix, uint32_t S, uint32_t nchains, uint32_t eof_chain, const uint32_t *__restrict__ start_sa,
                  uint32_t rate, uint32_t *__restrict__ mark_blocks, uint2 *__restrict__ pairs, unsigned long long *n_pairs, uint32_t text_rate,
                  uint32_t *__restrict__ tsamp) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const uint32_t j = blockIdx.x * kThreads + threadIdx.x;
    if (j >= nchains) return;
    uint32_t r = (j == eof_chain) ? ix.eof : j * S, v = start_sa[j];
    for (;;) {
        if (tsamp != nullptr && v % text_rate == 0) tsamp[v / text_rate] = r;
        if (rate != 0 && v % rate == 0) {
            const uint32_t b = r / kBitsPerBlock, o = r - b * kBitsPerBlock;
            atomicOr(&mark_blocks[(uint64_t)b * 16 + 1 + (o >> 5)], 1u << (o & 31));
            pairs[atomicAdd(n_pairs, 1ull)] = make_uint2(r, v);
        }
        r = lf_value<1, LAYOUT>(ix, tb, ix.bwt[r], r);
        v = (v == 0) ? ix.n - 1 : v - 1;
        if (r == ix.eof || r % S == 0 || r >= ix.n) break;
    }
}

__global__ void scatter_samples_kernel(const uint4 *__restrict__ mark, const uint2 *__restrict__ pairs, int64_t np, uint32_t *__restrict__ samples) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= np) return;
    const uint2 p = pairs[i];
    samples[rank_one<1>(mark, p.x, nullptr)] = p.y;
}

// full-SA variant of the second walk: every row gets its sa value; isa and T' fall out of the same walk
template <int LAYOUT>
__global__ void __launch_bounds__(kThreads)
chain_fullsa_kernel(const __grid_constant__ DevIndex ix, uint32_t S, uint32_t nchains, uint32_t eof_chain, const uint32_t *__restrict__ start_sa,
                    uint32_t *__restrict__ sa, uint32_t *__restrict__ isa, uint8_t *__restrict__ text) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const uint32_t j = blockIdx.x * kThreads + threadIdx.x;
    if (j >= nchains) return;
    uint32_t r = (j == eof_chain) ? ix.eof : j * S, v = start_sa[j];
    for (;;) {
        const uint32_t c = ix.bwt[r];
        sa[r] = v;
        isa[v] = r;
        if (v > 0) text[v - 1] = (uint8_t)c;          // BWT[r] = T'[sa[r]-1]
        else text[ix.n - 1] = 0;                      // the '$'
        r = lf_value<1, LAYOUT>(ix, tb, c, r);
        v = (v == 0) ? ix.n - 1 : v - 1;
        if (r == ix.eof || r % S == 0 || r >= ix.n) break;
    }
}

namespace {
struct Chains {
    uint32_t S = 1, nchains = 0, eof_chain = 0;
    uint32_t *d_start = nullptr;     // sa value of every chain's first row
};

// first walk + host linking (sa[eof] = 0, each LF step decrements the text position mod n)
cudaError_t prepare_chains(const DevIndex &ix, int layout, Chains &ch, cudaStream_t st, std::string &err) {
    const uint64_t n = ix.n;
    const uint64_t target = n < (1u << 20) ? n : (1u << 20);
    uint32_t S = (uint32_t)((n + target - 1) / target);
    if (S == 0) S = 1;
    const uint32_t base_chains = (uint32_t)((n + S - 1) / S);
    const bool eof_is_grid = (ix.eof % S) == 0;
    ch.S = S;
    ch.eof_chain = eof_is_grid ? ix.eof / S : base_chains;
    ch.nchains = eof_is_grid ? base_chains : base_chains + 1;
    const uint32_t nchains = ch.nchains;
    uint32_t *d_next, *d_len;
    CK(cudaMallocAsync(&d_next, nchains * 4ull, st));
    CK(cudaMallocAsync(&d_len, nchains * 4ull, st));
    CK(cudaMallocAsync(&ch.d_start, nchains * 4ull, st));
    const unsigned grid = (nchains + kThreads - 1) / kThreads;
    if (layout == FMX_LAYOUT_PLANES) chain_len_kernel<FMX_LAYOUT_PLANES><<<grid, kThreads, 0, st>>>(ix, S, nchains, ch.eof_chain, d_next, d_len);
    else if (layout == FMX_LAYOUT_WMX) chain_len_kernel<FMX_LAYOUT_WMX><<<grid, kThreads, 0, st>>>(ix, S, nchains, ch.eof_chain, d_next, d_len);
    else chain_len_kernel<FMX_LAYOUT_WM><<<grid, kThreads, 0, st>>>(ix, S, nchains, ch.eof_chain, d_next, d_len);
    std::vector<uint32_t> nx(nchains), ln(nchains), sv(nchains, 0);
    CK(cudaMemcpyAsync(nx.data(), d_next, nchains * 4ull, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(ln.data(), d_len, nchains * 4ull, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    cudaFreeAsync(d_next, st);
    cudaFreeAsync(d_len, st);
    uint64_t total = 0, v = 0;
    uint32_t cur = ch.eof_chain, visited = 0;
    do {
        sv[cur] = (uint32_t)v;
        total += ln[cur];
        v = (v + n - (ln[cur] % n)) % n;
        cur = nx[cur];
        ++visited;
    } while (cur != ch.eof_chain && visited <= nchains);
    if (cur != ch.eof_chain || visited != nchains || total != n) {
        err = "BWT is not a single LF cycle (corrupt .bwt/.aux?)";
        cudaFreeAsync(ch.d_start, st);
        ch.d_start = nullptr;
        return cudaErrorInvalidValue;
    }
    CK(cudaMemcpyAsync(ch.d_start, sv.data(), nchains * 4ull, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));                  // sv is a local
    return cudaSuccess;
}
}  // namespace

cudaError_t build_sa_samples(const DevIndex &ix, int layout, int rate, uint32_t *d_mark_blocks, int64_t nblk, uint32_t *d_samples,
                             int64_t n_samples, cudaStream_t st, std::string &err, int text_rate, uint32_t *d_tsamp) {
    Chains ch;
    CK(prepare_chains(ix, layout, ch, st, err));
    const unsigned grid = (ch.nchains + kThreads - 1) / kThreads;
    uint2 *d_pairs = nullptr; unsigned long long *d_np = nullptr;
    if (rate > 0) {
        CK(cudaMallocAsync(&d_pairs, (size_t)n_samples * 8, st));
        CK(cudaMallocAsync(&d_np, 8, st));
        CK(cudaMemsetAsync(d_np, 0, 8, st));
        CK(cudaMemsetAsync(d_mark_blocks, 0, (size_t)nblk * 64, st));
    }
    const uint32_t r32 = rate > 0 ? (uint32_t)rate : 0u, t32 = d_tsamp ? (uint32_t)text_rate : 0u;
    if (layout == FMX_LAYOUT_PLANES) chain_mark_kernel<FMX_LAYOUT_PLANES><<<grid, kThreads, 0, st>>>(ix, ch.S, ch.nchains, ch.eof_chain, ch.d_start, r32, d_mark_blocks, d_pairs, d_np, t32, d_tsamp);
    else if (layout == FMX_LAYOUT_WMX) chain_mark_kernel<FMX_LAYOUT_WMX><<<grid, kThreads, 0, st>>>(ix, ch.S, ch.nchains, ch.eof_chain, ch.d_start, r32, d_mark_blocks, d_pairs, d_np, t32, d_tsamp);
    else chain_mark_kernel<FMX_LAYOUT_WM><<<grid, kThreads, 0, st>>>(ix, ch.S, ch.nchains, ch.eof_chain, ch.d_start, r32, d_mark_blocks, d_pairs, d_np, t32, d_tsamp);
    if (rate <= 0) {                                         // text samples only
        cudaFreeAsync(ch.d_start, st);
        return cudaGetLastError();
    }
    CK(finish_headers(d_mark_blocks, nblk, 1, st));
    unsigned long long np = 0;
    CK(cudaMemcpyAsync(&np, d_np, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if ((int64_t)np != n_samples) { err = "sample count mismatch"; return cudaErrorInvalidValue; }
    scatter_samples_kernel<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(reinterpret_cast<const uint4 *>(d_mark_blocks), d_pairs, (int64_t)np, d_samples);
    cudaFreeAsync(d_pairs, st); cudaFreeAsync(d_np, st);
    cudaFreeAsync(ch.d_start, st);
    return cudaGetLastError();
}

// fused walk blocks for locate: 56 BWT bytes + their 56 mark bits per 64-byte block
__global__ void build_walk_blocks_kernel(const uint8_t *__restrict__ bwt, const uint32_t *__restrict__ mark_blocks, int64_t n, uint8_t *__restrict__ bm,
                                         int64_t nwb) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nwb) return;
    uint8_t out[64];
#pragma unroll
    for (int i = 0; i < 64; ++i) out[i] = 0;
    for (int o = 0; o < 56; ++o) {
        const int64_t r = b * 56 + o;
        if (r >= n) break;
        out[o] = bwt[r];
        const int64_t blk = r / kBitsPerBlock, off = r - blk * kBitsPerBlock;
        const uint32_t bit = (mark_blocks[blk * 16 + 1 + (off >> 5)] >> (off & 31)) & 1u;
        out[56 + (o >> 3)] |= (uint8_t)(bit << (o & 7));
    }
    uint4 *dst = reinterpret_cast<uint4 *>(bm + b * 64);
    const uint4 *src = reinterpret_cast<const uint4 *>(out);
    dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2]; dst[3] = src[3];
}
cudaError_t build_walk_blocks(const uint8_t *d_bwt, const uint32_t *d_mark_blocks, int64_t n, uint8_t *d_bm, int64_t nwb, cudaStream_t st) {
    build_walk_blocks_kernel<<<(unsigned)((nwb + 127) / 128), 128, 0, st>>>(d_bwt, d_mark_blocks, n, d_bm, nwb);
    return cudaGetLastError();
}

// isat[p] = { isa[p], 96 bits holding the next `syms` symbols of T' at `bits` bits each }: stored value = dense code + 1,
// 0 for the '$' and past the end
__global__ void build_isat_kernel(const uint32_t *__restrict__ isa, const uint8_t *__restrict__ text, const uint8_t *__restrict__ code, int64_t n,
                                  int bits, int syms, uint4 *__restrict__ isat) {
    __shared__ uint8_t sc[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sc[i] = code[i];
    __syncthreads();
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    unsigned long long lo = 0, hi = 0;                          // 96 bits: lo = bits 0..63, hi = bits 64..95
    for (int k = 0; k < syms; ++k) {
        unsigned long long v = 0;
        if (p + k < n) { const uint8_t t = text[p + k]; v = t ? (unsigned long long)sc[t] + 1ull : 0ull; }
        const int o = k * bits;
        if (o < 64) { lo |= v << o; if (o + bits > 64) hi |= v >> (64 - o); }
        else hi |= v << (o - 64);
    }
    isat[p] = make_uint4(isa[p], (uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi);
}
cudaError_t build_isat(const uint32_t *d_isa, const uint8_t *d_text, const uint8_t *d_code, int64_t n, int bits, int syms, uint4 *d_isat, cudaStream_t st) {
    build_isat_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_isa, d_text, d_code, n, bits, syms, d_isat);
    return cudaGetLastError();
}

// ctx[r] (32 B) = { isa[sa[r]-j] for the five hop lengths j = hops.h[0..4] (hops.h[4] = J), 96 bits = the J symbols T'[sa[r]-J .. sa[r]-1] in the
// isat packing }; positions before the start of T' read as symbol 0 / row 0 (symbol 0 never equals a pattern symbol, which is dense code + 1
// >= 1); raw = 1 (8-bit symbols): the text bytes themselves are stored (0 = '$' / before the start; patterns with a zero byte never take this path)
__global__ void build_ctx_kernel(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ isa, const uint8_t *__restrict__ text,
                                 const uint8_t *__restrict__ code, int64_t n, int bits, int J, int raw, CtxHops hops, uint4 *__restrict__ ctx) {
    __shared__ uint8_t sc[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sc[i] = code[i];
    __syncthreads();
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int64_t p = sa[r];
    uint32_t row[5];
#pragma unroll
    for (int t = 0; t < 5; ++t) { const int64_t q = p - hops.h[t]; row[t] = q >= 0 ? isa[q] : 0u; }
    unsigned long long lo = 0, hi = 0;
    for (int k = 0; k < J; ++k) {
        const int64_t q = p - J + k;
        unsigned long long v = 0;
        if (q >= 0) { const uint8_t t = text[q]; v = raw ? (unsigned long long)t : (t ? (unsigned long long)sc[t] + 1ull : 0ull); }
        const int o = k * bits;
        if (o < 64) { lo |= v << o; if (o + bits > 64) hi |= v >> (64 - o); }
        else hi |= v << (o - 64);
    }
    ctx[2 * r] = make_uint4(row[0], row[1], row[2], row[3]);
    ctx[2 * r + 1] = make_uint4(row[4], (uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi);
}
cudaError_t build_ctx(const uint32_t *d_sa, const uint32_t *d_isa, const uint8_t *d_text, const uint8_t *d_code, int64_t n, int bits, int J,
                      int raw, const CtxHops &hops, uint4 *d_ctx, cudaStream_t st) {
    build_ctx_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_sa, d_isa, d_text, d_code, n, bits, J, raw, hops, d_ctx);
    return cudaGetLastError();
}

// Hop lengths stored per context depth J = 96 / bits: the 5-subset of 1..J (with 1 and J) that minimises the worst excess of fetches over
// ceil(rem / J), then the mean, over rem <= 4J (offline exhaustive search); J = 12 prefers multiples of 4 (k-mer lengths 8/12/16/20/24/32
// after a depth-4 table finish in ceil(rem / 12) fetches).  plan[rem] = index of the first hop of a fewest-fetches decomposition of rem,
// plan[128 + rem] = that number of fetches (rem <= 127).
void ctx_hop_plan(int J, CtxHops &hops, uint8_t plan[256]) {
    static const int known[][6] = {{12, 1, 3, 4, 8, 12},  {13, 1, 3, 5, 6, 13},   {16, 1, 4, 6, 15, 16},  {19, 1, 4, 5, 16, 19},
                                   {24, 1, 4, 6, 15, 24}, {32, 1, 4, 9, 21, 32}, {48, 1, 5, 12, 33, 48}, {96, 1, 6, 16, 48, 96}};
    int S[5] = {1, (J + 7) / 8, (J + 3) / 4, (J + 1) / 2, J};
    for (const auto &k : known) if (k[0] == J) for (int t = 0; t < 5; ++t) S[t] = k[1 + t];
    for (int t = 0; t < 8; ++t) hops.h[t] = t < 5 ? S[t] : 0;
    int cost[128];
    cost[0] = 0;
    plan[0] = 0; plan[128] = 0;
    for (int r = 1; r < 128; ++r) {
        int best = 1 << 20, bt = 0;
        for (int t = 4; t >= 0; --t)                            // ties go to the longer hop
            if (S[t] <= r && cost[r - S[t]] + 1 < best) { best = cost[r - S[t]] + 1; bt = t; }
        cost[r] = best;
        plan[r] = (uint8_t)bt;
        plan[128 + r] = (uint8_t)best;
    }
}

// ctx8[r] (8 B) = { isa[sa[r]-J], the J <= 16 symbols T'[sa[r]-J .. sa[r]-1] as 2-bit dense codes }; row 0xFFFFFFFF when sa[r] < J
__global__ void build_ctx8_kernel(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ isa, const uint8_t *__restrict__ text,
                                  const uint8_t *__restrict__ code, int64_t n, int J, uint2 *__restrict__ ctx8) {
    __shared__ uint8_t sc[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) sc[i] = code[i];
    __syncthreads();
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int64_t q = (int64_t)sa[r] - J;
    if (q < 0) { ctx8[r] = make_uint2(0xFFFFFFFFu, 0u); return; }
    uint32_t syms = 0;
    for (int k = 0; k < J; ++k) syms |= ((uint32_t)sc[text[q + k]] & 3u) << (2 * k);
    ctx8[r] = make_uint2(isa[q], syms);
}
cudaError_t build_ctx8(const uint32_t *d_sa, const uint32_t *d_isa, const uint8_t *d_text, const uint8_t *d_code, int64_t n, int J,
                       uint2 *d_ctx8, cudaStream_t st) {
    build_ctx8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_sa, d_isa, d_text, d_code, n, J, d_ctx8);
    return cudaGetLastError();
}

cudaError_t build_full_sa(const DevIndex &ix, int layout, uint32_t *d_sa, uint32_t *d_isa, uint8_t *d_text, cudaStream_t st, std::string &err) {
    Chains ch;
    CK(prepare_chains(ix, layout, ch, st, err));
    const unsigned grid = (ch.nchains + kThreads - 1) / kThreads;
    if (layout == FMX_LAYOUT_PLANES) chain_fullsa_kernel<FMX_LAYOUT_PLANES><<<grid, kThreads, 0, st>>>(ix, ch.S, ch.nchains, ch.eof_chain, ch.d_start, d_sa, d_isa, d_text);
    else if (layout == FMX_LAYOUT_WMX) chain_fullsa_kernel<FMX_LAYOUT_WMX><<<grid, kThreads, 0, st>>>(ix, ch.S, ch.nchains, ch.eof_chain, ch.d_start, d_sa, d_isa, d_text);
    else chain_fullsa_kernel<FMX_LAYOUT_WM><<<grid, kThreads, 0, st>>>(ix, ch.S, ch.nchains, ch.eof_chain, ch.d_start, d_sa, d_isa, d_text);
    cudaFreeAsync(ch.d_start, st);
    return cudaGetLastError();
}

// LCP array = bwtFm2LCP (util.scala:153-212) / LCPCreator.create (bwtmerger.scala:583-650): lcp[r] = longest common prefix of the suffixes
// of rows r and r+1.  The reference walks the text positions in order carrying h-1 from one to the next (Kasai et al.); here every
// thread owns a run of kLcpRun consecutive text positions and does the same inside its run (h restarts at 0 at the run's first
// position, which only costs that one comparison its head start).  Characters are compared through T' directly; like the reference's
// fm walk, the neighbour's characters wrap around the end of T' (the unique '$' always stops the comparison first).
constexpr int kLcpRun = 64;
__global__ void lcp_kernel(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ isa, const uint8_t *__restrict__ text, int64_t n,
                           int32_t *__restrict__ lcp) {
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * kLcpRun;
    int64_t h = 0;
    for (int64_t i = i0; i < i0 + kLcpRun && i < n; ++i) {
        const uint32_t k = isa[i];
        if (k == 0) { h = 0; continue; }                    // row 0 ('$'): the reference stores LCP(0) = 0, row 1 stores it again
        const int64_t j = sa[k - 1];
        while (i + h < n) {
            int64_t q = j + h;
            if (q >= n) q -= n;
            if (text[i + h] != text[q]) break;
            ++h;
        }
        lcp[k - 1] = (int32_t)h;
        if (h > 0) --h;
    }
}
cudaError_t build_lcp(const uint32_t *d_sa, const uint32_t *d_isa, const uint8_t *d_text, int64_t n, int32_t *d_lcp, cudaStream_t st) {
    CK(cudaMemsetAsync(d_lcp, 0, (size_t)n * 4, st));
    const int64_t threads = (n + kLcpRun - 1) / kLcpRun;
    lcp_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(d_sa, d_isa, d_text, n, d_lcp);
    return cudaGetLastError();
}

// k-mer table: entry idx <-> the K-byte pattern P with P[K-1-j] = sym[digit_j(idx)] (digit 0 most significant = the byte search()
// consumes first, i.e. the LAST pattern byte); entry = (sp,ep) after those K backward steps, (0,0) when the interval is empty.
// Built level by level: level 1 is (C[c], C[c+1]); an entry of level j+1 is one backward step from its parent idx/sigma of level j
// with symbol idx%sigma — sigma^K * sigma/(sigma-1) steps in all instead of sigma^K * (K-1).  In lexicographic order (lex) the new symbol is
// the most significant digit instead: parent idx % sigma^(j), symbol idx / sigma^(j).  Dense codes ascend with the byte value, so there
// consecutive entries are consecutive intervals of rows.
__global__ void kmer_level1_kernel(const DevIndex ix, const uint8_t *__restrict__ sym, uint32_t sigma, uint2 *__restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= sigma) return;
    const uint32_t c = sym[t], a = ix.C[c], b = ix.C[c + 1];
    out[t] = a < b ? make_uint2(a, b) : make_uint2(0u, 0u);
}
template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
kmer_extend_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ sym, uint32_t sigma, const uint2 *__restrict__ prev,
                   unsigned long long count, bool lex, uint2 *__restrict__ out) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const unsigned long long t = (unsigned long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (t >= count) return;                                // group-uniform
    const unsigned long long sub = count / sigma;          // entries of the parent level
    const uint2 p = prev[lex ? t % sub : t / sigma];
    uint32_t sp = p.x, ep = p.y, touched = 0;
    if (sp < ep) backward_step<G, LAYOUT, false>(ix, tb, (uint32_t)sym[lex ? t / sub : t % sigma], sp, ep, touched);
    if ((threadIdx.x % G) == 0) out[t] = sp < ep ? make_uint2(sp, ep) : make_uint2(0u, 0u);
}

cudaError_t build_kmer_table(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_sym, uint32_t sigma, int K, uint2 *d_table, cudaStream_t st,
                             bool lex) {
    if (K < 1 || sigma < 1) return cudaErrorInvalidValue;
    std::vector<unsigned long long> size((size_t)K + 1, 1);
    for (int j = 1; j <= K; ++j) size[(size_t)j] = size[(size_t)j - 1] * sigma;
    uint2 *d_tmp = nullptr;
    if (K >= 2) CK(cudaMallocAsync(&d_tmp, size[(size_t)K - 1] * sizeof(uint2), st));
    auto buf = [&](int level) { return ((K - level) % 2 == 0) ? d_table : d_tmp; };      // level K lands in d_table
    kmer_level1_kernel<<<(sigma + 255) / 256, 256, 0, st>>>(ix, d_sym, sigma, buf(1));
    const int G = (cfg.lanes == 1 || cfg.lanes == 2 || cfg.lanes == 4) ? cfg.lanes : 2;
    for (int j = 2; j <= K; ++j) {
        const unsigned long long cnt = size[(size_t)j];
        const unsigned long long per = kThreads / G;
        const unsigned grid = (unsigned)((cnt + per - 1) / per);
#define CALL(GG, LAY) kmer_extend_kernel<GG, LAY><<<grid, kThreads, 0, st>>>(ix, d_sym, sigma, buf(j - 1), cnt, lex, buf(j))
        if (ix.layout == FMX_LAYOUT_PLANES) { if (G == 1) CALL(1, FMX_LAYOUT_PLANES); else if (G == 2) CALL(2, FMX_LAYOUT_PLANES); else CALL(4, FMX_LAYOUT_PLANES); }
        else if (ix.layout == FMX_LAYOUT_WMX) { if (G == 1) CALL(1, FMX_LAYOUT_WMX); else if (G == 2) CALL(2, FMX_LAYOUT_WMX); else CALL(4, FMX_LAYOUT_WMX); }
        else { if (G == 1) CALL(1, FMX_LAYOUT_WM); else if (G == 2) CALL(2, FMX_LAYOUT_WM); else CALL(4, FMX_LAYOUT_WM); }
#undef CALL
        CK(cudaGetLastError());
    }
    if (d_tmp) cudaFreeAsync(d_tmp, st);
    return cudaGetLastError();
}

// k-mer group blocks (layout: fmx_device.cuh, kmer_group): one thread per group of 8 lexicographically consecutive entries reads them and
// writes the block over the same 64 bytes.  A group is narrow when its non-empty intervals follow each other without a gap and span at most
// 255 rows; the J-hop halves of the row contexts of its first rows (up to kKmerInlineRows) then fill the rest of the block.
__global__ void pack_kmer_groups_kernel(uint2 *__restrict__ table, unsigned long long entries, const uint4 *__restrict__ ctx) {
    const unsigned long long g = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g * kKmerGroup >= entries) return;
    uint2 v[kKmerGroup];
#pragma unroll
    for (uint32_t e = 0; e < kKmerGroup; ++e) {
        const unsigned long long idx = g * kKmerGroup + e;
        v[e] = idx < entries ? table[idx] : make_uint2(0u, 0u);
        if (v[e].x >= v[e].y) v[e] = make_uint2(0u, 0u);
    }
    uint32_t base = 0, last = 0;
    bool any = false, gap = false;
#pragma unroll
    for (uint32_t e = 0; e < kKmerGroup; ++e) {
        if (v[e].x >= v[e].y) continue;
        if (!any) { base = v[e].x; any = true; }
        else if (v[e].x != last) gap = true;
        last = v[e].y;
    }
    uint32_t w[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) w[k] = 0;
    w[0] = base;
    if (gap || last - base > 255u) {
        uint32_t prev = base;
#pragma unroll
        for (uint32_t e = 0; e < kKmerGroup; ++e) {
            const bool ne = v[e].x < v[e].y;
            const uint32_t end = ne ? v[e].y : prev, lead = ne ? v[e].x - prev : 0u;      // lead <= k: rows of no k-mer
            w[4 + e] = end;
            w[12 + e / 4] |= (lead & 0xFFu) << (8 * (e % 4));
            prev = end;
        }
        w[3] = kKmerWide << 24;
    } else {
        uint32_t end = 0;
#pragma unroll
        for (uint32_t e = 0; e < kKmerGroup; ++e) {
            if (v[e].x < v[e].y) end = v[e].y - base;
            w[1 + e / 4] |= end << (8 * (e % 4));
        }
        const uint32_t kind = any ? min(last - base, kKmerInlineRows) : 0u;
        w[3] = kind << 24;
        for (uint32_t k = 0; k < kind; ++k) {
            const uint4 c = ctx[2ull * (base + k) + 1];
            w[4 + 4 * k] = c.x; w[5 + 4 * k] = c.y; w[6 + 4 * k] = c.z; w[7 + 4 * k] = c.w;
        }
    }
    uint4 *dst = reinterpret_cast<uint4 *>(table + g * kKmerGroup);
#pragma unroll
    for (int k = 0; k < 4; ++k) dst[k] = make_uint4(w[4 * k], w[4 * k + 1], w[4 * k + 2], w[4 * k + 3]);
}
cudaError_t pack_kmer_groups(uint2 *d_table, uint64_t entries, const uint4 *d_ctx, cudaStream_t st) {
    const unsigned long long groups = (entries + kKmerGroup - 1) / kKmerGroup;
    pack_kmer_groups_kernel<<<(unsigned)((groups + 255) / 256), 256, 0, st>>>(d_table, entries, d_ctx);
    return cudaGetLastError();
}

// Dictionary of wide intervals (DevIndex::dict): grown level by level from the dense k-mer table.  Level K = the table's entries of more
// than `min_rows` rows; level d+1 = one backward step from every level-d item with every symbol, kept when still wider than `min_rows`
// (a child of a narrow interval is narrow, so nothing is missed).  Items are appended to one array; the levels that fit `max_entries` are
// then hashed into 32-byte buckets (two {key, sp, ep} slots) at half load.
struct DictItem { unsigned long long key; uint32_t sp, ep; };

__global__ void dict_seed_kernel(const uint2 *__restrict__ kmer, unsigned long long entries, uint32_t sigma, int K, uint32_t bits, uint32_t min_rows,
                                 DictItem *__restrict__ out, unsigned long long cap, unsigned long long *__restrict__ counter) {
    const unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= entries) return;
    const uint2 v = kmer[idx];
    if (v.y - v.x <= min_rows || v.y <= v.x) return;
    // digit 0 of idx (most significant) is the first consumed symbol = the key's lowest field
    unsigned long long key = 0, r = idx;
    for (int j = K - 1; j >= 0; --j) { key |= (r % sigma) << (bits * (uint32_t)j); r /= sigma; }
    const unsigned long long slot = atomicAdd(counter, 1ull);
    if (slot < cap) out[slot] = DictItem{key | ((unsigned long long)(K - 1) << 60), v.x, v.y};
}

template <int G, int LAYOUT>
__global__ void __launch_bounds__(kThreads)
dict_extend_kernel(const __grid_constant__ DevIndex ix, const uint8_t *__restrict__ sym, uint32_t sigma, const DictItem *__restrict__ parents,
                   unsigned long long count, int d, int D, int Jc, uint32_t bits, uint32_t min_rows, DictItem *__restrict__ out,
                   unsigned long long cap, unsigned long long *__restrict__ counter) {
    __shared__ SharedTables tb;
    load_tables(tb, ix);
    __syncthreads();
    const unsigned long long t = (unsigned long long)blockIdx.x * (kThreads / G) + threadIdx.x / G;
    if (t >= count * sigma) return;                        // group-uniform
    const DictItem p = parents[t / sigma];
    const uint32_t code = (uint32_t)(t % sigma);
    uint32_t sp = p.sp, ep = p.ep, touched = 0;
    backward_step<G, LAYOUT, false>(ix, tb, (uint32_t)sym[code], sp, ep, touched);
    const bool keepit = (threadIdx.x % G) == 0 && sp < ep && ep - sp > min_rows;
    const uint32_t act = __activemask(), votes = __ballot_sync(act, keepit);
    unsigned long long wbase = 0;
    if (votes) {
        const int leader = __ffs(votes) - 1, wl = threadIdx.x & 31;
        if (wl == leader) wbase = atomicAdd(counter, (unsigned long long)__popc(votes));
        wbase = __shfl_sync(act, wbase, leader);
    }
    if (votes) {                                           // counter[1] += rows covered by the kept children (is the level worth having?)
        const uint32_t rows = __reduce_add_sync(act, keepit ? ep - sp : 0u);
        if ((int)(threadIdx.x & 31) == __ffs(votes) - 1) atomicAdd(counter + 1, (unsigned long long)rows);
    }
    if (keepit) {
        const unsigned long long slot = wbase + __popc(votes & ((1u << (threadIdx.x & 31)) - 1u));
        unsigned long long key;
        if (d <= D) key = (p.key & ((1ull << 60) - 1ull)) | ((unsigned long long)code << (bits * (uint32_t)(d - 1))) | ((unsigned long long)(d - 1) << 60);
        else {                                             // chain entry: tier t, j-th symbol past the tier's parent interval
            const int rel = d - D - 1, t = rel / Jc + 1, j = rel % Jc + 1;
            if (j == 1) key = dict_chain_key(p.sp, 1, t, (unsigned long long)code);
            else key = (p.key & ~(7ull << 32)) | ((unsigned long long)(j - 1) << 32) | ((unsigned long long)code << (38u + bits * (uint32_t)(j - 1)));
        }
        if (slot < cap) out[slot] = DictItem{key, sp, ep};
    }
}

__global__ void dict_insert_kernel(const DictItem *__restrict__ items, unsigned long long count, unsigned long long *__restrict__ table,
                                   unsigned long long buckets, unsigned long long *__restrict__ failed) {
    const unsigned long long t = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= count) return;
    const DictItem it = items[t];
    unsigned long long b = __umul64hi(dict_mix(it.key), buckets);
    for (unsigned long long tries = 0; tries < buckets; ++tries) {
        for (int s = 0; s < 2; ++s) {
            unsigned long long *slot = table + (b * 2 + (unsigned long long)s) * 2;      // 16-byte slots: key, then sp | ep << 32
            if (atomicCAS(slot, 0ull, it.key) == 0ull) { slot[1] = (unsigned long long)it.sp | ((unsigned long long)it.ep << 32); return; }
        }
        if (++b == buckets) b = 0;
    }
    atomicAdd(failed, 1ull);
}

cudaError_t build_dict(const DevIndex &ix, LaunchCfg cfg, const uint8_t *d_sym, uint32_t sigma, int bits, int Dmax, uint32_t min_rows, uint32_t min_rows_top,
                       int64_t max_entries, void **d_table_out, int64_t *buckets_out, int *depth_out, int *depth_x_out, int *jc_out, int64_t *entries_out,
                       cudaStream_t st) {
    *d_table_out = nullptr; *buckets_out = 0; *depth_out = 0; *depth_x_out = 0; *entries_out = 0;
    const int Jc = std::max(1, std::min(8, 22 / bits));
    *jc_out = Jc;
    const int K = ix.kmer_k;
    if (!ix.kmer || K < 1 || sigma < 2 || Dmax <= K || max_entries < 1) return cudaSuccess;
    unsigned long long table_entries = 1;
    for (int j = 0; j < K; ++j) table_entries *= sigma;
    struct Scratch {                                       // stream-ordered scratch, released on every way out
        void *p = nullptr; cudaStream_t st;
        explicit Scratch(cudaStream_t s) : st(s) {}
        ~Scratch() { if (p) cudaFreeAsync(p, st); }
    } cnt_mem(st), items_mem(st);
    unsigned long long *d_cnt = nullptr, h_cnt = 0;
    CK(cudaMallocAsync(&cnt_mem.p, 16, st));
    d_cnt = (unsigned long long *)cnt_mem.p;
    CK(cudaMemsetAsync(d_cnt, 0, 16, st));
    // the seeds: wide entries of the dense table (disjoint intervals, so at most n / (min_rows + 1)); counted first — a text without any
    // (uniform symbols under a deep table) gets no dictionary and costs no scratch
    if ((table_entries + 255) / 256 > 0x7FFFFFFFull) return cudaSuccess;
    dict_seed_kernel<<<(unsigned)((table_entries + 255) / 256), 256, 0, st>>>(ix.kmer, table_entries, sigma, K, (uint32_t)bits, min_rows, nullptr, 0, d_cnt);
    CK(cudaMemcpyAsync(&h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const unsigned long long seeds = h_cnt;
    if (seeds == 0) return cudaSuccess;
    const unsigned long long cap = seeds + (unsigned long long)max_entries;
    CK(cudaMallocAsync(&items_mem.p, cap * sizeof(DictItem), st));
    DictItem *items = (DictItem *)items_mem.p;
    CK(cudaMemsetAsync(d_cnt, 0, 16, st));
    dict_seed_kernel<<<(unsigned)((table_entries + 255) / 256), 256, 0, st>>>(ix.kmer, table_entries, sigma, K, (uint32_t)bits, min_rows, items, cap, d_cnt);
    unsigned long long lvl_begin = 0, lvl_count = seeds, total = seeds;
    int D = K;
    const int G = (cfg.lanes == 1 || cfg.lanes == 2 || cfg.lanes == 4) ? cfg.lanes : 2;
    for (int d = K + 1; d <= Dmax + kDictMaxTiers * Jc && lvl_count > 0; ++d) {
        const unsigned long long groups = lvl_count * sigma, per = kThreads / G;
        if ((groups + per - 1) / per > 0x7FFFFFFFull) break;
        const unsigned grid = (unsigned)((groups + per - 1) / per);
        // the deepest level the key can hold is where every pattern of at least that length probes first and nothing is grown from: it may
        // take narrower intervals too (min_rows_top < min_rows) when they fit
        // Chain levels (d > Dmax) keep what row contexts cannot take (more than kCtxMaxRows rows), whatever the threshold of the keyed levels.
        const uint32_t lvl_rows = d > Dmax ? std::max<uint32_t>(min_rows, kCtxMaxRows) : min_rows;
        uint32_t keep = (d == Dmax && min_rows_top < min_rows) ? min_rows_top : lvl_rows;
        for (;;) {
#define CALL(GG, LAY) dict_extend_kernel<GG, LAY><<<grid, kThreads, 0, st>>>(ix, d_sym, sigma, items + lvl_begin, lvl_count, d, Dmax, Jc, (uint32_t)bits, keep, items, cap, d_cnt)
            if (ix.layout == FMX_LAYOUT_PLANES) { if (G == 1) CALL(1, FMX_LAYOUT_PLANES); else if (G == 2) CALL(2, FMX_LAYOUT_PLANES); else CALL(4, FMX_LAYOUT_PLANES); }
            else if (ix.layout == FMX_LAYOUT_WMX) { if (G == 1) CALL(1, FMX_LAYOUT_WMX); else if (G == 2) CALL(2, FMX_LAYOUT_WMX); else CALL(4, FMX_LAYOUT_WMX); }
            else { if (G == 1) CALL(1, FMX_LAYOUT_WM); else if (G == 2) CALL(2, FMX_LAYOUT_WM); else CALL(4, FMX_LAYOUT_WM); }
#undef CALL
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(&h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            const bool fits = h_cnt <= cap && h_cnt - seeds <= (unsigned long long)max_entries;
            if (fits || keep == lvl_rows) break;
            keep = lvl_rows;                                                             // the narrow ones do not fit: the level as all others
            CK(cudaMemcpyAsync(d_cnt, &total, 8, cudaMemcpyHostToDevice, st));
            CK(cudaStreamSynchronize(st));
        }
        if (h_cnt > cap || h_cnt - seeds > (unsigned long long)max_entries) break;      // this level does not fit: the dictionary ends one level up
        if (d == K + 1) {
            // Worth having?  The first level past the table must cover a fair share of the rows: on a uniform text a few k-mers are wide by
            // chance, and a dictionary of those would make every query pay a probe that almost never hits.
            unsigned long long covered = 0;
            CK(cudaMemcpyAsync(&covered, d_cnt + 1, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            if (covered * 16ull < (unsigned long long)ix.n) return cudaSuccess;
        }
        lvl_begin = total;
        lvl_count = h_cnt - total;
        total = h_cnt;
        if (lvl_count > 0) D = d;
    }
    const unsigned long long entries = total - seeds;
    if (entries > 0 && D > K) {
        unsigned long long buckets = (entries + 3ull) & ~3ull;                          // two slots per bucket: half load
        if (buckets < 4) buckets = 4;
        void *table = nullptr;
        cudaError_t e = cudaMalloc(&table, buckets * 32);
        if (e != cudaSuccess) return e;
        CK(cudaMemsetAsync(table, 0, buckets * 32, st));
        CK(cudaMemsetAsync(d_cnt, 0, 16, st));
        dict_insert_kernel<<<(unsigned)((entries + 255) / 256), 256, 0, st>>>(items + seeds, entries, (unsigned long long *)table, buckets, d_cnt);
        CK(cudaMemcpyAsync(&h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (h_cnt != 0) { cudaFree(table); return cudaErrorUnknown; }
        *d_table_out = table; *buckets_out = (int64_t)buckets; *depth_out = std::min(D, Dmax); *depth_x_out = D; *entries_out = (int64_t)entries;
    }
    return cudaGetLastError();
}

// ======================================================================================================
// (c) suffix sorting by prefix doubling -> BWT
// ======================================================================================================
// t = T' without terminator (len bytes, none zero); suffix `len` is the '$' suffix.
__global__ void init_keys_kernel(const uint8_t *__restrict__ t, int64_t len, uint64_t *__restrict__ key, uint32_t *__restrict__ sa) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > len) return;
    uint64_t k = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) k = (k << 8) | (uint64_t)((i + j < len) ? t[i + j] : 0);
    key[i] = k;
    sa[i] = (uint32_t)i;
}
__global__ void head_flags_kernel(const uint64_t *__restrict__ key, int64_t n, uint32_t *__restrict__ head) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    head[j] = (j == 0 || key[j] != key[j - 1]) ? (uint32_t)j : 0u;
}
__global__ void assign_rank_kernel(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ grp, int64_t n, uint32_t *__restrict__ rank,
                                   unsigned long long *n_singleton_breaks) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    rank[sa[j]] = grp[j];
    if (grp[j] != (uint32_t)j) atomicAdd(n_singleton_breaks, 1ull);          // some group has more than one member
}
__global__ void doubled_keys_kernel(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ rank, int64_t n, int64_t h, uint64_t *__restrict__ key) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int64_t i = sa[j];
    const uint64_t lo = (i + h < n) ? (uint64_t)rank[i + h] + 1ull : 0ull;
    key[j] = ((uint64_t)rank[i] << 32) | lo;
}
__global__ void emit_bwt_kernel(const uint8_t *__restrict__ t, const uint32_t *__restrict__ sa, int64_t n, uint8_t *__restrict__ bwt, unsigned long long *eof) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t s = sa[j];
    if (s == 0) { bwt[j] = 0; *eof = (unsigned long long)j; }
    else bwt[j] = t[s - 1];
}
__global__ void histogram_kernel(const uint8_t *__restrict__ t, int64_t len, unsigned long long *__restrict__ counts) {
    __shared__ unsigned int h[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) h[i] = 0;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x) atomicAdd(&h[t[i]], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) if (h[i]) atomicAdd(&counts[i], (unsigned long long)h[i]);
}
__global__ void reverse_kernel(const uint8_t *__restrict__ src, int64_t len, uint8_t *__restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len) dst[i] = src[len - 1 - i];
}
__global__ void fm_iota_kernel(uint32_t *v, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (uint32_t)i;
}

cudaError_t byte_histogram(const uint8_t *d_bytes, int64_t n, int64_t counts_out[256], cudaStream_t st) {
    unsigned long long *d_counts = nullptr, h[256];
    CK(cudaMallocAsync(&d_counts, 256 * 8, st));
    CK(cudaMemsetAsync(d_counts, 0, 256 * 8, st));
    if (n > 0) histogram_kernel<<<148 * 4, 256, 0, st>>>(d_bytes, n, d_counts);
    CK(cudaMemcpyAsync(h, d_counts, 256 * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    cudaFreeAsync(d_counts, st);
    for (int i = 0; i < 256; ++i) counts_out[i] = (int64_t)h[i];
    return cudaGetLastError();
}

cudaError_t reverse_bytes(const uint8_t *d_src, int64_t len, uint8_t *d_dst, cudaStream_t st) {
    if (len > 0) reverse_kernel<<<(unsigned)((len + 255) / 256), 256, 0, st>>>(d_src, len, d_dst);
    return cudaGetLastError();
}

cudaError_t suffix_sort_bwt(const uint8_t *d_t, int64_t len, uint8_t *d_bwt, int64_t *eof_out, int64_t counts_out[256],
                            uint32_t *d_sa_out, int *rounds_out, cudaStream_t st) {
    const int64_t n = len + 1;
    if (n >= (1ll << 32)) return cudaErrorInvalidValue;
    uint64_t *k0, *k1; uint32_t *s0, *s1, *rank, *grp; unsigned long long *d_flag, *d_counts;
    CK(cudaMallocAsync(&k0, n * 8, st)); CK(cudaMallocAsync(&k1, n * 8, st));
    CK(cudaMallocAsync(&s0, n * 4, st)); CK(cudaMallocAsync(&s1, n * 4, st));
    CK(cudaMallocAsync(&rank, n * 4, st));
    grp = reinterpret_cast<uint32_t *>(k0);                  // the group heads live in k0, which is dead between a sort and the next doubled_keys (28 bytes per text byte in all)
    CK(cudaMallocAsync(&d_flag, 16, st)); CK(cudaMallocAsync(&d_counts, 256 * 8, st));
    const unsigned grid = (unsigned)((n + 255) / 256);
    init_keys_kernel<<<grid, 256, 0, st>>>(d_t, len, k0, s0);
    CK(sort_pairs_u64_u32(k0, k1, s0, s1, n, 0, 64, st));
    int64_t h = 8; int rounds = 1;
    for (;;) {
        // k1/s1 hold the sorted (key, suffix) pairs
        head_flags_kernel<<<grid, 256, 0, st>>>(k1, n, grp);
        CK(inclusive_max_u32(grp, grp, n, st));
        CK(cudaMemsetAsync(d_flag, 0, 16, st));
        assign_rank_kernel<<<grid, 256, 0, st>>>(s1, grp, n, rank, d_flag);
        unsigned long long dup = 0;
        CK(cudaMemcpyAsync(&dup, d_flag, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (dup == 0 || h >= n) break;
        doubled_keys_kernel<<<grid, 256, 0, st>>>(s1, rank, n, h, k0);
        CK(sort_pairs_u64_u32(k0, k1, s1, s0, n, 0, 64, st));
        uint32_t *t = s0; s0 = s1; s1 = t;
        h *= 2; ++rounds;
    }
    CK(cudaMemsetAsync(d_flag, 0, 16, st));
    emit_bwt_kernel<<<grid, 256, 0, st>>>(d_t, s1, n, d_bwt, d_flag);
    CK(cudaMemsetAsync(d_counts, 0, 256 * 8, st));
    if (len > 0) histogram_kernel<<<148 * 4, 256, 0, st>>>(d_t, len, d_counts);
    unsigned long long eof = 0, cnt[256];
    CK(cudaMemcpyAsync(&eof, d_flag, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(cnt, d_counts, 256 * 8, cudaMemcpyDeviceToHost, st));
    if (d_sa_out) CK(cudaMemcpyAsync(d_sa_out, s1, n * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaStreamSynchronize(st));
    *eof_out = (int64_t)eof;
    for (int i = 0; i < 256; ++i) counts_out[i] = (int64_t)cnt[i];
    if (rounds_out) *rounds_out = rounds;
    cudaFreeAsync(k0, st); cudaFreeAsync(k1, st); cudaFreeAsync(s0, st); cudaFreeAsync(s1, st);
    cudaFreeAsync(rank, st); cudaFreeAsync(d_flag, st); cudaFreeAsync(d_counts, st);
    return cudaGetLastError();
}

// FMCreator.create (bwtmerger.scala:452-532): fm = stable counting sort of rows by BWT byte (eof row -> 0)
cudaError_t build_fm_array(const uint8_t *d_bwt, int64_t n, uint32_t *d_fm, cudaStream_t st) {
    uint8_t *kout; uint32_t *iota;
    CK(cudaMallocAsync(&kout, n, st));
    CK(cudaMallocAsync(&iota, n * 4, st));
    fm_iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(iota, n);
    CK(sort_pairs_u8_u32(d_bwt, kout, iota, d_fm, n, st));
    cudaFreeAsync(kout, st); cudaFreeAsync(iota, st);
    return cudaGetLastError();
}

}  // namespace fmx

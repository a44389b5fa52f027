// GpuFMSearcher.hpp — header-only C++ mirror of the reference's operator interface over the libfmgpu C ABI.
//
// The reference is compiled (Scala/JVM) code whose toolchain is absent from this image, so the host side above the
// C ABI is written in C++: same member names, argument meaning and error behaviour as
//   trait SuffixAlgo / SuffixWalkingAlgo   src/main/scala/org/fmindex/findex.scala:9-57
//   class NaiveFMSearcher                  src/main/scala/org/fmindex/bwtmerger.scala:335-421
//   ReTree(post).matchSA(sa)               src/main/scala/org/fmindex/re2/retree.scala:156, 570
//   case class SAResult(sa,len,sp,ep)      src/main/scala/org/fmindex/re2/re2.scala:9-19
// Scala exceptions become std::runtime_error (MatchError -> fmx::MatchError).  Link with -lfmgpu.
#pragma once
#include <cstdint>
#include <optional>
#include <stdexcept>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "fmgpu.h"

namespace fmx {

struct MatchError : std::runtime_error { using std::runtime_error::runtime_error; };

inline void check(int rc) {
    if (rc == FMX_OK) return;
    if (rc == FMX_E_UNSUPPORTED) throw MatchError(fmx_last_error());
    throw std::runtime_error(fmx_last_error());
}

class GpuFMSearcher;

struct SAResult {                       // re2.scala:9-19
    const GpuFMSearcher *sa;
    int len;
    int64_t sp, ep;
    int64_t cnt() const { return ep - sp; }
    std::string toString() const;
    bool operator==(const SAResult &o) const { return len == o.len && sp == o.sp && ep == o.ep; }
};

class GpuFMSearcher {                   // new NaiveFMSearcher(filename, bigEndian)
public:
    explicit GpuFMSearcher(const std::string &filename, bool bigEndian = true, const fmx_opts *opts = nullptr) {
        check(fmx_open(filename.c_str(), bigEndian ? 1 : 0, opts, &h_));
        n = fmx_n(h_);
        eof = fmx_eof(h_);
        check(fmx_ctable(h_, C_));
    }
    ~GpuFMSearcher() { fmx_close(h_); }
    GpuFMSearcher(const GpuFMSearcher &) = delete;
    GpuFMSearcher &operator=(const GpuFMSearcher &) = delete;

    int64_t n = 0, eof = 0;
    fmx_index *handle() const { return h_; }

    // ---- SuffixAlgo
    int64_t cf(int c) const { return C_[c]; }
    int64_t occ(int c, int64_t i) const {
        uint8_t cc = (uint8_t)c; int64_t out = 0;
        check(fmx_occ_batch(h_, &cc, &i, 1, &out));
        return out;
    }
    std::optional<std::pair<int64_t, int64_t>> search(const std::string &in) const {
        int64_t off[2] = {0, (int64_t)in.size()}, sp = 0, ep = 0;
        check(fmx_count_batch(h_, reinterpret_cast<const uint8_t *>(in.data()), off, 1, &sp, &ep));
        if (sp < ep) return std::make_pair(sp, ep);
        return std::nullopt;
    }
    std::optional<std::pair<int64_t, int64_t>> getPrevRange(int64_t sp, int64_t ep, int c) const {
        uint8_t cc = (uint8_t)c; int64_t a = 0, b = 0;
        check(fmx_prev_range_batch(h_, &sp, &ep, &cc, 1, &a, &b));
        if (a < b) return std::make_pair(a, b);
        return std::nullopt;
    }
    std::vector<std::pair<int64_t, int64_t>> getIntervalPrevRange(int64_t sp, int64_t ep, int cstart, int cend) const {
        const int k = cend - cstart + 1 > 0 ? cend - cstart + 1 : 1;
        std::vector<int32_t> oc(k); std::vector<int64_t> a(k), b(k); int64_t m = 0;
        check(fmx_interval_prev_range(h_, sp, ep, cstart, cend, oc.data(), a.data(), b.data(), &m));
        std::vector<std::pair<int64_t, int64_t>> r;
        for (int64_t i = 0; i < m; ++i) r.emplace_back(a[i], b[i]);
        return r;
    }
    // ---- SuffixWalkingAlgo + NaiveFMSearcher extras
    int64_t getPrevI(int64_t i) const { int64_t o = 0; check(fmx_get_prev_i_batch(h_, &i, 1, &o)); return o; }
    int64_t getNextI(int64_t i) const { int64_t o = 0; check(fmx_get_next_i_batch(h_, &i, 1, &o)); return o; }
    int pos2char(int64_t key) const { int32_t c = 0; check(fmx_pos2char(h_, key, &c)); return c; }
    std::string prevSubstr(int64_t sp, int len) const {
        std::string out((size_t)(len > 0 ? len : 1), '\0'); int32_t ol = 0;
        check(fmx_prev_substr_batch(h_, &sp, 1, len, reinterpret_cast<uint8_t *>(&out[0]), &ol));
        out.resize((size_t)ol);
        return out;
    }
    // file bytes F[off .. off+len) (0x00 dropped; shorter at the text's end): needs fmx_opts.text_sample_rate or FMX_ACCEL_TEXT
    std::string text(int64_t off, int len) const { return textBatch({off}, len)[0]; }
    std::vector<std::string> textBatch(const std::vector<int64_t> &off, int len) const {
        std::vector<uint8_t> out(off.size() * (size_t)(len > 0 ? len : 0) + 1);
        std::vector<int32_t> ol(off.size() + 1);
        check(fmx_text_batch(h_, off.data(), (int64_t)off.size(), len, out.data(), ol.data()));
        std::vector<std::string> r;
        for (size_t i = 0; i < off.size(); ++i) r.emplace_back(reinterpret_cast<const char *>(out.data()) + i * (size_t)len, (size_t)ol[i]);
        return r;
    }
    // longest matches (index opened with fmx_opts.lcp = 1) of a query in file order: for every position j the length of the longest
    // match ending there and the interval of its reverse ((0, n) for length 0); the SMEMs of at least min_len bytes in increasing start order
    struct MatchStats { std::vector<int32_t> len; std::vector<int64_t> sp, ep; };
    MatchStats matchStats(const std::string &q) const {
        MatchStats r;
        r.len.resize(q.size()); r.sp.resize(q.size()); r.ep.resize(q.size());
        const int64_t off[2] = {0, (int64_t)q.size()};
        check(fmx_match_stats_batch(h_, reinterpret_cast<const uint8_t *>(q.data()), off, 1, r.len.data(), r.sp.data(), r.ep.data()));
        return r;
    }
    struct Smem { int32_t start, len; int64_t sp, ep; };
    std::vector<Smem> smems(const std::string &q, int32_t min_len = 1) const {
        const int64_t off[2] = {0, (int64_t)q.size()};
        int64_t oo[2] = {0, 0};
        const int64_t cap = (int64_t)q.size() + 1;                 // at most one SMEM ends at each position
        std::vector<int32_t> st((size_t)cap), ln((size_t)cap);
        std::vector<int64_t> sp((size_t)cap), ep((size_t)cap);
        check(fmx_smem_batch(h_, reinterpret_cast<const uint8_t *>(q.data()), off, 1, min_len, cap, oo, st.data(), ln.data(), sp.data(), ep.data()));
        std::vector<Smem> r;
        for (int64_t k = 0; k < oo[1]; ++k) r.push_back({st[(size_t)k], ln[(size_t)k], sp[(size_t)k], ep[(size_t)k]});
        return r;
    }
    // k-mer census (index opened with fmx_opts.lcp = 1): hist[b] = distinct k-mers occurring b+1 times (the last bucket: >= buckets
    // times); the intervals of the k-mers with min_count <= count <= max_count (0 = no bound) in row order, count = ep - sp
    struct KmerSpectrum { std::vector<int64_t> hist; int64_t distinct = 0, maxOcc = 0; };
    KmerSpectrum kmerSpectrum(int32_t k, int32_t buckets) const {
        KmerSpectrum r;
        r.hist.resize((size_t)(buckets > 0 ? buckets : 1));
        check(fmx_kmer_spectrum(h_, k, buckets, r.hist.data(), &r.distinct, &r.maxOcc));
        r.hist.resize((size_t)buckets);
        return r;
    }
    struct Kmers { std::vector<int64_t> sp, ep; };
    Kmers kmers(int32_t k, int64_t minCount = 1, int64_t maxCount = 0) const {
        Kmers r;
        int64_t total = 0;
        const int rc = fmx_kmer_list_batch(h_, k, minCount, maxCount, 0, &total, nullptr, nullptr);
        if (rc != FMX_E_CAPACITY) { check(rc); return r; }        // FMX_OK here: nothing to list
        r.sp.resize((size_t)total); r.ep.resize((size_t)total);
        check(fmx_kmer_list_batch(h_, k, minCount, maxCount, total, &total, r.sp.data(), r.ep.data()));
        return r;
    }
    std::string nextSubstr(int64_t sp, int len) const {
        std::string out((size_t)(len > 0 ? len : 1), '\0'); int32_t ol = 0;
        check(fmx_next_substr_batch(h_, &sp, 1, len, reinterpret_cast<uint8_t *>(&out[0]), &ol));
        out.resize((size_t)ol);
        return out;
    }
    // ---- batched
    void searchBatch(const std::vector<std::string> &pats, std::vector<int64_t> &sp, std::vector<int64_t> &ep) const {
        std::vector<int64_t> off(pats.size() + 1, 0);
        std::string flat;
        for (size_t i = 0; i < pats.size(); ++i) { flat += pats[i]; off[i + 1] = (int64_t)flat.size(); }
        sp.assign(pats.size(), 0); ep.assign(pats.size(), 0);
        check(fmx_count_batch(h_, reinterpret_cast<const uint8_t *>(flat.data()), off.data(), (int64_t)pats.size(), sp.data(), ep.data()));
    }
    // m patterns of `len` bytes back to back; (sp, ep) as the reference's Int rows (fmx_count_fixed_i32; None = (0, 0))
    void searchFixed(const uint8_t *pat, int32_t len, int64_t m, std::vector<int32_t> &sp, std::vector<int32_t> &ep) const {
        sp.assign((size_t)m, 0); ep.assign((size_t)m, 0);
        check(fmx_count_fixed_i32(h_, pat, len, m, sp.data(), ep.data()));
    }
    std::vector<int64_t> locate(int64_t sp, int64_t ep) const {
        std::vector<int64_t> pos((size_t)(ep > sp ? ep - sp : 1)); int64_t off[2];
        check(fmx_locate_batch(h_, &sp, &ep, 1, ep > sp ? ep - sp : 0, off, pos.data()));
        pos.resize((size_t)off[1]);
        return pos;
    }

private:
    fmx_index *h_ = nullptr;
    int64_t C_[256];
};

inline std::string SAResult::toString() const {
    if (cnt() == 1) return sa->nextSubstr(sp, len);
    if (cnt() > 0) return "[" + std::to_string(cnt()) + " Results] " + sa->nextSubstr(sp, len);
    return "[no results]";
}

class ReTree {                          // ReTree(REParser.re2post(str, lineOnly)); engine 1 = REParser.createNFA(re2post(str))
public:
    explicit ReTree(fmx_regex *adopted) : h_(adopted) {}
    explicit ReTree(const std::string &re, bool lineOnly = false, int engine = FMX_ENGINE_GLUSHKOV) {
        check(fmx_regex_compile_engine(reinterpret_cast<const uint8_t *>(re.data()), (int64_t)re.size(), lineOnly ? 1 : 0, engine, &h_));
    }
    ~ReTree() { fmx_regex_free(h_); }
    ReTree(const ReTree &) = delete;
    ReTree &operator=(const ReTree &) = delete;

    // matchSA(sa, maxBranching = Int.MaxValue, maxIterations = 0): sorted by (len, sp, ep)
    std::vector<SAResult> matchSA(const GpuFMSearcher &sa) const {
        int64_t cap = 1 << 12, off[2] = {0, 0};
        std::vector<int32_t> len; std::vector<int64_t> sp, ep;
        for (;;) {
            len.assign((size_t)cap, 0); sp.assign((size_t)cap, 0); ep.assign((size_t)cap, 0);
            fmx_regex *one[1] = {h_};
            int rc = fmx_regex_search_batch(sa.handle(), one, 1, cap, off, len.data(), sp.data(), ep.data());
            if (rc == FMX_E_CAPACITY) { cap = off[1]; continue; }
            check(rc);
            break;
        }
        std::vector<SAResult> r;
        for (int64_t i = 0; i < off[1]; ++i) r.push_back(SAResult{&sa, len[(size_t)i], sp[(size_t)i], ep[(size_t)i]});
        return r;
    }

    fmx_regex *handle() const { return h_; }

private:
    fmx_regex *h_ = nullptr;
};

// REParser.matchSA(REParser.createNFA(REParser.re2post(re)), sa)  — re2.scala:264-334, 568-693, uncapped
struct ThompsonNFA : ReTree {
    explicit ThompsonNFA(const std::string &re, bool lineOnly = false) : ReTree(re, lineOnly, FMX_ENGINE_THOMPSON) {}
};

// DFA engine (dfa.scala): states are added with addState(kind) and linked with link(from, to, chr) in the order the reference's
// s.link(...) calls were made; build() = DFA.processLinkList(start): numbering, moves, compileBuckets.  matchSA = DFA.matchSA, cap off.
class DFABuilder {
public:
    enum Kind { Start = 0, Plain = 1, Finish = 2 };        // StartState / State / FinishState  (dfa.scala:325-336)
    int addState(Kind k) { kind_.push_back((uint8_t)k); links_.emplace_back(); return (int)kind_.size() - 1; }
    void link(int from, int to, int chr) { links_[(size_t)from].insert(links_[(size_t)from].begin(), {to, chr}); }    // link() prepends (:299)
    struct DFA : ReTree {
        using ReTree::ReTree;
        std::string buckets(int state) const {             // buckets(state).mkString(",")
            int64_t need = 0;
            fmx_dfa_buckets(handle(), state, nullptr, 0, &need);
            std::string s((size_t)(need > 0 ? need : 1), '\0');
            check(fmx_dfa_buckets(handle(), state, &s[0], (int64_t)s.size(), nullptr));
            s.resize(std::char_traits<char>::length(s.c_str()));
            return s;
        }
        bool matchString(const std::string &w) const {
            int32_t m = 0;
            check(fmx_dfa_match_string(handle(), reinterpret_cast<const uint8_t *>(w.data()), (int64_t)w.size(), &m));
            return m != 0;
        }
    };
    std::unique_ptr<DFA> build() const {
        std::vector<int32_t> off(kind_.size() + 1, 0), to, chr;
        for (size_t i = 0; i < kind_.size(); ++i) {
            for (const auto &l : links_[i]) { to.push_back(l.first); chr.push_back(l.second); }
            off[i + 1] = (int32_t)to.size();
        }
        if (to.empty()) { to.push_back(0); chr.push_back(0); }
        fmx_regex *h = nullptr;
        check(fmx_dfa_create((int32_t)kind_.size(), kind_.data(), off.data(), to.data(), chr.data(), &h));
        return std::unique_ptr<DFA>(new DFA(h));
    }

private:
    std::vector<uint8_t> kind_;
    std::vector<std::vector<std::pair<int, int>>> links_;
};

}  // namespace fmx

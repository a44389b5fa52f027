"""
k-mer census on the GPU (fmx_kmer_spectrum / fmx_kmer_list_batch / fmx_kmer_list_dev; index opened with lcp=1).  The reference is
computed from the file, never from the GPU's LCP: the distinct k-mers and their counts by brute force over the windows of F, their
intervals by the oracle's backward search of the reversed k-mers, or, for alphabets of <= 4 symbols, by kmer_intervals() (a histogram of
k-mer codes, no suffix sorting).  The tier past 2^31 rows (FMX_LARGE_ROWS=0 switches it off) builds its own seeded DNA index.
"""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from findex_b200 import fmindex as fx
from oracle import fm_oracle as fo
from test_gpu_large_rows import kmer_intervals
from test_match_model import _texts, _words

pytestmark = pytest.mark.gpu
MODE = os.environ.get("FMX_LARGE_ROWS", "1")
TWO31 = 1 << 31
ACGT = np.frombuffer(b"ACGT", np.uint8)
LISTINGS = [(1, 0), (1, 1), (2, 0), (3, 5), (100, 0)]


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU; the product has no CPU path"
    from findex_b200 import build
    build.build()


def _open(F, **kw):
    bwt, eof, cnt = fx.build_bwt(F)
    return fx.GpuFMSearcher(bwt=bwt, eof=eof, counts=cnt, **kw)


def _ks(L):
    """the k of the model texts, |F| = L"""
    return sorted({k for k in (1, 2, 3, 5, 8, 16, 31, 64, 254, 255, 256, 300, 1000, 2999, 3000, 3001, L - 1, L, L + 1) if k >= 1})


def _kmers(Fz, k):
    """brute force: the distinct k-mers of Fz, reversed (uint8[D, k], in row order: sorted by reverse(K)) and their counts"""
    a = np.frombuffer(Fz, np.uint8)
    if k > len(a):
        return np.zeros((0, k), np.uint8), np.zeros(0, np.int64)
    w = np.lib.stride_tricks.sliding_window_view(a, k)[:, ::-1]
    rev, cnt = np.unique(w, axis=0, return_counts=True)
    return rev, cnt.astype(np.int64)


def _oracle_intervals(o, rev):
    D, k = rev.shape
    if D == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    return o.count_batch(np.ascontiguousarray(rev).reshape(-1), np.arange(0, D * k + 1, k, dtype=np.int64), threads=os.cpu_count())


def _spectrum_want(cnt, buckets):
    return np.bincount(np.minimum(cnt, buckets) - 1, minlength=buckets)[:buckets] if len(cnt) else np.zeros(buckets, np.int64)


def _keep(cnt, mn, mx):
    return (cnt >= mn) & ((cnt <= mx) if mx else True)


def _check_text(g, o, Fz, k):
    rev, cnt = _kmers(Fz, k)
    sp, ep = _oracle_intervals(o, rev)
    assert np.array_equal(ep - sp, cnt), k                        # the reference agrees with itself
    for buckets in (1, 2, 7, 1000):
        hist, distinct, max_occ = g.kmer_spectrum(k, buckets)
        assert np.array_equal(hist, _spectrum_want(cnt, buckets)), (k, buckets)
        assert distinct == len(cnt) and max_occ == (int(cnt.max()) if len(cnt) else 0), (k, buckets)
    for mn, mx in LISTINGS:
        gs, ge = g.kmers(k, mn, mx)
        keep = _keep(cnt, mn, mx)
        assert np.array_equal(gs, sp[keep]) and np.array_equal(ge, ep[keep]), (k, mn, mx)
    gs, ge = g.kmers(k)
    assert int((ge - gs).sum()) == max(len(Fz) - k + 1, 0), k    # the sum identity
    return sp, ep


@pytest.fixture(scope="module")
def model_texts():
    out = {}
    for name, F in _texts().items():
        Fz = F.replace(b"\0", b"")
        o = fo.OracleIndex.from_text_rev(fo.file_to_text_rev(F))
        want = {}
        for k in _ks(len(Fz)):
            rev, cnt = _kmers(Fz, k)
            want[k] = _oracle_intervals(o, rev)
        out[name] = (F, Fz, o, want)
    yield out
    for _, _, o, _ in out.values():
        o.close()


def test_model_texts(model_texts):
    for name, (F, Fz, o, _) in model_texts.items():
        g = _open(F, lcp=1)
        for k in _ks(len(Fz)):
            _check_text(g, o, Fz, k)
        g.close()


@pytest.mark.parametrize("layout", [fx.LAYOUT_PLANES, fx.LAYOUT_WM, fx.LAYOUT_WMX])
def test_listing_walk_every_layout_and_lane_count(model_texts, layout):
    """min_count = 1 walks k - 1 LF steps from row 0: the only part of the census that reads the rank structure"""
    for name, (F, Fz, o, want) in model_texts.items():
        for lanes in (1, 2, 4):
            g = _open(F, lcp=1, layout=layout, lanes_per_query=lanes, accel=fx.ACCEL_NONE)
            for k, (sp, ep) in want.items():
                gs, ge = g.kmers(k)
                assert np.array_equal(gs, sp) and np.array_equal(ge, ep), (name, layout, lanes, k)
            g.close()


def _edge_texts():
    rng = np.random.default_rng(3)
    t = {"1": b"a", "2": b"ab", "3": b"abc", "aa": b"aa", "aaa": b"aaa", "n40": rng.integers(1, 4, 40, dtype=np.uint8).tobytes()}
    for j in (1, 3, 300):
        for d in (-1, 0, 1):                                      # n = |F| + 1 = 64 j + d
            t["n%d" % (64 * j + d)] = rng.integers(97, 101, 64 * j + d - 1, dtype=np.uint8).tobytes()
    t["run"] = b"a" * 100_000                                    # one run across all seven tiles at small k
    t["periodic"] = rng.integers(1, 256, 37, dtype=np.uint8).tobytes() * 3000     # runs of ~3000 rows across tile boundaries
    return t


@pytest.mark.parametrize("name", list(_edge_texts()))
def test_edges(name):
    F = _edge_texts()[name]
    o = fo.OracleIndex.from_text_rev(fo.file_to_text_rev(F))
    g = _open(F, lcp=1)
    L = len(F)
    ks = [1, 2, 3, 5, 64, 300] if L > 5000 else [k for k in _ks(L) if k <= 64]
    for k in sorted(set(ks + [2, 3, 4, L - 1, L, L + 1]) - {0}):
        _check_text(g, o, F, k)
    g.close()
    o.close()


def test_scaled_dna_against_kmer_intervals():
    rng = np.random.default_rng(11)
    F = ACGT[rng.integers(0, 4, 2_000_000)].tobytes()
    g = _open(F, lcp=1)
    tp = np.frombuffer(F, np.uint8)[::-1]
    for k in (1, 2, 5, 8, 10):
        sp, ep = kmer_intervals(tp, ACGT, k)
        hit = ep > sp
        gs, ge = g.kmers(k)
        assert np.array_equal(gs, sp[hit]) and np.array_equal(ge, ep[hit]), k
        cnt = (ep - sp)[hit]
        hist, distinct, max_occ = g.kmer_spectrum(k, int(cnt.max()) + 2)
        assert np.array_equal(hist, _spectrum_want(cnt, int(cnt.max()) + 2)) and distinct == hit.sum() and max_occ == cnt.max(), k
        gs2, ge2 = g.kmers(k, 2)
        assert np.array_equal(gs2, sp[hit & (ep - sp >= 2)]), k
    g.close()


def _words_like(n, seed):
    vocab = [w for w in _words(60_000).split(b"\r\n") if w]
    rng = np.random.default_rng(seed)
    out, size = [], 0
    while size < n:
        w = vocab[int(rng.integers(0, len(vocab)))]
        out.append(w)
        size += len(w) + 1
    return b" ".join(out)[:n]


@pytest.mark.parametrize("kind", ["sigma255", "words"])
def test_scaled_bytes_against_unique_windows(kind):
    rng = np.random.default_rng(12)
    F = rng.integers(1, 256, 2_000_000, dtype=np.uint8).tobytes() if kind == "sigma255" else _words_like(2_000_000, 13)
    g = _open(F, lcp=1)
    for k in ((1, 2, 3, 4, 8) if kind == "sigma255" else (1, 4, 8, 16, 32, 64)):
        rev, cnt = _kmers(F, k)
        hist, distinct, max_occ = g.kmer_spectrum(k, 1000)
        assert np.array_equal(hist, _spectrum_want(cnt, 1000)) and distinct == len(cnt) and max_occ == cnt.max(), k
        for mn in (1, 2):
            gs, ge, txt = g.kmers(k, mn, text=True)
            assert np.array_equal(ge - gs, cnt[cnt >= mn]), (k, mn)
            if len(gs) == 0:
                continue
            assert (ge > gs).all() and (gs[1:] >= ge[:-1]).all()                       # disjoint and increasing
            rk = [x[::-1] for x in txt]                                                   # txt: the k-mers in file order
            cs, ce = g.count_batch(rk)                                                    # count(reverse(K)) == (sp, ep)
            assert np.array_equal(cs, gs) and np.array_equal(ce, ge), (k, mn)
            assert np.array_equal(np.frombuffer(b"".join(rk), np.uint8).reshape(-1, k), rev[cnt >= mn]), (k, mn)
    g.close()


def test_list_dev_chained_into_locate():
    import torch
    rng = np.random.default_rng(4)
    F = ACGT[rng.integers(0, 4, 400_000)].tobytes()
    g = _open(F, lcp=1, sa_sample_rate=8)
    n, k, t = g.n, 9, 3
    hsp, hep = g.kmers(k, t)
    assert len(hsp) > 100
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        cap = len(hsp)
        d_sp = torch.zeros(cap, dtype=torch.int32, device="cuda")
        d_ep = torch.zeros(cap, dtype=torch.int32, device="cuda")
        total = g.kmers_dev(k, d_sp.data_ptr(), d_ep.data_ptr(), cap, min_count=t, stream=st.cuda_stream)
        assert total == cap
        nocc = int((d_ep.to(torch.int64) - d_sp.to(torch.int64)).sum().item())
        d_off = torch.zeros(total + 1, dtype=torch.int64, device="cuda")
        d_pos = torch.zeros(nocc, dtype=torch.int32, device="cuda")
        got = g.locate_dev(d_sp.data_ptr(), d_ep.data_ptr(), total, d_off.data_ptr(), d_pos.data_ptr(), nocc, st.cuda_stream)
    st.synchronize()
    assert got == nocc and nocc >= t * total
    assert np.array_equal(d_sp.cpu().numpy().view(np.uint32), hsp) and np.array_equal(d_ep.cpu().numpy().view(np.uint32), hep)
    off, pos = d_off.cpu().numpy(), d_pos.cpu().numpy().view(np.uint32).astype(np.int64)
    kms = g.next_substr_batch(hsp, k)                            # the k-mers in file order
    for j in range(total):
        ps = pos[off[j]:off[j + 1]]
        assert len(ps) == hep[j] - hsp[j] >= t
        for p in ps:
            f = (n - 1) - int(p) - k
            assert F[f:f + k] == kms[j]
    g.close()


def test_errors_and_capacity():
    import torch
    rng = np.random.default_rng(8)
    F = ACGT[rng.integers(0, 4, 20_000)].tobytes()
    L = fx.lib()
    p = fx._ptr
    tot, d, mx = C.c_int64(), C.c_int64(), C.c_int64()
    h = np.zeros(4, np.int64)
    plain = _open(F)
    assert L.fmx_kmer_spectrum(plain.h, 3, 4, p(h), C.byref(d), C.byref(mx)) == fx.FMX_E_UNSUPPORTED
    assert L.fmx_kmer_list_batch(plain.h, 3, 1, 0, 0, C.byref(tot), None, None) == fx.FMX_E_UNSUPPORTED
    assert L.fmx_kmer_list_dev(plain.h, 3, 1, 0, None, None, 0, C.byref(tot), None) == fx.FMX_E_UNSUPPORTED
    with pytest.raises(fx.ReUnsupported):
        plain.kmer_spectrum(3, 4)
    plain.close()
    g = _open(F, lcp=1)
    sp, ep = np.zeros(4, np.int64), np.zeros(4, np.int64)
    for k, b in ((0, 4), (3, 0), (-1, 4)):
        assert L.fmx_kmer_spectrum(g.h, k, b, p(h), C.byref(d), C.byref(mx)) == fx.FMX_E_ARG
    assert L.fmx_kmer_spectrum(g.h, 3, 4, None, C.byref(d), C.byref(mx)) == fx.FMX_E_ARG
    assert L.fmx_kmer_spectrum(g.h, 3, 4, p(h), None, C.byref(mx)) == fx.FMX_E_ARG
    assert L.fmx_kmer_spectrum(g.h, 3, 4, p(h), C.byref(d), None) == fx.FMX_E_ARG
    for k, mn, mxc in ((0, 1, 0), (3, 0, 0), (3, 1, -1), (3, 3, 2), (3, -5, 0)):
        assert L.fmx_kmer_list_batch(g.h, k, mn, mxc, 4, C.byref(tot), p(sp), p(ep)) == fx.FMX_E_ARG, (k, mn, mxc)
        assert L.fmx_kmer_list_dev(g.h, k, mn, mxc, None, None, 0, C.byref(tot), None) == fx.FMX_E_ARG, (k, mn, mxc)
    assert L.fmx_kmer_list_batch(g.h, 3, 1, 0, 4, C.byref(tot), None, p(ep)) == fx.FMX_E_ARG
    assert L.fmx_kmer_list_batch(g.h, 3, 1, 0, 4, None, p(sp), p(ep)) == fx.FMX_E_ARG
    assert L.fmx_kmer_list_batch(g.h, 3, 1, 0, -1, C.byref(tot), p(sp), p(ep)) == fx.FMX_E_ARG
    assert L.fmx_kmer_list_dev(g.h, 3, 1, 0, None, None, 4, C.byref(tot), None) == fx.FMX_E_ARG
    assert L.fmx_kmer_list_dev(g.h, 3, 1, 0, None, None, 0, None, None) == fx.FMX_E_ARG
    with pytest.raises(fx.FmxError) as e:
        g.kmers(3, 0)
    assert e.value.code == fx.FMX_E_ARG
    # capacity: the required total, and nothing written
    want_sp, want_ep = g.kmers(5, 2)
    T = len(want_sp)
    assert T > 10
    gs, ge = np.full(T + 5, -7, np.int64), np.full(T + 5, -7, np.int64)
    assert L.fmx_kmer_list_batch(g.h, 5, 2, 0, T - 1, C.byref(tot), p(gs), p(ge)) == fx.FMX_E_CAPACITY and tot.value == T
    assert (gs == -7).all() and (ge == -7).all()
    assert L.fmx_kmer_list_batch(g.h, 5, 2, 0, T, C.byref(tot), p(gs), p(ge)) == fx.FMX_OK and tot.value == T
    assert np.array_equal(gs[:T], want_sp) and np.array_equal(ge[:T], want_ep) and (gs[T:] == -7).all() and (ge[T:] == -7).all()
    dsp = torch.full((T + 5,), -7, dtype=torch.int32, device="cuda")
    dep = torch.full((T + 5,), -7, dtype=torch.int32, device="cuda")
    with pytest.raises(fx.FmxError) as e:
        g.kmers_dev(5, dsp.data_ptr(), dep.data_ptr(), T - 1, min_count=2)
    assert e.value.code == fx.FMX_E_CAPACITY
    torch.cuda.synchronize()
    assert (dsp == -7).all() and (dep == -7).all()
    assert g.kmers_dev(5, dsp.data_ptr(), dep.data_ptr(), T, min_count=2) == T
    torch.cuda.synchronize()
    assert np.array_equal(dsp[:T].cpu().numpy(), want_sp) and (dsp[T:] == -7).all().item() and (dep[T:] == -7).all().item()
    # k > |F|: empty, FMX_OK
    n1 = g.n - 1
    for k in (n1 + 1, n1 + 1000):
        hist, distinct, max_occ = g.kmer_spectrum(k, 3)
        assert hist.tolist() == [0, 0, 0] and distinct == 0 and max_occ == 0
        assert len(g.kmers(k)[0]) == 0 and g.kmers_dev(k, 0, 0, 0) == 0
    g.close()


def test_top_kmers():
    rng = np.random.default_rng(17)
    F = _words_like(300_000, 5)
    g = _open(F, lcp=1)
    for k in (1, 3, 6):
        o = fo.OracleIndex.from_text_rev(fo.file_to_text_rev(F))
        rev, cnt = _kmers(F, k)
        sp, ep = _oracle_intervals(o, rev)
        o.close()
        order = np.lexsort((sp, -cnt))
        for t in (1, 5, 50, 333, len(cnt), len(cnt) + 3):
            gs, ge = g.top_kmers(k, t)
            assert np.array_equal(gs, sp[order][:t]) and np.array_equal(ge, ep[order][:t]), (k, t)
    F2 = rng.integers(1, 256, 50_000, dtype=np.uint8).tobytes()   # counts of 1 and 2 only: ties everywhere
    g2 = _open(F2, lcp=1)
    rev, cnt = _kmers(F2, 2)
    sp, ep = g2.kmers(2)
    order = np.lexsort((sp, -(ep - sp)))
    for t in (1, 10, 1000):
        gs, ge = g2.top_kmers(2, t)
        assert np.array_equal(gs, sp[order][:t]), t
    g2.close()
    g.close()


def test_concurrent_host_threads():
    rng = np.random.default_rng(31)
    F = ACGT[rng.integers(0, 4, 300_000)].tobytes()
    g = _open(F, lcp=1)
    ks = (4, 7, 9, 12)
    pats = [[ACGT[rng.integers(0, 4, 14)].tobytes() for _ in range(2000)] for _ in ks]
    want = [(g.kmer_spectrum(k, 50), g.kmers(k), g.kmers(k, 2, 9), g.count_batch(pats[i])) for i, k in enumerate(ks)]
    errors = []

    def work(i):
        try:
            k = ks[i]
            for _ in range(5):
                h, d, m = g.kmer_spectrum(k, 50)
                assert np.array_equal(h, want[i][0][0]) and (d, m) == want[i][0][1:]
                assert all(np.array_equal(x, y) for x, y in zip(g.kmers(k), want[i][1]))
                assert all(np.array_equal(x, y) for x, y in zip(g.kmers(k, 2, 9), want[i][2]))
                assert all(np.array_equal(x, y) for x, y in zip(g.count_batch(pats[i]), want[i][3]))
        except Exception as e:                               # noqa: BLE001 — reported below
            errors.append(e)
    th = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    g.close()
    assert not errors, errors


def test_past_2_31_rows():
    if MODE == "0":
        pytest.skip("FMX_LARGE_ROWS=0: the tier past 2^31 rows is switched off")
    L = 2_200_000_000
    lut = np.frombuffer(b"AAACCCGGGT", np.uint8)
    rng = np.random.default_rng(29)
    F = np.empty(L, np.uint8)
    for a in range(0, L, 1 << 28):
        F[a:a + (1 << 28)] = lut[rng.integers(0, 10, min(1 << 28, L - a), dtype=np.uint8)]
    g = _open(F, lcp=1, accel=fx.ACCEL_NONE, layout=fx.LAYOUT_WMX)
    assert g.n == L + 1
    sp, ep = kmer_intervals(F[::-1], ACGT, 12)
    hit = ep > sp
    gs, ge = g.kmers(12)
    assert np.array_equal(gs, sp[hit]) and np.array_equal(ge, ep[hit])
    assert ge.max() > TWO31 and gs.min() < TWO31
    cnt = (ep - sp)[hit]
    B = int(cnt.max()) + 1
    hist, distinct, max_occ = g.kmer_spectrum(12, B)
    assert np.array_equal(hist, np.bincount(cnt - 1, minlength=B)[:B]) and distinct == hit.sum() and max_occ == cnt.max()
    s1, e1 = g.kmers(1)
    C_ = [g.cf(c) for c in b"ACGT"] + [g.n]
    assert s1.tolist() == C_[:4] and e1.tolist() == C_[1:]
    g.close()

"""
Indexes of more than 2^31 rows.  The device keeps rows and positions as uint32 and indexes any n < 2^32 - 1; the range [2^31, 2^32) is
where 32-bit code goes wrong (signed/unsigned mix-ups, sign extension, values stored in 32 bits).  One seeded skewed DNA text of
2.4e9 bytes (p = 0.3, 0.3, 0.3, 0.1 over ACGT, so C['T'] > 2^31 too) is indexed once on the GPU and every operator is run in six
configurations, with rows, keys, positions and intervals on both sides of 2^31.

The GPU-built BWT is not trusted on its own word: kmer_intervals() computes the interval of every k-mer from the text alone (a
histogram of k-mer codes, no suffix sorting), and all 4^12 twelve-mers are counted against it.  Those intervals, with the suffixes
shorter than 12, tile [1, n), so every row's first 12 symbols are checked.  Longer patterns and the element-wise operators are then
compared with the CPU oracle loaded from the GPU-built files, and locate is checked by the text (located positions are real
occurrences, ascending and complete), never by the oracle's suffix array.

FMX_LARGE_ROWS=0 switches the GPU tier off; FMX_LARGE_ROWS=max runs configuration 1 on the longest text the builder accepts
(n = 2^32 - 2).  The CPU test of kmer_intervals() against the oracle always runs.
"""
import os

import numpy as np
import pytest

from findex_b200 import fmindex as fx
from findex_b200 import sharded
from oracle import fm_oracle as fo

MODE = os.environ.get("FMX_LARGE_ROWS", "1")
TWO31 = 1 << 31
ACGT = np.frombuffer(b"ACGT", np.uint8)
MASK = 0xFFFFFFFF
DEFAULT_BYTES = 2_400_000_000
MANY = 100                                                      # occurrences of each len-14 locate pattern, at least


# ---- the reference: k-mer intervals from the text ----------------------------------------------------------------------------------
def kmer_intervals(tp, alphabet, k, chunk=1 << 26):
    """(sp, ep) int64[sigma^k] of every k-mer over `alphabet` (sorted byte values; the k-mer with base-sigma code c is entry c), computed
    from T' = `tp` (the indexed text without '$') alone.  (0, 0) where the k-mer does not occur.

    Rows sort as: '$' (row 0), then by suffix.  A k-mer p starts at sp = 1 + #{k-mers of T' < p} + #{suffixes shorter than k, before '$',
    that are <= p's prefix of their length} (such a suffix sorts before p: '$' is the smallest symbol)."""
    tp = np.asarray(tp, np.uint8)
    alphabet = np.asarray(alphabet, np.uint8)
    s, L = len(alphabet), len(tp)
    nb = s ** k
    assert nb <= 1 << 32
    dt = np.uint32
    lut = np.zeros(256, dt)
    lut[alphabet] = np.arange(s, dtype=dt)
    hist = np.zeros(nb, np.int64)
    for a in range(0, L - k + 1, chunk):
        b = min(a + chunk, L - k + 1)                            # k-mers starting in [a, b)
        w = lut[tp[a:b + k - 1]]
        code = np.zeros(b - a, dt)
        for j in range(k):
            code *= dt(s)
            code += w[j:j + b - a]
        hist += np.bincount(code, minlength=nb)
    short = np.zeros(nb, np.int64)                               # suffix T'[i:L] of m < k symbols at the smallest code with that prefix
    for i in range(max(L - k + 1, 0), L):
        c = 0
        for x in lut[tp[i:L]]:
            c = c * s + int(x)
        short[c * s ** (k - (L - i))] += 1
    sp = 1 + np.cumsum(hist) - hist + np.cumsum(short)
    ep = sp + hist
    sp[hist == 0] = 0
    ep[hist == 0] = 0
    return sp, ep


def all_kmers(alphabet, k):
    """every k-mer over `alphabet` in code order: uint8[sigma^k, k]"""
    alphabet = np.asarray(alphabet, np.uint8)
    s = len(alphabet)
    codes = np.arange(s ** k, dtype=np.int64)
    return np.stack([alphabet[(codes // s ** (k - 1 - j)) % s] for j in range(k)], axis=1).copy()


def _oracle_fixed(o, pats):
    ln = pats.shape[1]
    return o.count_batch(pats.reshape(-1), np.arange(0, pats.size + 1, ln, dtype=np.int64), threads=os.cpu_count())


@pytest.mark.parametrize("alphabet", [b"\x01\x02", b"\x07\x28\xc8", b"ACGT"], ids=["sigma2", "sigma3_sparse", "sigma4_dna"])
def test_kmer_reference_matches_oracle(alphabet):
    """kmer_intervals() == the oracle's backward search for every k-mer, k = 1..6, texts of 1..2000 symbols (also shorter than k),
    uniform, skewed and repetitive"""
    alpha = np.frombuffer(alphabet, np.uint8)
    rng = np.random.default_rng(len(alphabet))
    texts = []
    for L in (1, 2, 3, 4, 5, 6, 7, 11, 64, 333, 1000, 2000):
        texts.append(alpha[rng.integers(0, len(alpha), L)])
        if L >= 64:
            texts.append(alpha[np.minimum(rng.geometric(0.6, L) - 1, len(alpha) - 1)])         # skewed
            texts.append(np.resize(alpha[rng.integers(0, len(alpha), 7)], L))                    # period 7
    texts.append(np.full(500, alpha[-1], np.uint8))
    for tp in texts:
        tp = np.ascontiguousarray(tp)
        o = fo.OracleIndex.from_text_rev(tp)
        for k in range(1, 7):
            sp, ep = kmer_intervals(tp, alpha, k, chunk=97)                                      # a chunk that does not divide the text
            osp, oep = o.count_batch(all_kmers(alpha, k).reshape(-1), np.arange(0, k * len(alpha) ** k + 1, k, dtype=np.int64))
            assert np.array_equal(sp, osp) and np.array_equal(ep, oep), (len(tp), k)
        o.close()


# ---- the GPU tier ----------------------------------------------------------------------------------------------------------------
def _dna(L, seed, chunk=1 << 28):
    """T': seeded DNA with p(A, C, G, T) = (0.3, 0.3, 0.3, 0.1)"""
    lut = np.frombuffer(b"AAACCCGGGT", np.uint8)
    rng = np.random.default_rng(seed)
    tp = np.empty(L, np.uint8)
    for a in range(0, L, chunk):
        tp[a:a + chunk] = lut[rng.integers(0, 10, min(chunk, L - a), dtype=np.uint8)]
    return tp


def _take(tp, offs, ln):
    return tp[offs[:, None] + np.arange(ln)[None, :]]


def _offsets(rng, L, ln, m):
    """m offsets of T' windows of ln symbols, half of them at or beyond 2^31"""
    lo = rng.integers(0, L - ln + 1, m - m // 2)
    hi = rng.integers(TWO31, L - ln + 1, m // 2)
    return np.concatenate([lo, hi])


def _windows(points, n, w=64):
    rows = np.unique(np.concatenate([np.arange(p - w, p + w) for p in points]))
    return rows[(rows >= 0) & (rows < n)]


@pytest.fixture(scope="module")
def big(tmp_path_factory):
    if MODE == "0":
        pytest.skip("FMX_LARGE_ROWS=0: the tier past 2^31 rows is switched off")
    import torch
    assert torch.cuda.is_available(), "the tier past 2^31 rows needs a GPU; the product has no CPU path"
    from findex_b200 import build
    build.build()
    L = (1 << 32) - 3 if MODE == "max" else DEFAULT_BYTES
    tp = _dna(L, 31)
    d = tmp_path_factory.mktemp("large_rows")
    base = str(d / "dna")
    fx.build_index_files(tp[::-1], base, bigEndian=True)          # the file holds T' reversed (no 0x00: T' is the file read backwards)
    o = fo.OracleIndex.load(base)
    n = L + 1
    assert o.n == n
    B = {"tp": tp, "L": L, "n": n, "base": base, "o": o, "eof": o.eof}
    B["C"] = {c: o.cf(c) for c in b"ACGT"}
    assert B["C"][ord("T")] > TWO31                              # the C table crosses 2^31 as well
    rng = np.random.default_rng(77)

    # count: all 12-mers against the text-only reference; fixed lengths 16 (the AUTO table's k), 20, 32; count_batch lengths 1..64
    B["k12"] = all_kmers(ACGT, 12)
    B["k12_want"] = kmer_intervals(tp, ACGT, 12)
    hit = B["k12_want"][1] > B["k12_want"][0]
    assert B["k12_want"][0][hit].min() >= 1 and B["k12_want"][1].max() <= n and B["k12_want"][1][hit].max() > TWO31
    fixed = {}
    for ln in (16, 20, 32):
        m = 200_000
        nh = m * 9 // 10
        pats = np.empty((m, ln), np.uint8)
        pats[:nh] = _take(tp, _offsets(rng, L, ln, nh), ln)
        pats[nh:] = ACGT[rng.integers(0, 4, (m - nh, ln))]
        fixed[ln] = (pats, _oracle_fixed(o, pats))
        assert (fixed[ln][1][1][:nh] > fixed[ln][1][0][:nh]).all()
    B["fixed"] = fixed
    var = []
    for ln in range(1, 65):
        var += [bytes(x) for x in _take(tp, _offsets(rng, L, ln, 150), ln)]
        var += [bytes(x) for x in ACGT[rng.integers(0, 4, (10, ln))]]
    voff = np.zeros(len(var) + 1, np.int64)
    np.cumsum([len(x) for x in var], out=voff[1:])
    B["var"] = (var, o.count_batch(np.frombuffer(b"".join(var), np.uint8), voff, threads=os.cpu_count()))

    # element-wise operators: windows around 0, eof, 2^31, every C[c] and n - 1, plus random rows >= 2^31
    C = B["C"]
    rows = np.concatenate([_windows([0, o.eof, TWO31, n - 1] + list(C.values()), n), rng.integers(TWO31, n, 100_000)])
    B["rows"] = rows
    B["occ_want"] = {c: np.array([o.occ(c, int(r)) for r in rows], np.int64) for c in b"ACGT"}
    B["prev_i_want"] = np.array([o.getPrevI(int(r)) for r in rows], np.int64)
    B["next_i_want"] = np.array([o.getNextI(int(r)) for r in rows], np.int64)
    sub = np.concatenate([rows[rows < TWO31 + 64][:4000], rows[-20_000:]])
    B["sub"] = sub
    B["prev_sub_want"] = [o.prevSubstr(int(r), 24) for r in sub]
    B["next_sub_want"] = [o.nextSubstr(int(r), 24) for r in sub]
    keys = _windows([0, o.eof, TWO31, n - 1] + list(C.values()), n, 8)
    B["pos2char"] = (keys, [o.pos2char(int(k)) for k in keys])
    d1 = rng.integers(0, 5000, len(rows))
    d2 = rng.integers(0, 5000, len(rows))
    psp, pep = np.clip(rows - d1, 0, n), np.clip(rows + d2, 0, n)
    straddle = np.array([[TWO31 - 1, TWO31 + 1], [TWO31 - 1000, TWO31 + 1000], [TWO31, TWO31 + 1], [TWO31 - 1, TWO31], [0, n],
                         [C[ord("T")], n], [C[ord("G")], C[ord("T")]], [n - 1, n]], np.int64)
    psp, pep = np.concatenate([straddle[:, 0], psp]), np.concatenate([straddle[:, 1], pep])
    pc = ACGT[rng.integers(0, 4, len(psp))]
    B["prev_range"] = (psp, pep, pc, [o.prev_range_raw(int(a), int(b), int(c)) for a, b, c in zip(psp, pep, pc)])
    B["interval"] = [(int(a), int(b), o.getIntervalPrevRange(int(a), int(b), ord("A"), ord("T"))[0]) for a, b in straddle]

    # locate: unique len-32 windows at known offsets (2^31 +- 1, the text's end, random on both sides) and len-14 patterns of
    # hundreds of occurrences
    s32 = np.concatenate([[0, 1, TWO31 - 1, TWO31, TWO31 + 1], np.arange(L - 40, L - 31), _offsets(rng, L, 32, 4000 - 14)])
    p32 = _take(tp, s32, 32)
    B["u32"] = (s32, p32, _oracle_fixed(o, p32))
    cand = _take(tp, _offsets(rng, L, 14, 40_000), 14)
    csp, cep = _oracle_fixed(o, cand)
    keep = np.flatnonzero((cep - csp >= MANY) & (cep - csp <= 5000))
    _, first = np.unique(cand[keep], axis=0, return_index=True)
    keep = keep[np.sort(first)][:2000]
    assert len(keep) == 2000
    B["r14"] = (cand[keep], (csp[keep], cep[keep]))

    # regex: literal runs, classes, alternations and '.'; some start with T (rows >= C['T'] > 2^31), some with A
    def lit(k, first=None):
        while True:
            s = int(rng.integers(0, L - k))
            if first is None or tp[s] == ord(first):
                return bytes(tp[s:s + k]).decode()
    rxs = []
    for i in range(5):
        rxs.append(lit(6, "T") + "." + lit(5))
        rxs.append(lit(6, "A") + "[CG]" + lit(5, "T"))
        rxs.append("T" + lit(5) + "(" + lit(3) + "|" + lit(3) + ")" + lit(4))
        rxs.append(lit(4, "G") + "[AT]" + lit(3) + "." + lit(4) + "T")
    B["rx"] = (rxs, [o.regex_match(r) for r in rxs])
    sps = [s for w in B["rx"][1] for (_, s, _) in w]
    assert min(sps) < TWO31 <= max(sps)
    yield B
    o.close()
    for ext in (".bwt", ".aux", ".sa", ".lcp", "_resident.sa"):
        if os.path.exists(base + ext):
            os.remove(base + ext)


def _checksum(parts):
    return int(sum(int((sp * 1315423911 + ep * 2654435761).sum()) for sp, ep in parts) & 0xFFFFFFFFFFFF)


def _check_counts(g, B):
    """every count entry point against the reference / the oracle; returns the checksum of the results"""
    import torch
    sp, ep = g.count_fixed(B["k12"])
    assert np.array_equal(sp, B["k12_want"][0]) and np.array_equal(ep, B["k12_want"][1])
    parts = [(sp, ep)]
    for ln, (pats, (osp, oep)) in B["fixed"].items():
        sp, ep = g.count_fixed(pats)
        assert np.array_equal(sp, osp) and np.array_equal(ep, oep), ln
        parts.append((sp, ep))
        assert np.array_equal(g.count_only_fixed(pats).astype(np.int64), oep - osp), ln
    var, (vsp, vep) = B["var"]
    sp, ep = g.count_batch(var)
    assert np.array_equal(sp, vsp) and np.array_equal(ep, vep)
    parts.append((sp, ep))
    pats, (osp, oep) = B["fixed"][20]
    codes = g.pack2(pats)
    for dt in (np.uint32, np.int64):
        psp, pep = np.full(len(pats), 7, dt), np.full(len(pats), 7, dt)
        g.count_packed2_into(codes, 20, psp, pep)
        assert np.array_equal(psp.astype(np.int64), osp) and np.array_equal(pep.astype(np.int64), oep), dt
    # device-resident rows: uint32 in int32 tensors
    pats, (osp, oep) = B["fixed"][16]
    m, ln = pats.shape
    d_pat = torch.from_numpy(pats).cuda()
    d_sp = torch.zeros(m, dtype=torch.int32, device="cuda")
    d_ep = torch.zeros(m, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    g.count_fixed_dev(d_pat.data_ptr(), ln, m, d_sp.data_ptr(), d_ep.data_ptr(), st)
    torch.cuda.synchronize()
    assert np.array_equal(d_sp.cpu().numpy().astype(np.int64) & MASK, osp) and np.array_equal(d_ep.cpu().numpy().astype(np.int64) & MASK, oep)
    world = 3                                                    # fused count + exchange, this GPU playing three ranks
    bufs = [fx.SharedDeviceBuffer(m) for _ in range(world)]
    d_sp.zero_()
    d_ep.zero_()
    for r in range(world):
        lo, hi = sharded.shard_bounds(m, r, world)
        g.count_fixed_dev_gather(d_pat.data_ptr() + lo * ln, ln, hi - lo, d_sp.data_ptr() + lo * 4, d_ep.data_ptr() + lo * 4,
                                 [b.ptr for b in bufs], lo, st)
    torch.cuda.synchronize()
    assert np.array_equal(d_sp.cpu().numpy().astype(np.int64) & MASK, osp) and np.array_equal(d_ep.cpu().numpy().astype(np.int64) & MASK, oep)
    for b in bufs:
        assert np.array_equal(b.to_host().astype(np.int64), oep - osp)
        b.close()
    blocks, steps = g.count_fixed_stats(pats[:20_000])
    assert blocks > 0 and steps >= 0
    with pytest.raises(fx.FmxError) as e:                        # the reference's Int rows cannot hold these rows
        g.count_fixed_into(pats[:100].copy(), np.zeros(100, np.int32), np.zeros(100, np.int32))
    assert e.value.code == fx.FMX_E_UNSUPPORTED
    return _checksum(parts)


def _check_elementwise(g, B):
    rows = B["rows"]
    for c in b"ACGT":
        assert np.array_equal(g.occ_batch(np.full(len(rows), c, np.uint8), rows), B["occ_want"][c]), chr(c)
    psp, pep, pc, want = B["prev_range"]
    a, b = g.prev_range_batch(psp, pep, pc)
    assert [(int(x), int(y)) for x, y in zip(a, b)] == want
    for s, e, w in B["interval"]:
        assert g.getIntervalPrevRange(s, e, ord("A"), ord("T")) == w, (s, e)
    assert np.array_equal(g.get_prev_i_batch(rows), B["prev_i_want"])
    assert np.array_equal(g.get_next_i_batch(rows), B["next_i_want"])
    keys, want = B["pos2char"]
    assert [g.pos2char(int(k)) for k in keys] == want
    sub = B["sub"]
    assert g.prev_substr_batch(sub, 24) == B["prev_sub_want"]
    assert g.next_substr_batch(sub, 24) == B["next_sub_want"]
    assert g.extract_batch(sub, 24, -1) == B["prev_sub_want"] and g.extract_batch(sub, 24, +1) == B["next_sub_want"]


def _locate_dev(g, sp, ep, cap):
    import torch
    m = len(sp)
    d_sp = torch.from_numpy(sp.astype(np.uint32).view(np.int32)).cuda()
    d_ep = torch.from_numpy(ep.astype(np.uint32).view(np.int32)).cuda()
    d_off = torch.zeros(m + 1, dtype=torch.int64, device="cuda")
    d_pos = torch.zeros(max(cap, 1), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    total = g.locate_dev(d_sp.data_ptr(), d_ep.data_ptr(), m, d_off.data_ptr(), d_pos.data_ptr(), cap, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return d_off.cpu().numpy(), d_pos.cpu().numpy()[:total].astype(np.int64) & MASK


def _locate_exchange(g, pats, want_off, want_pos):
    """the locate exchange with this GPU playing three ranks: every rank's gathered buffer holds the whole batch's positions"""
    import torch
    world, M, ln = 3, len(pats), pats.shape[1]
    total = int(want_off[-1])
    dev = torch.device("cuda", 0)
    ex = [sharded.GpuExchange(g, r, world, M, total + 16, dev, peers=([], []), barrier=lambda: None) for r in range(world)]
    for e in ex:
        e.set_peers([x.counts.ptr for x in ex], [x.values.ptr for x in ex])
    d_pat = torch.from_numpy(pats).cuda()
    bounds = [sharded.shard_bounds(M, r, world) for r in range(world)]
    for r, (lo, hi) in enumerate(bounds):
        ex[r].locate_count(d_pat[lo:hi].contiguous(), ln, lo, hi)
    torch.cuda.synchronize()
    outs = [ex[r].locate_values(lo, hi, total + 16) for r, (lo, hi) in enumerate(bounds)]
    torch.cuda.synchronize()
    for r in range(world):
        assert np.array_equal(outs[r][0].cpu().numpy(), want_off), r
        assert np.array_equal(ex[r].gathered_values(total).cpu().numpy().astype(np.int64) & MASK, want_pos), r
    for e in ex:
        e.close()


def _check_locate(g, B):
    tp, L = B["tp"], B["L"]
    s32, p32, (sp, ep) = B["u32"]
    assert (ep - sp == 1).all()
    off, pos = g.locate_batch(sp, ep)
    assert np.array_equal(off, np.arange(len(sp) + 1)) and np.array_equal(pos, s32)
    doff, dpos = _locate_dev(g, sp, ep, len(sp))
    assert np.array_equal(doff, off) and np.array_equal(dpos, s32)
    _locate_exchange(g, p32, off, s32)
    p14, (sp, ep) = B["r14"]
    off, pos = g.locate_batch(sp, ep)
    assert np.array_equal(np.diff(off), ep - sp)
    q = np.repeat(np.arange(len(sp)), ep - sp)
    assert (pos >= 0).all() and (pos <= L - 14).all()
    assert (np.diff(pos)[np.diff(q) == 0] > 0).all()            # strictly ascending inside each query
    assert (_take(tp, pos, 14) == p14[q]).all()                  # each one a real occurrence: with the count, exactly the occurrences
    assert (pos >= TWO31).any()
    doff, dpos = _locate_dev(g, sp, ep, len(pos))
    assert np.array_equal(doff, off) and np.array_equal(dpos, pos)
    _locate_exchange(g, p14, off, pos)


def _check_regex(g, B):
    import torch
    rxs, want = B["rx"]
    trees = [fx.ReTree(r) for r in rxs]
    assert g.regex_search_batch(trees) == want
    rset = g.regex_set(trees)
    off, ln, sp, ep = rset.search(g)
    cap = int(off[-1]) + 5
    d_res = torch.zeros((cap, 4), dtype=torch.int32, device="cuda")
    d_off = torch.zeros(len(rxs) + 1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    total = rset.search_dev(g, d_res.data_ptr(), cap, d_off.data_ptr())
    torch.cuda.synchronize()
    r = d_res.cpu().numpy().astype(np.int64) & MASK
    flat = np.array([(i, l, s, e) for i, w in enumerate(want) for (l, s, e) in w], np.int64).reshape(-1, 4)
    assert total == len(flat) and np.array_equal(d_off.cpu().numpy(), off) and np.array_equal(r[:total], flat)
    rset.close()


SUMS = {}
CONFIGS = [
    # name, options, FMX_TLB_REACH_GB, locate
    ("auto", {}, None, True),
    ("planes_none_rate32", dict(layout=fx.LAYOUT_PLANES, accel=fx.ACCEL_NONE, sa_sample_rate=32), None, True),
    ("wm_none_1lane", dict(layout=fx.LAYOUT_WM, accel=fx.ACCEL_NONE, lanes_per_query=1), None, False),
    ("wmx_kmer_2lanes", dict(layout=fx.LAYOUT_WMX, accel=fx.ACCEL_KMER, lanes_per_query=2), None, False),
    ("ctx32", dict(accel=fx.ACCEL_CTX | fx.ACCEL_KMER, kmer_table_bytes=1 << 27), "1000", False),
    ("auto_groups", dict(kmer_table_bytes=8 << 32), "1000", False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,opts,reach,locate", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_configuration(big, name, opts, reach, locate, monkeypatch):
    if MODE == "max" and name != "auto":
        pytest.skip("FMX_LARGE_ROWS=max runs configuration 1 (AUTO) only")
    B = big
    monkeypatch.delenv("FMX_KMER_ROWS", raising=False)
    if reach:
        monkeypatch.setenv("FMX_TLB_REACH_GB", reach)
    else:
        monkeypatch.delenv("FMX_TLB_REACH_GB", raising=False)
    g = fx.GpuFMSearcher(B["base"] + ".bwt", **opts)
    info = g.info()
    print("\n%s: %s" % (name, info))
    assert g.n == B["n"] and g.eof == B["eof"] and all(g.cf(c) == v for c, v in B["C"].items())
    if name == "auto":
        assert info["layout"] == "planes" and info["sigma"] == 4 and info["ctx_entry_bytes"] == 8 and info["sa_sample_rate"] == 0, info
        if info["kmer_k"] == 16:
            assert 4 ** 16 == 1 << 32                                # the table holds exactly 2^32 entries
    elif name == "planes_none_rate32":
        assert info["layout"] == "planes" and info["kmer_k"] == 0 and info["ctx_entry_bytes"] == 0 and info["sa_sample_rate"] == 32, info
    elif name == "wm_none_1lane":
        assert info["layout"] == "wm" and info["kmer_k"] == 0 and info["lanes_per_query"] == 1, info
    elif name == "wmx_kmer_2lanes":
        assert info["layout"] == "wmx" and info["kmer_k"] >= 2 and info["lanes_per_query"] == 2, info
    elif name == "ctx32":
        assert info["ctx_entry_bytes"] == 32 and info["kmer_k"] == 12 and info["kmer_rows"] == 0, info
    elif name == "auto_groups":
        assert info["ctx_entry_bytes"] == 32 and info["kmer_k"] == 16 and info["kmer_rows"] == 3, info
    sums = set()
    for lanes in ((1, 2, 4) if name == "auto" else (0,)):
        if lanes:
            g.set_lanes(lanes)
            assert g.info()["lanes_per_query"] == lanes
        sums.add(_check_counts(g, B))
    assert len(sums) == 1
    SUMS[name] = sums.pop()
    _check_elementwise(g, B)
    _check_regex(g, B)
    if locate:
        _check_locate(g, B)
    if name == "auto":                                           # the resident suffix array, written out as unsigned words
        g.write_sa_file(B["base"] + "_resident")
        sa = np.memmap(B["base"] + "_resident.sa", dtype=">u4", mode="r")
        s32, _, (sp, _) = B["u32"]
        assert np.array_equal(sa[sp].astype(np.int64), s32)
        del sa
        os.remove(B["base"] + "_resident.sa")
    g.close()


@pytest.mark.gpu
def test_count_checksums_agree_across_configurations(big):
    want = 1 if MODE == "max" else len(CONFIGS)
    assert len(SUMS) == want and len(set(SUMS.values())) == 1, SUMS


def _lcp(tp, a, b):
    """common prefix of T'[a:] + '$' and T'[b:] + '$'"""
    k = 0
    while True:
        x, y = tp[a + k:a + k + 256], tp[b + k:b + k + 256]
        m = min(len(x), len(y))
        ne = np.flatnonzero(x[:m] != y[:m])
        if len(ne):
            return k + int(ne[0])
        if m < 256:
            return k + m
        k += 256


@pytest.mark.gpu
def test_sa_and_lcp_files(big):
    """write_sa_file (built for the call) and LCPSearcher: getSA / getLCP at rows whose suffixes start at or beyond 2^31"""
    B = big
    tp, base, n = B["tp"], B["base"], B["n"]
    for ext in (".sa", ".lcp"):
        if os.path.exists(base + ext):
            os.remove(base + ext)
    ls = fx.LCPSearcher(base + ".bwt", accel=fx.ACCEL_NONE)
    s32, _, (sp, _) = B["u32"]
    assert (s32 >= TWO31).any()
    for r, s in zip(sp, s32):
        assert ls.getSA(int(r)) == s, (r, s)
    rows = np.unique(np.concatenate([sp[sp < n - 1][:500], _windows([TWO31, n - 2], n - 1, 16)]))
    for r in rows:
        a, b = ls.getSA(int(r)), ls.getSA(int(r) + 1)
        assert ls.getLCP(int(r)) == _lcp(tp, a, b), r
    ls.close()
    for ext in (".sa", ".lcp"):
        os.remove(base + ext)


@pytest.mark.gpu
def test_longest_text_bound(big):
    """2^32 - 3 bytes is the longest text the builder accepts (n = 2^32 - 2); one byte more needs 64-bit rows"""
    if MODE == "max":
        assert big["n"] == (1 << 32) - 2
    text = np.full((1 << 32) - 2, ord("A"), np.uint8)
    with pytest.raises(fx.FmxError) as e:
        fx.build_index_files(text, os.path.join(os.path.dirname(big["base"]), "too_long"))
    assert e.value.code == fx.FMX_E_UNSUPPORTED

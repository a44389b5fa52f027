"""
Matching statistics and SMEMs on the GPU (fmx_match_stats_batch / fmx_smem_batch / fmx_smem_dev; index opened with lcp=1).  On the model
texts, every layout and lane count must give the model's ms_len, intervals, SMEMs and index requests (tests/match_model.py; rank blocks
are compared on PLANES, where the model counts them); at n ~ 2e6 every result is checked through the count path alone; SMEMs found on the
device feed fmx_locate_dev and every occurrence is checked against the file.  The tier past 2^31 rows (FMX_LARGE_ROWS=0 switches it off)
builds its own seeded DNA index.
"""
import ctypes as C
import os
import threading

import numpy as np
import pytest

from findex_b200 import fmindex as fx
from match_model import LcpModel, Matcher, smems
from test_match_model import _index, _queries, _texts

pytestmark = pytest.mark.gpu
MODE = os.environ.get("FMX_LARGE_ROWS", "1")
TWO31 = 1 << 31


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU; the product has no CPU path"
    from findex_b200 import build
    build.build()


def _open(F, **kw):
    bwt, eof, cnt = fx.build_bwt(F)
    return fx.GpuFMSearcher(bwt=bwt, eof=eof, counts=cnt, **kw)


def _reads(F, count, length, sub, seed, random_frac=0.0):
    """reads taken from the file with a fraction `sub` of substituted symbols, plus random reads"""
    rng = np.random.default_rng(seed)
    Fa = np.frombuffer(F, np.uint8)
    alpha = np.unique(Fa)
    st = rng.integers(0, len(F) - length, count)
    R = Fa[st[:, None] + np.arange(length)].copy()
    mask = rng.random(R.shape) < sub
    R[mask] = alpha[rng.integers(0, len(alpha), int(mask.sum()))]
    k = int(count * random_frac)
    if k:
        R[:k] = alpha[rng.integers(0, len(alpha), (k, length))]
    return [r.tobytes() for r in R]


def _flat_smems(off, ln, sp, ep, min_len):
    out = []
    for q in range(len(off) - 1):
        a, b = off[q], off[q + 1]
        out.append(smems(ln[a:b].tolist(), sp[a:b].tolist(), ep[a:b].tolist(), min_len))
    return out


@pytest.fixture(scope="module")
def model_cases():
    cases = {}
    for name, F in _texts().items():
        Fz, o, lcp = _index(F)
        mt = Matcher(o, lcp)
        qs = _queries(Fz, len(F), count=16)
        runs = [mt.run(q) for q in qs]
        o.close()
        cases[name] = (F, qs, runs, mt.lm.nbytes())
    return cases


@pytest.mark.parametrize("layout", [fx.LAYOUT_PLANES, fx.LAYOUT_WM, fx.LAYOUT_WMX])
def test_every_layout_and_lane_count_equals_the_model(model_cases, layout):
    for name, (F, qs, runs, nbytes) in model_cases.items():
        for lanes in (1, 2, 4):
            g = _open(F, lcp=1, layout=layout, lanes_per_query=lanes, accel=fx.ACCEL_NONE)
            assert g.info()["lcp_bytes"] == nbytes
            g.set_stats(True)
            off, ln, sp, ep = g.match_stats(qs)
            got_req = g.last_match_requests()
            want_req = [sum(r[3][k] for r in runs) for k in range(3)]
            assert got_req[1:] == tuple(want_req[1:]), (name, layout, lanes)
            if layout == fx.LAYOUT_PLANES:
                assert got_req[0] == want_req[0], (name, lanes)
            assert g.last_steps() == sum(got_req)
            for q, r in enumerate(runs):
                a, b = off[q], off[q + 1]
                assert ln[a:b].tolist() == r[0], (name, layout, lanes, q)
                assert sp[a:b].tolist() == r[1] and ep[a:b].tolist() == r[2], (name, layout, lanes, q)
            _, ln2, none_sp, _ = g.match_stats(qs, intervals=False)
            assert none_sp is None and np.array_equal(ln, ln2)
            for min_len in (1, 5, 20):
                so, st, sl, ssp, sep = g.smems(qs, min_len=min_len)
                for q, r in enumerate(runs):
                    want = smems(r[0], r[1], r[2], min_len)
                    got = list(zip(st[so[q]:so[q + 1]].tolist(), sl[so[q]:so[q + 1]].tolist(), ssp[so[q]:so[q + 1]].tolist(), sep[so[q]:so[q + 1]].tolist()))
                    assert got == want, (name, layout, lanes, q, min_len)
            g.close()


def _check_by_count(g, qs, off, ln, sp, ep):
    """for every position: count(reverse(match)) = the interval, and the match one symbol longer does not occur"""
    pats, longer, want = [], [], []
    for q, Q in enumerate(qs):
        for j in range(len(Q)):
            i = off[q] + j
            l = int(ln[i])
            pats.append(Q[j - l + 1:j + 1][::-1])
            want.append((int(sp[i]), int(ep[i])) if l else (0, g.n))
            if j - l >= 0:
                longer.append(Q[j - l:j + 1][::-1])
    s, e = g.count_batch(pats)
    empty = np.array([len(p) == 0 for p in pats])
    s = np.where(empty, 0, s)
    e = np.where(empty, g.n, e)
    assert np.array_equal(np.stack([s, e], 1), np.array(want, np.int64))
    s2, e2 = g.count_batch(longer)
    assert (s2 >= e2).all()


@pytest.mark.parametrize("alpha", [b"ACGT", bytes(range(1, 256))])
def test_scaled_run_checked_by_the_count_path(alpha):
    rng = np.random.default_rng(len(alpha))
    F = np.frombuffer(alpha, np.uint8)[rng.integers(0, len(alpha), 2_000_000)].tobytes()
    g = _open(F, lcp=1)
    qs = _reads(F, 6000, 150, 0.02, 5)
    off, ln, sp, ep = g.match_stats(qs)
    _check_by_count(g, qs, off, ln, sp, ep)
    so, st, sl, ssp, sep = g.smems(qs, min_len=10)
    assert [len(x) for x in _flat_smems(off, ln, sp, ep, 10)] == np.diff(so).tolist()
    g.close()


def test_smem_dev_chained_into_locate():
    import torch
    rng = np.random.default_rng(4)
    F = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 400_000)].tobytes()
    g = _open(F, lcp=1, sa_sample_rate=8)
    n = g.n
    qs = _reads(F, 3000, 150, 0.01, 6, random_frac=0.1) + [b"", b"ACGT\0ACGT"]
    ho, hst, hln, hsp, hep = g.smems(qs, min_len=12)
    pat, off = g._queries(qs)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        d_pat = torch.from_numpy(pat.copy()).cuda()
        d_off = torch.from_numpy(off).cuda()
        m = len(qs)
        cap = int(ho[m])
        d_oo = torch.zeros(m + 1, dtype=torch.int64, device="cuda")
        d_st = torch.zeros(cap, dtype=torch.int32, device="cuda")
        d_ln = torch.zeros(cap, dtype=torch.int32, device="cuda")
        d_sp = torch.zeros(cap, dtype=torch.int32, device="cuda")
        d_ep = torch.zeros(cap, dtype=torch.int32, device="cuda")
        total = g.smems_dev(d_pat.data_ptr(), d_off.data_ptr(), m, 12, d_oo.data_ptr(), d_st.data_ptr(), d_ln.data_ptr(), d_sp.data_ptr(),
                            d_ep.data_ptr(), cap, st.cuda_stream)
        assert total == cap
        nocc = int((d_ep.to(torch.int64) - d_sp.to(torch.int64)).sum().item())
        d_loff = torch.zeros(total + 1, dtype=torch.int64, device="cuda")
        d_pos = torch.zeros(max(nocc, 1), dtype=torch.int32, device="cuda")
        got = g.locate_dev(d_sp.data_ptr(), d_ep.data_ptr(), total, d_loff.data_ptr(), d_pos.data_ptr(), nocc, st.cuda_stream)
    st.synchronize()
    assert got == nocc
    assert np.array_equal(d_oo.cpu().numpy(), ho)
    assert np.array_equal(d_st.cpu().numpy(), hst) and np.array_equal(d_ln.cpu().numpy(), hln)
    assert np.array_equal(d_sp.cpu().numpy().view(np.uint32), hsp) and np.array_equal(d_ep.cpu().numpy().view(np.uint32), hep)
    loff, pos = d_loff.cpu().numpy(), d_pos.cpu().numpy().view(np.uint32).astype(np.int64)
    checked = 0
    for q in range(m):
        for k in range(ho[q], ho[q + 1]):
            s, l = int(hst[k]), int(hln[k])
            seg = qs[q][s:s + l]
            if b"\0" in seg:
                continue
            for p in pos[loff[k]:loff[k + 1]]:
                f = (n - 1) - int(p) - l
                assert F[f:f + l] == seg
                checked += 1
    assert checked >= 3000
    g.close()


def test_capacity_errors_and_budget():
    rng = np.random.default_rng(8)
    F = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 20_000)].tobytes()
    plain = _open(F)
    with pytest.raises(fx.ReUnsupported):
        plain.match_stats([b"ACGT"])
    with pytest.raises(fx.ReUnsupported):
        plain.smems([b"ACGT"])
    plain.close()
    g = _open(F, lcp=1)
    qs = _reads(F, 50, 80, 0.05, 1)
    ho, hst, hln, hsp, hep = g.smems(qs, min_len=1, cap_total=1)         # the wrapper retries with the reported total
    total = int(ho[-1])
    assert total > 2
    L = fx.lib()
    pat, off = g._queries(qs)
    m = len(qs)
    oo = np.zeros(m + 1, np.int64)
    st, ln = np.full(3, -7, np.int32), np.full(3, -7, np.int32)
    sp, ep = np.full(3, -7, np.int64), np.full(3, -7, np.int64)
    p = fx._ptr
    rc = L.fmx_smem_batch(g.h, p(pat), p(off), m, 1, 2, p(oo), p(st), p(ln), p(sp), p(ep))
    assert rc == fx.FMX_E_CAPACITY and oo[m] == total and np.array_equal(oo, ho)
    assert (st == -7).all() and (ln == -7).all() and (sp == -7).all() and (ep == -7).all()
    with pytest.raises(fx.FmxError) as e:
        g.smems(qs, min_len=0)
    assert e.value.code == fx.FMX_E_ARG
    bad = off.copy()
    bad[2], bad[3] = bad[3], bad[2]
    assert L.fmx_smem_batch(g.h, p(pat), p(bad), m, 1, total, p(oo), p(st), p(ln), p(sp), p(ep)) == fx.FMX_E_ARG
    lnv = np.zeros(int(off[-1]), np.int32)
    assert L.fmx_match_stats_batch(g.h, p(pat), p(bad), m, p(lnv), None, None) == fx.FMX_E_ARG
    assert L.fmx_match_stats_batch(g.h, None, p(off), m, p(lnv), None, None) == fx.FMX_E_ARG
    assert L.fmx_match_stats_batch(g.h, p(pat), p(off), m, None, None, None) == fx.FMX_E_ARG
    assert L.fmx_smem_batch(g.h, p(pat), p(off), m, 1, total, None, p(st), p(ln), p(sp), p(ep)) == fx.FMX_E_ARG
    tot = C.c_int64()
    assert L.fmx_smem_dev(g.h, None, None, m, 1, None, None, None, None, None, 0, C.byref(tot), None) == fx.FMX_E_ARG
    off0, ln0, _, _ = g.match_stats([])
    assert len(off0) == 1 and len(ln0) == 0
    so, *_ = g.smems([b"", b""])
    assert so.tolist() == [0, 0, 0]
    g.close()
    for bad_lcp in (-1, 2):
        with pytest.raises(fx.FmxError) as e:
            _open(F, lcp=bad_lcp)
        assert e.value.code == fx.FMX_E_ARG
    w = _open(F, accel=fx.ACCEL_NONE, layout=fx.LAYOUT_WM)
    cap = w.info()["index_bytes"]
    w.close()
    with pytest.raises(fx.FmxError) as e:
        _open(F, accel=fx.ACCEL_NONE, layout=fx.LAYOUT_WM, max_total_bytes=cap, lcp=1)
    assert e.value.code == fx.FMX_E_ARG


@pytest.mark.parametrize("sa_rate", [0, 16])
def test_lcp_changes_nothing_else(sa_rate):
    rng = np.random.default_rng(21)
    F = np.frombuffer(bytes(range(1, 256)), np.uint8)[rng.integers(0, 255, 200_000)].tobytes()
    a = _open(F, sa_sample_rate=sa_rate)
    b = _open(F, sa_sample_rate=sa_rate, lcp=1)
    ia, ib = a.info(), b.info()
    assert ia["lcp_bytes"] == 0 and ib["lcp_bytes"] == LcpModel(b.build_lcp()).nbytes()
    assert ib["index_bytes"] - ia["index_bytes"] == ib["lcp_bytes"]
    for key in ia:
        if key not in ("index_bytes", "lcp_bytes"):
            assert ia[key] == ib[key], key
    Fa = np.frombuffer(F, np.uint8)
    for ln in (4, 12, 30):
        st = rng.integers(0, len(F) - ln, 3000)
        pats = Fa[st[:, None] + np.arange(ln)][:, ::-1].copy()
        pats[::5] = rng.integers(1, 256, (len(pats[::5]), ln))
        sa_, ea = a.count_fixed(pats)
        sb, eb = b.count_fixed(pats)
        assert np.array_equal(sa_, sb) and np.array_equal(ea, eb)
    a.close()
    b.close()


def test_concurrent_host_threads():
    rng = np.random.default_rng(31)
    F = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 300_000)].tobytes()
    g = _open(F, lcp=1)
    sets = [_reads(F, 800, 100, 0.03, s) for s in range(4)]
    want = [g.match_stats(qs) for qs in sets]
    want_sm = [g.smems(qs, min_len=8) for qs in sets]
    errors = []

    def work(k):
        try:
            for _ in range(5):
                got = g.match_stats(sets[k])
                assert all(np.array_equal(x, y) for x, y in zip(got, want[k]))
                got = g.smems(sets[k], min_len=8)
                assert all(np.array_equal(x, y) for x, y in zip(got, want_sm[k]))
        except Exception as e:                               # noqa: BLE001 — reported below
            errors.append(e)
    th = [threading.Thread(target=work, args=(k,)) for k in range(4)]
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
    assert g.n == L + 1 and g.info()["lcp_bytes"] > L
    # reads from both sides of 2^31 in T' (file offset f covers T' positions n-1-f-len .. n-2-f)
    starts = np.concatenate([rng.integers(0, L - 200, 1500), rng.integers(L - TWO31 - 5000, L - TWO31 + 5000, 1500)])
    qs = []
    alpha = np.frombuffer(b"ACGT", np.uint8)
    for s in starts:
        r = F[s:s + 150].copy()
        mask = rng.random(150) < 0.02
        r[mask] = alpha[rng.integers(0, 4, int(mask.sum()))]
        qs.append(r.tobytes())
    off, ln, sp, ep = g.match_stats(qs)
    assert (ep > TWO31).any() and (sp < TWO31).any()
    _check_by_count(g, qs, off, ln, sp, ep)
    g.close()

"""
Extract on the GPU (fmx_text_batch / fmx_text_dev; DESIGN.md §3): the indexed file bytes at any file offset, from the text samples
(fmx_opts.text_sample_rate) and the row-context hops, the compact contexts, the singleton shortcut or LF steps.  Every path must give the
file with its 0x00 bytes dropped, for every offset and the lengths around the hop length, on every layout and lane count; opening with
text samples must change nothing else.  The tier past 2^31 rows (FMX_LARGE_ROWS=0 switches it off) builds its own seeded DNA index.
"""
import os
import threading

import numpy as np
import pytest

from findex_b200 import fmindex as fx
from oracle import fm_oracle as fo

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
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


def _synthetic(sigma, n, seed, zeros=False):
    rng = np.random.default_rng(seed)
    alpha = np.arange(1, 256, dtype=np.uint8) if sigma == 255 else np.sort(rng.choice(np.arange(1, 256), sigma, replace=False)).astype(np.uint8)
    t = alpha[rng.integers(0, sigma, n)]
    if zeros:
        t[rng.integers(0, n, n // 10)] = 0
    return t.tobytes()


def _files():
    out = {}
    for name in sorted(os.listdir(os.path.join(ROOT, "tests", "golden", "ref"))):
        if name.endswith(".txt"):
            out[name] = open(os.path.join(ROOT, "tests", "golden", "ref", name), "rb").read()
    for sigma in (2, 4, 28, 255):
        out["sigma%d" % sigma] = _synthetic(sigma, 700, sigma)
    out["zeros"] = _synthetic(28, 700, 5, zeros=True)
    return out


def _lengths(J, nf):
    return sorted({0, 1, max(J - 1, 0), J, J + 1, 3 * J, nf})


def _check_all(g, F, J, note):
    """every offset x the lengths around J, against the file with zeros dropped"""
    Fz = F.replace(b"\0", b"")
    nf = len(Fz)
    assert g.n - 1 == nf
    offs = np.arange(nf + 1)
    for ln in _lengths(J, nf):
        got = g.text_batch(offs, ln)
        for f in range(nf + 1):
            assert got[f] == Fz[f:f + ln], (note, f, ln)


def test_every_offset_and_length_golden_and_synthetic():
    for name, F in _files().items():
        for rate in (1, 7, 32):
            g = _open(F, text_sample_rate=rate)
            assert g.info()["text_sample_rate"] == rate
            _check_all(g, F, max(g.info()["ctx_depth"], 12), (name, rate))
            g.close()


def _paths(F, dna):
    """(name, searcher) for every path on one text"""
    g = _open(F, text_sample_rate=5)
    yield "auto", g
    g.set_accel_mask(fx.ACCEL_KMER)                                    # contexts hidden: LF steps
    yield "auto-lf", g
    g.close()
    if dna:
        g = _open(F, text_sample_rate=5, accel=fx.ACCEL_CTX8)
        assert g.info()["ctx_entry_bytes"] == 8
        yield "ctx8", g
        g.close()
    for rate in (0, 5):
        g = _open(F, text_sample_rate=rate, accel=fx.ACCEL_TEXT)
        assert g.info()["text_shortcut"]
        yield "isat%d" % rate, g
        g.close()
    for layout in (fx.LAYOUT_PLANES, fx.LAYOUT_WM, fx.LAYOUT_WMX):
        for lanes in (1, 2, 4):
            g = _open(F, text_sample_rate=5, accel=fx.ACCEL_NONE, layout=layout, lanes_per_query=lanes)
            yield "none-%d-%d" % (layout, lanes), g
            g.close()


@pytest.mark.parametrize("sigma", [4, 28, 255])
def test_every_path_gives_the_same_bytes(sigma):
    F = _synthetic(sigma, 3000, 40 + sigma)
    Fz = F
    rng = np.random.default_rng(sigma)
    offs = np.concatenate([np.arange(0, 40), np.arange(len(F) - 40, len(F) + 1), rng.integers(0, len(F) + 1, 300)])
    lens = (0, 1, 11, 12, 13, 16, 19, 32, 33, 100, 600, 1500)
    want = {ln: [Fz[f:f + ln] for f in offs] for ln in lens}
    seen = []
    for name, g in _paths(F, sigma == 4):
        for ln in lens:
            assert g.text_batch(offs, ln) == want[ln], (name, ln)
        seen.append(name)
    assert len(seen) == 2 + (sigma == 4) + 2 + 9


def test_whole_text_in_one_request():
    F = _synthetic(28, 2_000_003, 77)
    g = _open(F, text_sample_rate=32)
    assert g.text_batch([0], len(F))[0] == F
    g.set_accel_mask(fx.ACCEL_KMER)
    assert g.text(0, len(F)) == F
    g.close()
    G = _synthetic(4, 2_000_001, 78)
    g = _open(G, text_sample_rate=32, accel=fx.ACCEL_CTX8)
    assert g.text(0, len(G)) == G
    g.close()


def test_locate_round_trip_and_device_form():
    import torch
    F = _synthetic(4, 500_000, 9)
    g = _open(F, text_sample_rate=16, sa_sample_rate=8)
    n = g.n
    rng = np.random.default_rng(3)
    k = 20
    Fa = np.frombuffer(F, np.uint8)
    starts = rng.integers(0, len(F) - k, 2000)
    pats = Fa[starts[:, None] + np.arange(k)][:, ::-1].copy()            # patterns are matched in T' = reverse(file)
    sp, ep = g.count_fixed(pats)
    off, pos = g.locate_batch(sp, ep)
    assert len(pos) >= 2000
    fo_ = (n - 1) - pos - k
    got = g.text_batch(fo_, k)
    for q in range(len(pats)):
        for i in range(off[q], off[q + 1]):
            assert got[i] == pats[q][::-1].tobytes()
    # device form on a user stream, chained after locate_dev through one torch conversion
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        d_pat = torch.from_numpy(pats).cuda()
        d_sp = torch.zeros(len(pats), dtype=torch.int32, device="cuda")
        d_ep = torch.zeros(len(pats), dtype=torch.int32, device="cuda")
        g.count_fixed_dev(d_pat.data_ptr(), k, len(pats), d_sp.data_ptr(), d_ep.data_ptr(), st.cuda_stream)
        d_off = torch.zeros(len(pats) + 1, dtype=torch.int64, device="cuda")
        d_pos = torch.zeros(len(pos), dtype=torch.int32, device="cuda")
        total = g.locate_dev(d_sp.data_ptr(), d_ep.data_ptr(), len(pats), d_off.data_ptr(), d_pos.data_ptr(), len(pos), st.cuda_stream)
        d_foff = ((n - 1 - k) - d_pos[:total].to(torch.int64)).to(torch.int32)
        d_out = torch.zeros((total, k), dtype=torch.uint8, device="cuda")
        d_len = torch.zeros(total, dtype=torch.int32, device="cuda")
        g.text_dev(d_foff.data_ptr(), total, k, d_out.data_ptr(), d_len.data_ptr(), st.cuda_stream)
    st.synchronize()
    assert total == len(pos)
    assert np.array_equal(d_len.cpu().numpy(), np.full(total, k))
    want = np.stack([np.frombuffer(b, np.uint8) for b in got])
    assert np.array_equal(d_out.cpu().numpy(), want)
    # text_dev == text_batch on arbitrary offsets, including the end of the text and one past it (out_len -1)
    offs = np.concatenate([rng.integers(0, n, 5000), [0, n - 2, n - 1, n]]).astype(np.int64)
    d_o = torch.from_numpy(offs.astype(np.uint32).view(np.int32)).cuda()
    d_out = torch.zeros((len(offs), 700), dtype=torch.uint8, device="cuda")
    d_len = torch.zeros(len(offs), dtype=torch.int32, device="cuda")
    g.text_dev(d_o.data_ptr(), len(offs), 700, d_out.data_ptr(), d_len.data_ptr(), 0)
    torch.cuda.synchronize()
    h_out, h_len = d_out.cpu().numpy(), d_len.cpu().numpy()
    assert h_len[-1] == -1
    ref = g.text_batch(offs[:-1], 700)
    for i in range(len(offs) - 1):
        assert h_out[i, :h_len[i]].tobytes() == ref[i]
    g.close()


def test_errors():
    F = _synthetic(28, 5000, 2)
    g = _open(F, accel=fx.ACCEL_CTX)
    with pytest.raises(fx.ReUnsupported):
        g.text_batch([0], 4)
    g.close()
    g = _open(F, text_sample_rate=8)
    n = g.n
    for bad in (-1, n):
        with pytest.raises(fx.FmxError) as e:
            g.text_batch([0, bad], 4)
        assert e.value.code == fx.FMX_E_ARG
    with pytest.raises(fx.FmxError) as e:
        g.text_batch([0], -1)
    assert e.value.code == fx.FMX_E_ARG
    assert g.text_batch([], 5) == [] and g.text_batch([3, n - 1], 0) == [b"", b""]
    g.close()
    for rate in (-1, 65537):
        with pytest.raises(fx.FmxError) as e:
            _open(F, text_sample_rate=rate)
        assert e.value.code == fx.FMX_E_ARG
    g = _open(F, text_sample_rate=0)
    assert g.info()["text_sample_rate"] == 0
    g.close()
    g = _open(F, text_sample_rate=65536)
    assert g.text(0, 100) == F[:100]
    base = g.info()["index_bytes"]
    g.close()
    # a cap the samples do not fit (rank structure + BWT take all of it)
    plain = _open(F, accel=fx.ACCEL_NONE, layout=fx.LAYOUT_WM)
    cap = plain.info()["index_bytes"]
    plain.close()
    with pytest.raises(fx.FmxError) as e:
        _open(F, accel=fx.ACCEL_NONE, layout=fx.LAYOUT_WM, max_total_bytes=cap, text_sample_rate=1)
    assert e.value.code == fx.FMX_E_ARG
    assert base > 0


@pytest.mark.parametrize("sa_rate", [0, 16])
def test_samples_change_nothing_else(sa_rate):
    F = _synthetic(255, 200_000, 21)
    a = _open(F, sa_sample_rate=sa_rate)
    b = _open(F, sa_sample_rate=sa_rate, text_sample_rate=7)
    n = a.n
    ia, ib = a.info(), b.info()
    assert ib["index_bytes"] - ia["index_bytes"] == 4 * ((n - 1) // 7 + 1)
    for key in ia:
        if key not in ("index_bytes", "text_sample_rate"):
            assert ia[key] == ib[key], key
    rng = np.random.default_rng(5)
    Fa = np.frombuffer(F, np.uint8)
    for ln in (4, 12, 16, 30):
        st = rng.integers(0, len(F) - ln, 3000)
        pats = Fa[st[:, None] + np.arange(ln)][:, ::-1].copy()
        pats[::5] = rng.integers(1, 256, (len(pats[::5]), ln))
        sa_, ea = a.count_fixed(pats)
        sb, eb = b.count_fixed(pats)
        assert np.array_equal(sa_, sb) and np.array_equal(ea, eb)
        if ln == 4:
            oa, pa = a.locate_batch(sa_, ea)
            ob, pb = b.locate_batch(sb, eb)
            assert np.array_equal(oa, ob) and np.array_equal(pa, pb)
    assert np.array_equal(a.build_lcp(), b.build_lcp())
    a.close()
    b.close()


def test_concurrent_host_threads():
    F = _synthetic(28, 300_000, 31)
    g = _open(F, text_sample_rate=32, sa_sample_rate=16)
    Fa = np.frombuffer(F, np.uint8)
    errors = []

    def work(seed):
        try:
            rng = np.random.default_rng(seed)
            for _ in range(6):
                offs = rng.integers(0, len(F) + 1, 3000)
                ln = int(rng.integers(1, 300))
                got = g.text_batch(offs, ln)
                assert all(got[i] == F[f:f + ln] for i, f in enumerate(offs))
                st = rng.integers(0, len(F) - 12, 2000)
                pats = Fa[st[:, None] + np.arange(12)][:, ::-1].copy()
                sp, ep = g.count_fixed(pats)
                assert (ep > sp).all()
                off, pos = g.locate_batch(sp[:200], ep[:200])
                assert (pos <= g.n - 1).all()
        except Exception as e:                               # noqa: BLE001 — reported below
            errors.append(e)
    th = [threading.Thread(target=work, args=(s,)) for s in range(4)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    g.close()
    assert not errors, errors


# ---- past 2^31 rows ------------------------------------------------------------------------------------------------------------------
def test_past_2_31_rows():
    if MODE == "0":
        pytest.skip("FMX_LARGE_ROWS=0: the tier past 2^31 rows is switched off")
    L = (1 << 32) - 3 if MODE == "max" else 2_200_000_000
    lut = np.frombuffer(b"AAACCCGGGT", np.uint8)
    rng = np.random.default_rng(23)
    F = np.empty(L, np.uint8)
    for a in range(0, L, 1 << 28):
        F[a:a + (1 << 28)] = lut[rng.integers(0, 10, min(1 << 28, L - a), dtype=np.uint8)]
    s = 32
    g = _open(F, text_sample_rate=s, accel=fx.ACCEL_CTX8 if MODE != "max" else fx.ACCEL_AUTO)
    n = g.n
    assert n == L + 1 and g.info()["text_sample_rate"] == s
    # file offsets f whose T' end q = n-1-f lies around 2^31, on every sample seam near it, and at both ends of the text
    qs = [TWO31 + d for d in range(-70, 70)] + [k * s + d for k in range(TWO31 // s - 3, TWO31 // s + 4) for d in (-1, 0, 1)]
    qs += list(range(0, 70)) + list(range(n - 1 - 70, n))
    qs += rng.integers(TWO31, n - 1, 2000).tolist()
    offs = np.array(sorted({(n - 1) - q for q in qs if 0 <= q <= n - 1}), np.int64)
    for ln in (1, 15, 16, 17, 64, 300):
        got = g.text_batch(offs, ln)
        for i, f in enumerate(offs):
            assert got[i] == F[f:f + ln].tobytes(), (ln, f)
    if MODE != "max":
        g.set_accel_mask(fx.ACCEL_KMER)
        got = g.text_batch(offs[:300], 64)
        for i, f in enumerate(offs[:300]):
            assert got[i] == F[f:f + 64].tobytes(), f
    g.close()

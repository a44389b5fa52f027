"""
Matching statistics and SMEMs (include/fmgpu.h) modelled on the CPU (tests/match_model.py): the LCP structure and both scans of the
widening, built from the oracle's exact LCP array, and the left-to-right algorithm over the oracle's backward steps.  Every ms_len must
equal brute force (the longest suffix of Q[..j] that is a substring of F + 0x00 + F), every interval the oracle's search of the reversed
match, every widening the plain linear scans of the recurrence; SMEMs must be the maximal occurring substrings.  Texts: binary, DNA,
sigma = 28 (the reference's words fixture), sigma = 255, a file with 0x00 bytes, a 3000-byte block three times and a 2000-byte run (LCPs
of >= 255: escapes spanning blocks and levels), and a 40000-symbol text with two levels of minima.
"""
import lzma
import os

import numpy as np
import pytest

from match_model import ESC, LcpModel, Matcher, brute_ms, smems, widen_by_scan
from oracle import fm_oracle as fo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _rand(alpha, n, seed):
    rng = np.random.default_rng(seed)
    return np.frombuffer(alpha, np.uint8)[rng.integers(0, len(alpha), n)].tobytes()


def _words(n):
    """the first n bytes of the reference's words fixture (its BWT walked back to the text)"""
    with lzma.open(os.path.join(ROOT, "tests", "golden", "ref", "words.bwt.xz"), "rb") as f:
        raw = f.read()
    nn, eof = np.frombuffer(raw[:16], ">i8")
    bwt = np.frombuffer(raw[16:], np.uint8).copy()
    cnt = np.frombuffer(open(os.path.join(ROOT, "tests", "golden", "ref", "words.aux"), "rb").read(), ">i8").astype(np.int64)
    o = fo.OracleIndex.from_bwt(bwt, int(eof), cnt)
    F = o.prevSubstr(0, int(nn) - 1)
    o.close()
    return F[:n]


def _texts():
    block = _rand(b"ACGT", 3000, 7)
    run = _rand(b"ab", 300, 8) + b"z" * 2000 + _rand(b"ab", 300, 9)
    zeros = bytearray(_rand(bytes(range(1, 29)), 900, 10))
    for i in range(0, 900, 37):
        zeros[i] = 0
    return {
        "binary": _rand(b"ab", 1500, 1),
        "dna": _rand(b"ACGT", 2000, 2) + b"ACGTTGCA" * 40,
        "words": _words(6000),
        "sigma255": _rand(bytes(range(1, 256)), 1500, 3),
        "zeros": bytes(zeros),
        "block3": block + block + block,
        "run2000": run,
    }


def _index(F):
    Fz = F.replace(b"\0", b"")
    o = fo.OracleIndex.from_text_rev(fo.file_to_text_rev(F))
    return Fz, o, o.lcp()


def _queries(Fz, seed, count=40):
    """edited substrings, random strings, 0x00 (also across the end and start of the file), absent bytes, lengths 0 / 1 / > |F|"""
    rng = np.random.default_rng(seed)
    nf = len(Fz)
    alpha = sorted(set(Fz)) or [65]
    qs = [b"", Fz[:1], bytes([alpha[0]]), b"\0", Fz + Fz[: nf // 3], b"\0" + Fz, Fz[nf // 2:] + b"\0" + Fz[:nf // 2]]
    for _ in range(count):
        ln = int(rng.integers(2, 120))
        s = int(rng.integers(0, max(nf - ln, 1)))
        q = bytearray(Fz[s:s + ln])
        for _ in range(int(rng.integers(0, 4))):
            if q:
                q[int(rng.integers(0, len(q)))] = int(rng.choice(alpha))
        qs.append(bytes(q))
    for _ in range(count // 4):
        qs.append(bytes(int(rng.choice(alpha)) for _ in range(int(rng.integers(1, 60)))))
    k = int(rng.integers(1, 30))
    qs.append(Fz[nf - k:] + b"\0" + Fz[:k])                                # across the file boundary
    qs.append(Fz[nf - k:] + b"\0" + Fz[:k] + b"\0" + Fz[:5])
    absent = next((c for c in range(1, 256) if c not in set(Fz)), None)
    if absent is not None:
        qs.append(Fz[:20] + bytes([absent]) + Fz[40:70])
    return qs


@pytest.fixture(scope="module")
def texts():
    return _texts()


def test_structure_layout():
    rng = np.random.default_rng(0)
    for n in (1, 2, 63, 64, 65, 1024, 1025, 16 * 64 + 1, 512 * 64 + 1, 40000):
        lcp = rng.integers(0, 300, n)
        lcp[-1] = 0
        lm = LcpModel(lcp)
        assert lm.nb == (n + 63) // 64
        assert np.array_equal(lm.lcp8[:n], np.minimum(lcp, ESC))
        assert np.array_equal(lm.lcpx, lcp[lcp >= ESC])
        for b in range(lm.nb):
            assert lm.levels[0][b] == lcp[b * 64:(b + 1) * 64].min()
            assert lm.rec_x[b] == (lcp[:b * 64] >= ESC).sum()
        assert len(lm.levels[-1]) <= (16 if lm.top == 0 else 32)
        assert lm.top == (0 if lm.nb <= 16 else 1 if lm.nb <= 512 else 2)
        for r in rng.integers(0, n, 50):
            assert lm.value(int(r))[0] == lcp[r]


def test_widening_equals_the_recurrence(texts):
    for name, F in list(texts.items()) + [("two-levels", _rand(b"ACGT", 40000, 11))]:
        Fz, o, lcp = _index(F)
        n = o.n
        lm = LcpModel(lcp)
        if name == "two-levels":
            assert lm.top == 2
        if name in ("block3", "run2000"):
            assert lcp.max() > 2 * ESC and len(lm.lcpx) > 64
        rng = np.random.default_rng(len(F))
        # every interval of a substring of T' that cannot be extended some way: intervals of the rows' prefixes of length l
        sa = o.sa().astype(np.int64)
        t = np.append(np.frombuffer(fo.file_to_text_rev(F).tobytes(), np.uint8), np.uint8(0))
        for r in rng.integers(0, n, 300):
            p = int(sa[r])
            l = int(rng.integers(1, min(n - p, 3000) + 1))
            iv = o.search(t[p:p + l].tobytes())
            assert iv is not None
            sp, ep = iv
            want = widen_by_scan(lcp, sp, ep)
            got = lm.widen(sp, ep)
            assert got[:3] == want, (name, sp, ep, l)
            assert want[2] < l
            if want[2] > 0:
                assert o.search(t[p:p + want[2]].tobytes()) == (want[0], want[1])
        o.close()


def test_matching_statistics_against_brute_force(texts):
    for name, F in texts.items():
        Fz, o, lcp = _index(F)
        mt = Matcher(o, lcp)
        n = o.n
        for qi, q in enumerate(_queries(Fz, len(F))):
            ms_l, ms_sp, ms_ep, req = mt.run(q)
            assert ms_l == brute_ms(Fz, q), (name, qi)
            for j, l in enumerate(ms_l):
                if l == 0:
                    assert (ms_sp[j], ms_ep[j]) == (0, n)
                else:
                    assert o.search(q[j - l + 1:j + 1][::-1]) == (ms_sp[j], ms_ep[j]), (name, qi, j)
            steps = sum(1 for _ in q)
            assert req[0] <= 2 * 2 * steps                                  # <= 2L steps of at most 2 blocks each
            for ml in (1, 5, 20):
                sm = smems(ms_l, ms_sp, ms_ep, ml)
                starts = [s for s, _, _, _ in sm]
                ends = [s + l for s, l, _, _ in sm]
                assert starts == sorted(set(starts)) and ends == sorted(set(ends))
                G = Fz + b"\0" + Fz
                for s, l, _, _ in sm:
                    assert q[s:s + l] in G and l >= ml
                    if s > 0:
                        assert q[s - 1:s + l] not in G
                    if s + l < len(q):
                        assert q[s:s + l + 1] not in G
        o.close()


def test_requests_of_a_widening_inside_a_block():
    """one request per side when both boundary rows and the answers are inside their 64-row blocks"""
    lcp = np.zeros(256, np.int64)
    lcp[10:20] = 5
    lcp[15] = 7
    lcp[-1] = 0
    lm = LcpModel(lcp)
    assert lm.widen(16, 17)[:3] == widen_by_scan(lcp, 16, 17)
    sp, ep, d, lreq, mreq = lm.widen(16, 17)
    assert (d, lreq, mreq) == (7, 1, 0)
    sp, ep, d, lreq, mreq = lm.widen(15, 17)
    assert (sp, ep, d) == widen_by_scan(lcp, 15, 17) and lreq == 1 and mreq == 0
    lcp2 = np.full(64 * 40, 3, np.int64)
    lcp2[-1] = 0
    lcp2[100] = 1
    lm2 = LcpModel(lcp2)
    sp, ep, d, lreq, mreq = lm2.widen(1500, 1501)
    assert (sp, ep, d) == widen_by_scan(lcp2, 1500, 1501) == (101, 64 * 40, 3)
    assert mreq >= 2 and lreq == 3

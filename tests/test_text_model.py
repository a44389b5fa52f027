"""
Extract (fmx_text_batch / fmx_text_dev; DESIGN.md §3) modelled on the CPU: the text samples, and the walk each path of text_kernel
(fmx_kernels.cu) takes — J-hops over ctx[2r+1] (raw bytes and packed dense codes, J = 12, 19, 32), 16-hops over ctx8 with LF steps for
the last positions, direct isat reads, plain LF steps.  The entries are built here from the oracle's suffix array (bwtFm2sa), not from
the GPU.  For every file offset and lengths around the hop length, on texts of 1 .. 301 symbols and sample rates 1, 2, 7, 32 and > n,
every path must give the file bytes, independently of the segment size, and the request counts of the model in the header.
"""
import numpy as np
import pytest

from oracle import fm_oracle as fo

SEG = 512                       # fmx_kernels.cu kTextSegment


def _index(text_rev):
    """T' (with '$' = 0 at n-1), sa, isa of text_rev + '$' from the oracle"""
    o = fo.OracleIndex.from_text_rev(text_rev)
    sa = np.array(o.sa(), dtype=np.int64)
    o.close()
    t = np.append(np.frombuffer(bytes(text_rev), np.uint8), np.uint8(0)).astype(np.int64)
    n = len(t)
    isa = np.zeros(n, np.int64)
    isa[sa] = np.arange(n)
    return t, sa, isa


class Model:
    """the structures of one index and the walks over them; each walk returns (bytes, requests)"""

    def __init__(self, text_rev, J, raw):
        self.t, self.sa, self.isa = _index(text_rev)
        self.n = len(self.t)
        syms = sorted(set(self.t[:-1].tolist()))
        self.code = {c: i for i, c in enumerate(syms)}
        self.sym = syms
        self.J, self.raw = J, raw

    def samples(self, s):
        return [int(self.isa[k * s]) for k in range((self.n - 1) // s + 1)]

    # the stored symbol of T' position p as the entries hold it: the byte (raw), dense code + 1 (packed), 2-bit code (ctx8); 0 outside
    def stored(self, p, form):
        if p < 0 or p >= self.n or self.t[p] == 0:
            return 0
        c = int(self.t[p])
        return c if form == "raw" else self.code[c] + 1 if form == "packed" else self.code[c]

    def decode(self, v, form):
        return v if form == "raw" else self.sym[v - 1] if form == "packed" else self.sym[v]

    def ctx_hop(self, r):                      # ctx[2r+1]: { isa[sa[r]-J] (0 before the text), T'[sa[r]-J .. sa[r]-1] }
        x = int(self.sa[r])
        return (int(self.isa[x - self.J]) if x >= self.J else 0), [self.stored(x - self.J + k, "raw" if self.raw else "packed") for k in range(self.J)]

    def ctx8(self, r):                         # ctx8[r]: row 0xFFFFFFFF and no symbols before position 16
        x = int(self.sa[r])
        if x < 16:
            return 0xFFFFFFFF, [0] * 16
        return int(self.isa[x - 16]), [self.stored(x - 16 + k, "ctx8") for k in range(16)]

    def isat(self, p, syms):
        return [self.stored(p + k, "packed") for k in range(syms)]

    def bwt(self, r):
        x = int(self.sa[r])
        return int(self.t[x - 1]) if x > 0 else 0

    def lf(self, r):
        x = int(self.sa[r])
        return int(self.isa[(x - 1) % self.n])

    def extract(self, f, ln, path, s=None, seg=SEG, syms=12):
        n, last = self.n, self.n - 1
        q = last - f
        olen = min(ln, q)
        out = [None] * olen
        req = 0
        tsamp = self.samples(s) if s else None
        for a in range(0, max(olen, 0), seg):
            b = min(a + seg, olen)
            lo, hi = q - b, q - a

            def put(p, v):
                assert lo <= p < hi and out[q - 1 - p] is None
                out[q - 1 - p] = v
            if path == "isat":
                for p in range(lo, hi, syms):
                    e = self.isat(p, syms)
                    req += 1
                    for k in range(min(syms, hi - p)):
                        put(p + k, self.decode(e[k], "packed"))
                continue
            k0 = -(-hi // s)
            x = k0 * s
            if x > last:
                x, r = last, 0
            else:
                r = tsamp[k0]
                req += 1
            if path == "ctx":
                form = "raw" if self.raw else "packed"
                while x > lo:
                    row, e = self.ctx_hop(r)
                    req += 1
                    for k in range(self.J):
                        if lo <= x - self.J + k < hi:
                            put(x - self.J + k, self.decode(e[k], form))
                    r, x = row, max(x - self.J, 0)
            elif path == "ctx8":
                while x > lo and x >= 16:
                    row, e = self.ctx8(r)
                    assert row != 0xFFFFFFFF
                    req += 1
                    for k in range(16):
                        if lo <= x - 16 + k < hi:
                            put(x - 16 + k, self.decode(e[k], "ctx8"))
                    r, x = row, x - 16
            while x > lo:                      # LF steps: the whole walk, or the tail of a ctx8 walk
                c = self.bwt(r)
                if x - 1 < hi:
                    put(x - 1, c)
                x -= 1
                if x > lo:
                    r = self.lf(r)
                    req += 2
                else:
                    req += 1
        assert all(v is not None for v in out)
        return bytes(out), req


def _file(text_rev):
    return bytes(np.frombuffer(bytes(text_rev), np.uint8)[::-1])


def _texts():
    rng = np.random.default_rng(11)
    for n in (1, 2, 3, 5, 11, 12, 13, 16, 17, 31, 32, 33, 64, 100, 301):
        for sigma in (2, 4, 28, 255):
            alpha = np.arange(1, 256) if sigma == 255 else np.sort(rng.choice(np.arange(1, 256), sigma, replace=False))
            yield n, sigma, alpha[rng.integers(0, sigma, n)].astype(np.uint8).tobytes()


def _lengths(J, nf):
    return sorted({0, 1, J - 1, J, J + 1, 3 * J, nf})


@pytest.mark.parametrize("J,raw", [(12, True), (12, False), (19, False), (32, False)])
def test_ctx_hop_walk_gives_the_file(J, raw):
    for n, sigma, tr in _texts():
        if raw and sigma < 28:
            continue
        m = Model(tr, J, raw)
        F = _file(tr)
        for s in (1, 2, 7, 32, n + 5):
            for f in range(0, n + 1):
                for ln in _lengths(J, n):
                    got, req = m.extract(f, ln, "ctx", s)
                    assert got == F[f:f + ln], (n, sigma, s, f, ln)
                    olen = min(ln, n - f)
                    if olen:
                        q = n - f
                        q0 = -(-q // s) * s
                        # model of the header: 1 + ceil((q0 - q + out_len) / J), and no sample read when q0 is past the text
                        want = 1 + -(-(q0 - q + olen) // J) if q0 <= n else -(-(n - q + olen) // J)
                        assert req == want, (n, s, f, ln, req, want)
                    if ln > 3:
                        assert m.extract(f, ln, "ctx", s, seg=3)[0] == got


def test_ctx8_walk_with_its_tail_gives_the_file():
    for n, sigma, tr in _texts():
        if sigma > 4:
            continue
        m = Model(tr, 16, False)
        F = _file(tr)
        for s in (1, 2, 7, 32, n + 5):
            for f in range(0, n + 1):
                for ln in _lengths(16, n):
                    got, req = m.extract(f, ln, "ctx8", s)
                    assert got == F[f:f + ln], (n, s, f, ln)
                    olen = min(ln, n - f)
                    if olen:
                        q = n - f
                        q0 = min(-(-q // s) * s, n)
                        assert req <= 1 + -(-(q0 - q + olen) // 16) + 2 * 15, (n, s, f, ln, req)
                    if ln > 5:
                        assert m.extract(f, ln, "ctx8", s, seg=5)[0] == got


@pytest.mark.parametrize("syms", [12, 19, 32])
def test_isat_reads_give_the_file(syms):
    for n, sigma, tr in _texts():
        m = Model(tr, 12, False)
        F = _file(tr)
        for f in range(0, n + 1):
            for ln in _lengths(syms, n):
                got, req = m.extract(f, ln, "isat", syms=syms)
                assert got == F[f:f + ln]
                assert req == -(-min(ln, n - f) // syms)


def test_lf_walk_gives_the_file():
    for n, sigma, tr in _texts():
        m = Model(tr, 12, False)
        F = _file(tr)
        for s in (1, 2, 7, 32, n + 5):
            for f in range(0, n + 1):
                for ln in _lengths(12, n):
                    got, req = m.extract(f, ln, "lf", s)
                    assert got == F[f:f + ln], (n, s, f, ln)
                    olen = min(ln, n - f)
                    if olen:
                        q = n - f
                        read = -(-q // s) * s <= n          # a sample is read unless the walk starts at position n-1 (row 0)
                        steps = min(-(-q // s) * s, n) - q + olen
                        assert req == read + 2 * steps - 1, (n, s, f, ln, req)
                    if ln > 2:
                        assert m.extract(f, ln, "lf", s, seg=2)[0] == got


def test_start_position_near_2_32():
    """q0 = ceil(q/s)*s exceeds 32 bits near n = 2^32 - 2; the walk then starts at position n-1 (row 0), at most s-1 before q"""
    last = (1 << 32) - 3
    for s in (1, 7, 32, 65535, 65536):
        k_max = last // s
        for q in (last, last - 1, k_max * s, k_max * s - 1, last - s + 1):
            k0 = -(-q // s)
            q0 = k0 * s
            start = last if q0 > last else q0
            assert q <= start < q + s and (q0 > last or k0 <= k_max)
    assert -(-last // 65536) * 65536 > 0xFFFFFFFF

"""
Matching statistics and SMEMs (fmx_match_stats_batch / fmx_smem_*) modelled on the CPU, shared by test_match_model.py and
test_gpu_match.py: the resident LCP structure as fmx_build.cu lays it out (64-row lcp8 blocks, one {minimum, first escape} record per
block, 16 records per 128-byte line, minima levels of 32 per line, the escaped values), the widening of lcp_widen (fmx_device.cuh) request
for request, and the left-to-right algorithm of match_kernel (fmx_kernels.cu) over the oracle's backward steps.
"""
import numpy as np

ROWS, REC_LINE, FAN, ESC = 64, 16, 32, 255
INF = 0xFFFFFFFF
RANK_ROWS = 480                                   # rows per 64-byte rank block (fmx_device.cuh kBitsPerBlock)


class LcpModel:
    """the structure built from the exact LCP array; widen() returns the parent interval and the requests it costs"""

    def __init__(self, lcp):
        self.lcp = np.asarray(lcp, dtype=np.int64)
        self.n = n = len(self.lcp)
        self.nb = nb = (n + ROWS - 1) // ROWS
        full = np.zeros(nb * ROWS, np.int64)
        full[:n] = self.lcp
        self.full = full
        self.lcp8 = np.minimum(full, ESC)
        blocks = full.reshape(nb, ROWS)
        esc = (blocks >= ESC).sum(axis=1)
        self.rec_x = np.concatenate([[0], np.cumsum(esc)[:-1]]).astype(np.int64)
        self.lcpx = full[full >= ESC]
        nrec = (nb + REC_LINE - 1) // REC_LINE * REC_LINE
        level0 = np.full(nrec, INF, np.int64)
        level0[:nb] = blocks.min(axis=1)
        self.levels = [level0]
        count, F = nb, REC_LINE
        while count > F:                               # level t+1: one minimum per line of level t (lcp_layout)
            prev = self.levels[-1]
            count = (count + F - 1) // F
            lv = np.full((count + FAN - 1) // FAN * FAN, INF, np.int64)
            lv[:count] = prev[:count * F].reshape(count, F).min(axis=1)
            self.levels.append(lv)
            F = FAN
        self.top = len(self.levels) - 1

    def nbytes(self):
        up = lambda b: (b + 127) // 128 * 128
        fixed = up(self.nb * ROWS) + up(len(self.levels[0]) * 8) + sum(len(lv) * 4 for lv in self.levels[1:])
        return fixed + 4 * len(self.lcpx)

    def value(self, r):
        """exact LCP[r] and the requests beyond its block: the record and the escaped value"""
        return (int(self.lcp8[r]), 0) if self.lcp8[r] != ESC else (int(self.full[r]), 2)

    def scan(self, blk, o, d, left):
        """last row <= o / first row >= o of the block with LCP < d (-1 / 64: none), requests"""
        dd = min(d, ESC)
        row = self.lcp8[blk * ROWS:(blk + 1) * ROWS]
        cand = [k for k in (range(0, o + 1) if left else range(o, ROWS)) if row[k] < dd]
        k1 = (max(cand) if cand else -1) if left else (min(cand) if cand else ROWS)
        if d <= ESC or k1 == o:
            return k1, 0
        req = 1                                                        # the record: where the block's escapes start
        for k in (range(o, k1, -1) if left else range(o, k1)):
            req += 1
            if self.full[blk * ROWS + k] < d:
                return k, req
        return k1, req

    def climb(self, b, d, left):
        """nearest block before / after b with a minimum below d (-1: none), 128-byte lines read"""
        p, t, req = b, 0, 0
        while True:
            if t > self.top:
                return -1, req
            F = REC_LINE if t == 0 else FAN
            line, slot = p // F, p % F
            vals = self.levels[t][line * F:(line + 1) * F]
            req += 1
            hits = [s for s in range(F) if vals[s] < d and (s < slot if left else s > slot)]
            if hits:
                q = line * F + (max(hits) if left else min(hits))
                break
            p, t = line, t + 1
        while t > 0:
            t -= 1
            F = REC_LINE if t == 0 else FAN
            vals = self.levels[t][q * F:(q + 1) * F]
            req += 1
            hits = [s for s in range(F) if vals[s] < d]
            q = q * F + (max(hits) if left else min(hits))
        return q, req

    def widen(self, sp, ep):
        """(sp, ep, d, lcp requests, minima lines) of the parent interval; d = 0 -> (0, n)"""
        has_a = sp > 0
        ra, rb = (sp - 1 if has_a else 0), ep - 1
        ba, bb, oa, ob = ra // ROWS, rb // ROWS, ra % ROWS, rb % ROWS
        lreq = 2 if (has_a and ba != bb) else 1
        mreq = 0
        vb, r = self.value(rb)
        lreq += r
        va = 0
        if has_a:
            va, r = self.value(ra)
            lreq += r
        d = max(va, vb)
        if d == 0:
            return 0, self.n, 0, lreq, mreq
        nsp = 0
        if has_a and va < d:
            nsp = sp
        elif has_a:
            k, r = self.scan(ba, oa, d, True)
            lreq += r
            if k >= 0:
                nsp = ba * ROWS + k + 1
            else:
                b2, r = self.climb(ba, d, True)
                mreq += r
                if b2 >= 0:
                    k, r = self.scan(b2, ROWS - 1, d, True)
                    lreq += 1 + r
                    nsp = b2 * ROWS + k + 1
        if vb < d:
            nep = ep
        else:
            k, r = self.scan(bb, ob, d, False)
            lreq += r
            if k < ROWS:
                nep = bb * ROWS + k + 1
            else:
                b2, r = self.climb(bb, d, False)
                mreq += r
                k, r = self.scan(b2, 0, d, False)
                lreq += 1 + r
                nep = b2 * ROWS + k + 1
        return nsp, nep, d, lreq, mreq


def widen_by_scan(lcp, sp, ep):
    """the parent interval by plain linear scans (the recurrence itself, without the structure)"""
    n = len(lcp)
    d = max(int(lcp[sp - 1]) if sp > 0 else 0, int(lcp[ep - 1]))
    if d == 0:
        return 0, n, 0
    k = sp - 1
    while k >= 0 and lcp[k] >= d:
        k -= 1
    a = k + 1
    k = ep - 1
    while lcp[k] >= d:
        k += 1
    return a, k + 1, d


class Matcher:
    """match_kernel over an oracle index: ms_len / intervals of a query and the requests by kind (rank blocks counted as PLANES fetches
    them: one 64-byte block per row position, shared when sp and ep fall into the same one)"""

    def __init__(self, oracle, lcp):
        self.o = oracle
        self.n = oracle.n
        self.lm = LcpModel(lcp)
        self.first = [oracle.prev_range_raw(0, self.n, c) for c in range(256)]     # (C[c], C[c+1])

    def run(self, q):
        n, o, lm = self.n, self.o, self.lm
        l, sp, ep = 0, 0, n
        out_l, out_sp, out_ep = [], [], []
        req = [0, 0, 0]
        for c in bytes(q):
            while True:
                if l == 0:
                    sp, ep = self.first[c]
                    if sp < ep:
                        l = 1
                    else:
                        sp, ep = 0, n
                    break
                s, e = o.prev_range_raw(sp, ep, c)
                if c != 0 and self.first[c][0] < self.first[c][1]:
                    req[0] += 1 if sp // RANK_ROWS == ep // RANK_ROWS else 2
                if s < e:
                    sp, ep, l = s, e, l + 1
                    break
                sp, ep, l, a, b = lm.widen(sp, ep)
                req[1] += a
                req[2] += b
            out_l.append(l)
            out_sp.append(sp)
            out_ep.append(ep)
        return out_l, out_sp, out_ep, req


def smems(ms_len, ms_sp, ms_ep, min_len):
    """(start, len, sp, ep) of every SMEM of at least min_len symbols from the matching statistics of one query"""
    out = []
    L = len(ms_len)
    for j in range(L):
        l = ms_len[j]
        if l >= min_len and (j == L - 1 or ms_len[j + 1] <= l):
            out.append((j - l + 1, l, ms_sp[j], ms_ep[j]))
    return out


def brute_ms(F, q):
    """ms_len by brute force: the longest suffix of q[..j] that is a substring of F + 0x00 + F (F without its 0x00 bytes)"""
    G = F + b"\0" + F
    out, prev = [], 0
    q = bytes(q)
    for j in range(len(q)):
        l = prev + 1
        while l > 0 and q[j - l + 1:j + 1] not in G:
            l -= 1
        out.append(l)
        prev = l
    return out

"""
The k-mer group blocks (DevIndex::kmer_rows; DESIGN.md §3) as an executable model on the CPU.  The 64-byte blocks are packed byte for byte
as pack_kmer_groups_kernel packs them (fmx_build.cu), from the oracle's suffix array: 8 lexicographically consecutive k-mers per block,
narrow (base row + eight u8 ends + the J-hop half of the row contexts of up to three first rows) or wide (u32 ends + u8 leading gaps, for
a group of more than 255 rows or one with a row of no k-mer — '$' or a suffix shorter than k — between its intervals).  The model decodes
every entry and checks it against the table's interval, then answers patterns the way search_pattern does (block, inline rows, the other
rows through their contexts, ordinary steps for the rest) and compares the answers with the oracle's backward search (findex.scala:15-31).
The CUDA code is checked against the oracle in tests/test_gpu_kmer_rows.py.
"""
import struct

import numpy as np
import pytest

from oracle import fm_oracle as fo

GROUP, INLINE, WIDE = 8, 3, 0xFF
CTX_MAX_ROWS = 8


def hop_plan(J):
    """ctx_hop_plan (fmx_build.cu): the five hop lengths and, per remaining length, the first hop / the fetches of a fewest-fetches plan"""
    known = {12: (1, 3, 4, 8, 12), 13: (1, 3, 5, 6, 13), 16: (1, 4, 6, 15, 16), 19: (1, 4, 5, 16, 19), 24: (1, 4, 6, 15, 24),
             32: (1, 4, 9, 21, 32), 48: (1, 5, 12, 33, 48), 96: (1, 6, 16, 48, 96)}
    S = known.get(J, (1, (J + 7) // 8, (J + 3) // 4, (J + 1) // 2, J))
    cost, first = [0] * 128, [0] * 128
    for r in range(1, 128):
        best, bt = 1 << 20, 0
        for t in range(4, -1, -1):                          # ties go to the longer hop
            if S[t] <= r and cost[r - S[t]] + 1 < best:
                best, bt = cost[r - S[t]] + 1, t
        cost[r], first[r] = best, bt
    return S, first, cost


class Model:
    def __init__(self, tp, K):
        self.tp, self.K = tp, K
        bwt, eof, cnt = fo.build_bwt(tp)
        self.o = fo.OracleIndex.from_bwt(bwt, eof, cnt)
        self.sa = self.o.sa().astype(np.int64)
        n = self.n = len(self.sa)
        self.isa = np.empty(n, np.int64)
        self.isa[self.sa] = np.arange(n)
        syms = sorted(set(tp))
        self.sigma = len(syms)
        self.code = {c: i for i, c in enumerate(syms)}      # dense codes ascend with the byte value
        self.bits = max(1, int(np.ceil(np.log2(self.sigma + 1))))
        self.J = 96 // self.bits
        self.raw = self.bits == 8
        self.S, self.plan, self.need = hop_plan(self.J)
        # the plain table in lexicographic order: entry idx = the k-mer's codes, its first byte most significant
        self.entries = self.sigma ** K
        self.table = np.zeros((self.entries, 2), np.int64)
        self.no_kmer_rows = 0
        txt = tp + b"\0"
        r = 0
        while r < n:
            pre = txt[self.sa[r]:self.sa[r] + K]
            if len(pre) < K or 0 in pre:
                self.no_kmer_rows += 1
                r += 1
                continue
            e = r + 1
            while e < n and txt[self.sa[e]:self.sa[e] + K] == pre:
                e += 1
            self.table[self.idx(pre)] = (r, e)
            r = e
        self.blocks = [self.pack(g) for g in range((self.entries + GROUP - 1) // GROUP)]

    def idx(self, kmer):
        v = 0
        for c in kmer:
            v = v * self.sigma + self.code[c]
        return v

    def ctx_half(self, r):
        """ctx[2r+1] of build_ctx_kernel: isa[sa[r]-J] (0 before the start), the J symbols T'[sa[r]-J .. sa[r]-1] (0 before the start)"""
        p = int(self.sa[r])
        row = int(self.isa[p - self.J]) if p >= self.J else 0
        v = 0
        for k in range(self.J):
            q = p - self.J + k
            s = 0 if q < 0 else (self.tp[q] if self.raw else self.code[self.tp[q]] + 1)
            v |= s << (k * self.bits)
        return struct.pack("<IQI", row, v & (2 ** 64 - 1), v >> 64)

    def pack(self, g):
        v = [tuple(self.table[i]) if i < self.entries else (0, 0) for i in range(g * GROUP, g * GROUP + GROUP)]
        v = [(int(a), int(b)) if a < b else (0, 0) for a, b in v]
        ne = [a < b for a, b in v]
        base = next((a for a, b in v if a < b), 0)
        last = max((b for a, b in v if a < b), default=0)
        gap = any(v[i][0] != v[j][1] for j, i in zip([k for k in range(GROUP) if ne[k]], [k for k in range(GROUP) if ne[k]][1:]))
        if gap or last - base > 255:
            ends, leads, prev = [], [], base
            for (a, b), e in zip(v, ne):
                ends.append(b if e else prev)
                leads.append(a - prev if e else 0)
                prev = ends[-1]
            blk = struct.pack("<I11xB", base, WIDE) + struct.pack("<8I", *ends) + bytes(leads) + bytes(8)
        else:
            ends, end = [], 0
            for (a, b), e in zip(v, ne):
                end = b - base if e else end
                ends.append(end)
            kind = min(last - base, INLINE) if any(ne) else 0
            blk = struct.pack("<I8B3xB", base, *ends, kind) + b"".join(self.ctx_half(base + k) for k in range(kind))
            blk += bytes(64 - len(blk))
        assert len(blk) == 64
        return blk

    def decode(self, idx):
        """kmer_group's decode: (sp, ep), base row, inline payloads"""
        blk, e = self.blocks[idx // GROUP], idx % GROUP
        base, kind = struct.unpack_from("<I", blk, 0)[0], blk[15]
        if kind != WIDE:
            hi, lo = base + blk[4 + e], base + (blk[3 + e] if e else 0)
            inline = [blk[16 + 16 * k:32 + 16 * k] for k in range(kind)]
        else:
            ends = struct.unpack_from("<8I", blk, 16)
            hi, lo = ends[e], (ends[e - 1] if e else base) + blk[48 + e]
            inline = []
        return ((lo, hi) if lo < hi else (0, 0)), base, inline

    def hop_matches(self, half, want):
        row, lo, hi = struct.unpack("<IQI", half)
        v = lo | (hi << 64)
        syms = [(v >> (k * self.bits)) & ((1 << self.bits) - 1) for k in range(self.J)]
        return row, syms == want

    def search(self, pat):
        """search_pattern over the group form; returns the answer and the requests it made (block + contexts fetched)"""
        K, o = self.K, self.o
        if len(pat) < K or any(c == 0 or c not in self.code for c in pat[len(pat) - K:]):
            return o.search(pat), None
        (sp, ep), base, inline = self.decode(self.idx(pat[len(pat) - K:]))
        requests, rem = 1, len(pat) - K
        if sp < ep and rem > 0:
            rows = ep - sp
            t = self.plan[rem] if rem <= 127 else 4
            need = self.need[rem] if rem <= 127 else rem // self.J + 3
            if rows <= CTX_MAX_ROWS and (rows == 1 or rows * need <= rem):
                j = self.S[t]
                hop = pat[rem - j:rem]
                if 0 not in hop and t == 4:                 # the full-depth hop: the block's inline rows count
                    want = [c if self.raw else self.code.get(c, -1) + 1 for c in hop]
                    got = []
                    absent = not self.raw and any(c not in self.code for c in hop)     # nothing matches (no row is fetched)
                    for r in range(sp, ep) if not absent else ():
                        if r - base < len(inline):
                            row, ok = self.hop_matches(inline[r - base], want)
                        else:
                            requests += 1
                            row, ok = self.hop_matches(self.ctx_half(r), want)
                        if ok:
                            got.append(row)
                    sp, ep = (min(got), min(got) + len(got)) if got else (0, 0)
                    rem -= j
        for c in reversed(pat[:rem]):                       # the rest: ordinary backward steps
            if sp >= ep:
                break
            r = o.getPrevRange(sp, ep, c)
            sp, ep = r if r else (0, 0)
        return ((sp, ep) if sp < ep else None), requests


def _texts():
    rng = np.random.default_rng(7)
    uni = bytes(rng.integers(1, 256, 30000, dtype=np.uint8))
    dna = bytes(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 12000)])
    al28 = np.frombuffer(b" abcdefghijklmnopqrstuvwxyz.", np.uint8)
    t28 = bytes(al28[rng.integers(0, 28, 20000)])
    # k-mers that pile up: a few short words repeated, so that one group holds far more than 255 rows
    words = [b"abab", b"abba", b"baab", b"ab"]
    pile = b"".join(words[i] for i in rng.integers(0, len(words), 3000))
    return [("uniform255", uni, 2), ("dna", dna, 7), ("sigma28", t28, 3), ("pileup", pile, 4)]


@pytest.mark.parametrize("name,tp,K", _texts(), ids=[t[0] for t in _texts()])
def test_group_blocks_equal_table_and_backward_search(name, tp, K):
    m = Model(tp, K)
    # every entry, empty ones included, decodes to the interval of the plain table
    for i in range(m.entries):
        a, b = (int(x) for x in m.table[i])
        assert m.decode(i)[0] == ((a, b) if a < b else (0, 0)), i
    kinds = [blk[15] for blk in m.blocks]
    wide = [g for g, k in enumerate(kinds) if k == WIDE]
    over255 = [g for g in wide if struct.unpack_from("<8I", m.blocks[g], 16)[7] - struct.unpack_from("<I", m.blocks[g], 0)[0] > 255]
    gapped = [g for g in wide if any(m.blocks[g][48:56])]
    assert m.no_kmer_rows == K                               # '$' and the K-1 suffixes shorter than K
    if name == "pileup":
        assert over255
    else:
        assert sum(1 for k in kinds if k in (1, 2, 3)) > len(kinds) // 4
    if name == "dna":
        assert gapped                                        # a row of no k-mer between two intervals of one group

    rng = np.random.default_rng(11)
    alpha = sorted(set(tp))
    one_request = hits = 0
    for ln in range(K, 3 * K + 6):
        for _ in range(40):
            s = int(rng.integers(0, len(tp) - ln))
            q = bytearray(tp[s:s + ln])
            u = rng.random()
            if u < 0.3:
                q = bytearray(bytes(alpha[int(x)] for x in rng.integers(0, len(alpha), ln)))
            elif u < 0.35:
                q[int(rng.integers(0, ln))] = 255 if 255 not in alpha else 1   # a byte that does not occur
            got, req = m.search(bytes(q))
            assert got == m.o.search(bytes(q)), (bytes(q), got)
            if got is not None:
                hits += 1
                one_request += req == 1
    # a 12-symbol tail after the table is answered from the block alone when the interval's rows are all inline
    for _ in range(200):
        s = int(rng.integers(0, len(tp) - K - m.J))
        q = tp[s:s + K + m.J]
        got, req = m.search(q)
        assert got == m.o.search(q)
        one_request += req == 1
    assert hits > 0 and one_request > 0
    # the answers of the oracle's batch count for the same patterns
    pats = [tp[s:s + K + m.J] for s in rng.integers(0, len(tp) - K - m.J, 50)]
    flat = np.frombuffer(b"".join(pats), np.uint8)
    off = np.arange(0, len(flat) + 1, K + m.J, dtype=np.int64)
    bsp, bep = m.o.count_batch(flat, off)
    for p, a, b in zip(pats, bsp, bep):
        got = m.search(p)[0]
        assert (got or (0, 0)) == (int(a), int(b))
    m.o.close()

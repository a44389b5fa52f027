"""
oracle/fm_oracle.py — TEST INFRASTRUCTURE ONLY. NOT PART OF THE PRODUCT.

ctypes binding of oracle/fm_oracle.c (the plain-C restatement of the reference's FM-index path) plus
the glue that runs oracle/retree.py automata through the C traversal loop.  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from . import retree

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "fm_oracle.c")
_SO = os.path.join(_HERE, "libfm_oracle.so")
_NATIVE_DIR = None


def build(force=False, native=False):
    """gcc -O3 the C restatement into oracle/libfm_oracle.so (git-ignored).  native=True builds a -march=native copy on the
    machine it will be timed on (bench.py's CPU legs), once per process and in a temporary directory so that a read-only tree
    works, and makes lib() use it."""
    global _SO, _lib, _NATIVE_DIR
    if native:
        if _NATIVE_DIR is None:
            _NATIVE_DIR = tempfile.mkdtemp(prefix="fm_oracle_")
            atexit.register(shutil.rmtree, _NATIVE_DIR, True)
        so = os.path.join(_NATIVE_DIR, "libfm_oracle_native.so")
    else:
        so = os.path.join(_HERE, "libfm_oracle.so")
    if force or (not os.path.exists(so)) or os.path.getmtime(so) < os.path.getmtime(_SRC):
        subprocess.check_call(["gcc", "-O3", "-march=native" if native else "-march=x86-64-v2", "-fPIC", "-shared", "-pthread",
                               "-Wno-format-truncation", "-o", so, _SRC])
    if so != _SO:
        _SO = so
        _lib = None
    return so


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build() if not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(_SRC) else _SO)
        p, i64, i32, u8p = C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_uint8)
        L.fmo_last_error.restype = C.c_char_p
        L.fmo_from_memory.restype = p
        L.fmo_from_memory.argtypes = [p, i64, i64, p]
        L.fmo_load.restype = p
        L.fmo_load.argtypes = [C.c_char_p, C.c_int]
        L.fmo_free.argtypes = [p]
        for name in ("fmo_n", "fmo_eof"):
            getattr(L, name).restype = i64
            getattr(L, name).argtypes = [p]
        L.fmo_bwt.restype = p
        L.fmo_bwt.argtypes = [p]
        L.fmo_fm.restype = p
        L.fmo_fm.argtypes = [p]
        L.fmo_cf.restype = i64
        L.fmo_cf.argtypes = [p, C.c_int]
        L.fmo_occ.restype = i64
        L.fmo_occ.argtypes = [p, C.c_int, i64]
        L.fmo_prev_range.restype = C.c_int
        L.fmo_prev_range.argtypes = [p, i64, i64, C.c_int, C.POINTER(i64), C.POINTER(i64)]
        L.fmo_search.restype = C.c_int
        L.fmo_search.argtypes = [p, p, i64, C.POINTER(i64), C.POINTER(i64)]
        L.fmo_interval_prev_range.restype = i64
        L.fmo_interval_prev_range.argtypes = [p, i64, i64, C.c_int, C.c_int, p, p, p]
        L.fmo_get_prev_i.restype = i64
        L.fmo_get_prev_i.argtypes = [p, i64]
        L.fmo_get_next_i.restype = i64
        L.fmo_get_next_i.argtypes = [p, i64]
        L.fmo_pos2char.restype = C.c_int
        L.fmo_pos2char.argtypes = [p, i64]
        L.fmo_next_substr.restype = i64
        L.fmo_next_substr.argtypes = [p, i64, i64, p]
        L.fmo_prev_substr.restype = i64
        L.fmo_prev_substr.argtypes = [p, i64, i64, p]
        L.fmo_build_sa.restype = p
        L.fmo_build_sa.argtypes = [p]
        L.fmo_build_lcp.argtypes = [p, p]
        L.fmo_build_lcp.restype = None
        L.fmo_locate.restype = i64
        L.fmo_locate.argtypes = [p, i64, i64, p]
        L.fmo_count_batch.argtypes = [p, p, p, i64, p, p, C.c_int]
        L.fmo_regex_match.restype = i64
        L.fmo_regex_match.argtypes = [p, i32, p, p, p, p, p, i32, i64, p, p, p, i64, C.POINTER(i64), C.c_int, i64]
        L.fmo_build_bwt.restype = C.c_int
        L.fmo_build_bwt.argtypes = [p, i64, p, C.POINTER(i64), p]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def build_bwt(text_rev):
    """BWT of text_rev+'$' ('$' smallest).  text_rev: bytes/uint8 array of T' WITHOUT the terminator.
    Returns (bwt uint8[n] with 0 at eof, eof, counts int64[256])."""
    t = np.ascontiguousarray(np.frombuffer(bytes(text_rev), dtype=np.uint8) if not isinstance(text_rev, np.ndarray) else text_rev, dtype=np.uint8)
    n = len(t) + 1
    bwt = np.zeros(n, dtype=np.uint8)
    cnt = np.zeros(256, dtype=np.int64)
    eof = C.c_int64(0)
    lib().fmo_build_bwt(_ptr(t), len(t), _ptr(bwt), C.byref(eof), _ptr(cnt))
    return bwt, int(eof.value), cnt


def file_to_text_rev(data):
    """FileBWTReader.copyReverse, M/bwtreader.scala:196-211: drop 0x00 bytes, reverse."""
    a = np.frombuffer(bytes(data), dtype=np.uint8)
    a = a[a > 0]
    return np.ascontiguousarray(a[::-1])


def write_index_files(base, bwt, eof, cnt, big_endian=True, write_fm=False):
    """Writes <base>.bwt/.aux (+ .fm) in the reference's on-disk layout (SURVEY Appendix A.1)."""
    bo = ">" if big_endian else "<"
    n = len(bwt)
    with open(base + ".bwt", "wb") as f:
        f.write(np.array([n, eof], dtype=bo + "i8").tobytes())
        f.write(np.asarray(bwt, dtype=np.uint8).tobytes())
    c = np.array(cnt, dtype=np.int64).copy()
    with open(base + ".aux", "wb") as f:
        f.write(c.astype(bo + "i8").tobytes())
    if write_fm:
        b = np.asarray(bwt, dtype=np.uint8).copy()
        b[eof] = 0
        fm = np.argsort(b, kind="stable").astype(">u4")       # == FMCreator placement (A.1)
        with open(base + ".fm", "wb") as f:
            f.write(bytes([4]))
            f.write(np.array([n], dtype=">i8").tobytes())      # RandomAccessFile.writeLong: always BE
            f.write(fm.tobytes())


class OracleIndex:
    """Mirror of NaiveFMSearcher (M/bwtmerger.scala:335-421) + SuffixAlgo (M/findex.scala:9-52)."""

    def __init__(self, handle):
        if not handle:
            raise RuntimeError(lib().fmo_last_error().decode())
        self.h = handle
        self.n = lib().fmo_n(handle)
        self.eof = lib().fmo_eof(handle)

    @classmethod
    def load(cls, base, big_endian=True):
        base = os.path.splitext(base)[0] if os.path.splitext(base)[1] in (".bwt", ".aux", ".fm") else base
        return cls(lib().fmo_load(base.encode(), 1 if big_endian else 0))

    @classmethod
    def from_bwt(cls, bwt, eof, cnt=None):
        b = np.ascontiguousarray(bwt, dtype=np.uint8)
        c = None if cnt is None else np.ascontiguousarray(cnt, dtype=np.int64)
        return cls(lib().fmo_from_memory(_ptr(b), len(b), eof, None if c is None else _ptr(c)))

    @classmethod
    def from_text_rev(cls, text_rev):
        bwt, eof, cnt = build_bwt(text_rev)
        return cls.from_bwt(bwt, eof, cnt)

    def close(self):
        if self.h:
            lib().fmo_free(self.h)
            self.h = None

    def bwt(self):
        return np.ctypeslib.as_array(C.cast(lib().fmo_bwt(self.h), C.POINTER(C.c_uint8)), shape=(self.n,))

    def fm(self):
        return np.ctypeslib.as_array(C.cast(lib().fmo_fm(self.h), C.POINTER(C.c_uint32)), shape=(self.n,))

    def cf(self, c):
        return lib().fmo_cf(self.h, int(c))

    def occ(self, c, key):
        return lib().fmo_occ(self.h, int(c), int(key))

    def search(self, pat):
        pat = bytes(pat)
        a = np.frombuffer(pat, dtype=np.uint8) if pat else np.zeros(1, np.uint8)
        sp, ep = C.c_int64(), C.c_int64()
        hit = lib().fmo_search(self.h, _ptr(a), len(pat), C.byref(sp), C.byref(ep))
        return (sp.value, ep.value) if hit else None

    def getPrevRange(self, sp, ep, c):
        a, b = C.c_int64(), C.c_int64()
        hit = lib().fmo_prev_range(self.h, sp, ep, int(c), C.byref(a), C.byref(b))
        return (a.value, b.value) if hit else None

    def prev_range_raw(self, sp, ep, c):
        a, b = C.c_int64(), C.c_int64()
        lib().fmo_prev_range(self.h, sp, ep, int(c), C.byref(a), C.byref(b))
        return a.value, b.value

    def getIntervalPrevRange(self, sp, ep, cstart, cend):
        k = max(0, cend - cstart + 1)
        oc = np.zeros(k, np.int32)
        osp = np.zeros(k, np.int64)
        oep = np.zeros(k, np.int64)
        m = lib().fmo_interval_prev_range(self.h, sp, ep, cstart, cend, _ptr(oc), _ptr(osp), _ptr(oep))
        return [(int(osp[i]), int(oep[i])) for i in range(m)], [int(x) for x in oc[:m]]

    def getPrevI(self, i):
        return lib().fmo_get_prev_i(self.h, i)

    def getNextI(self, i):
        return lib().fmo_get_next_i(self.h, i)

    def pos2char(self, k):
        return lib().fmo_pos2char(self.h, k)

    def nextSubstr(self, sp, ln):
        out = np.zeros(max(ln, 1), np.uint8)
        k = lib().fmo_next_substr(self.h, sp, ln, _ptr(out))
        return out[:k].tobytes()

    def prevSubstr(self, sp, ln):
        out = np.zeros(max(ln, 1), np.uint8)
        k = lib().fmo_prev_substr(self.h, sp, ln, _ptr(out))
        return out[:k].tobytes()

    def sa(self):
        return np.ctypeslib.as_array(C.cast(lib().fmo_build_sa(self.h), C.POINTER(C.c_uint32)), shape=(self.n,))

    def lcp(self):
        """bwtFm2LCP (M/util.scala:153-212): int32[n], LCP[r] = lcp(suffix of row r, suffix of row r+1), LCP[n-1] = 0 (never written);
        LCPCreator's .lcp file holds the first max(n-1, 1) entries, big-endian int32 (M/bwtmerger.scala:583-650, LCPLoader :176-211)."""
        out = np.zeros(self.n, np.int32)
        lib().fmo_build_lcp(self.h, _ptr(out))
        return out

    def locate(self, sp, ep):
        out = np.zeros(max(ep - sp, 1), np.int64)
        k = lib().fmo_locate(self.h, sp, ep, _ptr(out))
        return out[:k].copy()

    def count_batch(self, pat, off, threads=1):
        pat = np.ascontiguousarray(pat, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.int64)
        m = len(off) - 1
        sp = np.zeros(m, np.int64)
        ep = np.zeros(m, np.int64)
        if len(pat) == 0:
            pat = np.zeros(1, np.uint8)
        lib().fmo_count_batch(self.h, _ptr(pat), _ptr(off), m, _ptr(sp), _ptr(ep), threads)
        return sp, ep

    # ---- Glushkov regex over the index: ReTree.matchSA uncapped (M/re2/retree.scala:570-653)
    def regex_match_tables(self, tb, max_expansions=0, stop_on_emit=True, max_len=0):
        nst = len(tb["c"])
        if nst == 0 or not tb["firsts"]:
            return [], 0
        c = np.array(tb["c"], np.uint8)
        last = np.array(tb["last"], np.uint8)
        off = np.zeros(nst + 1, np.int32)
        for i, f in enumerate(tb["follows"]):
            off[i + 1] = off[i] + len(f)
        fol = np.array([x for f in tb["follows"] for x in f] or [0], np.int32)
        fst = np.array(tb["firsts"], np.int32)
        cap = 1 << 16
        while True:
            ol = np.zeros(cap, np.int32)
            osp = np.zeros(cap, np.int64)
            oep = np.zeros(cap, np.int64)
            nexp = C.c_int64(0)
            k = lib().fmo_regex_match(self.h, nst, _ptr(c), _ptr(last), _ptr(off), _ptr(fol), _ptr(fst), len(fst),
                                      cap, _ptr(ol), _ptr(osp), _ptr(oep), max_expansions, C.byref(nexp), 1 if stop_on_emit else 0, max_len)
            if k == -2:
                raise RuntimeError("regex traversal exceeded max_expansions")
            if k <= cap:
                break
            cap = int(k)
        res = sorted(zip(ol[:k].tolist(), osp[:k].tolist(), oep[:k].tolist()))
        return res, int(nexp.value)

    def regex_match(self, regex, line_only=False, max_expansions=0):
        """sorted multiset of (len, sp, ep) — the parity object of SURVEY §8(a) a13."""
        t = retree.compile_regex(regex, line_only)
        return self.regex_match_tables(t.tables(), max_expansions)[0]

    def regex_match_thompson(self, regex, line_only=False, max_expansions=0, max_len=0):
        """REParser.matchSA(createNFA(re2post(regex)), sa, maxIterations = 0, maxLength = max_len) (M/re2/re2.scala:568-693): sorted
        (len, sp, ep)."""
        tb = retree.compile_thompson(regex, line_only)
        return self.regex_match_tables(tb, max_expansions, stop_on_emit=False, max_len=max_len)[0]

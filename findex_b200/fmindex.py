"""
findex_b200.fmindex — host-side mirror of the reference's operator interface over the libfmgpu C ABI.

The reference's interface for this path is the Scala trait pair SuffixAlgo / SuffixWalkingAlgo
(src/main/scala/org/fmindex/findex.scala:9-57) implemented by NaiveFMSearcher (bwtmerger.scala:335-421) and
consumed by ReTree.matchSA (re2/retree.scala:570).  `GpuFMSearcher` keeps those member names and meanings
(n, cf, occ, search, getPrevRange, getIntervalPrevRange, getPrevI, getNextI, pos2char, nextSubstr, prevSubstr)
and adds the batched calls the GPU wants.  Everything computes on the GPU through include/fmgpu.h; there is
no CPU fallback — a missing library or device raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libfmgpu.so")

FMX_OK, FMX_E_IO, FMX_E_FORMAT, FMX_E_CUDA, FMX_E_ARG = 0, -1, -2, -3, -4
FMX_E_CAPACITY, FMX_E_SYNTAX, FMX_E_UNSUPPORTED, FMX_E_LIMIT = -5, -6, -7, -8
LAYOUT_AUTO, LAYOUT_WM, LAYOUT_PLANES, LAYOUT_WMX = 0, 1, 2, 3
ACCEL_AUTO, ACCEL_KMER, ACCEL_TEXT, ACCEL_CTX, ACCEL_NONE, ACCEL_CTX8, ACCEL_NO_SA, ACCEL_DICT = 0, 1, 2, 4, 8, 16, 32, 64


class FmxError(Exception):
    def __init__(self, code, msg):
        super().__init__("%s (code %d)" % (msg, code))
        self.code = code


class ReSyntaxError(FmxError):
    """Exception("re2post syntax") in the reference."""


class ReUnsupported(FmxError):
    """MatchError / NoSuchElementException in the reference's ReTree.apply."""


class fmx_opts(C.Structure):
    _fields_ = [("device", C.c_int32), ("layout", C.c_int32), ("sa_sample_rate", C.c_int32), ("require_fm", C.c_int32),
                ("max_index_bytes", C.c_int64), ("lanes_per_query", C.c_int32), ("accel", C.c_int32), ("kmer_table_bytes", C.c_int64),
                ("max_total_bytes", C.c_int64), ("dict_bytes", C.c_int64), ("dict_min_rows", C.c_int32), ("dict_top_min_rows", C.c_int32),
                ("text_sample_rate", C.c_int32), ("lcp", C.c_int32)]


_lib = None


def lib():
    """Loads libfmgpu.so (built by findex_b200.build).  Raises if it is missing: no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise ImportError("libfmgpu.so is not built (run `python -m findex_b200.build`); there is no CPU fallback")
    L = C.CDLL(_SO)
    p, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    pp = C.POINTER(C.c_void_p)
    L.fmx_last_error.restype = C.c_char_p
    L.fmx_version.restype = C.c_char_p
    L.fmx_opts_default.argtypes = [C.POINTER(fmx_opts)]
    L.fmx_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(fmx_opts), pp]
    L.fmx_open_mem.argtypes = [p, i64, i64, p, C.POINTER(fmx_opts), pp]
    L.fmx_close.argtypes = [p]
    L.fmx_n.restype = i64
    L.fmx_n.argtypes = [p]
    L.fmx_eof.restype = i64
    L.fmx_eof.argtypes = [p]
    L.fmx_ctable.argtypes = [p, p]
    L.fmx_info.argtypes = [p, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i64), C.POINTER(i32)]
    L.fmx_accel_info.argtypes = [p, C.POINTER(i32), C.POINTER(i32)]
    L.fmx_get_lanes.argtypes = [p]
    L.fmx_ctx_depth.argtypes = [p]
    L.fmx_kmer_rows.argtypes = [p]
    L.fmx_dict_info.argtypes = [p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    L.fmx_ctx_entry_bytes.argtypes = [p]
    L.fmx_occ_batch.argtypes = [p, p, p, i64, p]
    L.fmx_prev_range_batch.argtypes = [p, p, p, p, i64, p, p]
    L.fmx_interval_prev_range.argtypes = [p, i64, i64, C.c_int, C.c_int, p, p, p, C.POINTER(i64)]
    L.fmx_count_batch.argtypes = [p, p, p, i64, p, p]
    L.fmx_count_fixed.argtypes = [p, p, i32, i64, p, p]
    L.fmx_count_only_fixed.argtypes = [p, p, i32, i64, p]
    L.fmx_count_fixed_i32.argtypes = [p, p, i32, i64, p, p]
    L.fmx_count_fixed_packed2.argtypes = [p, p, p, i32, i64, p, p, i32]
    L.fmx_count_fixed_dev.argtypes = [p, p, i32, i64, p, p, p]
    L.fmx_count_fixed_dev_gather.argtypes = [p, p, i32, i64, p, p, p, i32, i64, p]
    L.fmx_dev_alloc.argtypes = [pp, i64]
    L.fmx_dev_free.argtypes = [p]
    L.fmx_ipc_export.argtypes = [p, p]
    L.fmx_ipc_import.argtypes = [p, pp]
    L.fmx_ipc_close.argtypes = [p]
    L.fmx_memcpy_d2h.argtypes = [p, p, i64]
    L.fmx_locate_batch.argtypes = [p, p, p, i64, i64, p, p]
    L.fmx_locate_dev.argtypes = [p, p, p, i64, p, p, i64, C.POINTER(i64), p]
    L.fmx_last_locate_ms.argtypes = [p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.fmx_scatter_dev.argtypes = [p, i64, p, i32, i64, p, i64, p]
    L.fmx_regex_set_search_dev.argtypes = [p, p, p, i64, p, C.POINTER(i64)]
    L.fmx_regex_set_ring.argtypes = [p, i64]
    L.fmx_regex_set_limits.argtypes = [p, i64]
    L.fmx_set_locate_slab.argtypes = [i64]
    L.fmx_set_stats.argtypes = [p, i32]
    L.fmx_last_steps.argtypes = [p]
    L.fmx_last_steps.restype = i64
    L.fmx_get_prev_i_batch.argtypes = [p, p, i64, p]
    L.fmx_get_next_i_batch.argtypes = [p, p, i64, p]
    L.fmx_pos2char.argtypes = [p, i64, C.POINTER(i32)]
    L.fmx_prev_substr_batch.argtypes = [p, p, i64, i32, p, p]
    L.fmx_text_sample_rate.argtypes = [p]
    L.fmx_text_batch.argtypes = [p, p, i64, i32, p, p]
    L.fmx_text_dev.argtypes = [p, p, i64, i32, p, p, p]
    L.fmx_next_substr_batch.argtypes = [p, p, i64, i32, p, p]
    L.fmx_lcp_bytes.restype = i64
    L.fmx_lcp_bytes.argtypes = [p]
    L.fmx_match_stats_batch.argtypes = [p, p, p, i64, p, p, p]
    L.fmx_smem_batch.argtypes = [p, p, p, i64, i32, i64, p, p, p, p, p]
    L.fmx_smem_dev.argtypes = [p, p, p, i64, i32, p, p, p, p, p, i64, C.POINTER(i64), p]
    L.fmx_last_match_requests.argtypes = [p, p]
    L.fmx_kmer_spectrum.argtypes = [p, i32, i32, p, C.POINTER(i64), C.POINTER(i64)]
    L.fmx_kmer_list_batch.argtypes = [p, i32, i64, i64, i64, C.POINTER(i64), p, p]
    L.fmx_kmer_list_dev.argtypes = [p, i32, i64, i64, p, p, i64, C.POINTER(i64), p]
    L.fmx_regex_compile.argtypes = [p, i64, C.c_int, pp]
    L.fmx_regex_compile_engine.argtypes = [p, i64, C.c_int, C.c_int, pp]
    L.fmx_regex_free.argtypes = [p]
    L.fmx_regex_free.restype = None
    L.fmx_regex_tables.argtypes = [p, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), p, p, p, p, p, p]
    L.fmx_regex_search_batch.argtypes = [p, p, i64, i64, p, p, p, p]
    L.fmx_regex_set_create.argtypes = [p, p, i64, pp]
    L.fmx_regex_set_search.argtypes = [p, p, i64, p, p, p, p]
    L.fmx_regex_set_free.argtypes = [p]
    L.fmx_regex_set_free.restype = None
    L.fmx_count_fixed_stats.argtypes = [p, p, i32, i64, C.POINTER(i64), C.POINTER(i64)]
    L.fmx_gather_bench.argtypes = [p, i32, i32, i64, i32, i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.fmx_set_lanes.argtypes = [p, i32]
    L.fmx_set_chunk.argtypes = [p, i64]
    L.fmx_set_accel_mask.argtypes = [p, i32]
    L.fmx_set_l2_fetch_granularity.argtypes = [i32, C.POINTER(i32)]
    L.fmx_host_alloc.argtypes = [pp, i64]
    L.fmx_host_free.argtypes = [p]
    L.fmx_last_kernel_ms.restype = C.c_double
    L.fmx_last_kernel_ms.argtypes = [p]
    L.fmx_last_kernel_launches.restype = i64
    L.fmx_last_kernel_launches.argtypes = [p]
    L.fmx_last_regex_levels.restype = i64
    L.fmx_last_regex_levels.argtypes = [p]
    L.fmx_build_index_files.argtypes = [p, i64, C.c_char_p, C.c_int, C.c_int, C.c_int]
    L.fmx_build_bwt.argtypes = [p, i64, p, C.POINTER(i64), C.POINTER(i64), p, C.c_int]
    _lib = L
    return L


def _check(rc):
    if rc == FMX_OK:
        return
    msg = lib().fmx_last_error().decode("latin-1")
    if rc == FMX_E_SYNTAX:
        raise ReSyntaxError(rc, msg)
    if rc == FMX_E_UNSUPPORTED:
        raise ReUnsupported(rc, msg)
    raise FmxError(rc, msg)


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def _u8(a):
    if isinstance(a, (bytes, bytearray)):
        return np.frombuffer(bytes(a), dtype=np.uint8)
    return np.ascontiguousarray(a, dtype=np.uint8)


def make_opts(device=-1, layout=LAYOUT_AUTO, sa_sample_rate=0, require_fm=False, max_index_bytes=0, lanes_per_query=0, accel=ACCEL_AUTO,
              kmer_table_bytes=0, max_total_bytes=0, dict_bytes=0, dict_min_rows=0, dict_top_min_rows=0, text_sample_rate=0, lcp=0):
    o = fmx_opts()
    lib().fmx_opts_default(C.byref(o))
    o.device, o.layout, o.sa_sample_rate = device, layout, sa_sample_rate
    o.require_fm, o.max_index_bytes, o.lanes_per_query, o.accel = int(require_fm), max_index_bytes, lanes_per_query, accel
    o.kmer_table_bytes = kmer_table_bytes
    o.max_total_bytes = max_total_bytes
    o.dict_bytes, o.dict_min_rows, o.dict_top_min_rows = dict_bytes, dict_min_rows, dict_top_min_rows
    o.text_sample_rate = text_sample_rate
    o.lcp = int(lcp)
    return o


class ReTree:
    """ReTree(REParser.re2post(regex, lineOnly)) — re2.scala:50-185 + retree.scala:156-370, compiled by libfmgpu."""

    ENGINE = 0

    def __init__(self, regex, lineOnly=False):
        if isinstance(regex, str):
            regex = regex.encode("latin-1")
        self.regex = bytes(regex)
        h = C.c_void_p()
        buf = _u8(self.regex) if self.regex else np.zeros(1, np.uint8)
        _check(lib().fmx_regex_compile_engine(_ptr(buf), len(self.regex), int(lineOnly), self.ENGINE, C.byref(h)))
        self.h = h

    def __del__(self):
        try:
            if getattr(self, "h", None):
                lib().fmx_regex_free(self.h)
                self.h = None
        except Exception:
            pass

    def tables(self):
        ns, nf, n1 = C.c_int32(), C.c_int32(), C.c_int32()
        _check(lib().fmx_regex_tables(self.h, C.byref(ns), C.byref(nf), C.byref(n1), None, None, None, None, None, None))
        c = np.zeros(max(ns.value, 1), np.uint8)
        last = np.zeros(max(ns.value, 1), np.uint8)
        num = np.zeros(max(ns.value, 1), np.int32)
        off = np.zeros(ns.value + 1, np.int32)
        fol = np.zeros(max(nf.value, 1), np.int32)
        fst = np.zeros(max(n1.value, 1), np.int32)
        _check(lib().fmx_regex_tables(self.h, None, None, None, _ptr(c), _ptr(last), _ptr(num), _ptr(off), _ptr(fol), _ptr(fst)))
        n = ns.value
        return {"c": c[:n].tolist(), "last": last[:n].tolist(), "num": num[:n].tolist(),
                "follows": [fol[off[i]:off[i + 1]].tolist() for i in range(n)], "firsts": fst[:n1.value].tolist()}

    def matchSA(self, sa):
        """ReTree.matchSA with the caps disabled: sorted list of (len, sp, ep)."""
        return sa.regex_search_batch([self])[0]


class RegexSet:
    """fmx_regex_set: the concatenated automata of a batch, resident on the searcher's device."""

    def __init__(self, searcher, trees):
        self.m = len(trees)
        arr = (C.c_void_p * max(self.m, 1))(*[t.h for t in trees])
        h = C.c_void_p()
        _check(lib().fmx_regex_set_create(searcher.h, arr, self.m, C.byref(h)))
        self.h = h

    def search(self, searcher, cap_total=1 << 20):
        m = self.m
        off = np.zeros(m + 1, np.int64)
        while True:
            ln = np.zeros(max(cap_total, 1), np.int32)
            sp = np.zeros(max(cap_total, 1), np.int64)
            ep = np.zeros(max(cap_total, 1), np.int64)
            rc = lib().fmx_regex_set_search(searcher.h, self.h, cap_total, _ptr(off), _ptr(ln), _ptr(sp), _ptr(ep))
            if rc == FMX_E_CAPACITY:
                cap_total = int(off[m])
                continue
            _check(rc)
            return off, ln[:off[m]], sp[:off[m]], ep[:off[m]]

    def set_limits(self, max_len=0):
        """REParser.matchSA's maxLength for later searches of this set (0 = off)"""
        _check(lib().fmx_regex_set_limits(self.h, max_len))

    def set_ring(self, slots):
        _check(lib().fmx_regex_set_ring(self.h, slots))

    def search_dev(self, searcher, d_res, cap, d_off=0):
        """device-resident results: {regex, len, sp, ep} uint32 records ordered by (regex, len, sp, ep); returns their number"""
        total = C.c_int64()
        _check(lib().fmx_regex_set_search_dev(searcher.h, self.h, C.c_void_p(d_res), cap, C.c_void_p(d_off), C.byref(total)))
        return total.value

    def close(self):
        if getattr(self, "h", None):
            lib().fmx_regex_set_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ThompsonNFA(ReTree):
    """REParser.createNFA(REParser.re2post(regex, lineOnly)) — re2.scala:264-334; matchSA = REParser.matchSA uncapped."""
    ENGINE = 1


class GpuFMSearcher:
    """new NaiveFMSearcher(filename, bigEndian) — on the GPU."""

    def __init__(self, filename=None, bigEndian=True, *, bwt=None, eof=None, counts=None, **opts):
        o = make_opts(**opts)
        h = C.c_void_p()
        if filename is not None:
            _check(lib().fmx_open(os.fsencode(filename), int(bigEndian), C.byref(o), C.byref(h)))
        else:
            b = _u8(bwt)
            c = _i64(counts)
            _check(lib().fmx_open_mem(_ptr(b), len(b), int(eof), _ptr(c), C.byref(o), C.byref(h)))
        self.h = h
        self.n = lib().fmx_n(h)
        self.eof = lib().fmx_eof(h)
        ct = np.zeros(256, np.int64)
        _check(lib().fmx_ctable(h, _ptr(ct)))
        self._C = ct

    def close(self):
        if getattr(self, "h", None):
            lib().fmx_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        lay, lev, sig, rate, nb = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
        _check(lib().fmx_info(self.h, C.byref(lay), C.byref(lev), C.byref(sig), C.byref(nb), C.byref(rate)))
        k, t = C.c_int32(), C.c_int32()
        _check(lib().fmx_accel_info(self.h, C.byref(k), C.byref(t)))
        dd, dx, de, db = C.c_int32(), C.c_int32(), C.c_int64(), C.c_int64()
        _check(lib().fmx_dict_info(self.h, C.byref(dd), C.byref(dx), C.byref(de), C.byref(db)))
        return {"layout": {1: "wm", 2: "planes", 3: "wmx"}[lay.value], "levels": lev.value, "sigma": sig.value,
                "dict_depth": dd.value, "dict_chain_depth": dx.value, "dict_entries": de.value, "dict_bytes": db.value,
                "index_bytes": nb.value, "sa_sample_rate": rate.value, "kmer_k": k.value, "kmer_rows": lib().fmx_kmer_rows(self.h), "text_shortcut": bool(t.value),
                "ctx_depth": lib().fmx_ctx_depth(self.h), "ctx_entry_bytes": lib().fmx_ctx_entry_bytes(self.h),
                "lanes_per_query": lib().fmx_get_lanes(self.h), "text_sample_rate": lib().fmx_text_sample_rate(self.h),
                "lcp_bytes": lib().fmx_lcp_bytes(self.h)}

    # ---- scalar trait members (each is a batch of one) -------------------------------------------------
    def cf(self, c):
        return int(self._C[c])

    def occ(self, c, key):
        return int(self.occ_batch([c], [key])[0])

    def search(self, pat):
        sp, ep = self.count_batch([bytes(pat)])
        return (int(sp[0]), int(ep[0])) if sp[0] < ep[0] else None

    def getPrevRange(self, sp, ep, c):
        a, b = self.prev_range_batch([sp], [ep], [c])
        return (int(a[0]), int(b[0])) if a[0] < b[0] else None

    def getIntervalPrevRange(self, sp, ep, cstart, cend):
        k = max(cend - cstart + 1, 1)
        oc, osp, oep = np.zeros(k, np.int32), np.zeros(k, np.int64), np.zeros(k, np.int64)
        m = C.c_int64()
        _check(lib().fmx_interval_prev_range(self.h, sp, ep, cstart, cend, _ptr(oc), _ptr(osp), _ptr(oep), C.byref(m)))
        return [(int(osp[i]), int(oep[i])) for i in range(m.value)]

    def getPrevI(self, i):
        return int(self.get_prev_i_batch([i])[0])

    def getNextI(self, i):
        return int(self.get_next_i_batch([i])[0])

    def pos2char(self, key):
        c = C.c_int32()
        _check(lib().fmx_pos2char(self.h, key, C.byref(c)))
        return c.value

    def prevSubstr(self, sp, ln):
        return self.prev_substr_batch([sp], ln)[0]

    def nextSubstr(self, sp, ln):
        return self.next_substr_batch([sp], ln)[0]

    # ---- batched calls ---------------------------------------------------------------------------------------
    def occ_batch(self, c, key):
        c, key = _u8(c), _i64(key)
        out = np.zeros(len(key), np.int64)
        _check(lib().fmx_occ_batch(self.h, _ptr(c), _ptr(key), len(key), _ptr(out)))
        return out

    def prev_range_batch(self, sp, ep, c):
        sp, ep, c = _i64(sp), _i64(ep), _u8(c)
        a, b = np.zeros(len(sp), np.int64), np.zeros(len(sp), np.int64)
        _check(lib().fmx_prev_range_batch(self.h, _ptr(sp), _ptr(ep), _ptr(c), len(sp), _ptr(a), _ptr(b)))
        return a, b

    def count_batch(self, patterns):
        """patterns: list of bytes.  Returns (sp, ep) int64 arrays; None is (0,0)."""
        off = np.zeros(len(patterns) + 1, np.int64)
        np.cumsum([len(x) for x in patterns], out=off[1:])
        pat = _u8(b"".join(bytes(x) for x in patterns)) if off[-1] else np.zeros(1, np.uint8)
        return self.count_offsets(pat, off)

    def count_offsets(self, pat, off):
        pat, off = _u8(pat), _i64(off)
        m = len(off) - 1
        sp, ep = np.zeros(m, np.int64), np.zeros(m, np.int64)
        _check(lib().fmx_count_batch(self.h, _ptr(pat), _ptr(off), m, _ptr(sp), _ptr(ep)))
        return sp, ep

    def count_fixed(self, pat2d):
        """pat2d: uint8 array [m, len]."""
        pat2d = np.ascontiguousarray(pat2d, dtype=np.uint8)
        m, ln = pat2d.shape
        sp, ep = np.zeros(m, np.int64), np.zeros(m, np.int64)
        _check(lib().fmx_count_fixed(self.h, _ptr(pat2d), ln, m, _ptr(sp), _ptr(ep)))
        return sp, ep

    def count_fixed_dev(self, d_pat, ln, m, d_sp, d_ep, stream=0):
        """Raw device pointers (ints); asynchronous on `stream`."""
        _check(lib().fmx_count_fixed_dev(self.h, C.c_void_p(d_pat), ln, m, C.c_void_p(d_sp), C.c_void_p(d_ep), C.c_void_p(stream)))

    def count_fixed_dev_gather(self, d_pat, ln, m, d_sp, d_ep, sinks, offset, stream=0):
        """Fused count + exchange: `sinks` = device pointers (ints) of every rank's gathered uint32 buffer."""
        arr = (C.c_void_p * max(len(sinks), 1))(*sinks)
        _check(lib().fmx_count_fixed_dev_gather(self.h, C.c_void_p(d_pat), ln, m, C.c_void_p(d_sp), C.c_void_p(d_ep), arr, len(sinks), offset,
                                                C.c_void_p(stream)))

    def count_fixed_stats(self, pat2d):
        pat2d = np.ascontiguousarray(pat2d, dtype=np.uint8)
        m, ln = pat2d.shape
        blocks, steps = C.c_int64(), C.c_int64()
        _check(lib().fmx_count_fixed_stats(self.h, _ptr(pat2d), ln, m, C.byref(blocks), C.byref(steps)))
        return blocks.value, steps.value

    def locate_batch(self, sp, ep):
        """Returns (off[m+1], pos) — pos ascending inside each query (T' coordinates)."""
        sp, ep = _i64(sp), _i64(ep)
        m = len(sp)
        total = int(np.maximum(ep - sp, 0).sum())
        off = np.zeros(m + 1, np.int64)
        pos = np.zeros(max(total, 1), np.int64)
        _check(lib().fmx_locate_batch(self.h, _ptr(sp), _ptr(ep), m, total, _ptr(off), _ptr(pos)))
        return off, pos[:total]

    def locate_dev(self, d_sp, d_ep, m, d_off, d_pos, cap, stream=0):
        """Device-resident locate (raw device pointers as ints): uint32 sp/ep in, int64 offsets [m+1] and uint32 positions out.
        Returns the number of positions; raises FmxError(FMX_E_CAPACITY) when cap is too small."""
        total = C.c_int64()
        _check(lib().fmx_locate_dev(self.h, C.c_void_p(d_sp), C.c_void_p(d_ep), m, C.c_void_p(d_off), C.c_void_p(d_pos), cap, C.byref(total),
                                    C.c_void_p(stream)))
        return total.value

    def set_stats(self, on):
        _check(lib().fmx_set_stats(self.h, int(on)))

    def last_steps(self):
        """LF steps of the last locate call (with set_stats(True)) / items of the last regex search"""
        return lib().fmx_last_steps(self.h)

    def last_locate_ms(self):
        """(LF-walk ms, per-query sort ms) of the last locate call"""
        a, b = C.c_double(), C.c_double()
        _check(lib().fmx_last_locate_ms(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def get_prev_i_batch(self, rows):
        rows = _i64(rows)
        out = np.zeros(len(rows), np.int64)
        _check(lib().fmx_get_prev_i_batch(self.h, _ptr(rows), len(rows), _ptr(out)))
        return out

    def get_next_i_batch(self, rows):
        rows = _i64(rows)
        out = np.zeros(len(rows), np.int64)
        _check(lib().fmx_get_next_i_batch(self.h, _ptr(rows), len(rows), _ptr(out)))
        return out

    def prev_substr_batch(self, rows, ln):
        rows = _i64(rows)
        out = np.zeros((len(rows), max(ln, 1)), np.uint8)
        olen = np.zeros(len(rows), np.int32)
        _check(lib().fmx_prev_substr_batch(self.h, _ptr(rows), len(rows), ln, _ptr(out), _ptr(olen)))
        return [out[i, :olen[i]].tobytes() for i in range(len(rows))]

    def next_substr_batch(self, rows, ln):
        rows = _i64(rows)
        out = np.zeros((len(rows), max(ln, 1)), np.uint8)
        olen = np.zeros(len(rows), np.int32)
        _check(lib().fmx_next_substr_batch(self.h, _ptr(rows), len(rows), ln, _ptr(out), _ptr(olen)))
        return [out[i, :olen[i]].tobytes() for i in range(len(rows))]

    def extract_batch(self, rows, ln, direction):
        """fmx_extract_batch: nextSubstr (direction > 0) or prevSubstr for a batch of rows"""
        rows = _i64(rows)
        out = np.zeros((len(rows), max(ln, 1)), np.uint8)
        olen = np.zeros(len(rows), np.int32)
        lib().fmx_extract_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
        _check(lib().fmx_extract_batch(self.h, _ptr(rows), len(rows), ln, direction, _ptr(out), _ptr(olen)))
        return [out[i, :olen[i]].tobytes() for i in range(len(rows))]

    def text(self, off, length):
        """the indexed file bytes F[off .. off+length) (0x00 dropped; shorter at the end of the text)"""
        return self.text_batch([off], length)[0]

    def text_batch(self, offs, length):
        """fmx_text_batch: F[off .. off+length) for every file offset in `offs` (0 <= off <= n-1); list of bytes"""
        offs = _i64(offs)
        out = np.zeros((len(offs), max(length, 1)), np.uint8)
        olen = np.zeros(len(offs), np.int32)
        _check(lib().fmx_text_batch(self.h, _ptr(offs), len(offs), length, _ptr(out), _ptr(olen)))
        return [out[i, :olen[i]].tobytes() for i in range(len(offs))]

    def text_dev(self, d_off, m, length, d_out, d_out_len, stream=0):
        """fmx_text_dev (raw device pointers as ints): uint32 file offsets [m] in, uint8 [m, length] rows and int32 lengths out;
        asynchronous on `stream`"""
        _check(lib().fmx_text_dev(self.h, C.c_void_p(d_off), m, length, C.c_void_p(d_out), C.c_void_p(d_out_len), C.c_void_p(stream)))

    # ---- longest matches (index opened with lcp=1; include/fmgpu.h) --------------------------------------------------------------------
    @staticmethod
    def _queries(queries):
        off = np.zeros(len(queries) + 1, np.int64)
        np.cumsum([len(x) for x in queries], out=off[1:])
        pat = _u8(b"".join(bytes(x) for x in queries)) if off[-1] else np.zeros(1, np.uint8)
        return pat, off

    def match_stats(self, queries, intervals=True):
        """fmx_match_stats_batch over queries in file order (list of bytes): (off[m+1], ms_len int32, ms_sp, ms_ep int64), entry off[q] + j
        for position j of query q; ms_len[i] = the longest l such that the l bytes ending there occur, (ms_sp, ms_ep) = count of their
        reverse ((0, n) when l = 0).  intervals=False skips the intervals (None)."""
        pat, off = self._queries(queries)
        T = int(off[-1])
        ln = np.zeros(max(T, 1), np.int32)
        sp = np.zeros(max(T, 1), np.int64) if intervals else None
        ep = np.zeros(max(T, 1), np.int64) if intervals else None
        _check(lib().fmx_match_stats_batch(self.h, _ptr(pat), _ptr(off), len(queries), _ptr(ln), None if sp is None else _ptr(sp),
                                           None if ep is None else _ptr(ep)))
        return off, ln[:T], (sp[:T] if intervals else None), (ep[:T] if intervals else None)

    def smems(self, queries, min_len=1, cap_total=1 << 20):
        """fmx_smem_batch: (out_off[m+1], start, len, sp, ep) — the SMEMs of at least min_len bytes of query q are entries
        out_off[q] .. out_off[q+1], in increasing start order; start is inside the query (file order)"""
        pat, off = self._queries(queries)
        m = len(queries)
        out_off = np.zeros(m + 1, np.int64)
        while True:
            k = max(cap_total, 1)
            st, ln, sp, ep = np.zeros(k, np.int32), np.zeros(k, np.int32), np.zeros(k, np.int64), np.zeros(k, np.int64)
            rc = lib().fmx_smem_batch(self.h, _ptr(pat), _ptr(off), m, min_len, cap_total, _ptr(out_off), _ptr(st), _ptr(ln), _ptr(sp), _ptr(ep))
            if rc == FMX_E_CAPACITY:
                cap_total = int(out_off[m])
                continue
            _check(rc)
            t = int(out_off[m])
            return out_off, st[:t], ln[:t], sp[:t], ep[:t]

    def smems_dev(self, d_pat, d_off, m, min_len, d_out_off, d_start, d_len, d_sp, d_ep, cap, stream=0):
        """fmx_smem_dev (raw device pointers as ints): uint8 queries and int64 offsets [m+1] in; int64 out_off [m+1], int32 start / len and
        uint32 sp / ep [cap] out.  Returns the number of SMEMs; raises FmxError(FMX_E_CAPACITY) when cap is too small."""
        total = C.c_int64()
        _check(lib().fmx_smem_dev(self.h, C.c_void_p(d_pat), C.c_void_p(d_off), m, min_len, C.c_void_p(d_out_off), C.c_void_p(d_start),
                                  C.c_void_p(d_len), C.c_void_p(d_sp), C.c_void_p(d_ep), cap, C.byref(total), C.c_void_p(stream)))
        return total.value

    def last_match_requests(self):
        """(rank blocks, LCP block / record / escape reads, minima lines) of the last match call with set_stats(True)"""
        r = np.zeros(3, np.int64)
        _check(lib().fmx_last_match_requests(self.h, _ptr(r)))
        return tuple(int(x) for x in r)

    # ---- k-mer census (index opened with lcp=1; include/fmgpu.h) -----------------------------------------------------------------------
    def kmer_spectrum(self, k, buckets):
        """fmx_kmer_spectrum: (hist int64[buckets], distinct, max_occ); hist[b] = distinct k-mers of F occurring exactly b+1 times, the last
        bucket those occurring >= buckets times"""
        hist = np.zeros(max(buckets, 1), np.int64)
        d, mx = C.c_int64(), C.c_int64()
        _check(lib().fmx_kmer_spectrum(self.h, k, buckets, _ptr(hist), C.byref(d), C.byref(mx)))
        return hist[:buckets], d.value, mx.value

    def kmers(self, k, min_count=1, max_count=0, text=False):
        """fmx_kmer_list_batch: (sp, ep) int64 of every distinct k-mer with min_count <= count <= max_count (0 = no bound), in row order
        (count = ep - sp).  text=True also returns the k-mers' bytes in file order: nextSubstr(sp, k) of each interval."""
        cap = min(self.n, 1 << 22)
        total = C.c_int64()
        while True:
            sp, ep = np.zeros(max(cap, 1), np.int64), np.zeros(max(cap, 1), np.int64)
            rc = lib().fmx_kmer_list_batch(self.h, k, min_count, max_count, cap, C.byref(total), _ptr(sp), _ptr(ep))
            if rc == FMX_E_CAPACITY:
                cap = total.value
                continue
            _check(rc)
            t = total.value
            sp, ep = sp[:t], ep[:t]
            if not text:
                return sp, ep
            return sp, ep, self.next_substr_batch(sp, k) if t else []

    def kmers_dev(self, k, d_sp, d_ep, cap, min_count=1, max_count=0, stream=0):
        """fmx_kmer_list_dev (raw device pointers as ints): uint32 sp / ep [cap] out, as locate_dev takes them.  Returns the number of
        k-mers listed; raises FmxError(FMX_E_CAPACITY) when cap is too small."""
        total = C.c_int64()
        _check(lib().fmx_kmer_list_dev(self.h, k, min_count, max_count, C.c_void_p(d_sp), C.c_void_p(d_ep), cap, C.byref(total), C.c_void_p(stream)))
        return total.value

    def top_kmers(self, k, t):
        """the t most frequent k-mers (fewer when there are fewer), by count descending, then sp ascending: (sp, ep) int64.  The threshold
        comes from the spectrum; the k-mers at or above it are listed and sorted here."""
        _, distinct, max_occ = self.kmer_spectrum(k, 1)
        if t <= 0 or distinct == 0:
            return np.zeros(0, np.int64), np.zeros(0, np.int64)
        buckets = min(max_occ, 1 << 16) + 1
        hist, _, _ = self.kmer_spectrum(k, buckets)
        above, threshold = 0, 1
        for b in range(buckets - 1, -1, -1):                     # the largest count c with at least t k-mers occurring >= c times
            above += int(hist[b])
            if above >= t:
                threshold = b + 1
                break
        sp, ep = self.kmers(k, min_count=threshold)
        order = np.lexsort((sp, -(ep - sp)))[:t]
        return sp[order], ep[order]

    def regex_search_batch(self, trees, cap_total=1 << 20):
        """trees: list of ReTree.  Returns per regex the sorted list of (len, sp, ep)."""
        m = len(trees)
        arr = (C.c_void_p * max(m, 1))(*[t.h for t in trees])
        off = np.zeros(m + 1, np.int64)
        while True:
            ln = np.zeros(max(cap_total, 1), np.int32)
            sp = np.zeros(max(cap_total, 1), np.int64)
            ep = np.zeros(max(cap_total, 1), np.int64)
            rc = lib().fmx_regex_search_batch(self.h, arr, m, cap_total, _ptr(off), _ptr(ln), _ptr(sp), _ptr(ep))
            if rc == FMX_E_CAPACITY:
                cap_total = int(off[m])
                continue
            _check(rc)
            break
        return [list(zip(ln[off[i]:off[i + 1]].tolist(), sp[off[i]:off[i + 1]].tolist(), ep[off[i]:off[i + 1]].tolist()))
                for i in range(m)]

    def regex_set(self, trees):
        """Device-resident batch of compiled regexes (compile once, search many times)."""
        return RegexSet(self, trees)

    def gather_bench(self, bytes_per_gather=64, lanes=4, gathers=1 << 24, chain=16, iters=3):
        gbs, ms = C.c_double(), C.c_double()
        _check(lib().fmx_gather_bench(self.h, bytes_per_gather, lanes, gathers, chain, iters, C.byref(gbs), C.byref(ms)))
        return gbs.value, ms.value

    def set_chunk(self, queries_per_chunk):
        _check(lib().fmx_set_chunk(self.h, queries_per_chunk))

    def count_fixed_into(self, pat2d, sp, ep):
        """Like count_fixed but into caller-owned arrays (pinned arrays make the copies asynchronous): int64, or int32 — the
        reference's own Int rows, half the result bytes over PCIe."""
        m, ln = pat2d.shape
        assert pat2d.flags.c_contiguous and pat2d.dtype == np.uint8 and sp.dtype == ep.dtype and sp.dtype in (np.int64, np.int32)
        assert len(sp) == m and len(ep) == m
        if sp.dtype == np.int32:
            _check(lib().fmx_count_fixed_i32(self.h, _ptr(pat2d), ln, m, _ptr(sp), _ptr(ep)))
        else:
            _check(lib().fmx_count_fixed(self.h, _ptr(pat2d), ln, m, _ptr(sp), _ptr(ep)))

    def pack2(self, pat2d):
        """2-bit codes of patterns over this index's (<= 4 symbol) alphabet, ceil(len/4) bytes per pattern; sets self.alphabet4"""
        syms = np.flatnonzero(np.diff(np.append(self._C, self.n))[1:] > 0) + 1          # bytes that occur in the text
        assert len(syms) <= 4, "packed upload needs an alphabet of at most 4 symbols"
        self.alphabet4 = np.zeros(4, np.uint8)
        self.alphabet4[:len(syms)] = syms
        lut = np.zeros(256, np.uint8)
        lut[syms] = np.arange(len(syms), dtype=np.uint8)
        m, ln = pat2d.shape
        pb = (ln + 3) // 4
        codes = np.zeros((m, pb * 4), np.uint8)
        codes[:, :ln] = lut[pat2d]
        c4 = codes.reshape(m, pb, 4)
        return (c4[:, :, 0] | (c4[:, :, 1] << 2) | (c4[:, :, 2] << 4) | (c4[:, :, 3] << 6)).astype(np.uint8)

    def count_packed2_into(self, codes, ln, sp, ep):
        """fmx_count_fixed_packed2: codes from pack2(); sp/ep uint32/int32 (4-byte rows) or int64"""
        m = codes.shape[0]
        assert codes.flags.c_contiguous and codes.dtype == np.uint8 and codes.shape[1] == (ln + 3) // 4 and sp.dtype == ep.dtype and len(sp) == m and len(ep) == m
        _check(lib().fmx_count_fixed_packed2(self.h, _ptr(codes), _ptr(self.alphabet4), ln, m, _ptr(sp), _ptr(ep), sp.dtype.itemsize))

    def count_only_fixed(self, pat2d, out=None):
        """Number of occurrences per pattern (ep - sp, uint32) without the interval."""
        pat2d = np.ascontiguousarray(pat2d, dtype=np.uint8)
        m, ln = pat2d.shape
        cnt = out if out is not None else np.zeros(m, np.uint32)
        assert cnt.dtype == np.uint32 and len(cnt) == m
        _check(lib().fmx_count_only_fixed(self.h, _ptr(pat2d), ln, m, _ptr(cnt)))
        return cnt

    def write_sa_file(self, path):
        """SACreator(path).create(): <base>.sa, n x 32-bit big-endian words, unsigned: positions at or beyond 2^31 are stored as they are,
        so read them back as >u4 (the reference's int32 reading agrees below 2^31)"""
        lib().fmx_write_sa_file.argtypes = [C.c_void_p, C.c_char_p]
        _check(lib().fmx_write_sa_file(self.h, os.fsencode(path)))

    def build_lcp(self):
        """bwtFm2LCP: int32[n], lcp[r] = lcp(suffix of row r, suffix of row r+1)"""
        lib().fmx_build_lcp.argtypes = [C.c_void_p, C.c_void_p]
        out = np.zeros(self.n, np.int32)
        _check(lib().fmx_build_lcp(self.h, _ptr(out)))
        return out

    def write_lcp_file(self, path):
        """LCPCreator(path).create(): <base>.lcp, max(n-1, 1) x int32 big-endian"""
        lib().fmx_write_lcp_file.argtypes = [C.c_void_p, C.c_char_p]
        _check(lib().fmx_write_lcp_file(self.h, os.fsencode(path)))

    def set_accel_mask(self, mask):
        """keep only the accelerators in `mask` (ACCEL_* bits; ACCEL_NONE = plain rank steps, ACCEL_AUTO = all built) for later calls"""
        _check(lib().fmx_set_accel_mask(self.h, mask))

    def set_lanes(self, lanes):
        _check(lib().fmx_set_lanes(self.h, lanes))

    def last_kernel_ms(self):
        return lib().fmx_last_kernel_ms(self.h)

    def last_kernel_launches(self):
        return lib().fmx_last_kernel_launches(self.h)

    def last_regex_levels(self):
        return lib().fmx_last_regex_levels(self.h)


class LCPSearcher(GpuFMSearcher):
    """new LCPSearcher(filename, bigEndian) — bwtmerger.scala:322-333: a NaiveFMSearcher that also opens <base>.lcp and <base>.sa
    (LCPLoader :176-211, SALoader :214-249; both created on demand here, by the GPU, when absent) and offers LCPSuffixWalkingAlgo's
    getLCP(i) and getStringOn(i).  The reference's getStringOn reads the cached forward text file from offset fsize - sa[i] up to
    the next 0 byte, i.e. the characters T'[sa[i]-1], T'[sa[i]-2], ... — the same bytes an LF walk from row i emits, which is how
    they are produced here (no .data file needed)."""

    def __init__(self, filename, bigEndian=True, **opts):
        super().__init__(filename, bigEndian, **opts)
        base = os.path.splitext(filename)[0]
        if not os.path.exists(base + ".lcp"):
            self.write_lcp_file(base)
        if not os.path.exists(base + ".sa"):
            self.write_sa_file(base)
        self._lcp = np.memmap(base + ".lcp", dtype=">i4", mode="r")
        self._sa = np.memmap(base + ".sa", dtype=">u4", mode="r")          # unsigned: texts past 2^31 (fmx_write_sa_file)

    def getLCP(self, i):
        return int(self._lcp[i])

    def getSA(self, i):
        return int(self._sa[i])

    def getStringOn(self, i, chunk=256):
        """iterator over the characters the reference's StringPosReader yields: up to (not including) the first 0 byte"""
        done = 0
        while True:
            s = self.prev_substr_batch([i], chunk)[0]              # one LF walk of `chunk` steps on the GPU; grown until the '\0' shows
            z = s.find(b"\0")
            for ch in s[done:(z if z >= 0 else len(s))]:
                yield chr(ch)
            if z >= 0 or chunk >= self.n:
                return
            done, chunk = len(s), min(self.n, chunk * 4)


class PinnedArray:
    """numpy view over page-locked host memory from fmx_host_alloc; keep the object alive while the view is used."""

    def __init__(self, shape, dtype):
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _check(lib().fmx_host_alloc(C.byref(p), self.nbytes))
        self.p = p
        buf = (C.c_uint8 * max(self.nbytes, 1)).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self.p:
            self.array = None
            lib().fmx_host_free(self.p)
            self.p = None


class SharedDeviceBuffer:
    """A cudaMalloc'ed uint32 buffer that the ranks of one node map into each other through CUDA IPC."""

    def __init__(self, n_elems):
        self.n = n_elems
        p = C.c_void_p()
        _check(lib().fmx_dev_alloc(C.byref(p), n_elems * 4))
        self.ptr = p.value
        self.peers = {}

    def export_handle(self):
        h = (C.c_uint8 * 64)()
        _check(lib().fmx_ipc_export(C.c_void_p(self.ptr), h))
        return bytes(h)

    def import_peer(self, rank, handle):
        p = C.c_void_p()
        buf = (C.c_uint8 * 64).from_buffer_copy(handle)
        _check(lib().fmx_ipc_import(buf, C.byref(p)))
        self.peers[rank] = p.value
        return p.value

    def to_host(self):
        out = np.zeros(self.n, np.uint32)
        _check(lib().fmx_memcpy_d2h(_ptr(out), C.c_void_p(self.ptr), self.n * 4))
        return out

    def close(self):
        for p in self.peers.values():
            lib().fmx_ipc_close(C.c_void_p(p))
        self.peers = {}
        if self.ptr:
            lib().fmx_dev_free(C.c_void_p(self.ptr))
            self.ptr = None


def scatter_dev(d_src, count_words, sinks, offset_words=0, d_dst_off=0, dst_scale=1, stream=0):
    """fmx_scatter_dev: `count_words` 4-byte words at d_src go to every sink at word offset offset_words + (*d_dst_off) * dst_scale"""
    arr = (C.c_void_p * max(len(sinks), 1))(*sinks)
    _check(lib().fmx_scatter_dev(C.c_void_p(d_src), count_words, arr, len(sinks), offset_words, C.c_void_p(d_dst_off), dst_scale, C.c_void_p(stream)))


def set_l2_fetch_granularity(nbytes=0):
    eff = C.c_int32()
    _check(lib().fmx_set_l2_fetch_granularity(nbytes, C.byref(eff)))
    return eff.value


def build_bwt(text, device=-1):
    """Device suffix sort of reverse(text without 0x00)+'$'.  Returns (bwt uint8[n], eof, counts int64[256])."""
    t = _u8(text)
    bwt = np.zeros(len(t) + 1, np.uint8)
    cnt = np.zeros(256, np.int64)
    n, eof = C.c_int64(), C.c_int64()
    buf = t if len(t) else np.zeros(1, np.uint8)
    _check(lib().fmx_build_bwt(_ptr(buf), len(t), _ptr(bwt), C.byref(n), C.byref(eof), _ptr(cnt), device))
    return bwt[:n.value], eof.value, cnt


def build_index_files(text, base, bigEndian=True, write_fm=False, device=-1):
    t = _u8(text)
    buf = t if len(t) else np.zeros(1, np.uint8)
    _check(lib().fmx_build_index_files(_ptr(buf), len(t), os.fsencode(base), int(bigEndian), int(write_fm), device))

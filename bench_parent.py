#!/usr/bin/env python
"""
bench.py — FM-index search throughput on B200 (BASELINE.json metric: FM count queries/s, len-16, 1 GB text; regex queries/s).

    python bench.py --gpus N --steps K --warmup W                       this repo's CUDA path through the C ABI (libfmgpu.so)
    python bench.py --impl reference --gpus N --steps K --warmup W      the reference algorithm on the host CPU cores (oracle/)
    python bench.py --workload cfg3|cfg4|cfg5 ...                       the other BASELINE configs as top-level lines

Default line = BASELINE configs[1] (SURVEY.md §8d cfg 2): 10^9 bytes i.i.d. uniform over 1..255 (seed 2), indexed as the reference
does (reverse(text)+'$', .bwt/.aux files); per GPU 10 M len-16 patterns, 90 % reversed text substrings, 10 % random (seed 3).  A "step"
is one pass of the batch through the count kernel.  With N GPUs the index is replicated, every rank owns its own 10 M-query shard
(weak scaling) and the per-query counts are exchanged by the count kernel itself (peer-memory stores) + a 4-byte NCCL barrier.
The same line carries, as extra keys, what bounds and qualifies that number:

    sweep      cfg-2 index at len 8..64, plain PLANES and the wavelet matrix at len 16, each with requests/query and oracle parity
    sustained  >= 2 s of back-to-back launches with the in-window clock / power record
    pcie       the box's concurrent pinned H2D+D2H copy ceiling for this step's bytes (what bounds e2e)
    english    cfg 3/4: 10^9-byte English-like text — count at len 8 / 12 / 16 / 24 with the dictionary of wide intervals and at len 12
               without it, locate (SA sample rate 32), 100 k Glushkov regexes
    cfg5       4*10^9-byte DNA text, len-32 count queries (2-bit packed upload for e2e)

One JSON line on stdout (rank 0).  Everything else goes to stderr.
"""
import argparse
import json
import lzma
import os
import subprocess
import sys
import threading
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OUT = sys.stdout
UNIT = "queries/s"
METRICS = {"cfg2": "fm_count_queries_per_s_len16_1GB_text", "cfg3": "fm_locate_queries_per_s_len12_1GB_english_text_sa32",
           "cfg4": "glushkov_regex_queries_per_s_1GB_english_text", "cfg5": "fm_count_queries_per_s_len32_4GB_dna_text"}
DEFAULTS = {"cfg2": (1_000_000_000, 10_000_000, 16), "cfg3": (1_000_000_000, 1_000_000, 12), "cfg4": (1_000_000_000, 100_000, 0),
            "cfg5": (4_000_000_000, 12_500_000, 32)}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------ workloads
def vocabulary(via):
    """words.txt vocabulary from the committed words.bwt fixture: through the GPU searcher (prevSubstr(eof, n) walks the whole file,
    T/Indexer.scala:1120) in our arm, through the oracle in the reference arm."""
    if via in _VOCAB:
        return _VOCAB[via]
    import tempfile
    d = tempfile.mkdtemp(prefix="fmx_words_%d_" % os.getpid())         # private to this process: N ranks of one box share /tmp
    with lzma.open(os.path.join(ROOT, "tests", "golden", "ref", "words.bwt.xz"), "rb") as f:
        data = f.read()
    with open(os.path.join(d, "words.bwt"), "wb") as f:
        f.write(data)
    with open(os.path.join(ROOT, "tests", "golden", "ref", "words.aux"), "rb") as f:
        aux = f.read()
    with open(os.path.join(d, "words.aux"), "wb") as f:
        f.write(aux)
    if via == "gpu":
        from findex_b200 import fmindex as fx
        g = fx.GpuFMSearcher(os.path.join(d, "words.bwt"), accel=fx.ACCEL_NONE)
        text = g.prevSubstr(g.eof, g.n)[1:]
        g.close()
    else:
        from oracle import fm_oracle as fo
        o = fo.OracleIndex.load(os.path.join(d, "words"))
        sa = o.sa()
        tp = np.zeros(o.n, np.uint8)
        tp[(sa.astype(np.int64) - 1) % o.n] = o.bwt()
        text = bytes(tp[:-1][::-1])
        o.close()
    import shutil
    shutil.rmtree(d, ignore_errors=True)
    _VOCAB[via] = [w for w in text.split(b"\r\n") if w]
    return _VOCAB[via]


_VOCAB = {}


def make_text(n, workload, via="gpu"):
    from findex_b200 import synth
    if workload == "cfg5":
        return synth.dna(n, 7)
    if workload in ("cfg3", "cfg4"):
        return synth.english_like(vocabulary(via), n, 4)
    return synth.uniform_bytes(n, 2)


def make_queries(text, m, ln, seed, rank, out=None, workload="cfg2"):
    """cfg 2/5: 90 % hits (reversed substrings at uniform offsets), 10 % uniform random symbols, shuffled.  cfg 3: substrings only."""
    rng = np.random.default_rng([seed, rank])
    nh = m if workload in ("cfg3", "cfg4") else int(m * 0.9)
    pats = out if out is not None else np.empty((m, ln), np.uint8)
    offs = rng.integers(0, len(text) - ln, nh)
    hits = text[offs[:, None] + np.arange(ln - 1, -1, -1)[None, :]]
    if nh == m:
        pats[:] = hits
        return pats, np.ones(m, bool)
    if workload == "cfg5":
        rnd = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, (m - nh, ln), dtype=np.uint8)]
    else:
        rnd = rng.integers(1, 256, (m - nh, ln), dtype=np.uint8)
    perm = rng.permutation(m)
    is_hit = np.zeros(m, bool)
    is_hit[:nh] = True
    pats[:] = np.concatenate([hits, rnd])[perm]
    return pats, is_hit[perm]


def index_base(n, workload):
    return "/tmp/fmx_bench_%s_%d" % ({"cfg4": "cfg3"}.get(workload, workload), n)


def workload_config(args, workload=None, n=None, m=None, ln=None):
    """identical in both arms (the driver compares the dicts)"""
    w = workload or args.workload
    n, m, ln = n or args.text_bytes, m or args.queries, args.len if ln is None else ln
    what = {"cfg2": "cfg2: %d-byte uniform text over bytes 1..255 (seed 2), %d len-%d count queries per GPU, 90%% hits / 10%% random (seed 3)" % (n, m, ln),
            "cfg3": "cfg3: %d-byte English-like text (Zipf words, seed 4), %d len-%d locate queries in all (text substrings, seed 5), SA sample rate 32" % (n, m, ln),
            "cfg4": "cfg4: %d-byte English-like text (Zipf words, seed 4), %d template regexes per GPU (classes, alternation, bounded repeats, \\d, '.'; seed 6)" % (n, m),
            "cfg5": "cfg5: %d-byte uniform DNA text (ACGT, seed 7), %d len-%d count queries per GPU, 90%% hits / 10%% random (seed 8)" % (n, m, ln)}[w]
    return {"workload": what, "text_bytes": n, "queries_per_gpu": m, "pattern_len": ln,
            "parallelism": "dp%d (index replicated, queries sharded)" % args.gpus,
            "l2": "inputs and index (GBs) exceed the 126 MB L2; no explicit flush"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled every 50 ms from before the warm-up until after the timed region; the summary uses
    the samples inside the timed window (all samples under load if the window is shorter than the sampling period)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc, self.window = gpu, [], None, [None, None]

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception as e:                       # nvidia-smi missing: report that, do not fail the bench
            log("clock sampler unavailable:", e)
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark_begin(self):
        self.window[0] = time.time()

    def mark_end(self):
        self.window[1] = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        parsed = []
        for ts, r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                parsed.append((ts, float(f[0]), float(f[1]), float(f[2]), [nme for nme, v in zip(names, f[3:7]) if v == "Active"]))
            except ValueError:
                continue
        inside = [p for p in parsed if self.window[0] is not None and self.window[0] <= p[0] <= (self.window[1] or 1e18) + 0.06]
        use = inside if inside else parsed
        reasons = sorted({x for p in use for x in p[4]})
        return {"sm_mhz": float(np.median([p[1] for p in use])) if use else None, "sm_mhz_min": min([p[1] for p in use]) if use else None,
                "sm_max_mhz": max([p[2] for p in use]) if use else None, "power_w_max": max([p[3] for p in use]) if use else None,
                "power_w_median": float(np.median([p[3] for p in use])) if use else None, "reasons": reasons, "samples": len(use),
                "samples_in_timed_window": len(inside)}


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path: NaiveFMSearcher.occ = binary search in the in-memory .fm array
    (bwtmerger.scala:354-375) driving SuffixAlgo.search (findex.scala:15-31), sorted sa[sp..ep) for locate (util.scala:213-224) and
    ReTree._matchSA (retree.scala:618-653) — the C restatement under oracle/ (no JVM exists in this image), all host threads, a bounded
    sample of the same workload per step."""
    if rank != 0:
        return
    from oracle import fm_oracle as fo
    cores = os.cpu_count() or 1
    w = args.workload
    n, m, ln = args.text_bytes, args.queries, args.len
    t0 = time.time()
    text = make_text(n, w, via="oracle")
    base = index_base(n, w)
    if not (os.path.exists(base + ".bwt") and os.path.exists(base + ".aux")):
        # index construction is setup, not the measured path; the device suffix sorter only writes the reference's files
        from findex_b200 import build as fbuild, fmindex as fx
        fbuild.build()
        try:
            fx.build_index_files(text, base, bigEndian=True)
        except fx.FmxError:
            # no CUDA device (CPU-only check of this arm): the oracle's own builder writes the same files; small texts only
            if n > 50_000_000:
                raise
            bwt, eof, cnt = fo.build_bwt(fo.file_to_text_rev(text.tobytes()))
            fo.write_index_files(base, bwt, eof, cnt, big_endian=True)
    fo.build(native=True)
    ix = fo.OracleIndex.load(base)
    log("reference arm: index loaded + fm array materialised in %.1f s" % (time.time() - t0))
    budget_s = min(8.0, 120.0 / max(args.steps + args.warmup, 1))
    unit = UNIT
    if w == "cfg4":
        from findex_b200 import synth
        rxs = synth.regex_templates(text, np.random.default_rng([6, 0]), min(m, 5000))
        rxs = [t for t in (_oracle_compile(r) for r in rxs) if t is not None]       # ReTree(post): compiled once, outside the timed traversal
        rate = _probe(lambda k: _oracle_regex(ix, rxs[:k], cores), 64)
        sample = int(min(len(rxs), max(64, rate * budget_s)))
        run = lambda: _oracle_regex(ix, rxs[:sample], cores)          # noqa: E731
        unit = "regexes/s"
        sdesc = "first %d regexes of the %d-regex batch per step, %d threads" % (sample, m, cores)
    else:
        pats, _ = make_queries(text, m, ln, {"cfg2": 3, "cfg3": 5, "cfg5": 8}[w], 0, workload=w)
        if w == "cfg3":
            t1 = time.time()
            ix.sa()                                                    # SACreator.create: the reference's one-off .sa (n FL steps)
            log("reference arm: suffix array materialised in %.1f s (setup, as SACreator.create)" % (time.time() - t1))
        fn = (lambda k: _oracle_locate(ix, pats[:k], ln, cores)) if w == "cfg3" else \
            (lambda k: ix.count_batch(pats[:k].reshape(-1), np.arange(0, k * ln + 1, ln, dtype=np.int64), threads=cores))
        rate = _probe(fn, 20000 if w != "cfg3" else 2000)
        sample = int(min(m, max(2000, rate * budget_s)))
        run = lambda: fn(sample)                                       # noqa: E731
        sdesc = "first %d of the %d-query batch per step, %d threads" % (sample, m, cores)
    for _ in range(args.warmup):
        run()
    t1 = time.time()
    for _ in range(args.steps):
        run()
    dt = time.time() - t1
    v = sample * args.steps / dt
    out = {"impl": "reference", "metric": METRICS[w], "value": v, "unit": unit, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong" if w == "cfg3" else "weak", "vs_baseline": None,
           "dtype": "u32", "data": "synthetic", "config": workload_config(args),
           "cpu_baseline": {"value": v, "unit": unit, "cores": cores, "kind": "port", "sample": sdesc,
                            "note": "JVM unavailable - C restatement of the reference algorithm (binary search in .fm)"},
           "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(out), file=OUT, flush=True)


def _probe(fn, k):
    t1 = time.time()
    fn(k)
    return k / max(time.time() - t1, 1e-6)


def _oracle_compile(rx):
    from oracle import retree
    try:
        return retree.compile_regex(rx).tables()
    except Exception:
        return None


def _oracle_regex(ix, tables, threads):
    """ReTree._matchSA (caps off) of precompiled automata, one regex per task on `threads` host threads"""
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max(threads, 1)) as ex:
        return list(ex.map(lambda t: ix.regex_match_tables(t, 50_000_000)[0], tables))


def _oracle_locate(ix, pats, ln, threads):
    """count (all threads) + sorted sa[sp..ep) per query"""
    k = len(pats)
    sp, ep = ix.count_batch(pats.reshape(-1), np.arange(0, k * ln + 1, ln, dtype=np.int64), threads=threads)
    sa = ix.sa()
    from concurrent.futures import ThreadPoolExecutor

    def part(r):
        return [np.sort(sa[a:b]) for a, b in zip(sp[r::threads], ep[r::threads])]
    with ThreadPoolExecutor(max(threads, 1)) as ex:
        return list(ex.map(part, range(threads)))


# ------------------------------------------------------------------------------------------------ our arm: shared plumbing
class Ctx:
    """torch / distributed plumbing of one rank"""

    def __init__(self, args, rank, world, local_rank):
        import torch
        import torch.distributed as dist
        from findex_b200 import build as fbuild, fmindex as fx, synth
        self.torch, self.dist, self.fx, self.synth = torch, dist, fx, synth
        self.args, self.rank, self.world, self.local = args, rank, world, local_rank
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        if rank == 0:
            fbuild.build()
        self.barrier()
        self.launches = 0

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v):
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def ensure_index(self, workload, n):
        """text (every rank) + index files (rank 0 builds them on the GPU when absent)"""
        t0 = time.time()
        import gc
        gc.collect()
        self.torch.cuda.empty_cache()                      # the suffix sort of a 4 GB text needs most of the device
        base = index_base(n, workload)
        err, text = None, None
        try:                                                 # every rank must reach the collective below and leave the same way
            text = make_text(n, workload)
            if self.rank == 0 and not (os.path.exists(base + ".bwt") and os.path.exists(base + ".aux")):
                tb = time.time()
                self.fx.build_index_files(text, base, bigEndian=True)
                log("%s: index files built on the GPU in %.1f s" % (workload, time.time() - tb))
        except Exception as e:                               # noqa: BLE001
            err = e
            log("rank %d: %s text / index files failed: %s: %s" % (self.rank, workload, type(e).__name__, e))
        if self.max_over_ranks(1.0 if err is not None else 0.0) > 0:
            raise err if err is not None else RuntimeError("another rank could not make the %s text / index files" % workload)
        log("rank %d: %s text + index files ready after %.1f s" % (self.rank, workload, time.time() - t0))
        return text, base

    def timed(self, fn, steps, warmup, wall=False, drain=None, sample_clocks=True):
        """warm-up, barrier + synchronize, `steps` calls between CUDA events on the current stream, barrier + synchronize; max over ranks.
        wall=True: host wall clock (host-API calls that return when the results are in host memory)."""
        torch = self.torch
        sampler = ClockSampler(self.local) if sample_clocks else None
        if sampler:
            sampler.start()
        for _ in range(warmup):
            fn()
        if drain:
            drain()
        torch.cuda.synchronize()
        self.barrier()
        torch.cuda.synchronize()
        if sampler:
            sampler.mark_begin()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall = time.time()
        e0.record()
        for _ in range(steps):
            fn()
        if drain:
            drain()
        e1.record()
        torch.cuda.synchronize()
        wall_ms = (time.time() - t_wall) * 1e3
        if sampler:
            sampler.mark_end()
        self.barrier()
        torch.cuda.synchronize()
        clocks = sampler.stop() if sampler else None
        ms = wall_ms if wall else e0.elapsed_time(e1)
        return self.max_over_ranks(ms), clocks


def device_count_rate(cx, g, pats, reps=5):
    """device-resident count of one batch: best-of-`reps` CUDA-event time, (sp, ep) as int64 arrays"""
    torch = cx.torch
    m, ln = pats.shape
    d_pat = torch.from_numpy(pats).to(cx.dev)
    d_sp = torch.zeros(m, dtype=torch.int32, device=cx.dev)
    d_ep = torch.zeros(m, dtype=torch.int32, device=cx.dev)
    st = torch.cuda.current_stream().cuda_stream
    for _ in range(3):
        g.count_fixed_dev(d_pat.data_ptr(), ln, m, d_sp.data_ptr(), d_ep.data_ptr(), st)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.count_fixed_dev(d_pat.data_ptr(), ln, m, d_sp.data_ptr(), d_ep.data_ptr(), st)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    cx.launches += 3 + reps
    sp = d_sp.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    ep = d_ep.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    return best, sp, ep


def oracle_parity(orc, pats, sp, ep, k):
    """GPU (sp, ep) of the first k queries == the oracle's (None reported as (0, 0))"""
    k = min(k, len(pats))
    ln = pats.shape[1]
    osp, oep = orc.count_batch(pats[:k].reshape(-1), np.arange(0, k * ln + 1, ln, dtype=np.int64), threads=os.cpu_count())
    hit = ep[:k] > sp[:k]
    return bool(np.array_equal(np.where(hit, sp[:k], 0), osp) and np.array_equal(np.where(hit, ep[:k], 0), oep)), k


def sweep_leg(cx, g, text, lens, m, seed, orc, label, workload="cfg2", sample=100_000):
    """count throughput vs pattern length on one index: device q/s, requests/query, steps skipped, oracle parity on a sample"""
    out = []
    for ln in lens:
        pats, _ = make_queries(text, m, ln, seed * 1000 + ln, cx.rank, workload=workload)
        ms, sp, ep = device_count_rate(cx, g, pats)
        req, steps = g.count_fixed_stats(pats)
        rec = {"index": label, "len": ln, "queries": m, "kernel_ms": ms, "queries_per_s": m / (ms * 1e-3), "requests_per_query": req / m,
               "steps_per_query": steps / m, "hits": int((ep > sp).sum())}
        if orc is not None:
            rec["parity_on_sample"], rec["parity_sample"] = oracle_parity(orc, pats, sp, ep, sample)
            assert rec["parity_on_sample"], "GPU (sp,ep) differ from the oracle: %s len %d" % (label, ln)
        out.append(rec)
    return out


def pcie_ceiling(cx, h2d_bytes, d2h_bytes, steps=10):
    """The box's copy ceiling for one step's bytes: pinned H2D and D2H on two streams, concurrently on every rank, no kernel.
    cudaMemcpyAsync one buffer per direction and step, as the host API does per chunk."""
    torch = cx.torch
    hin = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8).pin_memory()
    hout = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8).pin_memory()
    din = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8, device=cx.dev)
    dout = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8, device=cx.dev)
    s1, s2 = torch.cuda.Stream(device=cx.dev), torch.cuda.Stream(device=cx.dev)

    def step():
        with torch.cuda.stream(s1):
            din.copy_(hin, non_blocking=True)
        with torch.cuda.stream(s2):
            hout.copy_(dout, non_blocking=True)

    def drain():
        torch.cuda.current_stream().wait_stream(s1)
        torch.cuda.current_stream().wait_stream(s2)
    ms, _ = cx.timed(step, steps, 3, wall=True, drain=drain, sample_clocks=False)
    per = ms / steps
    return {"ms_per_step": per, "h2d_gbs_per_gpu": h2d_bytes / per / 1e6, "d2h_gbs_per_gpu": d2h_bytes / per / 1e6,
            "aggregate_h2d_gbs": cx.world * h2d_bytes / per / 1e6, "what": "concurrent pinned cudaMemcpyAsync H2D %d B + D2H %d B per rank and step, "
            "all %d ranks at once, no kernel" % (h2d_bytes, d2h_bytes, cx.world)}


def numa_report(local_rank):
    """Where this rank's GPU hangs in the host topology, and the binding taken (none when the box exposes no NUMA topology)."""
    rep = {"bound_node": None}
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (getattr(p, "pci_domain_id", 0), p.pci_bus_id, getattr(p, "pci_device_id", 0))
        rep["pci"] = bdf
        path = "/sys/bus/pci/devices/%s/numa_node" % bdf
        node = int(open(path).read().strip()) if os.path.exists(path) else None
        rep["numa_node"] = node
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")] if os.path.isdir("/sys/devices/system/node") else []
        rep["host_numa_nodes"] = len(nodes)
        if node is not None and node >= 0 and len(nodes) > 1:
            cpus = set()
            for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
            allowed = cpus & os.sched_getaffinity(0)
            if allowed:
                os.sched_setaffinity(0, allowed)                      # before any pinned allocation: first touch lands on this node
                rep["bound_node"] = node
        elif node is None or node < 0:
            rep["note"] = "the box exposes no NUMA topology for the GPU (numa_node = %s, %d host node(s)): nothing to bind to" % (node, len(nodes))
    except Exception as e:
        rep["error"] = str(e)
    return rep


# ------------------------------------------------------------------------------------------------ cfg 2 / cfg 5: count
class FusedExchange:
    """N > 1: the count kernel stores its hit counts straight into every rank's gathered buffer (CUDA IPC peer memory over
    NVLink/NVSwitch); NCCL is left with one 4-byte all-reduce per step as the cross-rank "all stores landed" barrier.  Three buffer
    sets rotate: kernel s (set s mod 3) is launched behind the barrier of step s-2, whose completion proves that every rank had
    enqueued — ahead of its kernel s-2 — the consumers of step s-3, the last user of that set."""

    def __init__(self, cx, m):
        fx, torch, dist = cx.fx, cx.torch, cx.dist
        self.cx, self.m = cx, m
        self.gath = [fx.SharedDeviceBuffer(m * cx.world) for _ in range(3)]
        mine = [gb.export_handle() for gb in self.gath]
        everyone = [None] * cx.world
        dist.all_gather_object(everyone, mine)
        self.sinks = [[self.gath[b].ptr if r == cx.rank else self.gath[b].import_peer(r, everyone[r][b]) for r in range(cx.world)] for b in range(3)]
        self.flag = torch.zeros(1, dtype=torch.int32, device=cx.dev)
        self.ev_k = [torch.cuda.Event() for _ in range(3)]
        self.ev_c = [torch.cuda.Event() for _ in range(3)]
        self.comm = torch.cuda.Stream(device=cx.dev)
        self.s = 0

    def step(self, g, d_pat, ln, d_sp, d_ep):
        torch, dist = self.cx.torch, self.cx.dist
        cur = torch.cuda.current_stream()
        b = self.s % 3
        if self.s >= 2:
            cur.wait_event(self.ev_c[(self.s - 2) % 3])
        g.count_fixed_dev_gather(d_pat.data_ptr(), ln, self.m, d_sp.data_ptr(), d_ep.data_ptr(), self.sinks[b], self.cx.rank * self.m, cur.cuda_stream)
        self.ev_k[b].record(cur)
        with torch.cuda.stream(self.comm):
            self.comm.wait_event(self.ev_k[b])
            dist.all_reduce(self.flag)                   # after this, every rank's stores of this step have landed everywhere
            self.ev_c[b].record(self.comm)
        self.s += 1

    def drain(self):
        self.cx.torch.cuda.current_stream().wait_stream(self.comm)

    def check(self, local_counts):
        """every rank holds every rank's counts of the last step, and all ranks agree"""
        torch, dist, cx = self.cx.torch, self.cx.dist, self.cx
        torch.cuda.synchronize()
        dist.barrier()
        got = torch.from_numpy(self.gath[(self.s - 1) % 3].to_host().astype(np.int64)).to(cx.dev)
        assert torch.equal(got[cx.rank * self.m:(cx.rank + 1) * self.m], local_counts.to(torch.int64) & 0xFFFFFFFF), "gathered counts differ from the local ones"
        cs = (got * torch.arange(1, got.numel() + 1, device=cx.dev) % 1000003).sum().reshape(1)
        lo_, hi_ = cs.clone(), cs.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        assert int(lo_) == int(hi_), "ranks disagree on the gathered counts"

    def close(self):
        """keeps the mappings until the end of the run (sharded.close_retired): closing the last IPC mapping of a peer takes the lazily
        enabled peer access down with it, under NCCL's feet"""
        from findex_b200 import sharded
        self.cx.torch.cuda.synchronize()
        sharded._RETIRED.append(self)

    def close_peers(self):
        for gb in self.gath:
            for ptr in list(gb.peers.values()):
                self.cx.fx.lib().fmx_ipc_close(ptr)
            gb.peers = {}

    def really_close(self):
        for gb in self.gath:
            gb.close()


def count_workload(cx, workload, n, m, ln, extras):
    """cfg 2 (default line) and cfg 5: device-resident count throughput, e2e through the host API, roofline, cpu baseline"""
    args, fx, torch = cx.args, cx.fx, cx.torch
    world, rank = cx.world, cx.rank
    text, base = cx.ensure_index(workload, n)
    t0 = time.time()
    layout = {"auto": fx.LAYOUT_AUTO, "wm": fx.LAYOUT_WM, "planes": fx.LAYOUT_PLANES}[args.layout]
    accel = {"auto": fx.ACCEL_AUTO, "none": fx.ACCEL_NONE, "kmer": fx.ACCEL_KMER, "text": fx.ACCEL_TEXT, "both": fx.ACCEL_KMER | fx.ACCEL_TEXT,
             "ctx": fx.ACCEL_KMER | fx.ACCEL_CTX}[args.accel]
    g = fx.GpuFMSearcher(base + ".bwt", bigEndian=True, device=cx.local, layout=layout, lanes_per_query=args.lanes, accel=accel,
                         max_total_bytes=args.max_total_bytes)
    if args.chunk:
        g.set_chunk(args.chunk)
    info = g.info()
    open_s = time.time() - t0
    log("rank %d: %s index open (%s, %.2f GB on device) after %.1f s" % (rank, workload, info["layout"], info["index_bytes"] / 1e9, open_s))

    seed = 8 if workload == "cfg5" else 3
    h_pat = fx.PinnedArray((m, ln), np.uint8)
    pats, is_hit = make_queries(text, m, ln, seed, rank, out=h_pat.array, workload=workload)
    d_pat = torch.from_numpy(pats).to(cx.dev)
    d_sp = torch.zeros(m, dtype=torch.int32, device=cx.dev)
    d_ep = torch.zeros(m, dtype=torch.int32, device=cx.dev)
    stream = torch.cuda.current_stream().cuda_stream
    fused = FusedExchange(cx, m) if (world > 1 and args.exchange == "p2p") else None
    nccl_all = torch.zeros(m * world, dtype=torch.int32, device=cx.dev) if (world > 1 and fused is None) else None
    nccl_cnt = torch.zeros(m, dtype=torch.int32, device=cx.dev) if nccl_all is not None else None

    def step():
        if fused is not None:
            fused.step(g, d_pat, ln, d_sp, d_ep)
        else:
            g.count_fixed_dev(d_pat.data_ptr(), ln, m, d_sp.data_ptr(), d_ep.data_ptr(), stream)
            if nccl_all is not None:
                torch.sub(d_ep, d_sp, out=nccl_cnt)
                cx.dist.all_gather_into_tensor(nccl_all, nccl_cnt)

    drain = fused.drain if fused is not None else None
    # ---- sanity at full size (parity proper lives in tests/ and in the cpu_baseline leg): hits are found, a few are verified by brute force
    step()
    if drain:
        drain()
    torch.cuda.synchronize()
    if fused is not None:
        fused.check(d_ep - d_sp)
    sp = d_sp.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    ep = d_ep.cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    cnt = ep - sp
    assert (cnt[is_hit] >= 1).all(), "a text substring was not found"
    if rank == 0 and n <= 1_500_000_000:
        tb = text.tobytes()
        for q in np.flatnonzero(is_hit)[:2]:
            assert tb.count(pats[q][::-1].tobytes()) == cnt[q], "count mismatch vs brute force"
        del tb
    checksum = int((sp * 1315423911 + ep * 2654435761).sum() & 0xFFFFFFFFFFFF)

    # ---- roofline inputs, outside the timed region
    requests, steps_exec = g.count_fixed_stats(pats)
    r_rand_gbs, _ = g.gather_bench(64, 4, 1 << 25, 16, 3)            # K4: random 64-B requests (four lanes x one 128-bit load = one request) over this index
    r_rand_req = r_rand_gbs * 1e9 / 64

    ms_total, clocks = cx.timed(step, args.steps, args.warmup, drain=drain)
    cx.launches += args.steps + args.warmup + 1
    # kernel-only time of the same launches (no exchange), per-launch events, for the roofline
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for a, b in kev:
        a.record()
        g.count_fixed_dev(d_pat.data_ptr(), ln, m, d_sp.data_ptr(), d_ep.data_ptr(), stream)
        b.record()
    torch.cuda.synchronize()
    cx.launches += args.steps
    k_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))

    sustained = None
    if "sustained" in extras:
        # >= 2 s of back-to-back launches: what the clocks and the power cap do to the number over time
        est = max(ms_total / args.steps, 1e-3)
        nlaunch = int(min(20000, max(200, 2200.0 / est)))
        ms_s, clocks_s = cx.timed(step, nlaunch, 3, drain=drain)
        cx.launches += nlaunch + 3
        sustained = {"launches": nlaunch, "seconds": ms_s / 1e3, "ms_per_step": ms_s / nlaunch, "value": world * m * nlaunch / (ms_s * 1e-3), "unit": UNIT,
                     "ratio_to_value": (ms_total / args.steps) / (ms_s / nlaunch), "clocks": clocks_s}

    # ---- end to end through the host API: (sp, ep) per query at the reference's own width (Option[(Int, Int)], findex.scala:15-31)
    narrow = g.n < 2 ** 31                                  # cfg 5 (n = 4e9) does not fit Int rows: int64 there
    rdt = np.int32 if narrow else np.int64
    h_sp, h_ep = fx.PinnedArray((m,), rdt), fx.PinnedArray((m,), rdt)
    e2e_steps = max(3, min(args.steps, 20))

    def e2e_step():
        g.count_fixed_into(h_pat.array, h_sp.array, h_ep.array)
    ms_e2e, clocks_e2e = cx.timed(e2e_step, e2e_steps, 3, wall=True)
    nchunks = (m + (args.chunk or (1 << 20)) - 1) // (args.chunk or (1 << 20))
    cx.launches += (e2e_steps + 3) * nchunks
    assert np.array_equal(h_sp.array, np.where(cnt > 0, sp, 0)) and np.array_equal(h_ep.array, np.where(cnt > 0, ep, 0)), "host API result differs from device API"
    e2e = {"value": world * m * e2e_steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": m * ln, "d2h_bytes_per_step": m * 2 * np.dtype(rdt).itemsize,
           "ms_per_step": ms_e2e / e2e_steps, "steps": e2e_steps, "clocks": clocks_e2e,
           "api": "fmx_count_fixed_i32 (host pinned buffers in/out, (sp, ep) as the reference's 32-bit Int rows)" if narrow else "fmx_count_fixed (host pinned buffers in/out, int64 sp/ep)"}
    # the same batch through the count-only call (uint32 ep-sp per query: 4 instead of 8/16 result bytes over PCIe)
    h_cnt = fx.PinnedArray((m,), np.uint32)

    def e2e_count_only_step():
        g.count_only_fixed(h_pat.array, out=h_cnt.array)
    ms_co, _ = cx.timed(e2e_count_only_step, e2e_steps, 2, wall=True, sample_clocks=False)
    cx.launches += (e2e_steps + 2) * nchunks
    assert np.array_equal(h_cnt.array.astype(np.int64), np.where(cnt > 0, cnt, 0)), "count-only API differs from ep-sp"
    e2e["count_only"] = {"value": world * m * e2e_steps / (ms_co * 1e-3), "unit": UNIT, "ms_per_step": ms_co / e2e_steps, "h2d_bytes_per_step": m * ln,
                         "d2h_bytes_per_step": m * 4, "api": "fmx_count_only_fixed (uint32 ep-sp)"}
    if info["sigma"] <= 4:
        # <= 4-symbol alphabets: the patterns cross PCIe as 2-bit codes (a quarter of the bytes) and are expanded on the device; rows come
        # back as uint32 (n < 2^32).  This is the call a DNA host makes, so it is the headline form of e2e where it applies.
        codes = g.pack2(pats)
        h_pk = fx.PinnedArray(codes.shape, np.uint8)
        h_pk.array[:] = codes
        h_sp4, h_ep4 = fx.PinnedArray((m,), np.uint32), fx.PinnedArray((m,), np.uint32)

        def e2e_packed_step():
            g.count_packed2_into(h_pk.array, ln, h_sp4.array, h_ep4.array)
        ms_pk, _ = cx.timed(e2e_packed_step, e2e_steps, 2, wall=True, sample_clocks=False)
        cx.launches += (e2e_steps + 2) * nchunks * 2
        assert np.array_equal(h_sp4.array.astype(np.int64), np.where(cnt > 0, sp, 0)) and np.array_equal(h_ep4.array.astype(np.int64), np.where(cnt > 0, ep, 0)), "packed host API result differs"
        unpacked = {k: e2e[k] for k in ("value", "ms_per_step", "h2d_bytes_per_step", "d2h_bytes_per_step", "api")}
        e2e.update({"value": world * m * e2e_steps / (ms_pk * 1e-3), "ms_per_step": ms_pk / e2e_steps, "h2d_bytes_per_step": int(codes.size), "d2h_bytes_per_step": m * 8,
                    "api": "fmx_count_fixed_packed2 (2-bit symbol codes in, expanded on the device; uint32 (sp, ep) out)", "unpacked_bytes": unpacked})
    if "pcie" in extras:
        pc = pcie_ceiling(cx, e2e["h2d_bytes_per_step"], e2e["d2h_bytes_per_step"])
        e2e["pcie_ceiling"] = pc
        e2e["frac_of_pcie_ceiling"] = pc["ms_per_step"] / e2e["ms_per_step"]

    value = world * m * args.steps / (ms_total * 1e-3)
    peak, peak_src = measured_peaks()
    # DRAM bytes one launch has to move at the 64-byte granule of a hinted random request: every request (table entry, row context, rank
    # block) is one granule, plus the streamed patterns and results
    granule_bytes = requests * 64 + m * (ln + 8)
    achieved = granule_bytes / (k_ms * 1e-3) / 1e9
    L = max(1, int(np.ceil(np.log2(max(info["sigma"], 2)))))
    roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": ncu_traffic(m, info),
            "peak_source": peak_src, "kernel": "count_fixed_kernel", "kernel_ms": k_ms, "algorithmic_bytes_per_launch": granule_bytes,
            "requests_per_query": requests / m, "steps_skipped_per_query": steps_exec / m - (requests / m),
            "request_rate": {"achieved_requests_per_s": requests / (k_ms * 1e-3), "r_rand_requests_per_s": r_rand_req,
                             "frac": requests / (k_ms * 1e-3) / r_rand_req, "r_rand_gbs": r_rand_gbs,
                             "note": "r_rand = live K4: dependent random 64-B requests over this index's rank blocks; what bounds a gather kernel on B200 is requests/s, not bytes"},
            "bytes_needed_per_query": {"table_entry": 8 if info["kmer_k"] else 0, "row_context": info["ctx_entry_bytes"], "pattern": ln, "result": 8},
            "survey_units": {"levels_L": L, "nominal_bytes_per_query": float(steps_exec / m * 2 * L * 64),
                             "note": "SURVEY 8(d): executed steps x 2 x L x 64 B of a wavelet-matrix search; this kernel answers the same queries bit-exactly "
                                     "from a k-mer table entry + row-context hops instead (steps skipped, not executed), so its bytes are the granules above"},
            "note": "achieved = (requests x 64-B granule + streamed pattern/result bytes) per launch / mean CUDA-event kernel time; frac vs the stream peak"}
    out = {"metric": METRICS[workload], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
           "config": workload_config(args, workload, n, m, ln),
           "impl_config": {"exchange": "none" if world == 1 else ("count kernel stores into peer gathered buffers + 4-byte NCCL barrier" if fused else "NCCL all_gather_into_tensor"),
                           "layout": info["layout"], "lanes_per_query": info["lanes_per_query"], "index_bytes": info["index_bytes"],
                           "index_bytes_per_text_byte": info["index_bytes"] / n, "kmer_k": info["kmer_k"], "ctx_depth": info["ctx_depth"],
                           "ctx_entry_bytes": info["ctx_entry_bytes"], "text_shortcut": info["text_shortcut"], "sigma": info["sigma"], "open_s": open_s, "checksum": checksum},
           "clocks": clocks, "e2e": e2e, "roofline": roof}
    if sustained:
        out["sustained"] = sustained
    state = {"g": g, "text": text, "base": base, "pats": pats, "sp": sp, "ep": ep, "cnt": cnt, "info": info, "fused": fused}
    return out, state


def ncu_traffic(m, info):
    """dram bytes per launch of the matching configuration from the committed ncu --set full capture (profiles/ncu_traffic.json)"""
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        try:
            for rec in json.load(open(tp)).get("count_fixed_kernel_captures", []):
                if (rec.get("queries") == m and rec.get("layout") == info["layout"] and rec.get("lanes") == info["lanes_per_query"]
                        and rec.get("kmer_k") == info["kmer_k"] and rec.get("ctx_depth", 0) == info["ctx_depth"] and rec.get("sigma") == info["sigma"]):
                    return rec.get("dram_bytes_per_launch")
        except Exception:
            pass
    return None


def cpu_count_baseline(orc, pats, sp, ep, cnt, unit=UNIT):
    """The oracle (C restatement of the reference algorithm) on the box's host cores, on a bounded sample of the same batch; doubles as
    the full-size parity check of that sample."""
    cores = os.cpu_count() or 1
    ln = pats.shape[1]
    rate = _probe(lambda k: orc.count_batch(pats[:k].reshape(-1), np.arange(0, k * ln + 1, ln, dtype=np.int64), threads=cores), 20000)
    sample = int(min(len(pats), max(20000, rate * 12.0)))
    off = np.arange(0, sample * ln + 1, ln, dtype=np.int64)
    t1 = time.time()
    osp, oep = orc.count_batch(pats[:sample].reshape(-1), off, threads=cores)
    dt = time.time() - t1
    parity = bool(np.array_equal(osp, np.where(cnt[:sample] > 0, sp[:sample], 0)) and np.array_equal(oep, np.where(cnt[:sample] > 0, ep[:sample], 0)))
    assert parity, "GPU (sp,ep) differ from the oracle on the CPU-baseline sample"
    one = int(min(sample, max(2000, rate / max(cores, 1) * 2.0)))     # single-thread figure (SURVEY §8d), about two seconds
    t1 = time.time()
    orc.count_batch(pats[:one].reshape(-1), off[:one + 1], threads=1)
    dt1 = time.time() - t1
    return {"value": sample / dt, "unit": unit, "cores": cores, "kind": "port",
            "sample": "first %d of the %d-query batch, %d threads, %.1f s" % (sample, len(pats), cores, dt), "parity_on_sample": parity,
            "note": "JVM unavailable - C restatement of the reference algorithm (binary search in .fm)",
            "single_thread": {"value": one / max(dt1, 1e-9), "unit": unit, "cores": 1, "sample": "first %d queries, %.1f s" % (one, dt1)}}


def load_oracle(base, what):
    from oracle import fm_oracle as fo
    t0 = time.time()
    fo.build(native=True)
    orc = fo.OracleIndex.load(base)
    log("%s: oracle index ready in %.1f s" % (what, time.time() - t0))
    return orc


# ------------------------------------------------------------------------------------------------ cfg 3 / cfg 4 on the English-like index
def english_open(cx, n):
    fx = cx.fx
    text, base = cx.ensure_index("cfg3", n)
    t0 = time.time()
    g = fx.GpuFMSearcher(base + ".bwt", bigEndian=True, device=cx.local, sa_sample_rate=32, max_total_bytes=cx.args.max_total_bytes)
    info = g.info()
    log("rank %d: cfg3 index open (%s, %.2f GB on device, k = %d, context depth %d) after %.1f s" % (cx.rank, info["layout"], info["index_bytes"] / 1e9,
                                                                                             info["kmer_k"], info["ctx_depth"], time.time() - t0))
    return text, base, g, dict(info, open_s=time.time() - t0)


def locate_leg(cx, g, text, n, m_total, ln, orc, steps, chunk_q=4000):
    """cfg 3: m_total len-`ln` text substrings (seed 5) in all, sharded over the ranks (strong scaling); count -> locate EVERY occurrence
    (sampled SA, rate 32) -> positions ascending per query.  On English-like text a len-12 pattern has ~10^5 occurrences on average
    (up to millions), so the batch is walked in chunks of `chunk_q` queries whose positions fit one device buffer; inside a chunk
    everything is device-resident: counts, scanned offsets and positions stay in HBM and, with N > 1, are exchanged by kernel stores
    into every rank's gathered buffers (sharded.GpuExchange)."""
    from findex_b200 import sharded
    torch, fx, world, rank = cx.torch, cx.fx, cx.world, cx.rank
    pats_all, _ = make_queries(text, m_total, ln, 5, 0, workload="cfg3")
    st = torch.cuda.current_stream().cuda_stream
    nchunk = (m_total + chunk_q - 1) // chunk_q
    chunks = []                                            # (global lo, global hi, device patterns of this rank's part)
    for c in range(nchunk):
        c0, c1 = c * chunk_q, min(m_total, (c + 1) * chunk_q)
        lo, hi = sharded.shard_bounds(c1 - c0, rank, world)
        chunks.append((c0 + lo, c0 + hi, c0, c1, torch.from_numpy(np.ascontiguousarray(pats_all[c0 + lo:c0 + hi])).to(cx.dev)))
    mloc = max(hi - lo for lo, hi, _, _, _ in chunks)
    d_sp = torch.zeros(max(mloc, 1), dtype=torch.int32, device=cx.dev)
    d_ep = torch.zeros(max(mloc, 1), dtype=torch.int32, device=cx.dev)
    d_off = torch.zeros(mloc + 1, dtype=torch.int64, device=cx.dev)
    # pre-pass (setup): hit counts of every chunk, to size the position buffers once
    loc_tot, sp_all, ep_all = [], [], []
    for lo, hi, _, _, d_pat in chunks:
        g.count_fixed_dev(d_pat.data_ptr(), ln, hi - lo, d_sp.data_ptr(), d_ep.data_ptr(), st)
        torch.cuda.synchronize()
        sp_all.append(d_sp[:hi - lo].cpu().numpy().astype(np.int64) & 0xFFFFFFFF)
        ep_all.append(d_ep[:hi - lo].cpu().numpy().astype(np.int64) & 0xFFFFFFFF)
        assert (ep_all[-1] > sp_all[-1]).all(), "a text substring was not found"
        loc_tot.append(int((ep_all[-1] - sp_all[-1]).sum()))
    tt = torch.tensor(loc_tot, dtype=torch.float64, device=cx.dev)
    if world > 1:
        cx.dist.all_reduce(tt)
    glob_tot = [int(x) for x in tt.cpu().tolist()]
    total_local, total_all = sum(loc_tot), sum(glob_tot)
    cap_local = max(loc_tot) + 16
    d_pos = torch.zeros(cap_local, dtype=torch.int32, device=cx.dev)
    ex = sharded.GpuExchange(g, rank, world, chunk_q, max(glob_tot) + 16, cx.dev) if world > 1 else None
    last = {}

    def step():
        for ci, (lo, hi, c0, c1, d_pat) in enumerate(chunks):
            if ex is not None:
                last["off"], _ = ex.locate(d_pat, ln, lo - c0, hi - c0, cap_local)
            else:
                g.count_fixed_dev(d_pat.data_ptr(), ln, hi - lo, d_sp.data_ptr(), d_ep.data_ptr(), st)
                g.locate_dev(d_sp.data_ptr(), d_ep.data_ptr(), hi - lo, d_off.data_ptr(), d_pos.data_ptr(), cap_local, st)
    g.set_stats(True)
    lf_steps = 0
    walk_ms = sort_ms = 0.0
    for ci, (lo, hi, c0, c1, d_pat) in enumerate(chunks):     # instrumented pass (untimed): LF steps per occurrence, walk/sort split
        g.count_fixed_dev(d_pat.data_ptr(), ln, hi - lo, d_sp.data_ptr(), d_ep.data_ptr(), st)
        g.locate_dev(d_sp.data_ptr(), d_ep.data_ptr(), hi - lo, d_off.data_ptr(), d_pos.data_ptr(), cap_local, st)
        lf_steps += g.last_steps()
        if nchunk > 8 and ci >= 3:                             # a sample of the chunks is enough for the per-occurrence figures
            break
    stat_occ = sum(loc_tot[:ci + 1])
    g.set_stats(False)
    for ci2, (lo, hi, c0, c1, d_pat) in enumerate(chunks[:ci + 1]):
        g.count_fixed_dev(d_pat.data_ptr(), ln, hi - lo, d_sp.data_ptr(), d_ep.data_ptr(), st)
        g.locate_dev(d_sp.data_ptr(), d_ep.data_ptr(), hi - lo, d_off.data_ptr(), d_pos.data_ptr(), cap_local, st)
        a, b = g.last_locate_ms()
        walk_ms += a
        sort_ms += b
    ms, clocks = cx.timed(step, steps, 1 if nchunk > 8 else 2)
    launches = int(g.last_kernel_launches())
    cx.launches += (steps + 2) * nchunk * (launches * 8 + 2)
    # ---- parity (last chunk): count vs the oracle; positions complete (count matches), ascending, and every one a real occurrence of the
    # pattern in the text — which makes them exactly sorted { sa[r] : r in [sp, ep) } (util.scala:213-224)
    lo, hi, c0, c1, d_pat = chunks[-1]
    sp, ep = sp_all[-1], ep_all[-1]
    occ = ep - sp
    pats = pats_all[lo:hi]
    if ex is not None:
        off_all = last["off"].cpu().numpy()
        pos_view = ex.gathered_values(int(off_all[c1 - c0]))
        off_local = off_all[lo - c0:hi - c0 + 1] - off_all[lo - c0]
        pos_local = pos_view[int(off_all[lo - c0]):int(off_all[hi - c0])]
    else:
        off_local = d_off[:hi - lo + 1].cpu().numpy()
        pos_local = d_pos[:loc_tot[-1]]
    assert off_local[-1] == loc_tot[-1] and np.array_equal(np.diff(off_local), occ)
    rng = np.random.default_rng(99)
    bad = 0
    chk = rng.choice(hi - lo, min(1500, hi - lo), replace=False)
    n1 = g.n
    for j in chk:
        q = pos_local[int(off_local[j]):int(off_local[j]) + min(int(occ[j]), 8192)].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
        if len(q) > 1 and not (np.diff(q) > 0).all():
            bad += 1
            continue
        qq = q[:: max(1, len(q) // 64)]
        fo_ = (n1 - 1) - qq - ln                                      # file offset = (n-1) - pos - len
        if not (text[fo_[:, None] + np.arange(ln)[None, :]] == pats[j][::-1][None, :]).all():
            bad += 1
    assert bad == 0, "located positions are not the pattern's occurrences"
    parity = {"positions_verified_queries": int(len(chk)), "mismatches": bad}
    if orc is not None:
        parity["count_parity_on_sample"], parity["count_parity_sample"] = oracle_parity(orc, pats, sp, ep, 100_000)
        assert parity["count_parity_on_sample"]
    # ---- e2e: host (sp, ep) in, host int64 positions out through fmx_locate_batch (pinned buffers), on a time-bounded slice of the shard
    sp0, ep0 = sp_all[0], ep_all[0]
    k = int(min(len(sp0), max(1, np.searchsorted(np.cumsum(ep0 - sp0), 120e6))))
    tot_k = int((ep0[:k] - sp0[:k]).sum())
    h_pos = fx.PinnedArray((max(tot_k, 1),), np.int64)
    h_off = np.zeros(k + 1, np.int64)
    sp_k, ep_k = np.ascontiguousarray(sp0[:k]), np.ascontiguousarray(ep0[:k])

    def e2e_step():
        rc = fx.lib().fmx_locate_batch(g.h, sp_k.ctypes.data, ep_k.ctypes.data, k, tot_k, h_off.ctypes.data, h_pos.array.ctypes.data)
        assert rc == 0, fx.lib().fmx_last_error()
    e2e_steps = max(2, min(steps, 5))
    ms_e2e, _ = cx.timed(e2e_step, e2e_steps, 1, wall=True, sample_clocks=False)
    hp = h_pos.array[:tot_k]
    assert all((np.diff(hp[h_off[j]:h_off[j + 1]]) > 0).all() for j in range(0, k, max(1, k // 50))), "host locate: positions not ascending"
    h_pos.free()
    per = ms / steps
    # one LF step of the sampled walk = one walk block (BWT byte + mark bit) + one rank block; plus the mark-rank block and the sample
    req_occ = 2.0 * lf_steps / max(stat_occ, 1) + 2.0
    r_rand_gbs, _ = g.gather_bench(64, 4, 1 << 25, 16, 3)
    peak, peak_src = measured_peaks()
    L = max(1, int(np.ceil(np.log2(max(g.info()["sigma"], 2)))))
    kern_ms = max(walk_ms + sort_ms, 1e-9)
    out = {"value": m_total / (per * 1e-3), "unit": UNIT, "positions_per_s": total_all / (per * 1e-3), "ms_per_step": per, "steps": steps, "queries": m_total,
           "occurrences": total_all, "occurrences_per_query": total_all / m_total, "pattern_len": ln, "sa_sample_rate": 32, "scaling": "strong",
           "chunks": nchunk, "queries_per_chunk": chunk_q, "walk_ms_sampled_chunks": walk_ms, "sort_ms_sampled_chunks": sort_ms,
           "sort_share_of_locate": sort_ms / kern_ms, "clocks": clocks, "parity_on_sample": bad == 0 and parity.get("count_parity_on_sample", True), "parity": parity,
           "exchange": "none" if ex is None else "kernel stores of counts + position slabs into every rank's gathered buffer (CUDA IPC) + 2 x 4-byte NCCL barrier per chunk",
           "e2e": {"value": cx.world * k / (ms_e2e / e2e_steps * 1e-3), "unit": UNIT, "positions_per_s": cx.world * tot_k / (ms_e2e / e2e_steps * 1e-3),
                   "ms_per_step": ms_e2e / e2e_steps, "queries": k, "h2d_bytes_per_step": k * 12 + 8, "d2h_bytes_per_step": tot_k * 8,
                   "api": "fmx_locate_batch (host int64 intervals in, pinned int64 positions out)", "slice": "first %d queries of the shard (%d positions; time-bounded)" % (k, tot_k)},
           "roofline": {"bound": "hbm", "unit": "GB/s", "achieved": req_occ * 64 * stat_occ / (kern_ms * 1e-3) / 1e9, "peak": peak, "peak_source": peak_src,
                        "frac": req_occ * 64 * stat_occ / (kern_ms * 1e-3) / 1e9 / peak, "traffic": None, "kernel": "locate_kernel (+ radix sort of the (query, position) keys)",
                        "kernel_ms": kern_ms, "lf_steps_per_occurrence": lf_steps / max(stat_occ, 1), "requests_per_occurrence": req_occ,
                        "request_rate": {"achieved_requests_per_s": req_occ * stat_occ / (max(walk_ms, 1e-9) * 1e-3), "r_rand_requests_per_s": r_rand_gbs * 1e9 / 64,
                                         "frac": req_occ * stat_occ / (max(walk_ms, 1e-9) * 1e-3) / (r_rand_gbs * 1e9 / 64)},
                        "survey_units": {"bytes_per_occurrence": 15.5 * L * 64 + 32, "note": "SURVEY 8(d): (rate-1)/2 LF steps x L x 64 B + one 32-B sample"}}}
    if ex is not None:
        ex.retire()
    return out


def regex_leg(cx, g, text, n_regexes, orc, steps):
    """cfg 4: `n_regexes` template regexes per GPU (SURVEY §8d: classes, alternation, desugared bounded repeats, \\d, '.') over the index,
    compiled once into a device-resident set.  value: device-resident search (traversal + ordering, results left in HBM); e2e: the host
    call fmx_regex_set_search (results to host buffers)."""
    import ctypes as C
    torch, fx = cx.torch, cx.fx
    rxs = cx.synth.regex_templates(text, np.random.default_rng([6, cx.rank]), n_regexes)
    t0 = time.time()
    trees, kept = [], []
    for r in rxs:
        try:
            trees.append(fx.ReTree(r))
            kept.append(r)
        except fx.FmxError:
            pass
    compile_s = time.time() - t0
    mr = len(trees)
    if cx.world > 1:                                       # equal shards: every rank searches the same number of regexes
        mr = int(-cx.max_over_ranks(-mr))
        trees, kept = trees[:mr], kept[:mr]
    t0 = time.time()
    rset = g.regex_set(trees)
    upload_s = time.time() - t0
    cap = 1 << 22
    off = np.zeros(mr + 1, np.int64)
    ln_, sp_, ep_ = fx.PinnedArray((cap,), np.int32), fx.PinnedArray((cap,), np.int64), fx.PinnedArray((cap,), np.int64)
    d_res = torch.zeros((cap, 4), dtype=torch.int32, device=cx.dev)
    d_off = torch.zeros(mr + 1, dtype=torch.int64, device=cx.dev)
    totals = []
    ex = None
    if cx.world > 1:
        # N > 1: the records of every rank's shard are exchanged on the device (sharded.GpuExchange): per-regex counts and the
        # {regex, len, sp, ep} slabs go by kernel stores into every rank's gathered buffers, 2 x 4-byte NCCL barrier
        from findex_b200 import sharded
        torch.cuda.synchronize()                           # d_res/d_off fills are on torch's stream, the search on the library's
        first = rset.search_dev(g, d_res.data_ptr(), cap, d_off.data_ptr())
        all_res = int(cx.sum_over_ranks(first))
        ex = sharded.GpuExchange(g, cx.rank, cx.world, cx.world * mr, 4 * all_res + 64, cx.dev)

    torch.cuda.synchronize()

    def dev_step():
        if ex is not None:
            _, t_ = ex.regex(rset, cx.rank * mr, (cx.rank + 1) * mr, cap)
            totals.append(t_)
        else:
            totals.append(rset.search_dev(g, d_res.data_ptr(), cap, d_off.data_ptr()))

    def host_step():
        rc = fx.lib().fmx_regex_set_search(g.h, rset.h, cap, off.ctypes.data_as(C.c_void_p), C.c_void_p(ln_.array.ctypes.data),
                                           C.c_void_p(sp_.array.ctypes.data), C.c_void_p(ep_.array.ctypes.data))
        assert rc == 0, fx.lib().fmx_last_error()
    steps = max(3, min(steps, 20))
    kms = []

    def dev_step_timed():
        dev_step()
        kms.append(g.last_kernel_ms())
    ms_dev, clocks = cx.timed(dev_step_timed, steps, 3, wall=True)
    kms = kms[-steps:]
    items = g.last_steps()
    launches = int(g.last_kernel_launches())
    max_len = int(g.last_regex_levels())
    ms_e2e, _ = cx.timed(host_step, steps, 2, wall=True, sample_clocks=False)
    cx.launches += (2 * steps + 5) * launches
    total = int(off[mr])
    assert total == totals[-1], "device-resident and host searches disagree on the number of results"
    if ex is not None:                                     # this rank's records inside the gathered buffer
        goff = ex.offsets().cpu().numpy()
        lo_w, hi_w = int(goff[cx.rank * mr]), int(goff[(cx.rank + 1) * mr])
        rec = ex.gathered_values(4 * int(goff[-1])).reshape(-1, 4)[lo_w:hi_w].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
        want_ids = np.repeat(np.arange(cx.rank * mr, (cx.rank + 1) * mr), np.diff(off))
        assert hi_w - lo_w == total, "gathered offsets give this rank %d records, it produced %d (all ranks: %d)" % (hi_w - lo_w, total, int(goff[-1]))
        assert np.array_equal(rec[:, 0], want_ids), "regex ids of the gathered records differ at %d of %d places (first: got %s want %s)" % (
            int((rec[:, 0] != want_ids).sum()), total, rec[:, 0][rec[:, 0] != want_ids][:4].tolist(), want_ids[rec[:, 0] != want_ids][:4].tolist())
    else:
        rec = d_res[:total].cpu().numpy().astype(np.int64) & 0xFFFFFFFF
    assert np.array_equal(rec[:, 1], ln_.array[:total]) and np.array_equal(rec[:, 2], sp_.array[:total]) and np.array_equal(rec[:, 3], ep_.array[:total])
    occurrences = int((ep_.array[:total] - sp_.array[:total]).sum())
    sample = [(kept[i], sorted(zip(ln_.array[off[i]:off[i + 1]].tolist(), sp_.array[off[i]:off[i + 1]].tolist(), ep_.array[off[i]:off[i + 1]].tolist())))
              for i in np.random.default_rng(9).choice(mr, min(200, mr), replace=False)]
    dev_ms = float(np.mean(kms)) if ex is None else ms_dev / steps          # N > 1: the step includes the exchange (wall clock, max over ranks)
    out = {"value": cx.world * mr / (dev_ms * 1e-3), "unit": "regexes/s", "ms_per_step": dev_ms, "steps": steps,
           "exchange": "none" if ex is None else "kernel stores of per-regex counts + record slabs into every rank's gathered buffer (CUDA IPC) + 2 x 4-byte NCCL barrier",
           "kernel_ms_per_step": float(np.mean(kms)),
           "what": "fmx_regex_set_search_dev: Glushkov engine, caps off, device-resident regex set; traversal (work-queue kernel) + ordering on the device, CUDA-event time",
           "call_value": cx.world * mr * steps / (ms_dev * 1e-3), "call_ms_per_step": ms_dev / steps,
           "regexes_per_gpu": mr, "rejected_by_compiler": len(rxs) - mr, "result_triples": total, "occurrences_covered": occurrences, "items_processed": int(items),
           "longest_match": max_len, "kernel_launches_per_step": launches, "clocks": clocks, "compile_s_once": compile_s, "set_upload_s_once": upload_s,
           "e2e": {"value": cx.world * mr * steps / (ms_e2e * 1e-3), "unit": "regexes/s", "ms_per_step": ms_e2e / steps, "h2d_bytes_per_step": 0,
                   "d2h_bytes_per_step": total * 20 + (mr + 1) * 8, "api": "fmx_regex_set_search (device-resident set, host result buffers)"}}
    # one item = one backward step = at most two rank-block requests + the 16-byte state record and the ring slot
    r_rand_gbs, _ = g.gather_bench(64, 4, 1 << 25, 16, 3)
    peak, peak_src = measured_peaks()
    out["roofline"] = {"bound": "hbm", "unit": "GB/s", "achieved": items * 2 * 64 / (float(np.mean(kms)) * 1e-3) / 1e9, "peak": peak, "peak_source": peak_src,
                       "frac": items * 2 * 64 / (float(np.mean(kms)) * 1e-3) / 1e9 / peak, "traffic": None, "kernel": "regex_queue_kernel", "kernel_ms": float(np.mean(kms)),
                       "items_per_regex": items / max(mr, 1), "request_rate": {"achieved_requests_per_s": items * 2 / (float(np.mean(kms)) * 1e-3),
                                                                              "r_rand_requests_per_s": r_rand_gbs * 1e9 / 64,
                                                                              "frac": items * 2 / (float(np.mean(kms)) * 1e-3) / (r_rand_gbs * 1e9 / 64)},
                       "note": "algorithmic bytes = items x one backward step (2 x 64-B rank blocks, SURVEY 8(d): 'one frontier expansion = one backward step')"}
    if orc is not None:
        cores = os.cpu_count() or 1
        tabs = [_oracle_compile(rx) for rx, _ in sample]
        t1 = time.time()
        got = _oracle_regex(orc, tabs, cores)
        dtr = time.time() - t1
        ok = all(a == want for a, (_, want) in zip(got, sample))
        assert ok, "GPU regex results differ from the oracle on the sample"
        out["parity_on_sample"] = bool(ok)
        out["cpu_baseline"] = {"value": len(sample) / dtr, "unit": "regexes/s", "cores": cores, "kind": "port",
                               "sample": "%d regexes of the batch (ReTree._matchSA, caps off, automata precompiled), %d threads, %.2f s" % (len(sample), cores, dtr),
                               "parity_on_sample": bool(ok)}
    if ex is not None:
        ex.retire()
    rset.close()
    for a in (ln_, sp_, ep_):
        a.free()
    return out


# ------------------------------------------------------------------------------------------------ drivers
class RunGuard:
    """Keeps a run bounded and its ranks in step across the secondary legs.

    * agreement: at N > 1 every leg ends with the ranks telling each other, through the process group's c10d store (host side, no NCCL
      stream involved), whether the leg succeeded.  A leg that failed on ANY rank counts as failed on all, and the remaining legs are
      skipped everywhere — a rank that went on alone would pair its collectives with the wrong ones of its peers and hang the job
      (seen on 8 x B200: two ranks lost a file race, the other six waited for them inside an all-reduce until the box's time limit).
    * watchdog: every leg (and the headline, and the teardown) has a time limit.  When one is exceeded — a rank stuck in a collective
      whose partner is gone — rank 0 prints the JSON line with what has been measured so far and every rank leaves with os._exit."""

    def __init__(self):
        self.rank, self.world, self.store = 0, 1, None
        self.broken = None                                   # name of the leg that failed on some rank (N > 1)
        self.out, self.printed = None, False
        self.limits = []                                     # stack of (name, deadline)
        self.seq = 0
        self.lock = threading.Lock()
        self.thread = None

    def attach(self, rank, world):
        self.rank, self.world = rank, world
        if world > 1:
            try:
                from torch.distributed import distributed_c10d as c10d
                self.store = c10d._get_default_store()
            except Exception as e:                           # noqa: BLE001
                log("rank %d: no c10d store for the leg agreement (%s); the watchdog alone bounds the run" % (rank, e))
        if self.thread is None:
            self.thread = threading.Thread(target=self._watch, daemon=True)
            self.thread.start()

    def push(self, name, seconds):
        with self.lock:
            self.limits.append((name, time.time() + seconds))

    def pop(self):
        with self.lock:
            if self.limits:
                self.limits.pop()

    def _watch(self):
        while True:
            time.sleep(1.0)
            with self.lock:
                late = [n for n, d in self.limits if time.time() > d]
            if late:
                self._fire(late[0])

    def _fire(self, name):
        log("rank %d: watchdog: '%s' exceeded its time limit — ending the run with what has been measured" % (self.rank, name))
        code = 0
        if self.rank == 0 and not self.printed:
            if self.out is not None:
                try:
                    self.emit(dict(self.out, watchdog="'%s' exceeded its time limit; later legs were not run" % name))
                except Exception as e:                       # noqa: BLE001
                    log("watchdog: could not print the partial line: %s" % e)
                    code = 3
            else:
                code = 3                                     # nothing measured yet
        sys.stderr.flush()
        os._exit(code)

    def emit(self, out):
        """the ONE JSON line (rank 0)"""
        with self.lock:
            if self.printed:
                return
            self.printed = True
        print(json.dumps(out), file=OUT, flush=True)

    def agree(self, name, ok, timeout_s=180):
        """True iff the leg succeeded on every rank (same answer on every rank, barring a timeout)"""
        if self.world == 1 or self.store is None:
            return ok
        from datetime import timedelta
        self.seq += 1
        keys = ["fmxleg/%d/%d" % (self.seq, r) for r in range(self.world)]
        try:
            self.store.set(keys[self.rank], "1" if ok else "0")
            self.store.wait(keys, timedelta(seconds=timeout_s))
            return all(bytes(self.store.get(k)) == b"1" for k in keys)
        except Exception as e:                               # noqa: BLE001 — a peer never got here
            log("rank %d: leg '%s': no answer from every rank (%s: %s)" % (self.rank, name, type(e).__name__, str(e)[:200]))
            return False


GUARD = RunGuard()


def guarded(name, fn, limit_s=480):
    """a secondary leg must not take the headline down with it — nor, at N > 1, leave the ranks out of step (RunGuard)"""
    if GUARD.broken is not None:
        log("leg %s skipped: leg '%s' failed on some rank" % (name, GUARD.broken))
        return {"skipped": "leg '%s' failed on some rank" % GUARD.broken}
    GUARD.push(name, limit_s)
    t0 = time.time()
    try:
        r, ok = fn(), True
    except Exception as e:                                           # noqa: BLE001
        log("leg %s FAILED:\n%s" % (name, traceback.format_exc()))
        r, ok = {"error": "%s: %s" % (type(e).__name__, e)}, False
    if GUARD.world > 1 and not GUARD.agree(name, ok):
        GUARD.broken = name
        if ok:
            r = {"error": "leg failed on another rank", "this_rank": r if isinstance(r, dict) and len(json.dumps(r, default=str)) < 4000 else "ok"}
    elif ok:
        log("leg %s done in %.1f s" % (name, time.time() - t0))
    GUARD.pop()
    return r


def run_default(cx):
    args, fx = cx.args, cx.fx
    extras = set(args.legs.split(",")) if args.legs else set()
    if cx.world > 1:
        extras -= {"sweep"}                                  # single-GPU characterisation; the scaling runs carry the multi-GPU legs
    n, m, ln = args.text_bytes, args.queries, args.len
    numa = numa_report(cx.local)
    out, stt = count_workload(cx, "cfg2", n, m, ln, extras)
    GUARD.out = out                                          # from here on a partial line can be printed
    out["host"] = {"numa": numa, "cores": os.cpu_count()}
    g, text, base = stt["g"], stt["text"], stt["base"]
    scale = n / DEFAULTS["cfg2"][0]
    orc = None
    if cx.world == 1 and cx.rank == 0 and not args.no_cpu:
        orc = load_oracle(base, "cfg2")
        out["cpu_baseline"] = guarded("cpu_baseline", lambda: cpu_count_baseline(orc, stt["pats"], stt["sp"], stt["ep"], stt["cnt"]))
    if "sweep" in extras:
        def sweep():
            ms = max(1000, min(m, int(4_000_000 * min(1.0, scale * 10))))
            recs = sweep_leg(cx, g, text, [8, 12, 16, 20, 24, 32, 64], ms, 3, orc, "cfg2, all accelerators (k-mer table + row-context hops)")
            g.set_accel_mask(fx.ACCEL_NONE)
            recs += sweep_leg(cx, g, text, [16], ms, 3, orc, "cfg2, %s rank structure alone (no accelerators)" % stt["info"]["layout"].upper())
            g.set_accel_mask(fx.ACCEL_AUTO)
            return recs
        out["sweep"] = guarded("sweep", sweep)
    if stt["fused"] is not None:
        stt["fused"].close()
    g.close()
    if "sweep" in extras and cx.rank == 0:
        def wm():
            recs = []
            for lay, name in ((fx.LAYOUT_WM, "wavelet matrix alone (north_star's structure: binary levels, 64-byte blocks"),
                              (fx.LAYOUT_WMX, "multi-ary wavelet matrix alone (16-ary levels, 128-byte blocks")):
                gw = fx.GpuFMSearcher(base + ".bwt", bigEndian=True, device=cx.local, layout=lay, accel=fx.ACCEL_NONE)
                try:
                    info = gw.info()
                    r = sweep_leg(cx, gw, text, [16], max(1000, min(m, int(2_000_000 * min(1.0, scale * 10)))), 3, orc,
                                  "cfg2, %s; %.2f GB)" % (name, info["index_bytes"] / 1e9))[0]
                    r["index_bytes"] = info["index_bytes"]
                    r["lanes_per_query"] = info["lanes_per_query"]
                    if lay == fx.LAYOUT_WM:
                        r["dedup_bytes_per_query"] = r["requests_per_query"] * 64          # SURVEY 8(d)'s dedup figure: distinct 64-B blocks of a WM search
                    recs.append(r)
                finally:
                    gw.close()
            return recs
        wm_recs = guarded("wm", wm)
        if isinstance(out.get("sweep"), list) and isinstance(wm_recs, list):
            out["sweep"] += wm_recs
            out["roofline"]["survey_units"]["dedup_bytes_per_query"] = wm_recs[0]["dedup_bytes_per_query"]
    if orc is not None:
        orc.close()
        orc = None
    del stt, text
    cx.barrier()
    if "english" in extras and args.regexes > 0:
        def english():
            ne = max(100_000, int(DEFAULTS["cfg3"][0] * scale))
            text_e, base_e, ge, info_e = english_open(cx, ne)
            try:
                orc_e = load_oracle(base_e, "cfg3") if (cx.world == 1 and cx.rank == 0 and not args.no_cpu) else None
                res = {"index": {k: info_e[k] for k in ("layout", "index_bytes", "kmer_k", "ctx_depth", "dict_depth", "dict_chain_depth", "dict_entries", "dict_bytes",
                                                        "sigma", "sa_sample_rate", "open_s")}}
                mq = max(1000, min(m, int(4_000_000 * min(1.0, scale * 10))))

                def english_count():
                    recs = sweep_leg(cx, ge, text_e, [8, 12, 16, 24], mq, 5, orc_e, "cfg3 English-like, all accelerators (table + row contexts + dictionary of wide intervals)", workload="cfg3")
                    ge.set_accel_mask(fx.ACCEL_KMER | fx.ACCEL_CTX)             # the same index without the dictionary
                    try:
                        recs += sweep_leg(cx, ge, text_e, [12], mq, 5, orc_e, "cfg3 English-like, table + row contexts only", workload="cfg3")
                    finally:
                        ge.set_accel_mask(fx.ACCEL_AUTO)
                    return recs
                res["count"] = guarded("english count", english_count)
                ml = max(400, int(4000 * min(1.0, scale * 10)))      # ~5 x 10^8 occurrences at full size: one chunk, a fraction of a second per step
                res["locate"] = guarded("locate", lambda: locate_leg(cx, ge, text_e, ne, ml, 12, orc_e, max(2, min(args.steps, 5)), chunk_q=ml))
                res["regex"] = guarded("regex", lambda: regex_leg(cx, ge, text_e, args.regexes, orc_e, args.steps))
                if orc_e is not None:
                    orc_e.close()
                return res
            finally:
                ge.close()
        eng = guarded("english", english)
        out["english"] = eng
        for k in ("locate", "regex"):                                 # the two halves BASELINE names, also at the top level
            if isinstance(eng, dict) and k in eng:
                out[k] = eng[k]
    cx.barrier()
    if "cfg5" in extras:
        def cfg5():
            n5 = max(100_000, int(DEFAULTS["cfg5"][0] * scale))
            m5 = max(1000, int(DEFAULTS["cfg5"][1] * min(1.0, scale * 10)))
            sub = argparse.Namespace(**vars(args))
            sub.steps, sub.warmup = max(3, min(args.steps, 20)), 3
            cx5 = cx
            old = cx.args
            cx.args = sub
            try:
                o5, st5 = count_workload(cx5, "cfg5", n5, m5, 32, {"pcie"} & extras)
            finally:
                cx.args = old
            try:
                if cx.world == 1 and cx.rank == 0 and not args.no_cpu:
                    orc5 = load_oracle(st5["base"], "cfg5")
                    o5["parity_on_sample"], o5["parity_sample"] = oracle_parity(orc5, st5["pats"], st5["sp"], st5["ep"], 200_000)
                    assert o5["parity_on_sample"], "cfg5: GPU (sp,ep) differ from the oracle"
                    orc5.close()
                else:
                    # without the oracle (N > 1): the accelerated answers equal plain rank stepping over the same index, on the whole batch
                    st5["g"].set_accel_mask(fx.ACCEL_NONE)
                    _, sp2, ep2 = device_count_rate(cx, st5["g"], st5["pats"], reps=1)
                    o5["parity_vs_plain_steps"] = bool(np.array_equal(sp2, st5["sp"]) and np.array_equal(ep2, st5["ep"]))
                    assert o5["parity_vs_plain_steps"]
            finally:
                if st5["fused"] is not None:
                    st5["fused"].close()
                st5["g"].close()
            keep = ("value", "unit", "ms_per_step", "steps", "config", "impl_config", "e2e", "roofline", "clocks", "parity_on_sample", "parity_sample", "parity_vs_plain_steps")
            return {k: o5[k] for k in keep if k in o5}
        out["cfg5"] = guarded("cfg5", cfg5)
    out["gpu_launches"] = cx.launches
    return out


def run_workload(cx):
    """--workload cfg3 | cfg4 | cfg5 as top-level lines"""
    args, fx = cx.args, cx.fx
    w, n, m, ln = args.workload, args.text_bytes, args.queries, args.len
    extras = set(args.legs.split(",")) if args.legs else set()
    if w == "cfg5":
        out, stt = count_workload(cx, "cfg5", n, m, ln, extras)
        if cx.world == 1 and cx.rank == 0 and not args.no_cpu:
            orc = load_oracle(stt["base"], "cfg5")
            out["cpu_baseline"] = cpu_count_baseline(orc, stt["pats"], stt["sp"], stt["ep"], stt["cnt"])
            orc.close()
        if stt["fused"] is not None:
            stt["fused"].close()
        stt["g"].close()
        out["gpu_launches"] = cx.launches
        return out
    text, base, g, info = english_open(cx, n)
    orc = load_oracle(base, w) if (cx.world == 1 and cx.rank == 0 and not args.no_cpu) else None
    common = {"n_gpus": cx.world, "steps": args.steps if w != "cfg3" else max(1, min(args.steps, 2 if m > 50_000 else args.steps)), "warmup": args.warmup, "higher_is_better": True, "vs_baseline": None, "dtype": "u32", "data": "synthetic",
              "config": workload_config(args), "impl_config": {k: info[k] for k in ("layout", "index_bytes", "kmer_k", "ctx_depth", "sigma", "sa_sample_rate", "open_s")}}
    if w == "cfg3":
        leg = locate_leg(cx, g, text, n, m, ln, orc, max(1, min(args.steps, 2 if m > 50_000 else args.steps)), chunk_q=4000)
        out = dict(common, metric=METRICS[w], value=leg["value"], unit=UNIT, ms_per_step=leg["ms_per_step"], scaling="strong", clocks=leg["clocks"], e2e=leg["e2e"],
                   roofline=leg["roofline"], locate={k: v for k, v in leg.items() if k not in ("e2e", "roofline", "clocks")})
        if orc is not None:
            cores = os.cpu_count() or 1
            pats, _ = make_queries(text, m, ln, 5, 0, workload="cfg3")
            t1 = time.time()
            orc.sa()
            sa_s = time.time() - t1
            k = int(min(m, max(2000, _probe(lambda kk: _oracle_locate(orc, pats[:kk], ln, cores), 2000) * 10.0)))
            t1 = time.time()
            _oracle_locate(orc, pats[:k], ln, cores)
            dt = time.time() - t1
            out["cpu_baseline"] = {"value": k / dt, "unit": UNIT, "cores": cores, "kind": "port", "sample": "first %d queries: count + sorted sa[sp..ep), %d threads, %.1f s "
                                   "(+ %.1f s one-off suffix array walk = SACreator.create)" % (k, cores, dt, sa_s)}
    else:
        leg = regex_leg(cx, g, text, m, orc, args.steps)
        out = dict(common, metric=METRICS[w], value=leg["value"], unit="regexes/s", ms_per_step=leg["ms_per_step"], scaling="weak", clocks=leg["clocks"], e2e=leg["e2e"],
                   roofline=leg["roofline"], regex={k: v for k, v in leg.items() if k not in ("e2e", "roofline", "clocks", "cpu_baseline")})
        if "cpu_baseline" in leg:
            out["cpu_baseline"] = leg["cpu_baseline"]
    if orc is not None:
        orc.close()
    g.close()
    out["gpu_launches"] = cx.launches
    return out


def protect_stdout():
    """Libraries (NCCL prints its version) may write to fd 1; the contract is ONE JSON line on stdout.  Point fd 1 at stderr and
    keep the real stdout for the final line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(real, "w")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"],
                    help="cfg2 = the metric's config (default line, carries the other configs as extra legs); cfg3 locate, cfg4 regex, cfg5 DNA count as their own lines")
    ap.add_argument("--legs", default="sweep,sustained,pcie,english,cfg5", help="extra legs of the default line (comma separated; empty = headline only)")
    ap.add_argument("--text-bytes", type=int, default=None)
    ap.add_argument("--queries", type=int, default=None)
    ap.add_argument("--len", type=int, default=None)
    ap.add_argument("--layout", default="auto", choices=["auto", "wm", "planes"])
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--accel", default="auto", choices=["auto", "none", "kmer", "text", "both", "ctx"])
    ap.add_argument("--max-total-bytes", type=int, default=0, help="fmx_opts.max_total_bytes: cap on everything resident for an index")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"], help="N>1 count: fused peer-memory stores (default) or NCCL all-gather")
    ap.add_argument("--regexes", type=int, default=100_000, help="regexes per GPU of the regex leg")
    ap.add_argument("--chunk", type=int, default=0, help="queries per pipeline chunk of the host-buffer calls (0 = library default)")
    ap.add_argument("--no-cpu", action="store_true")
    args = ap.parse_args()
    dflt = DEFAULTS[args.workload]
    args.text_bytes = args.text_bytes or dflt[0]
    args.queries = args.queries or dflt[1]
    args.len = dflt[2] if args.len is None else args.len
    if args.warmup < 3:
        log("note: contract asks for >= 3 warm-up steps; got", args.warmup)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    global OUT
    OUT = protect_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    GUARD.attach(rank, world)
    GUARD.push("the whole run", 1500 if args.workload != "cfg3" else 7200)
    try:
        cx = Ctx(args, rank, world, local_rank)
        out = run_default(cx) if args.workload == "cfg2" else run_workload(cx)
        if rank == 0:
            GUARD.emit(out)
        GUARD.out = None
        GUARD.push("teardown", 90)                           # the line is out: nothing below may keep the job alive
        if world > 1 and GUARD.broken is None:               # exchange buffers live as long as the process group: unmap, barrier, free
            from findex_b200 import sharded
            torch.cuda.synchronize()
            sharded.close_retired(cx.barrier)
    finally:
        if world > 1:
            if GUARD.broken is not None:                     # ranks possibly out of step: no collective teardown
                sys.stdout.flush()
                sys.stderr.flush()
                os._exit(0 if (GUARD.printed or rank != 0) else 1)
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()

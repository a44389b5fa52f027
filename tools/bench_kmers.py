"""
tools/bench_kmers.py — the k-mer census (fmx_kmer_spectrum, fmx_kmer_list_dev) on bench.py's cfg-2 and cfg-3 indexes and on a DNA
index (cfg 5's text at 10^9 symbols), each opened with the LCP structure.

    python tools/bench_kmers.py [--configs cfg2,cfg3,dna] [--scale 1.0] [--out-dir profiles]

The texts and index files are bench.py's (same seeds, same cached files in the temporary directory).  For every k the spectrum and the
listings (min_count, max_count) = (2, 0), (100, 0) and (1, 1) are timed with CUDA events over at least one second each and reported as
rows/s, model bytes, GB/s and that rate as a share of the 7.7 TB/s HBM3e data-sheet figure of one B200 (a data-sheet figure, not a
measured peak).  The model bytes are the n bytes of lcp8, plus the records and escaped values when k > 255 (bounded by lcp_bytes), plus
the 8 bytes of each listed interval; a listing reads lcp8 twice (a counting pass and an emitting pass), the model counts it once.
The same spectrum is then computed through the count path that existed before the census, on the same index: fmx_count_fixed_dev over
every window of T' in chunks, torch.unique of the rows and a bincount of the counts.  It must equal the census exactly (histogram at
1000 buckets, distinct, max_occ); both times are reported.  One JSON record per config goes to <out-dir>/r06_kmers_<config>.json; the
card's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KS = {"cfg2": (4, 8, 16, 32), "cfg3": (8, 16, 32, 300), "dna": (11, 21, 31)}
LISTINGS = [(2, 0), (100, 0), (1, 1)]
BUCKETS = 1000
DATASHEET_BPS = 7.7e12
CHUNK = 1 << 26


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn, min_s=1.0, warmup=2):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps, ms = 0, 0.0
    while ms < min_s * 1e3:
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms += e0.elapsed_time(e1)
        steps += 1
    return steps, ms


def rate(n, model_bytes, ms):
    s = ms / 1e3
    return {"ms": ms, "rows_per_s": n / s, "model_bytes": model_bytes, "model_GB_per_s": model_bytes / s / 1e9,
            "share_of_7.7TBps_datasheet": model_bytes / s / DATASHEET_BPS}


def baseline_spectrum(g, tp, k, fx):
    """the spectrum through the count path: every T' window counted (uint32 rows), torch.unique of the sp, bincount of the counts"""
    import torch
    W = len(tp) - k + 1
    sp = torch.empty(W, dtype=torch.int32, device="cuda")
    chunk = max(1 << 20, min(CHUNK, (1 << 31) // k))                       # at most 2 GB of pattern bytes per chunk
    ep = torch.empty(min(W, chunk), dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for a in range(0, W, chunk):
        c = min(chunk, W - a)
        pats = tp[a:a + c + k - 1].unfold(0, k, 1).contiguous()
        g.count_fixed_dev(pats.data_ptr(), k, c, sp[a:].data_ptr(), ep.data_ptr(), stream)
    _, counts = torch.unique(sp, return_counts=True)
    hist = torch.bincount(torch.clamp(counts, max=BUCKETS) - 1, minlength=BUCKETS)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1), hist.cpu().numpy().astype(np.int64), int(counts.numel()), int(counts.max().item())


def run_config(w, scale, fx, bench):
    import torch
    src = "cfg5" if w == "dna" else w
    n = max(100_000, int(1_000_000_000 * scale))
    t0 = time.time()
    text = np.asarray(bench.make_text(n, src), np.uint8)
    base = bench.index_base(n, src)
    if not (os.path.exists(base + ".bwt") and os.path.exists(base + ".aux")):
        fx.build_index_files(text, base, bigEndian=True)
    prep_s = time.time() - t0
    t0 = time.time()
    g = fx.GpuFMSearcher(base + ".bwt", bigEndian=True, device=0, lcp=1)
    open_s = time.time() - t0
    info = g.info()
    N = g.n
    Fz = text[text != 0]
    tp = torch.from_numpy(np.ascontiguousarray(Fz[::-1])).cuda()
    del text
    L = fx.lib()
    stream = torch.cuda.current_stream().cuda_stream
    recs = []
    for k in KS[w]:
        esc_bytes = info["lcp_bytes"] - N if k > 255 else 0
        hist, distinct, max_occ = g.kmer_spectrum(k, BUCKETS)
        steps, ms = timed(lambda: g.kmer_spectrum(k, BUCKETS))
        r = {"k": k, "distinct": distinct, "max_occ": max_occ, "spectrum": dict(rate(N, N + esc_bytes, ms / steps), steps=steps)}
        for mn, mx in LISTINGS:
            tot = C.c_int64()
            rc = L.fmx_kmer_list_dev(g.h, k, mn, mx, None, None, 0, C.byref(tot), C.c_void_p(stream))
            assert rc in (fx.FMX_OK, fx.FMX_E_CAPACITY), rc
            T = tot.value
            d_sp = torch.empty(max(T, 1), dtype=torch.int32, device="cuda")
            d_ep = torch.empty(max(T, 1), dtype=torch.int32, device="cuda")
            steps, ms = timed(lambda: g.kmers_dev(k, d_sp.data_ptr(), d_ep.data_ptr(), T, mn, mx, stream))
            r["list_%d_%d" % (mn, mx)] = dict(rate(N, N + esc_bytes + 8 * T, ms / steps), steps=steps, listed=T)
            del d_sp, d_ep
            torch.cuda.empty_cache()
        bms, bhist, bdistinct, bmax = baseline_spectrum(g, tp, k, fx)
        torch.cuda.empty_cache()
        assert np.array_equal(bhist, hist) and bdistinct == distinct and bmax == max_occ, ("baseline differs", w, k)
        r["count_path_baseline"] = {"ms": bms, "windows": int(len(Fz) - k + 1), "equal_to_census": True,
                                    "speedup_of_census": bms / r["spectrum"]["ms"]}
        print(json.dumps({"config": w, **r}), flush=True)
        recs.append(r)
    rec = {"config": w, "n": int(N), "card": card(), "torch_device": torch.cuda.get_device_name(0), "layout": info["layout"],
           "lcp_bytes": info["lcp_bytes"], "lcp_bytes_per_n": info["lcp_bytes"] / N, "buckets": BUCKETS, "open_s_with_lcp": round(open_s, 2),
           "text_and_files_s": round(prep_s, 1), "ks": recs}
    g.close()
    del tp
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg2,cfg3,dna")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the 10^9-symbol texts")
    ap.add_argument("--out-dir", default=None, help="write r06_kmers_<config>.json here")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_kmers.py measures the GPU; there is no CPU path"
    from findex_b200 import build
    build.build()
    from findex_b200 import fmindex as fx
    import bench
    for w in a.configs.split(","):
        rec = run_config(w, a.scale, fx, bench)
        line = json.dumps(rec)
        print(line, flush=True)
        if a.out_dir:
            os.makedirs(a.out_dir, exist_ok=True)
            with open(os.path.join(a.out_dir, "r06_kmers_%s.json" % w), "w") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()

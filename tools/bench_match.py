"""
tools/bench_match.py — SMEMs (fmx_smem_dev) on the cfg-2 byte index and on a DNA index (cfg 5's text, by default at a quarter of its size).

    python tools/bench_match.py [--configs cfg2,cfg5] [--scale 1.0] [--dna-scale 0.25] [--reads 1000000] [--out profiles/r05_match.json]

The texts and index files are bench.py's (same seeds, same cached files in the temporary directory).  Each index is opened without and
with the LCP structure (open times and lcp_bytes / n reported).  The reads are 150 symbols taken from the text with 1 % substitutions,
plus 10 % random reads (seeded).  fmx_smem_dev (min_len 16) is timed with CUDA events, as reads/s and query symbols/s; an untimed
counting run gives the index requests per query symbol by kind, printed beside the model's bound (at most 2 backward steps and one
widening per symbol); the request rate is set against fmx_gather_bench's 64-byte random-gather rate on the same index.  Every SMEM of one
timed step is checked through the count path: count(reverse(match)) = its interval, and the match grown by one symbol on either side
does not occur.  One JSON line per config goes to --out (appended); the card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

READ_LEN, SUB, RANDOM_FRAC, MIN_LEN = 150, 0.01, 0.10, 16


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make_reads(text, m, seed):
    rng = np.random.default_rng(seed)
    alpha = np.unique(text[: 1 << 24])
    st = rng.integers(0, len(text) - READ_LEN, m)
    R = text[st[:, None] + np.arange(READ_LEN)]
    mask = rng.random(R.shape) < SUB
    R[mask] = alpha[rng.integers(0, len(alpha), int(mask.sum()))]
    k = int(m * RANDOM_FRAC)
    R[:k] = alpha[rng.integers(0, len(alpha), (k, READ_LEN))]
    return np.ascontiguousarray(R)


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


def check(g, R, oo, st, ln, sp, ep):
    """every SMEM through the count path"""
    m = len(R)
    q_of = np.repeat(np.arange(m), np.diff(oo))
    pats, grow, want = [], [], []
    for k in range(len(st)):
        r = R[q_of[k]]
        s, l = int(st[k]), int(ln[k])
        pats.append(r[s:s + l][::-1].tobytes())
        want.append((int(sp[k]), int(ep[k])))
        if s > 0:
            grow.append(r[s - 1:s + l][::-1].tobytes())
        if s + l < READ_LEN:
            grow.append(r[s:s + l + 1][::-1].tobytes())
    a, b = g.count_batch(pats)
    assert np.array_equal(np.stack([a, b], 1), np.array(want, np.int64)), "SMEM intervals"
    a, b = g.count_batch(grow)
    assert (a >= b).all(), "an SMEM grown by one symbol occurs"
    return len(pats)


def run_config(w, scale, m, fx, bench):
    import torch
    n = max(100_000, int(bench.DEFAULTS[w][0] * scale))
    t0 = time.time()
    text = np.asarray(bench.make_text(n, w), np.uint8)
    base = bench.index_base(n, w)
    if not (os.path.exists(base + ".bwt") and os.path.exists(base + ".aux")):
        fx.build_index_files(text, base, bigEndian=True)
    prep_s = time.time() - t0
    t0 = time.time()
    g = fx.GpuFMSearcher(base + ".bwt", bigEndian=True, device=0)
    open_plain = time.time() - t0
    info_plain = g.info()
    g.close()
    torch.cuda.empty_cache()
    t0 = time.time()
    g = fx.GpuFMSearcher(base + ".bwt", bigEndian=True, device=0, lcp=1)
    open_lcp = time.time() - t0
    info = g.info()
    N = g.n
    R = make_reads(text, m, 505)
    pat = R.reshape(-1)
    off = np.arange(m + 1, dtype=np.int64) * READ_LEN
    T = m * READ_LEN
    d_pat, d_off = torch.from_numpy(pat).cuda(), torch.from_numpy(off).cuda()
    d_oo = torch.zeros(m + 1, dtype=torch.int64, device="cuda")
    cap = 16 * m
    d_st, d_ln = torch.zeros(cap, dtype=torch.int32, device="cuda"), torch.zeros(cap, dtype=torch.int32, device="cuda")
    d_sp, d_ep = torch.zeros(cap, dtype=torch.int32, device="cuda"), torch.zeros(cap, dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    total = [0]

    def step():
        total[0] = g.smems_dev(d_pat.data_ptr(), d_off.data_ptr(), m, MIN_LEN, d_oo.data_ptr(), d_st.data_ptr(), d_ln.data_ptr(), d_sp.data_ptr(),
                               d_ep.data_ptr(), cap, stream)
    g.set_stats(True)
    step()
    torch.cuda.synchronize()
    req = g.last_match_requests()
    g.set_stats(False)
    k, ms = timed(step)
    oo = d_oo.cpu().numpy()
    nsm = int(oo[m])
    checked = check(g, R, oo, d_st[:nsm].cpu().numpy(), d_ln[:nsm].cpu().numpy(), d_sp[:nsm].cpu().numpy().view(np.uint32),
                    d_ep[:nsm].cpu().numpy().view(np.uint32))
    rps = m * k / (ms / 1e3)
    req_sym = [x / T for x in req]
    gbs, _ = g.gather_bench(64, 4, 1 << 24, 16, 3)
    gather_rps = gbs * 1e9 / 64
    rank_per_step = 1 if info["layout"] == "planes" else info["levels"]
    rec = {"config": w, "n": int(N), "card": card(), "torch_device": torch.cuda.get_device_name(0), "layout": info["layout"],
           "count_lanes_per_query": info["lanes_per_query"], "match_lanes_per_query": 4 if info["layout"] == "wmx" else 2, "reads": m, "read_len": READ_LEN, "substitutions": SUB, "random_reads": RANDOM_FRAC,
           "min_len": MIN_LEN, "smems": nsm, "smems_per_read": nsm / m, "checked_smems": checked,
           "steps": k, "ms_per_step": ms / k, "reads_per_s": rps, "symbols_per_s": rps * READ_LEN,
           "requests_per_symbol": {"rank": req_sym[0], "lcp": req_sym[1], "minima": req_sym[2], "total": sum(req_sym)},
           "model_bound_requests_per_symbol": {"rank": 2 * 2 * rank_per_step, "lcp": "1-2 per widening in the common case", "widenings": 1},
           "requests_per_s": rps * READ_LEN * sum(req_sym), "gather64_requests_per_s": gather_rps,
           "request_rate_vs_gather": rps * READ_LEN * sum(req_sym) / gather_rps,
           "lcp_bytes": info["lcp_bytes"], "lcp_bytes_per_n": info["lcp_bytes"] / N, "index_bytes": info["index_bytes"],
           "index_bytes_without_lcp": info_plain["index_bytes"], "open_s_without_lcp": round(open_plain, 2), "open_s_with_lcp": round(open_lcp, 2),
           "text_and_files_s": round(prep_s, 1)}
    g.close()
    del d_pat, d_off, d_oo, d_st, d_ln, d_sp, d_ep
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg2,cfg5")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of cfg 2's text size (1.0 = bench.py's)")
    ap.add_argument("--dna-scale", type=float, default=0.25, help="fraction of cfg 5's text size")
    ap.add_argument("--reads", type=int, default=1_000_000)
    ap.add_argument("--out", default=None, help="append the JSON lines here")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_match.py measures the GPU; there is no CPU path"
    from findex_b200 import build
    build.build()
    from findex_b200 import fmindex as fx
    import bench
    for w in a.configs.split(","):
        rec = run_config(w, a.dna_scale if w == "cfg5" else a.scale, a.reads, fx, bench)
        line = json.dumps(rec)
        print(line, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()

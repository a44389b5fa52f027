"""
tools/bench_text.py — extract (fmx_text_dev) on the cfg-2, cfg-3 and cfg-5 indexes, against the LF walk on the same index.

    python tools/bench_text.py [--configs cfg2,cfg3,cfg5] [--scale 1.0] [--out profiles/r04_text.json]

The texts and index files are bench.py's (same seeds, same cached files in the temporary directory).  Each index is opened without and
with text samples (text_sample_rate = 32; open times of both are reported), then for len in 16, 64, 256, 4096 the device-resident call is
timed with CUDA events on 10^6 seeded random file offsets (10^5 at 4096): the index as built (row-context hops) and the same handle with
every accelerator hidden by fmx_set_accel_mask (LF steps), alternating the two.  An untimed counting run gives the index requests per
snippet, printed beside the model 1 + ceil((q0 - q + len) / J) (LF: 1 + 2 (q0 - q + len)).  Every snippet of one timed step of each
form is compared with the text.  Writes one JSON line per config to --out (appends) and prints it; the card's name and power limit
are read in the same run.
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

LENS = (16, 64, 256, 4096)
RATE = 32
SEG = 512                               # fmx_kernels.cu kTextSegment


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def model_requests(offs, ln, n, J, lf):
    """per-snippet requests of the model, summed over the segments the kernel cuts a request into"""
    q = (n - 1) - offs.astype(np.int64)
    olen = np.minimum(ln, q)
    tot = np.zeros(len(offs), np.float64)
    for a in range(0, ln, SEG):
        b = np.minimum(a + SEG, olen)
        live = b > a
        hi, lo = q - a, q - b
        x0 = -(-hi // RATE) * RATE
        read = x0 <= n - 1
        x0 = np.minimum(x0, n - 1)
        walk = x0 - lo
        cost = read + (2 * walk - 1 if lf else -(-walk // J))
        tot += np.where(live, cost, 0)
    return float(tot.mean())


def timed(fn, min_s=0.5, warmup=2):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps, ms = 0, 0.0
    while ms < min_s * 1e3:
        k = max(1, steps)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        e1.synchronize()
        ms += e0.elapsed_time(e1)
        steps += k
    return steps, ms


def check(text, offs, ln, d_out, d_len):
    """every snippet of a step against the text"""
    out = d_out.cpu().numpy()
    olen = d_len.cpu().numpy()
    n_file = len(text)
    want_len = np.minimum(ln, n_file - offs)
    assert np.array_equal(olen, want_len), "out_len"
    for a in range(0, len(offs), 1 << 14):
        o = offs[a:a + (1 << 14)]
        idx = np.minimum(o[:, None] + np.arange(ln)[None, :], n_file - 1)
        w = text[idx]
        mask = np.arange(ln)[None, :] < want_len[a:a + len(o), None]
        assert np.array_equal(np.where(mask, out[a:a + len(o)], 0), np.where(mask, w, 0)), "snippets %d.." % a
    return len(offs)


def run_config(w, scale, fx, bench):
    import torch
    n_full = bench.DEFAULTS[w][0]
    n = max(100_000, int(n_full * scale))
    t0 = time.time()
    text = bench.make_text(n, w)
    base = bench.index_base(n, w)
    if not (os.path.exists(base + ".bwt") and os.path.exists(base + ".aux")):
        fx.build_index_files(text, base, bigEndian=True)
    prep_s = time.time() - t0
    extra = {"sa_sample_rate": 32} if w == "cfg3" else {}
    t0 = time.time()
    g = fx.GpuFMSearcher(base + ".bwt", bigEndian=True, device=0, **extra)
    open_plain = time.time() - t0
    info_plain = g.info()
    g.close()
    torch.cuda.empty_cache()
    t0 = time.time()
    g = fx.GpuFMSearcher(base + ".bwt", bigEndian=True, device=0, text_sample_rate=RATE, **extra)
    open_samples = time.time() - t0
    info = g.info()
    N = g.n
    J = info["ctx_depth"]
    text = np.asarray(text, np.uint8)
    rec = {"config": w, "n": int(N), "card": card(), "torch_device": torch.cuda.get_device_name(0), "text_sample_rate": RATE,
           "layout": info["layout"], "ctx_depth": J, "ctx_entry_bytes": info["ctx_entry_bytes"],
           "index_bytes": info["index_bytes"], "index_bytes_without_samples": info_plain["index_bytes"],
           "open_s_without_samples": round(open_plain, 2), "open_s_with_samples": round(open_samples, 2), "text_and_files_s": round(prep_s, 1),
           "lens": {}}
    rng = np.random.default_rng(404)
    for ln in LENS:
        m = 100_000 if ln == 4096 else 1_000_000
        offs = rng.integers(0, N - 1 - ln, m).astype(np.int64)
        d_off = torch.from_numpy(offs.astype(np.uint32).view(np.int32)).cuda()
        d_out = torch.empty((m, ln), dtype=torch.uint8, device="cuda")
        d_len = torch.empty(m, dtype=torch.int32, device="cuda")
        st = torch.cuda.current_stream().cuda_stream

        def step():
            g.text_dev(d_off.data_ptr(), m, ln, d_out.data_ptr(), d_len.data_ptr(), st)
        r = {}
        forms = (("hop", fx.ACCEL_AUTO), ("lf", fx.ACCEL_NONE))
        for name, mask in forms:                             # untimed counting run
            g.set_accel_mask(mask)
            g.set_stats(True)
            step()
            torch.cuda.synchronize()
            r[name] = {"requests_per_snippet": g.last_steps() / m,
                       "model_requests_per_snippet": model_requests(offs, ln, N, J, name == "lf")}
            g.set_stats(False)
        acc = {name: [0, 0.0] for name, _ in forms}
        for _ in range(2):                                   # the two forms alternate
            for name, mask in forms:
                g.set_accel_mask(mask)
                k, ms = timed(step)
                acc[name][0] += k
                acc[name][1] += ms
        for name, mask in forms:                             # every snippet of one timed step
            g.set_accel_mask(mask)
            d_out.zero_()
            step()
            torch.cuda.synchronize()
            r[name]["checked_snippets"] = check(text, offs, ln, d_out, d_len)
            k, ms = acc[name]
            sps = m * k / (ms / 1e3)
            r[name].update({"steps": k, "ms_per_step": ms / k, "snippets_per_s": sps, "output_GB_per_s": sps * ln / 1e9,
                            "requests_per_s": sps * r[name]["requests_per_snippet"]})
            r[name]["requests_vs_model"] = r[name]["requests_per_snippet"] / r[name]["model_requests_per_snippet"]
        r["speedup_hop_over_lf"] = r["hop"]["snippets_per_s"] / r["lf"]["snippets_per_s"]
        rec["lens"][str(ln)] = r
        print(w, ln, json.dumps(r), flush=True)
        del d_off, d_out, d_len
    g.set_accel_mask(fx.ACCEL_AUTO)
    g.close()
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg2,cfg3,cfg5")
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the configs' text sizes (1.0 = bench.py's)")
    ap.add_argument("--out", default=None, help="append the JSON lines here")
    a = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bench_text.py measures the GPU; there is no CPU path"
    from findex_b200 import build
    build.build()
    from findex_b200 import fmindex as fx
    import bench
    for w in a.configs.split(","):
        rec = run_config(w, a.scale, fx, bench)
        line = json.dumps(rec)
        print(line, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()

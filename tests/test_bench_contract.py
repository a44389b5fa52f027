"""bench.py's contract: the reference arm (the CPU restatement of the reference's own search path, oracle/) runs on a tiny workload
and prints ONE JSON line with the agreed keys; our arm refuses to run without a CUDA device instead of falling back to anything; on
a GPU, --dump-outputs writes the rows of the last timed count step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, env=e, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    out = _run(["--impl", "reference", "--text-bytes", "150000", "--queries", "25000", "--steps", "2", "--warmup", "1"])
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"] == "fm_count_queries_per_s_len16_1GB_text" and d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0
    assert d["config"]["workload"].startswith("cfg2") and d["config"]["pattern_len"] == 16
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_other_workloads():
    """--workload cfg3 (count + sorted sa[sp..ep)) and cfg4 (ReTree._matchSA) through the oracle, scaled down"""
    for w, extra, unit in (("cfg3", ["--queries", "3000"], "queries/s"), ("cfg4", ["--queries", "200"], "regexes/s")):
        out = _run(["--impl", "reference", "--workload", w, "--text-bytes", "200000", "--steps", "1", "--warmup", "1"] + extra)
        assert out.returncode == 0, out.stderr[-2000:]
        d = json.loads([ln for ln in out.stdout.splitlines() if ln.strip()][-1])
        assert d["impl"] == "reference" and d["unit"] == unit and d["value"] > 0 and d["config"]["workload"].startswith(w)
        assert d["cpu_baseline"]["kind"] == "port"


def test_bad_arguments_are_refused():
    """--steps is the number of timed steps, so at least one; --dump-outputs only exists for this repo's count path"""
    for args in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"], ["--workload", "cfg3", "--dump-outputs", "d"]):
        out = _run(args)
        assert out.returncode == 2 and "error:" in out.stderr, (args, out.stderr[-2000:])
        assert not out.stdout.strip()


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """a small cfg2 line with --dump-outputs: the sampled (sp, ep) rows are the oracle's answers to the same seeded queries (a miss
    as (0, 0)), the sample stays under 64 MB, and the line reports the timed steps asked for"""
    import bench
    from oracle import fm_oracle as fo
    n, m, steps = 2_000_000, bench.DUMP_MAX_QUERIES + 50_000, 3
    d = tmp_path / "dump"
    out = _run(["--text-bytes", str(n), "--queries", str(m), "--steps", str(steps), "--warmup", "3", "--legs", "", "--no-cpu",
                "--dump-outputs", str(d)])
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    names = sorted(os.listdir(d))
    assert names == ["cfg2_count_ep.npy", "cfg2_count_query.npy", "cfg2_count_sp.npy"]
    assert sum(os.path.getsize(d / f) for f in names) <= 64_000_000
    q, sp, ep = (np.load(d / ("cfg2_count_%s.npy" % k)) for k in ("query", "sp", "ep"))
    assert q.dtype == sp.dtype == ep.dtype == np.float64 and len(q) == len(sp) == len(ep) == bench.DUMP_MAX_QUERIES
    q, sp, ep = q.astype(np.int64), sp.astype(np.int64), ep.astype(np.int64)
    assert q[0] >= 0 and q[-1] < m and (np.diff(q) > 0).all()
    text = bench.make_text(n, "cfg2")
    pats, is_hit = bench.make_queries(text, m, 16, 3, 0)
    o = fo.OracleIndex.from_text_rev(fo.file_to_text_rev(text.tobytes()))
    osp, oep = o.count_batch(pats[q].reshape(-1), np.arange(0, len(q) * 16 + 1, 16, dtype=np.int64), threads=os.cpu_count())
    o.close()
    assert (ep > sp)[is_hit[q]].all() and (ep > sp).sum() < len(q)
    assert np.array_equal(sp, osp) and np.array_equal(ep, oep)


@pytest.mark.gpu
@pytest.mark.parametrize("workload,queries,steps,warmup", [("cfg3", 60_000, 3, 2), ("cfg4", 200, 2, 0)])
def test_workload_lines_time_the_steps_asked_for(workload, queries, steps, warmup):
    """--steps and --warmup of a --workload cfg3 / cfg4 line are the counts its headline leg times, and the line reports them"""
    out = _run(["--workload", workload, "--text-bytes", "2000000", "--queries", str(queries), "--steps", str(steps), "--warmup", str(warmup),
                "--no-cpu"])
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    leg = d["locate" if workload == "cfg3" else "regex"]
    assert (d["steps"], d["warmup"]) == (steps, warmup) and (leg["steps"], leg["warmup"]) == (steps, warmup)
    assert d["value"] > 0


def test_our_arm_needs_a_gpu_and_says_so():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    out = _run(["--text-bytes", "150000", "--queries", "25000", "--steps", "1", "--warmup", "3", "--no-cpu", "--regexes", "0"])
    assert out.returncode != 0
    assert "needs a CUDA device" in (out.stderr + out.stdout)
    assert not [ln for ln in out.stdout.splitlines() if ln.strip().startswith("{")]       # no number without the device

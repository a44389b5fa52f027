"""
k-mer group blocks on the GPU (fmx_kmer_rows; DESIGN.md §3): under FMX_ACCEL_AUTO an index with 32-byte row contexts, a saturating k-mer
table and no dictionary stores its table as 64-byte group blocks that carry the row contexts' J-hop of their first rows.  Every count entry
point must give what the oracle and the same index with the plain table (FMX_KMER_ROWS=0) give, for every pattern length, with byte 0,
absent bytes and intervals larger than the inline rows, at 1, 2 and 4 lanes per query, with the accelerators partly hidden.
"""
import numpy as np
import pytest

from findex_b200 import fmindex as fx
from oracle import fm_oracle as fo

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU; the product has no CPU path"
    from findex_b200 import build
    build.build()


def _text(sigma, n, seed):
    """uniform symbols; sizes where the AUTO table (at most 8n entries) is saturating (sigma^k >= n/2): groups of a few rows"""
    rng = np.random.default_rng(seed)
    alpha = np.arange(1, 256, dtype=np.uint8) if sigma == 255 else np.sort(rng.choice(np.arange(2, 255), sigma, replace=False)).astype(np.uint8)
    tp = alpha[rng.integers(0, sigma, n)].tobytes()
    return tp, alpha


def _open(bwt, eof, cnt, monkeypatch, rows_env=None, **kw):
    if rows_env is None:
        monkeypatch.delenv("FMX_KMER_ROWS", raising=False)
    else:
        monkeypatch.setenv("FMX_KMER_ROWS", rows_env)
    return fx.GpuFMSearcher(bwt=bwt, eof=eof, counts=cnt, **kw)


def _batch(tp, alpha, rng, ln, m):
    offs = rng.integers(0, len(tp) - ln, m)
    arr = np.stack([np.frombuffer(tp[s:s + ln], np.uint8) for s in offs]).copy()
    arr[1::7, int(rng.integers(0, ln))] = alpha[rng.integers(0, len(alpha))]              # near misses
    arr[2::11] = alpha[rng.integers(0, len(alpha), (len(arr[2::11]), ln))]                  # random patterns
    arr[3::13, int(rng.integers(0, ln))] = 0                                                 # byte 0 ('$' wraps the text)
    if len(alpha) < 255:
        arr[4::17, int(rng.integers(0, ln))] = 1                                             # a byte the text does not hold
    return arr


def _oracle(o, arr):
    ln = arr.shape[1]
    return o.count_batch(arr.reshape(-1), np.arange(0, arr.size + 1, ln, dtype=np.int64))


@pytest.mark.parametrize("sigma,n", [(255, 100000), (28, 40000), (4, 50000)])
@pytest.mark.parametrize("layout", [fx.LAYOUT_PLANES, fx.LAYOUT_WM])
def test_group_form_every_length_and_lanes(sigma, n, layout, monkeypatch):
    tp, alpha = _text(sigma, n, 5 + sigma)
    bwt, eof, cnt = fo.build_bwt(tp)
    o = fo.OracleIndex.from_bwt(bwt, eof, cnt)
    plain = _open(bwt, eof, cnt, monkeypatch, "0", layout=layout)
    assert plain.info()["kmer_rows"] == 0
    rng = np.random.default_rng(sigma)
    batches = {ln: _batch(tp, alpha, rng, ln, 300) for ln in range(1, 65)}
    want = {}
    for ln, arr in batches.items():
        want[ln] = _oracle(o, arr)
        sp, ep = plain.count_fixed(arr)
        assert np.array_equal(sp, want[ln][0]) and np.array_equal(ep, want[ln][1]), ln
    plain.close()
    for lanes in (0, 1, 2, 4):
        g = _open(bwt, eof, cnt, monkeypatch, None, layout=layout, lanes_per_query=lanes)
        info = g.info()
        assert info["kmer_rows"] == 3 and info["ctx_entry_bytes"] == 32 and info["dict_depth"] == 0, info
        wide = 0
        for ln, arr in batches.items():
            sp, ep = g.count_fixed(arr)
            assert np.array_equal(sp, want[ln][0]) and np.array_equal(ep, want[ln][1]), (lanes, ln)
            if ln == info["kmer_k"]:
                wide += int(((ep - sp) > 3).sum())           # intervals larger than the inline rows
            assert np.array_equal(g.count_only_fixed(arr).astype(np.int64), want[ln][1] - want[ln][0])
        assert wide > 0 or sigma == 4                        # (DNA: the depth-9 table leaves intervals of 1-2 rows)
        # variable-length batches (count_var) and patterns too long for shared memory (count_fixed_gmem)
        pats = [bytes(batches[ln][i]) for ln in range(1, 65) for i in range(0, 300, 37)]
        sp, ep = g.count_batch(pats)
        for i, p in enumerate(pats):
            r = o.search(p)
            assert (int(sp[i]), int(ep[i])) == (r if r else (0, 0)), p
        long = _batch(tp, alpha, rng, 700, 64)
        osp, oep = _oracle(o, long)
        sp, ep = g.count_fixed(long)
        assert np.array_equal(sp, osp) and np.array_equal(ep, oep)
        g.close()
    o.close()


def test_group_form_with_accelerators_hidden(monkeypatch):
    """KMER alone: the blocks act as a plain table (no inline rows without the row contexts); KMER | CTX: the full path"""
    tp, alpha = _text(255, 100000, 9)
    bwt, eof, cnt = fo.build_bwt(tp)
    o = fo.OracleIndex.from_bwt(bwt, eof, cnt)
    g = _open(bwt, eof, cnt, monkeypatch)
    assert g.info()["kmer_rows"] == 3
    rng = np.random.default_rng(1)
    for mask in (fx.ACCEL_KMER, fx.ACCEL_KMER | fx.ACCEL_CTX, fx.ACCEL_CTX, fx.ACCEL_NONE, fx.ACCEL_AUTO):
        g.set_accel_mask(mask)
        assert g.info()["kmer_rows"] == (3 if mask & fx.ACCEL_KMER or mask == fx.ACCEL_AUTO else 0)
        for ln in (2, 3, 8, 14, 16, 20, 33):
            arr = _batch(tp, alpha, rng, ln, 500)
            osp, oep = _oracle(o, arr)
            sp, ep = g.count_fixed(arr)
            assert np.array_equal(sp, osp) and np.array_equal(ep, oep), (mask, ln)
    g.close()
    o.close()


def test_group_form_fused_exchange_single_gpu(monkeypatch):
    """the fused count + all-gather entry point over the group form, this GPU playing three ranks"""
    import torch
    tp, alpha = _text(255, 100000, 3)
    bwt, eof, cnt = fo.build_bwt(tp)
    o = fo.OracleIndex.from_bwt(bwt, eof, cnt)
    g = _open(bwt, eof, cnt, monkeypatch)
    assert g.info()["kmer_rows"] == 3
    pats = _batch(tp, alpha, np.random.default_rng(2), 16, 3003)
    m, ln, world = len(pats), 16, 3
    osp, oep = _oracle(o, pats)
    bufs = [fx.SharedDeviceBuffer(m) for _ in range(world)]
    d_pat = torch.from_numpy(pats).cuda()
    d_sp = torch.zeros(m, dtype=torch.int32, device="cuda")
    d_ep = torch.zeros(m, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    per = m // world
    for r in range(world):
        lo, hi = r * per, (r + 1) * per
        g.count_fixed_dev_gather(d_pat.data_ptr() + lo * ln, ln, hi - lo, d_sp.data_ptr() + lo * 4, d_ep.data_ptr() + lo * 4,
                                 [b.ptr for b in bufs], lo, st)
    torch.cuda.synchronize()
    assert np.array_equal(d_sp.cpu().numpy(), osp) and np.array_equal(d_ep.cpu().numpy(), oep)
    for b in bufs:
        assert np.array_equal(b.to_host().astype(np.int64), oep - osp)
        b.close()
    g.close()
    o.close()

"""The extreme-score scan over window plans (pgt_scan_plan_extreme) without a GPU: the entry points fail loudly, the Python
dispatch keeps the ExtremePlan signatures, and the numpy restatement of the row contract the GPU tests use (`xref`)
equals the oracle of ihsWindow / xpehhWindow on windows built to coincide with its own."""
import ctypes as C
import inspect

import numpy as np
import pytest

import oracle_lib as O

IHS, XPEHH = 0, 1
# the NaN of an empty row (CUDART_NAN, as pgt_scan_extreme writes it)
EMPTY_NAN = np.frombuffer(np.uint64(0xFFF8000000000000).tobytes(), np.float64)[0]


def xkey(stat, cutoff, score):
    """The key of every site: IHS |v|, XPEHH v (cutoff >= 0) or -v; a NaN key is -inf."""
    k = np.abs(score) if stat == IHS else (score if cutoff >= 0 else -score)
    return np.where(np.isnan(k), -np.inf, k)


def xbig(stat, cutoff, score):
    with np.errstate(invalid="ignore"):
        if stat == IHS:
            return np.abs(score) > cutoff
        return score > cutoff if cutoff >= 0 else score < cutoff


def _rmq_first_max(key, lo, hi):
    """For every window [lo, hi) (non-empty): the smallest index of the largest key, by a sparse table over the
    ranks of (key, -index) (largest key first, then smallest index)."""
    n = len(key)
    order = np.lexsort((-np.arange(n), key))  # ascending: key, then larger index first
    rank = np.empty(n, np.int64)
    rank[order] = np.arange(n)
    table = [rank]
    while (1 << len(table)) <= n:
        prev, h = table[-1], 1 << (len(table) - 1)
        table.append(np.maximum(prev[:-h], prev[h:]))
    length = hi - lo
    k = np.floor(np.log2(np.maximum(length, 1))).astype(np.int64)
    best = np.empty(len(lo), np.int64)
    for lev in np.unique(k):
        m = k == lev
        t = table[lev]
        best[m] = np.maximum(t[lo[m]], t[hi[m] - (1 << lev)])
    return order[best]


def xref(stat, cutoff, score, pos, lo, hi):
    """The rows of pgt_scan_plan_extreme for windows reducing sites [lo, hi) (global indices into score / pos)."""
    score = np.asarray(score, np.float64)
    lo, hi = np.asarray(lo, np.int64), np.asarray(hi, np.int64)
    n = (hi - lo).astype(np.uint32)
    cb = np.concatenate([[0], np.cumsum(xbig(stat, cutoff, score), dtype=np.int64)])
    nbig = (cb[hi] - cb[lo]).astype(np.uint32)
    full = n > 0
    site = np.full(len(lo), np.iinfo(np.uint64).max, np.uint64)
    if full.any():
        site[full] = _rmq_first_max(xkey(stat, cutoff, score), lo[full], hi[full])
    val = np.full(len(lo), EMPTY_NAN)
    val[full] = score[site[full].astype(np.int64)]
    out = dict(ext_value=val, ext_site=site, nbig=nbig, nsites=n, prop=np.full(len(lo), EMPTY_NAN))
    out["prop"][full] = nbig[full].astype(np.float64) / n[full].astype(np.float64)
    if pos is not None:
        out["ext_pos"] = np.zeros(len(lo), np.uint32)
        out["ext_pos"][full] = np.asarray(pos)[site[full].astype(np.int64)]
    return out


def coincident_layout(pos, contig_offsets, winsize, pgt):
    """Sites of the non-empty windows of an ExtremePlan, in order, and the site-mode plan whose windows are exactly
    those windows: contig_offsets = their boundaries, W = S = the longest + 1.  Returns (index of every plan site in
    the original columns, xplan window table, its non-empty rows, plan)."""
    xplan = pgt.ExtremePlan(pos, contig_offsets, winsize)
    xw = xplan.windows()
    keep = np.nonzero(xw["nsites"] > 0)[0]
    idx = np.concatenate([np.arange(int(xw["first_site"][w]), int(xw["first_site"][w]) + int(xw["nsites"][w])) for w in keep])
    offs = np.concatenate([[0], np.cumsum(xw["nsites"][keep], dtype=np.uint64)]).astype(np.uint64)
    W = int(xw["nsites"].max()) + 1
    return idx, xw, keep, pgt.WindowPlan(offs, W, W), xplan


def synth_positions(rng, lengths, gap):
    pos = []
    for L in lengths:
        pos.append(np.cumsum(rng.integers(1, gap, L)).astype(np.uint32))
    return np.concatenate(pos), np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)


@pytest.fixture(scope="module")
def pgt():
    import popgenomicstools_b200 as m
    return m


def test_entry_points_fail_loudly_without_device(pgt):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from popgenomicstools_b200 import _cabi
    lib = _cabi.load()
    off = np.array([0, 100], np.uint64)
    h = C.c_void_p()
    assert lib.pgt_plan_create(C.byref(h), 0, off.ctypes.data, 1, 10, 5, 0) == 0
    score = np.zeros(100)
    pos = np.arange(1, 101, dtype=np.uint32)
    val = np.zeros(19)
    xo = _cabi.PgtXWindows()
    xo.ext_value = val.ctypes.data
    nb = lib.pgt_scan_plan_extreme_workspace_bytes(h, None, _cabi.PGT_MEM_HOST)
    assert nb > 0
    ws = np.zeros(nb, np.uint8)
    assert lib.pgt_scan_plan_extreme(h, None, IHS, 2.0, pos.ctypes.data, score.ctypes.data, None, None, C.byref(xo), ws.ctypes.data,
                                     ws.nbytes, _cabi.PGT_MEM_HOST, None) == _cabi.PGT_ERR_CUDA
    assert b"no CPU fallback" in lib.pgt_last_error()
    dev = (C.c_int * 2)(0, 0)
    assert lib.pgt_scan_plan_extreme_sharded(h, XPEHH, -2.0, pos.ctypes.data, score.ctypes.data, None, None, C.byref(xo), dev,
                                             2) == _cabi.PGT_ERR_CUDA
    # the argument checks come first
    assert lib.pgt_scan_plan_extreme(h, None, 7, 2.0, pos.ctypes.data, score.ctypes.data, None, None, C.byref(xo), ws.ctypes.data,
                                     ws.nbytes, _cabi.PGT_MEM_HOST, None) == _cabi.PGT_ERR_ARGS
    assert lib.pgt_scan_plan_extreme(h, None, IHS, 2.0, pos.ctypes.data, None, None, None, C.byref(xo), ws.ctypes.data,
                                     ws.nbytes, _cabi.PGT_MEM_HOST, None) == _cabi.PGT_ERR_ARGS
    # pgt_scan and its workspace query know nothing of the new statistic
    assert lib.pgt_scan_workspace_bytes(h, None, 16, _cabi.PGT_MEM_HOST) == 0
    assert lib.pgt_plan_scan_path(h, 16) == _cabi.PGT_ERR_ARGS
    lib.pgt_plan_destroy(h)


def test_python_dispatch_keeps_extreme_plan_signatures(pgt):
    from popgenomicstools_b200 import extreme
    head = ["plan", "stat", "cutoff", "pos", "score", "window_range", "site_origin", "out", "device"]
    assert list(inspect.signature(extreme.scan_extreme).parameters)[:len(head)] == head
    assert list(inspect.signature(extreme.scan_extreme_sharded).parameters)[:6] == ["plan", "stat", "cutoff", "pos", "score", "devices"]
    assert list(inspect.signature(extreme.ihs_window).parameters)[:4] == ["plan", "pos", "score", "cutoff"]
    assert list(inspect.signature(extreme.xpehh_window).parameters)[:4] == ["plan", "pos", "score", "cutoff"]
    xplan = pgt.ExtremePlan(np.arange(1, 11, dtype=np.uint32), np.array([0, 10], np.uint64), 5)
    with pytest.raises(ValueError, match="WindowPlan"):
        pgt.scan_extreme(xplan, IHS, 2.0, None, np.zeros(10), site_offsets=np.array([0, 10], np.uint64))
    bp = pgt.WindowPlan(np.array([0, 1000], np.uint64), 100, 10, mode="bp")
    with pytest.raises(ValueError, match="site_offsets"):
        pgt.ihs_window(bp, np.arange(1, 11, dtype=np.uint32), np.zeros(10))


@pytest.mark.parametrize("stat,cutoff", [(IHS, 2.0), (XPEHH, 2.0), (XPEHH, -2.0)])
@pytest.mark.parametrize("seed", [1, 2])
def test_restatement_equals_oracle_on_coincident_windows(pgt, stat, cutoff, seed):
    rng = np.random.default_rng(seed)
    pos, offs = synth_positions(rng, [4000, 700, 2500, 50], 40)
    score = rng.standard_normal(len(pos)) * 1.5
    score[rng.random(len(pos)) < 0.05] = 2.0  # ties, and values exactly at the cutoff
    score[rng.random(len(pos)) < 0.05] = -2.0
    idx, xw, keep, plan, _ = coincident_layout(pos, offs, 10000, pgt)
    first, last, label = plan.windows()
    assert plan.num_windows == len(keep)
    assert np.array_equal(last - first + 1, xw["nsites"][keep].astype(np.uint64))
    ref = xref(stat, cutoff, score[idx], pos[idx], first.astype(np.int64), last.astype(np.int64) + 1)
    chr_id = np.repeat(np.arange(len(offs) - 1, dtype=np.uint32), np.diff(offs).astype(np.int64))
    orc = O.extreme("ihs" if stat == IHS else "xpehh", chr_id, pos, score, 10000, cutoff)
    assert len(orc["n"]) == len(xw["nsites"])
    for mine, theirs in (("ext_value", "ext"), ("ext_pos", "extpos"), ("nbig", "nbig"), ("nsites", "n"), ("prop", "prop")):
        assert ref[mine].tobytes() == orc[theirs][keep].tobytes(), mine


def test_restatement_edge_cases():
    score = np.array([np.nan, np.nan, -0.0, 0.0, 3.0, -3.0, np.inf, -np.inf, 1e308, -1e308])
    lo, hi = np.array([0, 2, 4, 6, 8, 3]), np.array([2, 4, 6, 8, 10, 3])
    r = xref(IHS, 2.0, score, None, lo, hi)
    assert list(r["ext_site"][:5]) == [0, 2, 4, 6, 8]  # all-NaN window: the first site; ties: the smaller index
    assert r["ext_site"][5] == np.iinfo(np.uint64).max and r["nsites"][5] == 0
    assert r["ext_value"][5].tobytes() == EMPTY_NAN.tobytes() and r["prop"][5].tobytes() == EMPTY_NAN.tobytes()
    assert list(r["nbig"][:5]) == [0, 0, 2, 2, 2]
    x = xref(XPEHH, -2.0, score, None, lo[:5], hi[:5])
    assert list(x["ext_site"]) == [0, 2, 5, 7, 9] and list(x["nbig"]) == [0, 0, 1, 1, 1]

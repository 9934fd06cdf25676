"""pgt_scan_plan_extreme on the GPU: every row, field by field and bit for bit, equals the numpy restatement of the
contract (test_plan_extreme_cpu.xref) -- on every kernel path, statistic, memory space and shard cut; the geometry equals
pgt_scan's fst rows; on windows built to coincide with ihsWindow's it equals pgt_scan_extreme."""
import ctypes as C

import numpy as np
import pytest

from test_plan_extreme_cpu import IHS, XPEHH, coincident_layout, synth_positions, xkey, xref

pytestmark = pytest.mark.gpu

STATS = [(IHS, 2.0), (XPEHH, 2.0), (XPEHH, -2.0)]
FIELDS = ("ext_value", "ext_pos", "ext_site", "nbig", "nsites", "prop")
KNOBS = [None, ("level1", 1), ("level1", 2), ("level2", 1), ("level2", 2), ("unittable", 1), ("unittable", 2), ("persite", 1)]


@pytest.fixture(scope="module")
def pgt():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import popgenomicstools_b200 as m
    return m


def to_dev(x, shift=0):
    """A CUDA copy of x; shift > 0: a view `shift` elements into a larger buffer (column pointer off its alignment)."""
    import torch
    x = np.ascontiguousarray(x)
    t = torch.from_numpy(x.view(np.int32) if x.dtype == np.uint32 else x)
    buf = torch.empty(len(x) + shift, dtype=t.dtype, device="cuda")
    buf[shift:] = t.cuda()
    v = buf[shift:]
    return v.view(torch.uint32) if x.dtype == np.uint32 else v


def npy(out):
    import torch
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items()}


def assert_rows(got, ref, what):
    for k in FIELDS:
        if k in ref:
            assert got[k].tobytes() == ref[k].tobytes(), f"{what}: {k} first bad at {np.nonzero(got[k] != ref[k])[0][:5]}"


def adversarial(rng, n, cutoff):
    pool = np.array([-3.0, -2.0, -1.0, -0.0, 0.0, 1.0, 2.0, 3.0, np.nan, np.inf, -np.inf, 1e308, -1e308, cutoff, -cutoff])
    s = pool[rng.integers(0, len(pool), n)]
    s[n // 3:n // 3 + 400] = np.nan  # windows of NaN only
    return s


def scores(pgt, kind, seed, n, cutoff):
    if kind == "synth":
        return pgt.synth_score(seed, 0, n).cpu().numpy()
    return adversarial(np.random.default_rng(seed), n, cutoff)


def site_windows(plan):
    first, last, _ = plan.windows()
    return first.astype(np.int64), last.astype(np.int64) + 1


def bp_windows(plan, pos, soff, boff):
    first, last, _ = plan.windows()
    chrom = np.repeat(np.arange(len(soff) - 1), np.diff(soff).astype(np.int64))
    e = boff[chrom].astype(np.int64) + pos.astype(np.int64) - 1
    return np.searchsorted(e, first.astype(np.int64), "left"), np.searchsorted(e, last.astype(np.int64), "right")


def fst_geometry(pgt, plan, pos, soff):
    n = len(pos)
    f = pgt.fst_window(plan, pos, np.zeros(n), np.ones(n), site_offsets=soff)
    return {k: f[k] for k in ("label", "start_pos", "end_pos", "mid_pos")}


def with_knob(pgt, knob, fn):
    if knob:
        pgt.tune(*knob)
    try:
        return fn()
    finally:
        if knob:
            pgt.tune(knob[0], 0)


# site layouts: contig lengths (the first a multiple of 100 and 10: the cross-contig carry; a tail not filling a window:
# the EOF drop), more than 32 contigs, chromosomes no longer than W - S (stale carry)
SITE_LAYOUTS = {
    "carry": [25000, 9000, 3100],
    "many": list(np.random.default_rng(3).integers(200, 3000, 40)),
    "short": [6000, 30, 4000, 7, 2500, 20],
}
GEOMS = [(50, 10), (1000, 100), (1000, 1), (37, 37), (1, 1)]


@pytest.mark.parametrize("layout", list(SITE_LAYOUTS))
@pytest.mark.parametrize("W,S", GEOMS)
def test_site_plans_every_path(pgt, layout, W, S):
    lens = SITE_LAYOUTS[layout]
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    n = int(offs[-1])
    pos = np.concatenate([np.cumsum(np.random.default_rng(L).integers(1, 30, L)) for L in lens]).astype(np.uint32)
    plan = pgt.WindowPlan(offs, W, S)
    lo, hi = site_windows(plan)
    geo = fst_geometry(pgt, plan, pos, None)
    shift = 1 if layout == "many" else 0  # unaligned column views
    for kind in ("synth", "adversarial"):
        for stat, cutoff in STATS:
            score = scores(pgt, kind, 11, n, cutoff)
            ref = xref(stat, cutoff, score, pos, lo, hi)
            dpos, dscore = to_dev(pos, shift), to_dev(score, shift)
            for knob in KNOBS:
                got = npy(with_knob(pgt, knob, lambda: pgt.scan_extreme(plan, stat, cutoff, dpos, dscore)))
                assert_rows(got, ref, f"{layout} {W}/{S} {kind} {stat} {cutoff} {knob}")
                for k in geo:
                    assert got[k].tobytes() == geo[k].tobytes(), (k, knob)
            host = pgt.scan_extreme(plan, stat, cutoff, pos, score)
            assert_rows(host, ref, f"host {layout} {W}/{S} {kind}")


def bp_input(seed, chr_len, density, empty_chrom=None, dense_run=None):
    """Sorted positions per chromosome: every bp (density 1) or about one per `density` bp; chromosome `empty_chrom`
    without sites; `dense_run` = (lo, hi): every bp of chromosome 0 in [lo, hi] a site."""
    rng = np.random.default_rng(seed)
    pos, nsites = [], []
    for c, L in enumerate(chr_len):
        if c == empty_chrom:
            p = np.zeros(0, np.uint32)
        elif density == 1:
            p = np.arange(1, L + 1, dtype=np.uint32)
        else:
            p = np.sort(rng.choice(L, size=max(1, L // density), replace=False)).astype(np.uint32) + 1
        if c == 0 and dense_run is not None:
            p = np.union1d(p, np.arange(dense_run[0], dense_run[1] + 1, dtype=np.uint32)).astype(np.uint32)
        pos.append(p)
        nsites.append(len(p))
    return np.concatenate(pos), np.concatenate([[0], np.cumsum(nsites)]).astype(np.uint64)


# (chromosome lengths, bp per site, W, S, dense run of chromosome 0).  The dense run inside sparse data: the tiled level-1
# kernel sizes its tiles for the average density, so the tiles over the run do not fit a stage and are read from global
# memory (level1=2 below).
BP_CASES = {
    "sparse_with_dense_run": ([9_000_000, 250_000, 31_000, 400_000], 30, 100_000, 10_000, (2_000_000, 2_600_000)),
    "dense_1000_100": ([120_000, 3_000, 57_000, 800], 1, 1000, 100),
    "sparse_1000_100": ([900_000, 25_000, 31_000, 400_000, 20_000], 30, 1000, 100),
    "dense_100k_10k": ([1_300_000, 250_000, 3_000, 570_000, 80_000], 1, 100_000, 10_000),
    "sparse_100k_10k": ([9_000_000, 250_000, 31_000, 4_000_000, 20_000], 30, 100_000, 10_000),
}


@pytest.mark.parametrize("case", list(BP_CASES))
def test_bp_plans_every_path(pgt, case):
    lens, density, W, S, *run = BP_CASES[case]
    pos, soff = bp_input(5, lens, density, empty_chrom=1, dense_run=run[0] if run else None)  # a chromosome without score sites (longer than W - S: rows of its own
    # with nsites 0 and NaN)
    boff = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    plan = pgt.WindowPlan(boff, W, S, mode="bp")
    lo, hi = bp_windows(plan, pos, soff, boff)
    assert np.any(hi == lo)
    geo = fst_geometry(pgt, plan, pos, soff)
    nsites_bp = pgt.bp_window_sites(plan, pos, soff)
    n = len(pos)
    dpos = to_dev(pos)
    for kind in ("synth", "adversarial"):
        for stat, cutoff in STATS:
            score = scores(pgt, kind, 12, n, cutoff)
            ref = xref(stat, cutoff, score, pos, lo, hi)
            assert np.array_equal(ref["nsites"], nsites_bp)
            dscore = to_dev(score)
            for knob in KNOBS:
                got = npy(with_knob(pgt, knob, lambda: pgt.scan_extreme(plan, stat, cutoff, dpos, dscore, site_offsets=soff)))
                assert_rows(got, ref, f"{case} {kind} {stat} {cutoff} {knob}")
                for k in geo:
                    assert got[k].tobytes() == geo[k].tobytes(), (k, knob)
            host = pgt.scan_extreme(plan, stat, cutoff, pos, score, site_offsets=soff)
            assert_rows(host, ref, f"host {case} {kind}")


@pytest.mark.parametrize("mode", ["sites", "bp"])
@pytest.mark.parametrize("W,S", [(1000, 100), (1, 1)])
def test_device_host_shards_and_sharded_agree(pgt, mode, W, S):
    import torch
    if mode == "bp" and W == 1:
        pytest.skip("W = S = 1 is a site-mode path")
    if mode == "sites":
        lens = [25000, 9000, 3100, 50, 7000]
        soff = None
        offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        pos = np.concatenate([np.arange(1, L + 1) for L in lens]).astype(np.uint32)
        plan, plan2 = pgt.WindowPlan(offs, W, S), pgt.WindowPlan(offs, W, S)
        lo, hi = site_windows(plan)
    else:
        lens = [300_000, 5_000, 120_000, 900]
        pos, soff = bp_input(9, lens, 7, empty_chrom=1)
        boff = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
        plan, plan2 = pgt.WindowPlan(boff, W, S, mode="bp"), pgt.WindowPlan(boff, W, S, mode="bp")
        lo, hi = bp_windows(plan, pos, soff, boff)
    score = adversarial(np.random.default_rng(4), len(pos), 2.0)
    for stat, cutoff in STATS:
        ref = xref(stat, cutoff, score, pos, lo, hi)
        dev = npy(pgt.scan_extreme(plan, stat, cutoff, to_dev(pos), to_dev(score), site_offsets=soff))
        host = pgt.scan_extreme(plan, stat, cutoff, pos, score, site_offsets=soff)
        pieces = []
        for i in range(5):
            w_lo, w_hi, _, _ = plan.shard(i, 5)
            if w_hi == w_lo:
                continue
            o = int(lo[w_lo])  # the window range's first site (bp: a data site index)
            pieces.append(pgt.scan_extreme(plan, stat, cutoff, pos[o:], score[o:], window_range=(w_lo, w_hi), site_origin=o,
                                           site_offsets=soff))
        cut = {k: np.concatenate([p[k] for p in pieces]) for k in pieces[0]}
        lists = [[0], [0, 0, 0]] + ([list(range(torch.cuda.device_count()))] if torch.cuda.device_count() > 1 else [])
        for res, what in [(dev, "device"), (host, "host"), (cut, "shards")] + [
                (pgt.scan_extreme_sharded(plan2, stat, cutoff, pos, score, d, site_offsets=soff), f"sharded {d}") for d in lists]:
            assert_rows(res, ref, f"{mode} {W}/{S} {stat} {cutoff} {what}")
            for k in ("label", "start_pos", "end_pos", "mid_pos"):
                assert res[k].tobytes() == host[k].tobytes(), (what, k)


def _c_rows(pgt, plan, pos, score, soff):
    """pgt_scan_plan_extreme with the geometry's nsites (which the Python rows leave out): (nsites, return code)."""
    from popgenomicstools_b200 import _cabi
    lib = _cabi.load()
    nw = plan.num_windows
    geo_n, val = np.zeros(nw, np.uint32), np.zeros(nw)
    rows, out = _cabi.PgtWindows(), _cabi.PgtXWindows()
    rows.nsites = geo_n.ctypes.data
    out.ext_value = val.ctypes.data
    nb = plan.extreme_workspace_bytes(_cabi.PGT_MEM_HOST)
    import torch
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    so = None if soff is None else np.ascontiguousarray(soff, np.uint64)
    rc = lib.pgt_scan_plan_extreme(plan.handle, None, IHS, 2.0, pos.ctypes.data, score.ctypes.data, so.ctypes.data if so is not None else None,
                                   C.byref(rows), C.byref(out), ws.data_ptr(), nb, _cabi.PGT_MEM_HOST, None)
    return geo_n, rc


def test_geometry_nsites_equals_fst(pgt):
    lens = [120_000, 3_000, 57_000, 800]
    pos, soff = bp_input(5, lens, 3)
    boff = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    for plan, so in ((pgt.WindowPlan(boff, 10_000, 1_000, mode="bp"), soff), (pgt.WindowPlan(soff, 50, 10), None)):
        score = np.zeros(len(pos))
        geo_n, rc = _c_rows(pgt, plan, pos, score, so)
        assert rc == 0
        f = pgt.fst_window(plan, pos, score, score, site_offsets=so)
        assert geo_n.tobytes() == f["nsites"].tobytes()


def test_coincident_windows_equal_scan_extreme(pgt):
    rng = np.random.default_rng(21)
    pos, offs = synth_positions(rng, [40000, 7000, 25000, 500, 30000], 40)
    score = pgt.synth_score(8, 0, len(pos)).cpu().numpy()
    score[rng.random(len(pos)) < 0.02] = 2.0
    idx, xw, keep, plan, xplan = coincident_layout(pos, offs, 100_000, pgt)
    for stat, cutoff in STATS:
        old = npy(pgt.scan_extreme(xplan, stat, cutoff, to_dev(pos), to_dev(score)))
        new = npy(pgt.scan_extreme(plan, stat, cutoff, to_dev(pos[idx]), to_dev(score[idx])))
        for k in FIELDS:
            want = old[k][keep]
            got = idx[new[k].astype(np.int64)].astype(np.uint64) if k == "ext_site" else new[k]
            assert got.tobytes() == want.tobytes(), k


def test_scale_1e8_sites(pgt):
    import torch
    from popgenomicstools_b200.workloads import human_like_contigs
    n, W, S = 100_000_000, 50_000, 10_000
    _, offs = human_like_contigs(n, S)
    plan = pgt.WindowPlan(offs, W, S)
    score_d = pgt.synth_score(31, 0, n)
    pos_d = pgt.synth_pos(31, 0, n, offs, 3)
    out = npy(pgt.ihs_window(plan, pos_d, score_d, 2.0))
    score = score_d.cpu().numpy()
    pos = pos_d.cpu().numpy()
    del score_d, pos_d
    torch.cuda.empty_cache()
    lo, hi = site_windows(plan)
    cb = np.concatenate([[0], np.cumsum(np.abs(score) > 2.0, dtype=np.int64)])
    assert np.array_equal(out["nbig"], (cb[hi] - cb[lo]).astype(np.uint32))
    assert np.array_equal(out["nsites"], (hi - lo).astype(np.uint32))
    key = xkey(IHS, 2.0, score)
    site = np.array([a + int(np.argmax(key[a:b])) for a, b in zip(lo, hi)], np.uint64)  # blockwise: one window at a time
    assert np.array_equal(out["ext_site"], site)
    assert out["ext_value"].tobytes() == score[site.astype(np.int64)].tobytes()
    assert np.array_equal(out["ext_pos"], pos[site.astype(np.int64)])


def test_errors(pgt):
    from popgenomicstools_b200 import _cabi
    lib = _cabi.load()
    lens = [10_000, 5_000]
    pos, soff = bp_input(2, lens, 5)
    boff = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    bp = pgt.WindowPlan(boff, 1000, 100, mode="bp")
    sites = pgt.WindowPlan(soff, 50, 10)
    score = np.zeros(len(pos))
    code = lambda f: pytest.raises(_cabi.PgtError, f).value.code  # noqa: E731
    assert code(lambda: pgt.scan_extreme(sites, 5, 2.0, pos, score)) == _cabi.PGT_ERR_ARGS
    assert code(lambda: pgt.scan_extreme(sites, IHS, 2.0, pos, score, window_range=(0, sites.num_windows + 1))) == _cabi.PGT_ERR_ARGS
    bad = pos.copy()
    bad[int(soff[1]) - 1] = lens[0] + 1  # beyond its chromosome
    assert code(lambda: pgt.scan_extreme_sharded(bp, IHS, 2.0, bad, score, [0], site_offsets=soff)) == _cabi.PGT_ERR_INPUT
    assert code(lambda: pgt.scan_extreme(bp, IHS, 2.0, bad, score, site_offsets=soff)) == _cabi.PGT_ERR_INPUT
    assert code(lambda: pgt.scan_extreme(bp, IHS, 2.0, to_dev(bad), to_dev(score), site_offsets=soff)) == _cabi.PGT_ERR_INPUT
    # NULL score, pos missing where it is required, rows asking for a non-geometry field, workspace too small
    nw = sites.num_windows
    val, fst = np.zeros(nw), np.zeros(nw)
    out, rows = _cabi.PgtXWindows(), _cabi.PgtWindows()
    out.ext_value = val.ctypes.data
    import torch
    nb = sites.extreme_workspace_bytes(_cabi.PGT_MEM_HOST)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    call = lambda p, s, r, o, b=nb, so=None: lib.pgt_scan_plan_extreme(sites.handle, None, IHS, 2.0, p, s, so, r, C.byref(o), ws.data_ptr(),  # noqa: E731
                                                                     b, _cabi.PGT_MEM_HOST, None)
    assert call(pos.ctypes.data, None, None, out) == _cabi.PGT_ERR_ARGS
    assert call(pos.ctypes.data, score.ctypes.data, None, out, nb - 1) == _cabi.PGT_ERR_NOMEM
    rows.fst = fst.ctypes.data
    assert call(pos.ctypes.data, score.ctypes.data, C.byref(rows), out) == _cabi.PGT_ERR_ARGS
    out.ext_pos = fst.ctypes.data
    assert call(None, score.ctypes.data, None, out) == _cabi.PGT_ERR_ARGS
    assert call(pos.ctypes.data, score.ctypes.data, None, out) == 0
    nb_bp = bp.extreme_workspace_bytes(_cabi.PGT_MEM_HOST)
    ws_bp = torch.empty(nb_bp, dtype=torch.uint8, device="cuda")
    assert lib.pgt_scan_plan_extreme(bp.handle, None, IHS, 2.0, pos.ctypes.data, score.ctypes.data, None, None, C.byref(out),
                                     ws_bp.data_ptr(), nb_bp, _cabi.PGT_MEM_HOST, None) == _cabi.PGT_ERR_ARGS  # bp without site_offsets

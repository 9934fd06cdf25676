"""fst, het and the fused scan over bp windows (PGT_MODE_BP plans), and the sites per bp window (bp_window_sites).

A bp window is one of the windows dxyWindow -fixedsite 0 prints for the same sizefile (the window list comes from
plan.windows(), which test_plan_cpu.py pins to the dxy oracle); it reduces the sites whose positions fall on its
entries, site i of chromosome c sitting on entry off_bp[c] + pos[i] - 1.  The reference below is computed here from
that definition alone: numpy searchsorted for the membership, math.fsum for the sums."""
import math

import numpy as np
import pytest

import oracle_lib as O
import parity as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pgt():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import popgenomicstools_b200 as m
    return m


def offsets(lengths):
    return np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)


def to_dev(x):
    import torch
    x = np.ascontiguousarray(x)
    if x.dtype == np.uint32:
        return torch.from_numpy(x.view(np.int32)).cuda().view(torch.uint32)
    return torch.from_numpy(x).cuda()


def npy(out):
    import torch
    torch.cuda.synchronize()
    if not isinstance(out, dict):
        return out.cpu().numpy() if hasattr(out, "cpu") else out
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items()}


def make_input(seed, chr_len, density, gap=None):
    """Sorted distinct positions in [1, L] per chromosome (every bp for density 1, about one site per `density` bp
    otherwise; `gap` = (lo, hi) bp of chromosome 0 left without sites), and random columns for every statistic."""
    rng = np.random.default_rng(seed)
    pos, nsites = [], []
    for L in chr_len:
        if density == 1:
            p = np.arange(1, L + 1, dtype=np.uint32)
        else:
            k = max(1, L // density)
            p = np.sort(rng.choice(L, size=min(k, L), replace=False)).astype(np.uint32) + 1
        if gap is not None and not pos:
            p = p[(p < gap[0]) | (p > gap[1])]
        pos.append(p)
        nsites.append(len(p))
    pos = np.concatenate(pos)
    n = len(pos)
    cols = dict(pos=pos,
                a=rng.standard_normal(n) * 0.01,
                b=np.where(rng.random(n) < 0.05, 0.0, rng.random(n) * 0.1),
                geno=rng.integers(-1, 3, n).astype(np.int8),
                f1=rng.random(n), f2=rng.random(n),
                n1=rng.integers(0, 12, n).astype(np.int32), n2=rng.integers(0, 12, n).astype(np.int32))
    return cols, offsets(nsites)


def entries(pos, soff, boff):
    """bp entry of every site: off_bp[c] + pos - 1."""
    chrom = np.repeat(np.arange(len(soff) - 1), np.diff(soff).astype(np.int64))
    return boff[chrom].astype(np.int64) + pos.astype(np.int64) - 1


def reference(plan, cols, soff, boff):
    first, last, label = plan.windows()
    e = entries(cols["pos"], soff, boff)
    assert np.all(np.diff(e) > 0)
    lo = np.searchsorted(e, first.astype(np.int64), "left")
    hi = np.searchsorted(e, last.astype(np.int64), "right")
    a, b, g = cols["a"], cols["b"], cols["geno"]
    ref = dict(first=first, last=last, label=label, count=(hi - lo).astype(np.uint32),
               asum=np.array([math.fsum(a[i:j]) for i, j in zip(lo, hi)]),
               bsum=np.array([math.fsum(b[i:j]) for i, j in zip(lo, hi)]),
               aabs=np.array([math.fsum(np.abs(a[i:j])) for i, j in zip(lo, hi)]),
               babs=np.array([math.fsum(np.abs(b[i:j])) for i, j in zip(lo, hi)]))
    csum = lambda m: np.concatenate([[0], np.cumsum(m, dtype=np.int64)])
    nm, nh = csum(g >= 0), csum(g == 1)
    ref["nonmissing"] = (nm[hi] - nm[lo]).astype(np.uint32)
    ref["nhet"] = (nh[hi] - nh[lo]).astype(np.uint32)
    return ref


def check_against_reference(res_f, res_h, ref, boff):
    nbp = (ref["last"] - ref["first"] + 1).astype(np.uint32)
    for res in (res_f, res_h):
        P.assert_exact(res["label"], ref["label"], "label")
        P.assert_exact(res["nsites"], nbp, "nsites (bp)")
        cf = np.searchsorted(boff, ref["first"], "right") - 1
        P.assert_exact(res["start_pos"], (ref["first"] - boff[cf] + 1).astype(np.uint32), "start_pos")
        P.assert_exact(res["end_pos"], (ref["last"] - boff[ref["label"]] + 1).astype(np.uint32), "end_pos")
        mid = ((res["start_pos"].astype(np.uint64) + res["end_pos"]) % (1 << 32) // 2).astype(np.uint32)
        P.assert_exact(res["mid_pos"], mid, "mid_pos")
    P.assert_sum_close(res_f["sum_a"], ref["asum"], ref["aabs"], "sum_a")
    P.assert_sum_close(res_f["sum_b"], ref["bsum"], ref["babs"], "sum_b")
    sa, sb = res_f["sum_a"], res_f["sum_b"]
    with np.errstate(divide="ignore", invalid="ignore"):
        P.assert_exact(res_f["fst"], np.where(sb != 0, sa / np.where(sb != 0, sb, 1.0), 0.0), "fst")
        P.assert_exact(res_h["nhet"], ref["nhet"], "nhet")
        P.assert_exact(res_h["nonmissing"], ref["nonmissing"], "nonmissing")
        nm = res_h["nonmissing"].astype(np.float64)
        P.assert_exact(res_h["het"], np.where(nm > 0, res_h["nhet"] / np.where(nm > 0, nm, 1.0), 0.0), "het")


def scan_all(pgt, plan, cols, soff, on_device):
    c = {k: to_dev(v) for k, v in cols.items()} if on_device else cols
    f = npy(pgt.fst_window(plan, c["pos"], c["a"], c["b"], site_offsets=soff))
    h = npy(pgt.het_window(plan, c["pos"], c["geno"], site_offsets=soff))
    d = npy(pgt.dxy_window(plan, c["pos"], c["f1"], c["f2"], c["n1"], c["n2"], minind=5, site_offsets=soff))
    u = npy(pgt.fused_window(plan, c["pos"], c["a"], c["b"], c["geno"], c["f1"], c["f2"], c["n1"], c["n2"], minind=5,
                             site_offsets=soff))
    return f, h, d, u


# (chromosome lengths in bp, W, S, bp per site, unit_sites)
CASES = {
    # a chromosome no longer than W - S in the middle (stale carry) and at the end (dropped at EOF)
    "dense": ([120_000, 3_000, 57_000, 800], 50_000, 10_000, 1, 0),
    "dense_u4096": ([120_000, 3_000, 57_000, 800], 50_000, 10_000, 1, 4096),
    "sparse": ([900_000, 25_000, 31_000, 400_000, 20_000], 50_000, 10_000, 30, 0),
    "sparse_u4096": ([900_000, 25_000, 31_000, 400_000, 20_000], 50_000, 10_000, 30, 4096),
    "many_short": (list(np.random.default_rng(7).integers(100, 3000, 300)), 5_000, 1_000, 3, 32),
    "w_eq_s": ([100_000, 77_777, 5_000], 10_000, 10_000, 1, 256),
    "fine_dense": ([20_000, 700, 15_000], 1_000, 1, 1, 0),
    "fine_sparse": ([60_000, 700, 45_000], 1_000, 1, 30, 0),
    "step100": ([300_000, 999, 77_000], 1_000, 100, 30, 64),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_bp_windows_match_reference_dxy_rows_and_fused(pgt, case):
    chr_len, W, S, density, unit = CASES[case]
    boff = offsets(chr_len)
    cols, soff = make_input(11, chr_len, density, gap=(30_000, 75_000) if case.startswith("sparse") else None)
    plan = pgt.WindowPlan(boff, W, S, mode="bp", unit_sites=unit)
    assert plan.scan_path(0) == plan.scan_path(1) == plan.scan_path(3) == "units"
    ref = reference(plan, cols, soff, boff)
    f, h, d, u = scan_all(pgt, plan, cols, soff, True)
    check_against_reference(f, h, ref, boff)
    # the rows line up with dxyWindow -fixedsite 0 over the same plan, bit for bit, and with the dxy oracle
    for res in (f, h, u):
        for k in ("label", "start_pos", "end_pos", "nsites"):
            assert res[k].tobytes() == d[k].tobytes(), k
    chr_id = np.repeat(np.arange(len(chr_len), dtype=np.uint32), np.diff(soff).astype(np.int64))
    dref = O.dxy(chr_id, cols["pos"], cols["f1"], cols["f2"], cols["n1"], cols["n2"], 5, W, S, 0, 0, chr_len)
    P.assert_exact(d["label"], dref["label"], "oracle label")
    P.assert_exact(d["start_pos"].astype(np.int64), dref["start"], "oracle start")
    P.assert_exact(d["end_pos"].astype(np.int64), dref["end"], "oracle end")
    # the fused scan equals the three single scans bit for bit
    for one in (f, h, d):
        for k, v in one.items():
            assert v.tobytes() == u[k].tobytes(), k
    # sites per window
    P.assert_exact(npy(pgt.bp_window_sites(plan, to_dev(cols["pos"]), soff)), ref["count"], "bp_window_sites")


@pytest.mark.parametrize("case", ["dense", "sparse_u4096", "many_short"])
def test_bp_het_level1_kernels_agree(pgt, case):
    """hetWindow's byte kernels over bp units, which start and end anywhere in the 1-byte column: the vectorised
    direct kernel (ragged heads and tails around its 16-byte chunks) and the tiled kernel give the same counts."""
    chr_len, W, S, density, unit = CASES[case]
    boff = offsets(chr_len)
    cols, soff = make_input(12, chr_len, density)
    plan = pgt.WindowPlan(boff, W, S, mode="bp", unit_sites=unit)
    ref = reference(plan, cols, soff, boff)
    pos, g = to_dev(cols["pos"]), to_dev(cols["geno"])
    try:
        for mode in (0, 1, 2):
            pgt.tune("level1", mode)
            res = npy(pgt.het_window(plan, pos, g, site_offsets=soff))
            P.assert_exact(res["nhet"], ref["nhet"], f"nhet level1={mode}")
            P.assert_exact(res["nonmissing"], ref["nonmissing"], f"nonmissing level1={mode}")
    finally:
        pgt.tune("level1", 0)


def test_bp_host_mode_and_shards_equal_device_mode(pgt):
    """Host-memory scans over several slabs of the bp axis, and the sharded scan over a repeated device list, give
    the device-mode tables bit for bit."""
    from popgenomicstools_b200 import _cabi
    chr_len = [9_000_000, 40_000, 3_500_000]  # > 3 host-mode slabs of entries
    boff = offsets(chr_len)
    cols, soff = make_input(13, chr_len, 30, gap=(1_000_000, 1_200_000))
    plan = pgt.WindowPlan(boff, 50_000, 10_000, mode="bp")
    dev = scan_all(pgt, plan, cols, soff, True)
    host = scan_all(pgt, plan, cols, soff, False)
    for dv, hv in zip(dev, host):
        for k, v in dv.items():
            assert hv[k].tobytes() == v.tobytes(), k
    fused = dev[3]
    unbound = pgt.WindowPlan(boff, 50_000, 10_000, mode="bp")  # (device-mode scans bound `plan` to one device)
    for stat, want in ((_cabi.PGT_STAT_FST, dev[0]), (_cabi.PGT_STAT_HET, dev[1]), (_cabi.PGT_STAT_FUSED, fused)):
        for devs in ([0, 0, 0], [0] * 5):
            res = pgt.scan_sharded(unbound, stat, cols, devs, minind=5, site_offsets=soff)
            for k, v in want.items():
                if k == "dxy_global":  # the shards' disjoint partial lines, added in shard order
                    assert res[k][1] == v[1] and res[k][2] == v[2] and abs(res[k][0] - v[0]) <= 1e-12 * abs(v[0])
                else:
                    assert res[k].tobytes() == v.tobytes(), (stat, devs, k)
    # sites per window: numpy and device tensors give the same counts, and so does a shard's range
    ref = reference(plan, cols, soff, boff)
    assert np.any(ref["count"] == 0)
    P.assert_exact(pgt.bp_window_sites(plan, cols["pos"], soff), ref["count"], "host bp_window_sites")
    wl, wh, el, eh = plan.shard(1, 3)  # (a bp plan's shard range is in entries: its sites are those on them)
    sl, sh = np.searchsorted(entries(cols["pos"], soff, boff), [el, eh])
    assert wh > wl and sh > sl
    part = npy(pgt.bp_window_sites(plan, to_dev(cols["pos"][sl:sh]), soff, window_range=(wl, wh), site_origin=sl,
                                   site_count=sh - sl))
    P.assert_exact(part, ref["count"][wl:wh], "shard bp_window_sites")
    part = pgt.bp_window_sites(plan, cols["pos"][sl:sh], soff, window_range=(wl, wh), site_origin=sl,
                               site_count=sh - sl)
    P.assert_exact(part, ref["count"][wl:wh], "host shard bp_window_sites")


def test_bp_window_sites_zero_windows_and_bad_positions(pgt):
    from popgenomicstools_b200 import _cabi
    chr_len = [100_000, 2_000, 60_000]
    boff = offsets(chr_len)
    cols, soff = make_input(14, chr_len, 50, gap=(10_000, 70_000))
    plan = pgt.WindowPlan(boff, 5_000, 1_000, mode="bp")
    ref = reference(plan, cols, soff, boff)
    assert np.sum(ref["count"] == 0) > 10
    for pos in (to_dev(cols["pos"]), cols["pos"]):
        P.assert_exact(npy(pgt.bp_window_sites(plan, pos, soff)), ref["count"], "bp_window_sites")
    # a site beyond its chromosome's length, or at position 0, is an input error
    for c, value in ((0, chr_len[0] + 1), (2, chr_len[2] + 7), (1, 0)):
        bad = cols["pos"].copy()
        i = int(soff[c + 1]) - 1 if value else int(soff[c])
        bad[i] = value
        for pos in (to_dev(bad), bad):
            with pytest.raises(pgt.PgtError) as e:
                pgt.bp_window_sites(plan, pos, soff)
            assert e.value.code == _cabi.PGT_ERR_INPUT and str(i) in str(e.value)
    # a site-mode plan has no bp windows
    with pytest.raises(pgt.PgtError) as e:
        pgt.bp_window_sites(pgt.WindowPlan(soff, 10, 5), cols["pos"], soff)
    assert e.value.code == _cabi.PGT_ERR_ARGS

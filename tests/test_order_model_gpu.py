"""Every kernel path against the summation-order model (tests/order_model.py), bit for bit.

DESIGN §4 states each window's floating-point result as a pure function of (W, S, u) and the segment origin; the
model restates that order on the CPU.  Here every statistic (fst, het, dxy, fused) on every path -- level 1 direct /
tiled, level 2 warp per window / thread per window / scan mode, the sliding tile (one crew and the fused two-crew
kernel), the per-site map (vector and scalar), the unit-start table, bp mode dense and sparse, host memory, shards and
the sharded scan -- must give the model's sum and ratio columns tobytes()-equal (NaN compared as NaN) on the synth,
wide and nonfinite value families, and the oracle's integer columns.  On the dyadic family every sum is exact, so
there the GPU equals the oracle bit for bit everywhere, dxyWindow's global line included.  A failure names the path,
the column and the first windows that differ."""
import contextlib

import numpy as np
import pytest

import oracle_lib as O
import order_model as M
import textfmt as T
from popgenomicstools_b200 import _cabi
from test_order_model_cpu import (MININD, SITE_SHAPES, bp_input, family, first_diff, many_contig_lengths, offsets, same_bits,
                                  site_lengths)

pytestmark = pytest.mark.gpu

KNOBS = ("level1", "level2", "slide", "fused2", "persite", "unittable")
STATS = {"fst": _cabi.PGT_STAT_FST, "het": _cabi.PGT_STAT_HET, "dxy": _cabi.PGT_STAT_DXY, "fused": _cabi.PGT_STAT_FUSED}
COLS = {"fst": ("a", "b"), "het": ("geno",), "dxy": ("f1", "f2", "n1", "n2"), "fused": ("a", "b", "geno", "f1", "f2", "n1", "n2")}


@pytest.fixture(scope="module")
def pgt():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import popgenomicstools_b200 as m
    yield m
    for k in KNOBS:
        m.tune(k, 0)


@contextlib.contextmanager
def knobs(pgt, **kv):
    try:
        for k, v in kv.items():
            pgt.tune(k, v)
        yield
    finally:
        for k in KNOBS:
            pgt.tune(k, 0)


def npy(out):
    import torch
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in out.items()}


def device(cols):
    import torch
    return {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in cols.items()}


def run(pgt, plan, stat, cols, **kw):
    return npy(pgt.scan(plan, STATS[stat], {k: cols[k] for k in ("pos",) + COLS[stat]}, minind=MININD, **kw))


def compare(res, model, stat, tag, oracle_ints=None):
    for k in M.FLOAT_COLS[stat]:
        if not same_bits(res[k], model[k]):
            w, g, m = first_diff(res[k], model[k])
            raise AssertionError(f"{tag}: windows {w.tolist()}, {k} differs from the documented order: gpu {g.tolist()} model {m.tolist()}")
    for k in M.INT_COLS[stat]:
        want = model[k] if oracle_ints is None else oracle_ints[k]
        assert np.array_equal(res[k], want), f"{tag}: {k} differs from the oracle at windows {np.nonzero(res[k] != want)[0][:5].tolist()}"


def oracle_site(lengths, pos, c, W, S):
    chr_id = T.expand_chr(lengths)
    rf = O.fst(chr_id, pos, c["a"], c["b"], W, S)
    rh = O.het(chr_id, pos, c["geno"], W, S)
    rd = O.dxy(chr_id, pos, c["f1"], c["f2"], c["n1"], c["n2"], MININD, W, S, 1)
    return dict(sum_a=rf["asum"], sum_b=rf["bsum"], fst=rf["fst"], het=rh["h"], nhet=rh["nhet"], nonmissing=rh["nonmissing"],
                dxy=rd["dxy"], neffective=rd["neff"], nskip=rd["nskip"], dxy_global=rd["global"])


def check_dyadic(res, ora, stat, tag):
    """dyadic: every sum is exact, so the GPU equals the oracle bit for bit, the global line included."""
    compare(res, ora, stat, tag + " (dyadic vs oracle)", ora)
    if "dxy_global" in res:
        assert same_bits(res["dxy_global"], ora["dxy_global"]), (tag, res["dxy_global"], ora["dxy_global"])


def site_configs(plan, W, S, u):
    """(tag, knobs, expected path) for every path a site-mode plan can be forced through."""
    g = M.Geom(W, S, u)
    cfg = [("auto", {}, None)]
    for l1 in ((0, 1, 2) if g.gw == 32 else (0, 2)):
        cfg.append((f"level1={l1} level2=1", dict(slide=1, level1=l1, level2=1), "tree"))
    if g.wunits >= 2:
        cfg.append(("level2=2", dict(slide=1, level2=2), "scan"))
        cfg.append(("level1=2 level2=2", dict(slide=1, level1=2, level2=2), "scan"))
    if W <= 1048:
        for f2 in (0, 1):
            cfg.append((f"slide=2 fused2={f2}", dict(slide=2, fused2=f2), "slide"))
    if W == 1 and S == 1:
        for ps in (0, 1):
            cfg.append((f"persite={ps}", dict(persite=ps), "persite"))
    return cfg


def check_plan(pgt, plan, lengths, W, S, u, fams=("synth", "wide", "nonfinite", "dyadic"), extra=True, configs=None):
    offs = plan.offsets
    n = int(offs[-1])
    pos = O.synth_pos(1, offs, 1)
    L = M.Layout(plan, u)
    for fam in fams:
        c = dict(family(fam, n, 7, huge=True), pos=pos)
        d = device(c)
        models = {}
        ora = oracle_site(lengths, pos, c, W, S)
        for tag, kv, want in (configs or site_configs(plan, W, S, u)):
            with knobs(pgt, **kv):
                path = M.path_of(plan, STATS["fused"], kv.get("level2", 0), u)
                assert want is None or path == want, (tag, path, want)
                if path not in models:
                    models[path] = M.window_table(plan, "fused", c, path, minind=MININD, layout=L)
                for stat in STATS:
                    res = run(pgt, plan, stat, d)
                    where = f"{fam} W={W} S={S} u={u} {tag} path {path} {stat}"
                    compare(res, models[path], stat, where, ora)
                    if fam == "dyadic":
                        check_dyadic(res, ora, stat, where)
        if not extra or fam not in ("wide", "dyadic"):
            continue
        # host memory, shards (device columns sliced per shard) and the sharded scan, under the automatic choice
        path = M.path_of(plan, STATS["fused"], 0, u)
        model = models.get(path) or M.window_table(plan, "fused", c, path, minind=MININD, layout=L)
        where = f"{fam} W={W} S={S} u={u} path {path}"
        compare(run(pgt, plan, "fused", c), model, "fused", where + " host memory", ora)
        parts, glob = [], np.zeros(3)
        for r in range(3):
            wl, wh, sl, sh = plan.shard(r, 3)
            if wh > wl:
                parts.append(run(pgt, plan, "fused", {k: v[sl:sh] for k, v in d.items()}, window_range=(wl, wh), site_origin=sl))
                glob = glob + parts[-1]["dxy_global"]
        cat = {k: np.concatenate([p[k] for p in parts]) for k in parts[0] if k != "dxy_global"}
        compare(cat, model, "fused", where + " 3 shards", ora)
        unbound = pgt.WindowPlan(offs, W, S, unit_sites=u)  # pgt_scan_sharded binds the plan on every device itself
        sh = pgt.scan_sharded(unbound, STATS["fused"], {k: c[k] for k in ("pos",) + COLS["fused"]}, [0, 0], minind=MININD)
        compare(sh, model, "fused", where + " pgt_scan_sharded", ora)
        if fam == "dyadic":
            assert same_bits(glob, ora["dxy_global"]), (where, "shard global lines", glob, ora["dxy_global"])
            assert same_bits(sh["dxy_global"], ora["dxy_global"]), (where, "sharded global line")


@pytest.mark.parametrize("W,S,u", SITE_SHAPES)
def test_site_mode_paths_match_the_model(pgt, W, S, u):
    lengths = site_lengths(W, S)
    check_plan(pgt, pgt.WindowPlan(offsets(lengths), W, S, unit_sites=u), lengths, W, S, u)


@pytest.mark.parametrize("W,S,u", [(1000, 1000, 0), (100, 10, 0), (5000, 1000, 512), (300, 300, 32)])
def test_many_contigs_unit_table_matches_the_model(pgt, W, S, u):
    """More than 32 segments: the unit-start table (unittable 1 / 2) under every level-1 kernel."""
    lengths = many_contig_lengths(W, S)
    plan = pgt.WindowPlan(offsets(lengths), W, S, unit_sites=u)
    assert plan.num_segments > 32
    g = M.Geom(W, S, u)
    cfg = [(f"unittable={t} level1={l1}", dict(unittable=t, level1=l1, slide=1), None)
           for t in (1, 2) for l1 in ((0, 1, 2) if g.gw == 32 else (0, 2))]
    check_plan(pgt, plan, lengths, W, S, u, fams=("wide", "dyadic"), configs=cfg)


def test_k_windows_many_row_batches_matches_the_model(pgt):
    """k_windows over many 32-row batches per block (1e5 windows of 80 units), contig ends inside batches."""
    lengths = [1_700_003, 2560 + 31, 900_000, 5, 700_017]
    W, S, u = 2560, 32, 32
    plan = pgt.WindowPlan(offsets(lengths), W, S, unit_sites=u)
    check_plan(pgt, plan, lengths, W, S, u, fams=("wide", "dyadic"), extra=False,
               configs=[("level2=1", dict(level2=1), "tree"), ("level1=2 level2=1", dict(level1=2, level2=1), "tree")])


@pytest.mark.parametrize("density", [10, 1])
@pytest.mark.parametrize("W,S", [(2000, 500), (100, 100), (1, 1), (777, 10)])
def test_bp_mode_matches_the_model(pgt, W, S, density):
    """bp windows (sparse: one site per 10 bp; dense: every bp) for every statistic, level-1 and level-2 kernels, host
    memory; the integer columns against dxyWindow -fixedsite 0's counts."""
    boff, soff, pos = bp_input(W, S, density)
    n = int(soff[-1])
    plan = pgt.WindowPlan(boff, W, S, mode="bp")
    L = M.Layout(plan)
    g = M.Geom(W, S, 0)
    chr_len = np.diff(boff.astype(np.int64))
    for fam in ("synth", "wide", "nonfinite", "dyadic"):
        c = dict(family(fam, n, 8, huge=True), pos=pos)
        d = device(c)
        rd = O.dxy(T.expand_chr(np.diff(soff.astype(np.int64))), pos, c["f1"], c["f2"], c["n1"], c["n2"], MININD, W, S, 0, 0, chr_len)
        models = {}
        cfg = [(f"level1={l1} level2={l2}", dict(level1=l1, level2=l2)) for l1 in (0, 2) for l2 in ((1, 2) if g.wunits >= 2 else (1,))]
        cfg.append(("auto", {}))
        for tag, kv in cfg:
            with knobs(pgt, **kv):
                path = M.path_of(plan, STATS["fused"], kv.get("level2", 0))
                if path not in models:
                    models[path] = M.window_table(plan, "fused", c, path, minind=MININD, site_offsets=soff, layout=L)
                m = models[path]
                assert np.array_equal(m["neffective"], rd["neff"]) and np.array_equal(m["nskip"], rd["nskip"]), "model counts vs oracle"
                for stat in STATS:
                    res = run(pgt, plan, stat, d, site_offsets=soff)
                    where = f"{fam} bp W={W} S={S} density={density} {tag} path {path} {stat}"
                    compare(res, m, stat, where)
                    if fam == "dyadic" and stat in ("dxy", "fused"):
                        assert same_bits(res["dxy"], rd["dxy"]), where + " dxy vs oracle"
                        assert same_bits(res["dxy_global"], rd["global"]), where + " global line vs oracle"
                if kv == {}:
                    compare(run(pgt, plan, "fused", c, site_offsets=soff), m, "fused", f"{fam} bp W={W} S={S} path {path} host memory")

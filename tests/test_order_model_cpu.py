"""The summation-order model (tests/order_model.py) against the oracle and against exactly rounded sums, and the unit
geometry it is built on.  No GPU: the plan functions of libpgtscan.so and numpy only.

Value families (also used by test_order_model_gpu.py):
  synth      the project's synthetic columns (oracle_lib's CPU twins);
  dyadic     a, b = k/1024 (|k| < 2^20, many zeros, sign-balanced b: Σb == 0 exactly in many windows), f = k/1024 in
             [0, 1], n in 0..20, genotypes of all 256 byte values: every sum is exact in any order;
  wide       ±m·2^e (53-bit m, e in [-40, 40]), exact ±0.0, subnormals, optionally a few values near 1e308 where the
             order decides between finite and Inf: order matters maximally;
  nonfinite  synth with a few NaN and ±Inf in a, b, f1, f2, and f outside [0, 1] (a site's dxy value < 0 but not -9).
"""
import math

import numpy as np
import pytest

import oracle_lib as O
import order_model as M
import parity as P
import textfmt as T
from popgenomicstools_b200 import WindowPlan

FAMILIES = ("synth", "dyadic", "wide", "nonfinite")
MININD = 5


def offsets(lengths):
    return np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)


def _wide(rng, n, huge):
    m = rng.integers(2 ** 52, 2 ** 53, n).astype(np.float64)
    x = np.ldexp(m, rng.integers(-40 - 52, 40 - 52 + 1, n)) * rng.choice([-1.0, 1.0], n)
    k = rng.random(n)
    x[k < 0.05] = 0.0
    x[(k >= 0.05) & (k < 0.08)] = -0.0
    sub = (k >= 0.08) & (k < 0.10)
    x[sub] = np.ldexp(rng.integers(1, 2 ** 40, int(sub.sum())).astype(np.float64), -1074) * rng.choice([-1.0, 1.0], int(sub.sum()))
    if huge:
        big = rng.random(n) < 0.002
        x[big] = rng.choice([-1.0, 1.0], int(big.sum())) * rng.uniform(0.6e308, 1.7e308, int(big.sum()))
    return x


def family(name, n, seed, huge=False):
    """Host columns a, b, geno, f1, f2, n1, n2 of `n` sites of value family `name`."""
    rng = np.random.default_rng(seed)
    if name in ("synth", "nonfinite"):
        a, b = O.synth_fst(seed, 0, n)
        g = O.synth_het(seed, 0, n)
        f1, f2, n1, n2 = O.synth_dxy(seed, 0, n)
        c = dict(a=a, b=b, geno=g, f1=f1, f2=f2, n1=n1, n2=n2)
        if name == "nonfinite":
            for k in ("a", "b", "f1", "f2"):
                x = c[k]
                sel = rng.random(n)
                x[sel < 0.002] = np.nan
                x[(sel >= 0.002) & (sel < 0.004)] = np.inf
                x[(sel >= 0.004) & (sel < 0.006)] = -np.inf
                if k in ("f1", "f2"):
                    out = (sel >= 0.006) & (sel < 0.05)
                    x[out] = rng.uniform(-3.0, 4.0, int(out.sum()))
        return c
    if name == "dyadic":
        a = rng.integers(-(2 ** 20) + 1, 2 ** 20, n) / 1024.0
        a[rng.random(n) < 0.3] = 0.0
        # b: zero stretches (Σb == 0, the fst epilogue's 0 branch) and sign-balanced pairs
        b = rng.integers(-(2 ** 20) + 1, 2 ** 20, n) / 1024.0
        b[1::2] = -b[0:-1:2][: len(b[1::2])]
        zero = (np.arange(n) // 1500) % 3 == 1
        b[zero] = 0.0
        b[rng.random(n) < 0.2] = 0.0
        f1 = rng.integers(0, 1025, n) / 1024.0
        f2 = rng.integers(0, 1025, n) / 1024.0
        n1 = rng.integers(0, 21, n).astype(np.int32)
        n2 = rng.integers(0, 21, n).astype(np.int32)
        g = rng.integers(-128, 128, n).astype(np.int8)
        common = rng.random(n) < 0.5
        g[common] = rng.choice(np.array([-1, 0, 1, 2], np.int8), int(common.sum()))
        return dict(a=a, b=b, geno=g, f1=f1, f2=f2, n1=n1, n2=n2)
    if name == "wide":
        a, b = _wide(rng, n, huge), _wide(rng, n, huge)
        # f = m·2^e in (0, 1): dxy values of every magnitude, nearly all of them counted
        f1 = np.ldexp(rng.integers(2 ** 52, 2 ** 53, n).astype(np.float64), rng.integers(-40 - 53, -53, n))
        f2 = np.ldexp(rng.integers(2 ** 52, 2 ** 53, n).astype(np.float64), rng.integers(-40 - 53, -53, n))
        n1 = rng.integers(0, 21, n).astype(np.int32)
        n2 = rng.integers(0, 21, n).astype(np.int32)
        g = rng.integers(-128, 128, n).astype(np.int8)
        return dict(a=a, b=b, geno=g, f1=f1, f2=f2, n1=n1, n2=n2)
    raise ValueError(name)


def oracle_tables(lengths, pos, c, W, S):
    chr_id = T.expand_chr(lengths)
    rf = O.fst(chr_id, pos, c["a"], c["b"], W, S)
    ra = O.fst(chr_id, pos, np.abs(c["a"]), np.abs(c["b"]), W, S)
    rh = O.het(chr_id, pos, c["geno"], W, S)
    rd = O.dxy(chr_id, pos, c["f1"], c["f2"], c["n1"], c["n2"], MININD, W, S, 1)
    return dict(sum_a=rf["asum"], sum_b=rf["bsum"], fst=rf["fst"], het=rh["h"], nhet=rh["nhet"], nonmissing=rh["nonmissing"],
                dxy=rd["dxy"], neffective=rd["neff"], nskip=rd["nskip"]), dict(sum_a=ra["asum"], sum_b=ra["bsum"])


def same_bits(x, y):
    """Bit for bit, every NaN equal to every NaN (the GPU makes the canonical NaN, x86 may set its sign bit)."""
    x, y = np.asarray(x), np.asarray(y)
    if x.dtype.kind != "f":
        return x.shape == y.shape and np.array_equal(x, y)
    nx, ny = np.isnan(x), np.isnan(y)
    return x.shape == y.shape and np.array_equal(nx, ny) and x[~nx].tobytes() == y[~ny].tobytes()


def first_diff(x, y):
    x, y = np.asarray(x), np.asarray(y)
    nx, ny = np.isnan(x), np.isnan(y)
    bad = np.nonzero((nx != ny) | (~nx & (x.view(np.uint64) != y.view(np.uint64))))[0]
    return bad[:5], x[bad[:5]], y[bad[:5]]


def paths_for(W, S, u=0):
    """The orders the model can be asked for at this shape (each forced through pgt_tune on the GPU)."""
    g = M.Geom(W, S, u)
    out = ["tree"]
    if g.wunits >= 2:
        out.append("scan")
    if W <= 1048:
        out.append("slide")
    if W == 1 and S == 1:
        out.append("persite")
    return out


# site-mode shapes: test_paths_gpu's list, test_slide_gpu's SHAPES, test_stats_gpu's scan-mode list
SITE_SHAPES = [(5000, 100, 0), (1000, 100, 0), (300, 299, 0), (1, 1, 0), (64, 1, 0), (777, 13, 32), (2560, 256, 0), (4096, 4096, 4096),
               (100, 10, 0), (24, 3, 32), (8, 4, 0), (31, 1, 0), (5000, 1000, 512),
               (2, 1, 0), (5, 2, 0), (64, 64, 0), (255, 7, 0), (256, 1, 0), (257, 3, 0), (1000, 1, 0), (1000, 7, 0), (1024, 32, 0),
               (1047, 5, 0), (1048, 1, 0), (1048, 1048, 0), (129, 1, 0), (192, 5, 0), (500, 3, 0), (700, 1, 0),
               (5000, 3, 0), (40, 40, 0)]


def site_lengths(W, S):
    return [W + 4 * S, 6011, 3, W // 2 + 1, 2 * W + 1, 4000, max(1, W - S)]


def many_contig_lengths(W, S):
    rng = np.random.default_rng(W * 7 + S)
    return rng.integers(1, 700, size=300).tolist() + [1, 2, W, W + S, 3 * W + 1]


def bp_input(W, S, density, seed=2):
    """bp-mode plan offsets (chromosome lengths), site offsets and sorted unique positions."""
    nsites = [3000, 1500, 40]
    chr_len = [x * density + 17 for x in nsites]
    rng = np.random.default_rng(seed)
    pos = np.concatenate([np.sort(rng.choice(np.arange(1, L + 1), size=ns, replace=False)) for ns, L in zip(nsites, chr_len)]).astype(np.uint32)
    return offsets(chr_len), offsets(nsites), pos


@pytest.mark.parametrize("W,S,u", SITE_SHAPES)
def test_geometry_units_tile_every_window(W, S, u):
    for lengths in (site_lengths(W, S), many_contig_lengths(W, S)):
        M.Layout(WindowPlan(offsets(lengths), W, S, unit_sites=u), u)


@pytest.mark.parametrize("density", [10, 1])
@pytest.mark.parametrize("W,S", [(2000, 500), (100, 100), (1, 1), (777, 10)])
def test_geometry_bp_mode(W, S, density):
    boff, soff, pos = bp_input(W, S, density)
    L = M.Layout(WindowPlan(boff, W, S, mode="bp"))
    lo, hi = L.unit_sites(pos, soff)
    assert lo[0] == 0 and hi[-1] == soff[-1] and np.array_equal(hi[:-1], lo[1:]), "bp units do not tile the sites"


def _check_table(tab, want, cols, what, exact, absref=None):
    for k in cols:
        if exact:
            assert same_bits(tab[k], want[k]), f"{what} {k}: {first_diff(tab[k], want[k])}"
        elif k in ("sum_a", "sum_b"):
            P.assert_sum_close(tab[k], want[k], absref[k], f"{what} {k}")
        elif k == "dxy":
            P.assert_sum_close(tab[k], want[k], want[k], f"{what} {k}")


CPU_SHAPES = [(1000, 100, 0), (300, 299, 0), (1, 1, 0), (64, 1, 0), (777, 13, 32), (24, 3, 32), (31, 1, 0), (1000, 1, 0), (255, 7, 0),
              (5000, 3, 0), (40, 40, 0)]


@pytest.mark.parametrize("fam", ["synth", "wide", "dyadic"])
@pytest.mark.parametrize("W,S,u", CPU_SHAPES)
def test_model_against_oracle(W, S, u, fam):
    """synth and wide: within parity.py's tolerance; dyadic (every sum exact): bit for bit, on every path."""
    lengths = site_lengths(W, S)
    offs = offsets(lengths)
    n = int(offs[-1])
    c = family(fam, n, 3)
    pos = O.synth_pos(1, offs, 1)
    want, absref = oracle_tables(lengths, pos, c, W, S)
    plan = WindowPlan(offs, W, S, unit_sites=u)
    L = M.Layout(plan, u)
    for path in paths_for(W, S, u):
        tab = M.window_table(plan, "fused", dict(c, pos=pos), path, minind=MININD, layout=L)
        for k in M.INT_COLS["fused"]:
            P.assert_exact(tab[k], want[k], f"{path} {k}")
        assert same_bits(tab["het"], want["het"]), f"{path} het"
        _check_table(tab, want, ("sum_a", "sum_b", "dxy") + (("fst",) if fam == "dyadic" else ()), f"{fam} W={W} S={S} {path}",
                     fam == "dyadic", absref)


@pytest.mark.parametrize("fam", FAMILIES)
def test_per_site_dxy_equals_oracle_on_every_family(fam):
    """W = S = 1: the window is the site (+0.0 + x); dxyWindow adds the same value to 0.  Bit for bit, NaN as NaN."""
    lengths = site_lengths(1, 1)
    offs = offsets(lengths)
    c = family(fam, int(offs[-1]), 4, huge=True)
    pos = O.synth_pos(1, offs, 1)
    want, _ = oracle_tables(lengths, pos, c, 1, 1)
    plan = WindowPlan(offs, 1, 1)
    tab = M.window_table(plan, "dxy", dict(c, pos=pos), "persite", minind=MININD)
    assert same_bits(tab["dxy"], want["dxy"]), first_diff(tab["dxy"], want["dxy"])
    P.assert_exact(tab["neffective"], want["neffective"], "neff")
    P.assert_exact(tab["nskip"], want["nskip"], "nskip")


@pytest.mark.parametrize("fam", ["synth", "wide"])
@pytest.mark.parametrize("W,S,u", [(1000, 100, 0), (777, 13, 32), (64, 1, 0), (1000, 1, 0), (5000, 3, 0), (24, 3, 32), (300, 299, 0)])
def test_model_within_tree_depth_bound_of_exact_sum(W, S, u, fam):
    """|model - fsum| <= γ_d Σ|x| with d the path's tree depth (order_model.depth): DESIGN's "true partial sums only, no
    cancellation" as a number.  (No values near 1e308 here: math.fsum raises on intermediate overflow.)"""
    lengths = site_lengths(W, S)
    offs = offsets(lengths)
    c = family(fam, int(offs[-1]), 5)
    plan = WindowPlan(offs, W, S, unit_sites=u)
    L = M.Layout(plan, u)
    lo, hi = L.window_sites()
    d, _ = M.site_channels("fused", c, MININD)
    exact = {k: M.exact_sums(x, lo, hi) for k, x in d.items()}
    mag = {k: M.exact_sums(np.abs(x), lo, hi) for k, x in d.items()}
    eps = 2.0 ** -53
    for path in paths_for(W, S, u):
        dep = M.depth(L, path)
        gamma = dep * eps / (1 - dep * eps)
        tab = M.window_table(plan, "fused", dict(c, pos=None), path, minind=MININD, layout=L)
        for k in d:
            err = np.abs(tab[k] - exact[k])
            bad = np.nonzero(~(err <= gamma * mag[k]))[0]
            assert len(bad) == 0, f"{path} {k}: depth {dep}, windows {bad[:5]} err {err[bad[:5]]} bound {gamma * mag[k][bad[:5]]}"
        # the bound is not vacuous: the model is off the exact sum somewhere on the wide family
        if fam == "wide" and path != "persite":
            assert any(np.any(tab[k] != exact[k]) for k in d) or W <= 2


def test_model_restates_kernel_details():
    """Small hand checks of the order the model states: the group butterfly pairs lanes l and l + G/2 first; the warp
    scans put the earlier item on the left; slide_team is the kernel's table."""
    assert M.slide_team(1000) == (5, 7, 1) and M.slide_team(256) == (4, 2, 3)
    x = np.array([1e16, 1.0, -1e16, 1.0])  # lanes 0..3: (x0 + x2) + (x1 + x3) = 0 + 2
    assert M.butterfly(x[None, :])[0] == 2.0
    y = np.array([1.0, 1e16, -1e16, 1.0, 0, 0, 0, 0])  # sequential lanes would give 1.0; the butterfly gives (1 - 1e16) + (1e16 + 1)
    assert M.butterfly(y[None, :])[0] == (1.0 + -1e16) + (1e16 + 1.0)
    lo, hi = np.array([0]), np.array([40])
    v = np.arange(40, dtype=np.float64)
    assert M.unit_partials(v, lo, hi, 8)[0] == 780.0

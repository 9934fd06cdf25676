"""CPU restatement of the summation order of every window kernel (DESIGN.md §4), bit for bit.

TEST INFRASTRUCTURE ONLY, like oracle_lib.py.  Given a WindowPlan, a statistic, host columns and the path a scan
takes, `window_table` returns the sum / ratio columns the kernels must produce, every addition one IEEE double
addition in the kernels' order.  Each function names the CUDA code it restates.  Rules:
  * additions are elementwise `+` on arrays (vectorised over units, windows or blocks); no pairwise reduction
    (np.sum / np.add.reduce) touches a floating-point value;
  * the geometry is ported from pgt_geom.h / pgt_plan.cpp and checked against the plan API first (units tile every
    window with no gap and no overlap);
  * dxyWindow's global line is not restated (its order depends on the grid).
"""
import numpy as np

from popgenomicstools_b200 import _cabi

F64 = np.float64
# the columns of each statistic that the model states bit for bit, and its integer counts
FLOAT_COLS = {"fst": ("sum_a", "sum_b", "fst"), "het": ("het",), "dxy": ("dxy",), "fused": ("sum_a", "sum_b", "fst", "het", "dxy")}
INT_COLS = {"fst": (), "het": ("nhet", "nonmissing"), "dxy": ("neffective", "nskip"),
            "fused": ("nhet", "nonmissing", "neffective", "nskip")}


# ----------------------------------------------------------------------------- geometry (pgt_geom.h, pgt_plan.cpp)

class Geom:
    """pgt_make_geom"""

    def __init__(self, W, S, u):
        u = u or 256
        self.W, self.S, self.u = W, S, u
        self.r, self.q = W % S, W // S
        self.upa = (self.r + u - 1) // u
        self.upb = (S - self.r + u - 1) // u
        self.upp = self.upa + self.upb
        self.wunits = self.q * self.upp + self.upa
        self.ueff = min(max(self.r, S - self.r), u)
        need, gw = (self.ueff + 7) // 8, 1
        while gw < need and gw < 32:
            gw <<= 1
        self.gw = gw

    def unit_range(self, N, j):
        """pgt_unit_range, vectorised over segment-local unit indices j: (start, length) segment-local."""
        j = np.asarray(j, np.int64)
        k, s = j // self.upp, j % self.upp
        in_a = s < self.upa
        st = np.where(in_a, k * self.S + s * self.u, k * self.S + self.r + (s - self.upa) * self.u)
        bound = np.where(in_a, k * self.S + self.r, (k + 1) * self.S)
        en = np.minimum(np.minimum(st + self.u, bound), N)
        return st, np.maximum(en - st, 0)

    def seg_nunits(self, N):
        if N == 0:
            return 0
        x = N - 1
        k, off = x // self.S, x % self.S
        s = off // self.u if off < self.r else self.upa + (off - self.r) // self.u
        return k * self.upp + s + 1


def segments(offsets, W, S, bp):
    """pgt_plan_create's segment loop: list of dicts (site_base, nsites, nfull, nwin, nunits, win_base, unit_base)."""
    off = [int(x) for x in offsets]
    nc = len(off) - 1
    last = nc
    for c in range(nc - 1, -1, -1):
        if off[c + 1] > off[c]:
            last = c
            break
    segs, N, base, nwin = [], 0, off[0], 0
    for c in range(nc):
        ln = off[c + 1] - off[c]
        if ln == 0:
            continue
        N += ln
        eof = c == last
        if not eof and ((N >= W and (N - W) % S == 0) or (bp and N <= W - S)):
            continue
        nfull = (N - W) // S + 1 if N >= W else 0
        partial = N < W or (N - W) % S != 0
        drop = (eof or bp) and N - nfull * S <= W - S
        segs.append(dict(site_base=base, nsites=N, nfull=nfull, nwin=nfull + (1 if partial and not drop else 0), win_base=nwin))
        nwin += segs[-1]["nwin"]
        base += N
        N = 0
    return segs


class Layout:
    """The plan's geometry, ported and checked against the library's plan (`plan`: WindowPlan built with `unit_sites`)."""

    def __init__(self, plan, unit_sites=0, check=True):
        self.plan = plan
        self.bp = plan.mode == _cabi.PGT_MODE_BP
        self.g = Geom(plan.winsize, plan.stepsize, unit_sites)
        self.segs = segments(plan.offsets, plan.winsize, plan.stepsize, self.bp)
        self.origin = int(plan.offsets[0])
        ub = 0
        for s in self.segs:
            s["nunits"] = self.g.seg_nunits(s["nsites"])
            s["unit_base"] = ub
            ub += s["nunits"]
        self.nunits = ub
        self.nwin = sum(s["nwin"] for s in self.segs)
        g = self.g
        # per unit: segment index, segment-local index, global start (site or bp entry), length
        seg_of_unit = np.repeat(np.arange(len(self.segs)), [s["nunits"] for s in self.segs])
        self.unit_seg = seg_of_unit
        self.unit_local = np.arange(self.nunits, dtype=np.int64) - np.array([s["unit_base"] for s in self.segs], np.int64)[seg_of_unit] \
            if self.nunits else np.zeros(0, np.int64)
        st = np.zeros(self.nunits, np.int64)
        ln = np.zeros(self.nunits, np.int64)
        for i, s in enumerate(self.segs):
            a, b = s["unit_base"], s["unit_base"] + s["nunits"]
            st[a:b], ln[a:b] = g.unit_range(s["nsites"], self.unit_local[a:b])
            st[a:b] += s["site_base"]
        self.unit_start, self.unit_len = st, ln
        # per window: segment, segment-local k, first / last site (entry), first unit, unit count
        wseg = np.repeat(np.arange(len(self.segs)), [s["nwin"] for s in self.segs])
        k = np.arange(self.nwin, dtype=np.int64) - np.array([s["win_base"] for s in self.segs], np.int64)[wseg] if self.nwin else np.zeros(0, np.int64)
        sb = np.array([s["site_base"] for s in self.segs], np.int64)[wseg] if self.nwin else np.zeros(0, np.int64)
        N = np.array([s["nsites"] for s in self.segs], np.int64)[wseg] if self.nwin else np.zeros(0, np.int64)
        nfull = np.array([s["nfull"] for s in self.segs], np.int64)[wseg] if self.nwin else np.zeros(0, np.int64)
        nun = np.array([s["nunits"] for s in self.segs], np.int64)[wseg] if self.nwin else np.zeros(0, np.int64)
        ubase = np.array([s["unit_base"] for s in self.segs], np.int64)[wseg] if self.nwin else np.zeros(0, np.int64)
        self.win_seg, self.win_k = wseg, k
        self.win_first = sb + k * g.S
        self.win_nsites = np.minimum(N - k * g.S, g.W)
        self.win_fu_local = k * g.upp
        self.win_cnt = np.where(k < nfull, g.wunits, nun - k * g.upp)  # pgt_window_units
        self.win_fu = ubase + self.win_fu_local
        self.win_seg_nunits = nun
        if check:
            self.check_against_plan()

    def check_against_plan(self):
        p, g = self.plan, self.g
        assert p.num_segments == len(self.segs), ("segments", p.num_segments, len(self.segs))
        assert p.num_windows == self.nwin and p.num_units == self.nunits, ("windows / units", p.num_windows, self.nwin, p.num_units, self.nunits)
        first, last, _ = p.windows()
        assert np.array_equal(first.astype(np.int64), self.win_first), "window first sites"
        assert np.array_equal(last.astype(np.int64), self.win_first + self.win_nsites - 1), "window last sites"
        # the plan's own unit and window-unit answers on a sample (every one when there are few)
        rng = np.random.default_rng(0)
        ws = np.unique(np.concatenate([np.arange(min(self.nwin, 512)), rng.integers(0, max(self.nwin, 1), 512),
                                       [max(self.nwin - 1, 0)]])) if self.nwin else []
        for w in ws:
            assert p.window_units(int(w)) == (int(self.win_fu[w]), int(self.win_cnt[w])), ("window_units", int(w))
        us = np.unique(np.concatenate([np.arange(min(self.nunits, 512)), rng.integers(0, max(self.nunits, 1), 512),
                                       [max(self.nunits - 1, 0)]])) if self.nunits else []
        for j in us:
            assert p.unit(int(j)) == (int(self.unit_start[j]), int(self.unit_len[j])), ("unit", int(j))
        # units tile every segment, hence every window, with no gap and no overlap
        assert np.all(self.unit_len >= 1), "empty unit"
        same = self.unit_seg[1:] == self.unit_seg[:-1]
        assert np.array_equal((self.unit_start[:-1] + self.unit_len[:-1])[same], self.unit_start[1:][same]), "units leave a gap or overlap"
        if self.nwin:
            lu = self.win_fu + self.win_cnt - 1
            assert np.all(self.win_cnt >= 1) and np.all(self.unit_seg[self.win_fu] == self.win_seg) and np.all(self.unit_seg[lu] == self.win_seg), \
                "a window's units leave its segment"
            assert np.array_equal(self.unit_start[self.win_fu], self.win_first), "a window does not start at its first unit"
            assert np.array_equal(self.unit_start[lu] + self.unit_len[lu], self.win_first + self.win_nsites), "a window does not end at its last unit"

    # ------------------------------------------------------------------ unit -> column element ranges
    def unit_sites(self, pos=None, site_offsets=None):
        """[lo, hi) column element ranges of every unit's sites.  Site mode: the unit itself.  bp mode: the lower bounds
        of the unit's first bp and of the next unit's first bp in `pos` (k_bp_bounds)."""
        if not self.bp:
            lo = self.unit_start - self.origin
            return lo, lo + self.unit_len
        off = np.asarray(self.plan.offsets, np.int64)
        soff = np.asarray(site_offsets, np.int64)
        pos = np.asarray(pos)
        e = self.unit_start
        c = np.searchsorted(off, e, side="right") - 1
        bounds = np.empty(self.nunits + 1, np.int64)
        for ci in np.unique(c):
            sel = c == ci
            p = (e[sel] - off[ci] + 1).astype(np.int64)
            bounds[:-1][sel] = soff[ci] + np.searchsorted(pos[soff[ci]:soff[ci + 1]].astype(np.int64), p, side="left")
        bounds[-1] = soff[-1]
        return bounds[:-1], bounds[1:]

    def window_sites(self, pos=None, site_offsets=None):
        """[lo, hi) column element ranges of every window's sites (its units')."""
        lo, hi = self.unit_sites(pos, site_offsets)
        lu = self.win_fu + self.win_cnt - 1
        return lo[self.win_fu], hi[lu]

    # ------------------------------------------------------------------ level-2 order
    def hgw(self, level2=0):
        """Does level 2 run in scan mode (make_layout)?  level2 = the pgt_tune knob."""
        g = self.g
        if level2 == 1:
            return False
        if level2 == 2 and g.wunits >= 2:
            return True
        direct = sum(s["nfull"] * g.wunits + (s["nunits"] - s["nfull"] * g.upp if s["nwin"] > s["nfull"] else 0) for s in self.segs)
        scan = 4.0 * (3.0 * sum((s["nunits"] + g.wunits - 1) // g.wunits * g.wunits for s in self.segs) + 2.0 * self.nwin)
        return g.wunits > 32 and float(direct) > scan


# ----------------------------------------------------------------------------- per-site values (pgt_kernels_common.cuh)

def site_channels(stat, cols, minind):
    """Per-site double channels (what a lane's fold adds: +0.0 where the fold adds nothing -- a partial is never -0.0,
    so that is the identity) and integer channels of `stat`."""
    d, i = {}, {}
    if stat in ("fst", "fused"):
        d["sum_a"], d["sum_b"] = np.asarray(cols["a"], F64), np.asarray(cols["b"], F64)
    if stat in ("dxy", "fused"):
        f1, f2 = np.asarray(cols["f1"], F64), np.asarray(cols["f2"], F64)
        with np.errstate(all="ignore"):
            v = f1 * (1.0 - f2) + f2 * (1.0 - f1)  # dxy_site_value: separate IEEE products and sums, no FMA
        v = np.where((np.asarray(cols["n1"]) >= minind) & (np.asarray(cols["n2"]) >= minind), v, -9.0)
        with np.errstate(invalid="ignore"):
            add = v >= 0.0
        d["dxy"] = np.where(add, v, 0.0)
        i["neffective"], i["nskip"] = add.astype(np.int64), (v == -9.0).astype(np.int64)
    if stat in ("het", "fused"):
        gt = np.asarray(cols["geno"], np.int8).astype(np.int64)
        i["nonmissing"], i["nhet"] = (gt >= 0).astype(np.int64), (gt == 1).astype(np.int64)
    return d, i


def _leaf(x):
    """A fold from Stat::zero(): +0.0 + x."""
    return F64(0.0) + x


# ----------------------------------------------------------------------------- level 1 (pgt_level1.cuh)

def unit_partials(x, lo, hi, G):
    """k_units (:22-52; G = 32), the tiled consumer (:410-418): lane g of a group of G adds sites g, g+G, ... of the
    unit from +0.0 in that order, then the group butterfly with m = G/2 ... 1.  x: one channel, lo / hi: unit ranges."""
    n = len(lo)
    ln = hi - lo
    rounds = int((ln.max() + G - 1) // G) if n else 0
    acc = np.zeros((n, G), F64)
    lane = np.arange(G, dtype=np.int64)
    for r in range(rounds):
        off = r * G + lane[None, :]
        ok = off < ln[:, None]
        idx = np.where(ok, lo[:, None] + off, 0)
        acc = acc + np.where(ok, x[idx] if len(x) else 0.0, 0.0)
    return butterfly(acc)


def butterfly(v):
    """xor butterfly over the last axis (length a power of two), m = n/2 ... 1: lane 0's value."""
    while v.shape[-1] > 1:
        h = v.shape[-1] // 2
        v = v[..., :h] + v[..., h:]
    return v[..., 0]


# ----------------------------------------------------------------------------- level 2 (pgt_level2.cuh)

def windows_tree(units, fu, cnt):
    """k_windows: lane l adds unit partials l, l+32, ... from +0.0, then the 5-level butterfly (k_windows_small
    evaluates the same tree depth-first)."""
    n = len(fu)
    rounds = int((cnt.max() + 31) // 32) if n else 0
    acc = np.zeros((n, 32), F64)
    lane = np.arange(32, dtype=np.int64)
    for r in range(rounds):
        off = r * 32 + lane[None, :]
        ok = off < cnt[:, None]
        acc = acc + np.where(ok, units[np.where(ok, fu[:, None] + off, 0)], 0.0)
    return butterfly(acc)


def _cta_scan(items, nthreads=256):
    """cta_scan_dir over rows of `items` (blocks x n, in scan order; +0.0 padding after the block's items): chunks of
    256; per chunk a Kogge-Stone scan inside each warp (earlier item on the left), then carry + the warp totals in
    warp order + v; the carry of the next chunk is the chunk's last inclusive value."""
    nb, n = items.shape
    nch = (n + nthreads - 1) // nthreads
    v_all = np.zeros((nb, nch * nthreads), F64)
    v_all[:, :n] = _leaf(items)
    out = np.empty_like(v_all)
    carry = np.zeros(nb, F64)
    nw = nthreads // 32
    for c in range(nch):
        v = v_all[:, c * nthreads:(c + 1) * nthreads].reshape(nb, nw, 32).copy()
        d = 1
        while d < 32:
            t = v.copy()
            t[:, :, d:] = v[:, :, :-d] + v[:, :, d:]
            v = t
            d <<= 1
        wtot = v[:, :, 31]
        pre_base = np.empty((nb, nw), F64)
        run = carry.copy()
        for w in range(nw):
            pre_base[:, w] = run
            run = run + wtot[:, w]
        pre = pre_base[:, :, None] + v
        out[:, c * nthreads:(c + 1) * nthreads] = pre.reshape(nb, nthreads)
        carry = pre[:, -1, -1]
    return out[:, :n]


def windows_scan(L, units, blocks_check=True):
    """Scan mode (k_block_scan + k_windows_hgw, pgt_level2.cuh:546-650): blocks of B = wunits units from every segment's
    first unit, PRE / SUF by _cta_scan; window = SUF[first] + PRE[last] over two blocks; inside one block PRE[last] when
    it starts the block, else SUF[first] -- which needs the window to run to the block's or the segment's end."""
    g = L.g
    B = g.wunits
    pre = np.empty(L.nunits, F64)
    suf = np.empty(L.nunits, F64)
    # blocks of all segments, padded to B items
    starts, lens = [], []
    for s in L.segs:
        for b0 in range(0, s["nunits"], B):
            starts.append(s["unit_base"] + b0)
            lens.append(min(B, s["nunits"] - b0))
    starts, lens = np.array(starts, np.int64), np.array(lens, np.int64)
    if len(starts):
        off = np.arange(B, dtype=np.int64)[None, :]
        ok = off < lens[:, None]
        fwd = np.where(ok, units[np.where(ok, starts[:, None] + off, 0)], 0.0)
        bwd_idx = starts[:, None] + lens[:, None] - 1 - off
        bwd = np.where(ok, units[np.where(ok, bwd_idx, 0)], 0.0)
        P, Sf = _cta_scan(fwd), _cta_scan(bwd)
        pre[(starts[:, None] + off)[ok]] = P[ok]
        suf[bwd_idx[ok]] = Sf[ok]
    fu, lu = L.win_fu_local, L.win_fu_local + L.win_cnt - 1
    gf, gl = L.win_fu, L.win_fu + L.win_cnt - 1
    one = fu // B == lu // B
    if blocks_check:
        runs_out = (lu == (lu // B + 1) * B - 1) | (lu == L.win_seg_nunits - 1)
        bad = np.nonzero(one & (fu % B != 0) & ~runs_out)[0]
        assert len(bad) == 0, f"scan mode: one-block windows {bad[:5]} neither start their block nor run to its end"
    return np.where(one, _leaf(np.where(fu % B == 0, pre[gl], suf[gf])), _leaf(suf[gf]) + pre[gl])


# ----------------------------------------------------------------------------- sliding tile (pgt_slide.cuh)

SLIDE_WARPS, SLIDE_MAX_E = 7, 6


def slide_team(W):
    """slide_team (pgt_slide.cuh:48): (E, wpb, G) with the most sites per step, the smaller E on ties."""
    best = (1, SLIDE_WARPS, 0)
    wp = (W + 31) // 32 * 32
    for E in range(1, SLIDE_MAX_E + 1):
        tpb = (W + E - 1) // E
        wpb = (tpb + 31) // 32
        if wpb > SLIDE_WARPS:
            continue
        G = max(1, min(SLIDE_WARPS // wpb, 1024 // wp))
        if G > best[2]:
            best = (E, wpb, G)
    return best


def slide_blocks(x, nblk, W, E, wpb):
    """PRE and SUF (nblk x W) of blocks of W sites given as x (nblk x W, +0.0 beyond the segment): thread q owns
    elements [qE, (q+1)E); its forward total; up / down Kogge-Stone warp scans; the team's warp totals -- those
    before in order, those after last first; PRE runs forward from (warps before + lanes before), SUF backward
    from (warps after + lanes after)."""
    nt = wpb * 32
    leaf = np.zeros((nblk, nt * E), F64)
    leaf[:, :W] = _leaf(x)
    leaf = leaf.reshape(nblk, wpb, 32, E)
    valid = (np.arange(nt * E) < W).reshape(wpb, 32, E)
    tot = np.zeros((nblk, wpb, 32), F64)
    for e in range(E):
        tot = tot + leaf[..., e]
    up, dn = tot.copy(), tot.copy()
    d = 1
    while d < 32:
        u2, d2 = up.copy(), dn.copy()
        u2[..., d:] = up[..., :-d] + up[..., d:]
        d2[..., :-d] = dn[..., d:] + dn[..., :-d]
        up, dn = u2, d2
        d <<= 1
    wt = up[..., 31]  # (nblk, wpb)
    bpre = np.zeros((nblk, wpb), F64)
    run = np.zeros(nblk, F64)
    for w in range(wpb):
        bpre[:, w] = run
        run = run + wt[:, w]
    bsuf = np.zeros((nblk, wpb), F64)
    run = np.zeros(nblk, F64)
    for w in range(wpb - 1, -1, -1):
        bsuf[:, w] = run
        run = run + wt[:, w]
    xu = np.zeros_like(up)
    xu[..., 1:] = up[..., :-1]
    xd = np.zeros_like(dn)
    xd[..., :-1] = dn[..., 1:]
    bp = bpre[..., None] + xu
    bs = bsuf[..., None] + xd
    PRE = np.zeros((nblk, wpb, 32, E), F64)
    SUF = np.zeros((nblk, wpb, 32, E), F64)
    for e in range(E):
        bp = np.where(valid[..., e], bp + leaf[..., e], bp)
        PRE[..., e] = bp
    for e in range(E - 1, -1, -1):
        bs = np.where(valid[..., e], bs + leaf[..., e], bs)
        SUF[..., e] = bs
    return PRE.reshape(nblk, nt * E)[:, :W], SUF.reshape(nblk, nt * E)[:, :W]


def windows_slide(L, x):
    """k_slide / k_slide_fused2: window k of a segment (first site f = kS, last l) = SUF_m[f mod W]
    (+ PRE_{m+1}[l mod W] when l lies in block m + 1), blocks of W sites from the segment origin."""
    g = L.g
    W = g.W
    E, wpb, _ = slide_team(W)
    out = np.empty(L.nwin, F64)
    for si, s in enumerate(L.segs):
        if s["nwin"] == 0:
            continue
        N = s["nsites"]
        nblk = (N + W - 1) // W
        base = s["site_base"] - L.origin
        xs = np.zeros(nblk * W, F64)
        xs[:N] = x[base:base + N]
        PRE, SUF = slide_blocks(xs.reshape(nblk, W), nblk, W, E, wpb)
        k = np.arange(s["nwin"], dtype=np.int64)
        f = k * g.S
        l = np.minimum(f + W - 1, N - 1)
        m = f // W
        acc = SUF[m, f % W]
        two = l // W == m + 1
        acc = np.where(two, acc + PRE[np.minimum(m + 1, nblk - 1), l % W], acc)
        out[s["win_base"]:s["win_base"] + s["nwin"]] = acc
    return out


# ----------------------------------------------------------------------------- the window table

def epilogue(stat, sums, counts):
    """Stat::emit: fst = Σb != 0 ? Σa / Σb : 0; het = nonmissing > 1 ? nhet / nonmissing : (nonmissing ? nhet : 0)."""
    out = dict(sums)
    if "sum_a" in sums:
        a, b = sums["sum_a"], sums["sum_b"]
        with np.errstate(all="ignore"):
            out["fst"] = np.where(b != 0.0, a / np.where(b != 0.0, b, 1.0), 0.0)
    if "nhet" in counts:
        nh, nm = counts["nhet"].astype(F64), counts["nonmissing"]
        with np.errstate(all="ignore"):
            out["het"] = np.where(nm > 1, nh / np.maximum(nm, 1).astype(F64), np.where(nm > 0, nh, 0.0))
    return out


def path_of(plan, stat_id, level2=0, unit_sites=0):
    """'tree' | 'scan' | 'slide' | 'persite': the order a scan of `stat_id` over `plan` takes under the current pgt_tune
    knobs (level2: the knob's value, which the model cannot read back)."""
    p = plan.scan_path(stat_id)
    if p != "units":
        return p
    return "scan" if Layout(plan, unit_sites, check=False).hgw(level2) else "tree"


def window_table(plan, stat, cols, path, minind=1, site_offsets=None, unit_sites=0, layout=None):
    """The columns the kernels produce for `stat` ('fst' | 'het' | 'dxy' | 'fused') over `plan`: the float sums and
    ratios bit for bit, and the integer counts.  path: 'tree' (level 1 + k_windows / k_windows_small), 'scan'
    (level 1 + scan mode), 'slide' (sliding tile), 'persite' (W = S = 1 map)."""
    with np.errstate(all="ignore"):  # Inf and NaN are values like any other here
        return _window_table(plan, stat, cols, path, minind, site_offsets, layout or Layout(plan, unit_sites))


def _window_table(plan, stat, cols, path, minind, site_offsets, L):
    d, ic = site_channels(stat, cols, minind)
    wlo, whi = L.window_sites(cols.get("pos"), site_offsets)
    counts = {}
    for k, v in ic.items():
        cs = np.concatenate([[0], np.cumsum(v)])
        counts[k] = (cs[whi] - cs[wlo]).astype(np.uint32)
    sums = {}
    if path in ("tree", "scan"):
        ulo, uhi = L.unit_sites(cols.get("pos"), site_offsets)
        for k, x in d.items():
            units = unit_partials(x, ulo, uhi, L.g.gw)
            sums[k] = windows_tree(units, L.win_fu, L.win_cnt) if path == "tree" else windows_scan(L, units)
    elif path == "slide":
        assert not L.bp
        for k, x in d.items():
            sums[k] = windows_slide(L, x)
    elif path == "persite":
        assert not L.bp and L.g.W == 1 and L.g.S == 1
        for k, x in d.items():
            sums[k] = _leaf(x[L.win_first - L.origin])
    else:
        raise ValueError(path)
    out = epilogue(stat, sums, counts)
    out.update(counts)
    return out


def depth(L, path):
    """An upper bound on the additions between a site and its window value on `path`, for the bound
    |model - exact| <= γ_d Σ|x|, γ_d = d u / (1 - d u)."""
    g = L.g
    unit = -(-g.ueff // g.gw) + g.gw.bit_length() - 1  # a lane's chain, then the group butterfly
    if path == "tree":
        return unit + 1 + -(-g.wunits // 32) + 5
    if path == "scan":  # leaf, warp scan, warp totals, the carry through every chunk, SUF + PRE
        return unit + 1 + 5 + 8 * (-(-g.wunits // 256) + 1) + 2
    if path == "slide":  # per side: leaf, thread total, warp scan, team warps, lanes before / after, PRE / SUF run
        E, wpb, _ = slide_team(g.W)
        return 2 * (1 + E + 5 + wpb + 1 + E) + 1
    return 1


def exact_sums(x, lo, hi):
    """math.fsum of x over each [lo, hi): the exactly rounded window sums."""
    import math
    return np.array([math.fsum(x[a:b]) for a, b in zip(lo, hi)], F64)

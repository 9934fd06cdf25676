"""Kernel time of the extreme-score scan over window plans (pgt_scan_plan_extreme), next to pgt_scan_extreme over 100 kb
windows of the same sites; and (--ab) the existing statistics of this library against another build, alternated.
One JSON line per point on stdout, the device name and power limit first.

usage: python tools/probe_plan_extreme.py [--reps 10] [--pkg DIR]
       python tools/probe_plan_extreme.py --ab DIR [--rounds 3]   (DIR holds another popgenomicstools_b200 package, built)

Time: CUDA events around a device-mode scan of the bound plan (every kernel of the scan), median of `reps` after two
warm-up scans; level-1 / level-2 kernel time from pgt_profile over the same scans.  Bytes (algorithmic): 8 B of score
per site, +4 B of position in bp mode; 36 B of extreme fields per window, +16 B of geometry (label, start, end, mid).
frac = bytes / time / the measured 6533.2 GB/s copy peak of one B200.  Inputs are far larger than L2 except where noted
by their size."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PEAK_GBS = 6533.2


def header(torch, lib_path):
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps(dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi[:1], lib=lib_path)), flush=True)


def timed(torch, run, reps):
    for _ in range(2):
        out = run()
    torch.cuda.synchronize()
    del out
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = run()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
        del out
    return float(np.median(ms)), float(min(ms)), float(max(ms))


def point(torch, pgt, what, run, reps, nbytes, profile_read, **kv):
    pgt.profile(True)
    med, lo, hi = timed(torch, run, reps)
    pgt.profile(False)
    p = profile_read()
    n = reps + 2
    print(json.dumps(dict(what=what, **kv, ms=round(med, 3), ms_min=round(lo, 3), ms_max=round(hi, 3),
                          level1_ms=round(p["units_ms"] / n, 3), level2_ms=round(p["windows_ms"] / n, 3),
                          gbytes=round(nbytes / 1e9, 3), gbs=round(nbytes / med / 1e6, 1), frac=round(nbytes / med / 1e6 / PEAK_GBS, 3))),
          flush=True)


def probe_extreme(pkg, reps):
    import torch
    sys.path.insert(0, pkg)
    import popgenomicstools_b200 as pgt
    from popgenomicstools_b200 import _cabi
    from popgenomicstools_b200.workloads import human_like_contigs
    header(torch, _cabi.LIB_PATH)
    IHS = _cabi.PGT_XSTAT_IHS
    row = 36 + 16
    # site mode, 1e9 sites
    n = 1_000_000_000
    _, soff = human_like_contigs(n, 10000)
    score = pgt.synth_score(7, 0, n)
    pos = pgt.synth_pos(7, 0, n, soff, 1)
    # (unit_sites 2048: the same windows reduced from units of 2048 sites instead of the plan's default -- how much of
    # level 1 is paid per unit)
    for W, S, unit in ((50000, 10000, 0), (50000, 10000, 2048), (500, 100, 0)):
        plan = pgt.WindowPlan(soff, W, S, unit_sites=unit)
        point(torch, pgt, "plan_extreme", lambda: pgt.ihs_window(plan, pos, score, 2.0), reps, n * 8 + plan.num_windows * row,
              pgt.profile_read, mode="sites", sites=n, W=W, S=S, unit_sites=unit, units=plan.num_units, windows=plan.num_windows)
        del plan
    # the yardstick: ihsWindow's own 100 kb windows over the same sites (one site per bp)
    xplan = pgt.ExtremePlan(pos.cpu().numpy(), soff, 100000)
    point(torch, pgt, "scan_extreme", lambda: pgt.ihs_window(xplan, pos, score, 2.0), reps, n * 8 + xplan.num_windows * 36,
          pgt.profile_read_extreme, mode="xplan", sites=n, W=100000, windows=xplan.num_windows)
    del xplan
    # bp 100000/10000: dense (every bp a site: the same 1e9 sites) and sparse (1e8 sites, one per ~30 bp)
    nsites = np.diff(soff).astype(np.int64)
    for layout, m, density in (("dense", n, 1), ("sparse", 100_000_000, 30)):
        if layout == "sparse":
            del score, pos
            torch.cuda.empty_cache()
            _, soff = human_like_contigs(m, 10000)
            nsites = np.diff(soff).astype(np.int64)
            score = pgt.synth_score(8, 0, m)
            pos = pgt.synth_pos(8, 0, m, soff, density)
        boff = np.concatenate([[0], np.cumsum(nsites * density + 17)]).astype(np.uint64)
        plan = pgt.WindowPlan(boff, 100000, 10000, mode="bp", unit_sites=0 if density == 1 else 4096)
        point(torch, pgt, "plan_extreme", lambda: pgt.ihs_window(plan, pos, score, 2.0, site_offsets=soff), reps,
              m * 12 + plan.num_windows * row, pgt.profile_read, mode="bp", layout=layout, sites=m, bp=int(boff[-1]), W=100000, S=10000,
              windows=plan.num_windows)
        del plan
    # 1e8 sites: W = S = 1 (per-site map) and 1000/1 (scan mode)
    score, pos = score[:m], pos[:m]
    for W, S in ((1, 1), (1000, 1)):
        plan = pgt.WindowPlan(soff, W, S)
        point(torch, pgt, "plan_extreme", lambda: pgt.ihs_window(plan, pos, score, 2.0), reps, m * 8 + plan.num_windows * row,
              pgt.profile_read, mode="sites", sites=m, W=W, S=S, windows=plan.num_windows)
        del plan


def probe_existing(pkg, reps):
    """The existing statistics with the package under `pkg` (this tree, or another build for --ab)."""
    import torch
    sys.path.insert(0, pkg)
    import popgenomicstools_b200 as pgt
    from popgenomicstools_b200 import _cabi
    from popgenomicstools_b200.workloads import human_like_contigs
    n = 1_000_000_000
    _, soff = human_like_contigs(n, 10000)
    a, b = pgt.synth_fst(4, 0, n)
    plan = pgt.WindowPlan(soff, 50000, 10000, unit_sites=512)
    point(torch, pgt, "fst", lambda: pgt.fst_window(plan, None, a, b), reps, n * 16, pgt.profile_read, lib=pkg, W=50000, S=10000, sites=n)
    del a, b, plan
    torch.cuda.empty_cache()
    m = 100_000_000
    _, soff = human_like_contigs(m, 100)
    a, b = pgt.synth_fst(5, 0, m)
    g = pgt.synth_het(5, 0, m)
    f1, f2, n1, n2 = pgt.synth_dxy(5, 0, m)
    pos = pgt.synth_pos(5, 0, m, soff, 1)
    for W, S in ((1000, 100), (1000, 1)):
        plan = pgt.WindowPlan(soff, W, S)
        point(torch, pgt, "fused", lambda: pgt.fused_window(plan, pos, a, b, g, f1, f2, n1, n2, minind=5), reps, m * 41, pgt.profile_read,
              lib=pkg, W=W, S=S, sites=m)
    plan = pgt.WindowPlan(soff, 1, 1)
    point(torch, pgt, "het", lambda: pgt.het_window(plan, pos, g), reps, m * 1, pgt.profile_read, lib=pkg, W=1, S=1, sites=m)
    point(torch, pgt, "dxy", lambda: pgt.dxy_window(plan, pos, f1, f2, n1, n2, minind=5), reps, m * 24, pgt.profile_read, lib=pkg, W=1,
          S=1, sites=m)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--ab", default=None, help="directory of another build: time the existing statistics, alternating")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--pkg", default=ROOT, help="directory holding the popgenomicstools_b200 package to probe (default: this tree)")
    ap.add_argument("--existing", default=None, help=argparse.SUPPRESS)  # one process of --ab
    args = ap.parse_args()
    if args.existing:
        probe_existing(args.existing, args.reps)
    elif args.ab:
        import torch
        header(torch, "ab")
        for r in range(args.rounds):
            for pkg in (os.path.abspath(args.ab), ROOT):
                subprocess.run([sys.executable, os.path.abspath(__file__), "--existing", pkg, "--reps", str(args.reps)], check=True)
    else:
        probe_extreme(os.path.abspath(args.pkg), args.reps)


if __name__ == "__main__":
    main()

"""Kernel time of fst, het, dxy and the fused scan over bp windows (PGT_MODE_BP plans), with site-mode fst over the same
sites for comparison.  One JSON line per point on stdout, plus the device name and power limit first.

usage: python tools/probe_bp_stats.py [--sites 1e9] [--reps 10] [--only dxy]

Layouts: "dense" = every bp a site; "sparse" = the same number of sites at about one per 30 bp (unit_sites 4096, the
dxyWindow CLI's choice for that density).  24 chromosomes of human-like proportions (popgenomicstools_b200.workloads).
Time: CUDA events around a device-mode scan of the bound plan (every kernel of the scan: bp unit bounds, level 1,
level 2, dxyWindow's global line), median of `reps` after two warm-up scans.  Bytes: the columns the statistic reads,
every site once (+4 B/site of positions in bp mode; site mode reads positions only at window edges), plus the window
rows written.  frac = bytes / time / the measured 6533.2 GB/s copy peak of one B200.  Inputs are far larger than L2.
Run it with PGT_LIB set to compare two builds of the library (e.g. dxy bp before and after a change: --only dxy)."""
import argparse
import json
import subprocess
import sys
import os

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import popgenomicstools_b200 as pgt  # noqa: E402
from popgenomicstools_b200 import _cabi  # noqa: E402
from popgenomicstools_b200.scan import _STAT_OUTS, _W_DTYPES  # noqa: E402
from popgenomicstools_b200.workloads import human_like_contigs  # noqa: E402

PEAK_GBS = 6533.2
STATS = {"fst": _cabi.PGT_STAT_FST, "het": _cabi.PGT_STAT_HET, "dxy": _cabi.PGT_STAT_DXY, "fused": _cabi.PGT_STAT_FUSED}
NAMES = {"fst": ("a", "b"), "het": ("geno",), "dxy": ("f1", "f2", "n1", "n2"), "fused": ("a", "b", "geno", "f1", "f2", "n1", "n2")}
COL_BYTES = {"pos": 4, "a": 8, "b": 8, "geno": 1, "f1": 8, "f2": 8, "n1": 4, "n2": 4}
GEOMS = [(50000, 10000), (1000, 100)]


def row_bytes(stat):
    return sum(np.dtype(_W_DTYPES[k]).itemsize for k in _STAT_OUTS[STATS[stat]] if k != "dxy_global")


def time_scan(plan, stat, cols, reps, **kw):
    def run():
        return pgt.scan(plan, STATS[stat], {k: cols[k] for k in ("pos",) + NAMES[stat]}, minind=5, **kw)
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=float, default=1e9)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--only", default=None, help="comma-separated statistics (fst, het, dxy, fused, fst_sites)")
    args = ap.parse_args()
    only = set(args.only.split(",")) if args.only else None
    want = lambda s: only is None or s in only
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps(dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi[:1], lib=os.path.basename(_cabi.LIB_PATH))), flush=True)
    n = int(args.sites)
    _, soff = human_like_contigs(n, 10000)
    nsites = np.diff(soff).astype(np.int64)
    cols = {}
    if want("fst") or want("fused") or want("fst_sites"):
        cols["a"], cols["b"] = pgt.synth_fst(7, 0, n)
    if want("het") or want("fused"):
        cols["geno"] = pgt.synth_het(7, 0, n)
    if want("dxy") or want("fused"):
        cols["f1"], cols["f2"], cols["n1"], cols["n2"] = pgt.synth_dxy(7, 0, n)
    for layout, density, unit in (("dense", 1, 0), ("sparse", 30, 4096)):
        cols["pos"] = pgt.synth_pos(7, 0, n, soff, density)
        chr_len = nsites * density + 17
        boff = np.concatenate([[0], np.cumsum(chr_len)]).astype(np.uint64)
        for W, S in GEOMS:
            plan = pgt.WindowPlan(boff, W, S, mode="bp", unit_sites=unit)
            for stat in ("dxy", "fst", "het", "fused"):
                if not want(stat):
                    continue
                med, lo, hi = time_scan(plan, stat, cols, args.reps, site_offsets=soff)
                nbytes = n * (4 + sum(COL_BYTES[c] for c in NAMES[stat])) + plan.num_windows * row_bytes(stat)
                print(json.dumps(dict(stat=stat, mode="bp", layout=layout, sites=n, bp=int(boff[-1]), W=W, S=S, unit=unit,
                                      windows=plan.num_windows, ms=round(med, 3), ms_min=round(lo, 3), ms_max=round(hi, 3),
                                      gbytes=round(nbytes / 1e9, 3), gbs=round(nbytes / med / 1e6, 1),
                                      frac=round(nbytes / med / 1e6 / PEAK_GBS, 3))), flush=True)
            del plan
            torch.cuda.empty_cache()
        if want("fst_sites") and layout == "dense":
            for W, S in GEOMS:
                plan = pgt.WindowPlan(soff, W, S)
                med, lo, hi = time_scan(plan, "fst", cols, args.reps)
                nbytes = n * 16 + plan.num_windows * row_bytes("fst")
                print(json.dumps(dict(stat="fst", mode="sites", layout="sites", sites=n, W=W, S=S, unit=0, windows=plan.num_windows,
                                      ms=round(med, 3), ms_min=round(lo, 3), ms_max=round(hi, 3), gbytes=round(nbytes / 1e9, 3),
                                      gbs=round(nbytes / med / 1e6, 1), frac=round(nbytes / med / 1e6 / PEAK_GBS, 3))), flush=True)
                del plan
                torch.cuda.empty_cache()


if __name__ == "__main__":
    main()

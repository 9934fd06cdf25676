#!/usr/bin/env python3
"""bench.py -- sites/sec of the fused window scan on 1..8 B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C4|C5] [--impl reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A step is one pass of the hot path (level-1 unit reduction + level-2 window combine) over the whole synthetic
genome, sharded by site range with a (W-S)-site halo (strong scaling: total work fixed).  There is no collective
on the data path and no gather: the window table lives once, in rank 0's HBM, and every rank's window kernel
writes its rows there directly (CUDA IPC mapping over NVLink, popgenomicstools_b200/sharding.py SharedTable).
Inputs are generated on the device by the counter-based generator and are resident in HBM when the timed region
starts; they are far larger than L2 (48 GB vs 126 MB), so no explicit flush is needed.

Prints ONE JSON line (rank 0).  `value` = total sites / max-over-ranks device time; `result_checksum` = an
order-sensitive checksum of the whole window table (identical for 1/2/4/8 GPUs: the summation order is a function
of (W, S, unit) only); `e2e` = the same scan through the C ABI with HOST (pinned) columns, H2D/D2H inside the timed
region -- at N > 1 ONE process (rank 0) drives all N GPUs through pgt_scan_sharded and ends with ONE table;
`roofline` = algorithmic bytes of the dominant kernel (level 1) / its mean CUDA-event duration over the timed
region, against MEASURED_PEAKS.json; `configs` = the other BASELINE.json configurations (C1, C2 sparse / dense, C3
per-site / 100 kb, C5 and its S = 1 stress variant), each sharded over the same N ranks: value, kernel time,
algorithmic bytes (columns in + window rows out, SURVEY 8d), fraction of the HBM peak and the table checksum;
`cpu_baseline` = the unmodified reference binary (oracle/_ref, g++ -O3) timed on this box's host cores on a
bounded text sample; its `compute_only` = the window arithmetic alone (oracle/pgt_oracle.c on pre-parsed arrays, one
core and all cores -- SURVEY 8d's second CPU figure: the reference itself cannot separate parsing from arithmetic).

--impl reference runs only that CPU arm (the reference's own implementation of the path); it never imports the
product package or loads libpgtscan.so.

--dump-outputs DIR writes the window table of the last timed step as .npy files (dump_outputs): the inputs come from
the seeded generator, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sites/sec for fused FST/dxy window scan at 1/2/4/8 B200; % of HBM peak"
UNIT = "sites/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4", choices=["C4", "C5"])
    ap.add_argument("--sites", type=float, default=0, help="override the workload's total site count (debug)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cli-large", action="store_true", help="skip the large-input legs of the drop-in fstWindow (N = 1 only)")
    ap.add_argument("--cli-large-cache-sites", type=float, default=6e8)
    ap.add_argument("--cli-large-text-sites", type=float, default=2.4e8)
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config legs (C1, C2, C3, C5, C5-S1)")
    ap.add_argument("--configs", default="", help="comma-separated subset of the per-config legs")
    ap.add_argument("--config-steps", type=int, default=5)
    ap.add_argument("--cpu-sample-sites", type=float, default=4.8e7)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the window table of the last one to DIR/<field>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the tables of the B200 scan (--impl b200)")
    return args


# ------------------------------------------------------------------------------ reference arm

def load_workloads():
    """workloads.py by path: the reference arm must not import the product package (its __init__ loads libpgtscan.so)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("pgt_workloads", os.path.join(ROOT, "popgenomicstools_b200", "workloads.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _write_contig(job):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    import numpy as np
    path, name, lo, hi, seed = job
    O.write_text("fst", path, [name], np.array([lo, hi], np.uint64), seed=seed, density=1)
    # write_text restarts local positions at 1 for the contig and hashes by global site index
    return path


def _run_ref(job):
    exe, path, W, S = job
    t0 = time.perf_counter()
    subprocess.run([exe, path, str(W), str(S)], stdout=subprocess.DEVNULL, check=True)
    return time.perf_counter() - t0


def cli_arm(tmp, jobs, W, S):
    """Our drop-in fstWindow on the same text, concatenated into one whole-genome file as a user
    would run it: text parsing (timed separately), scan through the C ABI, row formatting."""
    exe = os.path.join(ROOT, "popgenomicstools_b200", "bin", "fstWindow")
    if not os.access(exe, os.X_OK):
        return None
    allp = os.path.join(tmp, "all.fst")
    with open(allp, "wb") as w:
        for j in jobs:
            with open(j[0], "rb") as r:
                shutil.copyfileobj(r, w, 1 << 24)
    best, walls = None, []
    ours_out = os.path.join(tmp, "ours.tsv")
    for _ in range(3):  # best of three: CUDA start-up of a fresh process varies between 0.3 and 3.5 s on these boxes
        t0 = time.perf_counter()
        with open(ours_out, "wb") as fo:
            p = subprocess.run([exe, allp, str(W), str(S)], stdout=fo, stderr=subprocess.PIPE, text=True,
                               env=dict(os.environ, PGT_TIMING="1"))
        wall = time.perf_counter() - t0
        if p.returncode != 0:
            return {"error": p.stderr[-200:]}
        t = json.loads(p.stderr.strip().splitlines()[-1])
        t["wall_s_incl_process_and_cuda_startup"] = round(wall, 3)
        walls.append(round(wall, 3))
        if best is None or wall < best["wall_s_incl_process_and_cuda_startup"]:
            best = t
    best["walls_s_all_runs"] = walls
    best["sites_per_s_parse_scan_format"] = round(best["sites"] / (best["total_ms"] * 1e-3), 1)
    # the same input as a binary columnar cache (PGT_PACK, csrc/tools/pgt_colfile.h): no text parsing at all
    try:
        cache = os.path.join(tmp, "all.pgtc")
        t0 = time.perf_counter()
        subprocess.run([exe, allp, str(W), str(S)], check=True, env=dict(os.environ, PGT_PACK=cache))
        pack_s = time.perf_counter() - t0
        cache_out = os.path.join(tmp, "cache.tsv")
        ct, cwall = None, None
        for _ in range(3):
            t0 = time.perf_counter()
            with open(cache_out, "wb") as fo:
                p = subprocess.run([exe, cache, str(W), str(S)], stdout=fo, stderr=subprocess.PIPE, text=True,
                                   env=dict(os.environ, PGT_TIMING="1"), check=True)
            w1 = time.perf_counter() - t0
            if cwall is None or w1 < cwall:
                cwall, ct = w1, json.loads(p.stderr.strip().splitlines()[-1])
        best["columnar_cache"] = {"pack_s": round(pack_s, 3), "file_bytes": os.path.getsize(cache), "load_ms": ct["parse_ms"],
                                  "scan_ms": ct["scan_ms"], "format_ms": ct["format_ms"], "total_ms": ct["total_ms"],
                                  "wall_s_incl_process_and_cuda_startup": round(cwall, 3),
                                  "identical_stdout": open(cache_out, "rb").read() == open(ours_out, "rb").read()}
        os.remove(cache)
    except Exception as ex:
        best["columnar_cache"] = {"error": repr(ex)[:200]}
    # the same file through the unmodified reference binary, one process (how a user runs it), and a
    # row-by-row comparison of the two outputs (text after %g formatting)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    ref = O.ref_binary("fstWindow")
    if ref:
        ref_out = os.path.join(tmp, "ref.tsv")
        t0 = time.perf_counter()
        with open(ref_out, "wb") as fo:
            subprocess.run([ref, allp, str(W), str(S)], stdout=fo, check=True)
        rsec = time.perf_counter() - t0
        a, b = open(ours_out).read().splitlines(), open(ref_out).read().splitlines()
        diff = sum(1 for x, y in zip(a, b) if x != y) + abs(len(a) - len(b))
        best["reference_same_file_one_process"] = {"wall_s": round(rsec, 2), "sites_per_s": round(best["sites"] / rsec, 1),
                                                   "rows": len(b), "rows_differing_from_ours": diff}
    os.remove(allp)
    return best


def _port_contig(job):
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    lo, hi, seed, W, S = job
    a, b = O.synth_fst(seed, lo, hi - lo)
    pos = np.arange(1, hi - lo + 1, dtype=np.uint32)
    chr_id = np.zeros(hi - lo, np.uint32)
    best = None
    for _ in range(2):
        t0 = time.perf_counter()
        O.fst(chr_id, pos, a, b, W, S, count_only=True)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return best


def compute_only_port(offs, seed, W, S, nproc):
    """SURVEY 8(d) CPU timing (2): the window arithmetic alone -- oracle/pgt_oracle.c, the restatement of
    fstWindow.cpp:69-107 (re-sum of every window, no parsing, no printing) over pre-parsed arrays; one contig
    per process.  One core = the sum of the per-contig times; all cores = the contigs spread over nproc processes."""
    import multiprocessing as mp
    n = int(offs[-1])
    jobs = sorted(((int(offs[i]), int(offs[i + 1]), seed, W, S) for i in range(len(offs) - 1)), key=lambda j: j[0] - j[1])
    with mp.get_context("fork").Pool(nproc) as pool:
        t0 = time.perf_counter()
        secs = pool.map(_port_contig, jobs, chunksize=1)
        wall = time.perf_counter() - t0
    # greedy longest-first schedule of the measured compute times over nproc cores (generation excluded)
    load = [0.0] * nproc
    for t in secs:
        load[load.index(min(load))] += t
    return {"kind": "port", "what": "oracle/pgt_oracle.c window arithmetic only (pre-parsed arrays, no text, no output)",
            "sites": n, "one_core_sites_per_s": round(n / sum(secs), 1), "cores": nproc,
            "all_cores_sites_per_s": round(n / max(load), 1), "pool_wall_s_incl_generation": round(wall, 2)}


def reference_arm(wl, sample_sites, steps, warmup, with_cli=False):
    """Times the unmodified reference fstWindow (oracle/_ref, built from /root/reference with
    g++ -O3 -Wall) end to end -- text parsing is inseparable from its window arithmetic -- on a
    scaled twin of the workload: the same 24 contig-length ratios, one text file and one
    single-threaded reference process per contig, min(24, cores) processes at a time."""
    import multiprocessing as mp
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    human_like_contigs = load_workloads().human_like_contigs
    W, S = wl["winsize"], wl["stepsize"]
    exe = O.ref_binary("fstWindow")
    cores = os.cpu_count() or 1
    names, offs = human_like_contigs(int(sample_sites), S)
    n = int(offs[-1])
    if exe is None:
        # reference binary not built (oracle/_ref absent): time the oracle port, compute only
        import numpy as np
        a, b = O.synth_fst(wl["seed"], 0, n)
        pos = O.synth_pos(wl["seed"], offs, 1)
        chr_id = np.repeat(np.arange(24, dtype=np.uint32), np.diff(offs).astype(np.int64))
        times = []
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.fst(chr_id, pos, a, b, W, S, count_only=True)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
        sec = sum(times) / len(times)
        return dict(value=n / sec, unit=UNIT, cores=1, kind="port",
                    sample=f"oracle/pgt_oracle.c compute-only (pre-parsed arrays), {n} sites, 24 contigs, {W}/{S}"), sec
    tmp = tempfile.mkdtemp(prefix="pgt_ref_")
    try:
        O.build_oracle()
        jobs = [(os.path.join(tmp, f"{nm}.fst"), nm, int(offs[i]), int(offs[i + 1]), wl["seed"]) for i, nm in enumerate(names)]
        nproc = min(len(jobs), cores)
        with mp.get_context("fork").Pool(nproc) as pool:
            pool.map(_write_contig, jobs)
            rjobs = [(exe, j[0], W, S) for j in sorted(jobs, key=lambda j: j[2] - j[3])]  # longest first
            times = []
            for i in range(warmup + steps):
                t0 = time.perf_counter()
                pool.map(_run_ref, rjobs, chunksize=1)
                if i >= warmup:
                    times.append(time.perf_counter() - t0)
        sec = sum(times) / len(times)
        tb = sum(os.path.getsize(j[0]) for j in jobs)
        cli = cli_arm(tmp, jobs, W, S) if with_cli else None
        extra = {"our_cli_same_text": cli} if cli else {}
        if with_cli:
            try:
                extra["compute_only"] = compute_only_port(offs, wl["seed"], W, S, nproc)
            except Exception as ex:
                extra["compute_only"] = {"error": repr(ex)[:200]}
        return dict(value=n / sec, unit=UNIT, cores=nproc, kind="reference", **extra,
                    sample=(f"unmodified reference fstWindow (g++ -O3 -Wall) end to end incl. text parsing: scaled twin "
                            f"{n} sites / 24 contig files ({tb / 1e9:.2f} GB text), {W}/{S}, one process per contig, "
                            f"{nproc} at a time on {cores} host cores")), sec
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    WORKLOADS = load_workloads().WORKLOADS
    wl = WORKLOADS["C4"] if args.workload == "C5" else WORKLOADS[args.workload]  # the reference has no fused tool
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    # bound the whole run to a few minutes whatever K/W the driver passes
    per_step_budget = 240.0 / (steps + warmup)
    sample = min(args.cpu_sample_sites, max(2.4e6, per_step_budget * 1.0e7))
    cb, sec = reference_arm(wl, sample, steps, warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.workload]["desc"], "sample": cb["sample"]},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------ clocks

class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._h = None
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)  # NVML queries take milliseconds: keep them off the ranks' critical path

    def __enter__(self):
        if self._h is not None:
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._h is not None:
            self._t.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s), "window": "warm-up + timed steps (one contiguous load)"}


# ------------------------------------------------------------------------------ B200 arm

def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def recorded_traffic(workload, n_gpus):
    """dram bytes per level-1 launch from the committed ncu --set full capture, if it matches."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if n_gpus != 1 or not os.path.exists(p):
        return None
    try:
        return json.load(open(p)).get(workload, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


IN_BYTES = {"fst": 16, "het": 1, "dxy": 24, "fused": 41}     # compulsory column bytes per site (SURVEY 8d; pos at window edges only)
OUT_BYTES = {"fst": 44, "het": 36, "dxy": 32, "fused": 76}   # window row bytes the scan writes (label, positions, counts, statistics)
ACC_BYTES = {"fst": 16, "het": 8, "dxy": 16, "fused": 40}

# The other BASELINE.json configurations, run after the headline on the same ranks (short: a few steps each).
# `full`: every rank holds the whole (small) input and scans only its window range; otherwise its shard + halo.
CONFIGS = [
    dict(name="C1", stat="fst", n=1_000_000, contigs=1, W=50000, S=10000, seed=1, unit=0, full=True,
         desc="fstWindow, 1 Mb contig, 50 kb / 10 kb (configs[0])"),
    dict(name="C2-sparse", stat="dxy", n=1_000_000, contigs=1, W=20000, S=5000, seed=2, unit=0, full=True, bp=10,
         desc="dxyWindow bp mode, 10 Mb contig, 1 site per 10 bp, 20 kb / 5 kb (configs[1])"),
    dict(name="C2-dense", stat="dxy", n=10_000_000, contigs=1, W=20000, S=5000, seed=2, unit=0, full=True, bp=1,
         desc="dxyWindow bp mode, 10 Mb contig, every bp a site, 20 kb / 5 kb (configs[1])"),
    dict(name="C3-1/1", stat="het", n=100_000_000, contigs=1, W=1, S=1, seed=3, unit=0, full=True,
         desc="hetWindow, 100 Mb chromosome, single-site windows (configs[2]; output-bound: one row per site)"),
    dict(name="C3-100k", stat="het", n=100_000_000, contigs=1, W=100000, S=100000, seed=3, unit=4096, full=True,
         desc="hetWindow, 100 Mb chromosome, 100 kb windows (configs[2])"),
    dict(name="C5", stat="fused", n=3_000_000_000, contigs=24, W=1000, S=100, seed=5, unit=0, full=False,
         desc="fused fst+dxy+het, 3e9 sites / 24 contigs, 1000 / 100 (configs[4])"),
    dict(name="C5-S1", stat="fused", n=100_000_000, contigs=24, W=1000, S=1, seed=5, unit=0, full=True,
         desc="fused fst+dxy+het, 1e8-site subset, 1000 / 1: maximal overlap, sliding-tile path (configs[4] stress variant)"),
]


class Ranks:
    """torch.distributed plumbing of one bench process."""

    def __init__(self, torch, dist):
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device(f"cuda:{self.local}")
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, values, op="max"):
        t = self.torch.tensor([float(v) for v in values], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op={"max": self.dist.ReduceOp.MAX, "sum": self.dist.ReduceOp.SUM}[op])
        return [float(x) for x in t.tolist()]


def make_columns(pgt, stat, seed, s_lo, n_local, offs, dev, density=1):
    cols = dict(pos=pgt.synth_pos(seed, s_lo, n_local, offs, density, device=dev))
    if stat in ("fst", "fused"):
        cols["a"], cols["b"] = pgt.synth_fst(seed, s_lo, n_local, device=dev)
    if stat in ("het", "fused"):
        cols["geno"] = pgt.synth_het(seed, s_lo, n_local, device=dev)
    if stat in ("dxy", "fused"):
        cols["f1"], cols["f2"], cols["n1"], cols["n2"] = pgt.synth_dxy(seed, s_lo, n_local, device=dev)
    return cols


def local_units(plan, w_lo, w_hi):
    if w_hi <= w_lo:
        return 0
    fu0, _ = plan.window_units(w_lo)
    fu1, c1 = plan.window_units(w_hi - 1)
    return (plan.num_units if w_hi == plan.num_windows else fu1 + c1) - (0 if w_lo == 0 else fu0)


def run_config(cfg, R, pgt, steps, peak):
    """One BASELINE configuration on the ranks of this run: resident columns, window table in rank 0's HBM, a few
    warm-up and `steps` timed steps (CUDA events, max over ranks), per-kernel time from the library's own events."""
    import numpy as np
    torch, dist = R.torch, R.dist
    from popgenomicstools_b200 import _cabi
    from popgenomicstools_b200.scan import _STAT_OUTS
    from popgenomicstools_b200.sharding import SharedTable
    from popgenomicstools_b200.workloads import human_like_contigs
    stat_id = {"fst": _cabi.PGT_STAT_FST, "het": _cabi.PGT_STAT_HET, "dxy": _cabi.PGT_STAT_DXY, "fused": _cabi.PGT_STAT_FUSED}[cfg["stat"]]
    n, W, S = cfg["n"], cfg["W"], cfg["S"]
    free, _ = torch.cuda.mem_get_info()
    need = (IN_BYTES[cfg["stat"]] + 4) * (n if cfg["full"] else n // R.world) + OUT_BYTES[cfg["stat"]] * (n // S if R.rank == 0 else 0)
    f = R.reduce([1.0 if need * 1.08 + (4 << 30) > free else 0.0])[0]
    if f > 0:  # every rank takes the same decision
        return dict(name=cfg["name"], skipped=f"needs {need / 1e9:.0f} GB of HBM per GPU, {free / 1e9:.0f} GB free")
    if cfg["contigs"] == 1:
        offs = np.array([0, n], np.uint64)
    else:
        _, offs = human_like_contigs(n, S)
    extra, density = {}, cfg.get("bp", 0)
    if density:  # dxyWindow -fixedsite 0: windows on the bp axis of a chromosome of n * density bp
        plan = pgt.WindowPlan(np.array([0, n * density], np.uint64), W, S, mode="bp", unit_sites=cfg["unit"])
        extra = dict(site_offsets=offs)
    else:
        plan = pgt.WindowPlan(offs, W, S, unit_sites=cfg["unit"])
    w_lo, w_hi, s_lo, s_hi = plan.shard(R.rank, R.world)
    if cfg["full"] or density:
        s_lo, s_hi = 0, n
    cols = make_columns(pgt, cfg["stat"], cfg["seed"], s_lo, s_hi - s_lo, offs, R.dev, density or 1)
    tab = SharedTable(_STAT_OUTS[stat_id], plan.num_windows, R.rank, R.world, dist, torch, R.dev, w_lo=w_lo, w_hi=w_hi)
    out = tab.rows()
    kw = dict(minind=5, window_range=(w_lo, w_hi), site_origin=s_lo, out=out, **extra)
    try:
        for _ in range(3):
            pgt.scan(plan, stat_id, cols, **kw)
        R.barrier()
        pgt.profile(True)
        pgt.profile_read()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        R.barrier()
        e0.record()
        for _ in range(steps):
            pgt.scan(plan, stat_id, cols, **kw)
        e1.record()
        R.barrier()
        prof = pgt.profile_read()
        pgt.profile(False)
        ms_step = R.reduce([e0.elapsed_time(e1) / steps])[0]
        path = plan.scan_path(stat_id)
        nwin_l = w_hi - w_lo
        # sites this rank's scan reads: its windows' span (the halo is real work of the sharded run)
        fl = plan._lib
        import ctypes as C
        sites_l = 0
        if nwin_l:
            f0, l1 = C.c_uint64(), C.c_uint64()
            fl.pgt_plan_window(plan.handle, w_lo, C.byref(f0), None, None)
            fl.pgt_plan_window(plan.handle, w_hi - 1, None, C.byref(l1), None)
            sites_l = l1.value + 1 - f0.value
            if density:  # bp axis: the sites are those of the bp range; a shard reads its share of them
                sites_l = int(round(sites_l / density))
        in_b = IN_BYTES[cfg["stat"]] + (4 if density else 0)
        # positions: compulsory only where a window row prints them -- its first and its last site, so 8 B per window
        # and never more than the whole column (S = 1: every site starts a window); the bp axis streams them (in_b)
        pos_b = 0 if density else min(4 * sites_l, 8 * nwin_l)
        algo = in_b * sites_l + pos_b + OUT_BYTES[cfg["stat"]] * nwin_l
        k_ms = (prof["units_ms"] + prof["windows_ms"]) / steps
        ach = algo / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0
        tot = R.reduce([algo, ach, k_ms, prof["units_ms"] / steps, prof["windows_ms"] / steps, pos_b], "sum")
        res = dict(name=cfg["name"], desc=cfg["desc"], path=path, n_sites=n, windows=plan.num_windows, value=n / (ms_step * 1e-3),
                   unit=UNIT, ms_per_step=round(ms_step, 4), steps=steps,
                   kernel_ms=round(tot[2] / R.world, 4), level1_ms=round(tot[3] / R.world, 4), level2_ms=round(tot[4] / R.world, 4),
                   algorithmic_bytes=int(tot[0]), achieved_gbs=round(tot[1] / R.world, 1), frac=round(tot[1] / R.world / peak, 4),
                   bytes_per_site_in=in_b, bytes_per_window_out=OUT_BYTES[cfg["stat"]], window_edge_position_bytes=int(tot[5]))
        R.barrier()
        res["table"] = ("one table in rank 0's HBM, rows written in place by every rank" if tab.placement == "rank0"
                        else "sharded: every rank keeps its rows in its own HBM (table above 256 MB)")
        res["result_checksum"] = tab.checksum()
        return res
    finally:
        pgt.profile(False)
        del cols
        tab.close()
        torch.cuda.empty_cache()


DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this many bytes


def dump_outputs(out_dir, tab, R, glob=None, budget=DUMP_BYTES):
    """--dump-outputs: the window table the last timed step left, i.e. the arrays scan() hands its caller, one
    DIR/<field>.npy per field in float64 (exact for the uint32 fields too), DIR/window_index.npy with the global
    window index of each row and, for the fused scan, DIR/dxy_global.npy.  A table above `budget` bytes is written at
    a sample of rows drawn with a fixed seed: the same rows for the same arguments, so that two builds of the project
    can be compared output for output.  Collective when the table is sharded over the ranks."""
    import numpy as np
    torch = R.torch
    nwin = tab.nwin
    nrows = min(nwin, (budget - 4096) // (8 * (len(tab.fields) + 1)))  # 4 KB: .npy headers and dxy_global
    rows = np.arange(nwin) if nrows == nwin else np.sort(np.random.default_rng(0).choice(nwin, nrows, replace=False))
    lo, hi = (0, nwin) if tab.placement == "rank0" else (tab.w_lo, tab.w_hi)
    part = None
    if R.rank == 0 or tab.placement != "rank0":
        mine = rows[(rows >= lo) & (rows < hi)]
        idx = torch.as_tensor(mine - lo, device=R.dev)
        part = {"window_index": mine.astype(np.float64)}
        for k, a in tab.rows(lo, hi).items():
            if k == "dxy_global":
                continue
            t = torch.as_tensor(a, device=R.dev)
            if t.dtype == torch.float64:
                part[k] = t[idx].cpu().numpy()
            else:  # uint32: gathered through an int32 view of the same bits
                part[k] = t.view(torch.int32)[idx].cpu().numpy().view(np.uint32).astype(np.float64)
    if tab.placement != "rank0":
        parts = [None] * R.world if R.rank == 0 else None
        R.dist.gather_object(part, parts, dst=0)
        if R.rank == 0:
            part = {k: np.concatenate([p[k] for p in parts]) for k in part}
    if R.rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for k, v in part.items():
            np.save(os.path.join(out_dir, k + ".npy"), v)
        if glob is not None:
            np.save(os.path.join(out_dir, "dxy_global.npy"), np.asarray(glob, np.float64))


class PinnedColumns:
    """Host columns of the WHOLE genome in page-locked memory of exactly their size (pgt_host_alloc; torch's pinned
    allocator rounds every tensor up to a power of two, 64 GB for the 48 GB of C4)."""

    def __init__(self, pgt, torch, stat, seed, n_total, offs, dev, slab=1 << 27):
        import ctypes as C
        import numpy as np
        from popgenomicstools_b200 import _cabi
        self._lib, self._ptrs = _cabi.load(), []
        names = {"fst": ("a", "b"), "fused": ("a", "b", "geno", "f1", "f2", "n1", "n2")}[stat]
        dt = dict(a=np.float64, b=np.float64, geno=np.int8, f1=np.float64, f2=np.float64, n1=np.int32, n2=np.int32)
        self.cols = {}
        for k in names:
            p = C.c_void_p()
            nbytes = n_total * np.dtype(dt[k]).itemsize
            _cabi.check(self._lib.pgt_host_alloc(C.byref(p), nbytes))
            self._ptrs.append(p.value)
            self.cols[k] = np.frombuffer((C.c_char * nbytes).from_address(p.value), dtype=dt[k])
        self.cols["pos"] = np.empty(n_total, np.uint32)  # pageable: gathered on the host at window edges, never copied
        views = {k: torch.from_numpy(v) for k, v in self.cols.items() if k != "pos"}
        for s0 in range(0, n_total, slab):  # generated on the device slab by slab, copied out
            m = min(slab, n_total - s0)
            c = make_columns(pgt, stat, seed, s0, m, offs, dev)
            for k in names:
                views[k][s0:s0 + m].copy_(c[k])
            self.cols["pos"][s0:s0 + m] = c["pos"].cpu().numpy().view(np.uint32)
            del c
        torch.cuda.synchronize()

    def free(self):
        import ctypes as C
        self.cols = {}
        for p in self._ptrs:
            self._lib.pgt_host_free(C.c_void_p(p))
        self._ptrs = []


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import popgenomicstools_b200 as pgt
    from popgenomicstools_b200 import _cabi
    from popgenomicstools_b200.scan import _STAT_OUTS
    from popgenomicstools_b200.sharding import SharedTable
    from popgenomicstools_b200.workloads import WORKLOADS, human_like_contigs

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback")
    R = Ranks(torch, dist)
    rank, world, dev = R.rank, R.world, R.dev
    if args.gpus != world and rank == 0:
        print(f"bench.py: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)

    wl = WORKLOADS[args.workload]
    n_total = int(args.sites) if args.sites else wl["n_sites"]
    W, S, seed = wl["winsize"], wl["stepsize"], wl["seed"]
    fused = wl["stat"] == "fused"
    sname = "fused" if fused else "fst"
    names, offs = human_like_contigs(n_total, S)
    # reduction unit (part of the summation order, any value gives the same results within 1e-16):
    # 512 sites fills a 110 KB tile of the 16 B/site fst stream with 13 units = one round of the 15
    # consumer warps (+2 % over the default 256, measured); the 41 B/site fused tile is best at 256
    unit_sites = wl.get("unit_sites", 0)
    plan = pgt.WindowPlan(offs, W, S, unit_sites=unit_sites)
    w_lo, w_hi, s_lo, s_hi = plan.shard(rank, world)
    n_local, nwin_local = s_hi - s_lo, w_hi - w_lo

    # ---- resident synthetic columns of this rank's shard (incl. halo)
    cols = make_columns(pgt, sname, seed, s_lo, n_local, offs, dev)
    stat = _cabi.PGT_STAT_FUSED if fused else _cabi.PGT_STAT_FST
    bytes_per_site = IN_BYTES[sname]
    torch.cuda.synchronize()

    # ---- the window table lives once, in rank 0's HBM; every rank's window kernel writes its rows there
    fields = [k for k in _STAT_OUTS[stat] if k != "dxy_global"]
    tab = SharedTable(_STAT_OUTS[stat], plan.num_windows, rank, world, dist, torch, dev, w_lo=w_lo, w_hi=w_hi)
    out = tab.rows()

    def step():
        pgt.scan(plan, stat, cols, minind=5, window_range=(w_lo, w_hi), site_origin=s_lo, out=out)

    barrier = R.barrier
    # Clock warm-up first (uncounted: the same load for >= 0.3 s, so that the NVML sampler -- one query every
    # 50 ms, outside the ranks' critical path -- sees the clocks under load), then the W counted warm-up steps,
    # then the K timed steps; the sampler runs through all three.
    W_steps = max(0, args.warmup)
    with ClockSampler(R.local) as clk:
        t_w = time.perf_counter()
        for _ in range(3):
            step()
        barrier()
        per = R.reduce([(time.perf_counter() - t_w) / 3])[0]
        for _ in range(max(0, min(4000, int(0.3 / max(per, 1e-5))))):
            step()
        barrier()
        for _ in range(W_steps):
            step()
        barrier()
        launches0 = pgt.kernel_launch_count()
        pgt.profile(True)
        pgt.profile_read()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
    ms_total = e0.elapsed_time(e1)
    prof = pgt.profile_read()
    pgt.profile(False)
    launches = pgt.kernel_launch_count() - launches0
    ms_step = R.reduce([ms_total])[0] / args.steps
    total_launches = int(R.reduce([launches], "sum")[0])
    value = n_total / (ms_step * 1e-3)
    result_checksum = tab.checksum()
    glob = tab.global_line() if fused else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, tab, R, glob)

    # ---- roofline of the dominant kernel (level 1) on this rank
    peak, peak_src = hbm_peak()
    nunits_local = local_units(plan, w_lo, w_hi)
    acc_bytes = ACC_BYTES[sname]
    algo_bytes = bytes_per_site * n_local + acc_bytes * nunits_local
    l1_ms = prof["units_ms"] / max(1, prof["units_launches"])
    achieved = algo_bytes / (l1_ms * 1e-3) / 1e9 if l1_ms > 0 else 0.0
    ach = R.reduce([achieved, prof["units_ms"], prof["windows_ms"]], "sum")
    ach = [x / world for x in ach]
    traffic = recorded_traffic(args.workload, world)
    roofline = {"bound": "hbm", "achieved": round(ach[0], 1), "peak": peak, "unit": "GB/s",
                "frac": round(ach[0] / peak, 4), "traffic": traffic,
                "traffic_source": ("recorded: ncu --set full capture of this kernel, profiles/traffic.json (not measured in this run)"
                                   if traffic is not None else None),
                "kernel": "k_units_tiled (level 1: per-site statistic + unit reduction)",
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes,
                "bytes_per_site": bytes_per_site,
                "kernel_ms_per_launch": round(l1_ms, 4),
                "kernel_share_of_step": round(ach[1] / args.steps / ms_step, 4),
                "level2_ms_per_launch": round(ach[2] / args.steps, 4),
                "step_minus_kernels_ms": round(ms_step - (ach[1] + ach[2]) / args.steps, 4),
                "note": ("pos is gathered only at the two edges of each window, so the compulsory stream is "
                         "a+b = 16 B/site (SURVEY.md 8d conservative variant)" if not fused else
                         "a,b,f1,f2 f64 + n1,n2 i32 + genotype i8 = 41 B/site; pos gathered at window edges only")}
    if not fused:
        roofline["achieved_if_pos_counted_20B"] = round(ach[0] * 20 / 16, 1)

    # ---- end to end through the C ABI with host (pinned) columns: ONE process, ONE table.  At N > 1 rank 0
    # drives all N GPUs through pgt_scan_sharded (one host thread + stream pair per GPU, every shard's rows
    # D2H straight into the table at its window offset); the other ranks only wait.
    e2e = None
    if not args.no_e2e:
        try:
            if rank == 0:
                t_prep = time.perf_counter()
                pinned = PinnedColumns(pgt, torch, sname, seed, n_total, offs, dev)
                hcols = pinned.cols
                prep_s = time.perf_counter() - t_prep
                devices = list(range(world))
                plan_h = pgt.WindowPlan(offs, W, S, unit_sites=unit_sites)  # not bound to a device: every GPU uploads its own tables
                hout = pgt.scan_sharded(plan_h, stat, hcols, devices, minind=5)  # warm-up: contexts on all GPUs
                from popgenomicstools_b200.sharding import table_checksum
                e2e_sum = table_checksum(hout, fields)  # the host path returns exactly what the resident path computed
                assert e2e_sum == result_checksum, f"e2e table differs from the resident table: {e2e_sum} vs {result_checksum}"
                times = []
                for _ in range(args.e2e_steps):
                    t0 = time.perf_counter()
                    pgt.scan_sharded(plan_h, stat, hcols, devices, minind=5, out=hout)
                    times.append(time.perf_counter() - t0)
                e_ms = sum(times) / len(times) * 1e3
                h2d = bytes_per_site * n_total + (world - 1) * bytes_per_site * (W - S)
                d2h = sum(hout[k].nbytes for k in fields if k in ("sum_a", "sum_b", "fst", "nhet", "nonmissing", "het", "dxy",
                                                                   "neffective", "nskip"))
                e2e = {"value": n_total / (e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "ms_per_step": round(e_ms, 3), "steps": args.e2e_steps, "timer": "host wall clock around the (synchronous) call",
                       "n_devices": world, "one_process_one_table": True, "result_checksum": e2e_sum,
                       "host_columns_prep_s": round(prep_s, 1),
                       "api": "pgt_scan_sharded(plan, stat, host columns, devices[0..N-1]): pinned host columns of the whole genome -> "
                              "per GPU: 4M-site slabs H2D (double-buffered, copy stream) -> level 1 per slab -> level 2 -> D2H of the "
                              "shard's rows into the caller's table at its window offset; window positions/labels resolved on the host",
                       "h2d_gbs": round(h2d / (e_ms * 1e-3) / 1e9, 2)}
                del hcols, hout
                pinned.free()
            barrier()
        except Exception as ex:  # report, never fake
            e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "error": repr(ex)[:300]}
            barrier()
    del cols
    tab_placement = tab.placement
    tab.close()
    torch.cuda.empty_cache()

    # ---- the other BASELINE configurations, each sharded over the same ranks
    configs = []
    if not args.no_configs:
        want = [c for c in args.configs.split(",") if c]
        for cfg in CONFIGS:
            if want and cfg["name"] not in want:
                continue
            if cfg["name"] == args.workload:
                continue
            try:
                res = run_config(cfg, R, pgt, args.config_steps, peak)
            except Exception as ex:
                res = dict(name=cfg["name"], error=repr(ex)[:300])
                try:
                    barrier()
                except Exception:
                    pass
            configs.append(res)

    # ---- CPU baseline next to it (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu, _ = reference_arm(WORKLOADS["C4"] if fused else wl, min(args.cpu_sample_sites, n_total), 1, 0, with_cli=True)
            cpu["value"] = round(cpu["value"], 1)
        except Exception as ex:
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "failed: " + repr(ex)[:200]}

    # ---- the drop-in fstWindow on LARGE inputs (the 48 M-site sample above mostly measures CUDA start-up): a 12 GB
    # columnar cache and a 7.6 GB text file, streaming upload (default) against the host-memory path from pageable columns
    cli_large = None
    if rank == 0 and world == 1 and not args.no_cli_large and not args.no_cpu_baseline:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import probe_cli_large as PL
            work = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
            exe = os.path.join(ROOT, "popgenomicstools_b200", "bin", "fstWindow")
            cli_large = []
            nc, ntx = int(args.cli_large_cache_sites), int(args.cli_large_text_sites)
            if nc:
                path = os.path.join(work, "pgt_bench_large.pgtc")
                PL.write_cache(path, nc)
                torch.cuda.empty_cache()
                for env, label in (({}, "cache/stream"), ({"PGT_STREAM": "0"}, "cache/host-pageable")):
                    r = PL.run_tool(exe, path, env, label)
                    r["input_bytes"] = os.path.getsize(path)
                    cli_large.append(r)
                os.remove(path)
            if ntx:
                lnames, loffs = human_like_contigs(ntx, 10000)
                import multiprocessing as mp
                jobs = [(os.path.join(work, f"pgt_bench_large_{nm}.fst"), nm, int(loffs[i]), int(loffs[i + 1]), 4) for i, nm in enumerate(lnames)]
                with mp.get_context("fork").Pool(min(24, os.cpu_count() or 1)) as pool:
                    pool.map(PL._write_contig, jobs)
                path = os.path.join(work, "pgt_bench_large.fst")
                with open(path, "wb") as wf:
                    for j in jobs:
                        with open(j[0], "rb") as rf:
                            shutil.copyfileobj(rf, wf, 1 << 24)
                        os.remove(j[0])
                for env, label in (({}, "text/stream"), ({"PGT_STREAM": "0"}, "text/host-pageable")):
                    r = PL.run_tool(exe, path, env, label)
                    r["input_bytes"] = os.path.getsize(path)
                    cli_large.append(r)
                os.remove(path)
        except Exception as ex:
            cli_large = {"error": repr(ex)[:300]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W_steps,
            "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["desc"], "name": args.workload, "n_sites": n_total, "contigs": 24,
                       "winsize_sites": W, "stepsize_sites": S, "windows": plan.num_windows, "units": plan.num_units,
                       "unit_sites": unit_sites or 256, "sharding": f"site ranges cut at window starts, halo = W-S = {W - S} sites, {world} shard(s)",
                       "l2": "inputs (>= 6 GB per GPU) exceed the 126 MB L2; no flush needed",
                       "clock_warmup": "uncounted steps for >= 0.3 s before the W counted warm-up steps",
                       "gather": (("none: every rank's window kernel writes its rows into the one table in rank 0's HBM "
                                   "(CUDA IPC mapping over NVLink); no collective inside a step" if tab_placement == "rank0" else
                                   "none: the table (above 256 MB) stays sharded, every rank keeps its rows in its own HBM") if world > 1
                                  else "single GPU: results stay in HBM")},
            "result_checksum": result_checksum,
            "clocks": clk.summary(),
            "e2e": e2e if e2e is not None else {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": total_launches,
            "roofline": roofline,
            "configs": configs,
            "cpu_baseline": cpu,
            "our_cli_large": cli_large,
        }
        if glob is not None:
            line["dxy_global"] = [float(x) for x in glob]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    a = parse_args()
    sys.exit(run_reference(a) if a.impl == "reference" else run_b200(a))

"""bench.py's host-side pieces that need no GPU: the argument contract the driver uses, the workload table read
without importing the package (the reference arm must not load libpgtscan.so), the CPU legs' helpers."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_workloads_load_without_the_package_and_configs_are_named():
    code = ("import sys, bench; w = bench.load_workloads(); "
            "assert 'popgenomicstools_b200' not in sys.modules, 'the reference arm must not import the package'; "
            "print(sorted(w.WORKLOADS)); print([c['name'] for c in bench.CONFIGS])")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "C4" in r.stdout and "C5" in r.stdout
    assert "['C1', 'C2-sparse', 'C2-dense', 'C3-1/1', 'C3-100k', 'C5', 'C5-S1']" in r.stdout


def test_compute_only_port_times_the_oracle_on_preparsed_arrays():
    import bench
    wl = bench.load_workloads()
    _, offs = wl.human_like_contigs(480000, 10000)
    r = bench.compute_only_port(offs, 4, 50000, 10000, 2)
    assert r["kind"] == "port" and r["sites"] == int(offs[-1]) and r["cores"] == 2
    assert r["one_core_sites_per_s"] > 1e6 and r["all_cores_sites_per_s"] >= r["one_core_sites_per_s"] * 0.9


def test_reference_arm_line_on_a_tiny_sample():
    """`bench.py --impl reference` prints ONE JSON line with impl / cpu_baseline / e2e and never touches a GPU."""
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample-sites", "2.4e6"],
                       cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "sites/s" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_steps_and_dump_arguments_are_checked():
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, "bench.py", *argv], cwd=ROOT, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "error:" in r.stderr, (argv, r.stderr[-500:])


def test_dump_outputs_writes_the_whole_table_or_a_fixed_sample(tmp_path):
    """--dump-outputs on a window table (the /dev/shm layout of SharedTable, the same code path as in HBM): every field
    as float64, bit-exact; above the byte budget the same seeded rows on every call, and never more than the budget."""
    import types
    import numpy as np
    import torch
    import bench
    from popgenomicstools_b200.sharding import SharedTable
    nwin = 1000
    R = types.SimpleNamespace(rank=0, world=1, dev=torch.device("cpu"), torch=torch, dist=None)
    tab = SharedTable(("label", "start_pos", "nsites", "sum_a", "fst", "dxy_global"), nwin, 0, 1, None, torch=torch,
                      backend="shm", tag=f"pgt_dump_test_{os.getpid()}")
    try:
        rng = np.random.default_rng(1)
        want = {k: rng.random(nwin) if k in ("sum_a", "fst") else rng.integers(0, 1 << 32, nwin, dtype=np.uint32)
                for k in tab.fields}
        rows = tab.rows()
        for k, v in want.items():
            rows[k][:] = v
        full = tmp_path / "full"
        bench.dump_outputs(str(full), tab, R, glob=np.array([1.5, 7.0, 2.0]))
        assert sorted(os.listdir(full)) == sorted([k + ".npy" for k in want] + ["window_index.npy", "dxy_global.npy"])
        assert np.array_equal(np.load(full / "window_index.npy"), np.arange(nwin))
        assert np.array_equal(np.load(full / "dxy_global.npy"), [1.5, 7.0, 2.0])
        for k, v in want.items():
            got = np.load(full / f"{k}.npy")
            assert got.dtype == np.float64 and np.array_equal(got, v.astype(np.float64)), k
        budget = 4096 + 8 * (len(want) + 1) * 100  # 100 rows
        dirs = [tmp_path / "s1", tmp_path / "s2"]
        for d in dirs:
            bench.dump_outputs(str(d), tab, R, budget=budget)
            assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= budget
        idx = np.load(dirs[0] / "window_index.npy")
        assert len(idx) == 100 and np.all(np.diff(idx) > 0) and np.array_equal(idx, np.load(dirs[1] / "window_index.npy"))
        for k, v in want.items():
            assert np.array_equal(np.load(dirs[0] / f"{k}.npy"), v[idx.astype(np.int64)].astype(np.float64)), k
    finally:
        tab.close()

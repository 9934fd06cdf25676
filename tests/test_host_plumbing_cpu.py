"""Host plumbing without a device: the workspace and device-table sizes of the C ABI over a grid of plans, pinned in
tests/golden/host_plumbing_sizes.json, and the Python layer's column checks.

The pinned sizes are those of the library before the window scan, the extreme-score scan and their multi-GPU drivers
shared their host code; any change to them changes how much device memory a caller has to provide."""
import ctypes as C
import json
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "host_plumbing_sizes.json")
NSHARDS = 7


def window_plans():
    """(key, mode, contig offsets, W, S, unit_sites): site and bp mode, few / many (> 32 segments) / long contigs."""
    rng = np.random.default_rng(11)
    layouts = {"few": [25000, 9000, 3100], "many": [int(x) for x in rng.integers(1, 5000, size=40)],
               "long": [9_000_000, 7_000_000, 1_500_000]}
    shapes = {0: [(1, 1, 0), (300, 1, 0), (5000, 1000, 0), (100, 10, 32), (64, 64, 4096), (20000, 5000, 0)],
              1: [(1000, 1000, 0), (5000, 1000, 0), (100, 10, 32), (50000, 10000, 0)]}
    for mode, wsu in shapes.items():
        for name, lengths in layouts.items():
            offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)
            for W, S, unit in wsu:
                yield f"plan mode={mode} {name} W={W} S={S} unit={unit}", mode, offs, W, S, unit


def extreme_plans():
    """(key, pos, contig offsets, chrlen, W, unit_sites): dense and sparse runs, with and without -chrlen."""
    rng = np.random.default_rng(12)
    layouts = {"two": ([20000, 17100], [2_000_000, 1_000_000]), "many": ([int(x) for x in rng.integers(1, 3000, size=40)], None)}
    for name, (lengths, chrlen) in layouts.items():
        span = chrlen or [60 * n + 100 for n in lengths]
        pos = np.concatenate([np.sort(rng.integers(1, L + 1, size=n)) for n, L in zip(lengths, span)]).astype(np.uint32)
        offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)
        for W, unit in ((100000, 0), (10000, 64), (1000, 0), (100, 0)):
            yield f"xplan {name} W={W} unit={unit}", pos, offs, chrlen, W, unit


def ranges(shard_fn, nwin):
    """All windows, the NSHARDS shards' windows, the middle third."""
    out = [(0, nwin)]
    for i in range(NSHARDS):
        v = [C.c_uint64() for _ in range(4)]
        assert shard_fn(i, NSHARDS, *[C.byref(x) for x in v]) == 0
        out.append((v[0].value, v[1].value))
    out.append((nwin // 3, 2 * nwin // 3))
    return out


def size_table():
    from popgenomicstools_b200 import _cabi
    lib = _cabi.load()
    table = {}
    for key, mode, offs, W, S, unit in window_plans():
        h = C.c_void_p()
        assert lib.pgt_plan_create(C.byref(h), mode, offs.ctypes.data, len(offs) - 1, W, S, unit) == 0
        sizes = [int(lib.pgt_plan_device_bytes(h))]
        for lo, hi in ranges(lambda *a: lib.pgt_plan_shard(h, *a), int(lib.pgt_plan_num_windows(h))):
            r = _cabi.PgtRange(lo, hi, 0, 0)
            sizes += [int(lib.pgt_scan_workspace_bytes(h, C.byref(r), stat, mem)) for stat in range(4) for mem in (0, 1)]
        sizes += [int(lib.pgt_scan_sharded_workspace_bytes(h, stat, i, NSHARDS)) for stat in range(4) for i in range(NSHARDS)]
        lib.pgt_plan_destroy(h)
        table[key] = sizes
    for key, pos, offs, chrlen, W, unit in extreme_plans():
        h = C.c_void_p()
        cl = np.asarray(chrlen, np.uint32) if chrlen else None
        assert lib.pgt_xplan_create(C.byref(h), pos.ctypes.data, offs.ctypes.data, cl.ctypes.data if cl is not None else None,
                                    len(offs) - 1, W, unit) == 0
        sizes = [int(lib.pgt_xplan_device_bytes(h))]
        for lo, hi in ranges(lambda *a: lib.pgt_xplan_shard(h, *a), int(lib.pgt_xplan_num_windows(h))):
            r = _cabi.PgtRange(lo, hi, 0, 0)
            sizes += [int(lib.pgt_scan_extreme_workspace_bytes(h, C.byref(r), mem)) for mem in (0, 1)]
        lib.pgt_xplan_destroy(h)
        table[key] = sizes
    return table


def test_workspace_and_table_sizes_are_pinned():
    if os.environ.get("PGT_TUNE"):
        pytest.skip("PGT_TUNE knobs choose other kernels, and some need other workspaces")
    with open(GOLDEN) as f:
        want = json.load(f)
    got = size_table()
    assert list(got) == list(want)
    for key in want:
        assert got[key] == want[key], key


def test_columns_check_dtypes_and_layout():
    import torch
    from popgenomicstools_b200.scan import _columns
    a = np.zeros(8)
    with pytest.raises(TypeError, match=r"^a: expected contiguous float64, got float32$"):
        _columns(dict(a=a.astype(np.float32), b=a), ("pos", "a", "b"), ("a", "b"), False)
    with pytest.raises(TypeError, match=r"^b: expected contiguous float64, got float64$"):
        _columns(dict(a=a, b=np.zeros(16)[::2]), ("pos", "a", "b"), ("a", "b"), False)
    with pytest.raises(TypeError, match=r"^score: expected contiguous float64, got int64$"):
        _columns(dict(pos=None, score=np.zeros(8, np.int64)), ("pos", "score"), (), False)
    with pytest.raises(TypeError, match=r"^a: expected a contiguous CUDA tensor$"):
        _columns(dict(a=torch.zeros(8, dtype=torch.float64), b=a), ("pos", "a", "b"), ("a", "b"), True)
    with pytest.raises(TypeError, match=r"^pos: expected a contiguous CUDA tensor$"):
        _columns(dict(pos=np.zeros(8, np.uint32), score=a), ("pos", "score"), (), True)
    with pytest.raises(ValueError, match=r"^column 'geno' is required$"):
        _columns(dict(pos=np.zeros(8, np.uint32)), ("pos", "geno"), ("geno",), False)
    # CPU tensors are read as numpy arrays; columns the statistic does not read are ignored
    ptrs, keep = _columns(dict(a=torch.zeros(8, dtype=torch.float64), b=a, geno=np.zeros(8, np.float32)), ("pos", "a", "b"), ("a", "b"), False)
    assert set(ptrs) == {"a", "b"} and ptrs["b"] == a.ctypes.data and len(keep) == 2


@pytest.mark.parametrize("names,need", [(("pos", "a", "b"), ("a", "b")), (("pos", "score"), ())])
def test_columns_view_int32_positions_as_uint32(names, need):
    """Both the window scan and the extreme-score scan take int32 positions in host memory."""
    from popgenomicstools_b200.scan import _columns
    pos = np.arange(-3, 5, dtype=np.int32)
    cols = {k: np.zeros(8) for k in names}
    cols["pos"] = pos
    ptrs, keep = _columns(cols, names, need, False)
    assert ptrs["pos"] == pos.ctypes.data
    (p,) = [v for v in keep if v.ctypes.data == pos.ctypes.data]
    assert p.dtype == np.uint32 and np.array_equal(p, pos.view(np.uint32))

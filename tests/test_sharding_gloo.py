"""N > 1 host logic on CPU: world_size-2 (and 4) gloo process groups exercise the shard split,
the packed-buffer gather to rank 0 and the reassembly into one window table.  The per-shard
window values are taken from the oracle (no kernels run here); what is under test is that
shards tile the window list, that every shard's sites (incl. the W-S halo) suffice for its
windows, and that gather + unpack reproduces the unsharded table bit for bit."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle_lib as O
import textfmt as T


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, lengths, W, S, result_path):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import popgenomicstools_b200 as pgt
    from popgenomicstools_b200.sharding import PackedWindows, shard_counts
    offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)
    n = int(offs[-1])
    plan = pgt.WindowPlan(offs, W, S)
    w_lo, w_hi, s_lo, s_hi = plan.shard(rank, world)
    first, last, label = plan.windows()
    if w_hi > w_lo:  # the shard's site range covers all of its windows
        assert s_lo <= first[w_lo] and last[w_hi - 1] < s_hi
    # "compute" this shard: oracle over the whole genome, sliced to the shard's windows
    a, b = O.synth_fst(9, 0, n)
    pos = O.synth_pos(9, offs, 1)
    ref = O.fst(T.expand_chr(lengths), pos, a, b, W, S)
    fields = ("label", "start_pos", "end_pos", "mid_pos", "nsites", "sum_a", "sum_b", "fst")
    key = dict(label="label", start_pos="start", end_pos="end", mid_pos="mid", nsites="n", sum_a="asum", sum_b="bsum", fst="fst")
    counts = shard_counts(dist, w_hi - w_lo, world, "cpu", torch)
    assert sum(counts) == plan.num_windows
    pw = PackedWindows(fields, w_hi - w_lo, max(counts), "cpu", torch)
    for k in fields:
        src = np.ascontiguousarray(ref[key[k]][w_lo:w_hi])
        if src.dtype == np.uint32:
            pw.views[k].view(torch.int32).copy_(torch.from_numpy(src.view(np.int32)))
        else:
            pw.views[k].copy_(torch.from_numpy(src))
    g = pw.gather(dist, rank, world)
    if rank == 0:
        table = pw.unpack(g, counts)
        ok = all(table[k].tobytes() == np.ascontiguousarray(ref[key[k]]).tobytes() for k in fields)
        open(result_path, "w").write("ok" if ok else "mismatch")
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_shard_gather_roundtrip_gloo(world, tmp_path):
    lengths = [24117, 23000, 19876, 5000, 123, 9999]  # contig 0: (N-W)%S==0 -> carry across the cut region
    res = str(tmp_path / "res.txt")
    mp.spawn(_worker, args=(world, _free_port(), lengths, 500, 100, res), nprocs=world, join=True)
    assert open(res).read() == "ok"


def _xworker(rank, world, port, lengths, W, result_path):
    """Same for the ihsWindow / xpehhWindow extreme scan: shards are window ranges without halo."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import popgenomicstools_b200 as pgt
    from popgenomicstools_b200.sharding import PackedWindows, shard_counts
    offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)
    n = int(offs[-1])
    pos = O.synth_pos(9, offs, 23)
    val = O.synth_score(9, 0, n)
    plan = pgt.ExtremePlan(pos, offs, W)
    w_lo, w_hi, s_lo, s_hi = plan.shard(rank, world)
    tab = plan.windows()
    if w_hi > w_lo:  # the shard's site range is exactly the sites of its windows
        assert s_lo == tab["first_site"][w_lo] and s_hi == s_lo + int(tab["nsites"][w_lo:w_hi].sum())
    # "compute" this shard from its own slice of the columns only
    chr_id = T.expand_chr(lengths)
    ref = O.extreme("ihs", chr_id, pos, val, W, 2.0)
    fields = ("ext_value", "ext_pos", "nbig", "nsites", "prop")
    key = dict(ext_value="ext", ext_pos="extpos", nbig="nbig", nsites="n", prop="prop")
    counts = shard_counts(dist, w_hi - w_lo, world, "cpu", torch)
    assert sum(counts) == plan.num_windows == len(ref["n"])
    pw = PackedWindows(fields, w_hi - w_lo, max(counts), "cpu", torch)
    for k in fields:
        src = np.ascontiguousarray(ref[key[k]][w_lo:w_hi])
        if src.dtype == np.uint32:
            pw.views[k].view(torch.int32).copy_(torch.from_numpy(src.view(np.int32)))
        else:
            pw.views[k].copy_(torch.from_numpy(src))
    g = pw.gather(dist, rank, world)
    if rank == 0:
        table = pw.unpack(g, counts)
        ok = all(table[k].tobytes() == np.ascontiguousarray(ref[key[k]]).tobytes() for k in fields)
        open(result_path, "w").write("ok" if ok else "mismatch")
    dist.barrier()
    dist.destroy_process_group()


def test_extreme_shard_gather_roundtrip_gloo(tmp_path):
    res = str(tmp_path / "xres.txt")
    mp.spawn(_xworker, args=(2, _free_port(), [9000, 4000, 2500, 10], 5000, res), nprocs=2, join=True)
    assert open(res).read() == "ok"


def _tworker(rank, world, port, lengths, W, S, result_path):
    """SharedTable: every rank writes the rows of its shard IN PLACE into the one table rank 0 owns (the GPU build
    maps rank 0's HBM through CUDA IPC; here the same layout logic runs over a /dev/shm file)."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import popgenomicstools_b200 as pgt
    from popgenomicstools_b200.sharding import SharedTable
    offs = np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)
    n = int(offs[-1])
    plan = pgt.WindowPlan(offs, W, S)
    w_lo, w_hi, s_lo, s_hi = plan.shard(rank, world)
    f1, f2, n1, n2 = O.synth_dxy(9, 0, n)
    pos = O.synth_pos(9, offs, 1)
    ref = O.dxy(T.expand_chr(lengths), pos, f1, f2, n1, n2, 5, W, S, 1)
    fields = ("label", "start_pos", "end_pos", "dxy", "neffective", "nskip", "dxy_global")
    key = dict(label="label", start_pos="start", end_pos="end", dxy="dxy", neffective="neff", nskip="nskip")
    tab = SharedTable(fields, plan.num_windows, rank, world, dist, torch=torch, backend="shm", tag="pgt_gloo_test", w_lo=w_lo, w_hi=w_hi)
    rows = tab.rows()
    for k, kr in key.items():
        rows[k][:] = np.asarray(ref[kr][w_lo:w_hi]).astype(rows[k].dtype)
    # every rank's global line over the sites it owns: here simply its share of the oracle's line
    rows["dxy_global"][:] = np.array(ref["global"], np.float64) * (1.0 if rank == 0 else 0.0)
    dist.barrier()
    checksum = tab.checksum()  # collective: every rank sums the rows it wrote
    if rank == 0:
        from popgenomicstools_b200.sharding import table_checksum
        t = tab.table()
        ok = all(np.ascontiguousarray(t[k]).tobytes() == np.asarray(ref[kr]).astype(t[k].dtype).tobytes() for k, kr in key.items())
        ok = ok and np.array_equal(t["dxy_global"], np.array(ref["global"], np.float64))
        ok = ok and table_checksum(t, fields) == checksum
        open(result_path, "w").write(("ok " if ok else "mismatch ") + checksum)
    tab.close()
    dist.barrier()
    dist.destroy_process_group()


def test_shared_table_in_place_rows_gloo(tmp_path):
    lengths = [24117, 23000, 19876, 5000, 123, 9999]
    sums = []
    for world in (1, 2, 4):
        res = str(tmp_path / f"tres{world}.txt")
        mp.spawn(_tworker, args=(world, _free_port(), lengths, 500, 100, res), nprocs=world, join=True)
        status, checksum = open(res).read().split()
        assert status == "ok"
        sums.append(checksum)
    assert sums[0] == sums[1] == sums[2], sums  # the table's checksum does not depend on how many ranks wrote it


def _dworker(rank, world, port, nwin, budget, out_dir):
    """bench.dump_outputs on a window table sharded over the ranks: every rank sends its sampled rows to rank 0."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import types
    import bench
    from popgenomicstools_b200.sharding import SharedTable
    bounds = np.linspace(0, nwin, world + 1).astype(int)
    w_lo, w_hi = int(bounds[rank]), int(bounds[rank + 1])
    tab = SharedTable(("label", "sum_a", "fst"), nwin, rank, world, dist, torch=torch, backend="shm", tag="pgt_dump_gloo_test",
                      w_lo=w_lo, w_hi=w_hi)
    # the /dev/shm layout indexes rows globally, so every rank's rows stay valid; only the dump's gather path changes
    tab.placement = "sharded"
    want = _dump_table(nwin)
    rows = tab.rows()
    for k, v in want.items():
        rows[k][:] = v[w_lo:w_hi]
    dist.barrier()
    bench.dump_outputs(out_dir, tab, types.SimpleNamespace(rank=rank, world=world, dev=torch.device("cpu"), torch=torch, dist=dist),
                       budget=budget)
    dist.barrier()
    tab.close()
    dist.destroy_process_group()


def _dump_table(nwin):
    rng = np.random.default_rng(5)
    return dict(label=rng.integers(0, 1 << 32, nwin, dtype=np.uint32), sum_a=rng.random(nwin), fst=rng.random(nwin))


def test_bench_dump_gathers_a_sharded_table_gloo(tmp_path):
    nwin = 1000
    want = _dump_table(nwin)
    sampled = []
    for world, budget in ((2, 1 << 20), (2, 4096 + 8 * 4 * 300), (3, 4096 + 8 * 4 * 300)):
        d = tmp_path / f"dump_{world}_{budget}"
        mp.spawn(_dworker, args=(world, _free_port(), nwin, budget, str(d)), nprocs=world, join=True)
        idx = np.load(d / "window_index.npy")
        if budget == 1 << 20:
            assert np.array_equal(idx, np.arange(nwin))
        else:
            assert len(idx) == 300 and np.all(np.diff(idx) > 0)
            sampled.append(idx)
        for k, v in want.items():
            got = np.load(d / f"{k}.npy")
            assert got.dtype == np.float64 and np.array_equal(got, v[idx.astype(np.int64)].astype(np.float64)), (world, k)
    assert np.array_equal(sampled[0], sampled[1])  # the same rows whatever the number of ranks

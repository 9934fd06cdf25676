"""The text parsers cut their input into line-aligned chunks (one or eight per thread) and parse the chunks
concurrently, straight into the final columns.  Where the cuts fall must not show in the result: the .pgtc a
tool packs is the same for every thread count, and of two malformed lines in different chunks the first in
file order is the one reported.  Packing never touches the device, so all of this runs on the CPU."""
import pytest

import cli_util as U
from popgenomicstools_b200 import colfile

# PGT_PARALLEL_MIN_BYTES=1 sends these small texts through the multi-chunk path, so the chunk boundaries fall
# inside name runs, next to CRLF line ends and around blank lines
THREADS = [1, 2, 3, 7, 16]


def penv(threads, **kw):
    e = {"PGT_THREADS": str(threads), "PGT_PARALLEL_MIN_BYTES": "1"}
    e.update({k: str(v) for k, v in kw.items()})
    return e


def name_of(i):
    # runs of 33 or 34 lines; chr1 comes back later as a run of its own
    return ["chr1", "chr2", "chrUn_7", "chr1", "chrX"][(i * 3 // 101) % 5]


def site_lines(kind, n):
    lines = []
    for i in range(n):
        sep = "\t" if i % 3 else " "
        if kind == "fst":
            vals = f"0.{i * 7919 % 1000000:06d}{sep}{1 + i % 5}.25" if i % 17 else f"{i}e-4  +0.5"  # the general path too
        else:
            vals = str(i % 4 - 1)
        lines.append(f"{name_of(i)}{sep}{10 + 3 * i}{sep}{vals}" + ("\r" if i % 11 == 0 else ""))
    return lines


def maf_lines(n, seed):
    lines = ["chromo\tposition\tmajor\tminor\tref\tknownEM\tnInd"]
    for i in range(n):
        f = f"0.{(i * 7919 + seed) % 1000000:06d}" if i % 19 else f"{i + seed}e-5"
        lines.append(f"{name_of(i)}\t{5 + 2 * i}\tA\tC\tA\t{f}\t{(i + seed) % 12}" + ("\r" if i % 13 == 0 else ""))
    return lines


def norm_lines(tool, n):
    nfields = 6 if tool == "ihsWindow" else 8
    lines = ["id\tpos\tgpos\tp1\tihh1\tp2\tihh2\txpehh\tnormxpehh\tcrit"] if tool == "xpehhWindow" else []
    for i in range(n):
        if i % 23 == 5:
            lines.append("" if i % 2 else "  \t ")  # blank: the previous site again
            continue
        nm = name_of(i)
        fields = [f"{(i * 31 + k) % 200 / 50 - 2:.3f}" for k in range(nfields)]
        if i % 29 == 3:
            fields = fields[:i % nfields]  # short line: the score is the previous line's
        if i % 37 == 8 and fields:
            fields[-1] = "NA"  # non-numeric score
        locus = nm if nm == "chrUn_7" else f"{nm}_{100 + i}"
        lines.append("\t".join([locus, str(100 + i)] + fields) + ("\r" if i % 7 == 0 else ""))
    return lines


def pack_all_threads(tool, args, files, tmp_path):
    """Pack at every thread count: the files each tool writes, as bytes, must not depend on it."""
    first = None
    for th in THREADS:
        out = {k: tmp_path / f"{k}.{th}.pgtc" for k in files}
        rc, so, se = U.run(U.ours(tool), args, cwd=str(tmp_path), env=penv(th, **out))
        assert (rc, so, se) == (0, "", ""), (tool, th, se)
        got = {k: p.read_bytes() for k, p in out.items()}
        if first is None:
            first = got
        assert got == first, (tool, th)
    return {k: colfile.read(tmp_path / f"{k}.{THREADS[0]}.pgtc") for k in files}


@pytest.mark.parametrize("tool,kind", [("fstWindow", "fst"), ("hetWindow", "het")])
def test_site_columns_do_not_depend_on_the_thread_count(tool, kind, tmp_path):
    lines = site_lines(kind, 600)
    # the first empty line ends the input: 400 sites
    (tmp_path / "s.txt").write_text("\n".join(lines[:400]) + "\n\n" + "\n".join(lines[400:]) + "\n", newline="")
    r = pack_all_threads(tool, ["s.txt", 10, 5], ["PGT_PACK"], tmp_path)["PGT_PACK"]
    assert r["nsites"] == 400 and len(r["runs"]) > 5


def test_maf_columns_do_not_depend_on_the_thread_count(tmp_path):
    one, two = maf_lines(700, 1), maf_lines(650, 2)
    (tmp_path / "p1.maf").write_text("\n".join(one[:501]) + "\n\n" + "\n".join(one[501:]) + "\n", newline="")
    (tmp_path / "p2.maf").write_text("\n".join(two), newline="")  # no final newline
    r = pack_all_threads("dxyWindow", ["-fixedsite", 1, "-winsize", 10, "-stepsize", 5, "p1.maf", "p2.maf"], ["PGT_PACK", "PGT_PACK2"],
                         tmp_path)
    assert r["PGT_PACK"]["nsites"] == 500 and r["PGT_PACK2"]["nsites"] == 650 and len(r["PGT_PACK"]["runs"]) > 5


@pytest.mark.parametrize("tool", ["ihsWindow", "xpehhWindow"])
def test_score_columns_do_not_depend_on_the_thread_count(tool, tmp_path):
    (tmp_path / "s.norm").write_text("\n".join(norm_lines(tool, 600)) + "\n", newline="")
    args = ["s.norm"] if tool == "ihsWindow" else ["s.norm", 2]
    r = pack_all_threads(tool, args, ["PGT_PACK"], tmp_path)["PGT_PACK"]
    assert r["nsites"] == 600 and len(r["runs"]) > 5


@pytest.mark.parametrize("tool,kind", [("fstWindow", "fst"), ("hetWindow", "het"), ("dxyWindow", "maf")])
def test_the_first_malformed_line_is_reported(tool, kind, tmp_path):
    """Rows 50 and 350 do not parse; with two or more threads they lie in different chunks."""
    if kind == "maf":
        lines = maf_lines(400, 1)
        lines[1 + 50] = "chr1\t105\tA"
        lines[1 + 350] = "chr2 x"
        (tmp_path / "p1.maf").write_text("\n".join(lines) + "\n")
        (tmp_path / "p2.maf").write_text("\n".join(maf_lines(400, 2)) + "\n")
        args, want = ["-fixedsite", 1, "-winsize", 10, "-stepsize", 5, "p1.maf", "p2.maf"], "cannot parse line 52 of p1.maf\n"
    else:
        lines = site_lines(kind, 400)
        lines[50] = "chr1 x 0.5 0.5"
        lines[350] = "chr2"
        (tmp_path / "s.txt").write_text("\n".join(lines) + "\n")
        args, want = ["s.txt", 10, 5], "cannot parse line 51 of s.txt\n"
    for th in THREADS:
        out = tmp_path / f"o.{th}.pgtc"
        rc, so, se = U.run(U.ours(tool), args, cwd=str(tmp_path), env=penv(th, PGT_PACK=out, PGT_PACK2=out))
        assert (rc, so, se) == (255, "", f"{tool}: {want}"), th
        assert not out.exists()

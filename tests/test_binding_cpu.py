"""The reference-side binding of INTEGRATION.md §1 (tests/integration/sitewindow_binding.cpp): the
reference's own main/parseArgs/info translation units with calcFst / calcHeterozygosity replaced by
calls into libpgtscan.so through the C ABI.  It is compiled against the unmodified reference sources
where they lie (make -C oracle binding -> oracle/_ref/{fstWindow,hetWindow}_pgt); here, without a GPU:
it builds and links, keeps the reference's argv contract byte for byte, and fails loudly (no CPU
fallback) when it reaches the scan."""
import os
import subprocess

import pytest

import cli_util as U
import oracle_lib as O

ROOT = U.ROOT


def binding(tool):
    p = os.path.join(ROOT, "oracle", "_ref", tool + "_pgt")
    reference = os.environ.get("PGT_REFERENCE")  # directory of the original PopGenomicsTools sources
    if reference and os.path.isdir(reference):
        U.ours(tool)  # libpgtscan.so must exist to link against
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "binding", f"REFERENCE={reference}"], check=True)
    return p if os.access(p, os.X_OK) else None


@pytest.mark.parametrize("tool", ["fstWindow", "hetWindow"])
def test_binding_builds_and_keeps_the_argv_contract(tool, tmp_path):
    exe = binding(tool)
    if exe is None:
        pytest.skip("oracle/_ref/*_pgt not built (needs the reference sources)")
    ref = O.ref_binary(tool)
    f = tmp_path / "in.txt"
    f.write_text("chr1 1 0.1 0.2\nchr1 2 0.3 0.4\n" if tool == "fstWindow" else "chr1 1 0\nchr1 2 1\n")
    for args in ([], ["/nonexistent/file"], [f, 0], [f, "abc"]):
        got = U.run(exe, args)
        assert got == U.run(U.ours(tool), args), args  # same contract as the drop-in CLI
        if ref:
            assert got == U.run(ref, args), args
    # an empty input prints nothing and needs no device
    e = tmp_path / "empty.txt"
    e.write_text("")
    assert U.run(exe, [e, 2, 1]) == (0, "", "")
    import torch
    if not torch.cuda.is_available():
        rc, out, err = U.run(exe, [f, 2, 1])
        assert rc == 255 and out == "" and "cuda" in err.lower()

"""The shipped launcher (crispresso2_b200/launcher.py) against the UNMODIFIED reference CLI on a real GPU: the reference's own
`CRISPResso` main() (baseline/_ref, installed by the recipe in baseline/ref_shim.py; skipped where it is absent) is
run twice on the same FASTQ -- as it is (CPU), and through `python -m crispresso2_b200.launcher` (process_fastq, filterFastqs
and the table around the cut re-bound to the engine, sm_100a library) -- and every file of the two output folders must be
byte-identical (SURVEY.md Appendix B).  The CPU twin of this test (warp-emulator engine) is tests/test_cli_dropin.py."""
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import golden_util as G  # noqa: E402
from test_cli_dropin import _info_stats, _snapshot  # noqa: E402

pytestmark = pytest.mark.gpu

REF_MAIN = ("import sys; sys.path.insert(0, %r); from baseline import ref_shim; CORE = ref_shim.load_core(); "
            "sys.argv = ['CRISPResso'] + sys.argv[1:]; CORE.main()" % ROOT)


def _fastq(tmp_path, case):
    rec = G.load(case)
    fq = tmp_path / (case + ".fastq")
    with open(fq, "w") as fh:
        for k, s in enumerate(rec["reads"]):
            fh.write("@r%d\n%s\n+\n%s\n" % (k, s, "I" * len(s)))
    return rec, str(fq)


@pytest.mark.parametrize("case,extra", [("fanc_cas9", ["--write_detailed_allele_table"]),
                                        ("synth_hdr", []),
                                        ("synth_single", ["--ignore_substitutions", "-w", "10"])])
def test_launcher_output_folder_equals_the_reference(case, extra, tmp_path):
    from baseline import ref_shim
    if not ref_shim.available():
        pytest.skip("baseline/_ref (the pip-installed reference) did not travel")
    rec, fq = _fastq(tmp_path, case)
    names = rec["ref_names"]
    amp = rec["refs"][names[0]]["sequence"]
    guide = "GGAATCCCTTCTGCAGCACC" if case.startswith("fanc") else amp[110:130]
    argv = ["-r1", fq, "-a", amp, "-g", guide, "--suppress_plots", "--suppress_report"] + extra
    if len(names) > 1:
        argv += ["-e", rec["refs"][names[1]]["sequence"]]
    env = dict(os.environ, PYTHONPATH=ROOT)
    outs = {}
    for mode, cmd in (("ref", [sys.executable, "-c", REF_MAIN]), ("b200", [sys.executable, "-m", "crispresso2_b200.launcher"])):
        out = str(tmp_path / mode)
        os.makedirs(out)
        p = subprocess.run(cmd + argv + ["-o", out], capture_output=True, text=True, timeout=900, env=env, cwd=out)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
        outs[mode] = out
    a, b = _snapshot(outs["ref"]), _snapshot(outs["b200"])
    assert sorted(a) == sorted(b)
    diff = [k for k in a if a[k] != b[k]]
    assert not diff, diff
    assert len(a) >= 10
    assert _info_stats(outs["ref"]) == _info_stats(outs["b200"])


def _run_both(argv, tmp_path, env):
    outs = {}
    for mode, cmd in (("ref", [sys.executable, "-c", REF_MAIN]), ("b200", [sys.executable, "-m", "crispresso2_b200.launcher"])):
        out = str(tmp_path / mode)
        os.makedirs(out)
        p = subprocess.run(cmd + argv + ["--suppress_plots", "--suppress_report", "-o", out], capture_output=True, text=True, timeout=900,
                           env=env, cwd=out)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
        outs[mode] = out
    a, b = _snapshot(outs["ref"]), _snapshot(outs["b200"])
    assert sorted(a) == sorted(b)
    diff = [k for k in a if a[k] != b[k]]
    assert not diff, diff
    assert _info_stats(outs["ref"]) == _info_stats(outs["b200"])
    return a


def test_launcher_prime_editing_scaffold(tmp_path):
    """'Scaffold-incorporated' re-labelling (CRISPRessoCORE.py:789-796) through the sm_100a library: the reads and pegRNA of the
    reference-generated fixture tests/golden/fanc_pe_scaffold.json.gz."""
    from baseline import ref_shim
    if not ref_shim.available():
        pytest.skip("baseline/_ref (the pip-installed reference) did not travel")
    rec, fq = _fastq(tmp_path, "fanc_pe_scaffold")
    P = rec["params"]
    argv = ["-r1", fq, "-a", rec["refs"]["Reference"]["sequence"], "--prime_editing_pegRNA_spacer_seq", "GGAATCCCTTCTGCAGCACC",
            "--prime_editing_pegRNA_extension_seq", P["prime_editing_pegRNA_extension_seq"],
            "--prime_editing_pegRNA_scaffold_seq", P["prime_editing_pegRNA_scaffold_seq"]]
    snap = _run_both(argv, tmp_path, dict(os.environ, PYTHONPATH=ROOT))
    assert any(k.startswith("Scaffold-incorporated.") for k in snap) and "Scaffold_insertion_sizes.txt" in snap


def test_launcher_paired_end_merge_mode(tmp_path):
    """--crispresso_merge (process_paired_fastq, :1245-1733) through crispresso2_b200.paired on the GPU; `fastp`, which the
    reference runs first even in this mode, is the pass-through stand-in tests/fake_fastp.py put on PATH."""
    from baseline import ref_shim
    if not ref_shim.available():
        pytest.skip("baseline/_ref (the pip-installed reference) did not travel")
    import stat
    import pe_case
    amp = G.load("fanc_cas9")["refs"]["Reference"]["sequence"]
    r1, r2 = str(tmp_path / "R1.fastq"), str(tmp_path / "R2.fastq")
    pe_case.write_pairs(r1, r2, amp, n=600)
    bindir = tmp_path / "bin"
    bindir.mkdir()
    exe = bindir / "fastp"
    exe.write_text("#!/bin/sh\nexec %s %s \"$@\"\n" % (sys.executable, os.path.join(HERE, "fake_fastp.py")))
    exe.chmod(exe.stat().st_mode | stat.S_IXUSR | stat.S_IXGRP | stat.S_IXOTH)
    env = dict(os.environ, PYTHONPATH=ROOT, PATH=str(bindir) + os.pathsep + os.environ.get("PATH", ""))
    argv = ["-r1", r1, "-r2", r2, "-a", amp, "-g", "GGAATCCCTTCTGCAGCACC", "--crispresso_merge", "--fastq_output"]
    snap = _run_both(argv, tmp_path, env)
    assert len(snap) >= 10

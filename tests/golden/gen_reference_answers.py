#!/usr/bin/env python
"""Generates tests/golden/reference_answers.json.gz: what the UNMODIFIED reference returned for the inputs of the tests that
compare the replacement with it, so that those tests run without the reference.

Run from the repo root:  python tests/golden/gen_reference_answers.py <CRISPResso2 source tree>
Needs that source tree (its unit tests, filterFastqs.py and EDNAFULL / BLOSUM62), oracle/_ref (the reference's two Cython
modules, compiled by oracle/Makefile) and what tests/golden/gen_golden.py needs to import the reference's CRISPRessoCORE.

Sections:
  matrices, unit_tests  every call tests/unit_tests/test_CRISPResso2Align.py and test_CRISPRessoCOREResources.py make to the
                        two native modules, answered by the compiled modules (tests/test_reference_unit_tests.py)
  consensus_unit        the calls of test_CRISPRessoCORE.py's get_consensus_alignment_from_pairs test, and
  consensus_fuzz        a digest of the answer for each fuzz case of tests/test_paired_consensus.py
  oracle_fuzz, oracle_legacy   digests of global_align / find_indels_substitutions(_legacy) for tests/test_oracle.py's fuzz
  filter                digests of what filterFastqs wrote (or the exception it raised) for tests/test_filter_fastqs.py
"""
import contextlib
import gzip
import importlib.util
import io
import json
import os
import sys
import tempfile
import types

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
TESTS = os.path.join(REPO, "tests")
sys.path.insert(0, REPO)
sys.path.insert(0, TESTS)
sys.path.insert(0, os.path.join(TESTS, "emu"))

import golden_util as G  # noqa: E402
from oracle import oracle as O  # noqa: E402


def _exec(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@contextlib.contextmanager
def _modules(mods):
    saved = {k: sys.modules.get(k) for k in mods}
    sys.modules.update(mods)
    try:
        yield
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


class Recorder:
    """Wraps the reference's functions: every call is kept with its arguments and what it returned or raised."""

    def __init__(self, arrays):
        self.arrays, self.calls = arrays, []

    def wrap(self, name, fn):
        def call(*args, **kwargs):
            rec = {"fn": name, "args": G.encode_value(list(args), self.arrays), "kwargs": G.encode_value(kwargs, self.arrays)["d"]}
            self.calls.append(rec)
            try:
                out = fn(*args, **kwargs)
            except Exception as ex:
                rec["raises"] = type(ex).__name__
                raise
            rec["out"] = G.digest(out)
            return out
        return call

    def take(self):
        calls, self.calls = self.calls, []
        return calls


def unit_tests(ref, arrays):
    A, R = O.ref_modules()
    out = {}
    for test_file in ("test_CRISPResso2Align.py", "test_CRISPRessoCOREResources.py"):
        rec = Recorder(arrays)
        a = types.ModuleType("CRISPResso2.CRISPResso2Align")
        for n in ("read_matrix", "make_matrix", "global_align"):
            setattr(a, n, rec.wrap(n, getattr(A, n)))
        r = types.ModuleType("CRISPResso2.CRISPRessoCOREResources")
        for n in ("find_indels_substitutions", "find_indels_substitutions_legacy"):
            setattr(r, n, rec.wrap(n, getattr(R, n)))
        r.ResultsSlotsDict = R.ResultsSlotsDict
        pkg = types.ModuleType("CRISPResso2")
        pkg.CRISPResso2Align, pkg.CRISPRessoCOREResources = a, r
        cwd = os.getcwd()
        os.chdir(ref)                                          # the tests read ./CRISPResso2/EDNAFULL
        try:
            with _modules({"CRISPResso2": pkg, "CRISPResso2.CRISPResso2Align": a, "CRISPResso2.CRISPRessoCOREResources": r}):
                mod = _exec(os.path.join(ref, "tests", "unit_tests", test_file), "_ref_" + test_file[:-3])
                entry = {"module": rec.take(), "tests": {}}
                for name, fn in sorted(vars(mod).items()):
                    if name.startswith("test_") and callable(fn):
                        fn()                                  # each must pass against the reference itself
                        entry["tests"][name] = rec.take()
        finally:
            os.chdir(cwd)
        out[test_file] = entry
        print("%s: %d tests, %d calls" % (test_file, len(entry["tests"]), sum(len(v) for v in entry["tests"].values())))
    return out


def consensus_unit(ref, CORE, arrays):
    rec = Recorder(arrays)

    class _Check:                                              # pytest_check.check as a hard assertion
        def __enter__(self):
            return self

        def __exit__(self, *exc):
            return False

        @staticmethod
        def equal(a, b, msg=""):
            assert a == b, (a, b, msg)

        @staticmethod
        def is_true(x, msg=""):
            assert x, msg

        @staticmethod
        def is_false(x, msg=""):
            assert not x, msg

    stubs = {"pytest_check": types.ModuleType("pytest_check"), "inline_snapshot": types.ModuleType("inline_snapshot")}
    stubs["pytest_check"].check = _Check()
    stubs["inline_snapshot"].snapshot = lambda x=None: x
    pkg = types.ModuleType("CRISPResso2")
    A = types.ModuleType("CRISPResso2.CRISPResso2Align")
    A.read_matrix = O.read_matrix
    core = types.ModuleType("CRISPResso2.CRISPRessoCORE")
    core.get_consensus_alignment_from_pairs = rec.wrap("get_consensus_alignment_from_pairs", CORE.get_consensus_alignment_from_pairs)
    pkg.CRISPResso2Align, pkg.CRISPRessoCORE = A, core
    pkg.CRISPRessoShared = types.ModuleType("CRISPResso2.CRISPRessoShared")
    pkg.CRISPRessoCOREResources = types.ModuleType("CRISPResso2.CRISPRessoCOREResources")
    cwd = os.getcwd()
    os.chdir(ref)
    try:
        with _modules({"CRISPResso2": pkg, **stubs}):
            mod = _exec(os.path.join(ref, "tests", "unit_tests", "test_CRISPRessoCORE.py"), "_ref_test_core")
            mod.test_get_consensus_alignment_from_pairs()
    finally:
        os.chdir(cwd)
    calls = rec.take()
    print("consensus unit test: %d calls" % len(calls))
    return calls


def consensus_fuzz(CORE):
    import test_paired_consensus as T
    out = []
    for case in T.fuzz_cases():
        with contextlib.redirect_stdout(io.StringIO()):       # the reference prints when the amplicons disagree
            out.append(G.digest(T.fuzz_answer(CORE.get_consensus_alignment_from_pairs, case)))
    return out


def oracle_fuzz():
    import test_oracle as T
    A, R = O.ref_modules()
    m = np.ascontiguousarray(O.make_matrix())
    keys, out = None, []
    for read, ref, gi, go, ge, inc in T.live_fuzz_cases():
        want = A.global_align(read, ref, matrix=m, gap_incentive=gi, gap_open=go, gap_extend=ge)
        w = R.find_indels_substitutions(want[0], want[1], inc).__dict__
        keys = keys or sorted(w)
        out.append([G.digest(want), T.payload_digest(w, keys)])
    legacy = []
    m = A.make_matrix()
    for read, ref, gi, inc in T.legacy_cases():
        aln = A.global_align(read, ref, matrix=m, gap_incentive=gi, gap_open=-20, gap_extend=-2)
        legacy.append([G.digest(aln), T.legacy_digest(R.find_indels_substitutions_legacy(aln[0], aln[1], inc))])
    return out, keys, legacy


def filter_answers(ref):
    import test_filter_fastqs as T
    mod = _exec(os.path.join(ref, "CRISPResso2", "filterFastqs.py"), "_ref_filterFastqs")
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for inputs, thr, gz in T.reference_calls():
            ext = ".fastq.gz" if gz else ".fastq"
            src = [os.path.join(d, "in%d%s" % (k, ext)) for k in range(len(inputs))]
            dst = [os.path.join(d, "out%d%s" % (k, ext)) for k in range(len(inputs))]
            for p, data in zip(src, inputs):
                T.write(p, data, gz)
            kw = {"fastq_r1": src[0], "fastq_r1_out": dst[0]}
            if len(inputs) == 2:
                kw.update(fastq_r2=src[1], fastq_r2_out=dst[1])
            try:
                with contextlib.redirect_stdout(io.StringIO()):
                    mod.filterFastqs(min_bp_qual_in_read=thr[0], min_av_read_qual=thr[1], min_bp_qual_or_N=thr[2], **kw)
                ans = {"out": [G.digest(T.content(p)) for p in dst]}
            except Exception as ex:
                ans = {"raises": type(ex).__name__}
            out[T.answer_key(inputs, thr, gz)] = ans
    print("filter: %d reference calls" % len(out))
    return out


def main():
    ref = os.path.abspath(sys.argv[1])
    O.build()
    if O.ref_modules() is None:
        raise SystemExit("oracle/_ref is missing: build it with oracle/Makefile (REF=%s)" % ref)
    arrays = {}
    gold = {"matrices": {}}
    for name in ("EDNAFULL", "BLOSUM62"):
        with open(os.path.join(ref, "CRISPResso2", name)) as fh:
            gold["matrices"][name] = fh.read()
    gold["unit_tests"] = unit_tests(ref, arrays)
    import gen_golden as GG                                   # installs the stubs, imports the reference's CRISPRessoCORE
    gold["consensus_unit"] = consensus_unit(ref, GG.CRISPRessoCORE, arrays)
    gold["consensus_fuzz"] = consensus_fuzz(GG.CRISPRessoCORE)
    gold["oracle_fuzz"], gold["oracle_fuzz_keys"], gold["oracle_legacy"] = oracle_fuzz()
    gold["filter"] = filter_answers(ref)
    gold["arrays"] = arrays
    path = os.path.join(TESTS, "golden", "reference_answers.json.gz")
    with gzip.GzipFile(path, "wb", mtime=0) as fh:
        fh.write(json.dumps(gold, sort_keys=True, separators=(",", ":")).encode())
    print("wrote %s (%d bytes)" % (path, os.path.getsize(path)))


if __name__ == "__main__":
    main()

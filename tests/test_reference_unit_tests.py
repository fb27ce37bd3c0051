"""The reference's OWN unit tests for its two native modules (tests/unit_tests/test_CRISPResso2Align.py,
test_CRISPRessoCOREResources.py), replayed against the replacement modules: every call those tests make to
`CRISPResso2Align` / `CRISPRessoCOREResources`, with what the reference's compiled modules returned for it, is stored in
tests/golden/reference_answers.json.gz (tests/golden/gen_reference_answers.py), and the stand-ins exposing
crispresso2_b200.align / .resources on the warp-emulator build of the engine must return the same value or raise the same
exception for each.  All of them must pass (r02: the legacy insertion quantification, `find_indels_substitutions_legacy`,
included)."""
import functools
import os
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))
sys.path.insert(0, HERE)

import golden_util as G  # noqa: E402


def _replacement():
    """-> {name: callable} of the stand-in modules, as the reference's tests would call them."""
    import build_emu
    from crispresso2_b200 import align, resources
    from crispresso2_b200.engine import Engine
    eng = Engine(lib_path=build_emu.build())

    def find(read_al, ref_al, inc):
        a, ed = eng.classify_pair(read_al, ref_al, [int(v) for v in inc])
        return resources.payload_from_device(a, ed, read_al, ref_al)

    def find_legacy(read_al, ref_al, inc):
        a, ed = eng.classify_pair(read_al, ref_al, [int(v) for v in inc], legacy=True)
        return resources.payload_from_device(a, ed, read_al, ref_al, legacy=True)

    return {"read_matrix": align.read_matrix, "make_matrix": align.make_matrix,
            "global_align": functools.partial(align.global_align, engine=eng),
            "find_indels_substitutions": find, "find_indels_substitutions_legacy": find_legacy}


def replay(call, fns, arrays):
    """None when the replacement answers `call` as the reference did, else a description of the difference."""
    args = G.decode_value(call["args"], arrays)
    kwargs = {k: G.decode_value(v, arrays) for k, v in call["kwargs"].items()}
    try:
        got = fns[call["fn"]](*args, **kwargs)
    except Exception as ex:                                   # noqa: BLE001 -- compared with what the reference raised
        if call.get("raises") == type(ex).__name__:
            return None
        return "%s raised %s: %s" % (call["fn"], type(ex).__name__, str(ex)[:120])
    if "raises" in call:
        return "%s returned, the reference raised %s" % (call["fn"], call["raises"])
    if G.digest(got) != call["out"]:
        return "%s%r -> %r" % (call["fn"], tuple(args), got)
    return None


@pytest.mark.parametrize("test_file", ["test_CRISPResso2Align.py", "test_CRISPRessoCOREResources.py"])
def test_reference_unit_tests_pass_against_the_replacement(test_file, tmp_path, monkeypatch):
    gold = G.load_reference_answers()
    rec = gold["unit_tests"][test_file]
    tests = rec["tests"]
    assert len(tests) >= 7
    os.makedirs(tmp_path / "CRISPResso2")                     # the tests read ./CRISPResso2/EDNAFULL and ./CRISPResso2/BLOSUM62
    for name, text in gold["matrices"].items():
        (tmp_path / "CRISPResso2" / name).write_text(text)
    monkeypatch.chdir(tmp_path)
    fns = _replacement()
    for call in rec["module"]:                                # module-level calls (the matrices every test uses)
        assert replay(call, fns, gold["arrays"]) is None, call
    failed = {}
    for name, calls in sorted(tests.items()):
        for call in calls:
            why = replay(call, fns, gold["arrays"])
            if why:
                failed[name] = why
                break
    assert not failed, failed
    print("%s: %d of %d reference tests pass" % (test_file, len(tests) - len(failed), len(tests)))

"""get_consensus_alignment_from_pairs (CRISPRessoCORE.py:829-985), the per-column merge of the paired-end merge mode, natively
(c2b_consensus_from_pairs via crispresso2_b200.paired): the calls of the reference's OWN unit test for it (tests/unit_tests/
test_CRISPRessoCORE.py:27-468) and a differential fuzz on random alignment pairs -- overlapping and disjoint mates, insertions in
one or both, deletions, uncovered stretches, quality ties, leading / trailing gaps, quality strings that are too short
(IndexError on both sides) -- each against what the reference's Python function returned for the same arguments, stored in
tests/golden/reference_answers.json.gz (tests/golden/gen_reference_answers.py).  CPU only."""
import os
import random
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))
sys.path.insert(0, HERE)

import golden_util as G  # noqa: E402
from test_reference_unit_tests import replay  # noqa: E402


@pytest.fixture(scope="module")
def consensus():
    import functools
    import build_emu
    from crispresso2_b200 import paired
    return functools.partial(paired.get_consensus_alignment_from_pairs, lib_path=build_emu.build())


def test_the_references_own_unit_test(consensus):
    gold = G.load_reference_answers()
    calls = gold["consensus_unit"]
    assert len(calls) >= 10
    fns = {"get_consensus_alignment_from_pairs": consensus}
    for call in calls:
        why = replay(call, fns, gold["arrays"])
        assert why is None, why


def _random_alignment(rnd, ref, lo, hi):
    """a mate covering ref[lo:hi] with substitutions, insertions and deletions -> (aligned read, aligned ref, qualities)"""
    s, f = [], []
    for i, c in enumerate(ref):
        if not (lo <= i < hi):
            s.append("-"); f.append(c)
            continue
        u = rnd.random()
        if u < 0.06:
            s.append("-"); f.append(c)                                   # deletion
        elif u < 0.12:
            s.append(rnd.choice("ACGT")); f.append(c)                    # substitution
        else:
            s.append(c); f.append(c)
        if rnd.random() < 0.05:
            for _ in range(rnd.randint(1, 3)):
                s.append(rnd.choice("ACGT")); f.append("-")             # insertion
    if rnd.random() < 0.2:                                              # alignment shorter than the amplicon's columns
        cut = rnd.randint(1, 4)
        s, f = s[:-cut], f[:-cut]
    n_bases = sum(1 for c in s if c != "-")
    q = "".join(rnd.choice("#5I") for _ in range(n_bases))
    return "".join(s), "".join(f), q


def fuzz_cases():
    """The 6000 seeded argument tuples of the differential fuzz."""
    rnd = random.Random(11)
    for it in range(6000):
        L = rnd.randint(8, 60)
        ref = "".join(rnd.choice("ACGT") for _ in range(L))
        a = rnd.randint(0, L // 2)
        b = rnd.randint(a + 1, L)
        c = rnd.randint(0, L - 1)
        d = rnd.randint(c + 1, L)
        s1, f1, q1 = _random_alignment(rnd, ref, a, b)
        s2, f2, q2 = _random_alignment(rnd, ref, c, d)
        if rnd.random() < 0.1:
            q1 = q1[:rnd.randint(0, len(q1))]                            # too short: IndexError on both sides
        if rnd.random() < 0.1:
            q2 += "I" * rnd.randint(1, 5)                               # spare qualities: the gaps of a lone mate consume some
        sc1, sc2 = rnd.choice([(90.0, 80.0), (80.0, 90.0), (85.5, 85.5)])
        yield (s1, f1, sc1, q1, s2, f2, sc2, q2)


def fuzz_answer(fn, case):
    """-> the value `fn` returns for `case`, or "IndexError" """
    try:
        return fn(*case)
    except IndexError:
        return "IndexError"


def test_differential_fuzz_against_the_reference_function(consensus):
    wants = G.load_reference_answers()["consensus_fuzz"]
    assert len(wants) == 6000
    n_ok = n_err = n_nocache = 0
    for case, want in zip(fuzz_cases(), wants):
        got = fuzz_answer(consensus, case)
        assert G.digest(got) == want, (case, got)
        if got == "IndexError":
            n_err += 1
        else:
            n_ok += 1
            n_nocache += not got[4]
    assert n_ok > 3000 and n_err > 100 and n_nocache > 500, (n_ok, n_err, n_nocache)

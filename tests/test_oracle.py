"""Pins the CPU oracle (oracle/) against the reference: restated known-answer tests, golden vectors produced
by the compiled reference (tests/golden/gen_golden.py), and seeded fuzzing against the compiled reference's answers for the
same inputs (tests/golden/gen_reference_answers.py)."""
import gzip
import json
import os
import random

import numpy as np
import pytest

from oracle import oracle as O
import golden_util as G


def Z(n):
    return np.zeros(n, dtype=np.int64)


# ---- known answers restated from /root/reference/tests/unit_tests/test_CRISPResso2Align.py --------------
def test_kat_identity(ednafull):
    assert O.global_align("ATTA", "ATTA", ednafull, Z(5)) == ("ATTA", "ATTA", 100.0)           # :35-40


def test_kat_gap_incentive_sweep(ednafull):                                                  # :139-273
    want = {0: ("ATT-A", "ATTTA"), 1: ("A-TTA", "ATTTA"), 2: ("AT-TA", "ATTTA"), 3: ("ATT-A", "ATTTA"),
            4: ("ATT-A", "ATTTA")}
    for pos in range(5):
        gi = Z(6)
        gi[pos] = 1
        s1, s2, sc = O.global_align("ATTA", "ATTTA", ednafull, gi)
        assert sc == 80.0 and s2 == "ATTTA" and s1.replace("-", "") == "ATTA"
        if pos in (1, 2):
            assert (s1, s2) == want[pos]


def test_kat_n_and_mismatch(ednafull):
    assert O.global_align("ANNG", "ATCG", ednafull, Z(5)) == ("A-NNG", "ATC-G", 40.0)          # :292-300
    assert O.global_align("AAAA", "TTTT", ednafull, Z(5)) == ("---AAAA", "TTTT---", 0.0)      # :324-332
    assert O.global_align("A", "A", ednafull, Z(2)) == ("A", "A", 100.0)                       # :281-289


# ---- known answers restated from test_CRISPRessoCOREResources.py ---------------------------------------
def test_kat_deletions():
    p = O.find_indels_substitutions("-ATTA", "AATTA", [1, 2, 3])                              # :11-17 (shape)
    assert p["all_deletion_positions"] == [0] and p["all_deletion_coordinates"] == [(0, 1)]
    p = O.find_indels_substitutions("AT-TA", "ATTTA", [1, 2])
    assert p["deletion_positions"] == [2] and p["deletion_n"] == 1 and p["ref_positions"] == [0, 1, 2, 3, 4]
    p = O.find_indels_substitutions("ATTT-", "ATTTA", [4])                                     # trailing deletion
    assert p["all_deletion_coordinates"] == [(4, 5)] and p["deletion_sizes"] == [1]


def test_kat_insertions():
    p = O.find_indels_substitutions("ATGGTA", "AT--TA", [1, 2])
    assert p["all_insertion_positions"] == [1, 2] and p["insertion_sizes"] == [2] and p["insertion_n"] == 2
    assert p["ref_positions"] == [0, 1, -2, -2, 2, 3]
    p = O.find_indels_substitutions("GGATTA", "--ATTA", [0, 1])                                # leading: ignored
    assert p["all_insertion_positions"] == [] and p["ref_positions"][:2] == [-1, -1]
    p = O.find_indels_substitutions("ATTAGG", "ATTA--", [2, 3])                                # trailing: ignored
    assert p["all_insertion_positions"] == []


# ---- golden vectors from the compiled reference -----------------------------------------------------------
def test_align_vectors(ednafull):
    with gzip.open(os.path.join(G.GOLD, "align_vectors.json.gz"), "rt") as fh:
        cases = json.load(fh)
    assert len(cases) >= 200
    for c in cases:
        got = O.global_align(c["read"], c["ref"], ednafull, np.array(c["gi"], dtype=np.int64), c["go"], c["ge"])
        assert got == (c["s1"], c["s2"], c["score"]), c
        p = O.find_indels_substitutions(c["s1"], c["s2"], c["inc"])
        assert not G.payload_equal(c["payload"], p), (c, p)


@pytest.mark.parametrize("case", G.CASES)
def test_whole_path_golden(case, ednafull):
    rec = G.load(case)
    refs = G.refs_from(rec)
    params = O.Params(**rec["params"])
    cache, stats, lost = O.process_reads(rec["reads"], refs, rec["ref_names"], params, ednafull)
    assert stats == rec["aln_stats"]
    assert list(cache.keys()) == list(rec["variants"].keys())
    assert set(lost) == set(rec["not_aligned"])
    for s, want in rec["variants"].items():
        got = cache[s]
        for k in ("count", "aln_ref_names", "aln_scores", "best_match_score", "class_name", "best_match_name"):
            assert got[k] == want[k], (s, k)
        assert [list(d) for d in got["ref_aln_details"]] == want["ref_aln_details"]
        for r in want["aln_ref_names"]:
            bad = G.payload_equal(want["variant_" + r], got["variant_" + r])
            assert not bad, (s, r, bad)
    names = list(rec["ref_names"])
    if rec["params"].get("prime_editing_pegRNA_scaffold_seq"):          # the reference main() appends after process_fastq (:3759-3764)
        names.append("Scaffold-incorporated")
        refs["Scaffold-incorporated"] = dict(refs["Prime-edited"])
        assert any(v["class_name"] == "Scaffold-incorporated" for v in cache.values())
    vec, sca, classes, total = O.count_vectors(cache, refs, names, params)
    for r in names:
        seq = refs[r]["sequence"]
        assert G.mod_count_text(seq, vec[r], sca[r]["counts_total"]) == G.file_for(rec, r, "Modification_count_vectors.txt")
        assert G.qw_count_text(seq, vec[r], sca[r]["counts_total"]) == G.file_for(
            rec, r, "Quantification_window_modification_count_vectors.txt")
        nf = G.nuc_freq_rows(G.file_for(rec, r, "Nucleotide_frequency_table.txt"))
        for b in "ACGTN-":
            assert (nf[b] == vec[r]["all_base_count_" + b]).all(), (r, b)


# ---- seeded fuzz against the compiled reference's answers --------------------------------------------------
def live_fuzz_cases():
    """-> (read, ref, gap_incentive, gap_open, gap_extend, include_idxs) of the fuzz, seeded."""
    rng = random.Random(7)
    for _ in range(400):
        I = rng.choice([4, 9, 30, 77, 150])
        ref = "".join(rng.choice("ACGT") for _ in range(I))
        read = "".join(c if rng.random() > 0.08 else rng.choice("ACGTN") for c in ref)
        cut = rng.randrange(I)
        read = read[:cut] + read[cut + rng.randrange(0, 6):] if rng.random() < 0.5 else read[:cut] + "ACG" + read[cut:]
        if len(read) < 3:
            continue
        gi = Z(I + 1)
        gi[rng.randrange(I + 1)] = 1
        go, ge = rng.choice([(-20, -2), (-1, -1), (-7, -3)])
        inc = sorted(rng.sample(range(I), min(I, 3)))
        yield read, ref, gi, go, ge, inc


def payload_digest(p, keys):
    """digest of the payload fields `keys`, compared as golden_util.payload_equal compares them"""
    return G.digest({k: G._norm(p[k]) for k in keys})


def test_live_fuzz_against_compiled_reference(ednafull):
    gold = G.load_reference_answers()
    wants, keys = gold["oracle_fuzz"], gold["oracle_fuzz_keys"]
    m = np.ascontiguousarray(ednafull)
    n = 0
    for (read, ref, gi, go, ge, inc), want in zip(live_fuzz_cases(), wants):
        got = O.global_align(read, ref, m, gi, go, ge)
        assert G.digest(got) == want[0], (read, ref, go, ge, got)
        g = O.find_indels_substitutions(got[0], got[1], inc)
        assert payload_digest(g, keys) == want[1], (got, inc, g)
        n += 1
    assert n == len(wants) > 300


def legacy_cases():
    """-> (read, ref, gap_incentive, include_idxs) of the legacy-classification fuzz, seeded."""
    rng = random.Random(5)
    for _ in range(400):
        I = rng.choice([20, 41, 80, 150])
        ref = "".join(rng.choice("ACGT") for _ in range(I))
        read = list(ref)
        for _k in range(rng.randrange(0, 4)):
            p = rng.randrange(len(read))
            u = rng.random()
            if u < 0.4:
                del read[p:p + rng.randrange(1, 9)]
            elif u < 0.7:
                read[p:p] = [rng.choice("ACGT") for _q in range(rng.randrange(1, 7))]
            else:
                read[p] = rng.choice("ACGTN")
        read = "".join(read)
        if len(read) < 3:
            continue
        gi = np.zeros(I + 1, dtype=np.int64)
        gi[rng.randrange(I + 1)] = 1
        inc = sorted(rng.sample(range(I), rng.randrange(0, min(I, 10))))
        yield read, ref, gi, inc


def legacy_digest(p):
    """digest of a legacy payload: arrays by their elements, every other field by type and value"""
    return G.digest({k: ["nd", G.canon(v.tolist())] if isinstance(v, np.ndarray) else [type(v).__name__, G.canon(v)]
                     for k, v in p.items()})


def test_legacy_classification_restatement_against_compiled_reference():
    """oracle.find_indels_substitutions_legacy (checker for a future device path) == the reference's compiled function on real
    alignments (random reads aligned by global_align, itself checked against the reference's alignment)."""
    wants = G.load_reference_answers()["oracle_legacy"]
    m = O.make_matrix()
    n = 0
    for (read, ref, gi, inc), want in zip(legacy_cases(), wants):
        aln = O.global_align(read, ref, m, gi, -20, -2)
        assert G.digest(aln) == want[0], (read, ref, aln)
        got = O.find_indels_substitutions_legacy(aln[0], aln[1], inc)
        assert legacy_digest(got) == want[1], (aln, inc, got)
        n += 1
    assert n == len(wants) > 300

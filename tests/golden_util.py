"""Helpers shared by the parity tests: fixture loading and the reference's count-vector file layout."""
import gzip
import hashlib
import json
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = ["fanc_cas9", "fanc_params", "synth_single", "synth_hdr", "fanc_pe_scaffold"]


def load(name):
    with gzip.open(os.path.join(GOLD, name + ".json.gz"), "rt") as fh:
        return json.load(fh)


def refs_from(rec):
    refs = {}
    for r, d in rec["refs"].items():
        refs[r] = dict(d)
        refs[r]["gap_incentive"] = np.array(d["gap_incentive"], dtype=np.int64)
        refs[r]["include_idxs"] = np.array(d["include_idxs"], dtype=np.int64)
        refs[r]["sequence_length"] = len(d["sequence"])
    return refs


def _row(name, vals):
    return name + "\t" + "\t".join(str(x) for x in vals) + "\n"


def mod_count_text(seq, V, total):
    """Layout of save_count_vectors_to_file (CRISPRessoCORE.py:4604-4609, rows :4680-4688)."""
    allm = V["all_insertion_count"] + V["all_deletion_count"] + V["all_substitution_count"]
    return ("Sequence\t" + "\t".join(seq) + "\n" + _row("Insertions", V["all_insertion_count"])
            + _row("Insertions_Left", V["all_insertion_left_count"]) + _row("Deletions", V["all_deletion_count"])
            + _row("Substitutions", V["all_substitution_count"]) + _row("All_modifications", allm)
            + _row("Total", [total] * len(seq)))


def qw_count_text(seq, V, total):
    """rows of CRISPRessoCORE.py:4667-4675"""
    allm = V["insertion_count"] + V["deletion_count"] + V["substitution_count"]
    return ("Sequence\t" + "\t".join(seq) + "\n" + _row("Insertions", V["insertion_count"])
            + _row("Deletions", V["deletion_count"]) + _row("Substitutions", V["substitution_count"])
            + _row("All_modifications", allm) + _row("Total", [total] * len(seq)))


def nuc_freq_rows(text):
    """Nucleotide_frequency_table.txt -> {base: float array}"""
    out = {}
    for ln in text.strip("\n").split("\n")[1:]:
        t = ln.split("\t")
        out[t[0]] = np.array([float(x) for x in t[1:]])
    return out


def file_for(rec, ref_name, suffix):
    """Output files carry a '<ref>.' prefix when the run has more than one amplicon."""
    names = [f for f in rec["files"] if f.endswith(suffix)]
    if len(rec["ref_names"]) == 1:
        return rec["files"][suffix]
    for f in names:
        if f == ref_name + "." + suffix:
            return rec["files"][f]
    raise KeyError((ref_name, suffix, names))


def _norm(g):
    if hasattr(g, "tolist"):
        g = g.tolist()
    if isinstance(g, tuple):
        g = list(g)
    if isinstance(g, list):
        g = [list(x) if isinstance(x, tuple) else x for x in g]
    return g


def payload_equal(want, got):
    """Compares two payloads (dict or ResultsSlotsDict-like); returns the list of differing keys."""
    return [k for k, w in want.items() if _norm(got[k]) != _norm(w)]


def load_reference_answers():
    """tests/golden/reference_answers.json.gz: what the reference's own functions returned for the inputs of the tests that
    compare with it (written by tests/golden/gen_reference_answers.py)."""
    return load("reference_answers")


def canon(x):
    """JSON-able form of a returned value that keeps what `==` on the original objects would see: tuple vs list, the dtype
    kind of an array, int vs float vs bool.  Objects with a mapping or attribute interface become their items."""
    if isinstance(x, np.ndarray):
        return {"nd": x.dtype.kind, "v": canon(x.tolist())}
    if isinstance(x, np.generic):
        x = x.item()
    if x is None or isinstance(x, (bool, int, float, str)):
        return x
    if isinstance(x, tuple):
        return {"t": [canon(v) for v in x]}
    if isinstance(x, list):
        return [canon(v) for v in x]
    if isinstance(x, dict):
        return {"d": {str(k): canon(v) for k, v in x.items()}}
    if hasattr(x, "keys"):
        return {"d": {str(k): canon(x[k]) for k in x.keys()}}
    if hasattr(x, "__dict__"):
        return {"d": {str(k): canon(v) for k, v in vars(x).items()}}
    raise TypeError("no canonical form for %r" % type(x))


def digest(x):
    """Short hash of canon(x) (bytes are hashed as they are)."""
    raw = x if isinstance(x, bytes) else json.dumps(canon(x), sort_keys=True).encode()
    return hashlib.sha256(raw).hexdigest()[:16]


def encode_value(x, arrays):
    """canon() that can be decoded back into call arguments; arrays are stored once in `arrays` and referenced by digest."""
    if isinstance(x, np.ndarray):
        key = digest(x.tobytes() + str((x.dtype.str, x.shape)).encode())
        arrays[key] = {"dtype": x.dtype.str, "shape": list(x.shape), "v": x.ravel().tolist()}
        return {"array": key}
    if isinstance(x, tuple):
        return {"t": [encode_value(v, arrays) for v in x]}
    if isinstance(x, list):
        return [encode_value(v, arrays) for v in x]
    if isinstance(x, dict):
        return {"d": {str(k): encode_value(v, arrays) for k, v in x.items()}}
    return canon(x)


def decode_value(x, arrays):
    if isinstance(x, list):
        return [decode_value(v, arrays) for v in x]
    if isinstance(x, dict):
        if "array" in x:
            a = arrays[x["array"]]
            return np.array(a["v"], dtype=np.dtype(a["dtype"])).reshape(a["shape"])
        if "t" in x:
            return tuple(decode_value(v, arrays) for v in x["t"])
        if "d" in x:
            return {k: decode_value(v, arrays) for k, v in x["d"].items()}
    return x

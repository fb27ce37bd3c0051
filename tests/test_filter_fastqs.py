"""Native quality filter (c2b_fastq_filter behind crispresso2_b200.filter_fastqs.filterFastqs) against the reference's own
filterFastqs.filterFastqs (CRISPResso2/filterFastqs.py): byte-identical output text for every combination of the three
thresholds, plain and gzip, CRLF input, truncated files, qualities below '!' (uint8 wrap-around).  What the reference wrote
(a digest of the text) or raised for each input of these tests is stored in tests/golden/reference_answers.json.gz
(tests/golden/gen_reference_answers.py); where the reference itself is broken, a restatement of its record loop stands in."""
import gzip
import hashlib
import itertools
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "emu"))
sys.path.insert(0, HERE)

import golden_util as G  # noqa: E402
from crispresso2_b200 import filter_fastqs  # noqa: E402


@pytest.fixture(scope="module")
def lib():
    import build_emu
    return build_emu.build()


def reference_broken(mbp, mrq, mbpn):
    # min_bp_qual_in_read + min_bp_qual_or_N without the mean filter is broken in the reference itself: run_mBP_mBPN masks a
    # read-only numpy view, filterFastqs.py:191-192, and raises on the first record it keeps -- the restatement stands in there
    return bool(mbp and mbpn and not mrq)


def restated_filter(path_in, path_out, mbp, mrq, mbpn):
    """restatement of filterFastqs.py:128-229 (single-end record loop)"""
    opener = (lambda p: gzip.open(p, "rb")) if path_in.endswith(".gz") else (lambda p: open(p, "rb"))
    out = gzip.open(path_out, "wt") if path_out.endswith(".gz") else open(path_out, "w")
    with opener(path_in) as f, out:
        idl = f.readline().rstrip().decode()
        while idl:
            seq, plus, qual = f.readline().rstrip(), f.readline().rstrip(), f.readline().rstrip()
            q = np.frombuffer(qual, dtype=np.uint8) - 33
            keep = True
            if mbp and not (np.min(q) >= mbp):
                keep = False
            if keep and mrq and not (np.mean(q) >= mrq):
                keep = False
            if keep:
                s = np.frombuffer(seq, "c").copy()
                if mbpn:
                    s[q < mbpn] = b"N"
                out.write("%s\n%s\n%s\n%s\n" % (idl, s.tobytes().decode(), plus.decode(), qual.decode()))
            idl = f.readline().rstrip().decode()


def answer_key(inputs, thr, gz):
    """key of one reference call: the uncompressed input file(s), the three thresholds, plain or gzip"""
    h = hashlib.sha256()
    for data in inputs:
        h.update(hashlib.sha256(data).digest())
    return "%s %r %s" % (h.hexdigest()[:16], tuple(thr), "gz" if gz else "plain")


_ANSWERS = {}


def reference_answer(inputs, thr, gz=False):
    """What the reference's filterFastqs did on these inputs: {"out": [digest of each output's text]} or {"raises": name}."""
    if not _ANSWERS:
        _ANSWERS.update(G.load_reference_answers()["filter"])
    key = answer_key(inputs, thr, gz)
    assert key in _ANSWERS, "no stored reference answer for %s (tests/golden/gen_reference_answers.py)" % key
    return _ANSWERS[key]


def assert_same_as_reference(got_paths, inputs, thr, gz=False):
    want = reference_answer(inputs, thr, gz)
    assert "out" in want, want
    assert [G.digest(content(p)) for p in got_paths] == want["out"], (thr, gz)


def content(path):
    with (gzip.open(path, "rb") if path.endswith(".gz") else open(path, "rb")) as fh:
        return fh.read()


def make_fastq(rng, n, L=60, low=0.08, crlf=False, weird=False):
    recs = []
    for k in range(n):
        seq = "".join(rng.choice(list("ACGT"), L))
        q = rng.integers(20, 41, size=L)
        q[rng.random(L) < low] = rng.integers(0, 15)
        if weird and k % 17 == 0:
            q[0] = -1                                      # ' ' (32): wraps to 255 after the uint8 subtraction
        qual = "".join(chr(33 + int(v)) for v in q)
        recs.append("@read%d extra\n%s\n+\n%s\n" % (k, seq, qual))
    text = "".join(recs)
    if crlf:
        text = text.replace("\n", "\r\n")
    return text.encode()


SINGLE_THRESHOLDS = [t for t in itertools.product([None, 10], [None, 30], [None, 20]) if any(t)]
PAIRED_THRESHOLDS = [t for t in itertools.product([None, 12], [None, 31], [None, 20]) if any(t)]
CRLF_THRESHOLDS = ((None, 25, 20), (None, None, 25), (None, 25, None))
SHORT_MATE_THRESHOLDS = ((None, 25, None), (5, None, None), (5, 25, None))
LARGE_THRESHOLDS = (5, 28, 15)


def single_case(thr):
    return make_fastq(np.random.default_rng(hash(thr) % 1000), 700, weird=True)


def paired_case(thr):
    """two mates of 900 records; every third record has a constant quality ON a threshold"""
    rng = np.random.default_rng(abs(hash(thr)) % 1000 + 7)
    out = []
    for mate in (1, 2):
        recs = make_fastq(rng, 900, L=50, low=0.03).split(b"\n")
        for k in range(0, 900, 3):
            v = 12 if k % 2 else 31
            recs[4 * k + 3] = bytes([33 + v]) * 50
        out.append(b"\n".join(recs))
    return tuple(out)


def short_mate_case():
    rng = np.random.default_rng(21)
    return make_fastq(rng, 40), make_fastq(rng, 25)


def crlf_cases():
    rng = np.random.default_rng(3)
    return {
        "crlf": make_fastq(rng, 50, crlf=True),
        "truncated": make_fastq(rng, 20)[:-35],
        "blank_id_stops": make_fastq(rng, 10) + b"\n" + make_fastq(rng, 10),
        "no_final_newline": make_fastq(rng, 5).rstrip(b"\n"),
    }


def large_case():
    return make_fastq(np.random.default_rng(9), 20000, L=100)


def reference_calls():
    """Every (inputs, thresholds, gzip) the tests below compare with the reference's filterFastqs on."""
    for thr in SINGLE_THRESHOLDS:
        if not reference_broken(*thr):
            for gz in (False, True):
                yield (single_case(thr),), thr, gz
    for thr in PAIRED_THRESHOLDS:
        for gz in (False, True):
            yield paired_case(thr), thr, gz
    for thr in SHORT_MATE_THRESHOLDS:
        yield short_mate_case(), thr, False
    for data in crlf_cases().values():
        for thr in CRLF_THRESHOLDS:
            yield (data,), thr, False
    yield (large_case(),), LARGE_THRESHOLDS, True


def write(path, data, gz):
    with (gzip.open(path, "wb") if gz else open(path, "wb")) as fh:
        fh.write(data)


@pytest.mark.parametrize("gz", [False, True])
@pytest.mark.parametrize("thr", SINGLE_THRESHOLDS)
def test_all_threshold_combinations(lib, tmp_path, thr, gz):
    data = single_case(thr)
    src = str(tmp_path / ("in.fastq.gz" if gz else "in.fastq"))
    write(src, data, gz)
    got = str(tmp_path / ("got.fastq.gz" if gz else "got.fastq"))
    n_in, n_out = filter_fastqs.filterFastqs(fastq_r1=src, fastq_r1_out=got, min_bp_qual_in_read=thr[0], min_av_read_qual=thr[1],
                                             min_bp_qual_or_N=thr[2], lib_path=lib)
    if reference_broken(*thr):
        want = str(tmp_path / ("want.fastq.gz" if gz else "want.fastq"))
        restated_filter(src, want, *thr)
        assert content(got) == content(want)
    else:
        assert_same_as_reference([got], (data,), thr, gz)
    assert n_in == 700 and n_out == content(got).count(b"\n") // 4


@pytest.mark.parametrize("gz", [False, True])
@pytest.mark.parametrize("thr", PAIRED_THRESHOLDS)
def test_paired_all_threshold_combinations(lib, tmp_path, thr, gz):
    """Paired input, every combination of the three thresholds (the seven run_*_pair variants, including the two whose mate-2
    comparison is strict), thresholds chosen so that reads sit exactly ON them; byte-identical output for both mates."""
    ext = ".fastq.gz" if gz else ".fastq"
    inputs = paired_case(thr)
    paths = {}
    for mate in (1, 2):
        paths[mate] = str(tmp_path / ("in_r%d%s" % (mate, ext)))
        write(paths[mate], inputs[mate - 1], gz)
    got = [str(tmp_path / ("got%d%s" % (m, ext))) for m in (1, 2)]
    n_in, n_out = filter_fastqs.filterFastqs(fastq_r1=paths[1], fastq_r2=paths[2], fastq_r1_out=got[0], fastq_r2_out=got[1],
                                             min_bp_qual_in_read=thr[0], min_av_read_qual=thr[1], min_bp_qual_or_N=thr[2], lib_path=lib)
    assert_same_as_reference(got, inputs, thr, gz)
    assert n_in == 900 and n_out == content(got[0]).count(b"\n") // 4 == content(got[1]).count(b"\n") // 4
    assert 0 < n_out


def test_paired_shorter_mate_file_and_default_names(lib, tmp_path):
    """Mate 2 runs out first: its lines read as empty -- with the mean filter the pair is dropped (mean of nothing is nan), with the
    min filter numpy raises; default output names of filterFastqs.py:48-79."""
    inputs = short_mate_case()
    r1, r2 = str(tmp_path / "a_R1.fastq"), str(tmp_path / "a_R2.fastq")
    open(r1, "wb").write(inputs[0])
    open(r2, "wb").write(inputs[1])
    filter_fastqs.filterFastqs(fastq_r1=r1, fastq_r2=r2, min_av_read_qual=25, lib_path=lib)
    assert_same_as_reference([str(tmp_path / "a_R1_filtered.fastq"), str(tmp_path / "a_R2_filtered.fastq")], inputs, (None, 25, None))
    assert reference_answer(inputs, (5, None, None)) == {"raises": "ValueError"}
    with pytest.raises(ValueError):
        filter_fastqs.filterFastqs(fastq_r1=r1, fastq_r2=r2, min_bp_qual_in_read=5, lib_path=lib)
    # min + mean without masking: the mean is tested first, so the short file drops pairs instead of raising (:300)
    filter_fastqs.filterFastqs(fastq_r1=r1, fastq_r2=r2, fastq_r1_out=str(tmp_path / "g1.fastq"), fastq_r2_out=str(tmp_path / "g2.fastq"),
                               min_bp_qual_in_read=5, min_av_read_qual=25, lib_path=lib)
    assert_same_as_reference([str(tmp_path / "g1.fastq"), str(tmp_path / "g2.fastq")], inputs, (5, 25, None))


def test_crlf_truncated_and_blank_id(lib, tmp_path):
    for name, data in crlf_cases().items():
        src = str(tmp_path / (name + ".fastq"))
        open(src, "wb").write(data)
        got = str(tmp_path / (name + "_got.fastq"))
        for thr in CRLF_THRESHOLDS:
            if name == "truncated" and thr[2]:              # last record: quality shorter than the sequence -> IndexError in both
                assert reference_answer((data,), thr) == {"raises": "IndexError"}
                with pytest.raises(IndexError):
                    filter_fastqs.filterFastqs(fastq_r1=src, fastq_r1_out=got, min_bp_qual_in_read=thr[0], min_av_read_qual=thr[1],
                                               min_bp_qual_or_N=thr[2], lib_path=lib)
                continue
            filter_fastqs.filterFastqs(fastq_r1=src, fastq_r1_out=got, min_bp_qual_in_read=thr[0], min_av_read_qual=thr[1],
                                       min_bp_qual_or_N=thr[2], lib_path=lib)
            assert_same_as_reference([got], (data,), thr)


def test_large_multithreaded_and_default_output_name(lib, tmp_path):
    data = large_case()
    src = str(tmp_path / "big.fastq.gz")
    write(src, data, True)
    n_in, n_out = filter_fastqs.filterFastqs(fastq_r1=src, min_bp_qual_in_read=5, min_av_read_qual=28, min_bp_qual_or_N=15,
                                             lib_path=lib, n_threads=6)
    got = str(tmp_path / "big_filtered.fastq.gz")            # filterFastqs.py:50: default output name
    assert os.path.exists(got) and 0 < n_out < n_in == 20000
    assert_same_as_reference([got], (data,), LARGE_THRESHOLDS, True)


def test_error_behaviour(lib, tmp_path):
    src = str(tmp_path / "x.fastq")
    open(src, "wb").write(b"@a\nACGT\n+\nII\n")
    with pytest.raises(IndexError):
        filter_fastqs.filterFastqs(fastq_r1=src, min_bp_qual_or_N=20, lib_path=lib)
    open(src, "wb").write(b"@a\nACGT\n+\n\n")
    with pytest.raises(ValueError):
        filter_fastqs.filterFastqs(fastq_r1=src, min_bp_qual_in_read=20, lib_path=lib)
    with pytest.raises(SystemExit):
        filter_fastqs.filterFastqs(fastq_r1=src, lib_path=lib)
    with pytest.raises(Exception):
        filter_fastqs.filterFastqs(fastq_r1=str(tmp_path / "missing.fastq"), min_av_read_qual=3, lib_path=lib)

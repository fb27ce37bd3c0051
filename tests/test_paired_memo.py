"""crispresso2_b200.paired.AlignmentMemo: the batch that serves process_paired_fastq's global_align calls (CRISPRessoCORE.py:1035-
1053) -- every distinct mate sequence and its reverse complement, forward-only against every amplicon -- must hand out exactly
what global_align returns (the oracle's restatement of CRISPResso2Align.pyx:101-434), for the sequences the paired loop asks for:
mate 1 as read, mate 2 reverse-complemented, and the reverse complements of both.  Arguments that differ from what the batch was
built with (another gap penalty) must not be answered from it.  Kernel logic on the CPU warp emulator."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))

from crispresso2_b200 import paired, synth
from crispresso2_b200.engine import Engine
from oracle import oracle as O

import pe_case


@pytest.fixture(scope="module")
def emu():
    import build_emu
    return Engine(lib_path=build_emu.build())


def test_memo_equals_global_align_for_every_sequence_the_paired_loop_uses(emu, tmp_path):
    rng = np.random.default_rng(8)
    amp = synth.random_amplicon(rng, 223)
    other = amp[:100] + "ACGTTGCA" + amp[100:]
    refs = {"Reference": synth.amplicon_setup(amp), "HDR": synth.amplicon_setup(other)}
    names = ["Reference", "HDR"]
    r1, r2 = str(tmp_path / "R1.fastq"), str(tmp_path / "R2.fastq")
    pe_case.write_pairs(r1, r2, amp, n=60)
    m = O.make_matrix()
    seqs = paired.mate_sequences(r1, r2, lib_path=emu.lib_path)
    memo = paired.AlignmentMemo(emu, seqs, refs, names, m, -20, -2)
    asked = set()
    with open(r1) as f1, open(r2) as f2:
        l1, l2 = f1.read().split("\n"), f2.read().split("\n")
    for k in range(1, len(l1) - 1, 4):
        s1, s2 = l1[k], O.reverse_complement(l2[k])
        asked.update([s1, s2, O.reverse_complement(s1), O.reverse_complement(s2)])
    assert asked <= set(seqs) and len(asked) > 60
    for s in sorted(asked):
        for name in names:
            want = O.global_align(s, refs[name]["sequence"], m, refs[name]["gap_incentive"], -20, -2)
            got = memo.global_align(s, refs[name]["sequence"], matrix=m, gap_incentive=refs[name]["gap_incentive"], gap_open=-20, gap_extend=-2)
            assert tuple(got) == tuple(want), (s, name)
    assert memo.misses == 0 and memo.hits == 2 * len(asked)
    # a call the batch was not built for is not answered from it (here: another gap-extension penalty): it goes to a live call on
    # the default engine, which answers as global_align does on a machine with a GPU and fails on one without
    import torch
    args = (seqs[0], refs["Reference"]["sequence"])
    kw = dict(matrix=m, gap_incentive=refs["Reference"]["gap_incentive"], gap_open=-20, gap_extend=-3)
    if torch.cuda.is_available():
        want = O.global_align(*args, m, refs["Reference"]["gap_incentive"], -20, -3)
        assert tuple(memo.global_align(*args, **kw)) == tuple(want)
    else:
        with pytest.raises(Exception):
            memo.global_align(*args, **kw)
    assert memo.misses == 1

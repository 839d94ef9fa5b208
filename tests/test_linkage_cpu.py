"""CPU: the variant linkage rule of oracle/linkage_oracle.py on crafted reads (every branch of the state rule, the span
limit and pair numbering, the reads that do not count), the refusals, r2 known answers and the binding's layout."""
import numpy as np
import pytest

from helpers import po
from oracle import linkage_oracle as lo

REF = "ACGTTGCAAGGCTTACCGATCAGTACGGTAACTTGCAGCATG" * 3      # 126 letters, A/C/G/T only
OTHER_BASE = {"A": "C", "C": "G", "G": "T", "T": "A"}


def _read(pos, cigar, seq, qual=None, flag=0, mapq=60):
    return po.Read(flag, pos, mapq, cigar, seq, [30] * len(seq) if qual is None else qual)


def _alt(p):
    return {"A": "G", "C": "T", "G": "A", "T": "C"}[REF[p]]


def _states(reads, sites, min_bq=13, min_mapq=0):
    pos = [p for p, _ in sites]
    alt = "".join(a for _, a in sites)
    return lo.read_states(reads, REF, pos, alt, min_bq, min_mapq)


def test_base_states_ref_alt_other_and_quality():
    seq = list(REF[10:40])
    seq[5] = _alt(15)                    # ALT
    seq[7] = OTHER_BASE[REF[17]]         # neither the reference letter nor alt
    if seq[7] == _alt(17):
        seq[7] = OTHER_BASE[seq[7]]
    seq[9] = "N"                         # N is OTHER
    qual = [30] * 30
    qual[11] = 12                        # below min_bq 13: absent
    sites = [(12, _alt(12)), (15, _alt(15)), (17, _alt(17)), (19, _alt(19)), (21, _alt(21))]
    assert _states([_read(10, [(0, 30)], "".join(seq), qual)], sites) == {0: {0: lo.REF, 1: lo.ALT, 2: lo.OTHER,
                                                                            3: lo.OTHER}}
    # the same base at the threshold is present
    qual[11] = 13
    assert _states([_read(10, [(0, 30)], "".join(seq), qual)], sites)[0][4] == lo.REF


def test_absent_outside_the_span_and_in_soft_clips():
    sites = [(5, _alt(5)), (12, _alt(12)), (30, _alt(30)), (45, _alt(45))]
    # 3S20M at 10: the clipped bases are not placed; the span is [10, 30)
    r = _read(10, [(4, 3), (0, 20)], "TTT" + REF[10:30])
    assert _states([r], sites) == {0: {1: lo.REF}}
    # 20M5S at 25: [25, 45); 45 lies in the soft clip
    r = _read(25, [(0, 20), (4, 5)], REF[25:45] + "GGGGG")
    assert _states([r], sites) == {0: {2: lo.REF}}


def test_deletion_entries():
    # 10M 2I 3D 10M at 20: the deletion covers 30..32; resolve_cigar2 gives its entries qpos 12, the first base after the
    # I op -- the quality that decides them, not the inserted bases'
    seq = REF[20:30] + "GG" + REF[33:43]
    sites_del = [(31, "-")]
    sites_base = [(31, _alt(31))]
    for q_after, q_ins, present in ((30, 5, True), (5, 30, False), (13, 0, True), (12, 40, False)):
        qual = [30] * 10 + [q_ins] * 2 + [q_after] + [30] * 9
        r = _read(20, [(0, 10), (1, 2), (2, 3), (0, 10)], seq, qual)
        assert _states([r], sites_del) == ({0: {0: lo.ALT}} if present else {}), (q_after, q_ins)
        assert _states([r], sites_base) == ({0: {0: lo.OTHER}} if present else {}), (q_after, q_ins)


def test_ref_skip_and_deletion_at_the_end():
    r = _read(20, [(0, 5), (3, 10), (0, 5)], REF[20:25] + REF[35:40])
    assert _states([r], [(22, _alt(22)), (28, "-"), (30, _alt(30)), (37, _alt(37))]) == \
        {0: {0: lo.REF, 1: lo.ALT, 2: lo.OTHER, 3: lo.REF}}
    # a deletion that ends the read: qpos is past the end, quality 0
    r = _read(20, [(0, 5), (2, 3)], REF[20:25])
    assert _states([r], [(23, _alt(23)), (26, "-")]) == {0: {0: lo.REF}}
    assert _states([r], [(23, _alt(23)), (26, "-")], min_bq=0) == {0: {0: lo.REF, 1: lo.ALT}}


def test_reads_that_do_not_count():
    sites = [(12, _alt(12)), (15, _alt(15))]
    good = REF[10:30]
    reads = [_read(10, [(0, 20)], good, flag=0x4), _read(10, [(0, 20)], good, flag=0x400),
             _read(10, [(0, 20)], good, flag=0x100), _read(10, [(0, 20)], good, flag=0x200),
             _read(10, [(0, 20)], good, mapq=5), _read(10, [(0, 20)], good, flag=0x1),     # orphan: paired, not proper
             _read(10, [(4, 20)], good)]                                                    # no reference-consuming op
    past_end = _read(110, [(0, 20)], REF[110:] + "A" * 4)
    assert _states(reads + [past_end], sites, min_mapq=10) == {}
    st = _states(reads + [_read(10, [(0, 20)], good, flag=0x3), past_end], sites, min_mapq=10)
    assert st == {7: {0: lo.REF, 1: lo.REF}}
    # the max_depth rule: the third read starting at the same position is not admitted
    reads = [_read(10, [(0, 20)], good) for _ in range(3)]
    assert sorted(lo.read_states(reads, REF, [12], _alt(12), 13, 0, max_depth=2)) == [0, 1]


def test_pairs_span_and_offsets():
    pos = [10, 20, 40, 41, 100]
    assert lo.pairs(pos, 20) == [(0, 1), (1, 2), (2, 3)]
    assert lo.pairs(pos, 21) == [(0, 1), (1, 2), (1, 3), (2, 3)]
    assert lo.pairs(pos, 59) == [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3), (3, 4)]
    for span in (1, 20, 21, 59, 60, 90):
        prs, off = lo.pairs(pos, span), lo.pair_offsets(pos, span)
        assert [off[a] + b - a - 1 for a, b in prs] == list(range(len(prs))), span
    # counts land on their pair, once per read
    alt = "".join(_alt(p) for p in pos)
    seq = list(REF[5:105])
    for p in (20, 41):
        seq[p - 5] = _alt(p)
    reads = [_read(5, [(0, 100)], "".join(seq))] * 2
    c = lo.count_linkage(reads, REF, pos, alt, 21, 13, 0)
    assert c.shape == (4, 3, 3) and int(c.sum()) == 8
    assert c[0, 0, 1] == c[1, 1, 0] == c[2, 1, 1] == c[3, 0, 1] == 2


def test_window_limit_and_refusals():
    dense = [p for p in range(126) if REF[p] in "ACGT"][:65]
    alt = "".join(_alt(p) for p in dense)
    assert lo.window(dense, 64) == 65 and lo.window(dense, 63) == 64
    with pytest.raises(ValueError, match="65 sites"):
        lo.validate(REF, dense, alt, 64)
    lo.validate(REF, dense, alt, 63)
    lo.validate(REF, [], "", 0)                                                  # no sites: counting off
    for pos, alt, span in (([5, 5], "GG", 10), ([6, 5], "AA", 10), ([5], "N", 10), ([5], "g", 10), ([5], REF[5], 10),
                           ([126], "A", 10), ([-1], "A", 10), ([5], _alt(5), 0), ([5], _alt(5), 65536)):
        with pytest.raises(ValueError):
            lo.validate(REF, pos, alt, span)
    with pytest.raises(ValueError, match="reference letter"):
        lo.validate("ACGNA", [3], "A", 10)
    assert lo.validate("acgta", [1], "A", 10) is None                            # the reference letter is upper-cased
    with pytest.raises(ValueError, match="alt equals"):
        lo.validate("acgta", [1], "C", 10)


@pytest.mark.parametrize("counts,want", [
    ([[30, 0, 0], [0, 70, 0], [0, 0, 5]], 1.0),
    ([[0, 30, 4], [70, 0, 0], [0, 0, 0]], 1.0),                  # perfect repulsion
    ([[25, 25, 0], [25, 25, 0], [0, 0, 9]], 0.0),
    ([[40, 10, 0], [10, 40, 0], [0, 0, 0]], 0.36),
    ([[0, 0, 5], [0, 0, 0], [3, 0, 0]], None),                   # n == 0
    ([[10, 20, 0], [0, 0, 0], [0, 0, 0]], None),                 # site a never ALT
    ([[10, 0, 0], [20, 0, 0], [0, 0, 0]], None),                 # site b never ALT
    ([[0, 0, 0], [0, 7, 0], [0, 0, 0]], None),
])
def test_r2_known_answers(counts, want):
    from lvc_b200 import records
    got = records.linkage_r2(counts)
    assert (got is None) if want is None else got == pytest.approx(want, rel=1e-12, abs=1e-15)
    if want is not None:
        assert records.linkage_r2(np.array(counts, dtype=np.uint32)) == pytest.approx(want, rel=1e-12, abs=1e-15)


def test_binding_layout():
    from lvc_b200 import capi
    assert capi.LINKAGE_DTYPE.itemsize == 48
    assert capi.LINKAGE_DTYPE.fields["count"][1] == 12
    names = {s[0] for s in capi.SIGNATURES}
    assert {"lvc_set_linkage_sites", "lvc_copy_linkage"} <= names

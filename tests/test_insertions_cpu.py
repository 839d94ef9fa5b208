"""CPU: the insertion counting and call rules (oracle/insertion_oracle.py, include/lvc.h lvc_insertion_calls) branch by
branch, the splice, and the binding of the new symbols."""
from collections import Counter

import numpy as np
import pytest

from helpers import po
from oracle import insertion_oracle as io

G = 200
Q = 30


def read(pos, cigar, seq=None, qual=None, flag=0, mapq=60):
    ops = po.parse_cigar(cigar)
    lq = sum(n for op, n in ops if op in (0, 1, 4, 7, 8))
    seq = seq if seq is not None else "A" * lq
    qual = qual if qual is not None else [Q] * lq
    assert len(seq) == lq == len(qual)
    return po.Read(flag, pos, mapq, ops, seq, qual)


def counts(reads, min_bq=13, min_mapq=0, max_depth=po.MAX_DEPTH):
    return dict(io.count_insertions(reads, G, min_bq, min_mapq, max_depth))


def test_anchor_after_a_match_op():
    # 5M 3I 5M at 10: anchor 14, bases CGT
    assert counts([read(10, "5M3I5M", "AAAAACGTAAAAA")]) == {(14, 3, io.encode("CGT")): 1}
    for m in ("=", "X"):
        assert counts([read(10, f"5{m}2I5M", "AAAAAGGAAAAA")]) == {(14, 2, io.encode("GG")): 1}
    # P ops and empty ops between the match and the insertion are transparent
    assert counts([read(10, "5M1P2I5M", "AAAAATTAAAAA")]) == {(14, 2, io.encode("TT")): 1}
    assert counts([read(10, "5M0D2I5M", "AAAAATTAAAAA")]) == {(14, 2, io.encode("TT")): 1}
    # an I op after an I op is not anchored on a match
    assert counts([read(10, "5M2I2I5M", "AAAAACCGGAAAAA")]) == {(14, 2, io.encode("CC")): 1}


@pytest.mark.parametrize("cigar,seq", [("5S2I5M", "AAAAACCAAAAA"), ("5M2D2I5M", "AAAAACCAAAAA"),
                                       ("5M2N2I5M", "AAAAACCAAAAA"), ("2I5M", "CCAAAAA"), ("5M0I5M", "AAAAAAAAAA")])
def test_no_match_anchor_counts_nothing(cigar, seq):
    assert counts([read(10, cigar, seq)]) == {}


def test_anchor_quality():
    q = [Q] * 12
    q[4] = 12                                                         # the anchor: below 13
    assert counts([read(10, "5M2I5M", "AAAAACCAAAAA", q)]) == {}
    q[4] = 13
    assert counts([read(10, "5M2I5M", "AAAAACCAAAAA", q)]) == {(14, 2, io.encode("CC")): 1}


def test_unresolved_insertions():
    q = [Q] * 12
    q[6] = 12                                                         # an inserted base below the threshold
    assert counts([read(10, "5M2I5M", "AAAAACCAAAAA", q)]) == {(14, 0, 0): 1}
    assert counts([read(10, "5M2I5M", "AAAAACNAAAAA")]) == {(14, 0, 0): 1}
    assert counts([read(10, "5M2I5M", "AAAAACRAAAAA")]) == {(14, 0, 0): 1}
    ins32, ins33 = "ACGT" * 8, "ACGT" * 8 + "G"
    assert counts([read(10, "5M32I5M", "AAAAA" + ins32 + "AAAAA")]) == {(14, 32, io.encode(ins32)): 1}
    assert counts([read(10, "5M33I5M", "AAAAA" + ins33 + "AAAAA")]) == {(14, 0, 0): 1}
    assert io.decode(io.encode(ins32), 32) == ins32


def test_several_insertions_and_reads():
    reads = [read(10, "3M1I3M2I3M", "AAACAAAGGAAA"), read(10, "3M1I6M", "AAACAAAAAA"), read(12, "1M1I5M", "AAAAAAA")]
    assert counts(reads) == {(12, 1, io.encode("C")): 2, (15, 2, io.encode("GG")): 1, (12, 1, io.encode("A")): 1}


def test_filtered_dropped_and_out_of_range_reads():
    ins = "AAAAACCAAAAA"
    assert counts([read(10, "5M2I5M", ins, flag=0x4)]) == {}                          # unmapped
    assert counts([read(10, "5M2I5M", ins, flag=0x400)]) == {}                        # duplicate
    assert counts([read(10, "5M2I5M", ins, flag=0x1)]) == {}                          # orphan
    assert counts([read(10, "5M2I5M", ins, mapq=5)], min_mapq=20) == {}               # mapping quality
    assert counts([read(10, "5S2I5S", "AAAAACCAAAAA")]) == {}                         # no reference-consuming op
    assert counts([read(G - 5, "5M2I5M", ins)]) == {}                                 # past the contig's end
    assert counts([read(G - 10, "5M2I5M", ins)]) == {(G - 6, 2, io.encode("CC")): 1}  # ends exactly at G
    # max_depth: the third read at the same start is not admitted
    reads = [read(10, "5M2I5M", ins) for _ in range(3)]
    assert counts(reads, max_depth=2) == {(14, 2, io.encode("CC")): 2}


def test_overlap_rewrite_is_seen():
    """the qualities the mate-overlap handling rewrote decide the anchor"""
    a = po.Read(0x1 | 0x2 | 0x20, 10, 60, po.parse_cigar("5M2I5M"), "AAAAACCAAAAA", [Q] * 12, "p", 12, 1, 20)
    b = po.Read(0x1 | 0x2 | 0x10, 12, 60, po.parse_cigar("3M2I5M"), "AAACCAAAAA", [Q] * 10, "p", 10, 1, -20)
    off = io.count_insertions([a, b], G, 13, 0)
    on = io.count_insertions([a, b], G, 13, 0, overlap_model=po.OVERLAP_HTSLIB_1_13)
    assert off == {(14, 2, io.encode("CC")): 2}
    assert on == {(14, 2, io.encode("CC")): 1}                        # the first mate's anchor quality was zeroed


def call(keys, d, letter="A", threshold=0.0):
    """the call rule at one anchor (position 0)"""
    c = Counter({(0, k[0], k[1]) if isinstance(k, tuple) else (0, 0, 0): n for k, n in keys.items()})
    return io.call_insertions(c, [d], letter, threshold)


S1, S2 = (3, io.encode("GAG")), (3, io.encode("GAA"))


def test_call_rule_each_comparison():
    assert call({S1: 6}, 10) == [(0, 3, S1[1], 6, 10)]
    assert call({S1: 5}, 10) == []                                   # count == none (5)
    assert call({S1: 5, S2: 1}, 10) == [(0, 3, S1[1], 5, 10)]         # none = 4
    assert call({S1: 5, S2: 5}, 10) == []                            # tie between resolved keys
    assert call({S1: 5, S2: 4}, 10) == [(0, 3, S1[1], 5, 10)]
    assert call({S1: 4, "u": 4}, 10) == []                           # count == unresolved
    assert call({S1: 5, "u": 4}, 10) == [(0, 3, S1[1], 5, 10)]
    assert call({"u": 9}, 10) == []                                  # unresolved keys are never emitted


def test_call_rule_threshold_and_letters():
    assert call({S1: 7}, 10, threshold=0.7) == [(0, 3, S1[1], 7, 10)]   # 7 / 10 == 0.7
    assert call({S1: 7}, 10, threshold=0.71) == []
    assert call({S1: 7}, 100, threshold=0.07) == []                   # none = 93
    for letter in "N-":
        assert call({S1: 7}, 10, letter) == []
    assert call({S1: 7}, 10, "R") == [(0, 3, S1[1], 7, 10)]


def test_call_rule_min_depth_and_range_through_the_consensus_letters():
    mem = {5: {"reference": "A", "totalDepth": 4, "snvs": {"A": [Q] * 4}, "indels": {}}}
    c = Counter({(5, 1, io.encode("T")): 3})
    for md, want in ((4, 1), (5, 0)):
        depth, letters = io.depth_and_letters_from_memory(mem, 10, md, 0.0)
        assert len(io.call_insertions(c, depth, letters, 0.0)) == want
    depth, letters = io.depth_and_letters_from_memory(mem, 10, 0, 0.0)
    assert io.call_insertions(c, depth, letters, 0.0, 0, 5) == []
    assert io.call_insertions(c, depth, letters, 0.0, 5, 6) == [(5, 1, io.encode("T"), 3, 4)]
    planes = {Q: np.zeros((10, 4), np.uint32)}
    planes[Q][5, 0] = 4
    d2, l2 = io.depth_and_letters_from_tables(planes, np.zeros(10, np.uint32), "A" * 10, 0, 0.0)
    assert list(d2) == list(depth) and l2 == letters


def test_splice_product_and_oracle_agree():
    from lvc_b200 import capi, records
    calls = [(1, 2, io.encode("GT"), 5, 6), (4, 1, io.encode("C"), 5, 6)]
    cons = "AC-TAN"
    want = io.splice(cons, calls)
    assert want == "ACGT-TACN"
    arr = np.array([(p, ln, s, c, d) for p, ln, s, c, d in calls], dtype=capi.INSERTION_DTYPE)
    assert records.splice_insertions(cons, arr[::-1]) == want
    assert records.splice_insertions(cons, arr[:0]) == cons
    assert records.format_consensus_fasta("c", want) == ">c\nACGTTACN\n"


def test_struct_and_binding(lib):
    from lvc_b200 import capi
    assert capi.INSERTION_DTYPE.itemsize == 24
    assert [capi.INSERTION_DTYPE.fields[f][1] for f in ("pos", "len", "seq", "count", "depth")] == [0, 4, 8, 16, 20]
    names = {n for n, _, _ in capi.SIGNATURES}
    for n in ("lvc_enable_insertions", "lvc_copy_insertions", "lvc_insertion_calls"):
        assert n in names and hasattr(lib, n)

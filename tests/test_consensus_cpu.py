"""CPU: the consensus / coverage rule of lvc_consensus (oracle/consensus_oracle.py) on hand-made sites, the two oracle
formulations against each other, the FASTA layout, the statistics struct and the binding of the new symbol."""
import ctypes

import numpy as np
import pytest

import helpers  # noqa: F401  (puts the package and the oracle on sys.path)
from oracle import consensus_oracle as co

GS_TO_NIBBLE = [1, 2, 4, 8, 0, 3, 5, 6, 7, 9, 10, 11, 12, 13, 14, 15]


def site(ref="A", dels=0, other=None, **counts):
    """a memory Site: counts {base: n} of A/C/G/T, `other` {letter: n} of the other codes, `dels` deletion entries"""
    snvs = {b: [30] * n for b, n in counts.items() if n}
    for b, n in (other or {}).items():
        snvs[b] = [20] * n
    return {"reference": ref, "totalDepth": sum(len(q) for q in snvs.values()) + dels, "snvs": snvs, "indels": {}}


def call(s, min_depth=0, threshold=0.0):
    seq, _ = co.consensus_from_memory({0: s}, s["reference"], min_depth, threshold)
    return seq


def test_low_depth_zero_depth_and_min_depth_zero():
    assert call(site(A=5), min_depth=6) == "N"
    assert call(site(A=5), min_depth=5) == "A"
    assert co.consensus_from_memory({}, "A", 0, 0.0)[0] == "N"                 # not in memory: d = 0
    assert call(site(), min_depth=0) == "N"                                     # in memory, every base filtered
    seq, st = co.consensus_from_memory({1: site(C=3)}, "ACG", 0, 0.0)
    assert seq == "NCN" and st["n_low_depth"] == 0 and st["n_N"] == 2
    _, st = co.consensus_from_memory({1: site(C=3)}, "ACG", 4, 0.0)
    assert st["n_low_depth"] == 3 and st["n_N"] == 3


@pytest.mark.parametrize("base", "ACGT")
def test_single_base(base):
    assert call(site(**{base: 7})) == base
    assert call(site(**{base: 7}), threshold=1.0) == base


@pytest.mark.parametrize("bases,letter", [("AC", "M"), ("AG", "R"), ("AT", "W"), ("CG", "S"), ("CT", "Y"), ("GT", "K"),
                                          ("ACG", "V"), ("ACT", "H"), ("AGT", "D"), ("CGT", "B"), ("ACGT", "N")])
def test_every_mask(bases, letter):
    # equal counts: every base is needed to reach a threshold of 1
    assert call(site(**{b: 4 for b in bases}), threshold=1.0) == letter
    assert call(site(**{b: 4 for b in bases}), threshold=0.0) == bases[0]


def test_rank_tie_breaks():
    assert call(site(T=5, G=5)) == "G"
    assert call(site(T=5, C=5, A=2)) == "C"
    assert call(site(A=5, dels=5)) == "A"                                     # A ranks before the deletion
    assert call(site(T=3, dels=3, G=3)) == "G"
    # with a threshold: the tied pair is taken in rank order, the second only if the first is not enough
    assert call(site(T=5, G=5), threshold=0.5) == "G"
    assert call(site(T=5, G=5), threshold=0.51) == "K"


def test_deletion_on_top():
    assert call(site(A=3, dels=6)) == "-"
    assert call(site(A=3, dels=6), threshold=1.0) == "-"
    seq, st = co.consensus_from_memory({0: site(A=3, dels=6)}, "A", 0, 0.0)
    assert st["n_deleted"] == 1 and st["n_mismatch"] == 0


def test_deletion_taken_but_not_on_top_is_not_in_the_mask():
    # A 6, deletion 4, C 2: at 0.9 A, the deletion and C are taken; the mask holds A and C only
    assert call(site(A=6, C=2, dels=4), threshold=0.9) == "M"
    assert call(site(A=6, dels=4), threshold=1.0) == "A"


def test_other_codes_keep_the_threshold_out_of_reach():
    s = site(A=6, other={"N": 4})
    assert s["totalDepth"] == 10
    assert call(s, threshold=0.6) == "A"
    assert call(s, threshold=0.61) == "N"                                      # A..T and deletions hold 60 %
    assert call(site(other={"R": 3})) == "N"                                   # no member at all
    assert call(site(other={"R": 3}, C=1), min_depth=4) == "C"                # nO counts towards the depth


def test_threshold_zero_and_one():
    s = site(A=5, C=3, G=1, T=1)
    assert call(s, threshold=0.0) == "A"
    assert call(s, threshold=0.5) == "A"
    assert call(s, threshold=0.6) == "M"
    assert call(s, threshold=0.9) == "V"
    assert call(s, threshold=1.0) == "N"


def test_division_not_product_at_the_boundary():
    # 7 of 100 reach 0.07 under the division (7 / 100 == 0.07) but not under the product (0.07 * 100 > 7)
    assert 7 / 100 >= 0.07 and not 7 >= 0.07 * 100
    s = site(T=7, other={"N": 93})
    assert call(s, threshold=0.07) == "T"
    tables = _tables_of({0: s}, 1)
    assert co.consensus_from_tables(*tables, "A", 0, 0.07)[0] == "T"


def test_uppercase_and_mismatch_against_a_lowercase_reference():
    mem = {0: site("a", C=4), 1: site("c", C=4), 2: site("n", C=4), 3: site("g", C=2, G=2)}
    seq, st = co.consensus_from_memory(mem, "acng", 0, 0.5)
    assert seq == "CCCC"                                 # position 3: a C/G tie goes to C
    assert st["n_mismatch"] == 2                         # positions 0 and 3; position 2's reference is not A/C/G/T
    seq, st = co.consensus_from_memory(mem, "acng", 0, 0.75)
    assert seq == "CCCS" and st["n_ambiguous"] == 1 and st["n_mismatch"] == 1


def _tables_of(mem, G):
    """memory -> (planes {key: [G, 4]}, dels [G]) the way the device keeps them"""
    planes, dels = {}, np.zeros(G, dtype=np.uint32)
    for p, s in mem.items():
        listed = 0
        for b, quals in s["snvs"].items():
            gs = GS_TO_NIBBLE.index(co.NIBBLE_CHARS.index(b))
            for q in quals:
                key = (gs >> 2) << 8 | q
                planes.setdefault(key, np.zeros((G, 4), dtype=np.uint32))[p, gs & 3] += 1
            listed += len(quals)
        dels[p] = s["totalDepth"] - listed
    return planes, dels


def test_the_two_formulations_agree_on_random_tables():
    rng = np.random.default_rng(20261020)
    G = 3000
    ref = "".join(rng.choice(list("ACGTacgtN"), G))
    mem = {}
    for p in range(G):
        if rng.random() < 0.1:
            continue
        kind = rng.integers(0, 4)
        scale = [0, 3, 30, 300][kind]
        counts = {b: int(rng.integers(0, scale + 1)) if rng.random() < 0.6 else 0 for b in "ACGT"}
        if rng.random() < 0.3:                                     # ties
            counts["G"] = counts["A"]
        other = {c: int(rng.integers(0, 4)) for c in rng.choice(list("=MRSVWYHKDBN"), 2)} if rng.random() < 0.2 else None
        dels = int(rng.integers(0, scale + 1)) if rng.random() < 0.3 else 0
        mem[p] = site(ref[p], dels=dels, other=other, **counts)
    planes, dels = _tables_of(mem, G)
    depths = (1, 10, 20, 100)
    for md in (0, 1, 3, 10):
        for t in (0.0, 0.07, 0.25, 0.5, 0.75, 1.0):
            a = co.consensus_from_memory(mem, ref, md, t, depths)
            b = co.consensus_from_tables(planes, dels, ref, md, t, depths)
            assert a == b, (md, t)
            sub = co.consensus_from_memory(mem, ref, md, t, depths, 1000, 1700)
            assert sub[0] == a[0][1000:1700]
            assert sub == co.consensus_from_tables(planes, dels, ref, md, t, depths, 1000, 1700)
    seq, st = co.consensus_from_memory(mem, ref, 3, 0.75, depths)
    assert {"M", "-", "N"} <= set(seq) and st["n_ambiguous"] > 0 and st["n_mismatch"] > 0


def test_fasta_layout():
    from lvc_b200 import records
    seq = "ACGT" * 20 + "--" + "N" * 41
    text = records.format_consensus_fasta("NC_045512.2", seq)
    lines = text.split("\n")
    assert lines[0] == ">NC_045512.2"
    assert lines[1] == ("ACGT" * 20)[:60] and lines[2] == ("ACGT" * 20)[60:] + "N" * 40 and lines[3] == "N"
    assert lines[4:] == [""] and "-" not in text
    assert records.format_consensus_fasta("c", "-" * 5) == ">c\n"
    assert records.format_consensus_fasta("c", "A" * 60) == ">c\n" + "A" * 60 + "\n"


def test_stats_struct_and_binding(lib):
    from lvc_b200 import capi
    assert ctypes.sizeof(capi.ConsensusStats) == 128
    assert [f[0] for f in capi.ConsensusStats._fields_][:8] == list(co.COUNTERS)
    assert "lvc_consensus" in {n for n, _, _ in capi.SIGNATURES}
    assert hasattr(lib, "lvc_consensus")

"""CPU: the strand-count rule of oracle/strand_oracle.py on crafted reads (every branch), forward + reverse against the
oracle's `memory` on the reference fixture and the synthetic scenarios, the strand-bias statistics against scipy and known
answers, and the opt-in VCF text against a literal fixture."""
import os

import numpy as np
import pytest

from helpers import GOLD, po, synth_small
from oracle import strand_oracle as so

REF = "ACGTTGCAAGGCTTACCGATCAGTACGGTAACTTGCAGCATG" * 3      # 126 letters
G = len(REF)
A, C, GG, T = (so.row_of(x) for x in "ACGT")


def _read(pos, cigar, seq, qual=None, flag=0, mapq=60, name="r"):
    return po.Read(flag, pos, mapq, cigar, seq, [30] * len(seq) if qual is None else qual, name)


def _counts(reads, min_bq=13, min_mapq=0, **kw):
    return so.count_strands(reads, G, min_bq, min_mapq, **kw)


def _nz(t):
    """{(row, col): count} of the non-zero cells"""
    return {(int(r), int(c)): int(t[r, c]) for r, c in zip(*np.nonzero(t))}


def test_forward_and_reverse_reads_and_soft_clips():
    seq = "TTT" + REF[10:20]
    fwd, rev = _counts([_read(10, [(4, 3), (0, 10)], seq)])
    assert not rev.any()
    assert _nz(fwd) == {(so.row_of(REF[p]), p): 1 for p in range(10, 20)}      # the clipped bases are not placed
    fwd, rev = _counts([_read(10, [(4, 3), (0, 10)], seq, flag=0x10)])
    assert not fwd.any()
    assert _nz(rev) == {(so.row_of(REF[p]), p): 1 for p in range(10, 20)}


def test_base_quality_threshold_and_weird_bases():
    seq = list(REF[20:30])
    seq[2], seq[4], seq[6] = "N", "R", "="
    qual = [30] * 10
    qual[1], qual[3] = 12, 13                      # below the threshold, at it
    _, rev = _counts([_read(20, [(0, 10)], "".join(seq), qual, flag=0x10)])
    got = _nz(rev)
    assert (so.row_of(REF[21]), 21) not in got
    assert got[(so.row_of(REF[23]), 23)] == 1
    assert got[(so.row_of("N"), 22)] == 1 and got[(so.row_of("R"), 24)] == 1 and got[(so.row_of("="), 26)] == 1
    assert so.row_of("N") == 15 and so.row_of("=") == 4 and so.row_of("-") == so.DEL == 16
    assert sum(got.values()) == 9


def test_deletions_and_ref_skips():
    # 5M 3D 5M at 30: the deletion's entries take the quality of the query base after it (qpos 5)
    seq = REF[30:35] + REF[38:43]
    for q_after, counted in ((13, True), (12, False)):
        qual = [30] * 10
        qual[5] = q_after
        _, rev = _counts([_read(30, [(0, 5), (2, 3), (0, 5)], seq, qual, flag=0x10)])
        assert [int(rev[so.DEL, p]) for p in (35, 36, 37)] == [int(counted)] * 3
        assert int(rev[so.row_of(REF[38]), 38]) == int(q_after >= 13)        # the base itself follows its own quality
    # a ref skip counts as a deletion entry
    _, rev = _counts([_read(30, [(0, 5), (3, 4), (0, 5)], REF[30:35] + REF[39:44], flag=0x10)])
    assert [int(rev[so.DEL, p]) for p in range(35, 39)] == [1] * 4
    # a deletion as the last op: qpos is past the end of the read, quality 0 -- counted only at threshold 0
    r = _read(30, [(0, 5), (2, 2)], REF[30:35], flag=0x10)
    assert not _counts([r])[1][so.DEL].any()
    assert [int(x) for x in _counts([r], min_bq=0)[1][so.DEL, 35:37]] == [1, 1]


def test_reads_that_do_not_count():
    r = REF[40:50]
    reads = [_read(40, [(0, 10)], r, flag=0x10 | 0x4),            # unmapped
             _read(40, [(0, 10)], r, flag=0x10 | 0x100),          # secondary
             _read(40, [(0, 10)], r, flag=0x10 | 0x400),          # duplicate
             _read(40, [(0, 10)], r, flag=0x10, mapq=5),          # below minMQ
             _read(40, [(0, 10)], r, flag=0x10 | 0x1)]            # orphan: paired, not proper
    assert not any(t.any() for t in _counts(reads, min_mapq=10))
    assert _counts([_read(40, [(0, 10)], r, flag=0x10 | 0x1 | 0x2)], min_mapq=10)[1].sum() == 10      # a proper pair


def test_depth_capped_reads_do_not_count():
    reads = [_read(50, [(0, 10)], REF[50:60], flag=0x10 if k % 2 else 0, name=f"r{k}") for k in range(8)]
    fwd, rev = _counts(reads, max_depth=5)
    p = so.row_of(REF[50])
    # the pileup engine admits the first five reads of this start and drops the rest, reverse reads 5 and 7 among them
    assert (int(fwd[p, 50]), int(rev[p, 50])) == (3, 2)
    assert (int(fwd[p, 50]), int(rev[p, 50])) != tuple(int(x[p, 50]) for x in _counts(reads))


def _memory_check(reads, ref, th, **kw):
    oc = po.OracleCaller(ref, th["minBQ"], th["minMQ"], 1, 1, 0.0, **kw)
    oc.process_reads(reads)
    fwd, rev = so.count_strands(reads, len(ref), th["minBQ"], th["minMQ"], **kw)
    assert np.array_equal(fwd.astype(np.int64) + rev, so.from_memory(oc.memory, len(ref)))
    return int(rev.sum()), int(fwd.sum())


def test_reference_fixture_sums_to_memory(golden_testfile):
    ref = open(os.path.join(GOLD, "NC_045512.2.synthetic.fasta")).read().split("\n", 1)[1].replace("\n", "")
    _, reads = po.read_sam(os.path.join(GOLD, "testfile.sam"))
    total = 0
    for name in ("vc_config", "bq13", "all_zero", "bq13_dp3"):
        th = golden_testfile[name]["thresholds"]
        nr, nf = _memory_check(reads, ref, th, overlap_model=po.OVERLAP_HTSLIB_1_13)
        assert nr == 0                                   # its four reads are all on the forward strand
        total += nf
    assert total > 0


@pytest.mark.parametrize("scen", ["mixed_small", "ont_like", "amplicon_like", "deep_underflow", "maxdepth"])
def test_synthetic_scenarios_sum_to_memory(golden_synth, scen):
    g = golden_synth[scen]
    reads = synth_small.rows_to_reads(g["reads"])
    for tname, res in g["results"].items():
        nr, nf = _memory_check(reads, g["ref"], res["thresholds"])
        if res["thresholds"]["minBQ"] == 0 and nr + nf:
            assert nr > 0 and nf > 0, (scen, tname)


def test_fisher_against_scipy():
    from lvc_b200 import records
    stats = pytest.importorskip("scipy.stats")
    vals = (0, 1, 2, 3, 7, 20, 150, 9990, 10000)
    for a in vals:
        for b in vals:
            for c in (0, 1, 5, 40, 9997):
                for d in (0, 2, 30, 10003):
                    want = stats.fisher_exact([[a, b], [c, d]])[1]
                    got = records.fisher_p(a, b, c, d)
                    if want > 1e-300:
                        assert got == pytest.approx(want, rel=1e-6, abs=1e-300), (a, b, c, d)
                    else:
                        assert got < 1e-290, (a, b, c, d)


def test_fs_and_sor_known_answers():
    from lvc_b200 import records
    # [[4, 6], [5, 0]]: margins 10 / 5 / 9 of 15; P(x) = C(10, x) C(5, 9 - x) / 5005 for x = 4..9 is
    # 210, 1260, 2100, 1200, 225, 10 / 5005; the observed 210 and the 10 are at most it: p = 220 / 5005
    assert records.fisher_p(4, 6, 5, 0) == pytest.approx(220 / 5005, rel=1e-12)
    assert records.fisher_strand(4, 6, 5, 0) == pytest.approx(-10 * np.log10(220 / 5005), rel=1e-12)
    # SOR: t = 5, 7, 6, 1; R = 5 / 42; ln(R + 1 / R) + ln(5 / 7) - ln(1 / 6)
    r = 5 / 42
    assert records.strand_odds_ratio(4, 6, 5, 0) == pytest.approx(np.log(r + 1 / r) + np.log(5 / 7) - np.log(1 / 6), rel=1e-12)
    # no bias: p = 1, FS = 0 (not -0), SOR = ln 2
    assert records.fisher_p(10, 10, 10, 10) == 1.0
    assert str(records.fisher_strand(10, 10, 10, 10)) == "0.0"
    assert records.strand_odds_ratio(0, 0, 0, 0) == pytest.approx(np.log(2))
    # tens of thousands of reads, all ALT on one strand: p underflows a double, FS stays finite
    fs = records.fisher_strand(12000, 0, 0, 9000)
    assert records.fisher_p(12000, 0, 0, 9000) == 0.0 and 6e4 < fs < 7e4
    # symmetric: swapping the strands changes neither statistic
    assert records.fisher_strand(30, 2, 9, 14) == pytest.approx(records.fisher_strand(2, 30, 14, 9), rel=1e-12)
    assert records.strand_odds_ratio(30, 2, 9, 14) == pytest.approx(records.strand_odds_ratio(2, 30, 14, 9), rel=1e-12)


def _two_records():
    return [{"start": 9, "stop": 10, "alleles": ("A", "G"), "qual": 0.000316227766, "info":
             {"DP": 70, "AD": 60, "GL": -35.00824146158652, "PL": 350, "SCORE": 99}},
            {"start": 9, "stop": 10, "alleles": ("A", "T"), "qual": 0.001, "info":
             {"DP": 70, "AD": 5, "GL": 0, "PL": 0, "SCORE": 0}}]


def test_opt_in_vcf_against_literal_fixture():
    """tests/golden/expected_two_records_strand.vcf, reviewed by hand: the two records of expected_two_records.vcf with
    DP4 4,6,50,10 and 4,6,5,0; FS 21.459 / 13.570 (p = 0.0071472 / 220/5005), SOR 3.091 / 3.598"""
    from lvc_b200 import records
    v = _two_records()
    sb = [records.strand_row(v[0], (4, 6, 50, 10)), records.strand_row(v[1], (4, 6, 5, 0))]
    txt = records.format_vcf(v, [("NC_045512.2", 29903)], sb)
    with open(os.path.join(GOLD, "expected_two_records_strand.vcf")) as fh:
        assert txt == fh.read()
    # a record without counts (REF letter not a nibble code) keeps the plain INFO
    sb[1] = records.strand_row(v[1], None)
    assert sb[1]["fs"] is None and sb[1]["ref_fwd"] is None
    lines = records.format_vcf(v, [("NC_045512.2", 29903)], sb).strip().split("\n")
    assert lines[-2] == "NC_045512.2\t10\t.\tA\tT\t0.001\t.\tDP=70;AD=5;GL=0;PL=0;SCORE=0"


def test_default_vcf_unchanged():
    from lvc_b200 import records
    with open(os.path.join(GOLD, "expected_two_records.vcf")) as fh:
        assert records.format_vcf(_two_records(), [("NC_045512.2", 29903)]) == fh.read()
        fh.seek(0)
        assert records.format_vcf(_two_records(), [("NC_045512.2", 29903)], None) == fh.read()

"""Host finalisation: device candidates -> the reference's Variant dicts and VCF text.

Only the few emitted (position, allele) candidates reach this code.  log10 / round / formatting use
the host libm and Python's banker's rounding so the text matches the reference (SURVEY A6):
live_variant_caller.py:158-185 (record), :233-297 (VCF), utils.py:12-13 (to_phred_scale).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

NIBBLE_CHARS = "=ACMGRSVTWYHKDBN"


def phred_luts() -> Tuple[np.ndarray, np.ndarray]:
    """e[q] = math.pow(10, q / -10) (utils.py:9-10) and 1.0 - e[q], built with the HOST libm.
    CUDA/NumPy pow differ from math.pow in the last bit at a few q (SURVEY A6), so the tables are
    uploaded rather than recomputed on the device."""
    e = np.array([math.pow(10, q / -10) for q in range(256)], dtype=np.float64)
    return e, (1.0 - e)


def to_phred_scale(probability: float, threshold: int = 99) -> int:
    """utils.py:12-13."""
    return min(round(-10 * math.log10(probability)), threshold) if probability > 0.0 else threshold


def candidates_to_variants(cands: np.ndarray) -> List[dict]:
    """Build the Variant dicts of prepare_variants (live_variant_caller.py:170-185).

    Order: ascending position (dict insertion order of `memory` for a coordinate-sorted BAM), and
    within a position the first-seen order of the alleles (SURVEY A7)."""
    order = np.lexsort((cands["first"], cands["pos"]))
    out = []
    for c in cands[order]:
        L, S = float(c["L"]), float(c["S"])
        if L != 0:
            gl = math.log10(L)
            pl = round(-10.0 * gl)
        else:
            gl, pl = 0, 0
        score = to_phred_scale(1.0 - (L / S))
        ad = int(c["ad"])
        out.append({
            "start": int(c["pos"]),
            "stop": int(c["pos"]) + 1,
            "alleles": (chr(int(c["ref"])), NIBBLE_CHARS[int(c["code"])]),
            "qual": np.float64(float(c["esum"]) / ad),
            "info": {"DP": int(c["dp"]), "AD": ad, "GL": gl, "PL": pl, "SCORE": score},
        })
    return out


def fmt_g_float32(x) -> str:
    """htslib kputd of a float32 field: C '%g' of the value after rounding to float32 [EXT A8]."""
    return "%g" % float(np.float32(x))


VCF_INFO_META = [
    ("DP", "Integer", "Total Depth"),
    ("AD", "Integer", "Allele Depth"),
    ("GL", "Float", "Genotype likelihoods comprised of comma separated floating point log10-scaled likelihoods "
                    "for all possible genotypes given the set of alleles defined in the REF and ALT fields"),
    ("PL", "Integer", "The phred-scaled genotype likelihoods rounded to the closest integer (and otherwise defined "
                      "precisely as the GL field)"),
    ("SCORE", "Float", "Custom scoring function"),
]


# the INFO metas write_vcf(strandBias=True) adds after VCF_INFO_META
VCF_STRAND_META = [
    ("DP4", "4", "Integer", "Reference-forward, reference-reverse, alternate-forward and alternate-reverse entries counted "
                            "in DP"),
    ("FS", "1", "Float", "Phred-scaled p-value of the two-sided Fisher exact test on the DP4 table (strand bias)"),
    ("SOR", "1", "Float", "Symmetric odds ratio of the DP4 table with pseudocounts of 1 (strand bias)"),
]


def format_vcf(variants: List[dict], contigs: Sequence[Tuple[str, int]], strand: Optional[List[dict]] = None) -> str:
    """VCF 4.2 text the way pysam/htslib writes the reference's records (live_variant_caller.py:235-295):
    INFO metas DP, AD, GL, PL, SCORE; one ##contig per FASTA contig; records stably sorted by
    (start, SCORE); CHROM = first header contig (new_record is called without a contig).
    `strand`: the strand_bias rows of `variants`, in their order.  With them the header gains the VCF_STRAND_META lines and
    the INFO of every record with counts gains DP4, FS and SOR (3 decimals); without them the text is unchanged."""
    lines = ["##fileformat=VCFv4.2", '##FILTER=<ID=PASS,Description="All filters passed">']
    for vid, typ, desc in VCF_INFO_META:
        lines.append(f'##INFO=<ID={vid},Number=1,Type={typ},Description="{desc}">')
    if strand is not None:
        if len(strand) != len(variants):
            raise ValueError(f"{len(strand)} strand rows for {len(variants)} records")
        for vid, num, typ, desc in VCF_STRAND_META:
            lines.append(f'##INFO=<ID={vid},Number={num},Type={typ},Description="{desc}">')
    for name, length in contigs:
        lines.append(f"##contig=<ID={name},length={length}>")
    lines.append("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO")
    chrom = contigs[0][0]
    order = sorted(range(len(variants)), key=lambda k: (variants[k]["start"], variants[k]["info"]["SCORE"]))
    for k in order:
        v = variants[k]
        i = v["info"]
        line = (f'{chrom}\t{v["start"] + 1}\t.\t{v["alleles"][0]}\t{v["alleles"][1]}\t{fmt_g_float32(v["qual"])}'
                f'\t.\tDP={i["DP"]};AD={i["AD"]};GL={fmt_g_float32(i["GL"])};PL={i["PL"]};'
                f'SCORE={fmt_g_float32(i["SCORE"])}')
        if strand is not None and strand[k]["ref_fwd"] is not None:
            sb = strand[k]
            line += (f';DP4={sb["ref_fwd"]},{sb["ref_rev"]},{sb["alt_fwd"]},{sb["alt_rev"]}'
                     f';FS={sb["fs"]:.3f};SOR={sb["sor"]:.3f}')
        lines.append(line)
    return "\n".join(lines) + "\n"


# ---------------------------------------------------------------------------------------------------------------------
# strand bias
# ---------------------------------------------------------------------------------------------------------------------
_LN10 = math.log(10.0)


def _log_choose(n: int, k: int) -> float:
    return math.lgamma(n + 1) - math.lgamma(k + 1) - math.lgamma(n - k + 1)


def fisher_log_p(ref_fwd: int, ref_rev: int, alt_fwd: int, alt_rev: int) -> float:
    """natural log of the two-sided Fisher exact p-value of the 2x2 table [[ref_fwd, ref_rev], [alt_fwd, alt_rev]]: the sum
    of the hypergeometric probabilities (margins fixed) that are <= the observed one x (1 + 1e-7), at most 1.  Computed in
    log space, so tables of tens of thousands of reads do not underflow."""
    a, b, c, d = int(ref_fwd), int(ref_rev), int(alt_fwd), int(alt_rev)
    r1, r2, c1 = a + b, c + d, a + c
    n = r1 + r2
    lo, hi = max(0, c1 - r2), min(r1, c1)
    base = -_log_choose(n, c1)

    def lp(x):
        return _log_choose(r1, x) + _log_choose(r2, c1 - x) + base

    cut = lp(a) + math.log1p(1e-7)
    terms = [t for t in (lp(x) for x in range(lo, hi + 1)) if t <= cut]
    m = max(terms)
    return min(0.0, m + math.log(sum(math.exp(t - m) for t in terms)))


def fisher_p(ref_fwd: int, ref_rev: int, alt_fwd: int, alt_rev: int) -> float:
    """two-sided Fisher exact p-value (fisher_log_p); 0.0 where it is below the smallest double"""
    return math.exp(fisher_log_p(ref_fwd, ref_rev, alt_fwd, alt_rev))


def fisher_strand(ref_fwd: int, ref_rev: int, alt_fwd: int, alt_rev: int) -> float:
    """FS = -10 log10(fisher_p), from the log p-value (finite for any counts)"""
    return -10.0 * fisher_log_p(ref_fwd, ref_rev, alt_fwd, alt_rev) / _LN10 + 0.0


def strand_odds_ratio(ref_fwd: int, ref_rev: int, alt_fwd: int, alt_rev: int) -> float:
    """GATK's StrandOddsRatio: with t00, t01, t10, t11 = ref_fwd, ref_rev, alt_fwd, alt_rev each + 1 and
    R = (t00 t11) / (t01 t10), SOR = ln(R + 1/R) + ln(min(t00, t01) / max(t00, t01)) - ln(min(t10, t11) / max(t10, t11))"""
    t00, t01, t10, t11 = int(ref_fwd) + 1, int(ref_rev) + 1, int(alt_fwd) + 1, int(alt_rev) + 1
    r = (t00 * t11) / (t01 * t10)
    return math.log(r + 1.0 / r) + math.log(min(t00, t01) / max(t00, t01)) - math.log(min(t10, t11) / max(t10, t11))


def strand_row(v: dict, counts: Optional[Tuple[int, int, int, int]]) -> dict:
    """one row of LiveVariantCaller.strand_bias: the record's start and alleles, its DP4 counts and the statistics (all
    None without counts)"""
    row = {"start": v["start"], "alleles": v["alleles"]}
    if counts is None:
        row.update(ref_fwd=None, ref_rev=None, alt_fwd=None, alt_rev=None, fisher_p=None, fs=None, sor=None)
        return row
    rf, rr, af, ar = (int(x) for x in counts)
    row.update(ref_fwd=rf, ref_rev=rr, alt_fwd=af, alt_rev=ar, fisher_p=fisher_p(rf, rr, af, ar),
               fs=fisher_strand(rf, rr, af, ar), sor=strand_odds_ratio(rf, rr, af, ar))
    return row


def format_site_csv(depth: np.ndarray, ad: np.ndarray, ref: str) -> str:
    """README.md:4-8 of the reference sketches a per-position table POS, REF, DEPTH, A, A%, ...; the
    reference never writes it.  Additive output, not a parity target."""
    rows = ["POS,REF,DEPTH,A,A%,C,C%,G,G%,T,T%"]
    for p in np.nonzero(depth)[0]:
        d = int(depth[p])
        cells = []
        for k in range(4):
            n = int(ad[p, k])
            cells += [str(n), "%.4f" % (n / d)]
        rows.append(f"{p + 1},{ref[p]},{d}," + ",".join(cells))
    return "\n".join(rows) + "\n"


def format_consensus_fasta(contig: str, consensus: str, width: int = 60) -> str:
    """FASTA of a consensus (LiveVariantCaller.consensus): header `>contig`, the deletion calls '-' removed, `width`
    letters per line."""
    seq = consensus.replace("-", "")
    return f">{contig}\n" + "".join(seq[i:i + width] + "\n" for i in range(0, len(seq), width))


def decode_insertion(seq: int, length: int) -> str:
    """lvc_insertion.seq (2-bit codes A, C, G, T = 0..3, base k in bits 2k) -> the inserted bases"""
    return "".join("ACGT"[(int(seq) >> (2 * k)) & 3] for k in range(int(length)))


def splice_insertions(consensus: str, calls) -> str:
    """`consensus` (one letter per reference position) with each called insertion (INSERTION_DTYPE rows, positions
    relative to the consensus's first letter) placed after the letter of its anchor"""
    out, last = [], 0
    for c in sorted(calls, key=lambda c: int(c["pos"])):
        p = int(c["pos"]) + 1
        out.append(consensus[last:p])
        out.append(decode_insertion(c["seq"], c["len"]))
        last = p
    out.append(consensus[last:])
    return "".join(out)


def linkage_r2(counts) -> Optional[float]:
    """r^2 of two sites from the REF/ALT 2x2 of a linkage pair's 3x3 counts (count[state_a][state_b], REF 0, ALT 1):
    n = n00 + n01 + n10 + n11, pa = (n10 + n11) / n, pb = (n01 + n11) / n, D = n11 / n - pa * pb,
    r2 = D^2 / (pa (1 - pa) pb (1 - pb)); None when n == 0 or the denominator is 0"""
    n00, n01, n10, n11 = (int(counts[a][b]) for a, b in ((0, 0), (0, 1), (1, 0), (1, 1)))
    if n00 + n01 + n10 + n11 == 0:
        return None
    # the same in integers (D = (n00 n11 - n01 n10) / n^2, pa (1 - pa) = (n10 + n11)(n00 + n01) / n^2, ...), so that
    # perfect linkage gives exactly 1.0
    den = (n10 + n11) * (n00 + n01) * (n01 + n11) * (n00 + n10)
    if den == 0:
        return None
    return (n00 * n11 - n01 * n10) ** 2 / den

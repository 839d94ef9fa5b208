"""Host finalisation: device candidates -> the reference's Variant dicts and VCF text.

Only the few emitted (position, allele) candidates reach this code.  log10 / round / formatting use
the host libm and Python's banker's rounding so the text matches the reference (SURVEY A6):
live_variant_caller.py:158-185 (record), :233-297 (VCF), utils.py:12-13 (to_phred_scale).
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence, Tuple

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


def format_vcf(variants: List[dict], contigs: Sequence[Tuple[str, int]]) -> str:
    """VCF 4.2 text the way pysam/htslib writes the reference's records (live_variant_caller.py:235-295):
    INFO metas DP, AD, GL, PL, SCORE; one ##contig per FASTA contig; records stably sorted by
    (start, SCORE); CHROM = first header contig (new_record is called without a contig)."""
    lines = ["##fileformat=VCFv4.2", '##FILTER=<ID=PASS,Description="All filters passed">']
    for vid, typ, desc in VCF_INFO_META:
        lines.append(f'##INFO=<ID={vid},Number=1,Type={typ},Description="{desc}">')
    for name, length in contigs:
        lines.append(f"##contig=<ID={name},length={length}>")
    lines.append("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO")
    chrom = contigs[0][0]
    for v in sorted(variants, key=lambda v: (v["start"], v["info"]["SCORE"])):
        i = v["info"]
        lines.append(f'{chrom}\t{v["start"] + 1}\t.\t{v["alleles"][0]}\t{v["alleles"][1]}\t{fmt_g_float32(v["qual"])}'
                     f'\t.\tDP={i["DP"]};AD={i["AD"]};GL={fmt_g_float32(i["GL"])};PL={i["PL"]};'
                     f'SCORE={fmt_g_float32(i["SCORE"])}')
    return "\n".join(lines) + "\n"


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

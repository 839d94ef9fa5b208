"""CPU ORACLE (test infrastructure) of the strand counts of ``lvc_enable_strand_counts`` / ``lvc_strand_counts``
(include/lvc.h), written as the rule reads.

Which reads count: the reads the pileup engine admits (``pileup_oracle.pileup_columns``) that lie inside [0, G) and whose
flag has 0x10 (reverse strand).

What they count: every pileup entry at column p that passes the base-quality test of ``OracleCaller.process_reads``
(qual[qpos], 0 if qpos is past the end of the read; for a deletion or ref-skip entry qpos is the one resolve_cigar2 gives),
i.e. every entry the reference adds to totalDepth.  A base adds 1 to rev[gs][p], gs the plane slot of its BAM nibble
(group << 2 | slot: A, C, G, T = 0..3, then the other nibble codes in ascending order); a deletion or ref-skip entry adds 1
to rev[16][p].  The forward counts are the same sums over the forward reads, so fwd + rev is what the reference's `memory`
holds: len(snvs[base]) per base, and totalDepth minus the bases for the deletions.
"""
from __future__ import annotations

from typing import Sequence, Tuple

import numpy as np

from . import pileup_oracle as po

ROWS = 17                                                       # 16 allele slots, then deletions
DEL = 16
GS_TO_NIBBLE = [1, 2, 4, 8, 0, 3, 5, 6, 7, 9, 10, 11, 12, 13, 14, 15]
NIBBLE_TO_GS = {n: gs for gs, n in enumerate(GS_TO_NIBBLE)}


def row_of(letter: str) -> int:
    """the table row of an allele letter: a nibble letter (either case) or '-'"""
    if letter == "-":
        return DEL
    return NIBBLE_TO_GS[po.CHAR_TO_NIBBLE[letter.upper()]]


def count_strands(reads: Sequence[po.Read], G: int, min_bq: int, min_mapq: int, max_depth: int = po.MAX_DEPTH,
                  overlap_model: int = po.OVERLAP_OFF) -> Tuple[np.ndarray, np.ndarray]:
    """(fwd, rev), uint32 [17, G] each: the counted entries of forward and of reverse reads"""
    out = np.zeros((2, ROWS, G), dtype=np.uint32)
    for col, entries in po.pileup_columns(list(reads), min_mapq, max_depth, overlap_model=overlap_model):
        for _idx, r, is_del, is_skip, qpos in entries:
            if r.pos < 0 or r.pos + r.ref_len() > G:                  # the deposit skips it (LVC_ERANGE)
                continue
            q = r.qual[qpos] if qpos < len(r.qual) else 0
            if q < min_bq:
                continue
            row = DEL if (is_del or is_skip) else NIBBLE_TO_GS[po.CHAR_TO_NIBBLE.get(r.seq[qpos], 15)]
            out[1 if r.flag & 0x10 else 0, row, col] += 1
    return out[0], out[1]


def from_memory(memory: dict, G: int) -> np.ndarray:
    """uint32 [17, G]: the counts of the reference's `memory` per allele row (bases) and deletions (totalDepth minus
    the bases): what fwd + rev must equal"""
    out = np.zeros((ROWS, G), dtype=np.uint32)
    for p, site in memory.items():
        n_bases = 0
        for base, quals in site["snvs"].items():
            out[NIBBLE_TO_GS[po.CHAR_TO_NIBBLE[base]], p] += len(quals)
            n_bases += len(quals)
        out[DEL, p] = site["totalDepth"] - n_bases
    return out

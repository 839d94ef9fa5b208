"""CPU ORACLE (test infrastructure) of the variant linkage counts of ``lvc_set_linkage_sites`` / ``lvc_copy_linkage``
(include/lvc.h), written as the rules read.

Sites: (pos, alt) with pos 0-based, strictly ascending, inside [0, G); alt one of 'A' 'C' 'G' 'T' '-' ('-' = a
deletion); the reference letter at pos, upper-cased, is A/C/G/T and differs from alt.  A pair is two sites a < b with
pos_b - pos_a <= max_span; pairs are numbered in (a, b) order (pair (a, b) = off[a] + b - a - 1, off the exclusive prefix
sum of the partner counts).  At most 64 sites may lie inside any window of max_span + 1 positions.

Which reads count: the reads the pileup engine admits (``pileup_oracle.pileup_columns``) that lie inside [0, G).

State of a site on a read, from the read's pileup entry at pos (``pileup_columns``) and the base-quality test of
``OracleCaller.process_reads`` (qual[qpos], 0 if qpos is past the end of the read; for a deletion or ref-skip entry qpos
is the one resolve_cigar2 gives):
  absent     no entry, or the entry fails the quality test;
  REF   (0)  the base is the reference letter;
  ALT   (1)  the base is alt, or the entry is a deletion / ref-skip and alt is '-';
  OTHER (2)  anything else.
Every pair whose two sites are present on a read adds 1 to count[state_a][state_b].
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import numpy as np

from . import pileup_oracle as po

REF, ALT, OTHER = 0, 1, 2
MAX_SITES = 1 << 20
MAX_WINDOW = 64


def window(pos: Sequence[int], max_span: int) -> int:
    """the most sites inside any window of max_span + 1 positions"""
    w, a = 0, 0
    for k in range(len(pos)):
        while pos[k] - pos[a] > max_span:
            a += 1
        w = max(w, k - a + 1)
    return w


def validate(ref: str, pos: Sequence[int], alt: str, max_span: int) -> None:
    """the refusals of lvc_set_linkage_sites, as ValueError"""
    if len(pos) > MAX_SITES:
        raise ValueError(f"{len(pos)} sites, at most 2^20")
    if not pos:
        return
    if not 1 <= max_span <= 65535:
        raise ValueError(f"max_span {max_span} outside 1..65535")
    for k, (p, a) in enumerate(zip(pos, alt)):
        if not 0 <= p < len(ref):
            raise ValueError(f"site {k} at {p} outside [0, {len(ref)})")
        if k and p <= pos[k - 1]:
            raise ValueError(f"positions not strictly ascending at site {k}")
        if a not in "ACGT-":
            raise ValueError(f"site {k}: alt {a!r}")
        if ref[p].upper() not in "ACGT":
            raise ValueError(f"site {k}: reference letter {ref[p]!r}")
        if ref[p].upper() == a:
            raise ValueError(f"site {k}: alt equals the reference letter")
    w = window(pos, max_span)
    if w > MAX_WINDOW:
        raise ValueError(f"{w} sites inside a window of {max_span + 1} positions")


def pairs(pos: Sequence[int], max_span: int) -> List[Tuple[int, int]]:
    """every pair (a, b) in pair-index order"""
    return [(a, b) for a in range(len(pos)) for b in range(a + 1, len(pos)) if pos[b] - pos[a] <= max_span]


def pair_offsets(pos: Sequence[int], max_span: int) -> List[int]:
    """off[a]: the index of pair (a, a + 1); pair (a, b) is off[a] + b - a - 1"""
    off, n = [], 0
    for a in range(len(pos)):
        off.append(n)
        n += sum(1 for b in range(a + 1, len(pos)) if pos[b] - pos[a] <= max_span)
    return off


def entry_state(read: po.Read, is_del: bool, is_skip: bool, qpos: int, ref_letter: str, alt: str, min_bq: int):
    """the state of one pileup entry (None: absent); `read` carries the qualities the entry is tested with"""
    q = read.qual[qpos] if qpos < len(read.qual) else 0
    if q < min_bq:
        return None
    if is_del or is_skip:
        return ALT if alt == "-" else OTHER
    base = read.seq[qpos]
    return REF if base == ref_letter.upper() else ALT if base == alt else OTHER


def read_states(reads: Sequence[po.Read], ref: str, pos: Sequence[int], alt: str, min_bq: int, min_mapq: int,
                max_depth: int = po.MAX_DEPTH, overlap_model: int = po.OVERLAP_OFF) -> Dict[int, Dict[int, int]]:
    """{read index: {site index: state}} over the reads that count, present sites only"""
    reads = list(reads)
    G = len(ref)
    at = {p: k for k, p in enumerate(pos)}
    states: Dict[int, Dict[int, int]] = {}
    for col, entries in po.pileup_columns(reads, min_mapq, max_depth, overlap_model=overlap_model):
        k = at.get(col)
        if k is None:
            continue
        for idx, r, is_del, is_skip, qpos in entries:
            if r.pos < 0 or r.pos + r.ref_len() > G:              # the deposit skips it (LVC_ERANGE)
                continue
            st = entry_state(r, is_del, is_skip, qpos, ref[col], alt[k], min_bq)
            if st is not None:
                states.setdefault(idx, {})[k] = st
    return states


def count_linkage(reads: Sequence[po.Read], ref: str, pos: Sequence[int], alt: str, max_span: int, min_bq: int,
                  min_mapq: int, max_depth: int = po.MAX_DEPTH, overlap_model: int = po.OVERLAP_OFF) -> np.ndarray:
    """uint32 [n_pairs, 3, 3] in pair-index order"""
    validate(ref, pos, alt, max_span)
    prs = pairs(pos, max_span)
    index = {p: j for j, p in enumerate(prs)}
    out = np.zeros((len(prs), 3, 3), dtype=np.uint32)
    for st in read_states(reads, ref, pos, alt, min_bq, min_mapq, max_depth, overlap_model).values():
        present = sorted(st)
        for i, a in enumerate(present):
            for b in present[i + 1:]:
                j = index.get((a, b))
                if j is not None:
                    out[j, st[a], st[b]] += 1
    return out

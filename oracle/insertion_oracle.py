"""CPU ORACLE (test infrastructure) of the insertion counts and calls of ``lvc_copy_insertions`` /
``lvc_insertion_calls`` (include/lvc.h), written as the rules read.

Counting rule: the reads the pileup engine admits (``pileup_oracle.pileup_columns(admitted=...)``), with the qualities
the mate-overlap handling rewrote (``tweaked=...``), that lie inside [0, G) count each I op whose predecessor -- ignoring
P ops and ops of length 0 -- is a match op (M, =, X) and whose anchor, the last base of that match op at reference
position p, has quality >= min_base_quality.  Key (p, len, seq) when len <= 32 and every inserted base is A/C/G/T with
quality >= min_base_quality (seq: A, C, G, T = 0..3, base k in bits 2k), else (p, 0, 0).

Call rule, per anchor p: d = consensus depth, I = every count at p, none = d - I.  The resolved key s is called iff the
consensus letter of p (consensus_oracle.call_position) is neither 'N' nor '-', count(s) > none, count(s) > the
unresolved count, count(s) > every other resolved count, and count(s) / d >= threshold.
"""
from __future__ import annotations

from collections import Counter
from typing import Dict, List, Mapping, Optional, Sequence, Tuple

import numpy as np

from . import consensus_oracle as co
from . import pileup_oracle as po

MAX_LEN = 32
_MATCH = (0, 7, 8)
_REF = (0, 2, 3, 7, 8)
_QUERY = (0, 1, 4, 7, 8)

Key = Tuple[int, int, int]


def encode(bases: str) -> int:
    return sum("ACGT".index(b) << (2 * k) for k, b in enumerate(bases))


def decode(seq: int, length: int) -> str:
    return "".join("ACGT"[(seq >> (2 * k)) & 3] for k in range(length))


def count_read(read: po.Read, qual: Sequence[int], G: int, min_bq: int, counts: Counter) -> None:
    """the insertions of one admitted read (qualities as the batch carries them) into `counts`"""
    rlen = read.ref_len()
    if rlen == 0 or read.pos < 0 or read.pos + rlen > G:          # the deposit skips it (LVC_ERANGE)
        return
    r, qi, prev = read.pos, 0, None
    for op, ln in read.cigar:
        if ln == 0 or op == 6:
            continue
        if op == 1 and prev in _MATCH and qual[qi - 1] >= min_bq:
            bases, qs = read.seq[qi:qi + ln], qual[qi:qi + ln]
            if ln <= MAX_LEN and all(b in "ACGT" for b in bases) and all(q >= min_bq for q in qs):
                counts[(r - 1, ln, encode(bases))] += 1
            else:
                counts[(r - 1, 0, 0)] += 1
        if op in _REF:
            r += ln
        if op in _QUERY:
            qi += ln
        prev = op


def count_insertions(reads: Sequence[po.Read], G: int, min_bq: int, min_mapq: int, max_depth: int = po.MAX_DEPTH,
                     overlap_model: int = po.OVERLAP_OFF) -> Counter:
    """{(pos, len, seq): count} over the reads the pileup engine admits"""
    reads = list(reads)
    admitted: List[int] = []
    tweaked: Dict[int, List[int]] = {}
    for _ in po.pileup_columns(reads, min_mapq, max_depth, admitted=admitted, overlap_model=overlap_model,
                               tweaked=tweaked):
        pass
    counts: Counter = Counter()
    for idx in admitted:
        count_read(reads[idx], tweaked.get(idx, reads[idx].qual), G, min_bq, counts)
    return counts


def depth_and_letters_from_memory(memory: Mapping, G: int, min_depth: int, threshold: float) -> Tuple[np.ndarray, str]:
    """consensus depth and letters of every position from a `memory` dict (the letters of consensus_oracle)"""
    depth = np.zeros(G, dtype=np.int64)
    letters = ["N"] * G
    for p, s in memory.items():
        p = int(p)
        snvs = s["snvs"]
        n = {b: len(snvs.get(b, ())) for b in "ACGT"}
        listed = sum(len(q) for q in snvs.values())
        depth[p] = int(s["totalDepth"])
        letters[p] = co.call_position(n["A"], n["C"], n["G"], n["T"], listed - sum(n.values()),
                                      depth[p] - listed, min_depth, threshold)
    return depth, "".join(letters)


def depth_and_letters_from_tables(planes: Dict[int, np.ndarray], dels: np.ndarray, ref: str, min_depth: int,
                                  threshold: float) -> Tuple[np.ndarray, str]:
    """the same from copied tables (consensus_oracle.consensus_from_tables gives the letters)"""
    depth = np.asarray(dels, dtype=np.int64).copy()
    for arr in planes.values():
        depth += np.asarray(arr, dtype=np.int64).sum(axis=1)
    letters, _ = co.consensus_from_tables(planes, dels, ref, min_depth, threshold)
    return depth, letters


def call_insertions(counts: Mapping[Key, int], depth: Sequence[int], letters: str, threshold: float, p0: int = 0,
                    p1: Optional[int] = None) -> List[Tuple[int, int, int, int, int]]:
    """[(pos, len, seq, count, depth)] of the call rule, ascending position; `depth` / `letters` cover the contig"""
    p1 = len(letters) if p1 is None or p1 < 0 else p1
    at: Dict[int, Dict[Key, int]] = {}
    for key, n in counts.items():
        at.setdefault(key[0], {})[key] = n
    out = []
    for p in sorted(at):
        if not p0 <= p < p1 or letters[p] in "N-":
            continue
        keys = at[p]
        d = int(depth[p])
        total = sum(keys.values())
        unresolved = keys.get((p, 0, 0), 0)
        resolved = {k: n for k, n in keys.items() if k[1] > 0}
        if not resolved:
            continue
        best = max(resolved.values())
        winners = [k for k, n in resolved.items() if n == best]
        if len(winners) != 1:
            continue
        c = best
        if c > d - total and c > unresolved and c / d >= threshold:
            out.append((p, winners[0][1], winners[0][2], c, d))
    return out


def splice(consensus: str, calls: Sequence[Tuple[int, int, int, int, int]], p0: int = 0) -> str:
    """`consensus` (positions p0..) with each called insertion after the letter of its anchor"""
    text = list(consensus)
    for p, ln, seq, _, _ in sorted(calls, reverse=True):
        text.insert(p - p0 + 1, decode(seq, ln))
    return "".join(text)

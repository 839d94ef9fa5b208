"""CPU ORACLE (test infrastructure) of the consensus / coverage rule of ``lvc_consensus`` (include/lvc.h).

Two formulations of the same rule:

* ``consensus_from_memory``: the rule applied literally, position by position, to the reference's own state, the
  ``memory`` dict (``{pos: {"reference", "totalDepth", "snvs": {allele: [phred, ...]}, "indels"}}``).  nO is the
  number of qualities listed under alleles other than A/C/G/T, nD = totalDepth - all listed qualities.
* ``consensus_from_tables``: the rule vectorised with NumPy over copied device tables (``copy_plane`` / ``copy_dels``),
  for inputs where building the dict is too slow.
"""
from __future__ import annotations

from typing import Dict, Mapping, Optional, Sequence, Tuple

import numpy as np

NIBBLE_CHARS = "=ACMGRSVTWYHKDBN"
DELETION = 4                                      # rank of the deletion member (after A, C, G, T)
COUNTERS = ("n_positions", "depth_sum", "depth_max", "n_low_depth", "n_N", "n_deleted", "n_ambiguous", "n_mismatch")


def call_position(nA: int, nC: int, nG: int, nT: int, nO: int, nD: int, min_depth: int, threshold: float) -> str:
    """The consensus letter of one position (include/lvc.h, lvc_consensus), written as the rule reads."""
    d = nA + nC + nG + nT + nO + nD
    if d == 0 or d < min_depth:
        return "N"
    members = sorted(((n, rank) for rank, n in enumerate((nA, nC, nG, nT, nD)) if n > 0), key=lambda m: (-m[0], m[1]))
    cum, taken = 0, []
    for n, rank in members:
        taken.append(rank)
        cum += n
        if float(cum) / float(d) >= threshold:
            break
    else:
        return "N"
    if taken[0] == DELETION:
        return "-"
    mask = 0
    for rank in taken:
        if rank < 4:
            mask |= 1 << rank
    return NIBBLE_CHARS[mask]


def _stats(depth: np.ndarray, seq: bytes, ref: bytes, min_depth: int, depth_thresholds: Sequence[int]) -> dict:
    letters = np.frombuffer(seq, dtype=np.uint8)
    refu = np.frombuffer(ref.upper(), dtype=np.uint8)
    depth = depth.astype(np.uint64)
    is_base = np.isin(letters, np.frombuffer(b"ACGT", np.uint8))
    ref_acgt = np.isin(refu, np.frombuffer(b"ACGT", np.uint8))
    st = {
        "n_positions": int(len(letters)),
        "depth_sum": int(depth.sum(dtype=np.uint64)),
        "depth_max": int(depth.max()) if len(depth) else 0,
        "n_low_depth": int(np.count_nonzero(depth < np.uint64(min_depth))),
        "n_N": int(np.count_nonzero(letters == ord("N"))),
        "n_deleted": int(np.count_nonzero(letters == ord("-"))),
        "n_ambiguous": int(np.count_nonzero(np.isin(letters, np.frombuffer(b"MRWSYKVHDB", np.uint8)))),
        "n_mismatch": int(np.count_nonzero(is_base & ref_acgt & (letters != refu))),
        "depth_ge": [int(np.count_nonzero(depth >= np.uint64(t))) for t in depth_thresholds],
    }
    return st


def consensus_from_memory(memory: Mapping, ref: str, min_depth: int, threshold: float,
                          depth_thresholds: Sequence[int] = (), p0: int = 0, p1: Optional[int] = None
                          ) -> Tuple[str, dict]:
    """(consensus over [p0, p1), statistics) from a `memory` dict; keys may be int or str (golden JSON)."""
    p1 = len(ref) if p1 is None or p1 < 0 else p1
    sites = {int(p): s for p, s in memory.items()}
    letters, depth = [], np.zeros(p1 - p0, dtype=np.uint64)
    for p in range(p0, p1):
        s = sites.get(p)
        if s is None:                                      # d = 0
            letters.append("N")
            continue
        snvs = s["snvs"]
        n = {b: len(snvs.get(b, ())) for b in "ACGT"}
        listed = sum(len(q) for q in snvs.values())
        nO = listed - sum(n.values())
        nD = int(s["totalDepth"]) - listed
        depth[p - p0] = int(s["totalDepth"])
        letters.append(call_position(n["A"], n["C"], n["G"], n["T"], nO, nD, min_depth, threshold))
    seq = "".join(letters)
    return seq, _stats(depth, seq.encode(), ref[p0:p1].encode("latin-1"), min_depth, depth_thresholds)


def consensus_from_tables(planes: Dict[int, np.ndarray], dels: np.ndarray, ref: str, min_depth: int, threshold: float,
                          depth_thresholds: Sequence[int] = (), p0: int = 0, p1: Optional[int] = None
                          ) -> Tuple[str, dict]:
    """The same rule vectorised over the tables: planes {key: uint32 [G, 4]} (key = group << 8 | quality),
    dels uint32 [G]."""
    p1 = len(ref) if p1 is None or p1 < 0 else p1
    n = p1 - p0
    cnt = np.zeros((n, 5), dtype=np.int64)                 # A, C, G, T, deletion
    other = np.zeros(n, dtype=np.int64)
    for key, arr in planes.items():
        a = np.asarray(arr[p0:p1], dtype=np.int64)
        if key >> 8 == 0:
            cnt[:, :4] += a
        else:
            other += a.sum(axis=1)
    cnt[:, 4] = np.asarray(dels[p0:p1], dtype=np.int64)
    d = cnt.sum(axis=1) + other
    order = np.argsort(-cnt, axis=1, kind="stable")        # descending count, ties by rank
    srt = np.take_along_axis(cnt, order, axis=1)
    cum = np.cumsum(srt, axis=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        df = d.astype(np.float64)[:, None]
        prev_below = (cum - srt).astype(np.float64) / df < threshold
        reached = (cum[:, 4].astype(np.float64) / d.astype(np.float64)) >= threshold
    first = np.zeros((n, 5), dtype=bool)
    first[:, 0] = True
    taken = (srt > 0) & (first | prev_below)
    bit = np.where(order < 4, np.left_shift(1, np.minimum(order, 3)), 0)
    mask = (taken * bit).sum(axis=1)
    lut = np.frombuffer(NIBBLE_CHARS.encode(), dtype=np.uint8)
    letters = lut[mask]
    letters = np.where((order[:, 0] == DELETION) & (srt[:, 0] > 0), ord("-"), letters)
    letters = np.where((cum[:, 4] == 0) | ~reached, ord("N"), letters)
    letters = np.where((d == 0) | (d < min_depth), ord("N"), letters).astype(np.uint8)
    seq = letters.tobytes()
    return seq.decode("ascii"), _stats(d, seq, ref[p0:p1].encode("latin-1"), min_depth, depth_thresholds)

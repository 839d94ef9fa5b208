"""Drop-in ``LiveVariantCaller`` backed by the B200 kernels (liblvc_b200.so through ctypes).

Same module path, constructor and methods as the reference class
(``variant_caller/live_variant_caller.py:21-297`` of COVID-SpiNGS/covid-spings-variant-caller), so
``client_server/vc_queue.py:55-63,140-144`` and ``main.py:17-29`` keep working unchanged:

    LiveVariantCaller(referenceFasta, minBaseQuality, minMappingQuality, minTotalDepth,
                      minAlleleDepth, minEvidenceRatio, maxVariants)
    .process_bam(inputBam, referenceIndex=0)   incremental: state accumulates across calls
    .prepare_variants() -> List[Variant]
    .write_vcf(path)
    .create_checkpoint(path) / .load_checkpoint(path)      pickle of the reference's `memory` schema
    .reset_memory()
    .memory                                                 dict[int -> Site], materialised on demand

What differs, by design: the per-position state lives on the GPU as integer count tables
(A/C/G/T x quality histograms, deletion counts, first-seen ranks) instead of Python lists, the CIGAR
walk runs in a CUDA kernel instead of htslib's pileup engine, and pysam is not needed.  There is no
CPU fallback: without the CUDA library / a GPU, construction raises.
"""
from __future__ import annotations

import os
import pickle
import threading
from typing import Dict, List, Optional

import numpy as np

from lvc_b200 import capi, packing, records, samio
from lvc_b200.packing import ReadBatch, UnsupportedInput

from .structs import Site, Variant

try:  # inside the reference tree the real helper is used (live_variant_caller.py:15)
    import config_util.logging as log  # type: ignore
except Exception:  # standalone: same call signature, stdout only
    class log:  # noqa: N801
        DEBUG, ERROR, INFO, WARNING = "debug", "error", "info", "warning"

        @staticmethod
        def print_and_log(text, log_type):
            from time import strftime, localtime
            print(f"{strftime('[%Y-%m-%d %H:%M:%S]', localtime())} {text}")

NIBBLE_CHARS = records.NIBBLE_CHARS
_GS_TO_NIBBLE = [1, 2, 4, 8, 0, 3, 5, 6, 7, 9, 10, 11, 12, 13, 14, 15]      # (group<<2|slot) -> BAM nibble
_NIBBLE_TO_GS = {n: gs for gs, n in enumerate(_GS_TO_NIBBLE)}


def _default_device() -> int:
    for var in ("LVC_DEVICE", "LOCAL_RANK"):
        if os.environ.get(var, "") != "":
            return int(os.environ[var])
    return 0


class LiveVariantCaller:
    def __init__(self, referenceFasta: str, minBaseQuality: int, minMappingQuality: int, minTotalDepth: int,
                 minAlleleDepth: int, minEvidenceRatio: float, maxVariants: int, device: Optional[int] = None,
                 maxDepth: int = capi.MAX_DEPTH_DEFAULT, ignoreOverlaps: bool = True, overlapModel: Optional[str] = None,
                 countInsertions: bool = False, maxInsertionKeys: int = 1 << 20, countStrands: bool = False):
        self.minBaseQuality = minBaseQuality
        self.minMappingQuality = minMappingQuality
        self.minTotalDepth = minTotalDepth
        self.minAlleleDepth = minAlleleDepth
        self.minEvidenceRatio = minEvidenceRatio
        self.maxVariants = maxVariants                      # stored, never used (reference :29)
        self.maxDepth = maxDepth                            # pysam's pileup(max_depth=8000) default
        # pysam's pileup(ignore_overlaps=True) default: htslib rewrites the qualities of overlapping mates.  The rule
        # changed between htslib releases and the reference does not pin pysam: "htslib-1.13" (default) or "htslib-1.10"
        self.overlapModel = capi.overlap_model_id(overlapModel) if ignoreOverlaps else capi.OVERLAP_OFF
        # insertions for consensus(insertions=True) (include/lvc.h lvc_enable_insertions): a device hash table of at least
        # maxInsertionKeys keys; records, VCF, memory and checkpoints never contain insertions
        self.countInsertions = bool(countInsertions)
        self.maxInsertionKeys = int(maxInsertionKeys)
        # reverse-strand counts for strand_bias() and write_vcf(strandBias=True) (include/lvc.h lvc_enable_strand_counts):
        # 17 x 4 bytes per reference position on the device; nothing else changes
        self.countStrands = bool(countStrands)
        self.fastaFile = samio.Fasta(referenceFasta)
        self._device = _default_device() if device is None else device
        self._lock = threading.RLock()                      # the reference's callers use bare threads
        self._handle: Optional[capi.Handle] = None
        self._contig: Optional[str] = None
        self._e_lut, self._om_lut = records.phred_luts()
        self._open_contig(0)

    # ------------------------------------------------------------------ lifetime
    def _open_contig(self, referenceIndex: int):
        name = self.fastaFile.references[referenceIndex]
        if self._handle is not None:
            if name == self._contig:
                return
            raise UnsupportedInput("one LiveVariantCaller instance holds the tables of ONE contig "
                                   f"({self._contig!r}); got {name!r} (the reference keys its state by position only)")
        self._contig = name
        self._ref = self.fastaFile.fetch(reference=name)
        self._handle = capi.Handle(self._ref.encode("latin-1"), max(0, int(self.minBaseQuality)),
                                   int(self.minMappingQuality), self._device)
        if self.countInsertions:
            self._handle.enable_insertions(self.maxInsertionKeys)
        if self.countStrands:
            self._handle.enable_strand_counts()

    def close(self):
        with self._lock:
            if self._handle is not None:
                self._handle.close()
                self._handle = None

    def __del__(self):
        try:
            self.close()
            self.fastaFile.close()
        except Exception:
            pass

    def reset_memory(self):
        with self._lock:
            if self._handle is not None:
                self._handle.reset()

    # ------------------------------------------------------------------ deposit
    def process_bam(self, inputBam: str, referenceIndex=0):
        """live_variant_caller.py:54-72.  Reads the alignments of contig `referenceIndex` (BAM, or SAM text),
        packs them and deposits them into the device tables."""
        with self._lock:
            self._open_contig(referenceIndex)
            reads = samio.read_alignments_native(inputBam, self._contig, int(self.minMappingQuality), self.maxDepth,
                                                 overlap_model=self.overlapModel)
            try:
                reads.compact()                 # reads the admission dropped never reach the device
                if reads.n_reads:
                    # quality codes where the file qualifies, 2-bit base codes on top where its bases allow it
                    self._handle.push_batch(reads.batch_for(int(self.minBaseQuality)))
            finally:
                reads.close()

    def process_batch(self, batch: ReadBatch):
        """Deposit one packed, coordinate-sorted batch (the fast entry point for live batches)."""
        with self._lock:
            if batch.n_reads:
                self._handle.push_batch(batch.as_capi())

    # ------------------------------------------------------------------ genotype
    def _candidates(self, emit_all: bool = False) -> np.ndarray:
        return self._handle.genotype(int(self.minTotalDepth), int(self.minAlleleDepth), float(self.minEvidenceRatio),
                                     self._e_lut, self._om_lut, capi.GENO_EMIT_ALL if emit_all else 0)

    def prepare_variants(self) -> List[Variant]:
        """live_variant_caller.py:120-231."""
        with self._lock:
            return records.candidates_to_variants(self._candidates())

    def likelihoods(self) -> Dict[int, Dict[str, float]]:
        """L(allele) for every allele of every gated site (not in the reference API; parity tests)."""
        with self._lock:
            out: Dict[int, Dict[str, float]] = {}
            for c in self._candidates(emit_all=True):
                out.setdefault(int(c["pos"]), {})[NIBBLE_CHARS[int(c["code"])]] = float(c["L"])
            return out

    def write_vcf(self, outputVfc: str, strandBias: bool = False):
        """live_variant_caller.py:233-297.  strandBias=True (needs countStrands=True) adds DP4, FS and SOR to every record's
        INFO and their three ##INFO lines to the header (strand_bias); without it the text is the reference's."""
        with self._lock:
            contigs = [(r, self.fastaFile.get_reference_length(r)) for r in self.fastaFile.references]
            variants = self.prepare_variants()
            text = records.format_vcf(variants, contigs, self.strand_bias(variants) if strandBias else None)
        with open(outputVfc, "w") as fh:
            fh.write(text)

    def write_csv(self, path: str):
        """Per-position table sketched in the reference's README.md:4-8 (additive output)."""
        with self._lock:
            self._candidates()
            depth, ad, _ = self._handle.copy_dense()
        with open(path, "w") as fh:
            fh.write(records.format_site_csv(depth, ad, self._ref))

    # ------------------------------------------------------------------ consensus + coverage (not in the reference API)
    def _insertion_calls(self, minDepth, threshold):
        if not self.countInsertions:
            raise ValueError("this LiveVariantCaller does not count insertions: construct it with countInsertions=True")
        return self._handle.insertion_calls(int(minDepth), float(threshold))

    def consensus(self, minDepth: int = 10, threshold: float = 0.0, insertions: bool = False) -> str:
        """Consensus genome, one letter per reference position (include/lvc.h lvc_consensus): 'N' below minDepth, '-'
        where deletions are the majority, IUPAC codes where the bases needed to reach `threshold` of the depth differ.
        Computed on the device from the count tables.  It contains no insertions unless `insertions` is True, which needs a
        caller constructed with countInsertions=True: then each called insertion (insertion_calls) follows the letter of
        its anchor, uppercase.  After load_checkpoint, or with more distinct insertions than the table holds, that raises
        (capi.LvcError) until reset_memory: the insertion counts do not cover the loaded tables."""
        with self._lock:
            seq, _ = self._handle.consensus(int(minDepth), float(threshold))
            text = seq.decode("ascii")
            if insertions:
                text = records.splice_insertions(text, self._insertion_calls(minDepth, threshold))
        return text

    def insertion_calls(self, minDepth: int = 10, threshold: float = 0.0) -> List[dict]:
        """The insertions consensus(insertions=True) splices in (include/lvc.h lvc_insertion_calls), ascending position:
        [{"pos": anchor (0-based; the insertion follows this reference base), "seq": inserted bases, "count": reads
        carrying it, "depth": consensus depth at pos}].  Needs countInsertions=True; raises as consensus(insertions=True)."""
        with self._lock:
            calls = self._insertion_calls(minDepth, threshold)
        return [{"pos": int(c["pos"]), "seq": records.decode_insertion(c["seq"], c["len"]), "count": int(c["count"]),
                 "depth": int(c["depth"])} for c in calls]

    def write_consensus(self, outputFasta: str, minDepth: int = 10, threshold: float = 0.0, insertions: bool = False):
        """FASTA of `consensus()` with the deletion calls removed, 60 letters per line."""
        with self._lock:
            text = records.format_consensus_fasta(self._contig, self.consensus(minDepth, threshold, insertions))
        with open(outputFasta, "w") as fh:
            fh.write(text)

    def coverage_summary(self, depths=(1, 10, 20, 100), minDepth: int = 10, threshold: float = 0.0) -> dict:
        """Coverage and completeness of the contig: the counters of lvc_consensus_stats, `depth_ge` and `breadth`
        ({depth: positions with at least that depth, as a count and as a fraction}), `mean_depth` and `completeness`
        (the share of positions whose consensus letter is not 'N')."""
        depths = [int(x) for x in depths]
        with self._lock:
            _, st = self._handle.consensus(int(minDepth), float(threshold), depths)
        n = st["n_positions"]
        out = {k: v for k, v in st.items() if k != "depth_ge"}
        out["depth_ge"] = dict(zip(depths, st["depth_ge"]))
        out["mean_depth"] = st["depth_sum"] / n
        out["breadth"] = {x: c / n for x, c in zip(depths, st["depth_ge"])}
        out["completeness"] = (n - st["n_N"]) / n
        return out

    # ------------------------------------------------------------------ strand bias (not in the reference API)
    def strand_bias(self, variants: Optional[List[Variant]] = None) -> List[dict]:
        """Strand bias of each record of `variants` (default: prepare_variants()), in their order: {"start", "alleles",
        "ref_fwd", "ref_rev", "alt_fwd", "alt_rev": the forward / reverse pileup entries of the REF and ALT letters at the
        position, counted as DP counts them (bcftools DP4), "fisher_p": two-sided Fisher exact p-value of that 2x2 table,
        "fs": -10 log10(fisher_p) (GATK FS), "sor": GATK's symmetric odds ratio (SOR)}.  Counts and statistics are None for
        a record whose REF letter is not a nibble code.  Needs countStrands=True; after load_checkpoint it raises
        (capi.LvcError) until reset_memory: the strand counts do not cover loaded tables."""
        if not self.countStrands:
            raise ValueError("this LiveVariantCaller does not count strands: construct it with countStrands=True")
        with self._lock:
            if variants is None:
                variants = self.prepare_variants()
            asked = [k for k, v in enumerate(variants)
                     if all(len(a) == 1 and a.upper() in NIBBLE_CHARS for a in v["alleles"][:2])]
            pos = [variants[k]["start"] for k in asked for _ in (0, 1)]
            letters = "".join(variants[k]["alleles"][0] + variants[k]["alleles"][1] for k in asked)
            fwd, rev = self._handle.strand_counts(pos, letters)
        counts = {k: (fwd[2 * j], rev[2 * j], fwd[2 * j + 1], rev[2 * j + 1]) for j, k in enumerate(asked)}
        return [records.strand_row(v, counts.get(k)) for k, v in enumerate(variants)]

    # ------------------------------------------------------------------ variant linkage (not in the reference API)
    def track_linkage(self, sites, maxSpan: int = 300):
        """Count, from now on, how the `sites` -- an iterable of (pos0, alt), pos0 0-based and ascending, alt one of
        'A' 'C' 'G' 'T' or '-' for a deletion -- co-occur on the same reads (include/lvc.h lvc_set_linkage_sites): every two
        sites at most maxSpan apart form a pair.  Call it before process_bam / process_batch: the counts cover the batches
        pushed since, and calling it again starts them over; reset_memory and load_checkpoint clear them and keep the sites.
        An empty list turns counting off."""
        sites = [(int(p), str(a)) for p, a in sites]
        with self._lock:
            self._handle.set_linkage_sites([p for p, _ in sites], "".join(a for _, a in sites), int(maxSpan))

    def linkage(self, minReads: int = 1) -> List[dict]:
        """Every pair of tracked sites whose REF/ALT states were both seen on at least minReads reads, in (pos_a, pos_b)
        order: {"pos_a", "alt_a", "pos_b", "alt_b", "counts": 3x3 list [state_a][state_b] (REF 0, ALT 1, OTHER 2),
        "n": reads with REF or ALT at both sites, "r2": squared correlation of the ALT states on those reads, None when
        n is 0 or a site does not vary}."""
        with self._lock:
            pairs = self._handle.copy_linkage()
        out = []
        for p in pairs:
            counts = p["count"].tolist()
            n = counts[0][0] + counts[0][1] + counts[1][0] + counts[1][1]
            if n < minReads:
                continue
            out.append({"pos_a": int(p["pos_a"]), "alt_a": chr(p["alt_a"]), "pos_b": int(p["pos_b"]),
                        "alt_b": chr(p["alt_b"]), "counts": counts, "n": n, "r2": records.linkage_r2(counts)})
        return out

    # ------------------------------------------------------------------ state <-> reference schema
    def _export_tables(self):
        h = self._handle
        keys = [int(k) for k in h.plane_keys()]
        planes = {k: h.copy_plane(k) for k in keys}
        first = {g: h.copy_first(g) for g in range(4)}
        return keys, planes, first, h.copy_dels(), np.cumsum(h.copy_covdiff()[:-1])

    @property
    def memory(self) -> Dict[int, Site]:
        """The reference's `self.memory` (live_variant_caller.py:31, 77-103), rebuilt from the tables.
        Alleles appear in first-seen order (it decides record order, SURVEY A7); the qualities of one
        allele are listed in ascending order (their read order is not a sufficient statistic)."""
        with self._lock:
            keys, planes, first, dels, cov = self._export_tables()
        mem: Dict[int, Site] = {}
        sites = np.nonzero(cov > 0)[0]
        per_pos: Dict[int, Dict[int, List]] = {}
        for k in sorted(keys):
            g, q = k >> 8, k & 255
            nz_p, nz_s = np.nonzero(planes[k])
            for p, s in zip(nz_p.tolist(), nz_s.tolist()):
                per_pos.setdefault(p, {}).setdefault(g * 4 + s, []).append((q, int(planes[k][p, s])))
        for p in sites.tolist():
            alle = per_pos.get(p, {})
            order = sorted(alle, key=lambda gs: int(first[gs >> 2][p, gs & 3]))
            snvs, total = {}, int(dels[p])
            for gs in order:
                lst: List[int] = []
                for q, n in alle[gs]:
                    lst.extend([q] * n)
                    total += n
                snvs[NIBBLE_CHARS[_GS_TO_NIBBLE[gs]]] = lst
            mem[p] = {"reference": self._ref[p], "totalDepth": total, "snvs": snvs, "indels": {}}
        return mem

    @memory.setter
    def memory(self, mem: Dict[int, Site]):
        """Replace the device state by a `memory` dict in the reference's schema (load_checkpoint)."""
        with self._lock:
            h = self._handle
            h.reset()
            G = h.G
            planes: Dict[int, np.ndarray] = {}
            first = {g: None for g in range(4)}
            dels = np.zeros(G, dtype=np.uint32)
            covd = np.zeros(G + 1, dtype=np.int32)
            for p, site in mem.items():
                p = int(p)
                if not 0 <= p < G:
                    raise ValueError(f"checkpoint position {p} outside the reference (length {G})")
                covd[p] += 1
                covd[p + 1] -= 1
                n_bases = 0
                for rank, (base, quals) in enumerate(site["snvs"].items()):
                    gs = _NIBBLE_TO_GS[NIBBLE_CHARS.index(base)]
                    g = gs >> 2
                    if first[g] is None:
                        first[g] = np.full((G, 4), 0xFFFFFFFF, dtype=np.uint32)
                    first[g][p, gs & 3] = rank
                    qs, cnt = np.unique(np.asarray(quals, dtype=np.int64), return_counts=True)
                    for q, n in zip(qs.tolist(), cnt.tolist()):
                        key = (g << 8) | int(q)
                        if key not in planes:
                            planes[key] = np.zeros((G, 4), dtype=np.uint32)
                        planes[key][p, gs & 3] += n
                    n_bases += len(quals)
                dels[p] = int(site["totalDepth"]) - n_bases
            for key, arr in planes.items():
                h.import_plane(key, arr)
            for g, arr in first.items():
                if arr is not None:
                    h.import_first(g, arr)
            h.import_dels(dels)
            h.import_covdiff(covd)
            h.ordinal = 16          # imported first-seen ranks are 0..15; later reads rank after them

    def create_checkpoint(self, filename):
        """live_variant_caller.py:40-45: pickle of `memory` in the reference's schema."""
        log.print_and_log(f'Creating checkpoint {filename}', log.INFO)
        with open(filename, 'wb') as file:
            pickle.dump(self.memory, file)

    def load_checkpoint(self, filename):
        """live_variant_caller.py:47-52: replaces the whole state."""
        log.print_and_log(f'Loading checkpoint {filename}', log.INFO)
        with open(filename, 'rb') as file:
            self.memory = pickle.load(file)

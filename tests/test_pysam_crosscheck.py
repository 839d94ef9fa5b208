"""Cross-check against the REAL reference wherever pysam can be imported (SURVEY 8d(2), Appendix B checklist).

The pileup half of the oracle (CIGAR walk, deletion-entry quality rule, max_depth admission, mate overlaps) restates
htslib, which is neither in the reference project nor a dependency of this one, so it is "parity unpinned"
(oracle/pileup_oracle.py header).  This module is the pin: when `import pysam` succeeds AND the environment variable
LVC_REFERENCE names a checkout of the reference project, it writes BAMs with samio.write_bam, runs the UNMODIFIED
variant_caller/live_variant_caller.py:21 `LiveVariantCaller` (process_bam :54-72, prepare_variants :120-231) on them
and compares `memory` and the records with the oracle (no GPU needed) and with the drop-in class (GPU).  When the
import fails it says so -- with the reason -- so that the test log of every box records the pysam / htslib status.

Cases (SURVEY Appendix B): the reference's own fixture test/testdata/testfile.sam at the four threshold sets of the
goldens; 9,000 reads at one start (B4: max_depth admission); `...M 2I 3D ...` (B3: qpos of deletion entries);
a deletion as the last reference-consuming op; an overlapping proper pair (B5: which release line the installed
htslib follows)."""
import importlib
import os
import sys

import numpy as np
import pytest

from oracle import pileup_oracle as po
from conftest import GOLD


def _pysam_status():
    try:
        import pysam
        ver = getattr(pysam, "__version__", "?")
        hts = getattr(getattr(pysam, "version", None), "__htslib_version__", None) or \
            getattr(pysam, "__htslib_version__", "?")
        return pysam, f"pysam {ver} (htslib {hts})"
    except Exception as e:  # ModuleNotFoundError here and on the GPU boxes of this pool
        return None, f"pysam not importable: {type(e).__name__}: {e}"


def _reference_tree():
    cand = os.environ.get("LVC_REFERENCE")
    if cand and os.path.exists(os.path.join(cand, "variant_caller", "live_variant_caller.py")):
        return cand
    return None


PYSAM, STATUS = _pysam_status()
REFTREE = _reference_tree()
print(f"[pysam cross-check] {STATUS}; reference tree: {REFTREE}", file=sys.stderr)

needs_pysam = pytest.mark.skipif(PYSAM is None or REFTREE is None,
                                 reason=f"{STATUS}; reference tree: {REFTREE} -- the htslib half stays 'parity unpinned'")


def test_pysam_status_is_reported():
    """always runs: the log of this box says whether the real reference could be consulted"""
    print(f"[pysam cross-check] {STATUS}; reference tree: {REFTREE}")
    assert isinstance(STATUS, str)


def _real_class():
    """the reference's own class, imported from its tree under a private module name (the drop-in package is also
    called variant_caller)"""
    sys.path.insert(0, REFTREE)
    try:
        for m in [m for m in sys.modules if m == "variant_caller" or m.startswith("variant_caller.")]:
            sys.modules["dropin_" + m] = sys.modules.pop(m)
        mod = importlib.import_module("variant_caller.live_variant_caller")
        ref_cls = mod.LiveVariantCaller
        for m in [m for m in sys.modules if m == "variant_caller" or m.startswith("variant_caller.")]:
            sys.modules["reference_" + m] = sys.modules.pop(m)
        for m in [m for m in sys.modules if m.startswith("dropin_variant_caller")]:
            sys.modules[m[len("dropin_"):]] = sys.modules.pop(m)
        return ref_cls
    finally:
        sys.path.remove(REFTREE)


def _write_inputs(tmp_path, name, ref, reads):
    from lvc_b200 import samio
    fa = str(tmp_path / f"{name}.fasta")
    with open(fa, "w") as fh:
        fh.write(">NC_045512.2\n")
        for i in range(0, len(ref), 70):
            fh.write(ref[i:i + 70] + "\n")
    bam = str(tmp_path / f"{name}.bam")
    recs = [(r.flag, r.pos, r.mapq, r.cigar, r.seq, r.qual, r.name, r.mpos, r.mref, r.tlen) for r in reads]
    samio.write_bam(bam, [("NC_045512.2", len(ref))], recs)
    PYSAM.index(bam)
    return fa, bam


def _cases():
    rng = np.random.default_rng(5)
    ref = "".join("ACGT"[i] for i in rng.integers(0, 4, 3000))

    def read(pos, cigar, name, flag=0, q=40, mpos=-1, mref=-1, tlen=0, mutate=()):
        lq = sum(n for o, n in cigar if o in (0, 1, 4, 7, 8))
        seq, r = [], pos
        for o, n in cigar:
            if o in (0, 7, 8):
                seq.extend(ref[r:r + n]); r += n
            elif o in (1, 4):
                seq.extend("A" * n)
            elif o in (2, 3):
                r += n
        for i in mutate:
            seq[i] = "A" if seq[i] != "A" else "C"
        quals = [q] * lq if isinstance(q, int) else list(q)
        return po.Read(flag, pos, 60, cigar, "".join(seq), quals, name, mpos, mref, tlen)

    cases = {}
    # B4: 9,000 reads at one start, then a few more further on (pysam's max_depth = 8000)
    cases["b4_depth_cap"] = [read(100, [(0, 60)], f"d{i}") for i in range(9000)] + \
                            [read(130, [(0, 60)], f"e{i}") for i in range(50)]
    # B3: ... M 2I 3D M ...: the deletion entries are judged by the quality of the base AFTER the insertion
    q = [40] * 20 + [5, 5] + [3] + [40] * 29
    cases["b3_ins_then_del"] = [read(200, [(0, 20), (1, 2), (2, 3), (0, 30)], f"i{i}", q=q) for i in range(12)] + \
                               [read(200, [(0, 53)], f"p{i}") for i in range(12)]
    # a deletion as the last reference-consuming op (the next query base does not exist: quality 0)
    cases["del_last"] = [read(300, [(0, 30), (2, 4), (4, 5)], f"l{i}") for i in range(12)] + \
                        [read(300, [(0, 34)], f"m{i}") for i in range(12)]
    # B5: overlapping proper pairs, one mismatch in the overlap
    pairs = []
    for i in range(14):
        pairs.append(read(400, [(0, 50)], f"pair{i}", flag=99, q=30, mpos=430, mref=1, tlen=80))
        pairs.append(read(430, [(0, 50)], f"pair{i}", flag=147, q=30 if i % 2 else 25, mpos=400, mref=1, tlen=-80,
                          mutate=(5,)))
    cases["b5_overlap"] = po.samtools_sort(pairs)
    return ref, cases


TH_SETS = [dict(minBQ=30, minMQ=20, minDP=10, minAD=5, ratio=0.10), dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05),
           dict(minBQ=0, minMQ=0, minDP=1, minAD=1, ratio=0.0)]


def _norm_memory(mem):
    return {int(p): (s["reference"], int(s["totalDepth"]), {a: sorted(int(x) for x in v) for a, v in s["snvs"].items()},
                     list(s["snvs"])) for p, s in mem.items()}


def _run_reference(ref_cls, fa, bam, th):
    c = ref_cls(fa, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1)
    c.process_bam(bam)
    return c.memory, c.prepare_variants()


def _overlap_model_of_installed_htslib(ref_cls, tmp_path):
    """which release line the installed htslib follows, decided on one overlapping pair (SURVEY B5)"""
    ref, cases = _cases()
    fa, bam = _write_inputs(tmp_path, "probe", ref, cases["b5_overlap"][:2])
    mem, _ = _run_reference(ref_cls, fa, bam, dict(minBQ=0, minMQ=0, minDP=1, minAD=1, ratio=0.0))
    for model in (po.OVERLAP_HTSLIB_1_13, po.OVERLAP_HTSLIB_1_10):
        oc = po.OracleCaller(ref, 0, 0, 1, 1, 0.0, overlap_model=model)
        oc.process_reads(cases["b5_overlap"][:2])
        if _norm_memory(oc.memory) == _norm_memory(mem):
            return model
    pytest.fail("the installed htslib's mate-overlap handling matches neither restated model")


@needs_pysam
def test_oracle_equals_real_reference(tmp_path):
    """oracle (htslib restatement) == the unmodified reference class under the installed pysam: no GPU needed"""
    ref_cls = _real_class()
    model = _overlap_model_of_installed_htslib(ref_cls, tmp_path)
    print(f"[pysam cross-check] installed htslib follows overlap model {model}")
    ref, cases = _cases()
    contigs, t_reads = po.read_sam(os.path.join(GOLD, "testfile.sam"))
    t_ref = open(os.path.join(GOLD, "NC_045512.2.synthetic.fasta")).read().split("\n", 1)[1].replace("\n", "")
    todo = [("testfile", t_ref, t_reads)] + [(k, ref, v) for k, v in cases.items()]
    for name, rseq, reads in todo:
        fa, bam = _write_inputs(tmp_path, name, rseq, reads)
        for th in TH_SETS:
            mem, recs = _run_reference(ref_cls, fa, bam, th)
            oc = po.OracleCaller(rseq, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], overlap_model=model)
            oc.process_reads(reads)
            assert _norm_memory(oc.memory) == _norm_memory(mem), (name, th)
            got = oc.prepare_variants()
            assert len(got) == len(recs), (name, th)
            for a, b in zip(got, recs):
                assert a["start"] == b["start"] and a["alleles"] == tuple(b["alleles"]) and a["info"]["DP"] == b["info"]["DP"] \
                    and a["info"]["AD"] == b["info"]["AD"] and a["info"]["PL"] == b["info"]["PL"] \
                    and a["info"]["SCORE"] == b["info"]["SCORE"], (name, th, a, b)


@needs_pysam
@pytest.mark.gpu
def test_dropin_equals_real_reference(lib, tmp_path):
    """the drop-in class (CUDA path) == the unmodified reference class on the same BAMs"""
    from variant_caller.live_variant_caller import LiveVariantCaller
    from lvc_b200 import capi
    from helpers import assert_variants_equal
    ref_cls = _real_class()
    model = _overlap_model_of_installed_htslib(ref_cls, tmp_path)
    model_name = {po.OVERLAP_HTSLIB_1_13: "htslib-1.13", po.OVERLAP_HTSLIB_1_10: "htslib-1.10"}[model]
    ref, cases = _cases()
    contigs, t_reads = po.read_sam(os.path.join(GOLD, "testfile.sam"))
    t_ref = open(os.path.join(GOLD, "NC_045512.2.synthetic.fasta")).read().split("\n", 1)[1].replace("\n", "")
    todo = [("testfile", t_ref, t_reads)] + [(k, ref, v) for k, v in cases.items()]
    for name, rseq, reads in todo:
        fa, bam = _write_inputs(tmp_path, name + "_g", rseq, reads)
        for th in TH_SETS:
            mem, recs = _run_reference(ref_cls, fa, bam, th)
            lvc = LiveVariantCaller(fa, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0,
                                    overlapModel=model_name)
            lvc.process_bam(bam)
            assert _norm_memory(lvc.memory) == _norm_memory(mem), (name, th)
            assert_variants_equal(lvc.prepare_variants(), recs, f"{name} {th}")
            lvc.close()
    assert capi.OVERLAP_DEFAULT in (capi.OVERLAP_HTSLIB_1_13, capi.OVERLAP_HTSLIB_1_10)

"""GPU: lvc_consensus (consensus letters + coverage statistics from the device tables) against the oracle of
oracle/consensus_oracle.py -- the dict formulation on the reference's `memory`, the NumPy formulation on copied tables --
sequence and every counter identical."""
import math
import os
import pickle

import numpy as np
import pytest

from helpers import GOLD, po, synth_small, rows_to_tuples
from oracle import consensus_oracle as co

pytestmark = pytest.mark.gpu

MIN_DEPTHS = (0, 1, 3, 10)
THRESHOLDS = (0.0, 0.07, 0.25, 0.5, 0.75, 1.0)
DEPTHS = (1, 10, 20, 100)
FASTA = os.path.join(GOLD, "NC_045512.2.synthetic.fasta")


def _ref_of(fasta):
    return open(fasta).read().split("\n", 1)[1].replace("\n", "")


def _fasta(tmp_path, name, ref):
    p = str(tmp_path / f"{name}.fasta")
    with open(p, "w") as fh:
        fh.write(f">{name}\n{ref}\n")
    return p


def _lvc(fasta, th):
    from variant_caller.live_variant_caller import LiveVariantCaller
    return LiveVariantCaller(fasta, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0)


def _tables(h):
    return {int(k): h.copy_plane(int(k)) for k in h.plane_keys()}, h.copy_dels()


def _check_grid(h, want, what, min_depths=MIN_DEPTHS, thresholds=THRESHOLDS):
    """want(min_depth, threshold) -> (sequence, statistics) of the oracle"""
    for md in min_depths:
        for t in thresholds:
            seq, st = h.consensus(md, t, DEPTHS)
            wseq, wst = want(md, t)
            assert seq.decode("ascii") == wseq, (what, md, t, [i for i, (a, b) in enumerate(zip(seq.decode(), wseq)) if a != b][:10])
            assert st == wst, (what, md, t, st, wst)


def _check_memory(h, mem, ref, what):
    _check_grid(h, lambda md, t: co.consensus_from_memory(mem, ref, md, t, DEPTHS), what)


def _check_tables(h, ref, what, **kw):
    planes, dels = _tables(h)
    _check_grid(h, lambda md, t: co.consensus_from_tables(planes, dels, ref, md, t, DEPTHS), what, **kw)


@pytest.mark.parametrize("name", ["vc_config", "bq13", "all_zero", "bq13_dp3"])
def test_reference_fixture_against_golden_memory(lib, golden_testfile, name):
    g = golden_testfile[name]
    lvc = _lvc(FASTA, g["thresholds"])
    lvc.process_bam(os.path.join(GOLD, "testfile.sam"))
    ref = _ref_of(FASTA)
    _check_memory(lvc._handle, g["memory"], ref, name)
    # the public methods give the same answers
    want, wst = co.consensus_from_memory(g["memory"], ref, 3, 0.5, DEPTHS)
    assert lvc.consensus(minDepth=3, threshold=0.5) == want
    cs = lvc.coverage_summary(DEPTHS, minDepth=3, threshold=0.5)
    assert all(cs[k] == wst[k] for k in co.COUNTERS)
    assert cs["depth_ge"] == dict(zip(DEPTHS, wst["depth_ge"]))
    n = len(ref)
    assert cs["mean_depth"] == wst["depth_sum"] / n and cs["completeness"] == (n - wst["n_N"]) / n
    assert cs["breadth"] == {x: c / n for x, c in zip(DEPTHS, wst["depth_ge"])}
    lvc.close()


@pytest.mark.parametrize("scen", ["mixed_small", "ont_like", "deep_underflow", "amplicon_like", "maxdepth"])
def test_synthetic_scenarios(lib, golden_synth, tmp_path, scen):
    from lvc_b200 import packing
    g = golden_synth[scen]
    fa = _fasta(tmp_path, "chrS", g["ref"])
    for tname, res in g["results"].items():
        th = res["thresholds"]
        lvc = _lvc(fa, th)
        lvc.process_batch(packing.pack_reads(rows_to_tuples(g["reads"]), th["minMQ"]))
        mem = res["memory"] if "memory" in res else lvc.memory
        _check_memory(lvc._handle, mem, g["ref"], f"{scen}/{tname}")
        lvc.close()


def test_crafted_iupac_codes_and_deletions(lib, tmp_path):
    """passing bases that are IUPAC letters or N (groups 1..3), a majority deletion, a position where other codes keep
    the threshold out of reach, a lowercase reference"""
    from lvc_b200 import packing, synth
    ref = synth.random_reference(300, 41).lower()
    q = 30

    def rd(pos, ops, seq):
        return (0, pos, 60, ops, seq, [q] * len(seq))
    reads = []
    for k in range(12):                                  # 20M 5D 20M: columns 30..34 deleted in 12 reads
        s = list(ref[10:30].upper() + ref[35:55].upper())
        if k < 9:
            s[5] = "N"                                   # column 15: 9 N of 15
        if k < 4:
            s[8] = "R"                                   # column 18: R, Y and bases
        elif k < 6:
            s[8] = "Y"
        s[12] = "C" if k < 6 else "T"                    # column 22: 6 C, 6 T, 3 G
        reads.append(rd(10, [(0, 20), (2, 5), (0, 20)], "".join(s)))
    for k in range(3):
        s = list(ref[10:60].upper())
        s[5] = "A" if k else "C"
        s[12] = "G"
        s[22] = "G"                                      # column 32: 3 G against 12 deletions
        reads.append(rd(10, [(0, 50)], "".join(s)))
    for k in range(5):
        reads.append(rd(100 + k, [(0, 30)], ("ACGTM" * 7)[k:k + 30]))
    fa = _fasta(tmp_path, "crafted", ref)
    th = dict(minBQ=13, minMQ=0, minDP=1, minAD=1, ratio=0.0)
    lvc = _lvc(fa, th)
    lvc.process_batch(packing.pack_reads(reads, 0))
    assert any(int(k) >> 8 for k in lvc._handle.plane_keys()), "no plane of groups 1..3"
    mem = lvc.memory
    _check_memory(lvc._handle, mem, ref, "crafted / memory")
    _check_tables(lvc._handle, ref, "crafted / tables")
    assert lvc.consensus(minDepth=1, threshold=0.0)[30:35] == "-----"
    assert lvc.consensus(minDepth=1, threshold=0.5)[15] == "N"          # the bases hold 6 of 15
    assert lvc.consensus(minDepth=1, threshold=0.75)[22] == "Y"
    lvc.close()


def test_ont_tables_with_many_planes(lib):
    from lvc_b200 import capi, synth
    ref = synth.random_reference(29903, 20260199)
    b = synth.ont_batch_fast(20260200, ref, depth=120.0)
    h = capi.Handle(ref.encode("latin-1"), 0, 20, device=0)
    h.push_batch(b.as_capi())
    assert len(h.plane_keys()) >= 60
    _check_tables(h, ref, "ont")
    h.close()


def test_full_config2_amplicon_sample(lib):
    from lvc_b200 import capi, synth
    ref, b = synth.amplicon_sample()
    h = capi.Handle(ref.encode("latin-1"), 30, 20, device=0)
    h.push_batch(b.as_capi())
    _check_tables(h, ref, "config 2")
    h.close()


def _to_device(batch):
    import torch
    from lvc_b200 import capi
    keep = {}
    for name in ("pos", "flag", "mapq", "keep", "cigar_off", "cigar", "seq_off", "seq4", "qual"):
        keep[name] = torch.from_numpy(np.ascontiguousarray(getattr(batch, name)).view(np.uint8).reshape(-1)).to("cuda:0")
    db = capi.Handle.make_batch(batch.n_reads, batch.n_cigar, batch.n_qual,
                                *[keep[k].data_ptr() for k in ("pos", "flag", "mapq", "keep", "cigar_off", "cigar",
                                                               "seq_off", "seq4", "qual")])
    return db, keep


def test_live_batches_checked_after_each(lib, golden_synth, tmp_path):
    """five live batches, the last one enqueued with push_batch_device_async and read by the consensus kernel before
    anything synchronises; after each one the result equals the oracle of the reads seen so far"""
    import torch
    from lvc_b200 import packing
    g = golden_synth["amplicon_like"]
    reads, rows = synth_small.rows_to_reads(g["reads"]), g["reads"]
    th = dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05)
    lvc = _lvc(_fasta(tmp_path, "chrS", g["ref"]), th)
    oc = po.OracleCaller(g["ref"], th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"])
    for k in range(5):
        sel = list(range(k, len(rows), 5))
        batch = packing.pack_reads(rows_to_tuples([rows[i] for i in sel]), th["minMQ"])
        oc.process_reads([reads[i] for i in sel])
        if k < 4:
            lvc.process_batch(batch)
        else:
            h = lvc._handle
            quals = set(int(x) for x in batch.qual[:batch.n_qual] if x >= th["minBQ"])
            for grp in range(4):                       # every key the batch can need has a plane: no replay is possible
                for qv in quals:
                    h.ensure_plane(grp << 8 | qv)
            db, keepalive = _to_device(batch)
            torch.cuda.synchronize()                   # the copies ran on torch's stream, the handle has its own
            h.push_batch_device_async(db)
        _check_memory(lvc._handle, oc.memory, g["ref"], f"batch {k}")
    lvc._handle.check_async()
    lvc.close()


def test_state_restored_by_load_checkpoint(lib, golden_synth, tmp_path):
    g = golden_synth["mixed_small"]
    res = g["results"]["loose"]
    mem = {int(p): {"reference": s["reference"], "totalDepth": s["totalDepth"], "snvs": s["snvs"], "indels": {}}
           for p, s in res["memory"].items()}
    ck = str(tmp_path / "ref.pkl")
    with open(ck, "wb") as fh:
        pickle.dump(mem, fh)
    lvc = _lvc(_fasta(tmp_path, "chrS", g["ref"]), res["thresholds"])
    lvc.load_checkpoint(ck)
    _check_memory(lvc._handle, mem, g["ref"], "checkpoint")
    lvc.close()


def test_sub_range_is_the_slice_of_the_whole(lib, golden_testfile):
    g = golden_testfile["all_zero"]
    lvc = _lvc(FASTA, g["thresholds"])
    lvc.process_bam(os.path.join(GOLD, "testfile.sam"))
    h, ref = lvc._handle, _ref_of(FASTA)
    sites = sorted(int(p) for p in g["memory"])
    for p0, p1 in ((0, h.G), (max(sites[0] - 3, 0), sites[0] + 50), (sites[10], sites[-1] + 1), (sites[5], sites[5]),
                   (h.G - 1, h.G), (0, 1)):
        for md, t in ((0, 0.0), (3, 0.75)):
            whole, _ = h.consensus(md, t, DEPTHS)
            seq, st = h.consensus(md, t, DEPTHS, p0, p1)
            assert seq == whole[p0:p1]
            assert (seq.decode(), st) == co.consensus_from_memory(g["memory"], ref, md, t, DEPTHS, p0, p1), (p0, p1)
    lvc.close()


def test_invalid_arguments(lib):
    from lvc_b200 import capi
    h = capi.Handle(b"ACGT" * 100, 13, 0, device=0)
    for t in (math.nan, -0.1, 1.1):
        with pytest.raises(capi.LvcError) as ei:
            h.consensus(0, t)
        assert ei.value.code == -1
    with pytest.raises(capi.LvcError) as ei:
        h.consensus(0, 0.5, depths=range(1, 10))
    assert ei.value.code == -1
    for p0, p1 in ((0, h.G + 1), (5, 4), (-1, 10)):
        with pytest.raises(capi.LvcError) as ei:
            h.consensus(0, 0.5, p0=p0, p1=p1)
        assert ei.value.code == -1
    seq, st = h.consensus(0, 0.5, depths=range(1, 9))
    assert seq == b"N" * h.G and st["n_N"] == h.G and st["depth_ge"] == [0] * 8
    # kernel time slot 3; slot 4 does not exist
    h.set_timing(True)
    h.consensus(0, 0.5)
    ms, n = h.get_timing(3)
    assert n == 1 and ms > 0
    with pytest.raises(capi.LvcError):
        h.get_timing(4)
    h.close()


def test_calls_between_steps_change_nothing(lib, golden_synth, tmp_path):
    """consensus / coverage_summary / write_consensus between live batches leave records, likelihoods, memory, the CSV
    and later deposits exactly as in a run without them"""
    from lvc_b200 import packing, records
    g = golden_synth["amplicon_like"]
    rows = g["reads"]
    th = dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05)
    fa = _fasta(tmp_path, "chrS", g["ref"])
    plain, probed = _lvc(fa, th), _lvc(fa, th)
    for k in range(5):
        batch = packing.pack_reads(rows_to_tuples([rows[i] for i in range(k, len(rows), 5)]), th["minMQ"])
        plain.process_batch(batch)
        probed.process_batch(batch)
        seq = probed.consensus(minDepth=3, threshold=0.5)
        probed.coverage_summary()
        out = str(tmp_path / f"c{k}.fasta")
        probed.write_consensus(out, minDepth=3, threshold=0.5)
        assert open(out).read() == records.format_consensus_fasta("chrS", seq)
        assert probed.prepare_variants() == plain.prepare_variants()
        assert probed.likelihoods() == plain.likelihoods()
        assert probed.memory == plain.memory
        a, b = str(tmp_path / f"a{k}.csv"), str(tmp_path / f"b{k}.csv")
        plain.write_csv(a)
        probed.write_csv(b)
        assert open(a).read() == open(b).read()
    plain.close()
    probed.close()

"""GPU: insertion counts (lvc_copy_insertions), insertion calls and the spliced consensus against the oracle of
oracle/insertion_oracle.py, in every batch form and push path; the refusals, the overflow report, and that counting
changes nothing else."""
import os
import pickle
import re

import numpy as np
import pytest

from helpers import GOLD, po, synth_small, rows_to_tuples
from oracle import insertion_oracle as io

pytestmark = pytest.mark.gpu

MIN_DEPTHS = (0, 1, 3, 10)                       # the grid of test_gpu_consensus.py
THRESHOLDS = (0.0, 0.07, 0.25, 0.5, 0.75, 1.0)
FASTA = os.path.join(GOLD, "NC_045512.2.synthetic.fasta")
QBINS = (2, 12, 23, 37)
INDEL_DENSE = dict(seed=103, ref_len=700, n_reads=500, len_lo=80, len_hi=250, q_lo=0, q_hi=0, indel_rate=0.12, weird=False,
                   qbins=QBINS)
TH = dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05)


def _ref_of(fasta):
    return open(fasta).read().split("\n", 1)[1].replace("\n", "")


def _fasta(tmp_path, name, ref):
    p = str(tmp_path / f"{name}.fasta")
    with open(p, "w") as fh:
        fh.write(f">{name}\n{ref}\n")
    return p


def _lvc(fasta, th, count=True, **kw):
    from variant_caller.live_variant_caller import LiveVariantCaller
    return LiveVariantCaller(fasta, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0,
                             countInsertions=count, **kw)


def _handle(ref, th, max_keys=1 << 16):
    from lvc_b200 import capi
    h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    h.enable_insertions(max_keys)
    return h


def _tuples(reads):
    return [(r.flag, r.pos, r.mapq, r.cigar, r.seq, r.qual) for r in reads]


def _got(h):
    a = h.copy_insertions()
    keys = [(int(x["pos"]), int(x["len"]), int(x["seq"])) for x in a]
    assert keys == sorted(keys) and len(set(keys)) == len(keys)
    assert (a["depth"] == 0).all()
    return {k: int(c) for k, c in zip(keys, a["count"])}


def _want(reads, G, th, **kw):
    return dict(io.count_insertions(reads, G, th["minBQ"], th["minMQ"], **kw))


def _calls(h, md, t, p0=0, p1=-1):
    return [tuple(int(x[f]) for f in ("pos", "len", "seq", "count", "depth")) for x in h.insertion_calls(md, t, p0, p1)]


def _check_calls(h, ref, counts, what, grid=True):
    """insertion_calls and the spliced consensus against the oracle over the MIN_DEPTHS x THRESHOLDS grid"""
    planes = {int(k): h.copy_plane(int(k)) for k in h.plane_keys()}
    dels = h.copy_dels()
    pairs = [(md, t) for md in MIN_DEPTHS for t in THRESHOLDS] if grid else [(3, 0.5)]
    n_called = 0
    for md, t in pairs:
        depth, letters = io.depth_and_letters_from_tables(planes, dels, ref, md, t)
        want = io.call_insertions(counts, depth, letters, t)
        assert _calls(h, md, t) == want, (what, md, t)
        seq, _ = h.consensus(md, t)
        assert io.splice(seq.decode(), want) == io.splice(letters, want), (what, md, t)
        n_called += len(want)
    return n_called


def test_reference_fixture(lib, golden_testfile):
    """testfile.sam: all four reads carry I ops"""
    ref = _ref_of(FASTA)
    _, reads = po.read_sam(os.path.join(GOLD, "testfile.sam"))
    assert len(reads) == 4 and all(any(op == 1 for op, _ in r.cigar) for r in reads)
    for name in ("vc_config", "bq13", "all_zero", "bq13_dp3"):
        g = golden_testfile[name]
        th = g["thresholds"]
        lvc = _lvc(FASTA, th)
        lvc.process_bam(os.path.join(GOLD, "testfile.sam"))
        want = _want(reads, len(ref), th, overlap_model=po.OVERLAP_HTSLIB_1_13)
        assert _got(lvc._handle) == want and want, name
        for md in MIN_DEPTHS:
            for t in THRESHOLDS:
                depth, letters = io.depth_and_letters_from_memory(g["memory"], len(ref), md, t)
                calls = io.call_insertions(want, depth, letters, t)
                assert _calls(lvc._handle, md, t) == calls, (name, md, t)
                assert lvc.consensus(md, t, insertions=True) == io.splice(letters, calls), (name, md, t)
                assert lvc.insertion_calls(md, t) == [{"pos": p, "seq": io.decode(s, ln), "count": c, "depth": d}
                                                       for p, ln, s, c, d in calls]
        lvc.close()


@pytest.mark.parametrize("scen", ["mixed_small", "ont_like", "amplicon_like", "deep_underflow", "maxdepth", "indel_dense",
                                  "planted"])
def test_synthetic_scenarios(lib, golden_synth, tmp_path, scen):
    from lvc_b200 import packing
    if scen in ("indel_dense", "planted"):
        ref, reads = synth_small.make_scenario(**INDEL_DENSE) if scen == "indel_dense" else _planted()
        results = {k: {"thresholds": v} for k, v in synth_small.THRESHOLDS.items()}
    else:
        g = golden_synth[scen]
        ref, reads, results = g["ref"], synth_small.rows_to_reads(g["reads"]), g["results"]
    n_keys = n_called = 0
    for tname, res in results.items():
        th = res["thresholds"]
        h = _handle(ref, th)
        h.push_batch(packing.pack_reads(_tuples(reads), th["minMQ"]).as_capi())
        want = _want(reads, len(ref), th)
        assert _got(h) == want, (scen, tname)
        n_keys += len(want)
        n_called += _check_calls(h, ref, want, f"{scen}/{tname}")
        h.close()
    if scen in ("mixed_small", "ont_like", "indel_dense", "planted"):
        assert n_keys > 0
    if scen == "planted":
        assert n_called > 0


def _forms(reads, th):
    """the same reads in every batch form the push paths take"""
    from lvc_b200 import packing
    raw = packing.pack_reads(_tuples(reads), th["minMQ"], max_depth=60)
    assert not (raw.keep & 1).all(), "the scenario must drop reads at max_depth"
    coded = raw.with_quality_codes()
    assert coded.qcode is not None
    based = coded.with_base_codes(th["minBQ"])
    assert based.scode is not None
    return dict(bytes=raw, codes=coded, base_codes=based, admitted_only=raw.admitted_only(),
                admitted_codes=coded.admitted_only(), pinned_bytes=packing.pin_batch(raw), pinned_codes=packing.pin_batch(coded),
                pinned_base_codes=packing.pin_batch(based))


@pytest.mark.parametrize("tname", ["strict", "loose", "zero"])
def test_every_batch_form(lib, tname):
    th = synth_small.THRESHOLDS[tname]
    ref, reads = synth_small.make_scenario(**dict(INDEL_DENSE, n_reads=900, ref_len=400))
    want = _want(reads, len(ref), th, max_depth=60)
    assert want
    for form, b in _forms(reads, th).items():
        for impl in (0, 1, 5):
            h = _handle(ref, th)
            h.set_impl(impl)
            h.push_batch(b.as_capi())
            assert _got(h) == want, (form, impl)
            h.close()


def test_device_and_async_pushes(lib):
    import torch
    from test_gpu_consensus import _to_device
    from lvc_b200 import packing
    th = TH
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    batch = packing.pack_reads(_tuples(reads), th["minMQ"])
    want = _want(reads, len(ref), th)
    db, keep = _to_device(batch)
    torch.cuda.synchronize()
    h = _handle(ref, th)
    h.push_batch_device(db)
    assert _got(h) == want
    # async: every key the batch needs has a plane (no replay is possible); two pushes count twice
    h.push_batch_device_async(db)
    h.check_async()
    assert _got(h) == {k: 2 * n for k, n in want.items()}
    h.close()
    h = _handle(ref, th)
    for grp in range(4):
        for q in set(int(x) for x in batch.qual[:batch.n_qual] if x >= th["minBQ"]):
            h.ensure_plane(grp << 8 | q)
    h.push_batch_device_async(db)
    assert _got(h) == want                             # the query runs after the enqueued kernels
    h.check_async()
    h.close()
    del keep


def test_replay_counts_once(lib):
    """N bases make a key of allele group 3 that has no plane yet: the deposit runs again for it; the counts are made once"""
    from lvc_b200 import packing
    th = TH
    ref = synth_small.make_scenario(**INDEL_DENSE)[0]
    reads = []
    for k in range(40):
        s = list(ref[100:150] + "GAGCCAGAA" + ref[150:200])
        if k % 3 == 0:
            s[10] = "N"
        reads.append(po.Read(0, 100, 60, [(0, 50), (1, 9), (0, 50)], "".join(s), [30] * 109))
    h = _handle(ref, th)
    before = h.launch_count
    h.push_batch(packing.pack_reads(_tuples(reads), 0).as_capi())
    assert h.launch_count - before == 3              # deposit, insertion counts, replayed deposit
    assert any(int(k) >> 8 == 3 for k in h.plane_keys())
    assert _got(h) == _want(reads, len(ref), th) == {(149, 9, io.encode("GAGCCAGAA")): 40}
    h.close()


def test_several_batches_equal_one(lib):
    from lvc_b200 import packing
    th = TH
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    b = packing.pack_reads(_tuples(reads), th["minMQ"])
    one, many = _handle(ref, th), _handle(ref, th)
    one.push_batch(b.as_capi())
    cuts = [0, 97, 260, 261, b.n_reads]
    for a, z in zip(cuts, cuts[1:]):
        many.push_batch(b.slice(a, z).as_capi())
    assert _got(one) == _got(many) == _want(reads, len(ref), th)
    _check_calls(many, ref, _want(reads, len(ref), th), "several batches", grid=False)
    one.close(); many.close()


PLANTED = {149: "GAT", 299: "C", 519: "TTAG"}           # anchor -> inserted bases


def _planted(seed=7):
    """the indel_dense reference, a quarter of its reads and 400 reads of which ~90 % carry the insertion of PLANTED at
    an anchor they cover: random indels alone never reach a call, these do"""
    import random
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    rng = random.Random(seed)
    extra = []
    for _ in range(400):
        pos = rng.randrange(80, len(ref) - 110)
        ops, seq, r = [], "", pos
        for a in sorted(PLANTED):
            if pos <= a < pos + 99 and rng.random() < 0.9:
                ops.append((0, a + 1 - r))
                seq += ref[r:a + 1]
                ops.append((1, len(PLANTED[a])))
                seq += PLANTED[a]
                r = a + 1
        ops.append((0, pos + 100 - r))
        seq += ref[r:pos + 100]
        extra.append(po.Read(0, pos, 60, ops, seq, [rng.choice((23, 37)) for _ in seq]))
    return ref, sorted(reads[::4] + extra, key=lambda x: x.pos)


def test_sub_ranges(lib):
    from lvc_b200 import packing
    th = TH
    ref, reads = _planted()
    h = _handle(ref, th)
    h.push_batch(packing.pack_reads(_tuples(reads), th["minMQ"]).as_capi())
    counts = _want(reads, len(ref), th)
    planes = {int(k): h.copy_plane(int(k)) for k in h.plane_keys()}
    dels = h.copy_dels()
    for md, t in ((0, 0.0), (3, 0.25), (10, 0.5)):
        depth, letters = io.depth_and_letters_from_tables(planes, dels, ref, md, t)
        whole = _calls(h, md, t)
        assert whole
        for p0, p1 in ((0, len(ref)), (0, 1), (whole[0][0], whole[0][0] + 1), (whole[0][0] + 1, len(ref)),
                       (200, 450), (len(ref) - 1, len(ref)), (300, 300)):
            got = _calls(h, md, t, p0, p1)
            assert got == [c for c in whole if p0 <= c[0] < p1] == io.call_insertions(counts, depth, letters, t, p0, p1)
    h.close()


def test_ba1_like_insertion(lib, tmp_path):
    """a 9-base insertion (spike ins214EPE: GAG CCA GAA) in most reads, a one-base variant of it, unresolved and
    low-quality insertions at the same anchor, reads without it"""
    from lvc_b200 import synth
    ref = synth.random_reference(1000, 214).upper()
    ins, variant = "GAGCCAGAA", "GAGCCAGAT"
    rows = []

    def add(seq_ins, n, anchor_q=30, ins_q=30):
        for _ in range(n):
            q = [30] * 50 + [ins_q] * len(seq_ins) + [30] * 50
            q[49] = anchor_q
            rows.append((0, 450, 60, [(0, 50), (1, len(seq_ins)), (0, 50)] if seq_ins else [(0, 100)],
                         ref[450:500] + seq_ins + ref[500:550], q))
    add(ins, 20)
    add(variant, 4)
    add("GAGCCNGAA", 2)                               # unresolved: an N
    add(ins, 1, ins_q=5)                              # unresolved: low-quality inserted bases
    add(ins, 2, anchor_q=5)                           # not counted, and not in the depth at the anchor
    add("", 3)
    from lvc_b200 import packing
    lvc = _lvc(_fasta(tmp_path, "spike", ref), dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05))
    lvc.process_batch(packing.pack_reads(rows, 0))
    assert _got(lvc._handle) == {(499, 0, 0): 3, (499, 9, io.encode(ins)): 20, (499, 9, io.encode(variant)): 4}
    assert lvc.insertion_calls(10, 0.5) == [{"pos": 499, "seq": ins, "count": 20, "depth": 30}]
    cons = lvc.consensus(10, 0.5, insertions=True)
    assert cons[450:509] == ref[450:500] + ins and cons[509:559] == ref[500:550] and len(cons) == len(ref) + 9
    assert lvc.insertion_calls(10, 0.67) == []                           # 20 / 30 < 0.67
    assert lvc.consensus(10, 0.67, insertions=True) == lvc.consensus(10, 0.67)
    assert lvc.insertion_calls(31, 0.0) == []                            # 'N' at the anchor
    out = str(tmp_path / "c.fasta")
    lvc.write_consensus(out, 10, 0.5, insertions=True)
    assert open(out).read().split("\n", 1)[1].replace("\n", "") == cons.replace("-", "")
    lvc.close()


def test_refusals_reset_and_overflow(lib, tmp_path):
    from lvc_b200 import capi, packing
    th = TH
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    batch = packing.pack_reads(_tuples(reads), th["minMQ"])
    want = _want(reads, len(ref), th)
    h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    with pytest.raises(capi.LvcError) as ei:
        h.copy_insertions()                                              # counting is off
    assert ei.value.code == -1
    with pytest.raises(capi.LvcError):
        h.get_timing(4)
    h.push_batch(batch.as_capi())
    with pytest.raises(capi.LvcError) as ei:
        h.enable_insertions(1 << 10)                                     # after a push
    assert ei.value.code == -1 and "lvc_reset" in str(ei.value)
    h.reset()
    h.enable_insertions(1 << 10)
    h.set_timing(True)
    h.push_batch(batch.as_capi())
    ms, n = h.get_timing(4)
    assert n == 1 and ms > 0
    assert _got(h) == want
    with pytest.raises(capi.LvcError) as ei:
        h.peer_attach(0, [None, b"x" * 64])
    assert ei.value.code == -1 and "insertions" in str(ei.value)
    # imports: the tables hold counts the insertion table does not cover
    for imp in (lambda: h.import_dels(h.copy_dels(), True), lambda: h.import_covdiff(np.zeros(h.G + 1, np.int32), True),
                lambda: h.import_plane(int(h.plane_keys()[0]), h.copy_plane(int(h.plane_keys()[0]))),
                lambda: h.import_first(0, h.copy_first(0))):
        imp()
        for q in (h.copy_insertions, lambda: h.insertion_calls(0, 0.0)):
            with pytest.raises(capi.LvcError) as ei:
                q()
            assert ei.value.code == -1 and "lvc_reset" in str(ei.value)
        with pytest.raises(capi.LvcError):
            h.enable_insertions(1 << 10)
        h.reset()                                                        # counting stays on, the table is empty
        assert _got(h) == {}
        h.push_batch(batch.as_capi())
        assert _got(h) == want
    h.close()
    # overflow: 2 keys -> 4 slots
    h = _handle(ref, th, max_keys=2)
    h.push_batch(batch.as_capi())
    assert len(want) > 4
    for q in (h.copy_insertions, lambda: h.insertion_calls(0, 0.0)):
        with pytest.raises(capi.LvcError) as ei:
            q()
        assert ei.value.code == -3 and re.search(r"\b[1-9]\d* insertion\(s\) found no free slot .* \(4 slots\)", str(ei.value))
    h.close()
    # arguments
    h = _handle(ref, th)
    for bad in (dict(md=0, t=1.5), dict(md=0, t=float("nan"))):
        with pytest.raises(capi.LvcError):
            h.insertion_calls(bad["md"], bad["t"])
    for p0, p1 in ((0, h.G + 1), (5, 4), (-1, 10)):
        with pytest.raises(capi.LvcError):
            h.insertion_calls(0, 0.0, p0, p1)
    with pytest.raises(capi.LvcError):
        h.enable_insertions(0)
    h.close()


def test_counting_changes_nothing_else(lib, golden_synth, tmp_path):
    """planes, deletions, coverage, first-seen ordinals and records are those of a caller that does not count; one more
    launch per push with counting on, none without"""
    from lvc_b200 import packing
    g = golden_synth["amplicon_like"]
    rows = g["reads"]
    fa = _fasta(tmp_path, "chrS", g["ref"])
    ref2, reads2 = synth_small.make_scenario(**INDEL_DENSE)
    for fasta, batches in ((fa, [packing.pack_reads(rows_to_tuples([rows[i] for i in range(k, len(rows), 3)]), 0)
                                 for k in range(3)]),
                           (_fasta(tmp_path, "dense", ref2), [packing.pack_reads(_tuples(reads2), 0)])):
        off, on = _lvc(fasta, TH, count=False), _lvc(fasta, TH)
        for b in batches:
            n0, n1 = off._handle.launch_count, on._handle.launch_count
            off.process_batch(b)
            on.process_batch(b)
            assert on._handle.launch_count - n1 == off._handle.launch_count - n0 + 1
            ho, hn = off._handle, on._handle
            assert sorted(ho.plane_keys().tolist()) == sorted(hn.plane_keys().tolist())
            for k in ho.plane_keys():
                assert np.array_equal(ho.copy_plane(int(k)), hn.copy_plane(int(k)))
            assert np.array_equal(ho.copy_dels(), hn.copy_dels()) and np.array_equal(ho.copy_covdiff(), hn.copy_covdiff())
            for grp in range(4):
                a, c = ho.copy_first(grp), hn.copy_first(grp)
                assert (a is None) == (c is None) and (a is None or np.array_equal(a, c))
            assert off.prepare_variants() == on.prepare_variants()
            assert off.memory == on.memory
            assert off.consensus(3, 0.5) == on.consensus(3, 0.5)
        with pytest.raises(ValueError):
            off.consensus(3, 0.5, insertions=True)
        off.close(); on.close()
    # the launches of a push without counting: the deposit kernel only (no replay: every plane exists)
    lvc = _lvc(fa, TH, count=False)
    b = packing.pack_reads(rows_to_tuples(rows), 0)
    lvc.process_batch(b)
    n0 = lvc._handle.launch_count
    lvc.process_batch(b)
    assert lvc._handle.launch_count - n0 == 1
    lvc.close()


def test_checkpoint_and_reset(lib, golden_synth, tmp_path):
    g = golden_synth["mixed_small"]
    res = g["results"]["loose"]
    from lvc_b200 import capi, packing
    fa = _fasta(tmp_path, "chrS", g["ref"])
    lvc = _lvc(fa, res["thresholds"])
    lvc.process_batch(packing.pack_reads(rows_to_tuples(g["reads"]), res["thresholds"]["minMQ"]))
    ck = str(tmp_path / "ck.pkl")
    lvc.create_checkpoint(ck)
    lvc.load_checkpoint(ck)
    with pytest.raises(capi.LvcError) as ei:
        lvc.consensus(3, 0.5, insertions=True)
    assert ei.value.code == -1
    with pytest.raises(capi.LvcError):
        lvc.insertion_calls(3, 0.5)
    lvc.reset_memory()
    assert lvc.consensus(3, 0.5, insertions=True) == "N" * len(g["ref"])
    lvc.process_batch(packing.pack_reads(rows_to_tuples(g["reads"]), res["thresholds"]["minMQ"]))
    reads = synth_small.rows_to_reads(g["reads"])
    assert _got(lvc._handle) == _want(reads, len(g["ref"]), res["thresholds"])
    with open(ck, "rb") as fh:
        assert pickle.load(fh) == lvc.memory                             # checkpoints carry no insertions
    lvc.close()

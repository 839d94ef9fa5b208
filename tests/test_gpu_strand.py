"""GPU: strand counts (lvc_enable_strand_counts / lvc_strand_counts) against the oracle of oracle/strand_oracle.py, exactly,
in every batch form and push path; a cross-check at scale that needs no oracle; the refusals and the lifetime of the
counts; strand_bias and the opt-in VCF; and that counting changes nothing else."""
import dataclasses
import os

import numpy as np
import pytest

from helpers import GOLD, po, synth_small, rows_to_tuples
from oracle import strand_oracle as so
from test_gpu_insertions import FASTA, INDEL_DENSE, TH, _forms, _fasta, _ref_of, _tuples

pytestmark = pytest.mark.gpu

NIBBLE_CHARS = po.NIBBLE_CHARS
ROW_LETTER = "".join(NIBBLE_CHARS[n] for n in so.GS_TO_NIBBLE) + "-"        # table row -> query letter
WEIRD = dict(INDEL_DENSE, seed=211, weird=True)


def _table(h, G):
    """(fwd, rev) uint32 [17, G]: every cell through lvc_strand_counts"""
    pos = np.tile(np.arange(G, dtype=np.int32), so.ROWS)
    letters = "".join(c * G for c in ROW_LETTER)
    fwd, rev = h.strand_counts(pos, letters)
    return fwd.reshape(so.ROWS, G), rev.reshape(so.ROWS, G)


def _check(h, want):
    fwd, rev = _table(h, want[0].shape[1])
    assert np.array_equal(rev, want[1])
    assert np.array_equal(fwd, want[0])


def _want(reads, G, th, **kw):
    return so.count_strands(reads, G, th["minBQ"], th["minMQ"], **kw)


def _handle(ref, th):
    from lvc_b200 import capi
    h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    h.enable_strand_counts()
    return h


def test_reference_fixture(lib, golden_testfile, tmp_path):
    """testfile.sam as it is (four forward reads) and with reads 1 and 3 on the reverse strand"""
    from variant_caller.live_variant_caller import LiveVariantCaller
    ref = _ref_of(FASTA)
    src = os.path.join(GOLD, "testfile.sam")
    lines = open(src).read().split("\n")
    k = 0
    for i, line in enumerate(lines):
        if line and not line.startswith("@"):
            t = line.split("\t")
            if k % 2:
                t[1] = str(int(t[1]) | 0x10)
            lines[i] = "\t".join(t)
            k += 1
    flipped = str(tmp_path / "flipped.sam")
    open(flipped, "w").write("\n".join(lines))
    n_rev = 0
    for sam in (src, flipped):
        _, reads = po.read_sam(sam)
        for name in ("vc_config", "bq13", "all_zero", "bq13_dp3"):
            th = golden_testfile[name]["thresholds"]
            lvc = LiveVariantCaller(FASTA, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0,
                                    countStrands=True)
            lvc.process_bam(sam)
            want = _want(reads, len(ref), th, overlap_model=po.OVERLAP_HTSLIB_1_13)
            _check(lvc._handle, want)
            n_rev += int(want[1].sum())
            lvc.close()
    assert n_rev > 0


@pytest.mark.parametrize("scen", ["mixed_small", "ont_like", "amplicon_like", "deep_underflow", "maxdepth", "indel_dense",
                                  "weird"])
def test_synthetic_scenarios(lib, golden_synth, scen):
    from lvc_b200 import packing
    if scen in ("indel_dense", "weird"):
        ref, reads = synth_small.make_scenario(**(INDEL_DENSE if scen == "indel_dense" else WEIRD))
        results = {k: {"thresholds": v} for k, v in synth_small.THRESHOLDS.items()}
    else:
        g = golden_synth[scen]
        ref, reads, results = g["ref"], synth_small.rows_to_reads(g["reads"]), g["results"]
    n_rev = 0
    for tname, res in results.items():
        th = res["thresholds"]
        h = _handle(ref, th)
        h.push_batch(packing.pack_reads(_tuples(reads), th["minMQ"]).as_capi())
        want = _want(reads, len(ref), th)
        _check(h, want)
        n_rev += int(want[1].sum())
        if scen == "weird":
            assert want[1][4:16].sum() > 0                 # nibble codes other than A/C/G/T on reverse reads
        h.close()
    assert n_rev > 0


@pytest.mark.parametrize("tname", ["strict", "loose", "zero"])
def test_every_batch_form(lib, tname):
    th = synth_small.THRESHOLDS[tname]
    ref, reads = synth_small.make_scenario(**dict(INDEL_DENSE, n_reads=900, ref_len=400))
    want = _want(reads, len(ref), th, max_depth=60)
    assert want[1].sum() > 0 and want[1][so.DEL].sum() > 0
    for form, b in _forms(reads, th).items():
        for impl in (0, 1, 5):
            h = _handle(ref, th)
            h.set_impl(impl)
            h.push_batch(b.as_capi())
            _check(h, want)
            h.close()


def test_device_and_async_pushes(lib):
    import torch
    from test_gpu_consensus import _to_device
    from lvc_b200 import packing
    th = TH
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    batch = packing.pack_reads(_tuples(reads), th["minMQ"])
    want = _want(reads, len(ref), th)
    twice = (2 * want[0], 2 * want[1])
    db, keep = _to_device(batch)
    torch.cuda.synchronize()
    h = _handle(ref, th)
    h.push_batch_device(db)
    _check(h, want)
    h.push_batch_device_async(db)
    h.check_async()
    _check(h, twice)
    h.close()
    h = _handle(ref, th)
    for grp in range(4):
        for q in set(int(x) for x in batch.qual[:batch.n_qual] if x >= th["minBQ"]):
            h.ensure_plane(grp << 8 | q)
    h.push_batch_device_async(db)
    _check(h, want)                                  # the query runs after the enqueued kernels
    h.check_async()
    h.close()
    del keep


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
    want = _want(reads, len(ref), th)
    _check(one, want)
    _check(many, want)
    one.close(); many.close()


def test_replay_counts_once(lib):
    """N bases make a key of allele group 3 that has no plane yet: the deposit runs again for it; the counts are made once"""
    from lvc_b200 import packing
    th = TH
    ref = synth_small.make_scenario(**INDEL_DENSE)[0]
    reads = []
    for k in range(40):
        s = list(ref[100:200])
        if k % 3 == 0:
            s[10] = "N"
        reads.append(po.Read(0x10 if k % 2 else 0, 100, 60, [(0, 100)], "".join(s), [30] * 100))
    h = _handle(ref, th)
    before = h.launch_count
    h.push_batch(packing.pack_reads(_tuples(reads), 0).as_capi())
    assert h.launch_count - before == 3              # deposit, strand counts, replayed deposit
    assert any(int(k) >> 8 == 3 for k in h.plane_keys())
    want = _want(reads, len(ref), th)
    assert int(want[1][so.row_of("N"), 110]) == 7 and int(want[0][so.row_of("N"), 110]) == 7
    _check(h, want)
    h.close()


def test_lifetime_and_refusals(lib, tmp_path):
    from lvc_b200 import capi, packing
    th = TH
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    G = len(ref)
    batch = packing.pack_reads(_tuples(reads), th["minMQ"])
    want = _want(reads, G, th)
    zero = (np.zeros_like(want[0]), np.zeros_like(want[1]))
    h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    with pytest.raises(capi.LvcError) as ei:
        h.strand_counts([1], "A")                                         # counting is off
    assert ei.value.code == -1
    with pytest.raises(capi.LvcError):
        h.get_timing(6)
    h.push_batch(batch.as_capi())
    with pytest.raises(capi.LvcError) as ei:
        h.enable_strand_counts()                                          # the tables hold counts
    assert ei.value.code == -1 and "lvc_reset" in str(ei.value)
    h.reset()
    h.enable_strand_counts()
    h.enable_strand_counts()                                              # again: a no-op
    _check(h, zero)
    h.set_timing(True)
    h.push_batch(batch.as_capi())
    ms, n = h.get_timing(6)
    assert n == 1 and ms > 0
    _check(h, want)
    # unknown letters and positions outside [0, G)
    for pos, letter, msg in (([G], "A", str(G)), ([-1], "A", "-1"), ([3], "X", "0x58"), ([3], "*", "0x2a"),
                             ([3], "\0", "0x00")):
        with pytest.raises(capi.LvcError) as ei:
            h.strand_counts(pos, letter)
        assert ei.value.code == -1 and msg in str(ei.value), (msg, str(ei.value))
    # letters in either case
    p = [int(x) for x in np.nonzero(want[1][so.row_of("A")])[0][:5]]
    assert np.array_equal(h.strand_counts(p, "a" * len(p))[1], h.strand_counts(p, "A" * len(p))[1])
    assert h.strand_counts([], "")[0].size == 0
    h.reset()                                                             # clears the counts, keeps counting on
    _check(h, zero)
    h.push_batch(batch.as_capi())
    _check(h, want)
    # an import: the query fails until lvc_reset
    h.import_dels(h.copy_dels(), True)
    with pytest.raises(capi.LvcError) as ei:
        h.strand_counts([1], "A")
    assert ei.value.code == -1 and "lvc_reset" in str(ei.value)
    h.reset()
    h.push_batch(batch.as_capi())
    _check(h, want)
    h.import_plane(int(h.plane_keys()[0]), h.copy_plane(int(h.plane_keys()[0])))
    with pytest.raises(capi.LvcError):
        h.strand_counts([1], "A")
    h.close()


def test_peer_attach_refused(lib):
    """a handle that counts strands refuses peer tables, before it opens anything"""
    from lvc_b200 import capi
    ref = synth_small.make_scenario(**INDEL_DENSE)[0]
    h = _handle(ref, TH)
    with pytest.raises(capi.LvcError) as ei:
        h.peer_attach(0, [None, b"x" * 64])
    assert ei.value.code == -1 and "counts strands" in str(ei.value)
    h.close()


def _lvc(fasta, th, **kw):
    from variant_caller.live_variant_caller import LiveVariantCaller
    return LiveVariantCaller(fasta, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0, **kw)


def test_strand_bias_and_vcf(lib, tmp_path):
    """strand_bias on the records, in their order, against the oracle's counts; the opt-in VCF; the default VCF"""
    from lvc_b200 import packing, records
    th = TH
    ref, reads = synth_small.make_scenario(**dict(WEIRD, n_reads=900))
    fa = _fasta(tmp_path, "w", ref)
    off, on = _lvc(fa, th), _lvc(fa, th, countStrands=True)
    b = packing.pack_reads(_tuples(reads), th["minMQ"])
    for c in (off, on):
        c.process_batch(b)
    fwd, rev = _want(reads, len(ref), th)
    vs = on.prepare_variants()
    assert vs and vs == off.prepare_variants()
    sb = on.strand_bias()
    assert len(sb) == len(vs)
    for v, s in zip(vs, sb):
        p = v["start"]
        assert (s["start"], s["alleles"]) == (p, v["alleles"])
        rr, ar = so.row_of(v["alleles"][0]), so.row_of(v["alleles"][1])
        assert (s["ref_fwd"], s["ref_rev"], s["alt_fwd"], s["alt_rev"]) == \
            (int(fwd[rr, p]), int(rev[rr, p]), int(fwd[ar, p]), int(rev[ar, p]))
        assert s["alt_fwd"] + s["alt_rev"] == v["info"]["AD"]
        assert s["fs"] == records.fisher_strand(s["ref_fwd"], s["ref_rev"], s["alt_fwd"], s["alt_rev"])
    assert on.strand_bias(vs[::-1]) == sb[::-1]
    with pytest.raises(ValueError):
        off.strand_bias()
    a, d, e = (str(tmp_path / f"{k}.vcf") for k in "ade")
    off.write_vcf(a)
    on.write_vcf(d)
    on.write_vcf(e, strandBias=True)
    plain = open(a).read()
    assert open(d).read() == plain
    text = open(e).read()
    assert text == records.format_vcf(vs, [("w", len(ref))], sb)
    body = [ln for ln in text.split("\n") if ln and not ln.startswith("#")]
    assert len(body) == len(vs) and all(";DP4=" in ln and ";FS=" in ln and ";SOR=" in ln for ln in body)
    assert sum(ln.startswith("##INFO=<ID=DP4,") for ln in text.split("\n")) == 1
    off.close(); on.close()


def test_checkpoint_fails_until_reset(lib, golden_synth, tmp_path):
    from lvc_b200 import capi, packing
    g = golden_synth["mixed_small"]
    th = g["results"]["loose"]["thresholds"]
    lvc = _lvc(_fasta(tmp_path, "chrS", g["ref"]), th, countStrands=True)
    b = packing.pack_reads(rows_to_tuples(g["reads"]), th["minMQ"])
    lvc.process_batch(b)
    before = lvc.strand_bias()
    ck = str(tmp_path / "ck.pkl")
    lvc.create_checkpoint(ck)
    lvc.load_checkpoint(ck)
    with pytest.raises(capi.LvcError) as ei:
        lvc.strand_bias()
    assert ei.value.code == -1
    lvc.reset_memory()
    lvc.process_batch(b)
    assert lvc.strand_bias() == before
    lvc.close()


def test_counting_changes_nothing_else(lib, golden_synth, tmp_path):
    """planes, deletions, coverage, first-seen ordinals, records, the default VCF, the consensus and the insertion and
    linkage counts are those of callers that do not count strands; exactly one more launch per push"""
    from lvc_b200 import packing
    g = golden_synth["amplicon_like"]
    rows = g["reads"]
    fa = _fasta(tmp_path, "chrS", g["ref"])
    ref2, reads2 = synth_small.make_scenario(**INDEL_DENSE)
    for fasta, ref, batches in (
            (fa, g["ref"], [packing.pack_reads(rows_to_tuples([rows[i] for i in range(k, len(rows), 3)]), 0) for k in range(3)]),
            (_fasta(tmp_path, "dense", ref2), ref2, [packing.pack_reads(_tuples(reads2), 0)])):
        sites = [(p, {"A": "C", "C": "G", "G": "T", "T": "A"}[ref[p].upper()]) for p in range(20, len(ref) - 20, 37)
                 if ref[p].upper() in "ACGT"]
        off = _lvc(fasta, TH, countInsertions=True)
        on = _lvc(fasta, TH, countInsertions=True, countStrands=True)
        for c in (off, on):
            c.track_linkage(sites, 100)
        for b in batches:
            n = [c._handle.launch_count for c in (off, on)]
            for c in (off, on):
                c.process_batch(b)
            d = [c._handle.launch_count - n0 for c, n0 in zip((off, on), n)]
            assert d[1] == d[0] + 1
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
            assert off.consensus(3, 0.5, insertions=True) == on.consensus(3, 0.5, insertions=True)
            assert np.array_equal(ho.copy_insertions(), hn.copy_insertions())
            assert np.array_equal(ho.copy_linkage(), hn.copy_linkage())
        va, vb = str(tmp_path / "a.vcf"), str(tmp_path / "b.vcf")
        off.write_vcf(va); on.write_vcf(vb)
        assert open(va).read() == open(vb).read()
        assert on.strand_bias()
        for c in (off, on):
            c.close()


def _rev_crosscheck(ref, batch, th):
    """deposit `batch` into a handle that counts strands, and into a plain handle a copy whose forward reads are dropped
    (keep bit 0 cleared): the plain handle's plane sums and dels equal the first handle's rev, exactly"""
    from lvc_b200 import capi
    G = len(ref)
    h = _handle(ref, th)
    h.push_batch(batch.as_capi())
    keep = batch.keep.copy()
    keep[(batch.flag & 0x10) == 0] &= np.uint8(0xFE)
    plain = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    plain.push_batch(dataclasses.replace(batch, keep=keep).as_capi())
    want = np.zeros((so.ROWS, G), dtype=np.uint64)
    for k in plain.plane_keys():
        pl = plain.copy_plane(int(k))
        g = int(k) >> 8
        want[4 * g:4 * g + 4] += pl.T
    want[so.DEL] = plain.copy_dels()
    fwd, rev = _table(h, G)
    assert rev.sum() > 0 and fwd.sum() > 0
    assert np.array_equal(rev.astype(np.uint64), want)
    h.close(); plain.close()


def test_at_scale_config2(lib):
    """a config-2-sized amplicon batch as the packer hands it over: admitted reads, 2-bit quality and base codes"""
    from lvc_b200 import synth
    ref, b = synth.amplicon_sample()
    b2 = b.admitted_only().with_quality_codes().with_base_codes(30)
    del b
    _rev_crosscheck(ref, b2, dict(minBQ=30, minMQ=20))


def test_at_scale_ont(lib):
    from lvc_b200 import synth
    ref = synth.random_reference(29903, 20260199)
    _rev_crosscheck(ref, synth.ont_batch_fast(20260200, ref), dict(minBQ=30, minMQ=20))

"""GPU: variant linkage counts (lvc_copy_linkage) against the oracle of oracle/linkage_oracle.py, exactly, in every batch
form and push path; known linkage; the refusals and the lifetime of the counts; and that counting changes nothing else."""
import os
import random
from collections import Counter

import numpy as np
import pytest

from helpers import GOLD, po, synth_small, rows_to_tuples
from oracle import linkage_oracle as lo
from test_gpu_insertions import FASTA, INDEL_DENSE, TH, _forms, _fasta, _ref_of, _tuples

pytestmark = pytest.mark.gpu


def _span(pos, want=300):
    """the widest span of `want`, 150, 100, ... that keeps at most 64 sites inside any window"""
    for s in (want, 150, 100, 50, 25, 10, 5, 2, 1):
        if lo.window(pos, s) <= lo.MAX_WINDOW:
            return s


def _sites(reads, ref, th, dels=True, max_depth=po.MAX_DEPTH, min_reads=2):
    """one site per position: its most frequent non-reference allele (A/C/G/T, or '-' for deletion entries) among the
    entries that pass the quality test, if at least min_reads reads carry it"""
    out = []
    for col, entries in po.pileup_columns(reads, th["minMQ"], max_depth):
        rl = ref[col].upper() if col < len(ref) else "N"
        if rl not in "ACGT":
            continue
        c = Counter()
        for _, r, is_del, is_skip, qpos in entries:
            if (r.qual[qpos] if qpos < len(r.qual) else 0) < th["minBQ"]:
                continue
            a = "-" if is_del or is_skip else r.seq[qpos]
            if a in "ACGT-" and a != rl and (dels or a != "-"):
                c[a] += 1
        if c:
            a = max(sorted(c), key=lambda x: c[x])
            if c[a] >= min_reads:
                out.append((col, a))
    return out


def _set(h, sites, span):
    h.set_linkage_sites([p for p, _ in sites], "".join(a for _, a in sites), span)


def _want(reads, ref, sites, span, th, **kw):
    return lo.count_linkage(reads, ref, [p for p, _ in sites], "".join(a for _, a in sites), span, th["minBQ"],
                            th["minMQ"], **kw)


def _check(h, sites, span, want):
    got = h.copy_linkage()
    prs = lo.pairs([p for p, _ in sites], span)
    assert got["pos_a"].tolist() == [sites[a][0] for a, _ in prs]
    assert got["pos_b"].tolist() == [sites[b][0] for _, b in prs]
    assert bytes(got["alt_a"]).decode() == "".join(sites[a][1] for a, _ in prs)
    assert bytes(got["alt_b"]).decode() == "".join(sites[b][1] for _, b in prs)
    assert np.array_equal(got["count"], want)


def _handle(ref, th, sites, span):
    from lvc_b200 import capi
    h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    _set(h, sites, span)
    return h


def test_reference_fixture(lib, golden_testfile):
    """testfile.sam: sites = every position's most frequent non-reference allele with at least 2 reads in the oracle's
    memory"""
    from variant_caller.live_variant_caller import LiveVariantCaller
    ref = _ref_of(FASTA)
    _, reads = po.read_sam(os.path.join(GOLD, "testfile.sam"))
    n_sites = 0
    for name in ("vc_config", "bq13", "all_zero", "bq13_dp3"):
        th = golden_testfile[name]["thresholds"]
        oc = po.OracleCaller(ref, th["minBQ"], th["minMQ"], 1, 1, 0.0, overlap_model=po.OVERLAP_HTSLIB_1_13)
        oc.process_reads(reads)
        sites = []
        for p in sorted(oc.memory):
            n = {b: len(q) for b, q in oc.memory[p]["snvs"].items() if b in "ACGT" and b != ref[p].upper()}
            if ref[p].upper() in "ACGT" and n and max(n.values()) >= 2:
                sites.append((p, max(sorted(n), key=lambda b: n[b])))
        if not sites:                                    # minBQ 30: no allele of these ONT reads reaches 2 reads
            continue
        n_sites += len(sites)
        span = _span([p for p, _ in sites])
        lvc = LiveVariantCaller(FASTA, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0)
        lvc.track_linkage(sites, span)
        lvc.process_bam(os.path.join(GOLD, "testfile.sam"))
        want = _want(reads, ref, sites, span, th, overlap_model=po.OVERLAP_HTSLIB_1_13)
        assert want[:, 1, 1].sum() > 0, name
        _check(lvc._handle, sites, span, want)
        lvc.close()
    assert n_sites > 0


@pytest.mark.parametrize("scen", ["mixed_small", "ont_like", "amplicon_like", "deep_underflow", "maxdepth", "indel_dense"])
def test_synthetic_scenarios(lib, golden_synth, scen):
    from lvc_b200 import packing
    if scen == "indel_dense":
        ref, reads = synth_small.make_scenario(**INDEL_DENSE)
        results = {k: {"thresholds": v} for k, v in synth_small.THRESHOLDS.items()}
    else:
        g = golden_synth[scen]
        ref, reads, results = g["ref"], synth_small.rows_to_reads(g["reads"]), g["results"]
    n_pairs = 0
    for tname, res in results.items():
        th = res["thresholds"]
        sites = _sites(reads, ref, th)
        if not sites:
            continue
        if scen == "indel_dense":
            assert any(a == "-" for _, a in sites) and any(a != "-" for _, a in sites)
        span = _span([p for p, _ in sites])
        h = _handle(ref, th, sites, span)
        h.push_batch(packing.pack_reads(_tuples(reads), th["minMQ"]).as_capi())
        want = _want(reads, ref, sites, span, th)
        _check(h, sites, span, want)
        n_pairs += int((want.sum(axis=(1, 2)) > 0).sum())
        h.close()
    assert n_pairs > 0


@pytest.mark.parametrize("tname", ["strict", "loose", "zero"])
def test_every_batch_form(lib, tname):
    th = synth_small.THRESHOLDS[tname]
    ref, reads = synth_small.make_scenario(**dict(INDEL_DENSE, n_reads=900, ref_len=400))
    sites = _sites(reads, ref, th, max_depth=60)
    span = _span([p for p, _ in sites], 150)
    want = _want(reads, ref, sites, span, th, max_depth=60)
    assert want.sum() > 0
    for form, b in _forms(reads, th).items():
        for impl in (0, 1, 5):
            h = _handle(ref, th, sites, span)
            h.set_impl(impl)
            h.push_batch(b.as_capi())
            _check(h, sites, span, want)
            h.close()


def test_device_and_async_pushes(lib):
    import torch
    from test_gpu_consensus import _to_device
    from lvc_b200 import packing
    th = TH
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    sites = _sites(reads, ref, th)
    span = _span([p for p, _ in sites])
    batch = packing.pack_reads(_tuples(reads), th["minMQ"])
    want = _want(reads, ref, sites, span, th)
    db, keep = _to_device(batch)
    torch.cuda.synchronize()
    h = _handle(ref, th, sites, span)
    h.push_batch_device(db)
    _check(h, sites, span, want)
    h.push_batch_device_async(db)
    h.check_async()
    _check(h, sites, span, 2 * want)
    h.close()
    h = _handle(ref, th, sites, span)
    for grp in range(4):
        for q in set(int(x) for x in batch.qual[:batch.n_qual] if x >= th["minBQ"]):
            h.ensure_plane(grp << 8 | q)
    h.push_batch_device_async(db)
    _check(h, sites, span, want)                     # the copy runs after the enqueued kernels
    h.check_async()
    h.close()
    del keep


def test_several_batches_equal_one(lib):
    from lvc_b200 import packing
    th = TH
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    sites = _sites(reads, ref, th)
    span = _span([p for p, _ in sites])
    b = packing.pack_reads(_tuples(reads), th["minMQ"])
    one, many = _handle(ref, th, sites, span), _handle(ref, th, sites, span)
    one.push_batch(b.as_capi())
    cuts = [0, 97, 260, 261, b.n_reads]
    for a, z in zip(cuts, cuts[1:]):
        many.push_batch(b.slice(a, z).as_capi())
    want = _want(reads, ref, sites, span, th)
    _check(one, sites, span, want)
    _check(many, sites, span, want)
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
        if k % 2 == 0:
            s[30] = {"A": "C", "C": "G", "G": "T", "T": "A"}[s[30]]
        reads.append(po.Read(0, 100, 60, [(0, 100)], "".join(s), [30] * 100))
    sites = [(110, "A" if ref[110] != "A" else "C"), (130, {"A": "C", "C": "G", "G": "T", "T": "A"}[ref[130]])]
    h = _handle(ref, th, sites, 50)
    before = h.launch_count
    h.push_batch(packing.pack_reads(_tuples(reads), 0).as_capi())
    assert h.launch_count - before == 3              # deposit, linkage counts, replayed deposit
    assert any(int(k) >> 8 == 3 for k in h.plane_keys())
    want = _want(reads, ref, sites, 50, th)
    assert want.sum() == 40 and want[0, 2, 1] == 7 and want[0, 2, 0] == 7
    _check(h, sites, 50, want)
    h.close()


def _two_haplotypes(seed=5):
    """100 reads over four sites within 150 bp; read i carries haplotype A (every alt) iff i % 10 < 7, else B (none)"""
    ref = synth_small.make_scenario(**dict(INDEL_DENSE, seed=seed, n_reads=1))[0]
    rng = random.Random(seed)
    sites_pos = [300, 341, 390, 437]
    sites = [(p, {"A": "G", "C": "T", "G": "A", "T": "C"}[ref[p]]) for p in sites_pos]
    rows = []
    for i in range(100):
        pos = 280 + rng.randrange(0, 15)
        seq = list(ref[pos:pos + 170])
        if i % 10 < 7:
            for p, a in sites:
                seq[p - pos] = a
        rows.append((0, pos, 60, [(0, 170)], "".join(seq), [rng.choice((25, 37)) for _ in seq]))
    rows.sort(key=lambda r: r[1])
    return ref, sites, rows


def test_known_linkage(lib, tmp_path):
    from variant_caller.live_variant_caller import LiveVariantCaller
    from lvc_b200 import packing
    ref, sites, rows = _two_haplotypes()
    lvc = LiveVariantCaller(_fasta(tmp_path, "hap", ref), 13, 0, 3, 2, 0.05, 1, device=0)
    lvc.track_linkage(sites, maxSpan=150)
    lvc.process_batch(packing.pack_reads(rows, 0))
    got = lvc.linkage()
    assert [(d["pos_a"], d["alt_a"], d["pos_b"], d["alt_b"]) for d in got] == \
        [(sites[a][0], sites[a][1], sites[b][0], sites[b][1]) for a in range(4) for b in range(a + 1, 4)]
    for d in got:
        assert d["counts"] == [[30, 0, 0], [0, 70, 0], [0, 0, 0]] and d["n"] == 100 and d["r2"] == 1.0, d
    assert lvc.linkage(minReads=100) == got and lvc.linkage(minReads=101) == []
    # the sites are 41, 49 and 47 apart: a span of 48 keeps two pairs; setting the sites again starts the counts over
    lvc.track_linkage(sites, maxSpan=48)
    lvc.process_batch(packing.pack_reads(rows, 0))
    got = lvc.linkage()
    assert [(d["pos_a"], d["pos_b"]) for d in got] == [(300, 341), (390, 437)]
    assert all(d["counts"] == [[30, 0, 0], [0, 70, 0], [0, 0, 0]] for d in got)
    lvc.close()


def test_triple_substitution(lib, tmp_path):
    """GGG -> AAC (the B.1.1 N-gene triple at 28881-28883) on a crafted reference: three pairs, every read ALT/ALT or
    REF/REF"""
    from variant_caller.live_variant_caller import LiveVariantCaller
    from lvc_b200 import packing
    ref = synth_small.make_scenario(**dict(INDEL_DENSE, seed=9, n_reads=1))[0]
    ref = ref[:300] + "GGG" + ref[303:]
    rows = []
    for i in range(60):
        seq = ref[250:300] + ("AAC" if i % 3 else "GGG") + ref[303:350]
        rows.append((0, 250, 60, [(0, 100)], seq, [30] * 100))
    lvc = LiveVariantCaller(_fasta(tmp_path, "n", ref), 13, 0, 3, 2, 0.05, 1, device=0)
    lvc.track_linkage([(300, "A"), (301, "A"), (302, "C")])
    lvc.process_batch(packing.pack_reads(rows, 0))
    got = lvc.linkage()
    assert [(d["pos_a"], d["pos_b"]) for d in got] == [(300, 301), (300, 302), (301, 302)]
    for d in got:
        assert d["counts"] == [[20, 0, 0], [0, 40, 0], [0, 0, 0]] and d["r2"] == 1.0
    lvc.close()


def test_lifetime_and_refusals(lib, tmp_path):
    from lvc_b200 import capi, packing
    th = TH
    ref, reads = synth_small.make_scenario(**INDEL_DENSE)
    sites = _sites(reads, ref, th)
    span = _span([p for p, _ in sites])
    batch = packing.pack_reads(_tuples(reads), th["minMQ"])
    want = _want(reads, ref, sites, span, th)
    zero = np.zeros_like(want)
    h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    with pytest.raises(capi.LvcError) as ei:
        h.copy_linkage()                                                 # counting is off
    assert ei.value.code == -1
    with pytest.raises(capi.LvcError):
        h.get_timing(5)
    h.push_batch(batch.as_capi())                                        # sites may be set on tables that hold counts
    _set(h, sites, span)
    _check(h, sites, span, zero)
    h.set_timing(True)
    h.push_batch(batch.as_capi())
    ms, n = h.get_timing(5)
    assert n == 1 and ms > 0
    _check(h, sites, span, want)
    _set(h, sites, span)                                                 # setting sites clears the counts
    _check(h, sites, span, zero)
    h.push_batch(batch.as_capi())
    # imports and reductions do not touch the counts
    h.import_dels(h.copy_dels(), True)
    h.import_plane(int(h.plane_keys()[0]), h.copy_plane(int(h.plane_keys()[0])))
    _check(h, sites, span, want)
    h.reset()                                                            # clears the counts, keeps the sites
    _check(h, sites, span, zero)
    h.push_batch(batch.as_capi())
    _check(h, sites, span, want)
    # refusals: named numbers, and the previous sites and counts stay
    G = len(ref)
    ok = [p for p in range(G) if ref[p] in "ACGT"]
    alt_of = {"A": "C", "C": "G", "G": "T", "T": "A"}
    bad = [
        (np.zeros((1 << 20) + 1, np.int32), b"A" * ((1 << 20) + 1), 10, "1048577"),
        (ok[:65], "".join(alt_of[ref[p]] for p in ok[:65]), ok[64] - ok[0], "65 sites"),
        ([ok[3], ok[1]], alt_of[ref[ok[3]]] + alt_of[ref[ok[1]]], 10, "not strictly ascending"),
        ([ok[1], ok[1]], alt_of[ref[ok[1]]] * 2, 10, "not strictly ascending"),
        ([ok[1]], "N", 10, "alt"),
        ([ok[1]], "a", 10, "alt"),
        ([ok[1]], ref[ok[1]], 10, "equals the reference letter"),
        ([G], "A", 10, str(G)),
        ([-1], "A", 10, "-1"),
        ([ok[1]], alt_of[ref[ok[1]]], 0, "max_span 0"),
        ([ok[1]], alt_of[ref[ok[1]]], 65536, "max_span 65536"),
    ]
    for pos, alt, sp, msg in bad:
        with pytest.raises(capi.LvcError) as ei:
            h.set_linkage_sites(pos, alt, sp)
        assert ei.value.code == -1 and msg in str(ei.value), (msg, str(ei.value))
    _check(h, sites, span, want)
    # the 64-site limit itself is accepted
    h2 = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    h2.set_linkage_sites(ok[:64], "".join(alt_of[ref[p]] for p in ok[:64]), ok[63] - ok[0])
    assert len(h2.copy_linkage()) == 64 * 63 // 2
    h2.close()
    # n_sites = 0: off, timer 5 refused, no extra launch
    h.set_linkage_sites([], "", 0)
    with pytest.raises(capi.LvcError):
        h.copy_linkage()
    with pytest.raises(capi.LvcError):
        h.get_timing(5)
    n0 = h.launch_count
    h.push_batch(batch.as_capi())
    assert h.launch_count - n0 == 1
    h.close()
    # a reference letter that is not A/C/G/T
    nref = ref[:50] + "N" + ref[51:]
    h = capi.Handle(nref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    with pytest.raises(capi.LvcError) as ei:
        h.set_linkage_sites([50], "A", 10)
    assert ei.value.code == -1 and "reference letter 'N'" in str(ei.value)
    h.close()


def test_checkpoint_clears_the_counts(lib, tmp_path):
    from variant_caller.live_variant_caller import LiveVariantCaller
    from lvc_b200 import packing
    ref, sites, rows = _two_haplotypes()
    lvc = LiveVariantCaller(_fasta(tmp_path, "hap", ref), 13, 0, 3, 2, 0.05, 1, device=0)
    lvc.track_linkage(sites, maxSpan=150)
    lvc.process_batch(packing.pack_reads(rows, 0))
    ck = str(tmp_path / "ck.pkl")
    lvc.create_checkpoint(ck)
    assert all(d["n"] == 100 for d in lvc.linkage())
    lvc.load_checkpoint(ck)
    assert lvc.linkage() == [] and len(lvc.linkage(minReads=0)) == 6
    lvc.process_batch(packing.pack_reads(rows, 0))
    assert all(d["n"] == 100 and d["r2"] == 1.0 for d in lvc.linkage())
    lvc.track_linkage([])
    with pytest.raises(Exception):
        lvc.linkage()
    lvc.close()


def test_counting_changes_nothing_else(lib, golden_synth, tmp_path):
    """planes, deletions, coverage, first-seen ordinals, records, the consensus and the insertion counts are those of
    callers that do not count linkage; exactly one more launch per push"""
    from variant_caller.live_variant_caller import LiveVariantCaller
    from lvc_b200 import packing
    g = golden_synth["amplicon_like"]
    rows = g["reads"]
    fa = _fasta(tmp_path, "chrS", g["ref"])
    ref2, reads2 = synth_small.make_scenario(**INDEL_DENSE)
    for fasta, ref, reads, batches in (
            (fa, g["ref"], synth_small.rows_to_reads(rows),
             [packing.pack_reads(rows_to_tuples([rows[i] for i in range(k, len(rows), 3)]), 0) for k in range(3)]),
            (_fasta(tmp_path, "dense", ref2), ref2, reads2, [packing.pack_reads(_tuples(reads2), 0)])):
        sites = _sites(reads, ref, TH)
        span = _span([p for p, _ in sites])
        mk = lambda **kw: LiveVariantCaller(fasta, TH["minBQ"], TH["minMQ"], TH["minDP"], TH["minAD"], TH["ratio"], 1,
                                            device=0, **kw)
        off, ins, both = mk(), mk(countInsertions=True), mk(countInsertions=True)
        both.track_linkage(sites, span)
        for b in batches:
            n = [c._handle.launch_count for c in (off, ins, both)]
            for c in (off, ins, both):
                c.process_batch(b)
            d = [c._handle.launch_count - n0 for c, n0 in zip((off, ins, both), n)]
            assert d[2] == d[1] + 1 == d[0] + 2
            ho, hn = off._handle, both._handle
            assert sorted(ho.plane_keys().tolist()) == sorted(hn.plane_keys().tolist())
            for k in ho.plane_keys():
                assert np.array_equal(ho.copy_plane(int(k)), hn.copy_plane(int(k)))
            assert np.array_equal(ho.copy_dels(), hn.copy_dels()) and np.array_equal(ho.copy_covdiff(), hn.copy_covdiff())
            for grp in range(4):
                a, c = ho.copy_first(grp), hn.copy_first(grp)
                assert (a is None) == (c is None) and (a is None or np.array_equal(a, c))
            assert off.prepare_variants() == both.prepare_variants()
            assert off.memory == both.memory
            assert off.consensus(3, 0.5) == both.consensus(3, 0.5)
            assert np.array_equal(ins._handle.copy_insertions(), both._handle.copy_insertions())
        assert both.linkage(minReads=0)
        for c in (off, ins, both):
            c.close()

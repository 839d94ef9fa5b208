"""GPU parity at scale: the CUDA path against the C oracle (reference-order streaming products) on the
synthetic BASELINE workloads, plus size-independent properties (both kernels agree bit for bit;
re-depositing a batch doubles every count; sum of counts == bases that pass the filters)."""
import numpy as np
import pytest

from helpers import close_lik

pytestmark = pytest.mark.gpu

TH = dict(minBQ=30, minMQ=20, minDP=10, minAD=5, ratio=0.10)
GS_TO_NIB = [1, 2, 4, 8, 0, 3, 5, 6, 7, 9, 10, 11, 12, 13, 14, 15]


def device_tables(h):
    """(ad[G,16] by nibble code, qsum[G,16], first[G,16], dels[G], cov[G]) from the device planes."""
    G = h.G
    ad = np.zeros((G, 16), np.uint64)
    qsum = np.zeros((G, 16), np.uint64)
    first = np.full((G, 16), 0xFFFFFFFF, np.uint32)
    for key in h.plane_keys():
        g, q = int(key) >> 8, int(key) & 255
        pl = h.copy_plane(int(key)).astype(np.uint64)
        for s in range(4):
            nib = GS_TO_NIB[g * 4 + s]
            ad[:, nib] += pl[:, s]
            qsum[:, nib] += pl[:, s] * np.uint64(q)
    for g in range(4):
        f = h.copy_first(g)
        if f is not None:
            for s in range(4):
                first[:, GS_TO_NIB[g * 4 + s]] = f[:, s]
    return ad, qsum, first, h.copy_dels(), np.cumsum(h.copy_covdiff()[:-1])


def check_against_c_oracle(ref, batches, th, impl, max_depth=8000, geno_between=False):
    from lvc_b200 import capi, records
    from oracle.c_oracle import COracle
    e_lut, om_lut = records.phred_luts()
    h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    h.set_impl(impl)
    co = COracle(ref, th["minBQ"], th["minMQ"], max_depth)
    for b in batches:
        h.push_batch(b.as_capi())
        co.process(b)
        if geno_between:                       # live mode: a genotype pass after every batch (it also writes the first-seen hints)
            h.genotype(th["minDP"], th["minAD"], th["ratio"], e_lut, om_lut)
    ad, qsum, first, dels, cov = device_tables(h)
    assert np.array_equal(ad, co.ad.astype(np.uint64)), "allele depth tables differ"
    assert np.array_equal(qsum, co.qsum), "quality-sum checksum differs"
    assert np.array_equal(cov.astype(np.uint32), co.cov), "coverage (site set) differs"
    assert np.array_equal(ad.sum(axis=1) + dels, co.depth.astype(np.uint64)), "totalDepth differs"
    assert np.array_equal(first[ad > 0], co.first[co.ad > 0]), "first-seen ordinals differ"
    # likelihoods + emission
    L, S, emit, n_emit = co.genotype(th["minDP"], th["minAD"], th["ratio"])
    cands = h.genotype(th["minDP"], th["minAD"], th["ratio"], e_lut, om_lut)
    got = sorted((int(c["pos"]), int(c["code"])) for c in cands)
    want = sorted(zip(*[x.tolist() for x in np.nonzero(emit)]))
    assert got == want, "emitted (position, allele) set differs"
    for c in cands:
        p, code = int(c["pos"]), int(c["code"])
        assert close_lik(float(c["L"]), float(L[p, code]), int(co.depth[p]) + 4), (p, code, c["L"], L[p, code])
        assert close_lik(float(c["S"]), float(S[p]), int(co.depth[p]) + 4)
        assert int(c["dp"]) == int(co.depth[p]) and int(c["ad"]) == int(co.ad[p, code])
        assert abs(float(c["esum"]) - co.esum[p, code]) <= 1e-10 * co.esum[p, code]
    depth, dad, dlik = h.copy_dense()
    assert np.array_equal(depth, co.depth)
    for s, nib in enumerate((1, 2, 4, 8)):
        assert np.array_equal(dad[:, s], co.ad[:, nib])
        a, b = dlik[:, s], L[:, nib]
        bad = [p for p in np.nonzero(a != b)[0] if not close_lik(float(a[p]), float(b[p]), int(co.depth[p]) + 4)]
        assert not bad, (nib, bad[:5], a[bad[:5]], b[bad[:5]])
    h.close()
    return n_emit


@pytest.mark.parametrize("impl", [1, 2, 4, 5])
def test_amplicon_medium(lib, impl):
    from lvc_b200 import synth
    ref, b = synth.amplicon_sample(seed=7, n_pairs=120_000)
    n = check_against_c_oracle(ref, [b], TH, impl)
    assert n > 0


@pytest.mark.parametrize("th", [dict(minBQ=20, minMQ=0, minDP=5, minAD=2, ratio=0.02),
                                dict(minBQ=0, minMQ=0, minDP=1, minAD=1, ratio=0.0)])
def test_amplicon_multi_quality(lib, th):
    """several passing quality values: the non-primary ones take the tile kernel's per-base path"""
    from lvc_b200 import synth
    ref, b = synth.amplicon_sample(seed=8, n_pairs=30_000, min_mapq=th["minMQ"])
    check_against_c_oracle(ref, [b], th, 2)
    check_against_c_oracle(ref, [b], th, 4)


@pytest.mark.parametrize("impl", [1, 2, 4, 5])
def test_shotgun_small_genome(lib, impl):
    from lvc_b200 import synth
    ref, b = synth.shotgun_sample(seed=9, ref_len=200_000, depth=60.0)
    check_against_c_oracle(ref, [b], TH, impl)


def test_shotgun_low_max_depth(lib):
    """max_depth admission on shotgun data (drops are position dependent)"""
    from lvc_b200 import synth
    ref, b = synth.shotgun_sample(seed=10, ref_len=30_000, depth=400.0, max_depth=200)
    check_against_c_oracle(ref, [b], TH, 2, max_depth=200)
    check_against_c_oracle(ref, [b], TH, 4, max_depth=200)


def test_live_batches_ont(lib):
    from lvc_b200 import synth
    ref = synth.random_reference(6000, 3)
    batches = [synth.ont_batch(100 + k, ref, depth=40.0) for k in range(3)]
    th = dict(minBQ=13, minMQ=20, minDP=10, minAD=3, ratio=0.05)
    for impl in (0, 1, 2, 3, 4, 5, 6):          # 0 = auto: picks the warp-per-read kernel for these batches
        check_against_c_oracle(ref, batches, th, impl)


def test_config3_sized_ont_batches(lib):
    """SURVEY 8d config 3 at full batch size (74,758 reads, ~21 CIGAR ops each, qualities 2..90): two live batches
    through the automatic long-read deposit choice and the genotype pass over their wide quality alphabet, against the
    C oracle"""
    from lvc_b200 import synth
    ref = synth.random_reference(29903, 20260199)
    batches = [synth.ont_batch_fast(20260200 + k, ref) for k in range(2)]
    assert batches[0].n_reads == 74758 and batches[0].n_cigar == 21 * 74758
    check_against_c_oracle(ref, batches, dict(minBQ=30, minMQ=20, minDP=10, minAD=5, ratio=0.10), 0)
    check_against_c_oracle(ref, batches[:1], dict(minBQ=7, minMQ=20, minDP=10, minAD=5, ratio=0.02), 0)


def test_full_size_config2_properties(lib):
    """BASELINE configs[1] at full size: C-oracle parity + idempotence-style properties."""
    from lvc_b200 import synth, capi
    ref, b = synth.amplicon_sample()
    assert b.n_reads == 1_993_534 and abs(b.aligned_bases() - 2.99e8) < 1e6
    assert abs(b.algorithmic_bytes(len(ref)) - 0.498e9) < 2e6          # SURVEY 8d: 0.498 GB
    check_against_c_oracle(ref, [b], TH, 2)
    # both kernels agree bit for bit; depositing the batch twice doubles every count
    tabs = []
    for impl, times in ((1, 1), (4, 1), (2, 2), (5, 1)):
        h = capi.Handle(ref.encode("latin-1"), TH["minBQ"], TH["minMQ"], device=0)
        h.set_impl(impl)
        for _ in range(times):
            h.push_batch(b.as_capi())
        tabs.append(device_tables(h))
        h.close()
    for x, y in zip(tabs[0][:2] + tabs[0][3:], tabs[1][:2] + tabs[1][3:]):
        assert np.array_equal(x, y)
    assert np.array_equal(tabs[0][2], tabs[1][2])
    assert np.array_equal(tabs[2][0], 2 * tabs[1][0]) and np.array_equal(tabs[2][1], 2 * tabs[1][1])
    assert np.array_equal(tabs[2][2], tabs[1][2])                       # first-seen ranks do not move
    for x, y in zip(tabs[3], tabs[1]):                                  # generation-5 tiled kernel == generation 4
        assert np.array_equal(x, y)


def test_pinned_host_buffers_are_read_in_place(lib):
    """page-locked caller buffers: the kernels read the payload over PCIe in place (no payload H2D copy);
    results must equal the copy path and the oracle"""
    from lvc_b200 import synth, capi, packing
    from oracle.c_oracle import COracle
    ref, b = synth.amplicon_sample(seed=11, n_pairs=60_000)
    pinned = packing.pin_batch(b)
    tabs = []
    for batch in (b, pinned):
        h = capi.Handle(ref.encode("latin-1"), TH["minBQ"], TH["minMQ"], device=0)
        h.push_batch(batch.as_capi())
        h.push_batch(batch.as_capi())
        tabs.append(device_tables(h))
        h.close()
    for x, y in zip(tabs[0], tabs[1]):
        assert np.array_equal(x, y)
    co = COracle(ref, TH["minBQ"], TH["minMQ"])
    co.process(b)
    co.process(b)
    assert np.array_equal(tabs[1][0], co.ad.astype(np.uint64))
    assert np.array_equal(tabs[1][2][tabs[1][0] > 0], co.first[co.ad > 0])


def test_long_reads_with_many_cigar_ops(lib):
    """reads with 121 and 401 CIGAR ops (several groups of 32 ops in the warp-per-read kernel, ring flushes at every
    group boundary), two live batches, every kernel selection, low and high base-quality thresholds"""
    from lvc_b200 import synth
    ref = synth.random_reference(12000, 77)
    b1 = synth.ont_batch_fast(501, ref, depth=40.0, ref_span=2400, n_runs=60)
    b2 = synth.ont_batch_fast(502, ref, depth=25.0, ref_span=6000, n_runs=200)
    assert b1.n_cigar == 121 * b1.n_reads and b2.n_cigar == 401 * b2.n_reads
    for impl in (0, 3, 4, 5, 6):
        check_against_c_oracle(ref, [b1, b2], dict(minBQ=20, minMQ=20, minDP=5, minAD=2, ratio=0.05), impl)
    check_against_c_oracle(ref, [b2, b1], dict(minBQ=0, minMQ=0, minDP=1, minAD=1, ratio=0.0), 0)


def test_first_seen_hints_between_batches(lib):
    """Live mode: the genotype pass after batch k tells the long-read kernel which alleles already have a first-seen
    ordinal (TableView::seen), and the kernel then skips the first-seen test for them.  Shallow batches, so new
    (column, allele) pairs keep appearing in later batches; ordinals must equal the oracle's, with and without a
    genotype pass in between, and after a reset."""
    from lvc_b200 import capi, records, synth
    ref = synth.random_reference(5000, 11)
    batches = [synth.ont_batch_fast(700 + k, ref, depth=3.0) for k in range(6)]
    th = dict(minBQ=13, minMQ=20, minDP=2, minAD=1, ratio=0.0)
    for impl in (6, 0, 3):
        check_against_c_oracle(ref, batches, th, impl, geno_between=True)
        check_against_c_oracle(ref, batches, th, impl, geno_between=False)
    # reset clears the hints: the same handle, fed again, must give the first run's first-seen table
    e_lut, om_lut = records.phred_luts()
    h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    h.set_impl(6)
    runs = []
    for _ in range(2):
        for b in batches:
            h.push_batch(b.as_capi())
            h.genotype(th["minDP"], th["minAD"], th["ratio"], e_lut, om_lut)
        runs.append(h.copy_first(0).copy())
        h.reset()
    assert np.array_equal(runs[0], runs[1])
    h.close()


@pytest.mark.parametrize("impl", [1, 3, 4, 5, 6])
def test_read_leaving_the_reference_is_reported_and_not_deposited(lib, impl):
    """a read whose reference span ends past the contig: every kernel reports LVC_ERANGE (the reference would raise
    inside pysam) and deposits nothing of it; the other reads of the batch are deposited exactly"""
    from lvc_b200 import capi, packing, synth
    ref = synth.random_reference(600, 5)
    G = len(ref)
    q = [40] * 100

    def rd(pos, ops):
        lq = sum(l for o, l in ops if o in (0, 1, 4))
        return (0, pos, 60, ops, ref[pos:pos + lq] if pos + lq <= G else (ref[pos:] + "A" * lq)[:lq], [40] * lq)
    long_ops = [(4, 5), (0, 20), (1, 2), (0, 20), (2, 3), (0, 30), (4, 4)]        # S M I M D M S: 7 ops (long-read path)
    good = [rd(10, [(0, 100)]), rd(50, long_ops), rd(300, [(0, 60), (2, 2), (0, 40)])]
    bad = rd(G - 50, [(0, 100)])                                                  # 50 columns past the end
    bad_long = rd(G - 40, long_ops)                                               # 73 reference columns from G - 40
    th = dict(minBQ=20, minMQ=0)
    href = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
    href.set_impl(1)
    href.push_batch(packing.pack_reads(good, 0).as_capi())
    want = device_tables(href)
    href.close()
    for extra in (bad, bad_long):
        h = capi.Handle(ref.encode("latin-1"), th["minBQ"], th["minMQ"], device=0)
        h.set_impl(impl)
        with pytest.raises(capi.LvcError) as ei:
            h.push_batch(packing.pack_reads(good + [extra], 0).as_capi())
        assert ei.value.code == -5                                                # LVC_ERANGE
        got = device_tables(h)
        for a, b_, what in zip(got, want, ("ad", "qsum", "first", "dels", "cov")):
            assert np.array_equal(a, b_), (impl, what)
        h.close()

"""Strand counting (k_count_strands, lvc_enable_strand_counts) and the strand-bias query on the device.

    python tools/bench_strand.py [--steps 30]

One JSON line per workload on stdout:
  config2_amplicon   the config-2 amplicon sample as the packer hands it over: admitted reads only, 2-bit quality and base
                     codes, page-locked
  config5_1mb        shotgun 150 bp at 1,000x over a 1 Mb genome (bench.py's config-5 geometry on one GPU), byte qualities,
                     page-locked
  config3_ont        one config-3 ONT batch (~21 CIGAR ops per read, qualities 2..90), byte qualities, page-locked
  minBQ 30, minMQ 20 throughout.
  count_kernel_us          CUDA events around k_count_strands (lvc_get_timing slot 6), mean over --steps pushes
  deposit_kernel_us        the deposit kernel of the same pushes (slot 0 tiled, slot 1 ONT / warp / general)
  push_off_ms / push_on_ms host clock around lvc_push_batch (synchronous), median over --steps pushes of a handle without
                           and of a handle with strand counting, the two alternated push by push in the same run
  records                  the records of one push (genotype at minDP 10, minAD 5, ratio 0.10)
  query_us                 host clock around lvc_strand_counts for the REF and ALT of every record, median of 20
  stats_us                 host clock around DP4 / Fisher / FS / SOR of every record (records.strand_row), median of 5
  reverse_admitted_reads / reverse_entries  admitted reads with flag 0x10, and the entries counted after one push
The card's name, power limit and SM clocks are read in the same run.  LVC_LIB_PATH selects another build of the library.
"""
import argparse, json, os, subprocess, sys, time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "covid-spings-variant-caller_b200")):
    sys.path.insert(0, p)
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402

MIN_BQ, MIN_MQ = 30, 20


def card():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                  # the name from torch is still reported
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit_clocks": q}


def measure(name, what, ref, batch, steps, stream):
    from lvc_b200 import capi, packing, records
    pinned = packing.pin_batch(batch)
    cb = pinned.as_capi()
    off = capi.Handle(ref.encode("latin-1"), MIN_BQ, MIN_MQ, device=0, stream=stream.cuda_stream)
    on = capi.Handle(ref.encode("latin-1"), MIN_BQ, MIN_MQ, device=0, stream=stream.cuda_stream)
    on.enable_strand_counts()
    for h in (off, on):
        for _ in range(3):
            h.push_batch(cb)
    on.reset()
    on.push_batch(cb)
    G = len(ref)
    e, om = records.phred_luts()
    cands = on.genotype(10, 5, 0.10, e, om)
    pos = np.repeat(cands["pos"].astype(np.int32), 2)
    letters = "".join(chr(int(c["ref"])) + records.NIBBLE_CHARS[int(c["code"])] for c in cands)
    q_s = []
    for _ in range(20):
        t0 = time.perf_counter()
        fwd, rev = on.strand_counts(pos, letters)
        q_s.append(time.perf_counter() - t0)
    s_s = []
    for _ in range(5):
        t0 = time.perf_counter()
        rows = [records.strand_row({"start": int(p), "alleles": None}, (fwd[2 * k], rev[2 * k], fwd[2 * k + 1], rev[2 * k + 1]))
                for k, p in enumerate(pos[::2])]
        s_s.append(time.perf_counter() - t0)
    # every reverse entry of the push: the whole table through the query
    allpos = np.tile(np.arange(G, dtype=np.int32), 17)
    _, allrev = on.strand_counts(allpos, "".join(c * G for c in "ACTGNMRSVWYHKDB=-"))
    flag, keep = batch.flag, batch.keep
    n_rev = int((((flag & 0x10) != 0) & ((keep & 1) != 0)).sum())
    for h in (off, on):
        h.set_timing(True)
    t_off, t_on = [], []
    for _ in range(steps):
        for h, acc in ((off, t_off), (on, t_on)):
            h.sync()
            t0 = time.perf_counter()
            h.push_batch(cb)
            acc.append(time.perf_counter() - t0)
    count_ms, n_count = on.get_timing(6)
    dep = {}
    for label, h in (("off", off), ("on", on)):
        for slot in (0, 1):
            ms, n = h.get_timing(slot)
            if n:
                dep[label] = {"slot": slot, "kernel_us": ms * 1e3 / n, "launches": int(n)}
    for h in (off, on):
        h.set_timing(False)
    out = {"workload": name, "what": what, "reads": int(batch.n_reads), "cigar_ops": int(batch.n_cigar), "G": G,
           "reverse_admitted_reads": n_rev, "reverse_entries": int(allrev.sum(dtype=np.uint64)),
           "count_kernel_us": count_ms * 1e3 / n_count, "count_launches": int(n_count), "deposit_kernel_us": dep,
           "push_off_ms_median": float(np.median(t_off)) * 1e3, "push_on_ms_median": float(np.median(t_on)) * 1e3,
           "records": int(len(cands)), "query_us_median": float(np.median(q_s)) * 1e6,
           "stats_us_median": float(np.median(s_s)) * 1e6, "steps": steps, "library": os.path.basename(capi.LIB_PATH)}
    del rows
    off.close(); on.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    a = ap.parse_args()
    import torch
    from lvc_b200 import synth
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=0)
    info = card()
    ref, b = synth.amplicon_sample()
    b2 = b.admitted_only().with_quality_codes().with_base_codes(MIN_BQ)
    assert b2.qcode is not None and b2.scode is not None
    del b
    out = measure("config2_amplicon", "config-2 amplicon sample, admitted reads, 2-bit quality and base codes", ref, b2,
                  a.steps, stream)
    out.update(info)
    print(json.dumps(out), flush=True)
    del b2
    ref, b = synth.shotgun_sample(ref_len=1_000_000, n_snvs=100)[:2]
    out = measure("config5_1mb", "shotgun 150 bp, 1,000x, G = 1 Mb, byte qualities", ref, b, max(5, a.steps // 3), stream)
    out.update(info)
    print(json.dumps(out), flush=True)
    del b
    ref = synth.random_reference(29903, 20260199)
    ont = synth.ont_batch_fast(20260200, ref)
    out = measure("config3_ont", "one config-3 ONT batch, byte qualities", ref, ont, a.steps, stream)
    out.update(info)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()

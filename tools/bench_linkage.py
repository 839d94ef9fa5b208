"""Variant linkage counting (k_count_linkage, lvc_set_linkage_sites) and lvc_copy_linkage on the device.

    python tools/bench_linkage.py [--steps 30]

One JSON line per workload on stdout:
  config2_planted50       the config-2 amplicon sample as the packer hands it over: admitted reads only (800,098 of
                          1,993,534), 2-bit quality and base codes, page-locked; sites = its 50 planted SNVs, span 150
  config2_panel1000       the same batch; sites = a seeded panel of 1,000 positions (alt = the next base), span 300
  config3_ont             one config-3 ONT batch (74,758 reads, ~21 CIGAR ops each, qualities 2..90), page-locked, byte
                          qualities; sites = a seeded panel of 1,000 positions, span 1,000
  minBQ 30, minMQ 20 throughout.
  count_kernel_us         CUDA events around k_count_linkage (lvc_get_timing slot 5), mean over --steps pushes
  deposit_kernel_us       the deposit kernel of the same pushes (slot 0 tiled, slot 1 ONT / warp / general)
  push_off_ms / push_on_ms  host clock around lvc_push_batch (synchronous), median over --steps pushes of a handle without
                          and of a handle with linkage counting, the two alternated push by push in the same run
  copy_us                 host clock around lvc_copy_linkage into a preallocated buffer, median of 20
  pairs / window          pairs of the panel; most sites inside any window of span + 1 positions
  pair_reads              sum of all counts after one push (read-pair observations)
The card's name and power limit are read in the same run.  LVC_LIB_PATH selects another build of the library (kernel
variants), as everywhere.
"""
import argparse, ctypes, json, os, sys, time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "covid-spings-variant-caller_b200"), os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402

from bench_insertions import card  # noqa: E402

MIN_BQ, MIN_MQ = 30, 20
BASES = "ACGT"


def planted_snvs(ref, seed=20260101, n_snvs=50):
    """the planted SNVs of synth.amplicon_sample(seed): its first two draws"""
    from lvc_b200 import synth
    refc = synth._reference_codes(ref)
    rng = np.random.default_rng(seed)
    pos = np.sort(rng.choice(np.arange(50, len(ref) - 50), n_snvs, replace=False))
    alt = (refc[pos] + rng.integers(1, 4, n_snvs)) & 3
    return pos.astype(np.int32), "".join(BASES[int(a)] for a in alt)


def panel(ref, n, seed):
    rng = np.random.default_rng(seed)
    pos = np.sort(rng.choice(np.arange(len(ref)), n, replace=False)).astype(np.int32)
    return pos, "".join(BASES[(BASES.index(ref[p].upper()) + 1) & 3] for p in pos)


def window(pos, span):
    return int(max(np.searchsorted(pos, pos + span, "right") - np.arange(len(pos))))


def measure(name, what, ref, batch, steps, stream, pos, alt, span):
    from lvc_b200 import capi, packing
    pinned = packing.pin_batch(batch)
    cb = pinned.as_capi()
    off = capi.Handle(ref.encode("latin-1"), MIN_BQ, MIN_MQ, device=0, stream=stream.cuda_stream)
    on = capi.Handle(ref.encode("latin-1"), MIN_BQ, MIN_MQ, device=0, stream=stream.cuda_stream)
    on.set_linkage_sites(pos, alt, span)
    for h in (off, on):
        for _ in range(3):
            h.push_batch(cb)
    on.reset()
    on.push_batch(cb)
    pairs = on.copy_linkage()
    pair_reads = int(pairs["count"].sum(dtype=np.uint64))
    for h in (off, on):
        h.set_timing(True)
    t_off, t_on = [], []
    for _ in range(steps):
        for h, acc in ((off, t_off), (on, t_on)):
            h.sync()
            t0 = time.perf_counter()
            h.push_batch(cb)
            acc.append(time.perf_counter() - t0)
    count_ms, n_count = on.get_timing(5)
    dep = {}
    for label, h in (("off", off), ("on", on)):
        for slot in (0, 1):
            ms, n = h.get_timing(slot)
            if n:
                dep[label] = {"slot": slot, "kernel_us": ms * 1e3 / n, "launches": int(n)}
    for h in (off, on):
        h.set_timing(False)
    buf = np.zeros(len(pairs), dtype=capi.LINKAGE_DTYPE)
    n_out = ctypes.c_uint32(0)
    copy_s = []
    for _ in range(20):
        t0 = time.perf_counter()
        rc = on.lib.lvc_copy_linkage(on.h, buf.ctypes.data, len(buf), ctypes.byref(n_out))
        copy_s.append(time.perf_counter() - t0)
        assert rc == 0 and n_out.value == len(buf)
    out = {"workload": name, "what": what, "reads": int(batch.n_reads), "cigar_ops": int(batch.n_cigar),
           "sites": int(len(pos)), "span": span, "window": window(pos, span), "pairs": int(len(pairs)),
           "pair_reads": pair_reads, "count_kernel_us": count_ms * 1e3 / n_count, "count_launches": int(n_count),
           "deposit_kernel_us": dep, "push_off_ms_median": float(np.median(t_off)) * 1e3,
           "push_on_ms_median": float(np.median(t_on)) * 1e3, "copy_us_median": float(np.median(copy_s)) * 1e6,
           "steps": steps, "library": os.path.basename(capi.LIB_PATH)}
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
    what = "config-2 amplicon sample, admitted reads, 2-bit quality and base codes"
    pos, alt = planted_snvs(ref)
    for name, (p, al), span in (("config2_planted50", (pos, alt), 150), ("config2_panel1000", panel(ref, 1000, 7), 300)):
        out = measure(name, what, ref, b2, a.steps, stream, p, al, span)
        out.update(info)
        print(json.dumps(out), flush=True)
    del b2
    ref = synth.random_reference(29903, 20260199)
    ont = synth.ont_batch_fast(20260200, ref)
    p, al = panel(ref, 1000, 8)
    out = measure("config3_ont", "one config-3 ONT batch, byte qualities", ref, ont, a.steps, stream, p, al, 1000)
    out.update(info)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()

"""Consensus + coverage statistics on the device (lvc_consensus) against the host route a user has without it.

    python tools/bench_consensus.py [--calls 200] [--host-calls 3]

One JSON line per workload on stdout:
  sars2_config2   SARS-CoV-2 after the config-2 amplicon deposit (1,993,534 reads, minBQ 30: 1 plane)
  ont_config3     config-3 ONT tables (74,758 reads, qualities 2..90, minBQ 30: 61 planes)
  synth_5mb_1p    5 Mb x 1 plane, imported from a seeded generator (lvc_import_plane / lvc_import_dels)
  synth_5mb_4p    5 Mb x 4 planes (three of A/C/G/T, one of the other codes)
Every timed call is preceded by a read of a 256 MB buffer on the same stream, so the tables are read from HBM, not
from the 126 MB L2 (5 Mb x 1 plane is ~110 MB and would fit): all figures are cold-L2.  A read leaves no dirty lines
behind, whose write-back would otherwise be charged to the kernel.
  kernel_us     CUDA events around the kernel (lvc_get_timing slot 3), mean over --calls calls after warm-up
  call_us       host clock around lvc_consensus (synchronous: kernel + copy of the letters and counters back)
  bytes         (p1 - p0) * (16 * planes + 4 + 1 + 1): plane rows, deletion counts, reference, letter
  roofline_frac bytes / kernel time over 6543.7 GB/s, the measured copy bandwidth of DESIGN section 3
  host_route_ms genotype pass + lvc_copy_dense + lvc_copy_dels + the rule in NumPy (oracle/consensus_oracle.py), and
                whether its letters equal the device's
The card's name and power limit are read in the same run.
"""
import argparse, json, os, subprocess, sys, time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "covid-spings-variant-caller_b200")):
    sys.path.insert(0, p)
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402

PEAK_GBS = 6543.7
MIN_DEPTH, THRESHOLD, DEPTHS = 10, 0.75, (1, 10, 20, 100)


def card():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                  # the name from torch is still reported
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": q}


def synthetic_tables(h, G, n_planes, seed):
    """seeded counts: a majority base per position with ~40 reads, a few reads of the others, some deletions"""
    rng = np.random.default_rng(seed)
    major = rng.integers(0, 4, G)
    keys = [30, 20, 10][:max(n_planes - 1, 1)] + ([1 << 8 | 30] if n_planes > 1 else [])
    for k, key in enumerate(keys):
        arr = rng.integers(0, 3, (G, 4), dtype=np.uint32)
        if key >> 8 == 0:
            arr[np.arange(G), major] += np.uint32(40 if k == 0 else 10)
        h.import_plane(key, arr)
    h.import_dels(rng.integers(0, 4, G, dtype=np.uint32))


def host_route(h, ref, e_lut, om_lut):
    from oracle import consensus_oracle as co
    h.genotype_device(0, 0, 0.0, e_lut, om_lut)
    depth, ad, _ = h.copy_dense()
    dels = h.copy_dels()
    other = depth.astype(np.int64) - ad.sum(axis=1, dtype=np.int64) - dels
    planes = {0: ad, 1 << 8: np.column_stack([other, np.zeros((len(other), 3), np.int64)])}
    return co.consensus_from_tables(planes, dels, ref, MIN_DEPTH, THRESHOLD, DEPTHS)[0]


def measure(name, what, h, ref, flush, calls, host_calls, e_lut, om_lut):
    import torch
    G = h.G
    planes = len(h.plane_keys())
    for _ in range(20):
        h.consensus(MIN_DEPTH, THRESHOLD, DEPTHS)
    h.set_timing(True)
    h.get_timing(3)
    call_s = []
    for _ in range(calls):
        flush.sum()                                          # 256 MB read on the handle's stream: cold, clean L2
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        seq, st = h.consensus(MIN_DEPTH, THRESHOLD, DEPTHS)
        call_s.append(time.perf_counter() - t0)
    ms, n = h.get_timing(3)
    h.set_timing(False)
    kernel_s = ms * 1e-3 / n
    host_s, host_seq = [], None
    for _ in range(host_calls):
        t0 = time.perf_counter()
        host_seq = host_route(h, ref, e_lut, om_lut)
        host_s.append(time.perf_counter() - t0)
    byts = G * (16 * planes + 4 + 1 + 1)
    return {"workload": name, "what": what, "positions": G, "planes": planes, "calls": int(n),
            "kernel_us": kernel_s * 1e6, "call_us_median": float(np.median(call_s)) * 1e6,
            "bytes": byts, "achieved_GBps": byts / kernel_s / 1e9, "roofline_frac": byts / kernel_s / 1e9 / PEAK_GBS,
            "host_route_ms_median": float(np.median(host_s)) * 1e3, "host_route_same_letters": host_seq == seq.decode(),
            "n_N": st["n_N"], "n_ambiguous": st["n_ambiguous"], "cold_l2": True,
            "rule": {"min_depth": MIN_DEPTH, "threshold": THRESHOLD, "depths": list(DEPTHS)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--host-calls", type=int, default=3)
    a = ap.parse_args()
    import torch
    from lvc_b200 import capi, records, synth
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream(device=0)
    torch.cuda.set_stream(stream)
    flush = torch.empty(64 << 20, dtype=torch.int32, device="cuda:0")
    e_lut, om_lut = records.phred_luts()
    info = card()

    def run(name, what, ref, fill):
        h = capi.Handle(ref.encode("latin-1"), 30, 20, device=0, stream=stream.cuda_stream)
        fill(h)
        out = measure(name, what, h, ref, flush, a.calls, a.host_calls, e_lut, om_lut)
        h.close()
        out.update(info)
        print(json.dumps(out), flush=True)

    ref, b = synth.amplicon_sample()
    run("sars2_config2", "SARS-CoV-2 after the config-2 amplicon deposit", ref, lambda h: h.push_batch(b.as_capi()))
    del b
    ref = synth.random_reference(29903, 20260199)
    ont = synth.ont_batch_fast(20260200, ref)
    run("ont_config3", "config-3 ONT tables, minBQ 30", ref, lambda h: h.push_batch(ont.as_capi()))
    del ont
    ref = synth.random_reference(5_000_000, 20261020)
    run("synth_5mb_1p", "5 Mb x 1 plane, seeded import", ref, lambda h: synthetic_tables(h, len(ref), 1, 7))
    run("synth_5mb_4p", "5 Mb x 4 planes, seeded import", ref, lambda h: synthetic_tables(h, len(ref), 4, 8))


if __name__ == "__main__":
    main()

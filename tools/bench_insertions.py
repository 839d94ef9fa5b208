"""Insertion counting (k_count_insertions, lvc_enable_insertions) and insertion calls on the device.

    python tools/bench_insertions.py [--steps 30]

One JSON line per workload on stdout:
  config2_admitted_codes  the config-2 amplicon sample as the packer hands it over: admitted reads only (800,098 of
                          1,993,534), 2-bit quality and base codes, page-locked; minBQ 30, minMQ 20
  config3_ont             one config-3 ONT batch (74,758 reads, ~21 CIGAR ops each, qualities 2..90), page-locked, byte
                          qualities; minBQ 30, minMQ 20
  count_kernel_us         CUDA events around k_count_insertions (lvc_get_timing slot 4), mean over --steps pushes
  deposit_kernel_us       the deposit kernel of the same pushes (slot 0 tiled, slot 1 ONT / warp / general)
  push_off_ms / push_on_ms  host clock around lvc_push_batch (synchronous), median over --steps pushes of a handle without
                          and of a handle with insertion counting, the two alternated push by push in the same run
  calls_us                host clock around lvc_insertion_calls(min_depth 10, threshold 0.5) over the whole contig
                          (three passes over the table, the call pass, the copy back), median
  keys / calls            distinct insertion keys counted per push, insertions called
The card's name and power limit are read in the same run.
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
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                  # the name from torch is still reported
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": q}


def measure(name, what, ref, batch, steps, stream):
    from lvc_b200 import capi, packing
    pinned = packing.pin_batch(batch)
    cb = pinned.as_capi()
    off = capi.Handle(ref.encode("latin-1"), MIN_BQ, MIN_MQ, device=0, stream=stream.cuda_stream)
    on = capi.Handle(ref.encode("latin-1"), MIN_BQ, MIN_MQ, device=0, stream=stream.cuda_stream)
    on.enable_insertions(1 << 20)
    for h in (off, on):
        for _ in range(3):
            h.push_batch(cb)
    on.reset()
    on.push_batch(cb)
    keys = len(on.copy_insertions())
    for h in (off, on):
        h.set_timing(True)
    t_off, t_on = [], []
    for _ in range(steps):
        for h, acc in ((off, t_off), (on, t_on)):
            h.sync()
            t0 = time.perf_counter()
            h.push_batch(cb)
            acc.append(time.perf_counter() - t0)
    count_ms, n_count = on.get_timing(4)
    dep = {}
    for label, h in (("off", off), ("on", on)):
        for slot in (0, 1):
            ms, n = h.get_timing(slot)
            if n:
                dep[label] = {"slot": slot, "kernel_us": ms * 1e3 / n, "launches": int(n)}
    for h in (off, on):
        h.set_timing(False)
    calls_s = []
    calls = on.insertion_calls(10, 0.5)
    for _ in range(20):
        t0 = time.perf_counter()
        calls = on.insertion_calls(10, 0.5)
        calls_s.append(time.perf_counter() - t0)
    out = {"workload": name, "what": what, "reads": int(batch.n_reads), "cigar_ops": int(batch.n_cigar),
           "count_kernel_us": count_ms * 1e3 / n_count, "count_launches": int(n_count),
           "deposit_kernel_us": dep, "push_off_ms_median": float(np.median(t_off)) * 1e3,
           "push_on_ms_median": float(np.median(t_on)) * 1e3, "calls_us_median": float(np.median(calls_s)) * 1e6,
           "keys": keys, "calls": int(len(calls)), "steps": steps}
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
    out = measure("config2_admitted_codes", "config-2 amplicon sample, admitted reads, 2-bit quality and base codes", ref, b2,
                  a.steps, stream)
    out.update(info)
    print(json.dumps(out), flush=True)
    del b, b2
    ref = synth.random_reference(29903, 20260199)
    ont = synth.ont_batch_fast(20260200, ref)
    out = measure("config3_ont", "one config-3 ONT batch, byte qualities", ref, ont, a.steps, stream)
    out.update(info)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()

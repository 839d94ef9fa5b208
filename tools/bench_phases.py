"""Where a CTA of the tiled deposit kernel (generation 5) spends its cycles, phase by phase, on the device.

Builds the library with -DLVC5_PHASE_CLOCKS into a build directory of its own (the in-tree library is not touched),
runs the config-2 step and the config-5 step the way bench.py does, and reads back the clock64() stamps that thread 0
of every CTA of the last launch took at the phase boundaries:

  headers     kernel entry -> both read-level exits passed (header loads, edge-mask table)
  extents     -> byte extent of the chunk's tileable reads known (one barrier)
  classify    -> barrier A (payload prefetch, classification, per-warp run counts)
  run_table   -> barrier B (coverage / deletion updates, run table)
  stage_slabs -> barrier C (task table of the first column window, keys staged)
  tasks       -> every warp left the task loop (pass loop, reduce, flush)
  tail        -> exit of thread 0 (reads handed to the one-warp-per-read path)

Per phase it prints the median and p90 cycles over the CTAs that passed both boundaries, the CTA-cycles summed over
the grid and their share of all CTA-cycles (entry to exit), and that share of the SM-cycles the grid occupied (per SM,
first entry to last exit; the resident CTAs of an SM share its cycles).  In the same call it times the step with the
default build (the in-tree library unless --default-lib says otherwise), so the probe's own cost is visible.

  python tools/bench_phases.py [--configs 2,5] [--steps 20] [--reps 5] [--src TREE | --phase-lib SO] [--json OUT]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAMPS = ["entry", "headers", "extents", "barrier_a", "barrier_b", "barrier_c", "tasks_end", "exit"]
PHASES = ["headers", "extents", "classify", "run_table", "stage_slabs", "tasks", "tail"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")


def build(src: str, out_dir: str) -> str:
    sys.path.insert(0, ROOT)
    from __graft_entry__ import NVCC_FLAGS
    lib = os.path.join(out_dir, "liblvc_b200_phases.so")
    cu = os.path.join(src, "covid-spings-variant-caller_b200", "csrc", "lvc_api.cu")
    subprocess.run([NVCC] + NVCC_FLAGS + ["-DLVC5_PHASE_CLOCKS", "-o", lib, cu, "-lz"], check=True, cwd=out_dir)
    return lib


def phase_stats(rec: np.ndarray) -> dict:
    """rec: [n_cta, 1 + len(STAMPS)] uint64 (SM id, stamps; 0 = boundary not reached)"""
    sm, st = rec[:, 0], rec[:, 1:].astype(np.int64)
    live = (st[:, 0] != 0) & (st[:, -1] != 0)
    sm, st = sm[live], st[live]
    total = float((st[:, -1] - st[:, 0]).sum())
    # SM-cycles the grid occupied: per SM, first entry to last exit
    sm_span = 0.0
    for s in np.unique(sm):
        m = sm == s
        sm_span += float(st[m, -1].max() - st[m, 0].min())
    out = {"ctas": int(live.sum()), "cta_cycles": total, "sm_cycles": sm_span,
           "early_exit_ctas": int(((st[:, 1] == 0)).sum()), "phases": {}}
    # phase k runs from stamp k to stamp k+1; a CTA that skipped stamp k+1 (early exit, no runs) charges the
    # interval to the next stamp it reached, so every CTA-cycle is counted once
    for k, name in enumerate(PHASES):
        a = st[:, k]
        nxt = np.zeros_like(a)
        for j in range(len(STAMPS) - 1, k, -1):
            nxt = np.where(st[:, j] != 0, st[:, j], nxt)
        ok = (a != 0) & (nxt != 0) & (st[:, k + 1] != 0)
        d = (st[ok, k + 1] - a[ok]).astype(np.float64)
        charged = float(np.where((a != 0) & (nxt != 0), nxt - a, 0).sum())
        out["phases"][name] = {
            "ctas": int(ok.sum()),
            "median": float(np.median(d)) if d.size else None,
            "p90": float(np.percentile(d, 90)) if d.size else None,
            "cta_cycles": charged,
            "share": charged / total if total else None,
            "sm_cycles": sm_span * charged / total if total else None,
        }
    return out


def worker(args) -> None:
    """one library, one process: the step time of each config, and with a phase-clock library the phase table"""
    os.environ["LVC_LIB_PATH"] = args.lib
    sys.path.insert(0, ROOT)
    import bench                                     # workloads, batch form and device upload exactly as bench.py
    import torch
    from lvc_b200 import capi, records
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    e_lut, om_lut = records.phred_luts()
    T = bench.THRESH
    res = {"lib": args.lib, "phase_clocks": bool(args.phases), "configs": {}}
    for cfg in args.configs.split(","):
        if cfg == "2":
            ref, batch = bench.make_workload(20260101, bench.N_PAIRS)
            batch = bench.in_form(batch.admitted_only())
        elif cfg == "5":
            ref, batch = bench.config5_workload()
            batch = bench.in_form(batch)
        else:
            raise SystemExit(f"unknown config {cfg}")
        db, keep = bench.to_device(torch, capi, batch, dev)
        h = capi.Handle(ref.encode("latin-1"), T["minBQ"], T["minMQ"], device=0, stream=stream.cuda_stream)

        def step():
            h.push_batch_device_async(db)
            h.genotype_device_async(T["minDP"], T["minAD"], T["ratio"], e_lut, om_lut)
        h.push_batch_device(db)
        h.genotype_device(T["minDP"], T["minAD"], T["ratio"], e_lut, om_lut)
        for _ in range(5):
            step()
        h.check_async()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            step()
        e1.record(stream)
        torch.cuda.synchronize()
        h.check_async()
        r = {"n_reads": int(batch.n_reads), "ms_per_step": e0.elapsed_time(e1) / args.steps}
        if args.phases:
            lib = capi.load_library()
            lib.lvc_phase_clocks.restype = ctypes.c_int
            lib.lvc_phase_clocks.argtypes = [ctypes.c_void_p, ctypes.c_uint32]
            n_cta = (int(batch.n_reads) + 191) // 192
            recs = []
            for _ in range(args.reps):
                step()
                torch.cuda.synchronize()
                buf = np.zeros((n_cta, 1 + len(STAMPS)), np.uint64)
                cap = lib.lvc_phase_clocks(buf.ctypes.data, n_cta)
                if cap < 0:
                    raise SystemExit("lvc_phase_clocks failed")
                if n_cta > cap:
                    raise SystemExit(f"{n_cta} CTAs, the phase-clock build records {cap}")
                recs.append(buf)
            h.check_async()
            r["phases"] = phase_stats(np.concatenate(recs))
            r["reps"] = args.reps
        h.close()
        del keep
        res["configs"][cfg] = r
    print("RESULT " + json.dumps(res), flush=True)


def run_worker(lib: str, phases: bool, args) -> dict:
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--lib", lib, "--configs", args.configs,
           "--steps", str(args.steps), "--reps", str(args.reps)] + (["--phases"] if phases else [])
    p = subprocess.run(cmd, check=True, stdout=subprocess.PIPE, text=True)
    for line in p.stdout.splitlines():
        if line.startswith("RESULT "):
            return json.loads(line[7:])
    raise SystemExit("worker printed no result")


def print_table(cfg: str, ms_default: float, r: dict) -> None:
    ph = r["phases"]
    print(f"\nconfig {cfg}: {r['n_reads']} reads, {ph['ctas']} CTAs x {r['reps']} launches "
          f"({ph['early_exit_ctas']} left before the headers stamp); step {ms_default * 1e3:.1f} us default build, "
          f"{r['ms_per_step'] * 1e3:.1f} us phase-clock build")
    print(f"{'phase':<12} {'median':>8} {'p90':>8} {'CTA-cycles':>14} {'share':>7} {'SM-cycles':>12}")
    for name in PHASES:
        p = ph["phases"][name]
        med = f"{p['median']:.0f}" if p["median"] is not None else "-"
        p90 = f"{p['p90']:.0f}" if p["p90"] is not None else "-"
        print(f"{name:<12} {med:>8} {p90:>8} {p['cta_cycles']:>14.4g} {100 * p['share']:>6.1f}% {p['sm_cycles']:>12.4g}")
    print(f"{'total':<12} {'':>8} {'':>8} {ph['cta_cycles']:>14.4g} {'':>7} {ph['sm_cycles']:>12.4g}")


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--configs", default="2,5", help="comma list of 2 (bench.py's headline) and 5 (--legs config5)")
    ap.add_argument("--steps", type=int, default=20, help="timed steps per config")
    ap.add_argument("--reps", type=int, default=5, help="launches whose clocks are pooled")
    ap.add_argument("--src", default=ROOT, help="source tree to instrument (default: this repository)")
    ap.add_argument("--build-dir", default=None, help="where the phase-clock library goes (default: a temporary directory)")
    ap.add_argument("--phase-lib", default=None, help="a phase-clock library built before (skips the build)")
    ap.add_argument("--default-lib", default=None, help="library timed beside it (default: the in-tree build)")
    ap.add_argument("--json", default=None, help="also write the results here")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--lib", help=argparse.SUPPRESS)
    ap.add_argument("--phases", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    default_lib = args.default_lib or os.path.join(ROOT, "covid-spings-variant-caller_b200", "lvc_b200", "liblvc_b200.so")
    if not os.path.exists(default_lib):
        raise SystemExit(f"{default_lib} not found: run `python __graft_entry__.py` first")
    with tempfile.TemporaryDirectory(prefix="lvc_phases_") as tmp:
        out_dir = args.build_dir or tmp
        os.makedirs(out_dir, exist_ok=True)
        lib = args.phase_lib or build(os.path.abspath(args.src), out_dir)
        base = run_worker(default_lib, False, args)
        ph = run_worker(lib, True, args)
    for cfg in args.configs.split(","):
        print_table(cfg, base["configs"][cfg]["ms_per_step"], ph["configs"][cfg])
    if args.json:
        with open(args.json, "w") as fh:
            json.dump({"default": base, "phase_clocks": ph}, fh, indent=1)


if __name__ == "__main__":
    main()

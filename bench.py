#!/usr/bin/env python
"""bench.py -- pileup + genotype-likelihood throughput (aligned bases / s) on N B200s.

    python bench.py --gpus 1 --steps 50 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 5 --warmup 1      # the CPU arm (oracle port, host cores)

One "step" = one pass of the hot path over one batch: deposit every read of the batch into the
persistent device tables + the genotype pass over all G positions + candidate compaction.
Headline workload at N = 1: BASELINE.json configs[1] (SURVEY 8d config 2): synthetic SARS-CoV-2 Illumina 2x150
amplicon reads at 10,000x, 1,993,534 reads, 2.99e8 aligned bases, 0.498 GB algorithmic bytes.  At N > 1 every rank
processes its own sample of the same geometry (independent samples, no communication) -> weak scaling.

The same JSON line (rank 0, stdout) carries a `configs` block with the other SURVEY 8d workloads:
  config3  ONT-like live batches on one GPU (N = 1)
  config5  shotgun 150 bp at 1,000x over a 1 Mb genome: one GPU (N = 1) or read-chunk sharded over the N ranks with
           the NCCL exchange of the count tables (deposit / exchange / genotype-slice split, three exchange modes)
  config4  the 96-sample plate at 5,000x, samples round-robin over the N ranks, no communication (strong scaling)
and `e2e_api`: LiveVariantCaller.process_bam(BAM on disk) + prepare_variants() (N = 1).
`--legs main` runs the headline workload only (kernel experiments).
`--dump-outputs DIR` writes what the last timed step computed as .npy files, so that two builds can be compared output
for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "covid-spings-variant-caller_b200")
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from (which may be read-only)
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "pileup+GL aligned bases/sec"
UNIT = "aligned bases/s"
THRESH = dict(minBQ=30, minMQ=20, minDP=10, minAD=5, ratio=0.10)      # config_util/vc.config defaults
WORKLOAD = "config2: synthetic SARS-CoV-2 Illumina 2x150 amplicon, 10,000x, 1,993,534 reads (seed 20260101)"
N_PAIRS = 996_767
BATCH_FIELDS = ("pos", "flag", "mapq", "keep", "cigar_off", "cigar", "seq_off", "seq4", "qual")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------ workloads
def _cached(name: str, make):
    """(ref, ReadBatch) cached in the temporary directory so the arms of one machine do not regenerate it."""
    from lvc_b200 import packing
    cache = os.path.join(tempfile.gettempdir(), name)
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            return str(z["ref"]), packing.ReadBatch(*[z[k] for k in BATCH_FIELDS])
        except Exception as e:
            log("[bench] cache unreadable, regenerating:", e)
    t = time.time()
    ref, b = make()
    log(f"[bench] generated {os.path.basename(cache)}: {b.n_reads} reads in {time.time() - t:.1f}s")
    try:
        tmp = cache + f".{os.getpid()}.tmp.npz"
        np.savez(tmp, ref=np.array(ref), **{k: getattr(b, k) for k in BATCH_FIELDS})
        os.replace(tmp, cache)
    except Exception as e:  # cache is best effort
        log("[bench] cache write failed:", e)
    return ref, b


def make_workload(seed: int, n_pairs: int):
    from lvc_b200 import synth
    return _cached(f"lvc_bench_cfg2_{seed}_{n_pairs}.npz", lambda: synth.amplicon_sample(seed=seed, n_pairs=n_pairs))


def live_bytes(batch) -> int:
    """SURVEY 8d bytes of the reads the deposit kernel actually has to read: 20 + 4 n_cigar + ceil(l/2) + l of every
    read that passes the host admission (keep bit 0) and the read-level filter (flag, mapq, orphan)."""
    from lvc_b200 import packing
    n = batch.n_reads
    f = batch.flag[:n].astype(np.uint32)
    live = ((batch.keep[:n] & 1) != 0) & ((f & 0x704) == 0) & (batch.mapq[:n] >= THRESH["minMQ"]) & \
        ~(((f & 1) != 0) & ((f & 2) == 0))
    lq = packing.query_lengths(batch.cigar_off, batch.cigar)[:n]
    nc = np.diff(batch.cigar_off[:n + 1].astype(np.int64))
    return int((20 + 4 * nc[live] + (lq[live] + 1) // 2 + lq[live]).sum()), int(live.sum())


QUALITY_FORM = "codes"      # --quality-form: what the short-read legs ship (codes = lvc_batch.qual_bits 2 where a batch qualifies)


def in_form(batch):
    """the batch in the quality form the run was asked for (2-bit codes only where the batch qualifies)"""
    return batch.with_quality_codes() if QUALITY_FORM == "codes" else batch.without_quality_codes()


def form_of(batch) -> str:
    if batch.qcode is not None and getattr(batch, "scode", None) is not None:
        return "2-bit quality codes + 2-bit base codes (lvc_batch.qual_bits = 2, seq_form = 2), 0.5 B per base"
    return "2-bit quality codes (lvc_batch.qual_bits = 2), 0.75 B per base" if batch.qcode is not None else \
        "phred bytes, 1.5 B per base"


def to_device(torch, capi, batch, dev):
    keep = {name: torch.from_numpy(getattr(batch, name).view(np.uint8).reshape(-1)).to(dev) for name in BATCH_FIELDS
            if not (name == "qual" and batch.qcode is not None)}
    if batch.qcode is not None:
        keep["qual"] = torch.from_numpy(batch.qcode.view(np.uint8).reshape(-1)).to(dev)
    db = capi.Handle.make_batch(batch.n_reads, batch.n_cigar, batch.n_qual, *[keep[k].data_ptr() for k in BATCH_FIELDS],
                                qual_dict=batch.qdict if batch.qcode is not None else None)
    return db, keep


# ------------------------------------------------------------------------------------------------ clocks / NUMA
class ClockSampler(threading.Thread):
    """NVML polling of SM clock + throttle reasons during the timed region (in-process: the region can be
    shorter than nvidia-smi's sampling period)."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reason_bits, self.stop_flag, self.ok = index, [], 0, False, False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:
            log("[bench] NVML unavailable:", e)

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.dev, self.nv.NVML_CLOCK_SM))
                self.reason_bits |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.dev)) \
                    if hasattr(self.nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.dev))
            except Exception:
                pass
            time.sleep(0.002)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        reasons = [n for bit, n in self.REASONS.items() if self.reason_bits & bit and n != "gpu_idle"]
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.samples)}


def bind_numa(index: int) -> dict:
    """Run this process on the CPUs of the GPU's NUMA node and prefer that node's memory: the end-to-end path reads
    page-locked host buffers in place over PCIe, and 8 ranks pulling from one socket's memory saturate the
    inter-socket link (round 1: e2e efficiency 0.46 at 8 GPUs).  Best effort; says what it did."""
    info = {"gpu_numa_node": None, "cpus_bound": 0, "mempolicy": None}
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dom, rest = bus.lower().split(":", 1)
        path = f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/numa_node"
        node = int(open(path).read().strip())
        info["gpu_numa_node"] = node
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        target = cpus & os.sched_getaffinity(0)
        if target:
            os.sched_setaffinity(0, target)
            info["cpus_bound"] = len(target)
        # set_mempolicy(MPOL_PREFERRED, {node}): later allocations (cudaHostAlloc pages included) come from that node
        mask = (ctypes.c_ulong * 16)()
        mask[node // 64] = 1 << (node % 64)
        libc = ctypes.CDLL(None, use_errno=True)
        rc = libc.syscall(238, 1, ctypes.byref(mask), 16 * 64 + 1)
        info["mempolicy"] = "preferred" if rc == 0 else f"failed errno {ctypes.get_errno()}"
    except Exception as e:
        info["error"] = f"{type(e).__name__}: {e}"
    return info


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram bytes per launch of the tiled deposit kernel from the committed ncu capture (NOT measured by this run)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return d.get("dram_bytes_per_launch"), d.get("source")
        except Exception:
            pass
    return None, None


# ------------------------------------------------------------------------------------------------ reference arm
def _oracle_admit(pos, flag, mapq, cigar_off, cigar, min_mapq, max_depth=8000):
    """keep mask from the ORACLE's admission (oracle.c orc_admit): the reference arm never loads liblvc_b200.so"""
    from oracle import c_oracle
    lib = c_oracle._load()
    n = len(pos)
    keep = np.zeros(max(n, 1), dtype=np.uint8)
    pos = np.ascontiguousarray(pos, np.int32); flag = np.ascontiguousarray(flag, np.uint16)
    mapq = np.ascontiguousarray(mapq, np.uint8); cigar_off = np.ascontiguousarray(cigar_off, np.uint32)
    cigar = np.ascontiguousarray(cigar, np.uint32)
    rc = lib.orc_admit(n, pos.ctypes.data, flag.ctypes.data, mapq.ctypes.data, cigar_off.ctypes.data, cigar.ctypes.data,
                       int(min_mapq), int(max_depth), 0, keep.ctypes.data)
    if rc:
        raise RuntimeError(f"orc_admit failed: {rc}")
    return keep[:n]


def cpu_oracle_throughput(ref, batch, min_seconds: float, max_reps: int):
    """the oracle port (oracle/oracle.c, single thread) on the same batch: deposit + genotype per rep."""
    from oracle.c_oracle import COracle
    reps, t0 = 0, time.perf_counter()
    while reps < max_reps and (reps == 0 or time.perf_counter() - t0 < min_seconds):
        co = COracle(ref, THRESH["minBQ"], THRESH["minMQ"])
        co.process(batch)
        co.genotype(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"])
        reps += 1
    dt = time.perf_counter() - t0
    return batch.aligned_bases() * reps / dt, reps, dt


def main_config(batch, G, bases, alg_bytes, world):
    return {"workload": WORKLOAD if world == 1 else WORKLOAD + f"; one such sample per GPU per step x{world} "
            "(independent samples, no communication)",
            "reads_per_step_per_gpu": batch.n_reads, "aligned_bases_per_step_per_gpu": bases,
            "algorithmic_bytes_per_step_per_gpu": alg_bytes, "ref_len": G, "thresholds": THRESH,
            "l2": "inputs (0.50 GB/step; 0.27 GB when the batch ships 2-bit quality codes) larger than L2 (126 MB); no flush needed"}


def run_reference(args):
    """--impl reference: the reference's CPU algorithm (the reference itself is pure Python + pysam, which
    this image cannot run; the C port of its algorithm is the stronger baseline) on the host cores.  Nothing of the
    product library is loaded here: the workload's keep mask comes from the oracle's own admission."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from lvc_b200 import capi
    capi.admit = _oracle_admit                     # lvc_b200.packing calls capi.admit: keep liblvc_b200.so out of this arm
    ref, batch = make_workload(20260101, N_PAIRS)
    total_steps = args.steps + args.warmup
    frac = min(1.0, 150.0 / (1.3 * max(total_steps, 1)))
    n = max(1000, int(batch.n_reads * frac))
    sample = batch if n >= batch.n_reads else batch.slice(0, n)
    from oracle.c_oracle import COracle
    for _ in range(args.warmup):
        co = COracle(ref, THRESH["minBQ"], THRESH["minMQ"]); co.process(sample)
        co.genotype(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        co = COracle(ref, THRESH["minBQ"], THRESH["minMQ"]); co.process(sample)
        co.genotype(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"])
    dt = time.perf_counter() - t0
    value = sample.aligned_bases() * args.steps / dt
    desc = f"first {sample.n_reads} of {batch.n_reads} reads of the workload per step"
    cfg = main_config(batch, len(ref), batch.aligned_bases(), batch.algorithmic_bytes(len(ref)), 1)
    cfg["variants_per_step"] = None
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32+f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port", "sample": desc,
                             "host_cores": os.cpu_count(),
                             "note": "oracle/oracle.c, one thread: the reference is single-threaded Python on pysam, "
                                     "which cannot be installed here; at N > 1 this is still ONE core on ONE sample"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "product_library_loaded": capi._lib is not None}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ extra legs
def leg_config3(torch, capi, records, stream, dev, distinct=4, n_batches=100):
    """SURVEY 8d config 3: ONT-like live batches (1,000x per batch, ~21 CIGAR ops per read, qualities 2..90), tables
    persist on the device; after EVERY batch deposit + genotype + compaction.  `distinct` seeded batches are cycled."""
    from lvc_b200 import synth
    e_lut, om_lut = records.phred_luts()
    ref = synth.random_reference(29903, 20260199)
    t0 = time.time()
    batches = [synth.ont_batch_fast(20260200 + k, ref) for k in range(distinct)]
    gen_s = time.time() - t0
    h = capi.Handle(ref.encode("latin-1"), THRESH["minBQ"], THRESH["minMQ"], device=dev.index, stream=stream.cuda_stream)

    def geno(sync=False):
        (h.genotype_device if sync else h.genotype_device_async)(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"], e_lut, om_lut)
    dbs = [to_device(torch, capi, b, dev) for b in batches]
    for db, _ in dbs:                       # synchronous first pass: allocates every quality plane that occurs
        h.push_batch_device(db)
    geno(sync=True)
    for k in range(3):
        h.push_batch_device_async(dbs[k % distinct][0]); geno()
    h.check_async()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_batches)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = h.launch_count
    e0.record(stream)
    for k in range(n_batches):
        evs[k][0].record(stream)
        h.push_batch_device_async(dbs[k % distinct][0]); geno()
        evs[k][1].record(stream)
    e1.record(stream)
    torch.cuda.synchronize()
    h.check_async()
    ms = e0.elapsed_time(e1)
    lat = np.array([x.elapsed_time(y) for x, y in evs])
    h.set_timing(True)
    for w in range(3):
        h.get_timing(w)
    for k in range(20):
        h.push_batch_device_async(dbs[k % distinct][0]); geno()
    torch.cuda.synchronize()
    h.check_async()
    h.set_timing(False)
    kt = {name: (lambda t: t[0] / max(t[1], 1))(h.get_timing(w)) for w, name in ((0, "tiled_deposit_ms"), (1, "long_read_deposit_ms"), (2, "genotype_ms"))}
    bases = sum(batches[k % distinct].aligned_bases() for k in range(n_batches))
    byts = sum(batches[k % distinct].algorithmic_bytes(len(ref)) for k in range(n_batches))
    peak, _ = measured_peak_gbs()
    out = {"workload": f"ONT-like live batches, 1,000x per batch, {batches[0].n_reads} reads/batch, {n_batches} batches "
                       f"({distinct} distinct seeds 20260200+k, cycled), incremental on-device accumulation",
           "value": bases / (ms * 1e-3), "unit": UNIT, "batch_ms_p50": float(np.percentile(lat, 50)),
           "batch_ms_p99": float(np.percentile(lat, 99)), "algorithmic_bytes": int(byts),
           "roofline_frac": byts / (ms * 1e-3) / 1e9 / peak, "gpu_launches": int(h.launch_count - n0),
           "quality_planes": len(h.plane_keys()), "kernel_avg_ms": kt, "generation_s": round(gen_s, 1)}
    h.close()
    return out


def config5_workload(ref_len=1_000_000):
    from lvc_b200 import synth
    return _cached(f"lvc_bench_cfg5_{ref_len}.npz",
                   lambda: synth.shotgun_sample(ref_len=ref_len, n_snvs=max(10, ref_len // 10000))[:2])


def leg_config5_single(torch, capi, records, stream, dev, steps=10):
    """SURVEY 8d config 5 geometry on ONE GPU (1 Mb genome instead of 5 Mb: same depth, same per-chunk geometry;
    every read is live here, so the formula fraction IS the live-bytes fraction)."""
    e_lut, om_lut = records.phred_luts()
    ref, batch = config5_workload()
    batch = in_form(batch)
    h = capi.Handle(ref.encode("latin-1"), THRESH["minBQ"], THRESH["minMQ"], device=dev.index, stream=stream.cuda_stream)
    db, keep = to_device(torch, capi, batch, dev)

    def geno(sync=False):
        (h.genotype_device if sync else h.genotype_device_async)(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"], e_lut, om_lut)
    h.push_batch_device(db); geno(sync=True)
    for _ in range(3):
        h.push_batch_device_async(db); geno()
    h.check_async()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        h.push_batch_device_async(db); geno()
    e1.record(stream)
    torch.cuda.synchronize()
    h.check_async()
    ms = e0.elapsed_time(e1) / steps
    h.set_timing(True)
    for w in range(3):
        h.get_timing(w)
    for _ in range(steps):
        h.push_batch_device_async(db); geno()
    torch.cuda.synchronize()
    h.set_timing(False)
    tile_ms, tile_n = h.get_timing(0)
    byts = batch.algorithmic_bytes(len(ref))
    lb, n_live = live_bytes(batch)
    peak, _ = measured_peak_gbs()
    out = {"workload": f"shotgun 150 bp, 1,000x, G = {len(ref)} (SURVEY config 5 geometry at 1/5 of the genome), "
                       f"{batch.n_reads} reads, seed 20260400", "value": batch.aligned_bases() / (ms * 1e-3), "unit": UNIT,
           "ms_per_step": ms, "algorithmic_bytes": int(byts), "step_frac": byts / (ms * 1e-3) / 1e9 / peak,
           "deposit_kernel_ms": tile_ms / max(tile_n, 1), "live_reads": n_live, "live_bytes": lb,
           "quality_form": form_of(batch),
           "frac_live": (lb / (tile_ms / max(tile_n, 1) * 1e-3) / 1e9 / peak) if tile_n else None, "steps": steps}
    h.close()
    del keep
    return out


def leg_config5_sharded(torch, dist, capi, records, stream, dev, world, rank, steps=8):
    """SURVEY 8e row 2 / config 5: ONE sample, contiguous chunks of the coordinate-sorted reads per rank, then the ONE
    exchange of the integer tables over NCCL, then each rank genotypes its slice of positions.  Three exchange modes
    are timed with the same deposit: reduce-scatter and all-reduce through the C-ABI (lvc_reduce_tables, one grouped
    NCCL call on the device tables), the halo-only send/recv of lvc_b200.dist, and "peer": position ownership over NVLink
    peer memory (lvc_peer_attach), where the deposit kernel reduces into the owner's tables and the exchange is a barrier."""
    from lvc_b200 import dist as ldist
    e_lut, om_lut = records.phred_luts()
    ref, batch = config5_workload()             # the keep mask was computed over the WHOLE batch
    G = len(ref)
    shards = ldist.shard_reads(batch, world)
    a, b = shards[rank]
    mine = batch.slice(a, b)
    db, keep = to_device(torch, capi, mine, dev)
    comm = ldist.make_library_comm(dev.index)
    res = {"n_ranks": world, "reads_total": batch.n_reads, "reads_this_rank": int(b - a), "ref_len": G,
           "workload": f"shotgun 150 bp, 1,000x, G = {G}, {batch.n_reads} reads, read-chunk sharded over {world} ranks"}

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def run_mode(mode):
        h = capi.Handle(ref.encode("latin-1"), THRESH["minBQ"], THRESH["minMQ"], device=dev.index, stream=stream.cuda_stream)
        touched = ldist.touched_ranges(batch, shards)
        tabs = None
        if mode == "peer":
            # position ownership over NVLink peer memory: fix the plane set, map every rank's tables, then deposit
            for k in ldist.key_union(ldist.batch_keys(mine, THRESH["minBQ"])):
                h.ensure_plane(k)
            h.sync()
            blobs = [None] * world
            dist.all_gather_object(blobs, h.peer_export())
            h.peer_attach(rank, blobs)
            h.stream_barrier(comm)
            h.sync()
        t_dep, t_exc, t_gen, t_step, nbytes = [], [], [], [], 0
        for it in range(steps + 2):
            if mode == "all_reduce" and rank != 0 and it > 0:
                h.reset()                                    # only rank 0 keeps the history between batches
            base = batch.n_reads * it
            h.ordinal = base + a
            e = [ev() for _ in range(4)]
            dist.barrier()
            torch.cuda.synchronize()
            e[0].record(stream)
            if mode == "peer":
                h.stream_barrier(comm)                       # the previous genotype pass is complete on every rank
                h.push_batch_device_async(db)                # remote columns are reduced into their owner's tables
            elif it == 0:
                h.push_batch_device(db)                      # synchronous first push: creates the quality planes
            else:
                h.push_batch_device_async(db)
            e[1].record(stream)
            if mode == "peer":
                h.stream_barrier(comm)                       # every rank's reductions have landed
                nbytes = 0
            elif mode == "halo":
                if tabs is None:
                    h.sync()
                    for k in ldist.key_union([int(k) for k in h.plane_keys()]):
                        h.ensure_plane(k)
                    tabs = ldist.device_tables(h)
                    e[1].record(stream)
                with torch.cuda.stream(stream):
                    nbytes = ldist.halo_exchange(tabs, G, touched)
                p0, p1 = ldist.position_slice(G, world, rank)
                h.set_genotype_range(p0, p1)
            else:
                nbytes = h.reduce_tables(comm, capi.REDUCE_SCATTER if mode == "reduce_scatter" else capi.REDUCE_ALL)
                if mode == "all_reduce":
                    p0, p1 = h.position_slice(world, rank)
                    h.set_genotype_range(p0, p1)
            e[2].record(stream)
            h.ordinal = base + batch.n_reads
            h.genotype_device_async(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"], e_lut, om_lut)
            e[3].record(stream)
            torch.cuda.synchronize()
            if it >= 2:
                t_dep.append(e[0].elapsed_time(e[1])); t_exc.append(e[1].elapsed_time(e[2]))
                t_gen.append(e[2].elapsed_time(e[3])); t_step.append(e[0].elapsed_time(e[3]))
        n_cand = len(h.fetch_candidates())
        t = torch.tensor([np.mean(t_dep), np.mean(t_exc), np.mean(t_gen), np.mean(t_step)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        nb = torch.tensor([nbytes, n_cand], device=dev, dtype=torch.int64)
        dist.all_reduce(nb, op=dist.ReduceOp.SUM)
        if mode == "peer":
            h.peer_detach()                                  # nobody frees tables another rank still has mapped
            dist.barrier()
        h.close()
        dep, exc, gen, step = [float(x) for x in t.tolist()]
        return {"deposit_ms": dep, "exchange_ms": exc, "genotype_slice_ms": gen, "step_ms": step,
                "exchange_bytes_all_ranks": int(nb[0].item()), "records_all_ranks": int(nb[1].item()),
                "value": batch.aligned_bases() / (step * 1e-3), "unit": UNIT}

    for mode in ("reduce_scatter", "all_reduce", "halo", "peer"):
        try:
            res[mode] = run_mode(mode)
        except Exception as ex:  # a leg must never take the headline line down
            res[mode] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
            torch.cuda.synchronize()
    res["timing"] = "CUDA events on the launching stream per phase, mean over steps, max over ranks"
    comm.close()
    del keep
    return res


def leg_config4(torch, dist, capi, records, stream, dev, world, rank, n_samples=96, steps=3, distinct=4):
    """SURVEY 8d config 4: the 96-sample plate at 5,000x each (config-2 geometry at half depth, seed 20260300 + sample),
    samples round-robin over the ranks (lvc_b200.dist.assign_samples), one handle per sample, NO communication; records
    stay with their rank (their counts are summed for the line).  Strong scaling: the plate is fixed."""
    from lvc_b200 import dist as ldist, synth
    e_lut, om_lut = records.phred_luts()
    mine = ldist.assign_samples(n_samples, world, rank)
    gen = mine[:max(1, min(distinct, len(mine)))]
    t0 = time.time()
    data = [_cached(f"lvc_bench_cfg4_{20260300 + s}.npz",
                    lambda s=s: synth.amplicon_sample(seed=20260300 + s, n_pairs=N_PAIRS // 2)) for s in gen]
    data = [(r, in_form(b)) for r, b in data]
    gen_s = time.time() - t0
    dbs = [to_device(torch, capi, b, dev) for _, b in data]
    handles = []
    for i, s in enumerate(mine):
        ref, b = data[i % len(data)]
        h = capi.Handle(ref.encode("latin-1"), THRESH["minBQ"], THRESH["minMQ"], device=dev.index, stream=stream.cuda_stream)
        handles.append((h, dbs[i % len(data)][0], b))

    def step():
        for h, db, _ in handles:
            h.push_batch_device_async(db)
            h.genotype_device_async(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"], e_lut, om_lut)
    for h, db, _ in handles:                          # first push synchronous: creates the planes
        h.push_batch_device(db)
        h.genotype_device(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"], e_lut, om_lut)
    step()
    for h, _, _ in handles:
        h.check_async()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = sum(h.launch_count for h, _, _ in handles)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    launches = sum(h.launch_count for h, _, _ in handles) - n0
    n_rec = sum(len(h.fetch_candidates()) for h, _, _ in handles)
    bases_local = sum(b.aligned_bases() for _, _, b in handles)
    bytes_local = sum(b.algorithmic_bytes(29903) for _, _, b in handles)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    tot = torch.tensor([bases_local, bytes_local, n_rec, len(handles)], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    bases, byts, recs, nh = [int(x) for x in tot.tolist()]
    peak, _ = measured_peak_gbs()
    for h, _, _ in handles:
        h.close()
    return {"workload": f"{n_samples}-sample plate, 5,000x each ({N_PAIRS // 2} pairs per sample), samples round-robin "
                        f"over {world} rank(s): {len(mine)} live handles on this GPU, no communication; "
                        f"{len(data)} distinct seeded samples per rank (20260300 + sample), cycled over its handles",
            "value": bases / (ms * 1e-3), "unit": UNIT, "scaling": "strong", "ms_per_plate": ms, "handles_total": nh,
            "handles_this_gpu": len(handles), "aligned_bases_per_plate": bases, "algorithmic_bytes_per_plate": byts,
            "roofline_frac_per_gpu": byts / world / (ms * 1e-3) / 1e9 / peak, "records_per_plate": recs,
            "gpu_launches_per_plate_this_gpu": int(launches // steps), "steps": steps, "generation_s": round(gen_s, 1),
            "stream": "all handles of a GPU launch on one stream (programmatic dependent launch overlaps "
                      "neighbouring kernels); CUDA events, max over ranks"}


def leg_e2e_api(torch, ref, batch, stream, local, tmp, reps=3):
    """The call the reference's server makes (client_server/vc_queue.py:142-144): process_bam(BAM on disk) +
    prepare_variants(), BAM decode, admission and mate-overlap pass included.  The BAM is written to directory `tmp`."""
    from lvc_b200 import samio, synth
    from variant_caller.live_variant_caller import LiveVariantCaller
    bam, fasta = os.path.join(tmp, "cfg2.bam"), os.path.join(tmp, "ref.fasta")
    t0 = time.time()
    ids, mpos, tlen = synth.amplicon_pairing(batch, N_PAIRS, len(ref))
    samio.write_bam_batch(bam, ("NC_045512.2", len(ref)), batch, name_id=ids, mate_pos=mpos, tlen=tlen)
    write_s = time.time() - t0
    with open(fasta, "w") as fh:
        fh.write(">NC_045512.2\n" + ref + "\n")
    lvc = LiveVariantCaller(fasta, THRESH["minBQ"], THRESH["minMQ"], THRESH["minDP"], THRESH["minAD"], THRESH["ratio"], 1,
                            device=local)
    lvc.process_bam(bam); lvc.prepare_variants()            # first call pins the buffer pool
    t_ing = []
    for _ in range(2):
        t1 = time.perf_counter()
        nat = samio.read_alignments_native(bam, "NC_045512.2", THRESH["minMQ"])
        t_ing.append(time.perf_counter() - t1)
        n_reads, pairs = nat.n_reads, nat.overlap_pairs
        nat.close()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    for _ in range(reps):
        lvc.process_bam(bam)
        variants = lvc.prepare_variants()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t1) / reps
    size = os.path.getsize(bam)
    lvc.close()
    return {"api": "LiveVariantCaller.process_bam(BAM on disk) + prepare_variants()", "value": batch.aligned_bases() / dt,
            "unit": UNIT, "ms_per_step": dt * 1e3, "ingest_ms": min(t_ing) * 1e3, "bam_bytes": size, "reads": n_reads,
            "mate_pairs_rewritten": pairs, "variants": len(variants), "steps": reps, "host_threads": os.cpu_count(),
            "bam_write_s": round(write_s, 1), "timing": "host wall clock around the calls (the path is host bound)"}


def dump_outputs(h, out_dir: str) -> None:
    """What the caller of the timed step receives after its last step, as float64 .npy files in `out_dir` (2.2 MB for
    config 2): the candidate records of lvc_fetch_candidates, one array per field, sorted by position and allele (the
    kernel appends them through an atomic counter, in no fixed order), and the dense per-position outputs of the genotype pass (lvc_copy_dense:
    depth, allele depths and likelihoods of the four allele slots)."""
    h.check_async()
    cand = np.sort(h.fetch_candidates(), order=["pos", "code"])
    depth, ad, lik = h.copy_dense()
    arrays = {f"candidates_{k}": cand[k] for k in ("pos", "code", "ref", "ad", "dp", "first", "L", "S", "esum")}
    arrays.update(depth=depth, allele_depth=ad, likelihood=lik)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--kernel-impl", type=int, default=0, help="0 auto (the tiled kernel for short reads, 3 for long reads), 1 general kernel, 2 tiled kernel (raw TMA staging), 3 long-read kernel, 4 tiled kernel (SWAR counters), 5 tiled kernel (bit-sliced counters)")
    ap.add_argument("--n-pairs", type=int, default=N_PAIRS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--legs", default="all", help="all | main | comma list of: config3,config4,config5,e2e_api")
    ap.add_argument("--no-numa", action="store_true")
    ap.add_argument("--device-batch", default="admitted", choices=["admitted", "masked"],
                    help="admitted: the device-resident batch holds the admitted reads only, as the packer hands it over "
                         "(ReadBatch.admitted_only / lvc_reads_compact); masked: dropped reads stay in the batch with keep bit0 clear")
    ap.add_argument("--base-form", default="codes", choices=["codes", "nibbles"],
                    help="end-to-end legs: codes = a quality-code batch also ships 2-bit base codes where its bases allow it "
                         "(what process_bam does; 0.5 payload bytes per base over PCIe); nibbles: 4-bit BAM codes (0.75)")
    ap.add_argument("--quality-form", default="codes", choices=["codes", "bytes"],
                    help="codes: batches whose qualities take <= 4 values ship 2-bit codes (what process_bam does); bytes: one phred byte per base")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them computed to DIR/<name>.npy (rank 0; the "
                         "tables accumulate over the warm-up and timed steps, so equal arguments give equal outputs)")
    args = ap.parse_args()
    global QUALITY_FORM
    QUALITY_FORM = args.quality_form
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    legs = {"config3", "config4", "config5", "e2e_api"} if args.legs == "all" else \
        (set() if args.legs == "main" else set(args.legs.split(",")))

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = {"skipped": True} if args.no_numa else bind_numa(local)       # before any CUDA / pinned allocation

    import torch
    import torch.distributed as dist
    from lvc_b200 import capi, packing, records
    from variant_caller.live_variant_caller import LiveVariantCaller

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # every rank owns an independent sample of the same geometry (rank 0 = the canonical config-2 seed)
    ref, batch = make_workload(20260101 + 1000 * rank, args.n_pairs)
    batch = in_form(batch)
    G = len(ref)
    bases = batch.aligned_bases()
    alg_bytes = batch.algorithmic_bytes(G)
    alg_bytes_deposit = alg_bytes - 52 * G
    lb, n_live = live_bytes(batch)
    e_lut, om_lut = records.phred_luts()

    # ---- device-resident inputs
    dev = torch.device("cuda", local)
    dev_batch = in_form(batch.admitted_only()) if args.device_batch == "admitted" else batch
    dbatch, t_arr = to_device(torch, capi, dev_batch, dev)
    stream = torch.cuda.Stream(device=dev)          # a real (non-null) stream: the library launches on it
    torch.cuda.set_stream(stream)
    h = capi.Handle(ref.encode("latin-1"), THRESH["minBQ"], THRESH["minMQ"], device=local, stream=stream.cuda_stream)
    h.set_impl(args.kernel_impl)

    def step_async():
        h.push_batch_device_async(dbatch)
        h.genotype_device_async(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"], e_lut, om_lut)

    # ---- warm-up: the first push is synchronous (allocates the quality planes, may replay)
    h.push_batch_device(dbatch)
    h.genotype_device(THRESH["minDP"], THRESH["minAD"], THRESH["ratio"], e_lut, om_lut)
    n_cand = len(h.fetch_candidates())
    for _ in range(args.warmup - 1):
        step_async()
    h.check_async()

    def barrier():
        if world > 1:
            dist.barrier()

    sampler = ClockSampler(local)

    def timed_region(n_steps: int, kernel_events: bool):
        """n steps between two events on the launching stream; with kernel_events the library also brackets
        every kernel launch with its own pair of events (which serialises the two kernels of a step)."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h.set_timing(kernel_events)
        h.get_timing(0); h.get_timing(1); h.get_timing(2)
        barrier()
        torch.cuda.synchronize()
        n0 = h.launch_count
        e0.record(stream)
        for _ in range(n_steps):
            step_async()
        e1.record(stream)
        torch.cuda.synchronize()
        barrier()
        h.set_timing(False)
        return e0.elapsed_time(e1), h.launch_count - n0

    sampler.start()
    # (1) the step time: EXACTLY --steps steps, the two kernels of a step back to back, nothing else on the stream
    ms, launches = timed_region(args.steps, False)
    if args.dump_outputs and rank == 0:
        dump_outputs(h, args.dump_outputs)
    # (2) the same steps again with per-kernel events: the kernels' own durations for the roofline
    ms_ev, _ = timed_region(args.steps, True)
    tile_ms, tile_n = h.get_timing(0)
    gen_ms, gen_n = h.get_timing(1)
    geno_ms, geno_n = h.get_timing(2)
    # (3) a long pass (>= 60 ms of device time) so that the clock sampler and the driver's own sampling see the load
    n_long = int(min(5000, max(args.steps, np.ceil(60.0 / max(ms / args.steps, 1e-3)))))
    ms_long, _ = timed_region(n_long, False)
    sampler.stop_flag = True
    h.check_async()
    if world > 1:
        t = torch.tensor([ms, ms_long / n_long], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_long = float(t[0].item()), float(t[1].item()) * n_long
    value = world * bases * args.steps / (ms * 1e-3)

    # ---- end to end through the public API: pinned host SoA -> process_batch -> prepare_variants
    with tempfile.TemporaryDirectory(prefix="lvc_bench_") as tmp:
        fasta = os.path.join(tmp, "ref.fasta")
        with open(fasta, "w") as fh:
            fh.write(">NC_045512.2\n" + ref + "\n")
        lvc = LiveVariantCaller(fasta, THRESH["minBQ"], THRESH["minMQ"], THRESH["minDP"], THRESH["minAD"], THRESH["ratio"],
                                1, device=local)
    lvc._handle.set_stream(stream.cuda_stream)
    lvc._handle.set_impl(args.kernel_impl)

    e2e_forms = []

    def run_e2e(b):
        """process_batch(page-locked SoA) + prepare_variants, e2e_steps times between two events; (ms, h2d bytes per
        step, records)"""
        if args.base_form == "codes":
            b = b.with_base_codes(THRESH["minBQ"])
        e2e_forms.append(form_of(b))
        pinned = packing.pin_batch(b)
        small = sum(getattr(b, k).nbytes for k in ("pos", "flag", "mapq", "keep", "cigar_off", "cigar", "seq_off"))
        lvc.reset_memory()
        for _ in range(2):
            lvc.process_batch(pinned)
            recs = lvc.prepare_variants()
        payload0 = lvc._handle.h2d_payload_bytes
        barrier()
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(args.e2e_steps):
            lvc.process_batch(pinned)
            recs = lvc.prepare_variants()
        f1.record(stream)
        torch.cuda.synchronize()
        barrier()
        t_ms = f0.elapsed_time(f1)
        if world > 1:
            t = torch.tensor([t_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_ms = float(t.item())
        # bytes that cross PCIe per step: the small per-read arrays in full (copied) + the payload the kernel pulls in
        # place (library count: the 16-byte groups of every chunk's staged extent, i.e. what the kernel requests)
        moved = small + (lvc._handle.h2d_payload_bytes - payload0) // args.e2e_steps
        del pinned
        return t_ms, moved, recs

    # the batch as the packer hands it over: reads the admission dropped are left out (ReadBatch.admitted_only); the
    # keep-masked batch of the device-resident legs is timed beside it
    e2e_ms, h2d, variants = run_e2e(batch.admitted_only())
    e2e_masked_ms, h2d_masked, variants_masked = run_e2e(batch)
    assert [(v["start"], v["alleles"], v["info"]["DP"], v["info"]["AD"]) for v in variants] == \
           [(v["start"], v["alleles"], v["info"]["DP"], v["info"]["AD"]) for v in variants_masked], \
        "e2e: the admitted-only batch and the keep-masked batch must give the same records"
    e2e_value = world * bases * args.e2e_steps / (e2e_ms * 1e-3)
    d2h = len(variants) * 48 + 4 + 32 * 4 + 8 * 4
    # admission is part of the reference's process_bam; here it runs once at pack time: its cost for this batch
    t_adm = time.perf_counter()
    capi.admit(batch.pos, batch.flag, batch.mapq, batch.cigar_off, batch.cigar, THRESH["minMQ"])
    admit_ms = (time.perf_counter() - t_adm) * 1e3
    lvc.close()

    # ---- the other SURVEY 8d workloads (each leg is fail-safe: an error string instead of a crash)
    configs, e2e_api = {}, None

    def guarded(name, fn):
        t0 = time.time()
        try:
            out = fn()
        except Exception as ex:
            import traceback
            log(f"[bench] leg {name} failed:\n" + traceback.format_exc())
            out = {"error": f"{type(ex).__name__}: {ex}"[:300]}
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
        if isinstance(out, dict):
            out["leg_wall_s"] = round(time.time() - t0, 1)
        return out

    h.close()
    del t_arr
    if "config5" in legs:
        if world == 1:
            configs["config5"] = guarded("config5", lambda: leg_config5_single(torch, capi, records, stream, dev))
        else:
            configs["config5_sharded"] = guarded("config5_sharded", lambda: leg_config5_sharded(
                torch, dist, capi, records, stream, dev, world, rank))
    if "config4" in legs:
        configs["config4"] = guarded("config4", lambda: leg_config4(torch, dist, capi, records, stream, dev, world, rank))
    if "config3" in legs and world == 1:
        configs["config3"] = guarded("config3", lambda: leg_config3(torch, capi, records, stream, dev))
    if "e2e_api" in legs and world == 1:
        with tempfile.TemporaryDirectory(prefix="lvc_bench_") as tmp:
            e2e_api = guarded("e2e_api", lambda: leg_e2e_api(torch, ref, batch, stream, local, tmp))

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        if args.kernel_impl == 1:
            tile_ms, tile_n = gen_ms, gen_n
        tile_avg_ms = tile_ms / max(tile_n, 1)
        # algorithmic bytes per launch = SURVEY 8d bytes of the reads in the batch the kernel is given.  With the
        # admitted-only device batch that is the live bytes; the figure for every PRESENTED read (60 % of which the host
        # admission drops and nobody reads) is printed beside it as frac_presented and is not a bandwidth.
        achieved_presented = alg_bytes_deposit / (tile_avg_ms * 1e-3) / 1e9 if tile_n else None
        achieved_live = lb / (tile_avg_ms * 1e-3) / 1e9 if tile_n else None
        achieved = achieved_live if args.device_batch == "admitted" else achieved_presented
        traffic, traffic_src = ncu_traffic()
        kname = {0: "k_deposit_tile5", 5: "k_deposit_tile5", 4: "k_deposit_tile4", 2: "k_deposit_tile",
                 3: "k_deposit_ont"}.get(args.kernel_impl, "k_deposit_general")
        if os.environ.get("LVC_TILE_IMPL") == "4" and args.kernel_impl == 0:
            kname = "k_deposit_tile4"
        cfg = main_config(batch, G, bases, alg_bytes, world)
        cfg["variants_per_step"] = n_cand
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32+f64", "data": "synthetic", "config": cfg,
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None,
                         "frac_live": (achieved_live / peak) if achieved_live else None,
                         "frac_presented": (achieved_presented / peak) if achieved_presented else None,
                         "frac_note": "frac = frac_live: the SURVEY 8d bytes (20 + 4 n_cigar + 1.5 l per read) of the reads "
                                      "that pass the host admission (htslib max_depth) and the read filter, i.e. of the batch "
                                      "the kernel is given, over the kernel time.  frac_presented credits the bytes of EVERY "
                                      "presented read (60 % are dropped at the depth cap and never read): a throughput "
                                      "figure, not a bandwidth" if args.device_batch == "admitted" else
                                      "frac credits the SURVEY 8d bytes of EVERY presented read; frac_live only the reads that "
                                      "pass the host admission and the read filter.  frac_live is the honest HBM fraction.",
                         "achieved_live": achieved_live, "live_bytes_per_launch": lb, "live_reads": n_live,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": lb if args.device_batch == "admitted" else alg_bytes_deposit,
                         "algorithmic_bytes_presented": alg_bytes_deposit,
                         "avg_launch_ms": tile_avg_ms, "launches_timed": tile_n,
                         "timing": "per-kernel CUDA events (library, launching stream) over a second pass of the same "
                                   "K steps; the first pass (ms_per_step) has no events between the kernels",
                         "ms_per_step_with_kernel_events": ms_ev / args.steps,
                         "step_frac": ((lb + 52 * G if args.device_batch == "admitted" else alg_bytes) / (ms / args.steps * 1e-3) / 1e9) / peak,
                         "other_kernels_ms_per_step": {"general_deposit": gen_ms / args.steps,
                                                       "genotype": geno_ms / args.steps}},
            "long_pass": {"steps": n_long, "ms_per_step": ms_long / n_long, "ms_total": ms_long,
                          "note": "same step repeated for >= 60 ms of device time (clock sampling)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / args.e2e_steps, "steps": args.e2e_steps,
                    "api": "LiveVariantCaller.process_batch(pinned SoA, admitted at pack time) + prepare_variants()",
                    "batch_form": e2e_forms[0] + "; reads the admission dropped are left out of the batch at pack time",
                    "keep_masked_batch": {"ms_per_step": e2e_masked_ms / args.e2e_steps, "h2d_bytes_per_step": int(h2d_masked),
                                          "value": world * bases * args.e2e_steps / (e2e_masked_ms * 1e-3),
                                          "note": "the same step with the dropped reads still in the batch (keep bit clear)"},
                    "admit_ms": admit_ms,
                    "h2d_note": "per-read arrays copied in full; payload of an admitted-only batch copied in bulk (one copy per "
                                "array), payload of a keep-masked batch read in place over PCIe (the 16-byte groups of each "
                                "chunk's staged extent): counted by the library"},
            "e2e_api": e2e_api,
            "device_batch": f"{dev_batch.n_reads} reads on the device ({args.device_batch}: " + (
                "the reads the host admission dropped are left out at pack time, as process_bam does" if args.device_batch == "admitted"
                else "dropped reads stay in the batch with keep bit0 clear") + f") of {batch.n_reads} presented; value counts "
                "the aligned bases of every presented read",
            "batch_form": form_of(batch) + "; the algorithmic bytes of the roofline are SURVEY 8d's (1.5 B per base) "
                          "whatever the form; --quality-form bytes ships one phred byte per base",
            "configs": configs,
            "numa": numa,
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
        }
        if world == 1 and not args.no_cpu_baseline:
            v, reps, dt = cpu_oracle_throughput(ref, batch, 10.0, 12)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
                                    "sample": f"the full workload batch, {reps} repetitions, {dt:.1f} s of CPU work "
                                              "(oracle/oracle.c, single thread like the reference)",
                                    "host_cores": os.cpu_count()}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

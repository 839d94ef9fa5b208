"""GPU, 2 ranks over NCCL (skipped on a single-GPU box): read-chunk sharding with the all-reduce of the
integer tables must reproduce the single-GPU tables and records bit for bit, across live batches."""
import os
import socket

import numpy as np
import pytest

from helpers import rows_to_tuples, assert_variants_equal

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, rows, ref, q, workdir, mode="full"):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for p in (root, os.path.join(root, "covid-spings-variant-caller_b200"), os.path.join(root, "tests")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import torch
    import torch.distributed as dist
    from lvc_b200 import packing, dist as ldist
    from variant_caller.live_variant_caller import LiveVariantCaller
    from helpers import rows_to_tuples as r2t, memory_tables
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    fa = os.path.join(workdir, f"rank{rank}.fasta")
    with open(fa, "w") as fh:
        fh.write(">c\n" + ref + "\n")
    th = dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05)
    lvc = LiveVariantCaller(fa, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=rank)
    out = []
    comm = ldist.make_library_comm(rank) if mode in ("lib_scatter", "lib_all", "peer") else None
    if mode == "peer":
        # position ownership over NVLink peer memory: the plane set is fixed and the tables are mapped BEFORE the first deposit
        allb = packing.pack_reads(r2t(rows), th["minMQ"])
        ldist.peer_setup(lvc, comm, keys=ldist.batch_keys(allb, th["minBQ"]))
    for k in range(3):                                   # three live batches
        sel = list(range(k, len(rows), 3))
        batch = packing.pack_reads(r2t([rows[i] for i in sel]), th["minMQ"])
        if mode == "peer":
            ldist.process_batch_peer(lvc, batch, comm)
        elif comm is not None:
            nbytes = ldist.process_batch_library(lvc, batch, comm, "scatter" if mode == "lib_scatter" else "all")
            assert nbytes > 0
        elif mode == "halo":
            sent = ldist.process_batch_halo(lvc, batch)
            assert sent < 4 * 4 * len(ref) * len(lvc._handle.plane_keys())      # a halo, not the tables
        else:
            ldist.process_batch_sharded(lvc, batch)
        out.append(ldist.gather_variants(lvc))
    lvc._handle.set_genotype_range(0, -1)
    if mode in ("halo", "lib_scatter", "peer"):
        # every rank keeps the history of its own slice of positions only
        p0, p1 = ldist.position_slice(len(ref), world, rank)
        lvc._candidates()                                  # genotype pass over all positions: fills the dense outputs
        depth, ad, _lik = lvc._handle.copy_dense()
        mem = (p0, p1, depth[p0:p1].tolist(), ad[p0:p1].tolist(), bool(ad[:p0].any() or ad[p1:].any()))
        gathered = [None] * world
        dist.all_gather_object(gathered, mem)
        mem = gathered
    else:
        mem = memory_tables(lvc.memory)
    if rank == 0:
        q.put((out, mem))
    if mode == "peer":
        lvc._handle.peer_detach()                          # nobody frees tables another rank still has mapped
    dist.barrier()
    lvc.close()
    if comm is not None:
        comm.close()
    dist.destroy_process_group()


def test_two_ranks_equal_one(lib, golden_synth, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from lvc_b200 import packing
    from variant_caller.live_variant_caller import LiveVariantCaller
    from helpers import memory_tables
    g = golden_synth["amplicon_like"]
    rows, ref = g["reads"], g["ref"]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, rows, ref, q, str(tmp_path))) for r in range(2)]
    for p in procs:
        p.start()
    out, mem = q.get(timeout=300)
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    fa = str(tmp_path / "c.fasta")
    with open(fa, "w") as fh:
        fh.write(">c\n" + ref + "\n")
    th = dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05)
    one = LiveVariantCaller(fa, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0)
    for k in range(3):
        sel = list(range(k, len(rows), 3))
        one.process_batch(packing.pack_reads(rows_to_tuples([rows[i] for i in sel]), th["minMQ"]))
        assert_variants_equal(out[k], one.prepare_variants(), f"batch {k}")
    assert mem == memory_tables(one.memory)
    one.close()


def test_two_ranks_halo_exchange_equal_one(lib, golden_synth, tmp_path):
    """position ownership + halo-only exchange (NCCL send/recv): records of every live batch and the per-slice
    tables must equal the single-GPU run"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from lvc_b200 import packing
    from variant_caller.live_variant_caller import LiveVariantCaller
    g = golden_synth["amplicon_like"]
    rows, ref = g["reads"], g["ref"]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, rows, ref, q, str(tmp_path), "halo")) for r in range(2)]
    for p in procs:
        p.start()
    out, slices = q.get(timeout=300)
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    fa = str(tmp_path / "c.fasta")
    with open(fa, "w") as fh:
        fh.write(">c\n" + ref + "\n")
    th = dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05)
    one = LiveVariantCaller(fa, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0)
    for k in range(3):
        sel = list(range(k, len(rows), 3))
        one.process_batch(packing.pack_reads(rows_to_tuples([rows[i] for i in sel]), th["minMQ"]))
        assert_variants_equal(out[k], one.prepare_variants(), f"batch {k}")
    one._candidates()
    depth, ad, _ = one._handle.copy_dense()
    for p0, p1, d, a, outside in slices:
        assert d == depth[p0:p1].tolist() and a == ad[p0:p1].tolist()
        assert not outside
    one.close()


@pytest.mark.parametrize("mode", ["lib_scatter", "lib_all", "peer"])
def test_two_ranks_library_exchange_equal_one(lib, golden_synth, tmp_path, mode):
    """mode "peer": lvc_peer_attach (position ownership, the deposit kernel reduces into the owner's tables over NVLink, no
    exchange step).  Otherwise lvc_reduce_tables (the C-ABI exchange: one grouped NCCL reduce-scatter / all-reduce over the device tables):
    records of every live batch and the tables must equal the single-GPU run"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from lvc_b200 import packing
    from variant_caller.live_variant_caller import LiveVariantCaller
    from helpers import memory_tables
    g = golden_synth["amplicon_like"]
    rows, ref = g["reads"], g["ref"]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, rows, ref, q, str(tmp_path), mode)) for r in range(2)]
    for p in procs:
        p.start()
    out, res = q.get(timeout=300)
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    fa = str(tmp_path / "c.fasta")
    with open(fa, "w") as fh:
        fh.write(">c\n" + ref + "\n")
    th = dict(minBQ=13, minMQ=0, minDP=3, minAD=2, ratio=0.05)
    one = LiveVariantCaller(fa, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"], 1, device=0)
    for k in range(3):
        sel = list(range(k, len(rows), 3))
        one.process_batch(packing.pack_reads(rows_to_tuples([rows[i] for i in sel]), th["minMQ"]))
        assert_variants_equal(out[k], one.prepare_variants(), f"batch {k}")
    if mode == "lib_all":
        assert res == memory_tables(one.memory)
    else:
        one._candidates()
        depth, ad, _ = one._handle.copy_dense()
        for p0, p1, d, a, outside in res:
            assert d == depth[p0:p1].tolist() and a == ad[p0:p1].tolist()
            assert not outside
    one.close()

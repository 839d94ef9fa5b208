"""Server integration (SURVEY 8f-3): the reference's UNTOUCHED task queue drives the drop-in class.

`client_server/vc_queue.py:123-146` (`VCQueue._process_bam`: samtools sort + index -> load_checkpoint -> process_bam ->
create_checkpoint -> write_vcf) is imported from an unmodified checkout of the reference project named by the
LVC_REFERENCE environment variable (the test skips without one), with the drop-in `variant_caller` package on the
path instead of the reference's, exactly what a deployment that switches to this repo does.  pysam is not installable here, so `pysam.sort` / `pysam.index` are stubbed (the
drop-in sorts SAM input itself and needs no index).  The queue is fed like the reference's own test
(test/vc_queue_test.py:30-36: put(('process', 'testdata/testfile.sam')); process()), and the VCF and the checkpoint
it leaves on disk are compared with the oracle's.  Needs a GPU (the drop-in has no CPU path)."""
import importlib
import os
import pickle
import shutil
import sys
import time
import types

import pytest

from oracle import pileup_oracle as po
from conftest import GOLD, PKG

pytestmark = pytest.mark.gpu


def _reference_tree():
    cand = os.environ.get("LVC_REFERENCE")
    if cand and os.path.exists(os.path.join(cand, "client_server", "vc_queue.py")):
        return cand
    return None


def _norm(mem):
    return {int(p): (s["reference"], int(s["totalDepth"]), {a: sorted(int(x) for x in v) for a, v in s["snvs"].items()},
                     list(s["snvs"])) for p, s in mem.items()}


@pytest.mark.parametrize("relaxed", [False, True])
def test_vcqueue_process_with_dropin(lib, tmp_path, monkeypatch, relaxed):
    tree = _reference_tree()
    if tree is None:
        pytest.skip("LVC_REFERENCE does not name a checkout of the reference project")
    work = tmp_path / "server"
    work.mkdir()
    for sub in ("client_server", "config_util"):                       # unmodified copies in a scratch directory
        shutil.copytree(os.path.join(tree, sub), work / sub)
    for d in ("log", "tmp", "output", "input"):
        (work / d).mkdir()
    shutil.copy(os.path.join(GOLD, "NC_045512.2.synthetic.fasta"), work / "input" / "reference-covid.fasta")
    sam = work / "input" / "testfile.sam"
    shutil.copy(os.path.join(GOLD, "testfile.sam"), sam)
    th = dict(minBQ=30, minMQ=20, minDP=10, minAD=5, ratio=0.10)       # config_util/vc.config as shipped
    if relaxed:
        # vc.config is configuration, not code: relaxed thresholds so that the fixture yields records
        th = dict(minBQ=13, minMQ=0, minDP=1, minAD=1, ratio=0.0)           # golden set "bq13": 4 records
        cfg = (work / "config_util" / "vc.config").read_text()
        for k, v in (("MIN_EVIDENCE_DEPTH", th["minAD"]), ("MIN_EVIDENCE_RATIO", th["ratio"]), ("MIN_TOTAL_DEPTH", th["minDP"]),
                     ("MIN_MAPPING_QUALITY", th["minMQ"]), ("MIN_BASE_QUALITY", th["minBQ"])):
            cfg = "\n".join((f"{k} = {v}" if line.startswith(k + " ") else line) for line in cfg.split("\n"))
        (work / "config_util" / "vc.config").write_text(cfg)

    # pysam stub: samtools sort -> the drop-in reads (and sorts) SAM text itself, so "sorting to BAM" is a copy;
    # samtools index -> an empty .bai (vc_queue.py:136 only checks that it exists)
    calls = []
    stub = types.ModuleType("pysam")

    def sort(*args):
        calls.append(("sort",) + args)
        out = args[args.index("-o") + 1]
        shutil.copy(args[-1], out)

    def index(bam, bai=None):
        calls.append(("index", bam, bai))
        open(bai or bam + ".bai", "wb").close()
    stub.sort, stub.index = sort, index
    monkeypatch.setitem(sys.modules, "pysam", stub)
    for m in [m for m in sys.modules if m.split(".")[0] in ("client_server", "config_util", "variant_caller")]:
        monkeypatch.delitem(sys.modules, m)
    monkeypatch.syspath_prepend(PKG)                                   # the drop-in variant_caller package
    monkeypatch.syspath_prepend(str(work))                             # the reference's client_server + config_util
    monkeypatch.chdir(work)                                            # OUTPUT_DIR / TEMP_DIR are relative paths
    vq = importlib.import_module("client_server.vc_queue")
    assert os.path.dirname(vq.__file__) == str(work / "client_server")
    lvc_mod = sys.modules["variant_caller.live_variant_caller"]
    assert os.path.dirname(os.path.dirname(lvc_mod.__file__)) == PKG   # the queue really holds the drop-in class

    q = vq.VCQueue(5)
    vcf = work / "output" / "testfile.bam.vcf"
    ckpt = work / "tmp" / "testfile.bam.pkl"

    def run_once():
        if vcf.exists():
            vcf.unlink()
        q.put(("process", str(sam)))
        q.process()                                                    # starts the daemon thread (vc_queue.py:99-111)
        assert q.length() == 0                                         # what the reference's own test asserts
        t0 = time.time()
        while not vcf.exists() and time.time() - t0 < 120:
            time.sleep(0.05)
        assert vcf.exists(), "the worker thread died before writing the VCF"
        time.sleep(0.2)

    contigs, reads = po.read_sam(os.path.join(GOLD, "testfile.sam"))
    fasta = (work / "input" / "reference-covid.fasta").read_text().split("\n", 1)[1].replace("\n", "")
    oc = po.OracleCaller(fasta, th["minBQ"], th["minMQ"], th["minDP"], th["minAD"], th["ratio"])

    run_once()
    oc.process_reads(po.samtools_sort(reads))
    assert [c[0] for c in calls] == ["sort", "index"]
    assert vcf.read_text() == oc.vcf_text(contigs)
    with open(ckpt, "rb") as fh:
        assert _norm(pickle.load(fh)) == _norm(oc.memory)
    n_first = len(oc.prepare_variants())
    assert (n_first > 0) == relaxed                                    # vc.config as shipped: header-only VCF (SURVEY C)

    # the same file again: the checkpoint is loaded first, then the whole file is processed again (reference
    # behaviour, vc_queue.py:138-142: counts double)
    run_once()
    oc.process_reads(po.samtools_sort(reads))
    assert vcf.read_text() == oc.vcf_text(contigs)
    with open(ckpt, "rb") as fh:
        assert _norm(pickle.load(fh)) == _norm(oc.memory)
    q.live_variant_caller.close()

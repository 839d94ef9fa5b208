"""ctypes binding of liblvc_b200.so (the C-ABI declared in include/lvc.h).

There is NO CPU fallback: if the shared library is missing, or no CUDA device is visible when a
handle is created, this raises.  Nothing here imports anything from ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LVC_LIB_PATH") or os.path.join(_HERE, "liblvc_b200.so")   # override: kernel experiments

LVC_OK = 0
ERRORS = {-1: "LVC_EINVAL", -2: "LVC_ECUDA", -3: "LVC_ENOMEM", -4: "LVC_EUNSORTED", -5: "LVC_ERANGE",
          -6: "LVC_ENODEVICE", -7: "LVC_EAGAIN", -8: "LVC_EIO"}
GENO_EMIT_ALL = 1
MAX_DEPTH_DEFAULT = 8000
# htslib mate-overlap models (include/lvc.h): pysam's pileup() default is ignore_overlaps=True
OVERLAP_OFF, OVERLAP_HTSLIB_1_10, OVERLAP_HTSLIB_1_13 = 0, 1, 2
OVERLAP_DEFAULT = OVERLAP_HTSLIB_1_13
OVERLAP_MODELS = {None: OVERLAP_DEFAULT, "off": OVERLAP_OFF, "htslib-1.10": OVERLAP_HTSLIB_1_10,
                  "htslib-1.13": OVERLAP_HTSLIB_1_13}


class LvcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code


class Batch(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("qual_bits", C.c_uint32), ("n_cigar_ops", C.c_uint64),
                ("n_qual_bytes", C.c_uint64), ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p),
                ("keep", C.c_void_p), ("cigar_off", C.c_void_p), ("cigar", C.c_void_p), ("seq_off", C.c_void_p),
                ("seq4", C.c_void_p), ("qual", C.c_void_p), ("qual_dict", C.c_uint8 * 4), ("seq_form", C.c_uint32)]


class Candidate(C.Structure):
    _fields_ = [("pos", C.c_int32), ("code", C.c_uint8), ("ref", C.c_uint8), ("pad0", C.c_uint16),
                ("ad", C.c_uint32), ("dp", C.c_uint32), ("first", C.c_uint32), ("pad1", C.c_uint32),
                ("L", C.c_double), ("S", C.c_double), ("esum", C.c_double)]


CANDIDATE_DTYPE = np.dtype([("pos", "<i4"), ("code", "u1"), ("ref", "u1"), ("pad0", "<u2"), ("ad", "<u4"),
                            ("dp", "<u4"), ("first", "<u4"), ("pad1", "<u4"), ("L", "<f8"), ("S", "<f8"),
                            ("esum", "<f8")])
assert CANDIDATE_DTYPE.itemsize == C.sizeof(Candidate) == 48

CONSENSUS_COUNTERS = ("n_positions", "depth_sum", "depth_max", "n_low_depth", "n_N", "n_deleted", "n_ambiguous",
                      "n_mismatch")


class ConsensusStats(C.Structure):
    _fields_ = [(name, C.c_uint64) for name in CONSENSUS_COUNTERS] + [("depth_ge", C.c_uint64 * 8)]


assert C.sizeof(ConsensusStats) == 128

# lvc_insertion (include/lvc.h): anchor position, length (0 = unresolved), 2-bit codes (base k in bits 2k), reads, depth
INSERTION_DTYPE = np.dtype([("pos", "<i4"), ("len", "<u4"), ("seq", "<u8"), ("count", "<u4"), ("depth", "<u4")])
assert INSERTION_DTYPE.itemsize == 24

# lvc_linkage_pair (include/lvc.h): the two sites, their alts (ASCII) and count[state_a][state_b], REF 0 / ALT 1 / OTHER 2
LINKAGE_DTYPE = np.dtype([("pos_a", "<i4"), ("pos_b", "<i4"), ("alt_a", "u1"), ("alt_b", "u1"), ("pad", "<u2"),
                          ("count", "<u4", (3, 3))])
assert LINKAGE_DTYPE.itemsize == 48

_lib: Optional[C.CDLL] = None

# every symbol include/lvc.h declares: (name, restype, argtypes)
_H = C.c_void_p
SIGNATURES = [
    ("lvc_version", C.c_int, []),
    ("lvc_create", C.c_int, [C.POINTER(_H), C.c_int, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    ("lvc_destroy", None, [_H]),
    ("lvc_reset", C.c_int, [_H]),
    ("lvc_last_error", C.c_char_p, [_H]),
    ("lvc_set_stream", C.c_int, [_H, C.c_void_p]),
    ("lvc_sync", C.c_int, [_H]),
    ("lvc_admit", C.c_int, [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                            C.c_void_p]),
    ("lvc_admit_overlaps", C.c_int, [C.c_uint32] + [C.c_void_p] * 13 + [C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                                       C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ("lvc_read_alignments", C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.c_char_p,
                                      C.c_int]),
    ("lvc_read_alignments_ex", C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p),
                                         C.c_char_p, C.c_int]),
    ("lvc_reads_overlap_stats", C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ("lvc_reads_batch", C.c_int, [C.c_void_p, C.POINTER(Batch)]),
    ("lvc_reads_batch_bytes", C.c_int, [C.c_void_p, C.POINTER(Batch)]),
    ("lvc_reads_compact", C.c_int, [C.c_void_p, C.c_int]),
    ("lvc_pack_quality_codes", C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_void_p, C.c_void_p]),
    ("lvc_pack_base_codes", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    ("lvc_reads_batch_for", C.c_int, [C.c_void_p, C.c_int, C.POINTER(Batch)]),
    ("lvc_reads_info", C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int),
                                 C.POINTER(C.c_int)]),
    ("lvc_reads_free", None, [C.c_void_p]),
    ("lvc_push_batch", C.c_int, [_H, C.POINTER(Batch)]),
    ("lvc_push_batch_device", C.c_int, [_H, C.POINTER(Batch)]),
    ("lvc_set_impl", C.c_int, [_H, C.c_int]),
    ("lvc_push_batch_device_async", C.c_int, [_H, C.POINTER(Batch)]),
    ("lvc_check_async", C.c_int, [_H]),
    ("lvc_genotype_device_async", C.c_int, [_H, C.c_int64, C.c_int64, C.c_double, C.c_void_p, C.c_void_p, C.c_uint32]),
    ("lvc_set_timing", C.c_int, [_H, C.c_int]),
    ("lvc_get_timing", C.c_int, [_H, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    ("lvc_host_alloc", C.c_void_p, [C.c_uint64]),
    ("lvc_host_free", None, [C.c_void_p]),
    ("lvc_genotype", C.c_int, [_H, C.c_int64, C.c_int64, C.c_double, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p,
                               C.c_uint32, C.POINTER(C.c_uint32)]),
    ("lvc_genotype_device", C.c_int, [_H, C.c_int64, C.c_int64, C.c_double, C.c_void_p, C.c_void_p, C.c_uint32]),
    ("lvc_fetch_candidates", C.c_int, [_H, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]),
    ("lvc_set_genotype_range", C.c_int, [_H, C.c_int64, C.c_int64]),
    ("lvc_copy_dense", C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("lvc_consensus", C.c_int, [_H, C.c_int64, C.c_int64, C.c_uint64, C.c_double, C.c_void_p, C.c_int, C.c_void_p,
                                C.POINTER(ConsensusStats)]),
    ("lvc_enable_insertions", C.c_int, [_H, C.c_uint32]),
    ("lvc_copy_insertions", C.c_int, [_H, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]),
    ("lvc_insertion_calls", C.c_int, [_H, C.c_int64, C.c_int64, C.c_uint64, C.c_double, C.c_void_p, C.c_uint32,
                                      C.POINTER(C.c_uint32)]),
    ("lvc_set_linkage_sites", C.c_int, [_H, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32]),
    ("lvc_copy_linkage", C.c_int, [_H, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]),
    ("lvc_enable_strand_counts", C.c_int, [_H]),
    ("lvc_strand_counts", C.c_int, [_H, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("lvc_num_planes", C.c_int, [_H]),
    ("lvc_plane_keys", C.c_int, [_H, C.c_void_p]),
    ("lvc_ensure_plane", C.c_int, [_H, C.c_uint16]),
    ("lvc_copy_plane", C.c_int, [_H, C.c_uint16, C.c_void_p]),
    ("lvc_import_plane", C.c_int, [_H, C.c_uint16, C.c_void_p, C.c_int]),
    ("lvc_copy_dels", C.c_int, [_H, C.c_void_p]),
    ("lvc_import_dels", C.c_int, [_H, C.c_void_p, C.c_int]),
    ("lvc_copy_covdiff", C.c_int, [_H, C.c_void_p]),
    ("lvc_import_covdiff", C.c_int, [_H, C.c_void_p, C.c_int]),
    ("lvc_copy_first", C.c_int, [_H, C.c_int, C.c_void_p]),
    ("lvc_import_first", C.c_int, [_H, C.c_int, C.c_void_p]),
    ("lvc_ordinal", C.c_uint64, [_H]),
    ("lvc_set_ordinal", C.c_int, [_H, C.c_uint64]),
    ("lvc_plane_devptr", C.c_void_p, [_H, C.c_uint16]),
    ("lvc_dels_devptr", C.c_void_p, [_H]),
    ("lvc_covdiff_devptr", C.c_void_p, [_H]),
    ("lvc_first_devptr", C.c_void_p, [_H, C.c_int]),
    ("lvc_nccl_unique_id", C.c_int, [C.c_void_p]),
    ("lvc_nccl_comm_create", C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_void_p]),
    ("lvc_nccl_comm_destroy", None, [C.c_void_p]),
    ("lvc_position_slice", C.c_int, [_H, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("lvc_reduce_tables", C.c_int, [_H, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    ("lvc_last_exchange_bytes", C.c_uint64, [_H]),
    ("lvc_peer_export", C.c_int, [_H, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    ("lvc_peer_attach", C.c_int, [_H, C.c_int, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    ("lvc_peer_detach", C.c_int, [_H]),
    ("lvc_stream_barrier", C.c_int, [_H, C.c_void_p]),
    ("lvc_launch_count", C.c_uint64, [_H]),
    ("lvc_h2d_payload_bytes", C.c_uint64, [_H]),
]


def load_library() -> C.CDLL:
    """Load liblvc_b200.so (built in-tree by __graft_entry__.build()).  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: build it with `python __graft_entry__.py` "
                          "(nvcc, sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SIGNATURES:
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a) -> Optional[int]:
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return int(a)


def admit(pos: np.ndarray, flag: np.ndarray, mapq: np.ndarray, cigar_off: np.ndarray, cigar: np.ndarray,
          min_mapq: int, max_depth: int = MAX_DEPTH_DEFAULT) -> np.ndarray:
    """keep-mask (bit0) of the host-side admission rules; needs no GPU."""
    lib = load_library()
    n = len(pos)
    keep = np.zeros(n, dtype=np.uint8)
    if n == 0:
        return keep
    rc = lib.lvc_admit(n, _ptr(pos), _ptr(flag), _ptr(mapq), _ptr(cigar_off), _ptr(cigar), int(min_mapq),
                       int(max_depth), _ptr(keep))
    if rc == -4:
        raise ValueError("reads are not coordinate sorted (the reference's pileup engine errors out too)")
    if rc != LVC_OK:
        raise LvcError(rc, "lvc_admit failed")
    return keep


def overlap_model_id(model) -> int:
    """None / "off" / "htslib-1.10" / "htslib-1.13" (or the integer ids of include/lvc.h)"""
    if isinstance(model, int) and not isinstance(model, bool):
        if model in (OVERLAP_OFF, OVERLAP_HTSLIB_1_10, OVERLAP_HTSLIB_1_13):
            return model
    elif model in OVERLAP_MODELS:
        return OVERLAP_MODELS[model]
    raise ValueError(f"unknown overlap model {model!r}; one of {[k for k in OVERLAP_MODELS if k]}")


def admit_overlaps(pos, flag, mapq, cigar_off, cigar, seq_off, seq4, qual, names, mate_pos, mate_ref, tlen,
                   min_mapq: int, max_depth: int = MAX_DEPTH_DEFAULT, overlap_model: int = OVERLAP_DEFAULT):
    """lvc_admit_overlaps: keep mask + htslib's mate-overlap quality rewrite, IN PLACE on `qual`; needs no GPU.
    `names`: list of QNAME strings.  Returns (keep, pairs rewritten, quality bytes rewritten)."""
    lib = load_library()
    n = len(pos)
    keep = np.zeros(n, dtype=np.uint8)
    if n == 0:
        return keep, 0, 0
    enc = [x.encode("latin-1") for x in names]
    name_off = np.zeros(n + 1, dtype=np.uint32)
    np.cumsum([len(x) for x in enc], out=name_off[1:])
    blob = np.frombuffer(b"".join(enc) + b"\0", dtype=np.uint8)
    mate_pos = np.ascontiguousarray(mate_pos, dtype=np.int32)
    mate_ref = np.ascontiguousarray(mate_ref, dtype=np.int8)
    tlen = np.ascontiguousarray(tlen, dtype=np.int32)
    pairs, bases = C.c_uint64(0), C.c_uint64(0)
    rc = lib.lvc_admit_overlaps(n, _ptr(pos), _ptr(flag), _ptr(mapq), _ptr(cigar_off), _ptr(cigar), _ptr(seq_off),
                                _ptr(seq4), _ptr(qual), _ptr(name_off), _ptr(blob), _ptr(mate_pos), _ptr(mate_ref),
                                _ptr(tlen), int(min_mapq), int(max_depth), int(overlap_model), _ptr(keep),
                                C.byref(pairs), C.byref(bases))
    if rc == -4:
        raise ValueError("reads are not coordinate sorted (the reference's pileup engine errors out too)")
    if rc != LVC_OK:
        raise LvcError(rc, "lvc_admit_overlaps failed")
    return keep, int(pairs.value), int(bases.value)


def pack_quality_codes(qual: np.ndarray, n_qual: int, keep: Optional[np.ndarray] = None,
                       seq_off: Optional[np.ndarray] = None, cigar_off: Optional[np.ndarray] = None,
                       cigar: Optional[np.ndarray] = None, n_threads: int = 0):
    """lvc_pack_quality_codes: (codes uint8 [(n_qual+3)//4 + 64 slack], dict bytes[4]) or None if the qualities (of the
    l_qseq bases of the reads with keep bit0 set, when the per-read arrays are given) take more than four distinct
    values."""
    lib = load_library()
    qual = np.ascontiguousarray(qual, dtype=np.uint8)
    codes = np.zeros((n_qual + 3) // 4 + 64, dtype=np.uint8)
    d = np.zeros(4, dtype=np.uint8)
    n_reads = 0
    if keep is not None and seq_off is not None and cigar_off is not None and cigar is not None:
        keep = np.ascontiguousarray(keep, dtype=np.uint8)
        seq_off = np.ascontiguousarray(seq_off, dtype=np.uint64)
        cigar_off = np.ascontiguousarray(cigar_off, dtype=np.uint32)
        cigar = np.ascontiguousarray(cigar, dtype=np.uint32)
        n_reads = len(keep)
    rc = lib.lvc_pack_quality_codes(_ptr(qual), int(n_qual), int(n_reads), _ptr(keep) if n_reads else None,
                                    _ptr(seq_off) if n_reads else None, _ptr(cigar_off) if n_reads else None,
                                    _ptr(cigar) if n_reads else None, int(n_threads), _ptr(d), _ptr(codes))
    if rc < 0:
        raise LvcError(rc, "lvc_pack_quality_codes failed")
    if rc == 0:
        return None
    return codes, bytes(d)


def pack_base_codes(seq4: np.ndarray, qual: np.ndarray, n_qual: int, keep: np.ndarray, seq_off: np.ndarray,
                    cigar_off: np.ndarray, cigar: np.ndarray, min_base_quality: int, n_threads: int = 0):
    """lvc_pack_base_codes: 2-bit base codes (uint8 [(n_qual+3)//4 + 64 slack]) or None if a base that can reach the
    tables (admitted read, quality >= min_base_quality) is not A, C, G or T."""
    lib = load_library()
    arrs = [np.ascontiguousarray(seq4, dtype=np.uint8), np.ascontiguousarray(qual, dtype=np.uint8),
            np.ascontiguousarray(keep, dtype=np.uint8), np.ascontiguousarray(seq_off, dtype=np.uint64),
            np.ascontiguousarray(cigar_off, dtype=np.uint32), np.ascontiguousarray(cigar, dtype=np.uint32)]
    codes = np.zeros((n_qual + 3) // 4 + 64, dtype=np.uint8)
    rc = lib.lvc_pack_base_codes(_ptr(arrs[0]), _ptr(arrs[1]), int(n_qual), int(len(arrs[2])), _ptr(arrs[2]), _ptr(arrs[3]),
                                 _ptr(arrs[4]), _ptr(arrs[5]), int(min_base_quality), int(n_threads), _ptr(codes))
    if rc < 0:
        raise LvcError(rc, "lvc_pack_base_codes failed")
    return codes if rc == 1 else None


class NativeReads:
    """Alignments of one contig read and packed by the native ingest (lvc_read_alignments)."""

    def __init__(self, path: str, contig: Optional[str], min_mapq: int, max_depth: int = MAX_DEPTH_DEFAULT,
                 n_threads: int = 0, overlap_model: int = OVERLAP_DEFAULT):
        self.lib = load_library()
        if not os.path.exists(path):
            raise FileNotFoundError(path)                      # pysam raises OSError for a missing file too
        r = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = self.lib.lvc_read_alignments_ex(path.encode(), (contig or "").encode(), int(min_mapq), int(max_depth),
                                             int(n_threads), int(overlap_model), C.byref(r), err, 512)
        if rc != LVC_OK:
            msg = err.value.decode()
            if "invalid contig" in msg or "not coordinate sorted" in msg:
                raise ValueError(msg)
            from .packing import UnsupportedInput
            if rc == -1:
                raise UnsupportedInput(msg)
            raise LvcError(rc, msg)
        self.r = r
        self.n_threads = int(n_threads)
        self._take_batches()
        self.n_presented = int(self.batch_bytes.n_reads)       # reads of the contig in the file
        name = C.create_string_buffer(256)
        ln, nc, pinned = C.c_int64(0), C.c_int(0), C.c_int(0)
        self.lib.lvc_reads_info(self.r, name, 256, C.byref(ln), C.byref(nc), C.byref(pinned))
        self.contig, self.contig_len, self.pinned = name.value.decode(), ln.value, bool(pinned.value)
        op, ob = C.c_uint64(0), C.c_uint64(0)
        self.lib.lvc_reads_overlap_stats(self.r, C.byref(op), C.byref(ob))
        self.overlap_pairs, self.overlap_bases = int(op.value), int(ob.value)

    def _take_batches(self):
        self._batch = None
        self.batch_bytes = Batch()                             # always one phred byte per base
        self.lib.lvc_reads_batch_bytes(self.r, C.byref(self.batch_bytes))
        self.batch_bytes._keepalive = self

    @property
    def batch(self) -> Batch:
        """what process_bam pushes: 2-bit quality codes if the file qualifies (made on first use), else phred bytes"""
        if self._batch is None:
            self._batch = Batch()
            self.lib.lvc_reads_batch(self.r, C.byref(self._batch))
            self._batch._keepalive = self
        return self._batch

    def batch_for(self, min_base_quality: int) -> Batch:
        """lvc_reads_batch_for: `batch` for a handle with this base-quality threshold -- a quality-code batch also carries
        2-bit base codes when every base that can reach the tables is A, C, G or T (0.5 payload bytes per base)"""
        b = Batch()
        self.lib.lvc_reads_batch_for(self.r, int(min_base_quality), C.byref(b))
        b._keepalive = self
        return b

    def compact(self) -> bool:
        """lvc_reads_compact: leave out the reads the admission dropped (views taken before are invalid)"""
        rc = self.lib.lvc_reads_compact(self.r, self.n_threads)
        if rc < 0:
            raise LvcError(rc, "lvc_reads_compact failed")
        self._take_batches()
        return rc == 1

    @property
    def n_reads(self) -> int:
        return int(self.batch_bytes.n_reads)

    def as_readbatch(self):
        """numpy views (no copy) in the layout of packing.ReadBatch; valid while this object lives"""
        from .packing import ReadBatch
        b = self.batch_bytes
        n = b.n_reads

        def view(ptr, dtype, count):
            if count == 0:
                return np.zeros(0, dtype=dtype)
            buf = (C.c_uint8 * (count * np.dtype(dtype).itemsize)).from_address(ptr)
            return np.frombuffer(buf, dtype=dtype, count=count)
        rb = ReadBatch(view(b.pos, np.int32, n), view(b.flag, np.uint16, n), view(b.mapq, np.uint8, n),
                       view(b.keep, np.uint8, n), view(b.cigar_off, np.uint32, n + 1),
                       view(b.cigar, np.uint32, max(int(b.n_cigar_ops), 1)), view(b.seq_off, np.uint64, n + 1),
                       view(b.seq4, np.uint8, int(b.n_qual_bytes) // 2 + 64), view(b.qual, np.uint8, int(b.n_qual_bytes) + 64))
        if self.batch.qual_bits == 2:
            rb.qcode = view(self.batch.qual, np.uint8, int(b.n_qual_bytes) // 4 + 16)
            rb.qdict = bytes(self.batch.qual_dict)
        rb._keepalive = self
        return rb

    def close(self):
        if getattr(self, "r", None):
            self.lib.lvc_reads_free(self.r)
            self.r = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


REDUCE_ALL, REDUCE_SCATTER = 0, 1


def nccl_unique_id() -> bytes:
    """128 bytes identifying a new NCCL communicator (rank 0 creates it and ships it to the other ranks)."""
    lib = load_library()
    buf = C.create_string_buffer(128)
    rc = lib.lvc_nccl_unique_id(buf)
    if rc != LVC_OK:
        raise LvcError(rc, lib.lvc_last_error(None).decode())
    return buf.raw


class NcclComm:
    """An ncclComm_t owned by the library (one per process = per GPU)."""

    def __init__(self, device: int, n_ranks: int, rank: int, unique_id: bytes):
        self.lib = load_library()
        self.n_ranks, self.rank = int(n_ranks), int(rank)
        c = C.c_void_p()
        idb = C.create_string_buffer(unique_id, 128)
        rc = self.lib.lvc_nccl_comm_create(C.byref(c), int(device), self.n_ranks, self.rank, idb)
        if rc != LVC_OK:
            raise LvcError(rc, self.lib.lvc_last_error(None).decode())
        self.c = c

    def close(self):
        if getattr(self, "c", None):
            self.lib.lvc_nccl_comm_destroy(self.c)
            self.c = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Handle:
    """Owns one lvc_handle (one contig's persistent device tables)."""

    def __init__(self, ref_bytes: bytes, min_base_quality: int, min_mapping_quality: int, device: int = 0,
                 stream: Optional[int] = None):
        self.lib = load_library()
        self.G = len(ref_bytes)
        self._ref = np.frombuffer(ref_bytes, dtype=np.uint8).copy()
        h = _H()
        rc = self.lib.lvc_create(C.byref(h), int(device), self.G, self._ref.ctypes.data, int(min_base_quality),
                                 int(min_mapping_quality), stream)
        if rc != LVC_OK:
            msg = self.lib.lvc_last_error(None).decode()
            raise LvcError(rc, msg)
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.lib.lvc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != LVC_OK:
            raise LvcError(rc, self.lib.lvc_last_error(self.h).decode())

    # ---- lifetime
    def reset(self):
        self._check(self.lib.lvc_reset(self.h))

    def set_impl(self, impl: int):
        self._check(self.lib.lvc_set_impl(self.h, impl))

    def set_stream(self, stream: Optional[int]):
        self._check(self.lib.lvc_set_stream(self.h, stream))

    def sync(self):
        self._check(self.lib.lvc_sync(self.h))

    # ---- deposit
    @staticmethod
    def make_batch(n_reads, n_cigar, n_qual, pos, flag, mapq, keep, cigar_off, cigar, seq_off, seq4, qual,
                   qual_dict=None, base_codes_min_bq=None) -> Batch:
        """`qual_dict` (4 phred values): `qual` holds 2-bit quality codes (lvc_batch::qual_bits == 2), else phred bytes.
        `base_codes_min_bq` (with qual_dict): `seq4` holds 2-bit base codes made for that base-quality threshold"""
        b = Batch(int(n_reads), 2 if qual_dict is not None else 0, int(n_cigar), int(n_qual), _ptr(pos), _ptr(flag),
                  _ptr(mapq), _ptr(keep), _ptr(cigar_off), _ptr(cigar), _ptr(seq_off), _ptr(seq4), _ptr(qual))
        if qual_dict is not None:
            for k in range(4):
                b.qual_dict[k] = int(qual_dict[k])
        if base_codes_min_bq is not None:
            b.seq_form = 2 | (max(0, min(int(base_codes_min_bq), 255)) << 8)
        return b

    def push_batch(self, batch: Batch):
        self._check(self.lib.lvc_push_batch(self.h, C.byref(batch)))

    def push_batch_device(self, batch: Batch):
        self._check(self.lib.lvc_push_batch_device(self.h, C.byref(batch)))

    def push_batch_device_async(self, batch: Batch):
        self._check(self.lib.lvc_push_batch_device_async(self.h, C.byref(batch)))

    def check_async(self):
        self._check(self.lib.lvc_check_async(self.h))

    def genotype_device_async(self, min_total_depth, min_allele_depth, min_ratio, e_lut, om_lut, flags=0):
        self._check(self.lib.lvc_genotype_device_async(self.h, int(min_total_depth), int(min_allele_depth),
                                                       float(min_ratio), e_lut.ctypes.data, om_lut.ctypes.data,
                                                       int(flags)))

    def set_timing(self, on: bool):
        self._check(self.lib.lvc_set_timing(self.h, int(on)))

    def get_timing(self, which: int):
        ms, n = C.c_double(0), C.c_uint64(0)
        self._check(self.lib.lvc_get_timing(self.h, which, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # ---- genotype
    def genotype(self, min_total_depth: int, min_allele_depth: int, min_ratio: float, e_lut: np.ndarray,
                 om_lut: np.ndarray, flags: int = 0) -> np.ndarray:
        cap = 1 << 14
        while True:
            out = np.zeros(cap, dtype=CANDIDATE_DTYPE)
            n = C.c_uint32(0)
            self._check(self.lib.lvc_genotype(self.h, int(min_total_depth), int(min_allele_depth), float(min_ratio),
                                              e_lut.ctypes.data, om_lut.ctypes.data, int(flags), out.ctypes.data, cap,
                                              C.byref(n)))
            if n.value <= cap:
                return out[:n.value]
            cap = n.value

    def genotype_device(self, min_total_depth, min_allele_depth, min_ratio, e_lut, om_lut, flags=0):
        self._check(self.lib.lvc_genotype_device(self.h, int(min_total_depth), int(min_allele_depth), float(min_ratio),
                                                 e_lut.ctypes.data, om_lut.ctypes.data, int(flags)))

    def fetch_candidates(self) -> np.ndarray:
        n = C.c_uint32(0)
        self._check(self.lib.lvc_fetch_candidates(self.h, None, 0, C.byref(n)))
        out = np.zeros(max(n.value, 1), dtype=CANDIDATE_DTYPE)
        self._check(self.lib.lvc_fetch_candidates(self.h, out.ctypes.data, len(out), C.byref(n)))
        return out[:n.value]

    def reduce_tables(self, comm: NcclComm, mode: int = REDUCE_SCATTER) -> int:
        """the one exchange step of the read-chunk sharding (lvc_reduce_tables); returns the bytes fed in"""
        self._check(self.lib.lvc_reduce_tables(self.h, comm.c, comm.n_ranks, comm.rank, int(mode)))
        return int(self.lib.lvc_last_exchange_bytes(self.h))

    def peer_export(self) -> bytes:
        """CUDA IPC blob of this handle's tables (lvc_peer_export) for the other ranks' peer_attach"""
        n = C.c_size_t(0)
        self._check(self.lib.lvc_peer_export(self.h, None, 0, C.byref(n)))
        buf = C.create_string_buffer(n.value)
        self._check(self.lib.lvc_peer_export(self.h, buf, n.value, C.byref(n)))
        return buf.raw[:n.value]

    def peer_attach(self, rank: int, blobs) -> None:
        """map the other ranks' tables (blobs[r] = rank r's peer_export(); blobs[rank] is ignored): from now on the
        deposit kernels reduce into the owner's tables over NVLink and this handle genotypes its own position slice"""
        n = len(blobs)
        keep = [C.create_string_buffer(b, len(b)) if b is not None else None for b in blobs]
        ptrs = (C.c_void_p * n)(*[C.cast(k, C.c_void_p) if k is not None else None for k in keep])
        lens = (C.c_size_t * n)(*[len(b) if b is not None else 0 for b in blobs])
        self._check(self.lib.lvc_peer_attach(self.h, int(rank), n, ptrs, lens))

    def peer_detach(self) -> None:
        self._check(self.lib.lvc_peer_detach(self.h))

    def stream_barrier(self, comm: "NcclComm") -> None:
        """stream-ordered barrier over the ranks of `comm` (lvc_stream_barrier)"""
        self._check(self.lib.lvc_stream_barrier(self.h, comm.c))

    def position_slice(self, n_ranks: int, rank: int):
        p0, p1 = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.lvc_position_slice(self.h, int(n_ranks), int(rank), C.byref(p0), C.byref(p1)))
        return int(p0.value), int(p1.value)

    def set_genotype_range(self, p0: int, p1: int):
        self._check(self.lib.lvc_set_genotype_range(self.h, int(p0), int(p1)))

    def copy_dense(self):
        depth = np.zeros(self.G, dtype=np.uint32)
        ad = np.zeros((self.G, 4), dtype=np.uint32)
        lik = np.zeros((self.G, 4), dtype=np.float64)
        self._check(self.lib.lvc_copy_dense(self.h, depth.ctypes.data, ad.ctypes.data, lik.ctypes.data))
        return depth, ad, lik

    def consensus(self, min_depth: int, threshold: float, depths=(), p0: int = 0, p1: int = -1):
        """lvc_consensus over [p0, p1) (p1 < 0: the whole contig): (consensus letters, statistics).  The statistics dict
        holds the counters of lvc_consensus_stats and `depth_ge`, a list aligned with `depths`."""
        if int(min_depth) < 0:
            raise ValueError(f"min_depth must be >= 0, not {min_depth}")
        thr = np.asarray(depths, dtype=np.int64).reshape(-1)
        if thr.size and (thr.min() < 0 or thr.max() > 0xFFFFFFFF):
            raise ValueError(f"depth thresholds must be in [0, 2^32): {list(depths)}")
        thr = thr.astype(np.uint32)
        n = self.G if p1 < 0 else max(int(p1) - int(p0), 0)
        seq = np.zeros(max(n, 1), dtype=np.uint8)
        st = ConsensusStats()
        self._check(self.lib.lvc_consensus(self.h, int(p0), int(p1), int(min_depth), float(threshold),
                                           thr.ctypes.data if thr.size else None, int(thr.size), seq.ctypes.data,
                                           C.byref(st)))
        out = {name: int(getattr(st, name)) for name in CONSENSUS_COUNTERS}
        out["depth_ge"] = [int(st.depth_ge[i]) for i in range(min(thr.size, 8))]
        return seq[:n].tobytes(), out

    # ---- insertions in the consensus
    def enable_insertions(self, max_keys: int = 1 << 20):
        """lvc_enable_insertions: count insertions from the next push on (only on empty tables)"""
        self._check(self.lib.lvc_enable_insertions(self.h, int(max_keys)))

    def _insertion_query(self, call) -> np.ndarray:
        cap, n = 1 << 12, C.c_uint32(0)
        while True:
            out = np.zeros(cap, dtype=INSERTION_DTYPE)
            self._check(call(out.ctypes.data, cap, C.byref(n)))
            if n.value <= cap:
                return out[:n.value]
            cap = n.value

    def copy_insertions(self) -> np.ndarray:
        """every counted key (INSERTION_DTYPE, depth 0), sorted by (pos, len, seq)"""
        return self._insertion_query(lambda out, cap, n: self.lib.lvc_copy_insertions(self.h, out, cap, n))

    def insertion_calls(self, min_depth: int, threshold: float, p0: int = 0, p1: int = -1) -> np.ndarray:
        """lvc_insertion_calls over [p0, p1) (p1 < 0: the whole contig): the called insertions, sorted by position"""
        if int(min_depth) < 0:
            raise ValueError(f"min_depth must be >= 0, not {min_depth}")
        return self._insertion_query(lambda out, cap, n: self.lib.lvc_insertion_calls(
            self.h, int(p0), int(p1), int(min_depth), float(threshold), out, cap, n))

    # ---- variant linkage
    def set_linkage_sites(self, pos, alt, max_span: int):
        """lvc_set_linkage_sites: count how the sites (pos[k], alt[k]) co-occur on reads from the next push on; clears
        the counts.  `alt`: a str or bytes of 'A' 'C' 'G' 'T' '-', one per site.  No sites turns counting off."""
        pos = np.ascontiguousarray(pos, dtype=np.int32)
        alt = np.frombuffer(alt.encode("ascii") if isinstance(alt, str) else bytes(alt), dtype=np.uint8)
        if pos.ndim != 1 or pos.size != alt.size:
            raise ValueError(f"{pos.size} positions but {alt.size} alts")
        self._check(self.lib.lvc_set_linkage_sites(self.h, pos.size, _ptr(pos), _ptr(alt), int(max_span)))

    def copy_linkage(self) -> np.ndarray:
        """lvc_copy_linkage: every pair (LINKAGE_DTYPE) in (a, b) order, zero counts included"""
        cap, n = 0, C.c_uint32(0)
        while True:
            out = np.zeros(cap, dtype=LINKAGE_DTYPE)
            self._check(self.lib.lvc_copy_linkage(self.h, _ptr(out) if cap else None, cap, C.byref(n)))
            if n.value <= cap:
                return out[:n.value]
            cap = n.value

    # ---- strand counts
    def enable_strand_counts(self):
        """lvc_enable_strand_counts: count reverse-strand pileup entries from the next push on (only on empty tables)"""
        self._check(self.lib.lvc_enable_strand_counts(self.h))

    def strand_counts(self, pos, allele):
        """lvc_strand_counts: (fwd, rev) uint32 arrays, the forward and reverse entries of allele[k] at pos[k].  `allele`:
        a str or bytes of nibble letters (=ACMGRSVTWYHKDBN, either case) or '-' for deletions, one per position."""
        pos = np.ascontiguousarray(pos, dtype=np.int32).reshape(-1)
        allele = np.frombuffer(allele.encode("ascii") if isinstance(allele, str) else bytes(allele), dtype=np.uint8)
        if pos.size != allele.size:
            raise ValueError(f"{pos.size} positions but {allele.size} alleles")
        fwd = np.zeros(pos.size, dtype=np.uint32)
        rev = np.zeros(pos.size, dtype=np.uint32)
        self._check(self.lib.lvc_strand_counts(self.h, pos.size, _ptr(pos), _ptr(allele), _ptr(fwd), _ptr(rev)))
        return fwd, rev

    # ---- tables
    def plane_keys(self) -> np.ndarray:
        n = self.lib.lvc_num_planes(self.h)
        keys = np.zeros(max(n, 1), dtype=np.uint16)
        self._check(self.lib.lvc_plane_keys(self.h, keys.ctypes.data))
        return keys[:n]

    def copy_plane(self, key: int) -> np.ndarray:
        out = np.zeros((self.G, 4), dtype=np.uint32)
        self._check(self.lib.lvc_copy_plane(self.h, int(key), out.ctypes.data))
        return out

    def import_plane(self, key: int, arr: np.ndarray, accumulate: bool = False):
        arr = np.ascontiguousarray(arr, dtype=np.uint32)
        assert arr.size == self.G * 4
        self._check(self.lib.lvc_import_plane(self.h, int(key), arr.ctypes.data, int(accumulate)))

    def ensure_plane(self, key: int):
        self._check(self.lib.lvc_ensure_plane(self.h, int(key)))

    def copy_dels(self) -> np.ndarray:
        out = np.zeros(self.G, dtype=np.uint32)
        self._check(self.lib.lvc_copy_dels(self.h, out.ctypes.data))
        return out

    def import_dels(self, arr, accumulate=False):
        arr = np.ascontiguousarray(arr, dtype=np.uint32)
        self._check(self.lib.lvc_import_dels(self.h, arr.ctypes.data, int(accumulate)))

    def copy_covdiff(self) -> np.ndarray:
        out = np.zeros(self.G + 1, dtype=np.int32)
        self._check(self.lib.lvc_copy_covdiff(self.h, out.ctypes.data))
        return out

    def import_covdiff(self, arr, accumulate=False):
        arr = np.ascontiguousarray(arr, dtype=np.int32)
        self._check(self.lib.lvc_import_covdiff(self.h, arr.ctypes.data, int(accumulate)))

    def copy_first(self, group: int) -> Optional[np.ndarray]:
        if not self.lib.lvc_first_devptr(self.h, group):
            return None
        out = np.zeros((self.G, 4), dtype=np.uint32)
        self._check(self.lib.lvc_copy_first(self.h, group, out.ctypes.data))
        return out

    def import_first(self, group: int, arr):
        arr = np.ascontiguousarray(arr, dtype=np.uint32)
        self._check(self.lib.lvc_import_first(self.h, group, arr.ctypes.data))

    @property
    def ordinal(self) -> int:
        return int(self.lib.lvc_ordinal(self.h))

    @ordinal.setter
    def ordinal(self, v: int):
        self._check(self.lib.lvc_set_ordinal(self.h, int(v)))

    @property
    def launch_count(self) -> int:
        return int(self.lib.lvc_launch_count(self.h))

    @property
    def h2d_payload_bytes(self) -> int:
        return int(self.lib.lvc_h2d_payload_bytes(self.h))

    def plane_devptr(self, key: int) -> int:
        return self.lib.lvc_plane_devptr(self.h, int(key)) or 0

    def dels_devptr(self) -> int:
        return self.lib.lvc_dels_devptr(self.h) or 0

    def covdiff_devptr(self) -> int:
        return self.lib.lvc_covdiff_devptr(self.h) or 0

    def first_devptr(self, group: int) -> int:
        return self.lib.lvc_first_devptr(self.h, group) or 0

"""ctypes binding of include/faqcs_b200.h -- the host-side mirror of the FaQCs
``trim()`` seam (FaQCs.h:245-248) in Python.

The structures below are field-for-field copies of the C header.  The binding
is prefix-parametrised (``fq_`` for the CUDA library) so that the test-only CPU
checker, which deliberately exports the same shapes under another prefix, can
be driven by the same ``Engine`` class from ``tests/``; this module itself only
ever loads ``libfaqcs_b200.so``.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

NUM_STAT = 25
NUM_QUAL = 42
NUM_BASE = 5
NUM_COMPOSITION_BIN = 10001
NUM_COMPOSITION = 6
REF_BATCH = 32768
OFFSET_AUTO = -128
NUM_STREAM = 4
OUT_R1, OUT_R2, OUT_UNPAIRED, OUT_DISCARD = range(4)
MODE_HARD, MODE_BWA, MODE_BWA_PLUS = range(3)

FILTER_STAT_NAMES = [
    "TOTAL_COUNT", "TOTAL_NUMBER", "TOTAL_LENGTH", "TOTAL_TRIMMED_NUMBER", "TOTAL_TRIMMED_LENGTH",
    "PAIRED_READ_NUMBER", "PAIRED_BASE_LENGTH", "READ_LENGTH", "BASE_LENGTH", "READ_NN", "BASE_NN",
    "READ_PHIX", "BASE_PHIX", "READ_ADAPTER", "BASE_ADAPTER", "READ_AVG_Q", "BASE_AVG_Q",
    "READ_QUAL_TRIM", "BASE_QUAL_TRIM", "READ_LOW_COMPLEXITY", "BASE_LOW_COMPLEXITY",
    "N_TO_A", "N_TO_T", "N_TO_G", "N_TO_C",
]
STAT = {n: i for i, n in enumerate(FILTER_STAT_NAMES)}

RR_VALID, RR_F_LENGTH, RR_F_NN, RR_F_AVGQ, RR_F_LOWCOMP, RR_QUAL_TRIMMED, RR_ADAPTER = (
    0x1, 0x2, 0x4, 0x8, 0x10, 0x20, 0x40)

STATUS_NAMES = {0: "FQ_OK", 1: "FQ_ERR_ARG", 2: "FQ_ERR_CUDA", 3: "FQ_ERR_NO_DEVICE", 4: "FQ_ERR_FORMAT",
                5: "FQ_ERR_QUALITY", 6: "FQ_ERR_OFFSET", 7: "FQ_ERR_BASE", 8: "FQ_ERR_STATE"}

# Built-in adapter table, in reference order (options.cpp:576-625).  Sequence data.
BUILTIN_ADAPTERS: List[Tuple[str, str]] = [
    ("cre-loxp-forward", "TCGTATAACTTCGTATAATGTATGCTATACGAAGTTATTACG"),
    ("cre-loxp-reverse", "AGCATATTGAAGCATATTACATACGATATGCTTCAATAATGC"),
    ("TruSeq-adapter-1", "GGGGTAGTGTGGATCCTCCTCTAGGCAGTTGGGTTATTCTAGAAGCAGATGTGTTGGCTGTTTCTGAAACTCTGGAAAA"),
    ("TruSeq-adapter-3", "CAACAGCCGGTCAAAACATCTGGAGGGTAAGCCATAAACACCTCAACAGAAAA"),
    ("PCR-primer-1", "CGATAACTTCGTATAATGTATGCTATACGAAGTTATTACG"),
    ("PCR-primer-2", "GCATAACTTCGTATAGCATACATTATACGAAGTTATACGA"),
    ("Nextera-primer-adapter-1", "GATCGGAAGAGCACACGTCTGAACTCCAGTCAC"),
    ("Nextera-primer-adapter-2", "GATCGGAAGAGCGTCGTGTAGGGAAAGAGTGT"),
    ("Nextera-junction-adapter-1", "CTGTCTCTTATACACATCTAGATGTGTATAAGAGACAG"),
]
POLYA_ADAPTER = ("polyA", "A" * 20)


class CAdapter(C.Structure):
    _fields_ = [("name", C.c_char_p), ("seq", C.c_char_p)]


class COptions(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("quality", C.c_int32), ("trim_5", C.c_uint32), ("trim_3", C.c_uint32),
        ("min_read_length", C.c_uint32), ("max_num_poly_N", C.c_uint32),
        ("average_quality", C.c_float), ("low_complexity_cutoff_ratio", C.c_float),
        ("adapter_mismatch_rate", C.c_float),
        ("input_quality_offset", C.c_int32), ("output_quality_offset", C.c_int32),
        ("replace_to_N_q", C.c_uint32), ("qc_only", C.c_int32), ("protect_5", C.c_int32),
        ("filter_adapter", C.c_int32), ("discard_output", C.c_int32),
        ("num_thread", C.c_uint32), ("n_adapters", C.c_uint32), ("adapters", C.POINTER(CAdapter)),
    ]


class CReadResult(C.Structure):
    _fields_ = [("offset_5", C.c_uint32), ("length", C.c_uint32), ("flags", C.c_uint16),
                ("adapter", C.c_int16), ("avg_q", C.c_float)]


READ_RESULT_DTYPE = np.dtype([("offset_5", "<u4"), ("length", "<u4"), ("flags", "<u2"),
                              ("adapter", "<i2"), ("avg_q", "<f4")])


class CBatchOut(C.Structure):
    _fields_ = [
        ("data", C.POINTER(C.c_uint8) * NUM_STREAM), ("bytes", C.c_uint64 * NUM_STREAM),
        ("n_records", C.c_uint64), ("n_valid", C.c_uint64 * 2),
        ("paired_read_number", C.c_uint64), ("paired_base_length", C.c_uint64),
        ("results", C.POINTER(CReadResult) * 2),
        ("pieces", C.c_void_p * NUM_STREAM), ("n_pieces", C.c_uint64 * NUM_STREAM), ("literal_bytes", C.c_uint64 * NUM_STREAM),
    ]


PIECE_DTYPE = np.dtype([("offset", "<u8"), ("length", "<u4"), ("source", "<u4")])


U64P = C.POINTER(C.c_uint64)


class CKmerView(C.Structure):
    _fields_ = [("n_rarefaction", C.c_uint32), ("rarefaction", C.c_void_p),
                ("n_frequency", C.c_uint64), ("frequency", C.POINTER(C.c_uint64))]


class CDupView(C.Structure):
    _fields_ = [("units", C.c_uint64), ("distinct", C.c_uint64), ("n_levels", C.c_uint64), ("levels", C.POINTER(C.c_uint64))]


class COverlapView(C.Structure):
    _fields_ = [("pairs", C.c_uint64), ("too_short", C.c_uint64), ("overlapped", C.c_uint64), ("r1_adapter", C.c_uint64),
                ("r2_adapter", C.c_uint64), ("overlap_bases", C.c_uint64), ("mismatch_bases", C.c_uint64),
                ("n_insert", C.c_uint32), ("insert_hist", C.POINTER(C.c_uint64)),
                ("n_cycles", C.c_uint32), ("r1_overlap", C.POINTER(C.c_uint64)), ("r1_mismatch", C.POINTER(C.c_uint64)),
                ("r2_overlap", C.POINTER(C.c_uint64)), ("r2_mismatch", C.POINTER(C.c_uint64))]


class COverrepSeq(C.Structure):
    _fields_ = [("count", C.c_uint64), ("mate", C.c_uint32), ("len", C.c_uint32), ("offset", C.c_uint64)]


class COverrepView(C.Structure):
    _fields_ = [("prefix_len", C.c_uint32), ("min_ppm", C.c_uint32), ("reads", C.c_uint64 * 2), ("min_count", C.c_uint64 * 2),
                ("n_seqs", C.c_uint64), ("seqs", C.POINTER(COverrepSeq)), ("bytes", C.POINTER(C.c_uint8))]


class CTileQualView(C.Structure):
    _fields_ = [("n_mates", C.c_uint32), ("overflow", C.c_uint32), ("n_tiles", C.c_uint32), ("cycles", C.c_uint32),
                ("reads", C.c_uint64 * 2), ("untiled", C.c_uint64 * 2),
                ("lane", C.POINTER(C.c_uint32)), ("tile", C.POINTER(C.c_uint32)),
                ("tile_reads", C.POINTER(C.c_uint64)), ("tile_bases", C.POINTER(C.c_uint64)), ("tile_qsum", C.POINTER(C.c_uint64)),
                ("cycle_bases", C.POINTER(C.c_uint64)), ("cycle_qsum", C.POINTER(C.c_uint64))]


OVERLAP_SCALARS = ("pairs", "too_short", "overlapped", "r1_adapter", "r2_adapter", "overlap_bases", "mismatch_bases")
OVERLAP_CYCLE_ARRAYS = ("r1_overlap", "r1_mismatch", "r2_overlap", "r2_mismatch")


class CStatsView(C.Structure):
    _fields_ = [
        ("filter_stats", C.c_uint64 * NUM_STAT), ("n_adapters", C.c_uint32),
        ("adapter_reads", U64P), ("adapter_bases", U64P),
        ("pre_rows", C.c_uint32), ("post_rows", C.c_uint32),
        ("pre_len_size", C.c_uint32), ("post_len_size", C.c_uint32),
        ("pre_quality_matrix", U64P), ("post_quality_matrix", U64P),
        ("pre_base_matrix", U64P), ("post_base_matrix", U64P),
        ("pre_read_quality_hist", U64P), ("pre_base_quality_hist", U64P),
        ("post_read_quality_hist", U64P), ("post_base_quality_hist", U64P),
        ("pre_composition", U64P), ("post_composition", U64P),
        ("pre_length_hist", U64P), ("post_length_hist", U64P),
    ]


@dataclass
class Options:
    """Python view of the fields of ``struct Options`` (FaQCs.h:77-144) that ``trim()`` reads.
    Defaults are the reference's (options.cpp:98-133)."""
    mode: int = MODE_BWA_PLUS
    quality: int = 5
    trim_5: int = 0
    trim_3: int = 0
    min_read_length: int = 50
    max_num_poly_N: int = 2
    average_quality: float = 0.0
    low_complexity_cutoff_ratio: float = 0.85
    adapter_mismatch_rate: float = 0.2
    input_quality_offset: int = OFFSET_AUTO
    output_quality_offset: int = 33
    replace_to_N_q: int = 0
    qc_only: bool = False
    protect_5: bool = False
    filter_adapter: bool = False
    discard_output: bool = False
    num_thread: int = 0
    adapters: List[Tuple[str, str]] = field(default_factory=list)

    def to_c(self):
        n = len(self.adapters)
        arr = (CAdapter * max(n, 1))()
        keep = []
        for i, (name, seq) in enumerate(self.adapters):
            bn, bs = name.encode(), seq.encode()
            keep += [bn, bs]
            arr[i].name, arr[i].seq = bn, bs
        c = COptions(self.mode, self.quality, self.trim_5, self.trim_3, self.min_read_length,
                     self.max_num_poly_N, self.average_quality, self.low_complexity_cutoff_ratio,
                     self.adapter_mismatch_rate, self.input_quality_offset, self.output_quality_offset,
                     self.replace_to_N_q, int(self.qc_only), int(self.protect_5), int(self.filter_adapter),
                     int(self.discard_output), self.num_thread, n, arr)
        return c, (arr, keep)


@dataclass
class BatchResult:
    streams: List[bytes]
    stream_bytes: List[int]
    n_records: int
    n_valid: Tuple[int, int]
    paired_read_number: int
    paired_base_length: int
    results: List[Optional[np.ndarray]]
    pieces: Optional[List[np.ndarray]] = None          # pieces mode: per stream, array of PIECE_DTYPE; `streams` then hold the literal bytes

    def expand(self, r1, r2=None) -> List[bytes]:
        """Pieces mode: materialise the four streams from the caller's inputs, the literal bytes and the piece lists."""
        if self.pieces is None:
            return self.streams
        src = [np.frombuffer(r1, np.uint8) if isinstance(r1, (bytes, bytearray)) else np.asarray(r1, np.uint8),
               None if r2 is None else (np.frombuffer(r2, np.uint8) if isinstance(r2, (bytes, bytearray)) else np.asarray(r2, np.uint8))]
        out = []
        for s in range(NUM_STREAM):
            lit = np.frombuffer(self.streams[s], np.uint8)
            parts = []
            for off, ln, which in self.pieces[s]:
                buf = lit if which == 2 else src[int(which)]
                parts.append(buf[int(off):int(off) + int(ln)])
            out.append(np.concatenate(parts).tobytes() if parts else b"")
            assert len(out[-1]) == self.stream_bytes[s], (s, len(out[-1]), self.stream_bytes[s])
        return out


@dataclass
class Stats:
    filter_stats: np.ndarray
    adapter_reads: np.ndarray
    adapter_bases: np.ndarray
    pre_quality_matrix: np.ndarray
    post_quality_matrix: np.ndarray
    pre_base_matrix: np.ndarray
    post_base_matrix: np.ndarray
    pre_read_quality_hist: np.ndarray
    pre_base_quality_hist: np.ndarray
    post_read_quality_hist: np.ndarray
    post_base_quality_hist: np.ndarray
    pre_composition: np.ndarray
    post_composition: np.ndarray
    pre_length_hist: np.ndarray
    post_length_hist: np.ndarray

    FIELDS = ("filter_stats", "adapter_reads", "adapter_bases", "pre_quality_matrix", "post_quality_matrix",
              "pre_base_matrix", "post_base_matrix", "pre_read_quality_hist", "pre_base_quality_hist",
              "post_read_quality_hist", "post_base_quality_hist", "pre_composition", "post_composition",
              "pre_length_hist", "post_length_hist")

    def diff(self, other: "Stats") -> List[str]:
        out = []
        for f in self.FIELDS:
            a, b = getattr(self, f), getattr(other, f)
            if a.shape != b.shape:
                out.append(f"{f}: shape {a.shape} != {b.shape}")
            elif not np.array_equal(a, b):
                idx = np.argwhere(a != b)
                out.append(f"{f}: {len(idx)} cells differ, first {tuple(idx[0])}: {a[tuple(idx[0])]} != {b[tuple(idx[0])]}")
        return out


class FaqcsError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {message}")
        self.status = status
        self.message = message


def _np_from(ptr, n, dtype=np.uint64):
    if n == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).copy()


def default_library_path() -> str:
    """In-tree build output; FAQCS_B200_LIB selects another build of the same library (kernel tuning variants)."""
    return os.environ.get("FAQCS_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libfaqcs_b200.so")


def load_library(path: Optional[str] = None) -> C.CDLL:
    """Load the CUDA C-ABI library.  Fails loudly if it has not been built: there is no fallback."""
    path = path or default_library_path()
    if not os.path.exists(path):
        raise FileNotFoundError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  faqcs_b200 has no CPU fallback.")
    return C.CDLL(path)


class Engine:
    """One context of the C ABI (``fq_ctx``) -- the stand-in for the accumulators
    ``main`` owns (filter_stats, adaptor_stats, PlotInfo; FaQCs.cpp:67-69) plus the
    ``trim()`` + routing loop applied batch by batch."""

    def __init__(self, options: Options, device: int = 0, lib: Optional[C.CDLL] = None, prefix: str = "fq_"):
        self.lib = lib if lib is not None else load_library()
        self.p = prefix
        self._bind()
        self.options = options
        copt, self._keep = options.to_c()
        self.ctx = C.c_void_p()
        if prefix == "fq_":
            st = self._f("create")(C.byref(copt), C.c_int(device), C.byref(self.ctx))
        else:
            st = self._f("create")(C.byref(copt), C.byref(self.ctx))
        if st != 0:
            raise FaqcsError(st, self._f("last_error")(None).decode(errors="replace"))

    def _f(self, name):
        return getattr(self.lib, self.p + name)

    def _bind(self):
        L = self.lib
        p = self.p
        getattr(L, p + "last_error").restype = C.c_char_p
        getattr(L, p + "last_error").argtypes = [C.c_void_p]
        getattr(L, p + "destroy").argtypes = [C.c_void_p]
        getattr(L, p + "destroy").restype = None
        getattr(L, p + "set_debug_results").argtypes = [C.c_void_p, C.c_int]
        getattr(L, p + "set_quality").argtypes = [C.c_void_p, C.c_int32]
        getattr(L, p + "autodetect").argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                 C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
        getattr(L, p + "process_host").argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                   C.c_uint64, C.c_int, C.POINTER(CBatchOut)]
        getattr(L, p + "stats").argtypes = [C.c_void_p, C.POINTER(CStatsView)]
        getattr(L, p + "kmer_enable").argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint32]
        getattr(L, p + "kmer_end_pass").argtypes = [C.c_void_p]
        getattr(L, p + "kmer_results").argtypes = [C.c_void_p, C.POINTER(CKmerView)]
        if p == "fq_":
            L.fq_process_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                            C.c_uint64, C.c_int, C.c_int, C.POINTER(CBatchOut)]
            L.fq_last_timing.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_int]
            L.fq_launch_count.argtypes = [C.c_void_p]
            L.fq_launch_count.restype = C.c_uint64
            L.fq_stream.argtypes = [C.c_void_p]
            L.fq_stream.restype = C.c_void_p
            L.fq_stats_device_buffer.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t),
                                                 C.POINTER(C.c_void_p)]
            L.fq_submit_host.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint64, C.c_int,
                                         C.POINTER(C.c_uint64)]
            L.fq_run.argtypes = [C.c_void_p, C.c_uint64]
            L.fq_wait.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(CBatchOut)]
            L.fq_stats_reserve_rows.argtypes = [C.c_void_p, C.c_uint32]
            L.fq_set_check_pair_ids.argtypes = [C.c_void_p, C.c_int]
            L.fq_set_output_pieces.argtypes = [C.c_void_p, C.c_int]
            L.fq_host_alloc.argtypes = [C.c_size_t]
            L.fq_host_alloc.restype = C.c_void_p
            L.fq_host_free.argtypes = [C.c_void_p]
            L.fq_host_free.restype = None
            L.fq_reset_stats.argtypes = [C.c_void_p]
            L.fq_comm_unique_id.argtypes = [C.c_void_p]
            L.fq_comm_init_rank.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
            L.fq_comm_init_all.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
            L.fq_comm_destroy.argtypes = [C.c_void_p]
            L.fq_comm_destroy.restype = None
            L.fq_allreduce_stats.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
            L.fq_merge_stats.argtypes = [C.c_void_p, C.c_void_p]
            L.fq_kmer_end_pass_all.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
            L.fq_dup_enable.argtypes = [C.c_void_p]
            L.fq_dup_end_pass_all.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
            L.fq_dup_results.argtypes = [C.c_void_p, C.POINTER(CDupView)]
            L.fq_overlap_enable.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]
            L.fq_overlap_end_pass_all.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
            L.fq_overlap_results.argtypes = [C.c_void_p, C.POINTER(COverlapView)]
            L.fq_overrep_enable.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
            L.fq_overrep_end_pass_all.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
            L.fq_overrep_results.argtypes = [C.c_void_p, C.POINTER(COverrepView)]
            L.fq_tile_qual_enable.argtypes = [C.c_void_p]
            L.fq_tile_qual_end_pass_all.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.POINTER(C.c_void_p)]
            L.fq_tile_qual_results.argtypes = [C.c_void_p, C.POINTER(CTileQualView)]
            L.fq_last_allreduce_ms.argtypes = [C.c_void_p]
            L.fq_last_allreduce_ms.restype = C.c_float
            L.fq_device_outputs.argtypes = [C.c_void_p, C.POINTER(C.c_void_p * NUM_STREAM)]
            L.fq_build_info.restype = C.c_char_p

    def _check(self, st):
        if st != 0:
            raise FaqcsError(st, self._f("last_error")(self.ctx).decode(errors="replace"))

    def close(self):
        if getattr(self, "ctx", None) is not None and self.ctx:
            self._f("destroy")(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- API -------------------------------------------------------------
    def set_debug_results(self, enable: bool = True):
        self._check(self._f("set_debug_results")(self.ctx, int(enable)))

    def set_output_pieces(self, enable: bool = True):
        """Pieces mode (fq_set_output_pieces): streams come back as lists of pieces of the caller's input + literal bytes."""
        self._check(self.lib.fq_set_output_pieces(self.ctx, int(enable)))
        self._pieces = bool(enable)

    def merge_stats_from(self, other: "Engine"):
        """fq_merge_stats: add another context's accumulators (same device) into this one and zero them there."""
        self._check(self.lib.fq_merge_stats(self.ctx, other.ctx))

    def kmer_enable(self, k: int = 31, split_size: int = 1000000, num_subsample: int = 10):
        """--kmer_rarefaction: k = Options::kmer (-m), Options::split_size, Options::num_subsample (--subset, already
        doubled where options.cpp:506-523 doubles it).  Batches must then be multiples of 32768 records."""
        self._check(self._f("kmer_enable")(self.ctx, int(k), int(split_size), int(num_subsample)))

    def kmer_end_pass(self):
        """End of one input (the paired files, then the unpaired file): FaQCs.cpp:518-537 / 737-756."""
        self._check(self._f("kmer_end_pass")(self.ctx))

    def kmer_results(self):
        """(rarefaction [n,3] uint64 = num_seq, distinct, total; frequency [m,2] uint64 = count, k-mers), plot.cpp:683-733."""
        v = CKmerView()
        self._check(self._f("kmer_results")(self.ctx, C.byref(v)))
        rare = np.zeros((v.n_rarefaction, 3), np.uint64)
        if v.n_rarefaction:
            rare[:] = np.ctypeslib.as_array(C.cast(v.rarefaction, C.POINTER(C.c_uint64)), (v.n_rarefaction, 3))
        freq = np.zeros((v.n_frequency, 2), np.uint64)
        if v.n_frequency:
            freq[:] = np.ctypeslib.as_array(v.frequency, (v.n_frequency, 2))
        return rare, freq

    def dup_enable(self):
        """Sequence duplication statistics (fq_dup_enable): every read (single-end) or pair of the following batches is counted
        by the bytes of its sequence line(s) as framed.  Call before the first batch of a pass."""
        self._check(self.lib.fq_dup_enable(self.ctx))

    def dup_end_pass(self):
        """End of one input's pass on this context alone (fq_dup_end_pass_all with n = 1); dist_stats has the sharded forms."""
        ctxs = (C.c_void_p * 1)(self.ctx)
        self._check(self.lib.fq_dup_end_pass_all(ctxs, 1, None))

    def dup_results(self) -> dict:
        """The last finished pass: {"units", "distinct", "levels": [m, 2] uint64 = (multiplicity, distinct keys), ascending}."""
        v = CDupView()
        self._check(self.lib.fq_dup_results(self.ctx, C.byref(v)))
        levels = np.zeros((v.n_levels, 2), np.uint64)
        if v.n_levels:
            levels[:] = np.ctypeslib.as_array(v.levels, (v.n_levels, 2))
        return {"units": int(v.units), "distinct": int(v.distinct), "levels": levels}

    def overlap_enable(self, min_overlap: int = 30, diff_limit: int = 5, diff_percent: int = 20):
        """Insert size and overlap error profile (fq_overlap_enable): every pair of the following paired batches is searched for
        the overlap of R1 with reverse-complemented R2.  Call before the first batch of a pass."""
        self._check(self.lib.fq_overlap_enable(self.ctx, int(min_overlap), int(diff_limit), int(diff_percent)))

    def overlap_end_pass(self):
        """End of one input's pass on this context alone (fq_overlap_end_pass_all with n = 1); dist_stats has the other forms."""
        ctxs = (C.c_void_p * 1)(self.ctx)
        self._check(self.lib.fq_overlap_end_pass_all(ctxs, 1, None))

    def overlap_results(self) -> dict:
        """The last finished pass: the scalars of OVERLAP_SCALARS as ints, "insert_hist" (index = insert size) and the four
        OVERLAP_CYCLE_ARRAYS (index = 0-based cycle) as uint64 arrays without trailing zeros."""
        v = COverlapView()
        self._check(self.lib.fq_overlap_results(self.ctx, C.byref(v)))
        out = {k: int(getattr(v, k)) for k in OVERLAP_SCALARS}

        def arr(p, n):
            return np.ctypeslib.as_array(p, (n,)).copy() if n else np.zeros(0, np.uint64)
        out["insert_hist"] = arr(v.insert_hist, v.n_insert)
        for k in OVERLAP_CYCLE_ARRAYS:
            out[k] = arr(getattr(v, k), v.n_cycles)
        return out

    def overrep_enable(self, prefix_len: int = 50, min_ppm: int = 1000):
        """Overrepresented sequences (fq_overrep_enable): the first prefix_len bytes of every read of the following batches are
        counted, each mate on its own.  Call before the first batch of a pass."""
        self._check(self.lib.fq_overrep_enable(self.ctx, int(prefix_len), int(min_ppm)))

    def overrep_end_pass(self):
        """End of one input's pass on this context alone (fq_overrep_end_pass_all with n = 1); dist_stats has the sharded forms."""
        ctxs = (C.c_void_p * 1)(self.ctx)
        self._check(self.lib.fq_overrep_end_pass_all(ctxs, 1, None))

    def overrep_results(self) -> dict:
        """The last finished pass: {"prefix_len", "min_ppm", "reads": [mate 1, mate 2], "min_count": [mate 1, mate 2],
        "seqs": [(mate, bytes, count)] in the library's order (count descending, mate, bytes)}."""
        v = COverrepView()
        self._check(self.lib.fq_overrep_results(self.ctx, C.byref(v)))
        seqs = []
        for i in range(v.n_seqs):
            e = v.seqs[i]
            seqs.append((int(e.mate), C.string_at(C.addressof(v.bytes.contents) + e.offset, e.len), int(e.count)))
        return {"prefix_len": int(v.prefix_len), "min_ppm": int(v.min_ppm), "reads": [int(x) for x in v.reads],
                "min_count": [int(x) for x in v.min_count], "seqs": seqs}

    def tile_qual_enable(self):
        """Per flowcell tile quality (fq_tile_qual_enable): every read of the following batches is counted under the (lane,
        tile) of its header, each mate on its own.  Call before the first batch of a pass."""
        self._check(self.lib.fq_tile_qual_enable(self.ctx))

    def tile_qual_end_pass(self):
        """End of one input's pass on this context alone (fq_tile_qual_end_pass_all with n = 1); dist_stats has the other forms."""
        ctxs = (C.c_void_p * 1)(self.ctx)
        self._check(self.lib.fq_tile_qual_end_pass_all(ctxs, 1, None))

    def tile_qual_results(self) -> dict:
        """The last finished pass: ints "n_mates", "overflow", "n_tiles", "cycles"; uint64 arrays "reads" and "untiled" [2];
        uint32 arrays "lane" and "tile" [n_tiles] ascending; uint64 arrays "tile_reads", "tile_bases", "tile_qsum"
        [n_tiles, n_mates] and "cycle_bases", "cycle_qsum" [n_tiles, n_mates, cycles]."""
        v = CTileQualView()
        self._check(self.lib.fq_tile_qual_results(self.ctx, C.byref(v)))
        T, M, Cy = int(v.n_tiles), int(v.n_mates), int(v.cycles)

        def arr(p, shape, dt=np.uint64):
            n = int(np.prod(shape))
            return np.ctypeslib.as_array(p, (n,)).copy().reshape(shape) if n else np.zeros(shape, dt)
        out = {"n_mates": M, "overflow": int(v.overflow), "n_tiles": T, "cycles": Cy,
               "reads": np.array(list(v.reads), np.uint64), "untiled": np.array(list(v.untiled), np.uint64),
               "lane": arr(v.lane, (T,), np.uint32), "tile": arr(v.tile, (T,), np.uint32)}
        for k in ("tile_reads", "tile_bases", "tile_qsum"):
            out[k] = arr(getattr(v, k), (T, M))
        for k in ("cycle_bases", "cycle_qsum"):
            out[k] = arr(getattr(v, k), (T, M, Cy))
        return out

    def set_quality(self, quality: int):
        """Options::quality for the following batches (the reference's NextSeq adjustment, FaQCs.cpp:272-277)."""
        self._check(self._f("set_quality")(self.ctx, int(quality)))

    @staticmethod
    def _buf(b):
        if b is None:
            return None, 0, None
        if isinstance(b, (bytes, bytearray)):
            a = np.frombuffer(b, dtype=np.uint8)
        else:
            a = np.ascontiguousarray(b, dtype=np.uint8)
        return C.c_void_p(a.ctypes.data) if a.size else C.c_void_p(0), a.size, a

    def autodetect(self, r1, r2=None) -> Tuple[int, int]:
        p1, n1, k1 = self._buf(r1)
        p2, n2, k2 = self._buf(r2)
        off, q = C.c_int32(), C.c_int32()
        self._check(self._f("autodetect")(self.ctx, p1, n1, p2, n2, C.byref(off), C.byref(q)))
        return off.value, q.value

    def _collect(self, out: CBatchOut, paired: bool, want_data: bool = True) -> BatchResult:
        streams = []
        pieces = None
        in_pieces = any(int(out.n_pieces[s]) for s in range(NUM_STREAM))
        if in_pieces and want_data:
            pieces = []
            for s in range(NUM_STREAM):
                k = int(out.n_pieces[s])
                raw = C.string_at(out.pieces[s], k * PIECE_DTYPE.itemsize) if k else b""
                pieces.append(np.frombuffer(raw, dtype=PIECE_DTYPE).copy())
        for s in range(NUM_STREAM):
            n = int(out.literal_bytes[s]) if in_pieces else int(out.bytes[s])
            streams.append(C.string_at(out.data[s], n) if (n and want_data and out.data[s]) else b"")
        results: List[Optional[np.ndarray]] = [None, None]
        for m in range(2 if paired else 1):
            if out.results[m]:
                raw = C.string_at(out.results[m], int(out.n_records) * C.sizeof(CReadResult))
                results[m] = np.frombuffer(raw, dtype=READ_RESULT_DTYPE).copy()
        return BatchResult(streams, [int(out.bytes[s]) for s in range(NUM_STREAM)], int(out.n_records), (int(out.n_valid[0]), int(out.n_valid[1])),
                           int(out.paired_read_number), int(out.paired_base_length), results, pieces)

    def process(self, r1, r2=None, first_record_index: int = 0, is_final: bool = True) -> BatchResult:
        """Host buffers in, host buffers out (fq_process_host)."""
        p1, n1, k1 = self._buf(r1)
        p2, n2, k2 = self._buf(r2)
        out = CBatchOut()
        self._check(self._f("process_host")(self.ctx, p1, n1, p2, n2, first_record_index, int(is_final),
                                            C.byref(out)))
        return self._collect(out, r2 is not None)

    def process_device(self, d_r1: int, n1: int, d_r2: Optional[int] = None, n2: int = 0,
                       first_record_index: int = 0, is_final: bool = True, copy_out: bool = False) -> BatchResult:
        """Device pointers in (fq_process_device); outputs stay in HBM unless copy_out."""
        out = CBatchOut()
        self._check(self.lib.fq_process_device(self.ctx, C.c_void_p(d_r1), n1,
                                               C.c_void_p(d_r2) if d_r2 else None, n2,
                                               first_record_index, int(is_final), int(copy_out), C.byref(out)))
        return self._collect(out, d_r2 is not None, want_data=copy_out)

    # ---- pipelined host path (submit -> run -> wait) ---------------------------------------------
    def submit(self, r1, r2=None, first_record_index: int = 0, is_final: bool = True) -> int:
        p1, n1, k1 = self._buf(r1)
        p2, n2, k2 = self._buf(r2)
        t = C.c_uint64()
        self._check(self.lib.fq_submit_host(self.ctx, p1, n1, p2, n2, first_record_index, int(is_final), C.byref(t)))
        self._inflight = getattr(self, "_inflight", {})
        self._inflight[t.value] = (k1, k2, r2 is not None)       # keep the host buffers alive until run()
        return t.value

    def run(self, ticket: int):
        self._check(self.lib.fq_run(self.ctx, ticket))

    def wait(self, ticket: int, want_data: bool = True) -> BatchResult:
        out = CBatchOut()
        self._check(self.lib.fq_wait(self.ctx, ticket, C.byref(out)))
        _, _, paired = self._inflight.pop(ticket)
        return self._collect(out, paired, want_data=want_data)

    def last_timing(self) -> dict:
        """Device ms of the last batch by segment (CUDA events on the context's stream)."""
        ms = (C.c_float * 5)()
        self._check(self.lib.fq_last_timing(self.ctx, ms, 5))
        return dict(zip(("all", "frame", "adapter", "trim", "emit"), [float(x) for x in ms]))

    def host_alloc(self, nbytes: int) -> np.ndarray:
        """Pinned host buffer (fq_host_alloc) viewed as a uint8 array; free with host_free."""
        p = self.lib.fq_host_alloc(nbytes)
        if not p:
            raise MemoryError("fq_host_alloc failed")
        arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(nbytes,))
        return arr

    def host_free(self, arr: np.ndarray):
        self.lib.fq_host_free(C.c_void_p(arr.ctypes.data))

    def launch_count(self) -> int:
        return int(self.lib.fq_launch_count(self.ctx))

    def stream(self) -> int:
        return int(self.lib.fq_stream(self.ctx) or 0)

    def stats_device_buffer(self) -> Tuple[int, int, int]:
        d, n, r = C.c_void_p(), C.c_size_t(), C.c_void_p()
        self._check(self.lib.fq_stats_device_buffer(self.ctx, C.byref(d), C.byref(n), C.byref(r)))
        return int(d.value), int(n.value), int(r.value)

    def stats_reserve_rows(self, rows: int):
        self._check(self.lib.fq_stats_reserve_rows(self.ctx, rows))

    def reset_stats(self):
        self._check(self.lib.fq_reset_stats(self.ctx))

    def stats(self) -> Stats:
        v = CStatsView()
        self._check(self._f("stats")(self.ctx, C.byref(v)))
        na = v.n_adapters
        return Stats(
            filter_stats=np.array(list(v.filter_stats), dtype=np.uint64),
            adapter_reads=_np_from(v.adapter_reads, na), adapter_bases=_np_from(v.adapter_bases, na),
            pre_quality_matrix=_np_from(v.pre_quality_matrix, v.pre_rows * NUM_QUAL).reshape(-1, NUM_QUAL),
            post_quality_matrix=_np_from(v.post_quality_matrix, v.post_rows * NUM_QUAL).reshape(-1, NUM_QUAL),
            pre_base_matrix=_np_from(v.pre_base_matrix, v.pre_rows * NUM_BASE).reshape(-1, NUM_BASE),
            post_base_matrix=_np_from(v.post_base_matrix, v.post_rows * NUM_BASE).reshape(-1, NUM_BASE),
            pre_read_quality_hist=_np_from(v.pre_read_quality_hist, NUM_QUAL),
            pre_base_quality_hist=_np_from(v.pre_base_quality_hist, NUM_QUAL),
            post_read_quality_hist=_np_from(v.post_read_quality_hist, NUM_QUAL),
            post_base_quality_hist=_np_from(v.post_base_quality_hist, NUM_QUAL),
            pre_composition=_np_from(v.pre_composition, NUM_COMPOSITION * NUM_COMPOSITION_BIN).reshape(
                NUM_COMPOSITION, NUM_COMPOSITION_BIN),
            post_composition=_np_from(v.post_composition, NUM_COMPOSITION * NUM_COMPOSITION_BIN).reshape(
                NUM_COMPOSITION, NUM_COMPOSITION_BIN),
            pre_length_hist=_np_from(v.pre_length_hist, v.pre_len_size),
            post_length_hist=_np_from(v.post_length_hist, v.post_len_size),
        )

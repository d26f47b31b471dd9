"""ctypes bindings of the two in-tree shared libraries.

  libraxtax_b200.so  device C ABI   (include/raxtax_b200.h)   -> class Context
  libraxtax_host.so  host   C ABI   (include/raxtax_host.h)   -> classes Tree, Queries, function raxtax()

There is no fallback path: if the CUDA extension is missing this module raises at load time, and without a
GPU `Context()` raises RtxError(RTX_ERR_NO_DEVICE).
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

from . import _build

u8p, u16p, u32p, u64p, f64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint16, C.c_uint32, C.c_uint64, C.c_double))

RTX_OK, RTX_ERR_INVALID, RTX_ERR_CUDA, RTX_ERR_NO_DEVICE, RTX_ERR_NO_INDEX, RTX_ERR_UNSUPPORTED, RTX_ERR_ASSERT = 0, -1, -2, -3, -4, -5, -6
RTX_SKIP_EXACT_MATCHES, RTX_RAW_CONFIDENCE, RTX_BOTH_STRANDS = 1, 2, 4
RTX_HITCOUNT_BITROWS, RTX_HITCOUNT_CSR = 0, 1
RTX_OPT_HITCOUNT_VARIANT, RTX_OPT_SUB_BATCH, RTX_OPT_KEEP_CSR, RTX_OPT_PROFILE, RTX_OPT_HITCOUNT_MAX_TILES = 1, 2, 3, 4, 6
RTX_OPT_HITCOUNT_GROUP, RTX_OPT_WALK_VARIANT, RTX_OPT_WALK_LOG_CAP, RTX_OPT_PIPELINE, RTX_OPT_BEST_HITS = 7, 9, 10, 11, 12
KERNEL_NAMES = ["kmers", "hitcount", "fixup", "prob", "index", "walk", "prefix", "allreduce", "allgather", "shard", "gather"]

# every symbol include/raxtax_b200.h declares
DEVICE_SYMBOLS = [
    "rtx_abi_version", "rtx_ctx_create", "rtx_ctx_destroy", "rtx_last_error", "rtx_ctx_set_option", "rtx_ctx_stream", "rtx_ctx_device",
    "rtx_ctx_synchronize", "rtx_host_alloc", "rtx_host_free", "rtx_index_upload", "rtx_index_n_refs", "rtx_index_shard_refs", "rtx_index_max_levels", "rtx_batch_sub_batch",
    "rtx_index_device_bytes", "rtx_index_bitrow_bytes", "rtx_hitcount_kernel_name", "rtx_classify_batch", "rtx_batch_upload", "rtx_batch_run", "rtx_batch_download", "rtx_batch_slot",
    "rtx_batch_strands", "rtx_batch_best_hits",
    "rtx_shard_phase1", "rtx_shard_hist_buffer", "rtx_shard_phase2", "rtx_shard_records_buffers", "rtx_shard_phase3", "rtx_shard_exchange_hist_local", "rtx_shard_exchange_records_local",
    "rtx_comm_unique_id", "rtx_comm_init", "rtx_comm_destroy", "rtx_shard_run", "rtx_shard_gather", "rtx_shard_classify",
    "rtx_profile_reset", "rtx_profile_get",
]
# every symbol include/raxtax_host.h declares
HOST_SYMBOLS = [
    "rxh_last_error", "rxh_tree_from_fasta", "rxh_tree_from_file", "rxh_queries_from_file", "rxh_tree_from_bin", "rxh_tree_save_bin", "rxh_queries_skip", "rxh_tree_new", "rxh_tree_free", "rxh_tree_num_tips", "rxh_tree_lineage",
    "rxh_tree_csr", "rxh_tree_build_kmer_map", "rxh_tree_has_kmer_map", "rxh_tree_exact", "rxh_tree_index_desc", "rxh_tree_upload", "rxh_tree_upload_sharded", "rxh_queries_from_fasta", "rxh_queries_new",
    "rxh_queries_free", "rxh_queries_len", "rxh_queries_label", "rxh_queries_arrays", "rxh_raxtax", "rxh_raxtax_multi", "rxh_raxtax_both_strands", "rxh_raxtax_best_hits", "rxh_raxtax_sharded", "rxh_merge_shard_results", "rxh_exact_batch", "rxh_count_sender", "rxh_count_logger", "rxh_format_fixed", "rxh_release_buffers", "rxh_plan_chunks",
]


class IndexDesc(C.Structure):
    _fields_ = [("n_refs", C.c_uint64), ("csr_offsets", u64p), ("csr_ids", u32p), ("n_nodes", C.c_uint32), ("node_lo", u32p),
                ("node_hi", u32p), ("node_type", u8p), ("child_first", u32p), ("child_count", u32p), ("ref_levels", u8p),
                ("ref_shard_begin", C.c_uint64), ("ref_shard_end", C.c_uint64), ("n_shards", C.c_uint32), ("shard_rank", C.c_uint32),
                ("shard_cuts", u64p), ("ref_seq_offsets", u64p), ("ref_seq_codes", u8p)]


class Batch(C.Structure):
    _fields_ = [("n_queries", C.c_uint32), ("seq_offsets", u64p), ("seq_codes", u8p), ("exact_offsets", u32p),
                ("exact_ids", u32p), ("flags", C.c_uint32)]


class ResultsStruct(C.Structure):
    _fields_ = [("n_kmers", u16p), ("result_begin", u32p), ("global_signal", f64p), ("result_capacity", C.c_uint64),
                ("first_ref", u32p), ("n_levels", u8p), ("confidence", f64p), ("local_signal", f64p), ("n_results", C.c_uint64),
                ("tap_counts", u16p), ("tap_hist", u32p), ("tap_hist_stride", C.c_uint64), ("tap_kmers", u16p),
                ("tap_kmer_stride", C.c_uint64), ("tap_probs", f64p), ("tap_prob_stride", C.c_uint64)]


class KernelStat(C.Structure):
    _fields_ = [("launches", C.c_uint64), ("total_ms", C.c_double)]


class Profile(C.Structure):
    _fields_ = [("kernel", KernelStat * 11), ("queries", C.c_uint64), ("hits", C.c_uint64), ("bitrow_bytes", C.c_uint64),
                ("csr_equiv_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("allreduce_bytes", C.c_uint64),
                ("allgather_bytes", C.c_uint64), ("gather_bytes", C.c_uint64)]


SENDER = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_char_p, C.c_char_p, C.c_char_p)
LOGGER = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_char_p)
HITS_SENDER = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_char_p, C.c_char_p)

_dev = None
_host = None


class RtxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rtx error {code}: {msg}")
        self.code = code
        self.msg = msg


def device_lib():
    """Load libraxtax_b200.so (building it in-tree if a source is newer).  Raises if the CUDA extension is absent."""
    global _dev
    if _dev is not None:
        return _dev
    path = _build.DEVICE_LIB
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run `python -m raxtax_b200._build` (needs nvcc); there is no fallback path")
    L = C.CDLL(path, mode=C.RTLD_GLOBAL)
    L.rtx_last_error.restype = C.c_char_p
    L.rtx_last_error.argtypes = [C.c_void_p]
    L.rtx_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.rtx_ctx_destroy.argtypes = [C.c_void_p]
    L.rtx_ctx_destroy.restype = None
    L.rtx_ctx_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int64]
    L.rtx_ctx_stream.restype = C.c_void_p
    L.rtx_ctx_stream.argtypes = [C.c_void_p]
    L.rtx_ctx_synchronize.argtypes = [C.c_void_p]
    L.rtx_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    L.rtx_host_free.argtypes = [C.c_void_p]
    L.rtx_index_upload.argtypes = [C.c_void_p, C.POINTER(IndexDesc)]
    L.rtx_hitcount_kernel_name.restype = C.c_char_p
    L.rtx_hitcount_kernel_name.argtypes = [C.c_void_p]
    for f in ("rtx_index_n_refs", "rtx_index_shard_refs", "rtx_index_device_bytes", "rtx_index_bitrow_bytes"):
        getattr(L, f).restype = C.c_uint64
        getattr(L, f).argtypes = [C.c_void_p]
    L.rtx_index_max_levels.restype = C.c_uint32
    L.rtx_index_max_levels.argtypes = [C.c_void_p]
    L.rtx_batch_sub_batch.restype = C.c_uint32
    L.rtx_batch_sub_batch.argtypes = [C.c_void_p]
    L.rtx_classify_batch.argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(ResultsStruct)]
    L.rtx_batch_upload.argtypes = [C.c_void_p, C.POINTER(Batch)]
    L.rtx_batch_run.argtypes = [C.c_void_p]
    L.rtx_batch_slot.argtypes = [C.c_void_p, C.c_int]
    L.rtx_batch_download.argtypes = [C.c_void_p, C.POINTER(ResultsStruct)]
    L.rtx_batch_strands.argtypes = [C.c_void_p, u8p]
    L.rtx_batch_best_hits.argtypes = [C.c_void_p, u32p, u32p, u16p]
    for f in ("rtx_shard_phase1", "rtx_shard_phase2", "rtx_shard_phase3", "rtx_profile_reset"):
        getattr(L, f).argtypes = [C.c_void_p]
    L.rtx_shard_hist_buffer.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.rtx_shard_records_buffers.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
    L.rtx_comm_unique_id.argtypes = [C.c_char_p]
    L.rtx_comm_init.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int]
    L.rtx_comm_destroy.argtypes = [C.c_void_p]
    L.rtx_shard_run.argtypes = [C.c_void_p]
    L.rtx_shard_gather.argtypes = [C.c_void_p, C.c_int]
    L.rtx_shard_classify.argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(ResultsStruct), C.c_int]
    L.rtx_shard_exchange_hist_local.argtypes = [C.POINTER(C.c_void_p), C.c_uint32]
    L.rtx_shard_exchange_records_local.argtypes = [C.POINTER(C.c_void_p), C.c_uint32]
    L.rtx_profile_get.argtypes = [C.c_void_p, C.POINTER(Profile)]
    _dev = L
    return L


def host_lib():
    global _host
    if _host is not None:
        return _host
    device_lib()
    path = _build.HOST_LIB
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run `python -m raxtax_b200._build`")
    L = C.CDLL(path)
    L.rxh_last_error.restype = C.c_char_p
    L.rxh_tree_from_fasta.restype = C.c_void_p
    L.rxh_tree_from_fasta.argtypes = [C.c_char_p, C.c_size_t]
    L.rxh_tree_from_file.restype = C.c_void_p
    L.rxh_tree_from_file.argtypes = [C.c_char_p, C.POINTER(C.c_int)]
    L.rxh_queries_from_file.restype = C.c_void_p
    L.rxh_queries_from_file.argtypes = [C.c_char_p]
    L.rxh_tree_from_bin.restype = C.c_void_p
    L.rxh_tree_from_bin.argtypes = [C.c_char_p, C.c_size_t]
    L.rxh_tree_save_bin.argtypes = [C.c_void_p, C.c_char_p]
    L.rxh_queries_skip.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t]
    L.rxh_tree_new.restype = C.c_void_p
    L.rxh_tree_new.argtypes = [C.c_size_t, C.c_char_p, C.c_size_t, u64p, u8p]
    L.rxh_tree_free.argtypes = [C.c_void_p]
    L.rxh_tree_free.restype = None
    L.rxh_tree_num_tips.restype = C.c_size_t
    L.rxh_tree_num_tips.argtypes = [C.c_void_p]
    L.rxh_tree_lineage.restype = C.c_char_p
    L.rxh_tree_lineage.argtypes = [C.c_void_p, C.c_size_t]
    L.rxh_tree_csr.argtypes = [C.c_void_p, C.POINTER(u64p), C.POINTER(u32p)]
    L.rxh_tree_csr.restype = None
    L.rxh_tree_build_kmer_map.argtypes = [C.c_void_p]
    L.rxh_tree_build_kmer_map.restype = None
    L.rxh_tree_has_kmer_map.argtypes = [C.c_void_p]
    L.rxh_tree_has_kmer_map.restype = C.c_int
    L.rxh_tree_exact.restype = C.c_size_t
    L.rxh_tree_exact.argtypes = [C.c_void_p, u8p, C.c_size_t, u32p, C.c_size_t]
    L.rxh_tree_index_desc.argtypes = [C.c_void_p, C.POINTER(IndexDesc)]
    L.rxh_tree_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]
    L.rxh_tree_upload_sharded.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, u64p]
    L.rxh_queries_from_fasta.restype = C.c_void_p
    L.rxh_queries_from_fasta.argtypes = [C.c_char_p, C.c_size_t]
    L.rxh_queries_new.restype = C.c_void_p
    L.rxh_queries_new.argtypes = [C.c_size_t, C.c_char_p, C.c_size_t, u64p, u8p]
    L.rxh_queries_free.argtypes = [C.c_void_p]
    L.rxh_queries_free.restype = None
    L.rxh_queries_len.restype = C.c_size_t
    L.rxh_queries_len.argtypes = [C.c_void_p]
    L.rxh_queries_label.restype = C.c_char_p
    L.rxh_queries_label.argtypes = [C.c_void_p, C.c_size_t]
    L.rxh_queries_arrays.argtypes = [C.c_void_p, C.POINTER(u64p), C.POINTER(u8p)]
    L.rxh_queries_arrays.restype = None
    L.rxh_raxtax.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, SENDER, C.c_void_p, C.c_int,
                             LOGGER, C.c_void_p, C.POINTER(C.c_int)]
    L.rxh_raxtax_multi.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, SENDER, C.c_void_p,
                                   C.c_int, LOGGER, C.c_void_p, C.POINTER(C.c_int)]
    L.rxh_raxtax_both_strands.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, SENDER,
                                          C.c_void_p, C.c_int, LOGGER, C.c_void_p, C.POINTER(C.c_int)]
    L.rxh_raxtax_best_hits.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, SENDER,
                                       C.c_void_p, C.c_int, LOGGER, C.c_void_p, C.POINTER(C.c_int), C.c_int, C.c_uint32, HITS_SENDER,
                                       C.c_void_p]
    L.rxh_raxtax_sharded.argtypes = [C.POINTER(C.c_void_p), C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, SENDER, C.c_void_p,
                                     C.c_int, LOGGER, C.c_void_p, C.POINTER(C.c_int)]
    L.rxh_merge_shard_results.argtypes = [C.c_size_t, C.c_size_t, C.c_uint32, C.POINTER(u32p), C.POINTER(u32p), C.POINTER(u8p), C.POINTER(f64p),
                                          C.POINTER(f64p), u32p, u32p, u8p, C.c_int, C.c_int, u32p, u32p, u8p, f64p, f64p, C.c_uint64,
                                          C.POINTER(C.c_uint64)]
    L.rxh_format_fixed.restype = C.c_size_t
    L.rxh_format_fixed.argtypes = [C.c_double, C.c_int, C.c_char_p, C.c_size_t]
    L.rxh_plan_chunks.restype = C.c_size_t
    L.rxh_plan_chunks.argtypes = [C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.c_size_t), C.c_size_t]
    L.rxh_exact_batch.restype = C.c_uint64
    L.rxh_exact_batch.argtypes = [C.c_void_p, C.c_size_t, u64p, u8p, u32p, u32p, C.c_uint64]
    _host = L
    return L


def _ptr(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


class HostError(RuntimeError):
    pass


def _host_err():
    return HostError(host_lib().rxh_last_error().decode(errors="replace"))


# ---------------------------------------------------------------------------------------------------------------
@dataclass
class ClassifyOutput:
    """`Vec<EvaluationResult>` per query (lineage.rs:7-14) in flat arrays, plus optional parity taps."""
    n_kmers: np.ndarray
    result_begin: np.ndarray
    global_signal: np.ndarray
    first_ref: np.ndarray
    n_levels: np.ndarray
    confidence: np.ndarray  # [n_results, max_levels]
    local_signal: np.ndarray
    counts: np.ndarray | None = None
    hist: np.ndarray | None = None
    kmers: np.ndarray | None = None
    probs: np.ndarray | None = None  # [nq, kmax + 1] normalised P(m) by count (valid where the histogram is non-zero)
    strand: np.ndarray | None = None  # both-strand batches: u8 [nq], 0 = classified as given, 1 = as its reverse complement
    # batches with best_hits = T > 0: (n_hits u32 [nq], ref u32 [nq, T], count u16 [nq, T]); row q is valid up to n_hits[q]
    best_hits: tuple | None = None

    def for_query(self, q):
        a, b = int(self.result_begin[q]), int(self.result_begin[q + 1])
        return [(int(self.first_ref[i]), self.confidence[i, : self.n_levels[i]].copy(), float(self.local_signal[i]),
                 float(self.global_signal[q])) for i in range(a, b)]


class Context:
    """One GPU's rtx_ctx."""

    def __init__(self, device: int = 0):
        L = device_lib()
        h = C.c_void_p()
        rc = L.rtx_ctx_create(device, C.byref(h))
        if rc != 0:
            raise RtxError(rc, L.rtx_last_error(None).decode())
        self._h = h
        self._pinned = []
        self._keep = []
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            for p in getattr(self, "_pinned", []):
                device_lib().rtx_host_free(p)
            self._pinned = []
            device_lib().rtx_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise RtxError(rc, device_lib().rtx_last_error(self._h).decode())

    def set_option(self, opt, value):
        self._check(device_lib().rtx_ctx_set_option(self._h, opt, int(value)))

    @property
    def stream(self) -> int:
        return device_lib().rtx_ctx_stream(self._h) or 0

    def synchronize(self):
        self._check(device_lib().rtx_ctx_synchronize(self._h))

    @property
    def n_refs(self):
        return device_lib().rtx_index_n_refs(self._h)

    @property
    def shard_refs(self):
        return device_lib().rtx_index_shard_refs(self._h)

    @property
    def sub_batch(self):
        return int(device_lib().rtx_batch_sub_batch(self._h))

    @property
    def max_levels(self):
        return device_lib().rtx_index_max_levels(self._h)

    @property
    def index_bytes(self):
        return device_lib().rtx_index_device_bytes(self._h)

    @property
    def index_bitrow_bytes(self):
        return device_lib().rtx_index_bitrow_bytes(self._h)

    def hitcount_kernel_name(self) -> str:
        return (device_lib().rtx_hitcount_kernel_name(self._h) or b"").decode()

    def batch_slot(self, slot: int):
        """rtx_batch_slot: the batch slot (0 / 1) that batch_upload / batch_run / batch_download / classify act on."""
        self._check(device_lib().rtx_batch_slot(self._h, int(slot)))
        self._slot = int(slot)

    def upload_index_arrays(self, n_refs, csr_off, csr_ids, node_lo, node_hi, node_type, child_first, child_count, ref_levels,
                            shard=(0, 0)):
        d = IndexDesc()
        arrs = dict(csr_off=np.ascontiguousarray(csr_off, np.uint64), csr_ids=np.ascontiguousarray(csr_ids, np.uint32),
                    node_lo=np.ascontiguousarray(node_lo, np.uint32), node_hi=np.ascontiguousarray(node_hi, np.uint32),
                    node_type=np.ascontiguousarray(node_type, np.uint8), child_first=np.ascontiguousarray(child_first, np.uint32),
                    child_count=np.ascontiguousarray(child_count, np.uint32), ref_levels=np.ascontiguousarray(ref_levels, np.uint8))
        d.n_refs = n_refs
        d.csr_offsets = _ptr(arrs["csr_off"], C.c_uint64)
        d.csr_ids = _ptr(arrs["csr_ids"], C.c_uint32)
        d.n_nodes = len(arrs["node_lo"])
        d.node_lo, d.node_hi = _ptr(arrs["node_lo"], C.c_uint32), _ptr(arrs["node_hi"], C.c_uint32)
        d.node_type = _ptr(arrs["node_type"], C.c_uint8)
        d.child_first, d.child_count = _ptr(arrs["child_first"], C.c_uint32), _ptr(arrs["child_count"], C.c_uint32)
        d.ref_levels = _ptr(arrs["ref_levels"], C.c_uint8)
        d.ref_shard_begin, d.ref_shard_end = shard
        self._check(device_lib().rtx_index_upload(self._h, C.byref(d)))

    def upload_tree(self, tree: "Tree", shard=(0, 0)):
        rc = host_lib().rxh_tree_upload(tree._h, self._h, shard[0], shard[1])
        self._check(rc)

    def upload_tree_sharded(self, tree: "Tree", n_shards: int, rank: int, cuts):
        cuts = np.ascontiguousarray(cuts, np.uint64)
        assert len(cuts) == n_shards + 1
        rc = host_lib().rxh_tree_upload_sharded(tree._h, self._h, n_shards, rank, _ptr(cuts, C.c_uint64))
        self._check(rc)

    # ---- reference-sharded phases (see raxtax_b200/dist.py for the exchange between them) --------------------
    def shard_phase(self, n):
        f = getattr(device_lib(), f"rtx_shard_phase{n}")
        self._check(f(self._h))

    def shard_hist_buffer(self):
        p, n = C.c_void_p(), C.c_uint64()
        self._check(device_lib().rtx_shard_hist_buffer(self._h, C.byref(p), C.byref(n)))
        return p.value or 0, int(n.value)

    def shard_records_buffers(self):
        sp, sb, rp, rb = C.c_void_p(), C.c_uint64(), C.c_void_p(), C.c_uint64()
        self._check(device_lib().rtx_shard_records_buffers(self._h, C.byref(sp), C.byref(sb), C.byref(rp), C.byref(rb)))
        return (sp.value or 0, int(sb.value)), (rp.value or 0, int(rb.value))

    # ---- reference-sharded mode over NCCL inside the library --------------------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        rc = device_lib().rtx_comm_unique_id(buf)
        if rc != 0:
            raise RtxError(rc, device_lib().rtx_last_error(None).decode())
        return buf.raw

    def comm_init(self, unique_id: bytes, rank: int, nranks: int):
        self._check(device_lib().rtx_comm_init(self._h, unique_id, int(rank), int(nranks)))

    def comm_destroy(self):
        self._check(device_lib().rtx_comm_destroy(self._h))

    def shard_run(self):
        self._check(device_lib().rtx_shard_run(self._h))

    def shard_gather(self, root: int = 0):
        self._check(device_lib().rtx_shard_gather(self._h, int(root)))

    # ---- batches -------------------------------------------------------------------------------------------
    def _make_batch(self, seq_off, codes, exact_off, exact_ids, flags):
        b = Batch()
        seq_off = np.ascontiguousarray(seq_off, np.uint64)
        codes = np.ascontiguousarray(codes, np.uint8)
        keep = [seq_off, codes]
        b.n_queries = len(seq_off) - 1
        b.seq_offsets = _ptr(seq_off, C.c_uint64)
        b.seq_codes = _ptr(codes if codes.size else np.zeros(1, np.uint8), C.c_uint8)
        if exact_off is not None:
            exact_off = np.ascontiguousarray(exact_off, np.uint32)
            exact_ids = np.ascontiguousarray(exact_ids if exact_ids is not None and len(exact_ids) else np.zeros(1, np.uint32), np.uint32)
            keep += [exact_off, exact_ids]
            b.exact_offsets = _ptr(exact_off, C.c_uint32)
            b.exact_ids = _ptr(exact_ids, C.c_uint32)
        b.flags = flags
        return b, keep

    def pinned_array(self, shape, dtype) -> np.ndarray:
        """numpy array over rtx_host_alloc memory (freed with the context): results land in it by DMA, no staging copy."""
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        self._check(device_lib().rtx_host_alloc(max(n, 1), C.byref(p)))
        self._pinned.append(p)
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def pinned_results(self, nq, cap=0):
        """Reusable page-locked result buffers for classify(..., out=...) / batch_download(out=...): (ClassifyOutput, capacity)."""
        ML = max(self.max_levels, 1)
        cap = cap or nq * 8 + 64
        pa = self.pinned_array
        return ClassifyOutput(pa(nq, np.uint16), pa(nq + 1, np.uint32), pa(nq, np.float64), pa(cap, np.uint32), pa(cap, np.uint8),
                              pa((cap, ML), np.float64), pa(cap, np.float64)), cap

    def _alloc_results(self, nq, cap, max_len, taps, reuse=None):
        ML = max(self.max_levels, 1)
        kmax = max(max_len - 7, 0)
        if reuse is not None:  # caller-owned (pinned) buffers; the views handed back alias them until the next call
            buf, bcap = reuse
            if len(buf.n_kmers) < nq:
                raise ValueError("pinned result buffers hold fewer queries than this batch")
            out = ClassifyOutput(buf.n_kmers[:nq], buf.result_begin[:nq + 1], buf.global_signal[:nq], buf.first_ref, buf.n_levels,
                                 buf.confidence, buf.local_signal)
            cap = bcap
        else:
            out = ClassifyOutput(np.zeros(nq, np.uint16), np.zeros(nq + 1, np.uint32), np.zeros(nq, np.float64), np.empty(cap, np.uint32),
                                 np.empty(cap, np.uint8), np.empty((cap, ML), np.float64), np.empty(cap, np.float64))
        r = ResultsStruct()
        r.n_kmers = _ptr(out.n_kmers, C.c_uint16)
        r.result_begin = _ptr(out.result_begin, C.c_uint32)
        r.global_signal = _ptr(out.global_signal, C.c_double)
        r.result_capacity = cap
        r.first_ref = _ptr(out.first_ref, C.c_uint32)
        r.n_levels = _ptr(out.n_levels, C.c_uint8)
        r.confidence = _ptr(out.confidence, C.c_double)
        r.local_signal = _ptr(out.local_signal, C.c_double)
        if "counts" in taps:
            out.counts = np.zeros((nq, self.shard_refs), np.uint16)
            r.tap_counts = _ptr(out.counts, C.c_uint16)
        if "hist" in taps:
            out.hist = np.zeros((nq, kmax + 1), np.uint32)
            r.tap_hist = _ptr(out.hist, C.c_uint32)
            r.tap_hist_stride = kmax + 1
        if "kmers" in taps:
            out.kmers = np.zeros((nq, max(kmax, 1)), np.uint16)
            r.tap_kmers = _ptr(out.kmers, C.c_uint16)
            r.tap_kmer_stride = max(kmax, 1)
        if "probs" in taps:
            out.probs = np.zeros((nq, kmax + 1), np.float64)
            r.tap_probs = _ptr(out.probs, C.c_double)
            r.tap_prob_stride = kmax + 1
        return out, r

    @staticmethod
    def _trim(out: ClassifyOutput, n):
        out.first_ref, out.n_levels = out.first_ref[:n], out.n_levels[:n]
        out.confidence, out.local_signal = out.confidence[:n], out.local_signal[:n]
        return out

    @staticmethod
    def _flags(skip_exact, raw_conf, both_strands):
        return (RTX_SKIP_EXACT_MATCHES if skip_exact else 0) | (RTX_RAW_CONFIDENCE if raw_conf else 0) | (RTX_BOTH_STRANDS if both_strands else 0)

    def batch_strands(self, nq) -> np.ndarray:
        """rtx_batch_strands: per query of the downloaded both-strand batch, 0 = classified as given, 1 = as its reverse complement."""
        s = np.zeros(max(nq, 1), np.uint8)
        self._check(device_lib().rtx_batch_strands(self._h, _ptr(s, C.c_uint8)))
        return s[:nq]

    def batch_best_hits(self, nq):
        """rtx_batch_best_hits of the downloaded batch in the active slot: (n_hits [nq], ref [nq, T], count [nq, T]), the references
        with the most shared 8-mers by count descending, then id ascending; entries of row q past n_hits[q] are unspecified."""
        T = max(getattr(self, "_best_hits", {}).get(getattr(self, "_slot", 0), 0), 1)
        n = np.zeros(max(nq, 1), np.uint32)
        ref = np.zeros((max(nq, 1), T), np.uint32)
        cnt = np.zeros((max(nq, 1), T), np.uint16)
        self._check(device_lib().rtx_batch_best_hits(self._h, _ptr(n, C.c_uint32), _ptr(ref, C.c_uint32), _ptr(cnt, C.c_uint16)))
        return n[:nq], ref[:nq], cnt[:nq]

    def _set_best_hits(self, best_hits):
        self.set_option(RTX_OPT_BEST_HITS, best_hits)
        if not hasattr(self, "_best_hits"):
            self._best_hits = {}
        self._best_hits[getattr(self, "_slot", 0)] = int(best_hits)

    def classify(self, seq_off, codes, exact_off=None, exact_ids=None, skip_exact=False, raw_conf=False, taps=(), out=None, shard_root=None,
                 both_strands=False, best_hits=0) -> ClassifyOutput:
        """rtx_classify_batch: H2D + kernels + D2H in one call.  out = pinned_results(...) reuses page-locked result buffers.
        shard_root = r: rtx_shard_classify instead (reference-sharded mode over NCCL, every rank calls it with the same batch; the
        final lines come back on rank r, nothing on the others).  both_strands: every query is classified in the orientation that
        shares more 8-mers with some reference (RTX_BOTH_STRANDS); exact_off then has 2n + 1 entries (Tree.exact_batch_both_strands)
        and the result's .strand tells the orientation.  best_hits = T in 1..64: the result's .best_hits holds each query's T best
        hits (RTX_OPT_BEST_HITS, batch_best_hits)."""
        L = device_lib()
        self._set_best_hits(best_hits)
        flags = self._flags(skip_exact, raw_conf, both_strands)
        b, keep = self._make_batch(seq_off, codes, exact_off, exact_ids, flags)
        nq = b.n_queries
        so = keep[0]
        max_len = int((so[1:] - so[:-1]).max()) if nq else 0
        cap = max(nq * 8 + 64, getattr(self, "_cap_hint", 0))
        reuse = out
        while True:
            out, r = self._alloc_results(nq, cap, max_len, taps, reuse)
            if shard_root is None:
                rc = L.rtx_classify_batch(self._h, C.byref(b), C.byref(r))
            else:
                rc = L.rtx_shard_classify(self._h, C.byref(b), C.byref(r), int(shard_root))
                if rc == RTX_ERR_INVALID and r.n_results > r.result_capacity:  # the batch is resident and merged: only the copy is repeated
                    cap = int(r.n_results) + 64
                    out, r = self._alloc_results(nq, cap, max_len, taps, None)
                    rc = L.rtx_batch_download(self._h, C.byref(r))
            if rc == RTX_ERR_INVALID and r.n_results > r.result_capacity and reuse is not None:
                raise ValueError(f"pinned result buffers too small: {int(r.n_results)} result lines, capacity {int(r.result_capacity)}")
            if rc == RTX_ERR_INVALID and r.n_results > cap:
                cap = int(r.n_results) + int(r.n_results) // 4 + 64
                self._cap_hint = cap
                continue
            self._check(rc)
            if both_strands:
                out.strand = self.batch_strands(nq)
            if best_hits:
                out.best_hits = self.batch_best_hits(nq)
            return self._trim(out, int(r.n_results))

    def batch_upload(self, seq_off, codes, exact_off=None, exact_ids=None, skip_exact=False, raw_conf=False, both_strands=False, best_hits=0):
        self._set_best_hits(best_hits)
        flags = self._flags(skip_exact, raw_conf, both_strands)
        b, keep = self._make_batch(seq_off, codes, exact_off, exact_ids, flags)
        self._check(device_lib().rtx_batch_upload(self._h, C.byref(b)))
        so = keep[0]
        if not hasattr(self, "_batch_infos"):
            self._batch_infos = {}
        self._batch_infos[getattr(self, "_slot", 0)] = (b.n_queries, int((so[1:] - so[:-1]).max()) if b.n_queries else 0, both_strands)

    def batch_run(self):
        self._check(device_lib().rtx_batch_run(self._h))

    def batch_download(self, taps=()) -> ClassifyOutput:
        L = device_lib()
        nq, max_len, both_strands = self._batch_infos[getattr(self, "_slot", 0)]
        cap = max(nq * 8 + 64, getattr(self, "_cap_hint", 0))
        while True:
            out, r = self._alloc_results(nq, cap, max_len, taps)
            rc = L.rtx_batch_download(self._h, C.byref(r))
            if rc == RTX_ERR_INVALID and r.n_results > cap:
                cap = int(r.n_results) + int(r.n_results) // 4 + 64
                self._cap_hint = cap
                continue
            self._check(rc)
            if both_strands:
                out.strand = self.batch_strands(nq)
            if self._best_hits.get(getattr(self, "_slot", 0), 0):
                out.best_hits = self.batch_best_hits(nq)
            return self._trim(out, int(r.n_results))

    def profile_reset(self):
        self._check(device_lib().rtx_profile_reset(self._h))

    def profile(self) -> dict:
        p = Profile()
        self._check(device_lib().rtx_profile_get(self._h, C.byref(p)))
        d = {n: dict(launches=int(p.kernel[i].launches), total_ms=float(p.kernel[i].total_ms)) for i, n in enumerate(KERNEL_NAMES)}
        d.update(queries=int(p.queries), hits=int(p.hits), bitrow_bytes=int(p.bitrow_bytes), csr_equiv_bytes=int(p.csr_equiv_bytes),
                 h2d_bytes=int(p.h2d_bytes), d2h_bytes=int(p.d2h_bytes), allreduce_bytes=int(p.allreduce_bytes),
                 allgather_bytes=int(p.allgather_bytes), gather_bytes=int(p.gather_bytes))
        return d


# ---------------------------------------------------------------------------------------------------------------
class Counts(C.Structure):
    """rxh_counts: what rxh_count_sender / rxh_count_logger accumulate."""
    _fields_ = [(n, C.c_uint64) for n in ("queries", "lines", "label_bytes", "primary_bytes", "tsv_bytes", "checksum", "log_lines", "log_bytes", "warn_lines")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


def plan_chunks(n_queries: int, n_ctx: int = 1, chunk_size: int = 0) -> list:
    """rxh_plan_chunks: the chunk boundaries the host driver uses (chunk_size 0 = the library's choice)."""
    n = host_lib().rxh_plan_chunks(n_queries, n_ctx, chunk_size, None, 0)
    buf = (C.c_size_t * n)()
    host_lib().rxh_plan_chunks(n_queries, n_ctx, chunk_size, buf, n)
    return list(buf)


def format_fixed(value: float, precision: int) -> str:
    buf = C.create_string_buffer(512)
    n = host_lib().rxh_format_fixed(float(value), int(precision), buf, 512)
    return buf.raw[:n].decode()


def raxtax_counted(ctx, queries: "Queries", tree: "Tree", skip_exact_matches=False, raw_confidence=False, chunk_size=0, tsv=False) -> dict:
    """rxh_raxtax / rxh_raxtax_multi with the library's counting sender and logger (no Python in the loop): returns the counts."""
    L = host_lib()
    cnt = Counts()
    send = C.cast(L.rxh_count_sender, SENDER)
    log = C.cast(L.rxh_count_logger, LOGGER)
    warn = C.c_int(0)
    ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else [ctx]
    arr = (C.c_void_p * len(ctxs))(*[c._h for c in ctxs])
    rc = L.rxh_raxtax_multi(arr, len(ctxs), queries._h, tree._h, int(skip_exact_matches), int(raw_confidence), int(chunk_size), send,
                            C.addressof(cnt), int(tsv), log, C.addressof(cnt), C.byref(warn))
    if rc != 0:
        raise _host_err()
    d = cnt.as_dict()
    d["warnings"] = bool(warn.value)
    return d


class Tree:
    """raxtax::tree::Tree (tree.rs:36-43) built by the C++ host library."""

    def __init__(self, handle):
        if not handle:
            raise _host_err()
        self._h = C.c_void_p(handle)

    @classmethod
    def from_fasta(cls, text: str) -> "Tree":  # parser::parse_reference_fasta_str
        b = text.encode()
        return cls(host_lib().rxh_tree_from_fasta(b, len(b)))

    @classmethod
    def from_file(cls, path: str):  # parser::parse_reference_fasta_file (parser.rs:37-44) -> (tree, was_database)
        was = C.c_int(0)
        t = cls(host_lib().rxh_tree_from_file(path.encode(), C.byref(was)))
        return t, bool(was.value)

    @classmethod
    def from_bin(cls, data: bytes):  # Tree::load_from_file (tree.rs:154-164); None when the bytes are not a database
        h = host_lib().rxh_tree_from_bin(data, len(data))
        return cls(h) if h else None

    def save_bin(self, path: str):  # Tree::save_to_file (tree.rs:146-152)
        if host_lib().rxh_tree_save_bin(self._h, path.encode()) != 0:
            raise _host_err()

    @classmethod
    def new(cls, lineages, seq_off, codes, eager_kmer_map=False) -> "Tree":  # Tree::new
        """k_mer_map (the CSR postings) is built on first use only unless eager_kmer_map: the device derives its index from the
        sorted sequences, and uploads of a tree WITH a materialised k_mer_map go through the CSR instead."""
        blob = "\n".join(lineages).encode()
        seq_off = np.ascontiguousarray(seq_off, np.uint64)
        codes = np.ascontiguousarray(codes, np.uint8)
        if codes.size == 0:
            codes = np.zeros(1, np.uint8)
        t = cls(host_lib().rxh_tree_new(len(lineages), blob, len(blob), _ptr(seq_off, C.c_uint64), _ptr(codes, C.c_uint8)))
        if eager_kmer_map:
            t.build_kmer_map()
        return t

    def build_kmer_map(self):
        host_lib().rxh_tree_build_kmer_map(self._h)

    @property
    def has_kmer_map(self) -> bool:
        return bool(host_lib().rxh_tree_has_kmer_map(self._h))

    def __del__(self):
        try:
            if self._h:
                host_lib().rxh_tree_free(self._h)
                self._h = None
        except Exception:
            pass

    @property
    def num_tips(self):
        return host_lib().rxh_tree_num_tips(self._h)

    def lineage(self, i):
        return host_lib().rxh_tree_lineage(self._h, i).decode()

    @property
    def lineages(self):
        return [self.lineage(i) for i in range(self.num_tips)]

    def csr(self):
        off, ids = u64p(), u32p()
        host_lib().rxh_tree_csr(self._h, C.byref(off), C.byref(ids))
        o = np.ctypeslib.as_array(off, (65537,)).copy()
        nnz = int(o[-1])
        i = np.ctypeslib.as_array(ids, (nnz,)).copy() if nnz else np.zeros(0, np.uint32)  # no postings at all: the vector's data() is NULL
        return o, i

    def k_mer_map(self, kmer):
        o, i = self.csr()
        return i[int(o[kmer]): int(o[kmer + 1])]

    def exact(self, codes):
        codes = np.ascontiguousarray(codes, np.uint8)
        buf = np.zeros(64, np.uint32)
        p = _ptr(codes if codes.size else np.zeros(1, np.uint8), C.c_uint8)
        n = host_lib().rxh_tree_exact(self._h, p, len(codes), _ptr(buf, C.c_uint32), len(buf))
        if n > len(buf):
            buf = np.zeros(n, np.uint32)
            host_lib().rxh_tree_exact(self._h, p, len(codes), _ptr(buf, C.c_uint32), len(buf))
        return buf[:n].copy()

    def exact_batch(self, seq_off, codes):
        seq_off = np.ascontiguousarray(seq_off, np.uint64)
        codes = np.ascontiguousarray(codes, np.uint8)
        n = len(seq_off) - 1
        eo = np.zeros(n + 1, np.uint32)
        p = _ptr(codes if codes.size else np.zeros(1, np.uint8), C.c_uint8)
        cap = max(64, n)
        while True:
            ids = np.zeros(cap, np.uint32)
            tot = host_lib().rxh_exact_batch(self._h, n, _ptr(seq_off, C.c_uint64), p, _ptr(eo, C.c_uint32), _ptr(ids, C.c_uint32), cap)
            if tot <= cap:
                return eo, ids[:tot].copy()
            cap = int(tot)

    def exact_batch_both_strands(self, seq_off, codes):
        """exact_batch for a both-strand batch (RTX_BOTH_STRANDS): 2n + 1 offsets, [0, n) the queries as given, [n, 2n) their
        reverse complements."""
        from .synth import reverse_complement_batch

        seq_off = np.asarray(seq_off, np.uint64)
        codes = np.asarray(codes, np.uint8)
        rc = reverse_complement_batch(seq_off - seq_off[0], codes[int(seq_off[0]): int(seq_off[-1])])
        base = seq_off - seq_off[0]
        both_off = np.concatenate([base, base[1:] + base[-1]])
        return self.exact_batch(both_off, np.concatenate([codes[int(seq_off[0]): int(seq_off[-1])], rc]))

    def index_arrays(self) -> dict:
        self.build_kmer_map()
        d = IndexDesc()
        host_lib().rxh_tree_index_desc(self._h, C.byref(d))
        nn, N = d.n_nodes, d.n_refs
        g = lambda p, n: np.ctypeslib.as_array(p, (n,)).copy() if n and p else np.zeros(0, p._type_)
        off = g(d.csr_offsets, 65537)
        return dict(n_refs=N, csr_off=off, csr_ids=g(d.csr_ids, int(off[-1])), node_lo=g(d.node_lo, nn), node_hi=g(d.node_hi, nn),
                    node_type=g(d.node_type, nn), child_first=g(d.child_first, nn), child_count=g(d.child_count, nn),
                    ref_levels=g(d.ref_levels, N))


class Queries:
    """`Vec<(String, Vec<u8>)>` (parser.rs:108-154)."""

    def __init__(self, handle):
        if not handle:
            raise _host_err()
        self._h = C.c_void_p(handle)

    @classmethod
    def from_fasta(cls, text: str) -> "Queries":
        b = text.encode()
        return cls(host_lib().rxh_queries_from_fasta(b, len(b)))

    @classmethod
    def from_file(cls, path: str) -> "Queries":  # parser::parse_query_fasta_file (plain or gz, streamed)
        return cls(host_lib().rxh_queries_from_file(path.encode()))

    @classmethod
    def new(cls, labels, seq_off, codes) -> "Queries":
        blob = "\n".join(labels).encode()
        seq_off = np.ascontiguousarray(seq_off, np.uint64)
        codes = np.ascontiguousarray(codes, np.uint8)
        if codes.size == 0:
            codes = np.zeros(1, np.uint8)
        return cls(host_lib().rxh_queries_new(len(labels), blob, len(blob), _ptr(seq_off, C.c_uint64), _ptr(codes, C.c_uint8)))

    def skip(self, labels):  # queries_to_skip of parse_query_fasta_file (parser.rs:108-115)
        blob = "\n".join(labels).encode()
        if host_lib().rxh_queries_skip(self._h, blob, len(blob)) != 0:
            raise _host_err()

    def __del__(self):
        try:
            if self._h:
                host_lib().rxh_queries_free(self._h)
                self._h = None
        except Exception:
            pass

    def __len__(self):
        return host_lib().rxh_queries_len(self._h)

    @property
    def labels(self):
        return [host_lib().rxh_queries_label(self._h, i).decode() for i in range(len(self))]

    def arrays(self):
        off, codes = u64p(), u8p()
        host_lib().rxh_queries_arrays(self._h, C.byref(off), C.byref(codes))
        n = len(self)
        o = np.ctypeslib.as_array(off, (n + 1,)).copy()
        c = np.ctypeslib.as_array(codes, (max(int(o[-1]), 1),))[: int(o[-1])].copy()
        return o, c


def raxtax(ctx: Context, queries: Queries, tree: Tree, skip_exact_matches=False, raw_confidence=False, chunk_size=0, tsv=False, sharded=False,
           both_strands=False, best_hits=0):
    """raxtax::raxtax (raxtax.rs:14-97).  Returns (results, log_lines, warnings) where results is the list of
    (query_label, primary_results, tsv_results_or_None) tuples the reference sends to its writer thread.  both_strands: every query
    is classified in the orientation that shares more 8-mers with some reference (rxh_raxtax_both_strands, one or several contexts);
    every line then ends in a strand column (`+` / `-`).  best_hits = N in 1..64 (rxh_raxtax_best_hits): returns
    (results, log_lines, warnings, hits) with hits the list of (query_label, hit_lines) in the order the queries were sent."""
    if (both_strands or best_hits) and sharded:
        raise ValueError("both_strands and best_hits are not available over a reference-sharded index")
    sent, logs, hits = [], [], []

    def _send(_u, label, primary, tsv_s):
        sent.append((label.decode(), primary.decode(), tsv_s.decode() if tsv_s is not None else None))
        return 0

    def _log(_u, level, msg):
        logs.append((level, msg.decode()))

    def _hits(_u, label, lines):
        hits.append((label.decode(), lines.decode()))
        return 0

    warn = C.c_int(0)
    if best_hits:
        ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else [ctx]
        arr = (C.c_void_p * len(ctxs))(*[c._h for c in ctxs])
        rc = host_lib().rxh_raxtax_best_hits(arr, len(ctxs), queries._h, tree._h, int(skip_exact_matches), int(raw_confidence), int(chunk_size),
                                             SENDER(_send), None, int(tsv), LOGGER(_log), None, C.byref(warn), int(both_strands),
                                             int(best_hits), HITS_SENDER(_hits), None)
    elif both_strands:
        ctxs = list(ctx) if isinstance(ctx, (list, tuple)) else [ctx]
        arr = (C.c_void_p * len(ctxs))(*[c._h for c in ctxs])
        rc = host_lib().rxh_raxtax_both_strands(arr, len(ctxs), queries._h, tree._h, int(skip_exact_matches), int(raw_confidence), int(chunk_size),
                                                SENDER(_send), None, int(tsv), LOGGER(_log), None, C.byref(warn))
    elif sharded:  # ctx = the shards' contexts in shard order (upload_tree_sharded): rxh_raxtax_sharded, results in query order
        arr = (C.c_void_p * len(ctx))(*[c._h for c in ctx])
        rc = host_lib().rxh_raxtax_sharded(arr, len(ctx), queries._h, tree._h, int(skip_exact_matches), int(raw_confidence), int(chunk_size),
                                           SENDER(_send), None, int(tsv), LOGGER(_log), None, C.byref(warn))
    elif isinstance(ctx, (list, tuple)):  # several GPUs (or several contexts on one): rxh_raxtax_multi, results in completion order
        arr = (C.c_void_p * len(ctx))(*[c._h for c in ctx])
        rc = host_lib().rxh_raxtax_multi(arr, len(ctx), queries._h, tree._h, int(skip_exact_matches), int(raw_confidence), int(chunk_size),
                                         SENDER(_send), None, int(tsv), LOGGER(_log), None, C.byref(warn))
    else:
        rc = host_lib().rxh_raxtax(ctx._h, queries._h, tree._h, int(skip_exact_matches), int(raw_confidence), int(chunk_size), SENDER(_send),
                                   None, int(tsv), LOGGER(_log), None, C.byref(warn))
    if rc != 0:
        raise _host_err()
    if best_hits:
        return sent, logs, bool(warn.value), hits
    return sent, logs, bool(warn.value)

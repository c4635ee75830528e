"""ctypes binding of the C ABI (include/ebwt2snp_b200.h) -- the host-side mirror used by the tests
and bench.py.  The names follow the reference's functions for this path:

    cluster_lm   <-> ref:ebwt2clust.cpp:68-139      statistics  <-> ref:clust2snp.cpp:877-966
    find_events  <-> ref:clust2snp.cpp:788-872      to_file     <-> ref:clust2snp.cpp:633-780

There is no CPU fallback and nothing here imports oracle/: if the CUDA library is missing the
import of this module raises, and if no B200 is visible `Context()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libebwt2snp_b200.so")
MAX_C_LEN = 150
MAX_K = 128
HIST_BINS = MAX_C_LEN + 1

KERNEL_FLAGS, KERNEL_EMIT, KERNEL_SCAN, KERNEL_EXACT, KERNEL_SCAN1, KERNEL_RESOLVE, KERNEL_CAND, KERNEL_EVENTS, KERNEL_MERGE = 0, 1, 2, 3, 4, 5, 6, 7, 8
OK, ERR_CUDA, ERR_ARG, ERR_NOMEM, ERR_UNSUPPORTED, ERR_STATE = range(6)


class E2SError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"e2s error {code}: {msg}")
        self.code = code


class ClusterSummary(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "n_local", "global_off", "n_global", "n_end", "n_written", "head_end", "any_event", "open_start",
        "end_nm2_start", "tail_lcp_nm2", "tail_lcp_nm1", "tail_bwt_nm1", "k", "min_len", "lcp_bytes")]


SUMMARY_WORDS = C.sizeof(ClusterSummary) // 8


class ClusterMerged(C.Structure):
    _fields_ = [
        ("record_offset", C.c_uint64), ("total_written", C.c_uint64), ("n_clust_out", C.c_uint64),
        ("phantom_lcp", C.c_uint32), ("n_prepend", C.c_uint32), ("n_append", C.c_uint32), ("n_adopt", C.c_uint32),
        ("prepend_start", C.c_uint64), ("prepend_len", C.c_uint64), ("prepend_written", C.c_uint64),
        ("append_start", C.c_uint64 * 2), ("append_len", C.c_uint64 * 2),
        ("adopt_start", C.c_uint64 * 3), ("adopt_len", C.c_uint64 * 3),
    ]


class Stats(C.Structure):
    _fields_ = [("hist", C.c_uint64 * HIST_BINS), ("n_clust", C.c_uint64), ("n_bases", C.c_uint64),
                ("last_len", C.c_uint64), ("max_len", C.c_uint64), ("max_clust_length", C.c_int32),
                ("reserved", C.c_int32)]


class SnpParams(C.Structure):
    _fields_ = [("k_left", C.c_int32), ("k_right", C.c_int32), ("mcov_out", C.c_int32), ("max_gap", C.c_int32),
                ("consensus_reads", C.c_int32), ("max_err", C.c_int32), ("max_snvs", C.c_int32),
                ("reserved", C.c_int32), ("pval", C.c_double), ("nr_reads1", C.c_uint64)]


class Event(C.Structure):
    _fields_ = [("D", C.c_int32), ("gap", C.c_int32), ("supp0", C.c_int32), ("supp1", C.c_int32),
                ("right_len", C.c_int32), ("keep", C.c_int32), ("cluster_start", C.c_uint64),
                ("left0", C.c_char * MAX_K), ("left1", C.c_char * MAX_K), ("right", C.c_char * MAX_K)]


class SnpCounts(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_analysed", "n_flagged", "n_candidates", "n_variants", "n_events", "saw_n")]


class PipelineResult(C.Structure):
    _fields_ = [("n_written", C.c_uint64), ("n_clust_out", C.c_uint64), ("max_clust_length", C.c_int32),
                ("reserved", C.c_int32), ("snp", SnpCounts), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64)]


# every symbol include/ebwt2snp_b200.h declares (tests/test_abi.py checks the list against the header)
SYMBOLS = [
    "e2s_version", "e2s_ctx_create", "e2s_ctx_destroy", "e2s_last_error", "e2s_ctx_set_stream",
    "e2s_ctx_synchronize", "e2s_ctx_mem_info", "e2s_ctx_launch_count", "e2s_ctx_timing", "e2s_ctx_kernel_time", "e2s_shard_create", "e2s_shard_destroy", "e2s_shard_load_gesa", "e2s_shard_load_gesa_fd",
    "e2s_shard_load_soa", "e2s_shard_load_soa_dev", "e2s_build_egsa_dev", "e2s_build_egsa", "e2s_build_egsa_ragged_dev", "e2s_build_egsa_ragged", "e2s_build_egsa_range_dev", "e2s_build_egsa_ragged_range_dev", "e2s_shard_set_layout", "e2s_shard_seal", "e2s_shard_lcp_bytes_resident", "e2s_reads_stage", "e2s_reads_stage_dev",
    "e2s_cluster_prefilter", "e2s_cluster_run", "e2s_cluster_merge", "e2s_cluster_finalize", "e2s_cluster_lm", "e2s_cluster_count",
    "e2s_cluster_fetch", "e2s_cluster_fetch_packed", "e2s_clusters_stage_packed", "e2s_clusters_stage",
    "e2s_statistics", "e2s_statistics_finish", "e2s_exchange_finish", "e2s_snp_default_params", "e2s_find_events", "e2s_events_fetch",
    "e2s_events_format", "e2s_free", "e2s_pipeline_resident", "e2s_pipeline_host",
    "e2s_comm_unique_id", "e2s_comm_create", "e2s_comm_destroy", "e2s_pipeline_sharded",
    "e2s_exchange_row_words", "e2s_exchange_rows_finish",
    "e2s_pipeline_host_soa", "e2s_shard_host_gsa", "e2s_shard_load_lcp_bwt", "e2s_shard_load_bcr", "e2s_chunk_stage_clusters", "e2s_chunked_clusters_finish",
    "e2s_pipeline_host_sharded", "e2s_shard_create_chunked", "e2s_shard_chunk_positions", "e2s_chunk_begin", "e2s_chunk_scan", "e2s_chunked_finish", "e2s_chunked_reset", "e2s_chunked_exchange",
]

_lib = None


def load_library():
    """Loads the in-tree CUDA library; raises (loudly) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -m ebwt2snp_b200.build` "
                          "(there is no CPU fallback for this package)")
    lib = C.CDLL(LIB_PATH)
    lib.e2s_last_error.restype = C.c_char_p
    lib.e2s_last_error.argtypes = [C.c_void_p]
    lib.e2s_ctx_launch_count.restype = C.c_uint64
    lib.e2s_ctx_launch_count.argtypes = [C.c_void_p]
    lib.e2s_ctx_destroy.restype = None
    lib.e2s_shard_destroy.restype = None
    lib.e2s_free.restype = None
    lib.e2s_snp_default_params.restype = None
    lib.e2s_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.e2s_ctx_destroy.argtypes = [C.c_void_p]
    lib.e2s_ctx_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    lib.e2s_ctx_synchronize.argtypes = [C.c_void_p]
    lib.e2s_ctx_mem_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.e2s_ctx_timing.argtypes = [C.c_void_p, C.c_int]
    lib.e2s_ctx_kernel_time.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    lib.e2s_shard_create.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p)]
    lib.e2s_shard_destroy.argtypes = [C.c_void_p]
    lib.e2s_shard_load_gesa.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int]
    lib.e2s_shard_load_gesa_fd.argtypes = [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int]
    lib.e2s_shard_load_soa.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.c_uint64, C.c_uint64]
    lib.e2s_shard_load_soa_dev.argtypes = [C.c_void_p] + [C.c_void_p] * 4 + [C.c_uint64, C.c_uint64]
    lib.e2s_shard_seal.argtypes = [C.c_void_p]
    lib.e2s_build_egsa_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32] + [C.c_void_p] * 4
    lib.e2s_build_egsa.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32] + [C.c_void_p] * 4
    lib.e2s_build_egsa_ragged_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64] + [C.c_void_p] * 4
    lib.e2s_build_egsa_ragged.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64] + [C.c_void_p] * 4
    lib.e2s_build_egsa_range_dev.argtypes = ([C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32,
                                              C.c_uint64] + [C.c_void_p] * 4 + [C.POINTER(C.c_uint64)] * 2)
    lib.e2s_build_egsa_ragged_range_dev.argtypes = ([C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32,
                                                     C.c_uint32, C.c_uint64] + [C.c_void_p] * 4 + [C.POINTER(C.c_uint64)] * 2)
    lib.e2s_shard_lcp_bytes_resident.argtypes = [C.c_void_p]
    lib.e2s_shard_set_layout.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.e2s_reads_stage.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.e2s_reads_stage_dev.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]
    lib.e2s_cluster_prefilter.argtypes = [C.c_void_p, C.c_int]
    lib.e2s_cluster_run.argtypes = [C.c_void_p, C.c_uint32, C.c_int32, C.POINTER(ClusterSummary)]
    lib.e2s_cluster_merge.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(ClusterMerged)]
    lib.e2s_cluster_finalize.argtypes = [C.c_void_p, C.POINTER(ClusterMerged)]
    lib.e2s_cluster_lm.argtypes = [C.c_void_p, C.c_uint32, C.c_int32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.e2s_cluster_count.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
    lib.e2s_cluster_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.e2s_cluster_fetch_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.e2s_clusters_stage_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
    lib.e2s_clusters_stage.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.e2s_statistics.argtypes = [C.c_void_p, C.POINTER(Stats)]
    lib.e2s_statistics_finish.argtypes = [C.POINTER(Stats), C.c_uint64, C.c_int, C.c_double]
    lib.e2s_exchange_finish.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double,
                                        C.POINTER(ClusterMerged), C.POINTER(Stats)]
    lib.e2s_snp_default_params.argtypes = [C.POINTER(SnpParams)]
    lib.e2s_find_events.argtypes = [C.c_void_p, C.POINTER(SnpParams), C.c_int, C.POINTER(SnpCounts)]
    lib.e2s_events_fetch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.e2s_events_format.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(SnpParams), C.POINTER(C.c_void_p),
                                      C.POINTER(C.c_size_t)]
    lib.e2s_free.argtypes = [C.c_void_p]
    lib.e2s_pipeline_resident.argtypes = [C.c_void_p, C.c_uint32, C.c_int32, C.POINTER(SnpParams), C.POINTER(PipelineResult)]
    lib.e2s_comm_unique_id.argtypes = [C.c_void_p]
    lib.e2s_exchange_row_words.restype = C.c_uint64
    lib.e2s_exchange_row_words.argtypes = []
    lib.e2s_exchange_rows_finish.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_int32, C.c_int, C.c_double,
                                             C.POINTER(ClusterMerged), C.POINTER(Stats)]
    lib.e2s_comm_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    lib.e2s_comm_destroy.argtypes = [C.c_void_p]
    lib.e2s_comm_destroy.restype = None
    lib.e2s_pipeline_sharded.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int32, C.POINTER(SnpParams),
                                         C.POINTER(ClusterMerged), C.POINTER(Stats), C.POINTER(SnpCounts)]
    lib.e2s_shard_create_chunked.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p)]
    lib.e2s_shard_chunk_positions.restype = C.c_uint64
    lib.e2s_shard_chunk_positions.argtypes = [C.c_void_p]
    lib.e2s_chunk_begin.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
    lib.e2s_chunk_scan.argtypes = [C.c_void_p, C.c_uint32, C.c_int32, C.c_int, C.POINTER(C.c_uint64)]
    lib.e2s_chunked_finish.argtypes = [C.c_void_p, C.c_uint32, C.c_int32, C.POINTER(ClusterSummary)]
    lib.e2s_chunked_reset.argtypes = [C.c_void_p]
    lib.e2s_chunked_exchange.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int32, C.c_int, C.c_double, C.POINTER(ClusterMerged), C.POINTER(Stats)]
    lib.e2s_pipeline_host.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.POINTER(SnpParams), C.c_void_p,
                                      C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(PipelineResult)]
    lib.e2s_pipeline_host_soa.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_void_p,
                                          C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.POINTER(SnpParams), C.c_void_p,
                                          C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(PipelineResult)]
    lib.e2s_shard_host_gsa.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.e2s_chunk_stage_clusters.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_uint64)]
    lib.e2s_chunked_clusters_finish.argtypes = [C.c_void_p]
    lib.e2s_shard_load_lcp_bwt.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64]
    lib.e2s_shard_load_bcr.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_uint64]
    lib.e2s_pipeline_host_sharded.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_int,
                                              C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int32, C.POINTER(SnpParams),
                                              C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p, C.c_uint64,
                                              C.POINTER(ClusterMerged), C.POINTER(Stats), C.POINTER(PipelineResult)]
    _lib = lib
    return lib


def default_params(nr_reads1=0, **kw) -> SnpParams:
    p = SnpParams()
    load_library().e2s_snp_default_params(C.byref(p))
    p.nr_reads1 = nr_reads1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def _ptr(a):
    """pointer of a numpy array / torch tensor / int / None"""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(type(a))


def cluster_merge(summaries, my) -> ClusterMerged:
    """Host-only (no CUDA): e2s_cluster_merge over a list of ClusterSummary."""
    lib = load_library()
    arr = (ClusterSummary * len(summaries))(*summaries)
    out = ClusterMerged()
    rc = lib.e2s_cluster_merge(C.cast(arr, C.c_void_p), len(summaries), my, C.byref(out))
    if rc:
        raise E2SError(rc, lib.e2s_last_error(None).decode())
    return out


def exchange_finish(sum_rows, stat_rows, my, mcov_out=5, pval=0.99):
    """e2s_exchange_finish over contiguous arrays of ClusterSummary / Stats records (numpy uint8/uint64 buffers or
    ctypes arrays): -> (ClusterMerged of shard `my`, global Stats)"""
    lib = load_library()
    n = len(sum_rows)
    mg, tot = ClusterMerged(), Stats()
    rc = lib.e2s_exchange_finish(_ptr(sum_rows) if not isinstance(sum_rows, C.Array) else C.cast(sum_rows, C.c_void_p),
                                 _ptr(stat_rows) if not isinstance(stat_rows, C.Array) else C.cast(stat_rows, C.c_void_p),
                                 n, my, int(mcov_out), float(pval), C.byref(mg), C.byref(tot))
    if rc:
        raise E2SError(rc, lib.e2s_last_error(None).decode())
    return mg, tot


class ClusterDev(C.Structure):
    """mirror of the scan's device accumulators (csrc/internal.h) = the leading words of one exchange row"""
    _fields_ = [(n, C.c_uint64) for n in ("n_end", "n_written", "head_end", "any_event", "open_start", "end_nm2_start", "overflow",
                                          "ticket", "n_pf", "last_rec", "tail_lcp_nm2", "tail_lcp_nm1", "tail_bwt_nm1", "n_bases")] + \
               [("hist", C.c_uint64 * HIST_BINS)]


def exchange_row_words() -> int:
    return int(load_library().e2s_exchange_row_words())


def exchange_rows_finish(rows, my, n_global, k, min_len, mcov_out=5, pval=0.99):
    """e2s_exchange_rows_finish over the gathered (world, exchange_row_words()) uint64 rows -> (ClusterMerged, global Stats)"""
    lib = load_library()
    rows = np.ascontiguousarray(rows, dtype=np.uint64)
    mg, tot = ClusterMerged(), Stats()
    rc = lib.e2s_exchange_rows_finish(_ptr(rows), rows.shape[0], int(my), int(n_global), int(k), int(min_len), int(mcov_out),
                                      float(pval), C.byref(mg), C.byref(tot))
    if rc:
        raise E2SError(rc, lib.e2s_last_error(None).decode())
    return mg, tot


def statistics_finish(st: Stats, last_len, mcov_out=5, pval=0.99) -> Stats:
    lib = load_library()
    rc = lib.e2s_statistics_finish(C.byref(st), int(last_len), int(mcov_out), float(pval))
    if rc:
        raise E2SError(rc, lib.e2s_last_error(None).decode())
    return st


def events_format(events, params: SnpParams, first_id=1) -> bytes:
    """to_file(): .snp text of the kept events (host-only)."""
    lib = load_library()
    n = len(events)
    arr = (Event * n)(*events) if n else None
    text, ln = C.c_void_p(), C.c_size_t()
    rc = lib.e2s_events_format(C.cast(arr, C.c_void_p) if n else None, n, first_id, C.byref(params), C.byref(text), C.byref(ln))
    if rc:
        raise E2SError(rc, lib.e2s_last_error(None).decode())
    data = C.string_at(text, ln.value)
    lib.e2s_free(text)
    return data


class Context:
    def __init__(self, device=0, stream=None):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.e2s_ctx_create(device, C.byref(h))
        if rc:
            raise E2SError(rc, self.lib.e2s_last_error(None).decode())
        self.h = h
        self.device = int(device)
        if stream is not None:
            self._ck(self.lib.e2s_ctx_set_stream(self.h, C.c_void_p(stream)))

    def _ck(self, rc):
        if rc:
            raise E2SError(rc, self.lib.e2s_last_error(self.h).decode())

    def close(self):
        if self.h:
            self.lib.e2s_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def synchronize(self):
        self._ck(self.lib.e2s_ctx_synchronize(self.h))

    @property
    def launches(self):
        return int(self.lib.e2s_ctx_launch_count(self.h))

    def timing(self, enable=True):
        self._ck(self.lib.e2s_ctx_timing(self.h, int(enable)))

    def kernel_time(self, kernel):
        """(total ms, launches) of KERNEL_FLAGS / _EMIT / _SCAN / _EXACT since the last call (CUDA events on the stream)"""
        ms, cnt = C.c_double(), C.c_uint64()
        self._ck(self.lib.e2s_ctx_kernel_time(self.h, kernel, C.byref(ms), C.byref(cnt)))
        return ms.value, cnt.value

    def stage_reads(self, bases, offsets, device=False, n_bases=None):
        n_reads = len(offsets) - 1
        if device:
            self._keep = (bases, offsets)
            self._ck(self.lib.e2s_reads_stage_dev(self.h, _ptr(bases), _ptr(offsets), n_reads, int(n_bases)))
        else:
            bases = np.ascontiguousarray(bases, dtype=np.uint8).reshape(-1)
            offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
            self._ck(self.lib.e2s_reads_stage(self.h, _ptr(bases), _ptr(offsets), n_reads))
            self.synchronize()

    def build_egsa(self, reads):
        """EGSA construction on the GPU (e2s_build_egsa_dev): `reads` = (R, L) uint8 ASCII, a numpy array or a torch
        tensor on this context's device.  Returns the same dict of torch tensors as synth.build_egsa (lcp / text /
        suff as int32 holding u32, bwt uint8, n, L, R), resident on the device."""
        import torch
        dev = torch.device("cuda", self.device)
        reads_t = (torch.from_numpy(np.ascontiguousarray(reads, dtype=np.uint8)) if isinstance(reads, np.ndarray) else reads)
        reads_t = reads_t.to(dev).contiguous()
        R, L = int(reads_t.shape[0]), int(reads_t.shape[1])
        n = R * (L + 1)
        out = {k: torch.empty(n, dtype=torch.int32, device=dev) for k in ("lcp", "text", "suff")}
        out["bwt"] = torch.empty(n, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)  # the library works on its own stream
        self._ck(self.lib.e2s_build_egsa_dev(self.h, _ptr(reads_t), R, L, _ptr(out["lcp"]), _ptr(out["text"]),
                                             _ptr(out["suff"]), _ptr(out["bwt"])))
        out.update(n=n, L=L, R=R)
        return out

    def build_egsa_range(self, reads, key_lo, key_hi, before=None, capacity=None):
        """One key range of the index (e2s_build_egsa_range_dev): the records of the suffixes whose first 32 symbols, as a 64-bit
        word at 2 bits per base, lie in [key_lo, key_hi) (key_hi = 0: no upper bound).  before = (text, suff) of the record that
        precedes the range (for lcp[0]) or None.  Returns the dict of build_egsa cut to the range + first = its index position."""
        import torch
        dev = torch.device("cuda", self.device)
        reads_t = (torch.from_numpy(np.ascontiguousarray(reads, dtype=np.uint8)) if isinstance(reads, np.ndarray) else reads)
        reads_t = reads_t.to(dev).contiguous()
        R, L = int(reads_t.shape[0]), int(reads_t.shape[1])
        cap = R * (L + 1) if capacity is None else int(capacity)
        out = {k: torch.empty(cap, dtype=torch.int32, device=dev) for k in ("lcp", "text", "suff")}
        out["bwt"] = torch.empty(cap, dtype=torch.uint8, device=dev)
        n_rec, first = C.c_uint64(0), C.c_uint64(0)
        bt, bs = (0xFFFFFFFF, 0) if before is None else (int(before[0]), int(before[1]))
        torch.cuda.synchronize(dev)
        self._ck(self.lib.e2s_build_egsa_range_dev(self.h, _ptr(reads_t), R, L, int(key_lo), int(key_hi), bt, bs, cap, _ptr(out["lcp"]),
                                                   _ptr(out["text"]), _ptr(out["suff"]), _ptr(out["bwt"]), C.byref(n_rec), C.byref(first)))
        m = int(n_rec.value)
        out = {k: v[:m] for k, v in out.items()}
        out.update(n=m, L=L, R=R, first=int(first.value))
        return out

    def build_egsa_ragged(self, bases, off):
        """The same for reads of any lengths (e2s_build_egsa_ragged_dev): `bases` = all reads back to back (numpy uint8 or a
        torch tensor on this context's device), `off` = R + 1 offsets (host).  n = off[R] + R records."""
        import torch
        dev = torch.device("cuda", self.device)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        R = len(off) - 1
        n = int(off[R]) + R
        bases_t = (torch.from_numpy(np.ascontiguousarray(bases, dtype=np.uint8).reshape(-1)) if isinstance(bases, np.ndarray) else bases)
        if bases_t.numel() == 0:
            bases_t = torch.zeros(1, dtype=torch.uint8)
        bases_t = bases_t.to(dev).contiguous()
        out = {k: torch.empty(n, dtype=torch.int32, device=dev) for k in ("lcp", "text", "suff")}
        out["bwt"] = torch.empty(n, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        self._ck(self.lib.e2s_build_egsa_ragged_dev(self.h, _ptr(bases_t), off.ctypes.data, R, _ptr(out["lcp"]), _ptr(out["text"]),
                                                    _ptr(out["suff"]), _ptr(out["bwt"])))
        out.update(n=n, R=R)
        return out

    def build_egsa_ragged_range(self, bases, off, key_lo, key_hi, before=None, capacity=None):
        """One key range of the index of reads of any lengths (e2s_build_egsa_ragged_range_dev): `bases` / `off` as for
        build_egsa_ragged, the range, `before` and `capacity` as for build_egsa_range.  Returns the dict of build_egsa_ragged cut to the
        range + first = its index position."""
        import torch
        dev = torch.device("cuda", self.device)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        R = len(off) - 1
        cap = int(off[R]) + R if capacity is None else int(capacity)
        bases_t = (torch.from_numpy(np.ascontiguousarray(bases, dtype=np.uint8).reshape(-1)) if isinstance(bases, np.ndarray) else bases)
        if bases_t.numel() == 0:
            bases_t = torch.zeros(1, dtype=torch.uint8)
        bases_t = bases_t.to(dev).contiguous()
        out = {k: torch.empty(max(cap, 1), dtype=torch.int32, device=dev) for k in ("lcp", "text", "suff")}
        out["bwt"] = torch.empty(max(cap, 1), dtype=torch.uint8, device=dev)
        n_rec, first = C.c_uint64(0), C.c_uint64(0)
        bt, bs = (0xFFFFFFFF, 0) if before is None else (int(before[0]), int(before[1]))
        torch.cuda.synchronize(dev)
        self._ck(self.lib.e2s_build_egsa_ragged_range_dev(self.h, _ptr(bases_t), off.ctypes.data, R, int(key_lo), int(key_hi), bt, bs, cap,
                                                          _ptr(out["lcp"]), _ptr(out["text"]), _ptr(out["suff"]), _ptr(out["bwt"]),
                                                          C.byref(n_rec), C.byref(first)))
        m = int(n_rec.value)
        out = {k: v[:m] for k, v in out.items()}
        out.update(n=m, R=R, first=int(first.value))
        return out

    def shard(self, n_local, global_off=0, n_global=None, chunk_positions=None):
        """chunk_positions: a CHUNKED shard -- the device buffers hold one chunk of the range at a time (streaming)"""
        return Shard(self, n_local, global_off, n_local if n_global is None else n_global, chunk_positions)

    def pipeline_host(self, gesa_records, n, reads_bases, reads_off, params, k=16, min_len=2, x=4, y=4, z=4,
                      rec10=None, events=None):
        """ebwt2clust + clust2snp from host buffers (pointers may be pinned torch tensors / numpy arrays)."""
        res = PipelineResult()
        n_reads = (len(reads_off) - 1) if reads_off is not None else 0
        cap_r = (rec10.nbytes // 10) if rec10 is not None else 0
        cap_e = len(events) if events is not None else 0
        self._ck(self.lib.e2s_pipeline_host(self.h, _ptr(gesa_records), n, x, y, z, _ptr(reads_bases), _ptr(reads_off),
                                            n_reads, k, min_len, C.byref(params), _ptr(rec10), cap_r,
                                            C.cast(events, C.c_void_p) if events is not None else None, cap_e,
                                            C.byref(res)))
        return res

    def pipeline_host_soa(self, lcp, bwt, pair_sa, n, reads_bases, reads_off, params, k=16, min_len=2, x=4, y=4, z=4,
                          rec10=None, events=None):
        """The same from the BCR triple (X.out.lcp, X.out, X.out.pairSA as byte buffers): only lcp + bwt cross PCIe in full,
        the survivors' text / suff are fetched from the host's pairSA (e2s_pipeline_host_soa)."""
        res = PipelineResult()
        n_reads = (len(reads_off) - 1) if reads_off is not None else 0
        cap_r = (rec10.nbytes // 10) if rec10 is not None else 0
        cap_e = len(events) if events is not None else 0
        self._ck(self.lib.e2s_pipeline_host_soa(self.h, _ptr(lcp), x, _ptr(bwt), _ptr(pair_sa), y, z, n, _ptr(reads_bases),
                                                _ptr(reads_off), n_reads, k, min_len, C.byref(params), _ptr(rec10), cap_r,
                                                C.cast(events, C.c_void_p) if events is not None else None, cap_e,
                                                C.byref(res)))
        return res


def pipeline_host_sharded(ctx, comm, records, first, range_lo, range_n, n_global, reads_bases, reads_off, params, k=16, min_len=2,
                          x=4, y=4, z=4, rec10=None, events=None):
    """e2s_pipeline_host_sharded: this rank's range of ONE eBWT from host records -> (PipelineResult, ClusterMerged, Stats, records in rec10)"""
    res, mg, st = PipelineResult(), ClusterMerged(), Stats()
    n_reads = (len(reads_off) - 1) if reads_off is not None else 0
    cap_r = (rec10.nbytes // 10) if rec10 is not None else 0
    cap_e = len(events) if events is not None else 0
    m = C.c_uint64()
    ctx._ck(ctx.lib.e2s_pipeline_host_sharded(ctx.h, comm.h, _ptr(records), int(first), int(range_lo), int(range_n), int(n_global), x, y, z,
                                              _ptr(reads_bases), _ptr(reads_off), n_reads, k, min_len, C.byref(params), _ptr(rec10), cap_r,
                                              C.byref(m), C.cast(events, C.c_void_p) if events is not None else None, cap_e,
                                              C.byref(mg), C.byref(st), C.byref(res)))
    return res, mg, st, m.value


class Comm:
    """The library's own NCCL communicator for the exchange between the phases (one process per GPU).  The 128-byte
    unique id is created on rank 0 and broadcast by the caller's launcher plumbing (torch.distributed)."""

    def __init__(self, ctx: Context, rank: int, world: int, broadcast_bytes):
        """broadcast_bytes(bytes | None) -> bytes: collective; returns on every rank what rank 0 passed in"""
        self.ctx, self.lib = ctx, ctx.lib
        buf = (C.c_uint8 * 128)()
        if rank == 0:
            ctx._ck(self.lib.e2s_comm_unique_id(buf))
        got = broadcast_bytes(bytes(buf) if rank == 0 else None)
        idb = (C.c_uint8 * 128).from_buffer_copy(got)
        h = C.c_void_p()
        ctx._ck(self.lib.e2s_comm_create(ctx.h, idb, rank, world, C.byref(h)))
        self.h, self.rank, self.world = h, rank, world

    def close(self):
        if self.h:
            self.lib.e2s_comm_destroy(self.h)
            self.h = None


class Shard:
    """A contiguous eBWT range resident on the GPU (see the header)."""

    def __init__(self, ctx: Context, n_local, global_off, n_global, chunk_positions=None):
        self.ctx, self.lib = ctx, ctx.lib
        self.n_local, self.global_off, self.n_global = int(n_local), int(global_off), int(n_global)
        h = C.c_void_p()
        if chunk_positions:
            ctx._ck(self.lib.e2s_shard_create_chunked(ctx.h, self.n_local, self.global_off, self.n_global, int(chunk_positions), C.byref(h)))
        else:
            ctx._ck(self.lib.e2s_shard_create(ctx.h, self.n_local, self.global_off, self.n_global, C.byref(h)))
        self.h = h

    # ---- chunked shards (streaming) ------------------------------------------------------
    @property
    def chunk_positions(self) -> int:
        return int(self.lib.e2s_shard_chunk_positions(self.h))

    def chunks(self):
        """the (lo, n) of every chunk of the range, in order"""
        cp, lo, end = self.chunk_positions, self.global_off, self.global_off + self.n_local
        while lo < end:
            yield lo, min(cp, end - lo)
            lo += cp

    def chunk_begin(self, lo, n):
        self.ctx._ck(self.lib.e2s_chunk_begin(self.h, int(lo), int(n)))

    def chunk_scan(self, k=16, min_len=2, mcov_out=0) -> int:
        m = C.c_uint64()
        self.ctx._ck(self.lib.e2s_chunk_scan(self.h, k, min_len, int(mcov_out), C.byref(m)))
        return m.value

    def chunk_stage_clusters(self, rec10, mcov_out, max_clust_length) -> int:
        """clust2snp on a chunked shard: the .clusters records (10-byte, uint8 array) that start in the open chunk -> #survivors"""
        rec10 = np.ascontiguousarray(rec10, dtype=np.uint8)
        ns = C.c_uint64()
        self.ctx._ck(self.lib.e2s_chunk_stage_clusters(self.h, _ptr(rec10) if len(rec10) else None, len(rec10) // 10, int(mcov_out),
                                                       int(max_clust_length), C.byref(ns)))
        return ns.value

    def chunked_clusters_finish(self):
        self.ctx._ck(self.lib.e2s_chunked_clusters_finish(self.h))

    def host_gsa(self, pair_sa, y, z):
        """lean SoA mode of a chunked shard: text / suff of the captured records come from this host buffer (kept alive by the caller)"""
        self.ctx._ck(self.lib.e2s_shard_host_gsa(self.h, _ptr(pair_sa), y, z))

    def chunked_finish(self, k=16, min_len=2) -> ClusterSummary:
        s = ClusterSummary()
        self.ctx._ck(self.lib.e2s_chunked_finish(self.h, k, min_len, C.byref(s)))
        return s

    def chunked_exchange(self, comm, k=16, min_len=2, mcov_out=5, pval=0.99):
        """multi-GPU: finish + all-gather of the ranks' accumulators + merge + statistics + finalize (collective)"""
        mg, st = ClusterMerged(), Stats()
        self.ctx._ck(self.lib.e2s_chunked_exchange(self.h, comm.h, k, min_len, int(mcov_out), float(pval), C.byref(mg), C.byref(st)))
        return mg, st

    def chunked_reset(self):
        self.ctx._ck(self.lib.e2s_chunked_reset(self.h))

    def close(self):
        if self.h:
            self.lib.e2s_shard_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- residency ---------------------------------------------------------------------
    def load_gesa(self, records, first=0, count=None, x=4, y=4, z=4):
        rs = x + y + z + 1
        if count is None:
            count = records.nbytes // rs if isinstance(records, np.ndarray) else records.numel() * records.element_size() // rs
        self.ctx._ck(self.lib.e2s_shard_load_gesa(self.h, _ptr(records), int(first), int(count), x, y, z))
        self.ctx.synchronize()

    def load_gesa_fd(self, fd, first, count, x=4, y=4, z=4):
        """records [first, first + count) of the X.gesa file open at the descriptor fd (pinned ring + reader threads)"""
        self.ctx._ck(self.lib.e2s_shard_load_gesa_fd(self.h, int(fd), int(first), int(count), x, y, z))

    def load_soa(self, lcp, text, suff, bwt, first=0, device=False):
        count = len(lcp) if lcp is not None else len(bwt)
        if device:
            self.ctx._ck(self.lib.e2s_shard_load_soa_dev(self.h, _ptr(lcp), _ptr(text), _ptr(suff), _ptr(bwt), int(first), count))
        else:
            arrs = [None if a is None else np.ascontiguousarray(a, dtype=t) for a, t in
                    ((lcp, np.uint32), (text, np.uint32), (suff, np.uint32), (bwt, np.uint8))]
            self.ctx._ck(self.lib.e2s_shard_load_soa(self.h, *[_ptr(a) for a in arrs], int(first), count))
        self.ctx.synchronize()

    def load_bcr(self, lcp, bwt, pair_sa, x, y, z, first=0):
        """the BCR triple as byte buffers (lcp at x bytes, BWT, pairSA = suff(z) text(y)); pair_sa=None: lcp + BWT only"""
        count = len(bwt)
        lcp, bwt = np.ascontiguousarray(lcp).view(np.uint8), np.ascontiguousarray(bwt, dtype=np.uint8)
        if pair_sa is None:
            self.ctx._ck(self.lib.e2s_shard_load_lcp_bwt(self.h, _ptr(lcp), x, _ptr(bwt), int(first), count))
        else:
            pair_sa = np.ascontiguousarray(pair_sa).view(np.uint8)
            self.ctx._ck(self.lib.e2s_shard_load_bcr(self.h, _ptr(lcp), x, _ptr(bwt), _ptr(pair_sa), y, z, int(first), count))
        self.ctx.synchronize()

    def set_layout(self, x=4, y=4, z=4, bcr=False):
        """byte widths / format of the index files the arrays came from (the reference's phantom record depends on it)"""
        self.ctx._ck(self.lib.e2s_shard_set_layout(self.h, x, y, z, int(bcr)))

    def seal(self):
        self.ctx._ck(self.lib.e2s_shard_seal(self.h))

    def lcp_bytes_resident(self) -> int:
        """1 when the scan streams the bit-sliced LCP copy the loads wrote (values above 127 saturated: exact for -k <= 127), else 4"""
        return int(self.lib.e2s_shard_lcp_bytes_resident(self.h))

    # ---- phase 1 -----------------------------------------------------------------------
    def cluster_prefilter(self, mcov_out):
        """fused mode: later cluster_run calls also run clust2snp's BWT prefilter for this -m (0 = off)"""
        self.ctx._ck(self.lib.e2s_cluster_prefilter(self.h, int(mcov_out)))

    def cluster_run(self, k=16, min_len=2) -> ClusterSummary:
        s = ClusterSummary()
        self.ctx._ck(self.lib.e2s_cluster_run(self.h, k, min_len, C.byref(s)))
        return s

    def cluster_finalize(self, merged: ClusterMerged):
        self.ctx._ck(self.lib.e2s_cluster_finalize(self.h, C.byref(merged)))

    def cluster_lm(self, k=16, min_len=2):
        """-> (n_written, n_clust_out) ; ref:ebwt2clust.cpp:68-139"""
        nw, nc = C.c_uint64(), C.c_uint64()
        self.ctx._ck(self.lib.e2s_cluster_lm(self.h, k, min_len, C.byref(nw), C.byref(nc)))
        return nw.value, nc.value

    def cluster_count(self):
        m = C.c_uint64()
        self.ctx._ck(self.lib.e2s_cluster_count(self.h, C.byref(m)))
        return m.value

    def cluster_fetch(self):
        m = self.cluster_count()
        start = np.empty(m, dtype=np.uint64)
        ln = np.empty(m, dtype=np.uint16)
        mm = C.c_uint64()
        if m:
            self.ctx._ck(self.lib.e2s_cluster_fetch(self.h, _ptr(start), _ptr(ln), m, C.byref(mm)))
        return start, ln

    def cluster_fetch_packed(self) -> bytes:
        m = self.cluster_count()
        buf = np.empty(m * 10 + 1, dtype=np.uint8)
        mm = C.c_uint64()
        self.ctx._ck(self.lib.e2s_cluster_fetch_packed(self.h, _ptr(buf), m, C.byref(mm)))
        return buf[: m * 10].tobytes()

    # ---- phase 2 -----------------------------------------------------------------------
    def stage_clusters(self, start, ln):
        start = np.ascontiguousarray(start, dtype=np.uint64)
        ln = np.ascontiguousarray(ln, dtype=np.uint16)
        self.ctx._ck(self.lib.e2s_clusters_stage(self.h, _ptr(start), _ptr(ln), len(ln)))

    def stage_clusters_packed(self, data: bytes):
        buf = np.frombuffer(data, dtype=np.uint8)
        self.ctx._ck(self.lib.e2s_clusters_stage_packed(self.h, _ptr(buf), len(data) // 10))

    def statistics(self, mcov_out=5, pval=0.99, finish=True) -> Stats:
        st = Stats()
        self.ctx._ck(self.lib.e2s_statistics(self.h, C.byref(st)))
        if finish:
            statistics_finish(st, st.last_len, mcov_out, pval)
        return st

    def find_events(self, params: SnpParams, max_clust_length) -> SnpCounts:
        cnt = SnpCounts()
        try:
            self.ctx._ck(self.lib.e2s_find_events(self.h, C.byref(params), int(max_clust_length), C.byref(cnt)))
        except E2SError as e:
            e.counts = cnt  # the counters up to the failure (e.g. candidates found before a read lookup failed)
            raise
        return cnt

    def pipeline_resident(self, params: SnpParams, k=16, min_len=2) -> PipelineResult:
        """cluster_lm + statistics + find_events on a sealed whole-eBWT shard in one C call"""
        res = PipelineResult()
        self.ctx._ck(self.lib.e2s_pipeline_resident(self.h, k, min_len, C.byref(params), C.byref(res)))
        return res

    def pipeline_sharded(self, comm: "Comm", params: SnpParams, k=16, min_len=2):
        """the sharded step in one C call (collective): -> (ClusterMerged of this shard, global Stats, SnpCounts)"""
        mg, st, cnt = ClusterMerged(), Stats(), SnpCounts()
        self.ctx._ck(self.lib.e2s_pipeline_sharded(self.h, comm.h, k, min_len, C.byref(params), C.byref(mg), C.byref(st),
                                                   C.byref(cnt)))
        return mg, st, cnt

    def events(self):
        n = C.c_uint64()
        self.ctx._ck(self.lib.e2s_events_fetch(self.h, None, 0, C.byref(n)))
        arr = (Event * n.value)()
        if n.value:
            self.ctx._ck(self.lib.e2s_events_fetch(self.h, C.cast(arr, C.c_void_p), n.value, C.byref(n)))
        return list(arr)

"""ctypes wrapper of oracle/_build/liboracle.so and a runner for oracle/_ref -- TEST INFRASTRUCTURE ONLY.

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference legs (see oracle/oracle.h).  Nothing here touches a GPU.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_build", "liboracle.so")
REF_DIR = os.path.join(HERE, "_ref")
MAX_C_LEN = 150
FLAG_SAW_N = 1         # oracle.h ORACLE_FLAG_SAW_N
FLAG_BAD_READ_REF = 2  # oracle.h ORACLE_FLAG_BAD_READ_REF


class Params(C.Structure):
    _fields_ = [
        ("k_left", C.c_int), ("k_right", C.c_int), ("mcov_out", C.c_int), ("max_gap", C.c_int),
        ("consensus_reads", C.c_int), ("max_err", C.c_int), ("max_snvs", C.c_int),
        ("pval", C.c_double), ("nr_reads1", C.c_uint64),
    ]


class ClusterResult(C.Structure):
    _fields_ = [("n_written", C.c_uint64), ("n_clust_out", C.c_uint32), ("phantom_lcp", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("hist", C.c_uint64 * (MAX_C_LEN + 1)), ("n_clust", C.c_uint64), ("n_bases", C.c_uint64),
                ("max_len", C.c_uint64), ("max_clust_length", C.c_int)]


class SnpResult(C.Structure):
    _fields_ = [("n_candidates", C.c_uint64), ("n_variants", C.c_uint64), ("n_events", C.c_uint64),
                ("n_analysed", C.c_uint64), ("flags", C.c_uint32)]


_lib = None


def build(force=False):
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(os.path.join(HERE, "oracle.c")):
        subprocess.run(["make", "-C", HERE, "port"], check=True, capture_output=True)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(LIB_PATH)
        _lib.oracle_cluster_lm.restype = C.c_int
        _lib.oracle_statistics.restype = C.c_int
        _lib.oracle_find_events.restype = C.c_int
        _lib.oracle_phantom_field.restype = C.c_uint32
    return _lib


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


def default_params(nr_reads1=0, **kw) -> Params:
    p = Params()
    lib().oracle_default_params(C.byref(p))
    p.nr_reads1 = nr_reads1
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def cluster_lm(lcp, bwt, k=16, min_len=2, x=4):
    """-> (start u64[], len u16[], n_clust_out, phantom_lcp); ref:ebwt2clust.cpp:68-139."""
    lcp = np.ascontiguousarray(lcp, dtype=np.uint32)
    bwt = np.ascontiguousarray(bwt, dtype=np.uint8)
    n = len(lcp)
    start = np.empty(n + 1, dtype=np.uint64)
    ln = np.empty(n + 1, dtype=np.uint16)
    res = ClusterResult()
    rc = lib().oracle_cluster_lm_x(_p(lcp, C.c_uint32), _p(bwt, C.c_uint8), C.c_uint64(n), C.c_uint32(k), C.c_int(min_len),
                                   C.c_int(x), _p(start, C.c_uint64), _p(ln, C.c_uint16), C.c_uint64(n + 1), C.byref(res))
    if rc:
        raise ValueError("oracle_cluster_lm: input outside the reference's domain")
    m = res.n_written
    return start[:m].copy(), ln[:m].copy(), int(res.n_clust_out), int(res.phantom_lcp)


def statistics(start, ln, mcov_out=5, pval=0.99) -> Stats:
    start = np.ascontiguousarray(start, dtype=np.uint64)
    ln = np.ascontiguousarray(ln, dtype=np.uint16)
    st = Stats()
    rc = lib().oracle_statistics(_p(start, C.c_uint64), _p(ln, C.c_uint16), C.c_uint64(len(ln)), C.c_int(mcov_out),
                                 C.c_double(pval), C.byref(st))
    if rc:
        raise ValueError("oracle_statistics: input outside the reference's domain")
    return st


def find_events(lcp, text, suff, bwt, start, ln, params: Params, max_clust_length, read_bases, read_off,
                x=4, y=4, z=4, bcr=False, strict=True):
    """-> (snp_bytes, SnpResult); ref:clust2snp.cpp:788-872.  x/y/z/bcr: layout of the index files (phantom record only)."""
    lcp = np.ascontiguousarray(lcp, dtype=np.uint32)
    text = np.ascontiguousarray(text, dtype=np.uint32)
    suff = np.ascontiguousarray(suff, dtype=np.uint32)
    bwt = np.ascontiguousarray(bwt, dtype=np.uint8)
    start = np.ascontiguousarray(start, dtype=np.uint64)
    ln = np.ascontiguousarray(ln, dtype=np.uint16)
    read_bases = np.ascontiguousarray(read_bases, dtype=np.uint8).reshape(-1)
    read_off = np.ascontiguousarray(read_off, dtype=np.uint64)
    out = C.c_char_p()
    out_len = C.c_size_t()
    res = SnpResult()
    rc = lib().oracle_find_events_w(_p(lcp, C.c_uint32), _p(text, C.c_uint32), _p(suff, C.c_uint32), _p(bwt, C.c_uint8),
                                    C.c_uint64(len(lcp)), _p(start, C.c_uint64), _p(ln, C.c_uint16), C.c_uint64(len(ln)),
                                    C.byref(params), C.c_int(max_clust_length), _p(read_bases, C.c_uint8),
                                    _p(read_off, C.c_uint64), C.c_uint64(len(read_off) - 1),
                                    C.c_int(x), C.c_int(y), C.c_int(z), C.c_int(int(bcr)),
                                    C.byref(out), C.byref(out_len), C.byref(res))
    if rc:
        if not strict:  # the candidate count is printed by the reference before it crashes (ref:clust2snp.cpp:859)
            return None, res
        if res.flags & FLAG_BAD_READ_REF:
            raise ValueError(f"oracle_find_events: input the reference would crash on (flags={res.flags})")
        raise ValueError("oracle_find_events: options outside what the restatement supports (consensus_reads < 1, k_left > 256, "
                         "max_gap > k_left, max_clust_length > 150) or an empty index")
    data = C.string_at(out, out_len.value)
    lib().oracle_free(out)
    return data, res


def distance(a: bytes, b: bytes, max_gap=10):
    assert len(a) == len(b)
    D, g = C.c_int(), C.c_int()
    lib().oracle_distance(a, b, C.c_int(len(a)), C.c_int(max_gap), C.byref(D), C.byref(g))
    return D.value, g.value


def clusters_to_bytes(start, ln) -> bytes:
    """.clusters layout: {u64 start LE, u16 length LE} x m, ref:ebwt2clust.cpp:58-59."""
    rec = np.empty(len(ln), dtype=np.dtype([("s", "<u8"), ("l", "<u2")]))
    rec["s"] = start
    rec["l"] = ln
    return rec.tobytes()


def clusters_from_bytes(data: bytes):
    rec = np.frombuffer(data, dtype=np.dtype([("s", "<u8"), ("l", "<u2")]))
    return rec["s"].copy(), rec["l"].copy()


def uniform_read_offsets(R, L):
    return (np.arange(R + 1, dtype=np.uint64) * np.uint64(L)).astype(np.uint64)


# ------------------------------------------------------------------------------------------
# the unmodified reference binaries (oracle/_ref), when present
# ------------------------------------------------------------------------------------------

def ref_available() -> bool:
    return all(os.access(os.path.join(REF_DIR, t), os.X_OK) for t in ("ebwt2clust", "clust2snp"))


def ref_ebwt2clust(fasta, k=None, m=None, x=4, y=4, z=4, timeout=3600):
    """Runs oracle/_ref/ebwt2clust -i fasta; returns (stdout, n_clust_out printed)."""
    cmd = [os.path.join(REF_DIR, "ebwt2clust"), "-i", fasta, "-x", str(x), "-y", str(y), "-z", str(z)]
    if k is not None:
        cmd += ["-k", str(k)]
    if m is not None:
        cmd += ["-m", str(m)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
    n = None
    for line in r.stdout.splitlines():
        if line.startswith("Done. ") and "clusters saved" in line:
            n = int(line.split()[1])
    return r, n


def ref_clust2snp(fasta, nreads1, x=4, y=4, z=4, extra=(), timeout=3600):
    cmd = [os.path.join(REF_DIR, "clust2snp"), "-i", fasta, "-n", str(nreads1), "-x", str(x), "-y", str(y), "-z", str(z)]
    cmd += list(extra)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
    info = {"returncode": r.returncode}
    for line in r.stdout.splitlines():
        if line.startswith("Cluster sizes allowed:"):
            a, b = line.split("[")[1].rstrip("]").split(",")
            info["allowed"] = (int(a), int(b))
        if line.startswith("Done. ") and "potential variants" in line:
            info["n_candidates"] = int(line.split()[1])
    return r, info


def build_egsa(reads: np.ndarray):
    """oracle_build_egsa: comparison sort of all suffixes (small inputs only).  Same dict as synth.build_egsa, numpy."""
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    R, L = reads.shape
    n = R * (L + 1)
    out = {k: np.empty(n, dtype=np.uint32) for k in ("lcp", "text", "suff")}
    out["bwt"] = np.empty(n, dtype=np.uint8)
    f = lib().oracle_build_egsa
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32] + [C.c_void_p] * 4
    rc = f(reads.ctypes.data, R, L, out["lcp"].ctypes.data, out["text"].ctypes.data, out["suff"].ctypes.data,
           out["bwt"].ctypes.data)
    if rc:
        raise MemoryError("oracle_build_egsa")
    out.update(n=n, L=L, R=R)
    return out


def build_egsa_ragged(bases: np.ndarray, off: np.ndarray):
    """oracle_build_egsa_ragged: reads of any lengths (bases back to back, off = R + 1 offsets); numpy dict as build_egsa."""
    bases = np.ascontiguousarray(bases, dtype=np.uint8).reshape(-1)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    R = len(off) - 1
    n = int(off[R]) + R
    out = {k: np.empty(n, dtype=np.uint32) for k in ("lcp", "text", "suff")}
    out["bwt"] = np.empty(n, dtype=np.uint8)
    pad = bases if bases.size else np.zeros(1, dtype=np.uint8)
    f = lib().oracle_build_egsa_ragged
    f.restype = C.c_int
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64] + [C.c_void_p] * 4
    rc = f(pad.ctypes.data, off.ctypes.data, R, out["lcp"].ctypes.data, out["text"].ctypes.data, out["suff"].ctypes.data,
           out["bwt"].ctypes.data)
    if rc:
        raise MemoryError("oracle_build_egsa_ragged")
    out.update(n=n, R=R)
    return out

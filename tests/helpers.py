"""Test-side helpers (numpy): random LCP arrays, a vectorised shard emulation of what the CUDA scan
reports for one shard (used to test the host-side merge logic without a GPU), dataset cache."""
from __future__ import annotations

import os

import numpy as np

from ebwt2snp_b200 import api, synth

BWT_ALPHABET = np.frombuffer(b"ACGT$acgt\x00\xff", dtype=np.uint8)


def random_lcp(rng, n, k, mode):
    if mode == 0:
        lcp = rng.integers(0, 2 * k + 2, size=n)
    elif mode == 1:
        lcp = rng.integers(0, 70000, size=n)
    elif mode == 2:
        lcp = np.maximum(0, np.cumsum(rng.integers(-3, 4, size=n)) + k)
    elif mode == 3:
        lcp = rng.integers(k, k + 3, size=n)  # long runs, few local minima
    else:
        lcp = np.full(n, k + 1)  # one giant cluster
        lcp[rng.integers(0, n, size=max(1, n // 5000))] = 0
    return lcp.astype(np.uint32)


def flags(lcp, k):
    """START/END masks of the stencil form (SURVEY.md §8(a) A2) for positions 0..n-1, END(n-1) left out."""
    n = len(lcp)
    l = lcp.astype(np.int64)
    ge = l >= k
    prev = np.concatenate([[0], l[:-1]])
    nxt = np.concatenate([l[1:], [0]])
    ge_n = np.concatenate([ge[1:], [False]])
    end = ge & (((prev > l) & (l <= nxt)) | ~ge_n)
    end[0] = False
    if n > 2 and ge[0] and not ge[1]:
        end[1] = True
    end[n - 1] = False
    ge_p = np.concatenate([[False], ge[:-1]])
    end_p = np.concatenate([[False], end[:-1]])
    start = ge & (~ge_p | end_p)
    return start, end


def emulate_shard(lcp, bwt, lo, hi, k, min_len, lcp_bytes=4):
    """What e2s_cluster_run reports for the shard [lo, hi) of the global arrays: (summary, start[], len[])."""
    n = len(lcp)
    start, end = flags(lcp, k)
    s = api.ClusterSummary()
    s.n_local, s.global_off, s.n_global = hi - lo, lo, n
    s.k, s.min_len = k, min_len & 0xFFFFFFFFFFFFFFFF
    s.lcp_bytes = lcp_bytes
    st_pos = np.flatnonzero(start[lo:hi]) + lo
    en_pos = np.flatnonzero(end[lo:hi]) + lo
    s.n_end = len(en_pos)
    s.any_event = int(len(st_pos) + len(en_pos) > 0)
    recs_s, recs_l = [], []
    ens = list(en_pos)
    if ens and (len(st_pos) == 0 or ens[0] < st_pos[0]):
        s.head_end = int(ens[0]) + 1
        if ens[0] == n - 2:
            s.end_nm2_start = 0xFFFFFFFFFFFFFFFF
        ens = ens[1:]
    for j, e in enumerate(ens):
        st = int(st_pos[j])
        ln = (int(e) - st + 1) & 0xFFFF
        if ln >= min_len:
            recs_s.append(st)
            recs_l.append(ln)
        if e == n - 2:
            s.end_nm2_start = st + 1
    s.n_written = len(recs_s)
    if len(st_pos) > len(ens):
        s.open_start = int(st_pos[-1]) + 1
    if hi == n:
        s.tail_lcp_nm2, s.tail_lcp_nm1, s.tail_bwt_nm1 = int(lcp[n - 2]), int(lcp[n - 1]), int(bwt[n - 1])
    return s, np.array(recs_s, dtype=np.uint64), np.array(recs_l, dtype=np.uint16)


def assemble(summaries, shard_records):
    """Global .clusters (start, len) from per-shard results + e2s_cluster_merge; also n_clust_out."""
    S, L = [], []
    mg = None
    for g, (rs, rl) in enumerate(shard_records):
        mg = api.cluster_merge(summaries, g)
        assert mg.record_offset == len(S)
        if mg.n_prepend and mg.prepend_written:
            S.append(mg.prepend_start)
            L.append(mg.prepend_len)
        S += list(rs)
        L += list(rl)
        for i in range(mg.n_append):
            S.append(mg.append_start[i])
            L.append(mg.append_len[i])
    assert mg.total_written == len(S)
    return np.array(S, dtype=np.uint64), np.array(L, dtype=np.uint16), mg


def reference_outputs(fa, eg, reads, nreads1):
    """What the unmodified reference's ebwt2clust + clust2snp (defaults, -x 4 -y 4 -z 4) make of the dataset `fa` (written by
    synth.write_dataset from the index `eg` and `reads`): (.clusters bytes, .snp bytes or None where clust2snp fails, the
    n_clust_out it prints, {"returncode", "allowed", "n_candidates", and with the binaries "stdout" of clust2snp}).
    The binaries themselves (oracle/_ref) where they are built, then the files they wrote are removed.  Elsewhere the oracle's
    restatement of them (oracle/oracle.c): the committed outputs of the binaries under tests/golden pin it byte for byte on
    their read sets (micro fixtures, equal-length fuzz, field widths), but not on the caller's inputs, so there the caller
    compares with the restatement and not with the binaries."""
    from oracle import oracle as O
    snp_path = os.path.join(os.path.dirname(fa), os.path.basename(fa).rsplit(".fast", 1)[0] + ".snp")
    if O.ref_available():
        r1, ncl = O.ref_ebwt2clust(fa)
        assert r1.returncode == 0, r1.stderr
        r2, info = O.ref_clust2snp(fa, nreads1)
        info["stdout"] = r2.stdout
        cl = open(fa + ".clusters", "rb").read()
        os.remove(fa + ".clusters")
        snp = open(snp_path, "rb").read() if info["returncode"] == 0 else None
        if os.path.exists(snp_path):
            os.remove(snp_path)
        return cl, snp, ncl, info
    lcp, text, suff, bwt = (np.asarray(eg[k]) for k in ("lcp", "text", "suff", "bwt"))
    s, l, ncl, _ = O.cluster_lm(lcp, bwt, 16, 2)
    cl = O.clusters_to_bytes(s, l)
    if len(l) == 0:  # the reference divides by zero in its statistics
        return cl, None, ncl, {"returncode": 1}
    p = O.default_params(nreads1)
    st = O.statistics(s, l, p.mcov_out, p.pval)
    snp, res = O.find_events(lcp, text, suff, bwt, s, l, p, st.max_clust_length, reads, O.uniform_read_offsets(*reads.shape),
                             strict=False)
    return cl, snp, ncl, {"returncode": 0 if snp is not None else 1, "allowed": (2 * p.mcov_out, st.max_clust_length),
                          "n_candidates": int(res.n_candidates)}


_DS_CACHE = {}


def dataset(name, seed=1, device="cpu"):
    """(ReadSet, egsa dict of numpy arrays) of a named config, cached per session."""
    key = (name, seed)
    if key not in _DS_CACHE:
        rs = synth.make_config(name, seed=seed)
        e = synth.build_egsa(rs.reads, device=device)
        eg = {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in e.items()}
        for f in ("lcp", "text", "suff"):
            eg[f] = eg[f].view(np.uint32)
        _DS_CACHE[key] = (rs, eg)
    return _DS_CACHE[key]

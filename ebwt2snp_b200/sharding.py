"""Multi-GPU plumbing: one process per GPU, contiguous eBWT shards (SURVEY.md §8(e)).

The path shards by contiguous eBWT ranges and has **no data-path collective**: the only exchanges are
a few words per rank between the phases,

    1. halo records (2 left / 151 right) once, when the shards are loaded,
    2. the 14-word scan summary of every shard        -> e2s_cluster_merge (host integer logic),
    3. the 151-bin length histogram + 3 counters      -> e2s_statistics_finish (max_clust_length),
    4. the kept-event count (when the text is written) -> global id_nr offsets of the .snp records,

all done with `torch.distributed.all_gather` on small int64 tensors (NCCL over NVLink on the GPUs,
gloo in the CPU tests).  The functions take ctypes structs of `api` in and out so that the same code
runs in `bench.py` under torchrun and in `tests/test_sharding_gloo.py` without a GPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
import torch.distributed as dist

from . import api

HALO_L = 2                      # END(i) needs lcp[i-1], START(i) needs END(i-1)
HALO_R = api.MAX_C_LEN + 1      # clusters analysed in phase 2 are <= 150 long (+1 for the LCP stencil)


def shard_cuts(n, parts):
    """contiguous, nearly equal shards, every one with >= 2 positions (mirrors host_io.hpp:shard_cuts)"""
    parts = max(1, int(parts))
    while parts > 1 and n // parts < 2:
        parts -= 1
    base, rem = divmod(n, parts)
    cuts = [base * g + min(g, rem) for g in range(parts)] + [n]
    return cuts


def first_key_words(reads, rows, cols):
    """the 64-bit first key word (32 symbols at 2 bits, A=0 C=1 G=2 T=3, first symbol most significant, zero padded) of the suffixes
    (rows[i], cols[i]) = (read, offset): what e2s_build_egsa_range_dev / e2s_build_egsa_ragged_range_dev compare with their key range.
    `reads` = the (R, L) read matrix, or a ragged collection (bases, off): all reads back to back + R + 1 offsets."""
    code = np.zeros(256, dtype=np.uint64)
    for c, v in ((b"C", 1), (b"c", 1), (b"G", 2), (b"g", 2), (b"T", 3), (b"t", 3)):
        code[c[0]] = v
    rows = np.asarray(rows, dtype=np.int64)
    cols = np.asarray(cols, dtype=np.int64)
    if isinstance(reads, tuple):
        bases = np.asarray(reads[0], dtype=np.uint8).reshape(-1)
        off = np.asarray(reads[1], dtype=np.int64)
        start, end = off[rows] + cols, off[rows + 1]
        last = max(len(bases) - 1, 0)
        fetch = lambda at: code[bases[np.minimum(at, last)]] if len(bases) else np.zeros(len(at), dtype=np.uint64)  # noqa: E731
    else:
        reads = np.asarray(reads)
        L = reads.shape[1]
        start, end = cols, np.full(len(rows), L, dtype=np.int64)
        fetch = lambda at: code[reads[rows, np.minimum(at, L - 1)]]  # noqa: E731
    key = np.zeros(len(rows), dtype=np.uint64)
    for j in range(32):
        at = start + j
        sym = np.where(at < end, fetch(at), np.uint64(0))
        key = (key << np.uint64(2)) | sym
    return key


def key_range_cuts(parts, reads=None, sample=1 << 16, seed=0):
    """`parts` key ranges [(lo, hi), ...] that tile the 64-bit key space (hi = 0 on the last one: no upper bound) -- one per rank (or
    per pass) for e2s_build_egsa_range_dev / e2s_build_egsa_ragged_range_dev.  Without reads: equal slices of the key space.  With the
    (R, L) read matrix or a ragged collection (bases, off): the cuts are quantiles of the first key words of `sample` suffixes drawn
    uniformly over all suffix slots, terminator suffixes included, so the ranges hold about the same number of records whatever the
    base composition (the terminator suffixes, and every suffix with an all-A first word, share key 0 and stay in the first range)."""
    parts = max(1, int(parts))
    if reads is None:
        cuts = [(i << 64) // parts for i in range(parts)]
    else:
        rng = np.random.default_rng(seed)
        if isinstance(reads, tuple):
            off = np.asarray(reads[1], dtype=np.int64)
            R = len(off) - 1
            slot0 = off + np.arange(R + 1)  # slot of (r, 0); read r owns slots [slot0[r], slot0[r + 1])
            m = int(min(sample, slot0[R]))
            slots = rng.integers(0, slot0[R], size=m)
            rows = np.searchsorted(slot0, slots, side="right") - 1
            cols = slots - slot0[rows]
        else:
            reads = np.asarray(reads)
            R, L = reads.shape
            m = int(min(sample, R * (L + 1)))
            rows, cols = rng.integers(0, R, size=m), rng.integers(0, L + 1, size=m)
        keys = np.sort(first_key_words(reads, rows, cols))
        cuts = [0] + [int(keys[(i * m) // parts]) for i in range(1, parts)]
        for i in range(1, parts):  # strictly increasing (a heavy key value cannot be cut: the ranges after it start past it)
            cuts[i] = max(cuts[i], cuts[i - 1] + 1)
    return [(cuts[i], cuts[i + 1] if i + 1 < parts else 0) for i in range(parts)]


def _world(group=None):
    if not (dist.is_available() and dist.is_initialized()):
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


_STAGE = {}


def _staging(n_words, world, device):
    """reusable buffers of one collective: pinned host send/recv + device send/recv (int64 words)"""
    key = (n_words, world, str(device))
    if key not in _STAGE:
        pin = torch.device(device).type == "cuda"
        _STAGE[key] = (torch.empty(n_words, dtype=torch.int64, pin_memory=pin),
                       torch.empty(n_words * world, dtype=torch.int64, pin_memory=pin),
                       torch.empty(n_words, dtype=torch.int64, device=device),
                       torch.empty(n_words * world, dtype=torch.int64, device=device))
    return _STAGE[key]


def all_gather_words(words, device, group=None):
    """all-gather of a short list of unsigned 64-bit words (one collective, one host synchronisation);
    returns a (world, n_words) uint64 numpy array"""
    rank, world = _world(group)
    w = np.ascontiguousarray(words, dtype=np.uint64)
    if world == 1:
        return w.reshape(1, -1).copy()
    h_send, h_recv, d_send, d_recv = _staging(len(w), world, device)
    h_send.numpy()[:] = w.view(np.int64)
    d_send.copy_(h_send, non_blocking=True)
    dist.all_gather_into_tensor(d_recv, d_send, group=group)
    h_recv.copy_(d_recv, non_blocking=True)
    if torch.device(device).type == "cuda":
        torch.cuda.current_stream(device).synchronize()
    return h_recv.numpy().view(np.uint64).reshape(world, len(w)).copy()


def exchange_summaries(summary: api.ClusterSummary, device, group=None):
    """step 2: every rank gets the scan summaries of all shards, in rank (= eBWT) order"""
    words = np.frombuffer(bytes(summary), dtype=np.uint64)
    gathered = all_gather_words(words, device, group)
    return [api.ClusterSummary.from_buffer_copy(g.tobytes()) for g in gathered]


def merge_clusters(summary: api.ClusterSummary, device, group=None):
    """-> (merged view of this rank, list of all summaries); ref:ebwt2clust.cpp:90-135 across shards"""
    rank, world = _world(group)
    sums = [summary] if world == 1 else exchange_summaries(summary, device, group)
    return api.cluster_merge(sums, rank), sums


def merge_statistics(st: api.Stats, mcov_out, pval, device, group=None) -> api.Stats:
    """step 3: global statistics() = sum of the shards' histograms; the reference's double count of the
    last record (ref:clust2snp.cpp:889) uses the LAST record of the global file, i.e. of the last
    shard that has any record.  Runs the pval loop (one IEEE double division per step, on the host)."""
    if _world(group)[1] == 1:
        api.statistics_finish(st, st.last_len, mcov_out, pval)
        return st
    gathered = all_gather_words(_stats_words(st), device, group)
    return _sum_statistics(gathered, mcov_out, pval)


def _stats_words(st: api.Stats):
    """the 154 leading u64 words of an e2s_stats (hist[151], n_clust, n_bases, last_len) as a numpy view"""
    return np.frombuffer(st, dtype=np.uint64, count=api.HIST_BINS + 3)


def _sum_statistics(rows, mcov_out, pval) -> api.Stats:
    """rows[g] = hist[151], n_clust, n_bases, last_len of shard g's records in file order"""
    tot = api.Stats()
    H = api.HIST_BINS
    w = _stats_words(tot)
    w[:H + 2] = rows[:, :H + 2].sum(axis=0)
    nz = np.flatnonzero(rows[:, H])
    last_len = int(rows[nz[-1], H + 2]) if len(nz) else 0
    tot.last_len = last_len
    api.statistics_finish(tot, last_len, mcov_out, pval)
    return tot


def event_id_offset(n_events, device, group=None):
    """step 4: -> (first id_nr of this rank's kept events, total kept events); ids start at 1 (ref:clust2snp.cpp:637)"""
    rank, world = _world(group)
    if world == 1:
        return 1, int(n_events)
    counts = [int(g[0]) for g in all_gather_words([int(n_events)], device, group)]
    return 1 + sum(counts[:rank]), sum(counts)


class EventIdOffset:
    """Step 4, deferred: global id_nr offsets are only needed when the .snp text is formatted (ref:clust2snp.cpp:637,764),
    so the all-gather of the kept-event counts runs when `resolve()` asks for them, not inside the hot path."""

    def __init__(self, n_events, device, group=None):
        self.n, self.device, self.group = int(n_events), device, group
        self._res = None

    def resolve(self):
        """-> (first id_nr of this rank's kept events, total kept events); a collective: every rank must call it"""
        if self._res is None:
            self._res = event_id_offset(self.n, self.device, self.group)
        return self._res


def exchange_halo(lcp, text, suff, bwt, device, group=None):
    """step 1 for shards that were BORN on their GPUs (bench.py): returns
    (left: dict of 2-element tensors from the previous rank or None,
     right: dict of 151-element tensors from the next rank or None).
    Inputs are this rank's torch tensors (int32 lcp/text/suff, uint8 bwt) of >= 151 elements."""
    rank, world = _world(group)
    if world == 1:
        return None, None
    n = lcp.numel()
    if n < HALO_R:
        raise ValueError("shard shorter than the halo")

    def pack(a, b):
        return torch.cat([lcp[a:b].to(torch.int32), text[a:b].to(torch.int32), suff[a:b].to(torch.int32),
                          bwt[a:b].to(torch.int32)])

    mine = torch.cat([pack(n - HALO_L, n), pack(0, HALO_R)]).to(device)
    allv = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allv, mine, group=group)

    def unpack(v, w):
        v = v.view(4, w)
        return {"lcp": v[0].contiguous(), "text": v[1].contiguous(), "suff": v[2].contiguous(),
                "bwt": v[3].to(torch.uint8).contiguous()}

    left = unpack(allv[rank - 1][: 4 * HALO_L], HALO_L) if rank > 0 else None
    right = unpack(allv[rank + 1][4 * HALO_L:], HALO_R) if rank < world - 1 else None
    return left, right


def shard_from_reads(ctx: "api.Context", bases, off, x, y, z, device, group=None) -> "api.Shard":
    """This rank's resident shard of ONE index built from all the reads (one process per rank, every rank passes the same reads):
    the reads are staged, the key cuts computed locally (the same on every rank, no collective), this rank's key range built into
    its shard, the halo rows exchanged with one all-gather and applied, and the shard sealed.  hot_path_step runs on it next."""
    rank, world = _world(group)
    bases = np.ascontiguousarray(bases, dtype=np.uint8).reshape(-1)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    ctx.stage_reads(bases if bases.size else np.zeros(1, dtype=np.uint8), off)
    key_lo, position = ctx.key_cuts(off, world)
    lo, hi = int(position[rank]), int(position[rank + 1])
    sh = ctx.shard(hi - lo, lo, int(position[world]))
    sh.build_egsa_range(off, int(key_lo[rank]), int(key_lo[rank + 1]) if rank + 1 < world else 0, x, y, z)
    rows = all_gather_words(sh.halo_row(), device, group)
    sh.halo_apply(rows, rank)
    sh.seal()
    return sh


def exchange_and_merge(summary: api.ClusterSummary, own: api.Stats, mcov_out, pval, device, group=None):
    """ONE collective between the phases: every rank contributes its scan summary and the length histogram of its OWN
    records; every rank then runs the (host, integer) merge for all shards, adds the records the merge creates at shard
    heads / at the tail to the histogram itself and finishes statistics().
    -> (ClusterMerged of this rank, global Stats with max_clust_length)"""
    rank, world = _world(group)
    W, SW = api.SUMMARY_WORDS, C.sizeof(api.Stats) // 8
    words = np.concatenate([np.frombuffer(summary, dtype=np.uint64), np.frombuffer(own, dtype=np.uint64)])
    rows = all_gather_words(words, device, group)
    sum_rows = np.ascontiguousarray(rows[:, :W])
    stat_rows = np.ascontiguousarray(rows[:, W:W + SW])
    return api.exchange_finish(sum_rows, stat_rows, rank, mcov_out, pval)


def make_comm(ctx: "api.Context", device, group=None) -> "api.Comm":
    """The library's own NCCL communicator over the ranks of the process group (its unique id travels through one
    torch.distributed broadcast).  With it, hot_path_step runs as ONE C call per step (e2s_pipeline_sharded): the
    exchange between the phases is an ncclAllGather on the library's stream instead of Python-driven collectives."""
    rank, world = _world(group)

    def bcast(data):
        t = torch.zeros(128, dtype=torch.uint8, device=device)
        if rank == 0:
            t.copy_(torch.frombuffer(bytearray(data), dtype=torch.uint8))
        dist.broadcast(t, src=0, group=group)
        return bytes(t.cpu().numpy().tobytes())

    return api.Comm(ctx, rank, world, bcast)


def hot_path_step(shard: "api.Shard", params: api.SnpParams, k, min_len, device, group=None, comm=None):
    """One pass of the hot path on this rank's resident shard, collectives included.
    -> (ClusterMerged, Stats (global), SnpCounts (this shard), EventIdOffset: .resolve() gives the first id_nr of this shard)
    comm (make_comm): the whole step is one library call, the exchange an ncclAllGather on the library's stream."""
    rank, world = _world(group)
    if comm is not None and world > 1:
        mg, st, cnt = shard.pipeline_sharded(comm, params, k, min_len)
        return mg, st, cnt, EventIdOffset(cnt.n_events, device, group)
    shard.cluster_prefilter(params.mcov_out)  # both phases run here: K2 applies the BWT prefilter while it writes the records
    s = shard.cluster_run(k, min_len)
    if world == 1:
        mg = api.cluster_merge([s], 0)
        shard.cluster_finalize(mg)
        st = shard.statistics(params.mcov_out, params.pval)
        cnt = shard.find_events(params, st.max_clust_length)
        return mg, st, cnt, EventIdOffset(cnt.n_events, device, group)
    own = shard.statistics(finish=False)  # before finalize: the shard's own records only
    mg, st = exchange_and_merge(s, own, params.mcov_out, params.pval, device, group)
    shard.cluster_finalize(mg)
    cnt = shard.find_events(params, st.max_clust_length)
    ids = EventIdOffset(cnt.n_events, device, group)  # resolved (one small all-gather) when the text is formatted
    return mg, st, cnt, ids

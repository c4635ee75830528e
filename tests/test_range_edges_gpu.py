"""-m gpu: byte parity with the oracle where the scan's ranges end -- scan tiles, streamed chunks, shards.

(a) An END at position n - 2 decides the reference's post-EOF phantom value (SURVEY.md A3), and with it the tail records and
    n_clust_out.  The inputs close a cluster at n - 2 and open one at n - 1, with k and bwt[n - 1] chosen so that the phantom
    value of the closed cluster's start and the fallback of an eBWT without such an END fall on opposite sides of k.  The
    cluster starts in the tile of n - 2, in the tile before, or before the chunk / shard.  The tile of n - 2 is interior in
    some of these shapes (n % 16384 == 1, a streamed range whose last chunk holds one position) and on the edge in others.
(b) Records a chunked shard adopts from the merge (the next shard's head record, the tail-rule records), of any length and
    starting in any chunk, while the fused BWT prefilter is armed.
(c) Inputs the streamed pipeline refuses in a later chunk (-k > 127 over an LCP value above 127, a wrapped-length cluster
    whose start has left the device): e2s_pipeline_host takes them on a resident shard; e2s_pipeline_host_soa refuses them.
(d) The ebwt2clust CLI on the shapes of (a) and (c).
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from ebwt2snp_b200 import api, synth
from oracle import oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu

T = 16384  # positions per scan tile; the chunks of a chunked shard start at whole tiles
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
R, L, NR1 = 400, 100, 200  # synthetic read set: R random reads of L bases, the first NR1 of sample 1
BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ebwt2snp_b200", "bin")


@pytest.fixture(scope="module")
def ctx(built):
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def reads():
    rng = np.random.default_rng(2024)
    rd = ACGT[rng.integers(0, 4, size=(R, L))]
    return rd, O.uniform_read_offsets(R, L)


def index_arrays(rng, lcp):
    """text / suff / bwt around an LCP array: every record points into the synthetic reads, far enough from their ends for
    clust2snp's left and right contexts"""
    n = len(lcp)
    text = rng.integers(0, R, size=n).astype(np.uint32)
    suff = rng.integers(31, 60, size=n).astype(np.uint32)
    bwt = ACGT[rng.integers(0, 4, size=n)].copy()
    return text, suff, bwt


def plant_cluster(lcp, lo, ln, v):
    """one cluster [lo, lo + ln): LCP v >= k inside, 0 on both sides"""
    lcp[lo - 1] = 0
    lcp[lo:lo + ln] = v
    lcp[lo + ln] = 0


def plant_snp(rng, lcp, text, bwt, lo, ln, v):
    """an analysable cluster that looks like a SNP: sample 1's records all 'A', sample 2's all 'C'"""
    plant_cluster(lcp, lo, ln, v)
    h = ln // 2
    text[lo:lo + h] = rng.integers(0, NR1, size=h)
    bwt[lo:lo + h] = ord("A")
    text[lo + h:lo + ln] = rng.integers(NR1, R, size=ln - h)
    bwt[lo + h:lo + ln] = ord("C")


def phantom_input(rng, n, k, s):
    """(lcp, text, suff, bwt) with random clusters everywhere, two SNP-like clusters early on, and one cluster [s, n - 2]
    closed by an END at n - 2 (lcp[n-3] > lcp[n-2] <= lcp[n-1], all >= k) so that a START follows at n - 1.  bwt[n - 1] = 'A'
    makes the fallback phantom value 65 < k; the value the reference uses is s (masked to the LCP width)."""
    lcp = np.minimum(rng.integers(0, 2 * k + 2, size=n), 255).astype(np.uint32)
    text, suff, bwt = index_arrays(rng, lcp)
    for lo in (1000, 3000):
        plant_snp(rng, lcp, text, bwt, lo, 30, k + 10)
    lcp[s - 1] = 0
    lcp[s:n - 2] = k + 6
    lcp[n - 2] = k + 5
    lcp[n - 1] = k + 5
    bwt[n - 1] = ord("A")
    return lcp, text, suff, bwt


def at_200(s):
    """s moved down (by < 256) to a position whose low byte is 200: the phantom value stays >= k under a 1-byte LCP field"""
    return s - ((s & 0xFF) - 200) % 256


def phantom_starts(n, lo=0):
    """where the cluster closed at n - 2 starts: in the scan tile of n - 2 (tiles counted from lo), in the tile before, and
    far back (before lo, or near the start of the eBWT)"""
    e = n - 2
    t0 = lo + (e - lo) // T * T
    out = {}
    if e - t0 >= 600:
        out["tile"] = at_200(e - 300)
    if t0 - 600 > max(lo, 300):
        out["prev"] = at_200(t0 - 300)
    out["far"] = at_200(lo - 300) if lo >= 600 else at_200(5300)
    return out


def check_phantom(lcp, bwt, k, m, x=4):
    """the oracle's outputs; and the input really separates the two phantom rules"""
    es, el, enc, P = O.cluster_lm(lcp, bwt, k, m, x=x)
    fallback = ((int(lcp[-1]) & ~0xFF) | int(bwt[-1])) & ((1 << (8 * x)) - 1)
    assert P >= k > fallback, (P, fallback, k)
    return es, el, enc


def oracle_snp(lcp, text, suff, bwt, es, el, rd, off, p_kw=None, x=4):
    op = O.default_params(NR1, **(p_kw or {}))
    ost = O.statistics(es, el, op.mcov_out, op.pval)
    otext, ores = O.find_events(lcp, text, suff, bwt, es, el, op, ost.max_clust_length, rd, off, x=x)
    return otext, ores, ost


def summary_equals(got, want, where):
    for f, _ in api.ClusterSummary._fields_:
        assert getattr(got, f) == getattr(want, f), (f, getattr(got, f), getattr(want, f), where)


def stream_range(ctx, lcp, bwt, k, m, chunk, lo=0, hi=None, text=None, suff=None, mcov=0):
    """the range [lo, hi) through a chunked shard, chunk by chunk -> (summary, records, shard)"""
    n = len(lcp)
    hi = n if hi is None else hi
    sh = ctx.shard(hi - lo, lo, n, chunk_positions=chunk)
    S, Ls = [], []
    for clo, cn in sh.chunks():
        sh.chunk_begin(clo, cn)
        a, b = max(0, clo - 176), min(n, clo + cn + 152)
        sh.load_soa(lcp[a:b], None if text is None else text[a:b], None if suff is None else suff[a:b], bwt[a:b], first=a)
        cnt = sh.chunk_scan(k, m, mcov)
        s, l = sh.cluster_fetch()
        assert len(s) == cnt
        S.append(s)
        Ls.append(l)
    return sh.chunked_finish(k, m), np.concatenate(S), np.concatenate(Ls), sh


def gesa(lcp, text, suff, bwt):
    return synth.gesa_records({"n": len(lcp), "lcp": lcp, "text": text, "suff": suff, "bwt": bwt}).view(np.uint8).reshape(-1)


def pipeline_host_equals_oracle(ctx, rec, lcp, text, suff, bwt, rd, off, k, m, what):
    n = len(lcp)
    es, el, enc, _ = O.cluster_lm(lcp, bwt, k, m)
    otext, ores, ost = oracle_snp(lcp, text, suff, bwt, es, el, rd, off)
    p = api.default_params(NR1)
    rec10 = np.empty((len(es) + 16) * 10, dtype=np.uint8)
    evbuf = (api.Event * (ores.n_candidates + 16))()
    res = ctx.pipeline_host(rec, n, rd.reshape(-1), off, p, k, m, rec10=rec10, events=evbuf)
    assert res.n_written == len(es) and rec10[: len(es) * 10].tobytes() == O.clusters_to_bytes(es, el), what
    assert (res.n_clust_out, res.max_clust_length) == (enc, ost.max_clust_length), what
    assert (res.snp.n_analysed, res.snp.n_candidates, res.snp.n_events) == (ores.n_analysed, ores.n_candidates, ores.n_events), what
    assert api.events_format(list(evbuf)[: res.snp.n_variants], p) == otext, what
    return res


# ---------------------------------------------------------------------------------------------------------------------------
# (a) END at n - 2
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [32769, 49153, 5 * T + 1, 16385, 32770])
def test_phantom_end_nm2_resident(ctx, n):
    """cluster_lm on one resident shard.  n % 16384 == 1 with 3 tiles or more: n - 2 is the last position of an interior
    tile; 16385 (n - 2 in the eBWT's first tile) and 32770 (n - 2 in the tile of n - 1) are the controls.  k = 130 over LCP
    values above 127 runs the 4-byte kernels, k = 100 the one-pass scan; x = 1, 2 mask the phantom value to the field."""
    rng = np.random.default_rng(n)
    for where, s in phantom_starts(n).items():
        for k in (100, 130):
            lcp, _, _, bwt = phantom_input(rng, n, k, s)
            for x in (4, 1, 2):
                for m in (-1, 1, 2):
                    es, el, enc = check_phantom(lcp, bwt, k, m, x)
                    sh = ctx.shard(n)
                    sh.load_soa(lcp, None, None, bwt)
                    sh.set_layout(x, 4, 4)
                    sh.seal()
                    nw, nc = sh.cluster_lm(k, m)
                    got = sh.cluster_fetch_packed()
                    sh.close()
                    assert (nw, nc) == (len(es), enc) and got == O.clusters_to_bytes(es, el), (n, where, k, x, m)


@pytest.mark.parametrize("n_last", [16385, 32769])
def test_phantom_end_nm2_last_shard(ctx, n_last):
    """two resident shards, the last one at global_off != 0 with n - 2 in an interior tile of its own: cluster_run summaries
    field by field against helpers.emulate_shard, the assembled .clusters against the oracle"""
    off = 20000
    n = off + n_last
    rng = np.random.default_rng(n_last)
    for where, s in phantom_starts(n, off).items():
        for k in (100, 130):
            lcp, _, _, bwt = phantom_input(rng, n, k, s)
            for m in (-1, 1, 2):
                es, el, enc = check_phantom(lcp, bwt, k, m)
                sums, recs = [], []
                for lo, hi in ((0, off), (off, n)):
                    sh = ctx.shard(hi - lo, lo, n)
                    a, b = max(0, lo - 2), min(n, hi + 151)
                    sh.load_soa(lcp[a:b], None, None, bwt[a:b], first=a)
                    sh.seal()
                    sums.append(sh.cluster_run(k, m))
                    sh.cluster_finalize(api.ClusterMerged())
                    recs.append(sh.cluster_fetch())
                    sh.close()
                    want, ws, wl = H.emulate_shard(lcp, bwt, lo, hi, k, m)
                    summary_equals(sums[-1], want, (n_last, where, k, m, lo))
                    assert np.array_equal(recs[-1][0], ws) and np.array_equal(recs[-1][1], wl)
                S, Ls, mg = H.assemble(sums, recs)
                assert mg.n_clust_out == enc and np.array_equal(S, es) and np.array_equal(Ls, el), (n_last, where, k, m)


@pytest.mark.parametrize("r", [0, 1, 2])
def test_phantom_end_nm2_chunked(ctx, r):
    """the chunk API over a range of 3 * 16384 + r positions: r = 1 leaves a last chunk of one position, so n - 2 is the last
    position of a full chunk.  Chunks of one tile and of two (then the tile before n - 2's is in the same chunk)."""
    n = 3 * T + r
    rng = np.random.default_rng(100 + r)
    for where, s in phantom_starts(n).items():
        k = 100
        lcp, _, _, bwt = phantom_input(rng, n, k, s)
        for m in (-1, 1, 2):
            es, el, enc = check_phantom(lcp, bwt, k, m)
            want, _, _ = H.emulate_shard(lcp, bwt, 0, n, k, m)
            for chunk in (T, 2 * T):
                sm, s_, l_, sh = stream_range(ctx, lcp, bwt, k, m, chunk)
                sh.close()
                summary_equals(sm, want, (r, where, m, chunk))
                S, Ls, mg = H.assemble([sm], [(s_, l_)])
                assert mg.n_clust_out == enc and np.array_equal(S, es) and np.array_equal(Ls, el), (r, where, m, chunk)


@pytest.mark.parametrize("n", [32769, 3 * T + 1])
def test_phantom_end_nm2_pipelines(ctx, reads, n, monkeypatch):
    """both tools in one call: e2s_pipeline_resident (its merge runs on the device, k_merge_stats) and e2s_pipeline_host
    streaming chunks of 16384 positions -- .clusters bytes, n_clust_out, candidates and .snp text"""
    rd, off = reads
    ctx.stage_reads(rd, off)
    rng = np.random.default_rng(7 * n)
    monkeypatch.setenv("E2S_CHUNK_POSITIONS", str(T))
    p = api.default_params(NR1)
    for where, s in phantom_starts(n).items():
        for k, m in ((100, 2), (100, 1), (130, 2)):
            lcp, text, suff, bwt = phantom_input(rng, n, k, s)
            es, el, enc = check_phantom(lcp, bwt, k, m)
            otext, ores, ost = oracle_snp(lcp, text, suff, bwt, es, el, rd, off)
            assert ores.n_candidates > 0
            sh = ctx.shard(n)
            sh.load_soa(lcp, text, suff, bwt)
            sh.seal()
            res = sh.pipeline_resident(p, k, m)
            assert sh.cluster_fetch_packed() == O.clusters_to_bytes(es, el), (n, where, k, m)
            assert (res.n_written, res.n_clust_out, res.max_clust_length) == (len(es), enc, ost.max_clust_length), (n, where, k, m)
            assert res.snp.n_candidates == ores.n_candidates and api.events_format(sh.events(), p) == otext, (n, where, k, m)
            sh.close()
            pipeline_host_equals_oracle(ctx, gesa(lcp, text, suff, bwt), lcp, text, suff, bwt, rd, off, k, m, (n, where, k, m))


# ---------------------------------------------------------------------------------------------------------------------------
# (b) long adopted records on chunked shards with the prefilter armed
# ---------------------------------------------------------------------------------------------------------------------------
def long_cluster_input(rng, n, lo, ln):
    """random small clusters (k = 16), SNP-like clusters on both sides of the middle, and one cluster [lo, lo + ln)"""
    lcp = H.random_lcp(rng, n, 16, 0)
    text, suff, bwt = index_arrays(rng, lcp)
    for a in (2000, 30000, n // 2 + 9000, n - 9000):
        plant_snp(rng, lcp, text, bwt, a, 24, 35)
    plant_cluster(lcp, lo, ln, 40)
    return lcp, text, suff, bwt


def two_chunked_shards(ctx, lcp, text, suff, bwt, cut, k, m, mcov):
    """both shards of [0, n) streamed in chunks of 16384 with the fused prefilter armed -> (summaries, records, shards)"""
    sums, recs, shards = [], [], []
    for lo, hi in ((0, cut), (cut, len(lcp))):
        sm, s, l, sh = stream_range(ctx, lcp, bwt, k, m, T, lo, hi, text=text, suff=suff, mcov=mcov)
        sums.append(sm)
        recs.append((s, l))
        shards.append(sh)
    return sums, recs, shards


@pytest.mark.parametrize("lo,ln", [(49500, 1000), (48000, 2500), (49800, 300)])
def test_adopted_long_record_chunked_shards(ctx, reads, lo, ln):
    """a cluster of 300..3000 positions that straddles the cut between two chunked shards is shard 1's head record, adopted
    by shard 0.  It starts in shard 0's last chunk (49152..50000) or in the chunk before; it is never analysed (longer than
    150), so it must neither fail the capture nor change the events"""
    rd, off = reads
    ctx.stage_reads(rd, off)
    n, cut, k, m = 120_000, 50_000, 16, 2
    rng = np.random.default_rng(lo)
    lcp, text, suff, bwt = long_cluster_input(rng, n, lo, ln)
    es, el, enc, _ = O.cluster_lm(lcp, bwt, k, m)
    assert ln in el.tolist()
    otext, ores, ost = oracle_snp(lcp, text, suff, bwt, es, el, rd, off)
    assert ores.n_candidates > 0
    p = api.default_params(NR1)
    sums, recs, shards = two_chunked_shards(ctx, lcp, text, suff, bwt, cut, k, m, p.mcov_out)
    S, Ls, mg = H.assemble(sums, recs)
    assert mg.n_clust_out == enc and np.array_equal(S, es) and np.array_equal(Ls, el)
    mg0 = api.cluster_merge(sums, 0)
    assert mg0.n_adopt >= 1 and ln in [mg0.adopt_len[i] for i in range(mg0.n_adopt)]
    texts, first_id, ncand, nanal = [], 1, 0, 0
    for g, sh in enumerate(shards):
        sh.cluster_finalize(api.cluster_merge(sums, g))
        cnt = sh.find_events(p, ost.max_clust_length)
        texts.append(api.events_format(sh.events(), p, first_id=first_id))
        first_id += cnt.n_events
        ncand += cnt.n_candidates
        nanal += cnt.n_analysed
        sh.close()
    assert (nanal, ncand) == (ores.n_analysed, ores.n_candidates) and b"".join(texts) == otext


def test_adopted_wrapped_record_chunked_shards(ctx, reads, monkeypatch):
    """a cluster of 65536 + 40 positions across the cut: its wrapped length (40) passes the filters, but its start left the
    device 4 chunks before the adopting shard's last one -- the chunk API refuses it cleanly; e2s_pipeline_host over the same
    eBWT as one range takes it on a resident shard and matches the oracle"""
    rd, off = reads
    ctx.stage_reads(rd, off)
    n, cut, k, m = 120_000, 50_000, 16, 2
    rng = np.random.default_rng(65576)
    lcp, text, suff, bwt = long_cluster_input(rng, n, 20_000, 65536 + 40)
    es, el, _, _ = O.cluster_lm(lcp, bwt, k, m)
    assert 40 in el.tolist()
    p = api.default_params(NR1)
    sums, recs, shards = two_chunked_shards(ctx, lcp, text, suff, bwt, cut, k, m, p.mcov_out)
    with pytest.raises(api.E2SError) as ei:
        shards[0].cluster_finalize(api.cluster_merge(sums, 0))
    assert ei.value.code == api.ERR_UNSUPPORTED
    for sh in shards:
        sh.close()
    monkeypatch.setenv("E2S_CHUNK_POSITIONS", str(T))
    pipeline_host_equals_oracle(ctx, gesa(lcp, text, suff, bwt), lcp, text, suff, bwt, rd, off, k, m, "wrapped")


@pytest.mark.parametrize("last_chunk", [5000, 1000])
def test_tail_rule_long_record_pipeline_host(ctx, reads, last_chunk, monkeypatch):
    """the last 3000 positions of the eBWT are one cluster: the tail rule writes it and the range adopts it.  It lies inside
    the last chunk of 5000 positions, or starts in the chunk before a last chunk of 1000"""
    rd, off = reads
    ctx.stage_reads(rd, off)
    n = 5 * T + last_chunk
    rng = np.random.default_rng(last_chunk)
    lcp, text, suff, bwt = long_cluster_input(rng, n, n - 3000, 2000)
    lcp[n - 3000:] = 40  # (open up to the last position: the tail rule closes it)
    es, el, _, _ = O.cluster_lm(lcp, bwt, 16, 2)
    assert es[-1] == n - 3000 and el[-1] >= 3000
    monkeypatch.setenv("E2S_CHUNK_POSITIONS", str(T))
    pipeline_host_equals_oracle(ctx, gesa(lcp, text, suff, bwt), lcp, text, suff, bwt, rd, off, 16, 2, last_chunk)


# ---------------------------------------------------------------------------------------------------------------------------
# (c) refused in a later chunk
# ---------------------------------------------------------------------------------------------------------------------------
def late_lcp_above_127():
    """the tiny dataset with LCP values 128..255 planted only at positions >= 2 * 16384"""
    rs, e = H.dataset("tiny", 4)
    n = e["n"]
    lcp = e["lcp"].copy()
    rng = np.random.default_rng(9)
    at = rng.integers(2 * T, n, size=n // 50)
    lcp[at] = rng.integers(128, 256, size=len(at))
    return rs, e, lcp


def wrapped_run():
    """the 65560-long run of test_wrapped_length_cluster_in_phase2 (wrapped length 24) and an ordinary cluster"""
    rng = np.random.default_rng(31)
    n = 200_000
    rd = ACGT[rng.integers(0, 4, size=(R, L))]
    lcp = np.zeros(n, dtype=np.uint32)
    lcp[5000:5000 + 65536 + 24] = 40
    lcp[150_000:150_030] = 35
    text = rng.integers(0, R, size=n).astype(np.uint32)
    suff = rng.integers(31, 60, size=n).astype(np.uint32)
    bwt = ACGT[rng.integers(0, 4, size=n)].copy()
    for lo_, hi_ in ((5000, 5024), (150_000, 150_030)):
        half = (hi_ - lo_) // 2
        text[lo_:lo_ + half] = rng.integers(0, NR1, size=half)
        bwt[lo_:lo_ + half] = ord("A")
        text[lo_ + half:hi_] = rng.integers(NR1, R, size=hi_ - lo_ - half)
        bwt[lo_ + half:hi_] = ord("C")
    return rd, lcp, text, suff, bwt


def soa_refused(ctx, lcp, text, suff, bwt, rd, off, nreads1, k, m):
    """e2s_pipeline_host_soa (no resident path): a clean E2S_ERR_UNSUPPORTED and no result claimed"""
    n = len(lcp)
    pair = np.empty(n, dtype=np.dtype([("suff", "<u4"), ("text", "<u4")]))
    pair["suff"], pair["text"] = suff, text
    pair = pair.view(np.uint8)
    lcp4 = np.ascontiguousarray(lcp, dtype=np.uint32)
    bwt = np.ascontiguousarray(bwt)
    bases = np.ascontiguousarray(rd).reshape(-1)
    off = np.ascontiguousarray(off, dtype=np.uint64)
    p = api.default_params(nreads1)
    rec10 = np.empty(1 << 20, dtype=np.uint8)
    res = api.PipelineResult()
    rc = ctx.lib.e2s_pipeline_host_soa(ctx.h, api._ptr(lcp4), 4, api._ptr(bwt), api._ptr(pair), 4, 4, n, api._ptr(bases),
                                       api._ptr(off), len(off) - 1, k, m, C.byref(p), api._ptr(rec10), len(rec10) // 10, None, 0,
                                       C.byref(res))
    assert rc == api.ERR_UNSUPPORTED, (rc, ctx.lib.e2s_last_error(ctx.h))
    assert (res.n_written, res.n_clust_out, res.max_clust_length, res.snp.n_candidates, res.snp.n_events) == (0, 0, 0, 0, 0)


def test_late_unsupported_pipeline_host(ctx, monkeypatch):
    """chunks of 16384 positions: the first chunks stream, a later one is refused -- e2s_pipeline_host starts again on a
    resident shard and matches the oracle; e2s_pipeline_host_soa refuses the input"""
    monkeypatch.setenv("E2S_CHUNK_POSITIONS", str(T))
    rs, e, lcp = late_lcp_above_127()
    off = O.uniform_read_offsets(*rs.reads.shape)
    ctx.stage_reads(rs.reads, off)
    k, m = 128, 2
    es, el, enc, _ = O.cluster_lm(lcp, e["bwt"], k, m)
    op = O.default_params(rs.nreads1)
    ost = O.statistics(es, el, op.mcov_out, op.pval)
    otext, ores = O.find_events(lcp, e["text"], e["suff"], e["bwt"], es, el, op, ost.max_clust_length, rs.reads, off, strict=False)
    p = api.default_params(rs.nreads1)
    eg = dict(e)
    eg["lcp"] = lcp
    rec = synth.gesa_records(eg).view(np.uint8).reshape(-1)
    rec10 = np.empty((len(es) + 16) * 10, dtype=np.uint8)
    evbuf = (api.Event * (ores.n_candidates + 16))()
    res = ctx.pipeline_host(rec, e["n"], rs.reads.reshape(-1), off, p, k, m, rec10=rec10, events=evbuf)
    assert res.n_written == len(es) and rec10[: len(es) * 10].tobytes() == O.clusters_to_bytes(es, el)
    assert (res.n_clust_out, res.max_clust_length) == (enc, ost.max_clust_length)
    assert (res.snp.n_analysed, res.snp.n_candidates, res.snp.n_events) == (ores.n_analysed, ores.n_candidates, ores.n_events)
    if otext is not None:
        assert api.events_format(list(evbuf)[: res.snp.n_variants], p) == otext
    soa_refused(ctx, lcp, e["text"], e["suff"], e["bwt"], rs.reads, off, rs.nreads1, k, m)

    rd, lcp, text, suff, bwt = wrapped_run()
    woff = O.uniform_read_offsets(R, L)
    ctx.stage_reads(rd, woff)
    es, el, _, _ = O.cluster_lm(lcp, bwt, 16, 2)
    assert 24 in el.tolist()
    pipeline_host_equals_oracle(ctx, gesa(lcp, text, suff, bwt), lcp, text, suff, bwt, rd, woff, 16, 2, "wrapped run")
    soa_refused(ctx, lcp, text, suff, bwt, rd, woff, NR1, 16, 2)


# ---------------------------------------------------------------------------------------------------------------------------
# (d) the CLI
# ---------------------------------------------------------------------------------------------------------------------------
def ebwt2clust(fa, k, m):
    env = dict(os.environ, E2S_CHUNK_POSITIONS=str(T))
    r = subprocess.run([os.path.join(BIN, "ebwt2clust"), "-i", fa, "-k", str(k), "-m", str(m), "-x", "4", "-y", "4", "-z", "4"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr
    done = [ln for ln in r.stdout.splitlines() if ln.startswith("Done. ")]
    assert len(done) == 1, r.stdout
    return open(fa + ".clusters", "rb").read(), int(done[0].split()[1])


def test_cli_range_edges(ctx, reads, tmp_path):
    """ebwt2clust streaming chunks of 16384 positions: the END at n - 2 of an n = 2 * 16384 + 1 eBWT, and LCP values above
    127 first met in a later chunk under -k 128 (the CLI takes the whole range on a resident shard)"""
    rd, _ = reads
    rng = np.random.default_rng(32769)
    n = 2 * T + 1
    for where, s in phantom_starts(n).items():
        for m in (1, 2):
            lcp, text, suff, bwt = phantom_input(rng, n, 100, s)
            es, el, enc = check_phantom(lcp, bwt, 100, m)
            rs = synth.ReadSet(reads=rd, nreads1=NR1, genome1=None, genome2=None, snp_pos=None, indels=[])
            fa = synth.write_dataset(str(tmp_path / f"{where}{m}"), rs, {"n": n, "lcp": lcp, "text": text, "suff": suff, "bwt": bwt})
            cl, done = ebwt2clust(fa, 100, m)
            assert cl == O.clusters_to_bytes(es, el) and done == enc, (where, m)
    rs, e, lcp = late_lcp_above_127()
    eg = dict(e)
    eg["lcp"] = lcp
    fa = synth.write_dataset(str(tmp_path / "late127"), rs, eg)
    es, el, enc, _ = O.cluster_lm(lcp, e["bwt"], 128, 2)
    cl, done = ebwt2clust(fa, 128, 2)
    assert cl == O.clusters_to_bytes(es, el) and done == enc

"""-m gpu: repeated calls on reused shards, contexts and chunked ranges against the oracle.

The benchmark times many steps on one resident shard, the streamed pipelines reuse the context's cached shard, the C4 loop
resets one chunked shard between passes, and a sharded job reruns the phases on the same shards every step.  Every call
here is compared with the oracle, not only the first: .clusters bytes, n_written / n_clust_out / max_clust_length,
n_analysed / n_candidates / n_events and the .snp text.

(A) e2s_pipeline_resident repeated on one shard, options changed and changed back, plain calls and capacity retries in between;
    launch counts say which scan ran.
(B) three fused shards of one index (cut through clusters: adopted records) rerun three times.
(C) one resident shard reloaded with another index of the same n through every loader, whole and in pieces; the seal
    verdict (an LCP value above 127) follows the data.
(D) e2s_pipeline_host / e2s_pipeline_host_soa in sequence on one context (its cached shard); a fresh context whose first
    streamed call is the lean one, then .gesa loads.
(E) one chunked shard over several passes with e2s_chunked_reset: scan passes, an abandoned pass, a clust2snp pass, lean;
    E2S_SCAN_LEGACY, which a chunked shard does not follow.
(F) a one-rank NCCL communicator: e2s_pipeline_sharded (with and without E2S_NO_FUSED_PREFILTER, which it ignores) and
    e2s_chunked_exchange repeated; e2s_pipeline_host_sharded under two chunk sizes.
(G) reads restaged between steps: bigger, smaller, with non-ACGT bytes, ragged.
"""
import os

import numpy as np
import pytest

from ebwt2snp_b200 import api, synth
from oracle import oracle as O
from tests import helpers as H
from tests import phase2_cases as P

pytestmark = pytest.mark.gpu

T = 16384
TAIL = 40  # the planted cluster at the end of the eBWT: written by the tail rule, adopted by the last shard


@pytest.fixture(scope="module")
def ctx(built):
    c = api.Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------------------------------------------------------------------
# data: the tiny dataset (1 616 000 positions whatever the seed), with planted LCP values above 127 and a cluster at the end
# ---------------------------------------------------------------------------------------------------------------------------
class Data:
    def __init__(self, name, lcp, text, suff, bwt, reads, nreads1):
        self.name, self.lcp, self.text, self.suff, self.bwt = name, lcp, text, suff, bwt
        self.reads, self.nreads1 = reads, nreads1
        self.off = O.uniform_read_offsets(*reads.shape)

    @property
    def n(self):
        return len(self.lcp)

    def eg(self):
        return dict(n=self.n, lcp=self.lcp, text=self.text, suff=self.suff, bwt=self.bwt)

    def cut(self, n):
        """the first n positions: an eBWT of its own for both tools"""
        return Data(f"{self.name}[:{n}]", self.lcp[:n], self.text[:n], self.suff[:n], self.bwt[:n], self.reads, self.nreads1)


_DATA = {}


def data(seed, hi=None, tail=False):
    """hi: None, "all" (runs of LCP values 128..255 everywhere) or (lo, hi) (only in that range of positions)"""
    key = (seed, str(hi), tail)
    if key not in _DATA:
        rs, e = H.dataset("tiny", seed)
        lcp, text, suff, bwt = (e[f].copy() for f in ("lcp", "text", "suff", "bwt"))
        n = len(lcp)
        rng = np.random.default_rng(1000 + seed)
        if hi is not None:
            lo_, hi_ = (1000, n - 1000) if hi == "all" else hi
            for a in rng.integers(lo_, hi_ - 8, size=max(4, (hi_ - lo_) // 2000)):
                lcp[a:a + 6] = rng.integers(128, 256, size=6)
        if tail:  # SNP-like: sample 1's records all 'A', sample 2's all 'C', contexts inside the reads
            lcp[n - TAIL - 1] = 0
            lcp[n - TAIL:] = 40
            h = TAIL // 2
            R = rs.reads.shape[0]
            text[n - TAIL:n - h] = rng.integers(0, rs.nreads1, size=TAIL - h)
            text[n - h:] = rng.integers(rs.nreads1, R, size=h)
            suff[n - TAIL:] = rng.integers(31, 60, size=TAIL)
            bwt[n - TAIL:n - h] = ord("A")
            bwt[n - h:] = ord("C")
        _DATA[key] = Data(f"tiny{seed}{'' if hi is None else '-hi' + str(hi)}{'-tail' if tail else ''}", lcp, text, suff, bwt,
                          rs.reads, rs.nreads1)
    return _DATA[key]


class Want:
    def __init__(self, es, el, enc, mcl, text, res):
        self.es, self.el, self.enc, self.mcl, self.text, self.res = es, el, enc, mcl, text, res
        self.clusters = O.clusters_to_bytes(es, el)


_WANT = {}


def want(d, k=16, m=2, mcov=5, xyz=(4, 4, 4), bcr=False, phase1=False) -> Want:
    """the oracle's outputs (phase1: ebwt2clust only)"""
    key = (d.name, k, m, mcov, xyz, bcr, phase1)
    if key not in _WANT:
        x, y, z = xyz
        es, el, enc, _ = O.cluster_lm(d.lcp, d.bwt, k, m, x=x)
        if phase1:
            _WANT[key] = Want(es, el, enc, None, None, None)
        else:
            op = O.default_params(d.nreads1, mcov_out=mcov)
            st = O.statistics(es, el, mcov, op.pval)
            text, res = O.find_events(d.lcp, d.text, d.suff, d.bwt, es, el, op, st.max_clust_length, d.reads, d.off, x=x, y=y, z=z,
                                      bcr=bcr)
            _WANT[key] = Want(es, el, enc, st.max_clust_length, text, res)
    return _WANT[key]


def params(d, mcov=5):
    return api.default_params(d.nreads1, mcov_out=mcov)


def check_counts(cnt, w, what):
    got = (cnt.n_analysed, cnt.n_candidates, cnt.n_events)
    assert got == (w.res.n_analysed, w.res.n_candidates, w.res.n_events), (what, got)


def check_step(sh, res, d, w, mcov, what):
    """an e2s_pipeline_resident result and what the shard holds afterwards"""
    assert (res.n_written, res.n_clust_out, res.max_clust_length) == (len(w.es), w.enc, w.mcl), what
    check_counts(res.snp, w, what)
    assert sh.cluster_fetch_packed() == w.clusters, what
    assert api.events_format(sh.events(), params(d, mcov)) == w.text, what


def step(sh, d, k=16, m=2, mcov=5, what=""):
    res = sh.pipeline_resident(params(d, mcov), k, m)
    check_step(sh, res, d, want(d, k, m, mcov), mcov, (what, d.name, k, m, mcov))
    return res


def two_phase(sh, d, k=16, m=2, mcov=5, what=""):
    """cluster_lm -> statistics -> find_events on the same shard"""
    w = want(d, k, m, mcov)
    nw, nc = sh.cluster_lm(k, m)
    assert (nw, nc) == (len(w.es), w.enc) and sh.cluster_fetch_packed() == w.clusters, what
    st = sh.statistics(mcov, 0.99)
    assert st.max_clust_length == w.mcl, what
    cnt = sh.find_events(params(d, mcov), st.max_clust_length)
    check_counts(cnt, w, what)
    assert api.events_format(sh.events(), params(d, mcov)) == w.text, what


def find_only(sh, d, k, m, mcov, what):
    """find_events with another -m on the records the last step left (the two-phase pass over the record list)"""
    w = want(d, k, m, mcov)
    st = sh.statistics(mcov, 0.99)
    assert st.max_clust_length == w.mcl, what
    cnt = sh.find_events(params(d, mcov), st.max_clust_length)
    check_counts(cnt, w, what)
    assert api.events_format(sh.events(), params(d, mcov)) == w.text, what


def drain(ctx):
    for kk in range(9):
        ctx.kernel_time(kk)


def scans(ctx):
    """(k_cluster_scan launches, k_lcp_flags launches) since the last call; the other timers are emptied as well"""
    s1, fl = ctx.kernel_time(api.KERNEL_SCAN1)[1], ctx.kernel_time(api.KERNEL_FLAGS)[1]
    drain(ctx)
    return s1, fl


def path(ctx, one_pass):
    """which scan ran since the last call (a capacity retry runs it twice)"""
    s1, fl = scans(ctx)
    assert (s1 > 0, fl > 0) == (one_pass, not one_pass), (s1, fl)


def one_pass_expected(d, k, m):
    """one_pass_ok: the byte LCP compares exactly for k <= 127, and for any k when no value above 127 was loaded; -m <= 33"""
    return m <= 33 and (k <= 127 or int(d.lcp.max()) <= 127)


def resident(ctx, d):
    sh = ctx.shard(d.n)
    sh.load_soa(d.lcp, d.text, d.suff, d.bwt)
    sh.seal()
    return sh


# ---------------------------------------------------------------------------------------------------------------------------
# (A) resident steps, repeated
# ---------------------------------------------------------------------------------------------------------------------------
def test_resident_steps_repeated(ctx, monkeypatch):
    d = data(1, hi="all", tail=True)
    assert int(d.lcp.max()) > 127 and want(d).es[-1] == d.n - TAIL  # (the tail rule writes the planted cluster)
    assert want(d, m=34).es[-1] == d.n - TAIL
    ctx.stage_reads(d.reads, d.off)
    sh = resident(ctx, d)
    ctx.timing(True)
    try:
        drain(ctx)
        first = None
        for i in range(5):
            res = step(sh, d, what=f"repeat {i}")
            if i:
                assert scans(ctx) == (1, 0), i  # (the first step on a fresh shard may grow its buffers and scan again)
            else:
                path(ctx, True)
            got = (bytes(res), sh.cluster_fetch_packed(), api.events_format(sh.events(), params(d)))
            assert first is None or got == first, i
            first = got
        for mcov in (3, 8, 5):
            step(sh, d, mcov=mcov, what="mcov")
            path(ctx, True)
        # -m 34: k_lcp_flags + k_cluster_emit on the same shard; then the one-pass scan again
        for m in (34, 2):
            step(sh, d, m=m, what="-m")
            path(ctx, one_pass_expected(d, 16, m))
        # -k 128 over LCP values above 127: the 4-byte stream
        for k in (128, 16):
            step(sh, d, k=k, what="-k")
            path(ctx, one_pass_expected(d, k, 2))
        assert not one_pass_expected(d, 128, 2)
        for fused in (False, True, False):
            if fused:
                monkeypatch.delenv("E2S_NO_FUSED_PREFILTER", raising=False)
            else:
                monkeypatch.setenv("E2S_NO_FUSED_PREFILTER", "1")
            step(sh, d, what=f"fused={fused}")
            path(ctx, True)
        monkeypatch.delenv("E2S_NO_FUSED_PREFILTER")
        # plain calls between the steps: the two-phase path walks the record list (own records + the adopted tail record)
        two_phase(sh, d, what="two-phase after steps")
        step(sh, d, what="after two-phase")
        find_only(sh, d, 16, 2, 6, "other -m after a step")
        s, ln = sh.cluster_fetch()
        assert np.array_equal(s, want(d).es) and np.array_equal(ln, want(d).el)
        step(sh, d, m=34, what="-m 34 after the record list got the adopted record")
        find_only(sh, d, 16, 34, 6, "other -m after a -m 34 step")
        step(sh, d, what="back")
        find_only(sh, d, 16, 2, 6, "other -m, again")
        drain(ctx)
        # capacity retries, then the hooks removed
        monkeypatch.setenv("E2S_PF_CAPACITY", "3")
        step(sh, d, what="E2S_PF_CAPACITY")
        monkeypatch.delenv("E2S_PF_CAPACITY")
        for i in range(2):
            step(sh, d, what=f"after E2S_PF_CAPACITY {i}")
        monkeypatch.setenv("E2S_SNP_FIRST_CAPACITY", "1")
        step(sh, d, mcov=3, what="E2S_SNP_FIRST_CAPACITY")
        monkeypatch.delenv("E2S_SNP_FIRST_CAPACITY")
        for mcov in (3, 5):
            step(sh, d, mcov=mcov, what="after E2S_SNP_FIRST_CAPACITY")
    finally:
        ctx.timing(False)
        drain(ctx)
        sh.close()


# ---------------------------------------------------------------------------------------------------------------------------
# (B) emulated shards, repeated
# ---------------------------------------------------------------------------------------------------------------------------
def test_fused_shards_rerun(ctx):
    d = data(3, tail=True)
    n = d.n
    w5 = want(d)
    # cuts through analysable clusters at a third and two thirds: the next shard's head record is adopted
    big = np.flatnonzero((w5.el >= 12) & (w5.el <= 150))
    cuts = [0] + [int(w5.es[j] + w5.el[j] // 2) for j in (big[len(big) // 3], big[2 * len(big) // 3])] + [n]
    ctx.stage_reads(d.reads, d.off)
    shards = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        sh = ctx.shard(hi - lo, lo, n)
        a, b = max(0, lo - 2), min(n, hi + 151)
        sh.load_soa(d.lcp[a:b], d.text[a:b], d.suff[a:b], d.bwt[a:b], first=a)
        sh.seal()
        shards.append(sh)
    try:
        for rnd, mcov in enumerate((5, 3, 5)):
            w = want(d, mcov=mcov)
            p = params(d, mcov)
            sums, recs = [], []
            for sh in shards:
                sh.cluster_prefilter(mcov)
                sums.append(sh.cluster_run(16, 2))
                recs.append(sh.cluster_fetch())  # (own records: nothing merged yet)
            S, L, mg = H.assemble(sums, recs)
            assert mg.n_clust_out == w.enc and np.array_equal(S, w.es) and np.array_equal(L, w.el), rnd
            mgs = [api.cluster_merge(sums, g) for g in range(len(shards))]
            assert sum(mg.n_adopt for mg in mgs[:-1]) >= 2 and mgs[-1].n_adopt >= 1
            texts, first_id, tot = [], 1, np.zeros(3, dtype=np.int64)
            for sh, mg in zip(shards, mgs):
                sh.cluster_finalize(mg)
                cnt = sh.find_events(p, w.mcl)
                texts.append(api.events_format(sh.events(), p, first_id=first_id))
                first_id += cnt.n_events
                tot += (cnt.n_analysed, cnt.n_candidates, cnt.n_events)
            assert b"".join(sh.cluster_fetch_packed() for sh in shards) == w.clusters, rnd  # head + own + tail, shard by shard
            assert tuple(tot) == (w.res.n_analysed, w.res.n_candidates, w.res.n_events), rnd
            assert b"".join(texts) == w.text, rnd
    finally:
        for sh in shards:
            sh.close()


# ---------------------------------------------------------------------------------------------------------------------------
# (C) reloading a resident shard
# ---------------------------------------------------------------------------------------------------------------------------
# gesa_fd: the .gesa file through e2s_shard_load_gesa_fd, which loads it in pieces of 2^20 records (the tiny index is larger)
LOADERS = [("soa", (4, 4, 4)), ("gesa", (4, 4, 4)), ("gesa", (1, 4, 1)), ("gesa", (8, 8, 8)), ("gesa_fd", (4, 4, 4)),
           ("bcr", (4, 4, 4))]


@pytest.fixture(scope="module")
def gesa_file(tmp_path_factory):
    """-> path of the .gesa file of (data, xyz), written once"""
    d0 = tmp_path_factory.mktemp("gesa")
    made = {}

    def get(d, xyz):
        key = (d.name, xyz)
        if key not in made:
            made[key] = str(d0 / f"{len(made)}.gesa")
            synth.write_gesa(made[key], d.eg(), *xyz)
        return made[key]
    return get


def pieces(n, rng):
    """5..9 pieces of [0, n) in shuffled order, cuts off every power-of-two grid, two of one position, one loaded twice"""
    cuts = set()
    while len(cuts) < int(rng.integers(2, 6)):
        c = int(rng.integers(100, n - 100))
        if c % 16:
            cuts.add(c)
    one = int(rng.integers(1000, n - 1000)) | 1
    cuts |= {one, one + 1, n - 1}
    b = sorted(cuts | {0, n})
    out = list(zip(b[:-1], b[1:]))
    assert 5 <= len(out) <= 9 and sum(1 for a, c in out if c - a == 1) >= 2
    rng.shuffle(out)
    out.append(out[len(out) // 2])
    return out


def load(sh, d, kind, xyz, a, b, gesa_file):
    x, y, z = xyz
    if kind == "gesa_fd":
        fd = os.open(gesa_file(d, xyz), os.O_RDONLY)
        try:
            sh.load_gesa_fd(fd, a, b - a, x, y, z)
            sh.ctx.synchronize()
        finally:
            os.close(fd)
    elif kind == "soa":
        sh.load_soa(d.lcp[a:b], d.text[a:b], d.suff[a:b], d.bwt[a:b], first=a)
    elif kind == "gesa":
        rec = synth.gesa_records(d.eg(), x, y, z).view(np.uint8).reshape(-1)
        rs = x + y + z + 1
        sh.load_gesa(rec[a * rs:b * rs], first=a, count=b - a, x=x, y=y, z=z)
    else:
        lcp = np.ascontiguousarray(d.lcp.astype(f"<u{x}")).view(np.uint8)
        pair = np.empty(d.n, dtype=np.dtype([("suff", f"<u{z}"), ("text", f"<u{y}")]))
        pair["suff"], pair["text"] = d.suff, d.text
        pair = pair.view(np.uint8)
        sh.load_bcr(lcp[a * x:b * x], d.bwt[a:b], pair[a * (y + z):b * (y + z)], x, y, z, first=a)


@pytest.mark.parametrize("kind,xyz", LOADERS, ids=[f"{k}{''.join(map(str, x))}" for k, x in LOADERS])
@pytest.mark.parametrize("hi_first", [True, False], ids=["hi-then-clean", "clean-then-hi"])
def test_resident_reload(ctx, kind, xyz, hi_first, gesa_file):
    dh, dc = data(2, hi="all"), data(4)
    assert dh.n == dc.n and int(dh.lcp.max()) > 127 >= int(dc.lcp.max())
    # whole / in pieces; every order ends with a whole reload whose LCP holds no value above 127 after one that held some
    seq = [(dh, True), (dc, False), (dh, False), (dc, True)] if hi_first else [(dc, True), (dh, False), (dc, True), (dh, True)]
    bcr = kind == "bcr"
    ctx.stage_reads(dh.reads, dh.off)  # (phase 2 of each step stages its own reads below)
    rng = np.random.default_rng(sum(xyz) + 7 * hi_first + len(kind))
    sh = ctx.shard(dh.n)
    ctx.timing(True)
    try:
        for i, (d, whole) in enumerate(seq):
            for a, b in ([(0, d.n)] if whole else pieces(d.n, rng)):
                load(sh, d, kind, xyz, a, b, gesa_file)
            sh.seal()
            ctx.stage_reads(d.reads, d.off)
            what = (kind, xyz, i, d.name, whole)
            drain(ctx)
            w = want(d, xyz=xyz, bcr=bcr)
            res = sh.pipeline_resident(params(d), 16, 2)
            check_step(sh, res, d, w, 5, what)
            path(ctx, True)
            w1 = want(d, k=128, xyz=xyz, phase1=True)
            nw, nc = sh.cluster_lm(128, 2)
            assert (nw, nc) == (len(w1.es), w1.enc) and sh.cluster_fetch_packed() == w1.clusters, what
            s1, fl = scans(ctx)
            if int(d.lcp.max()) > 127:
                assert (s1, fl) == (0, 1), what  # the saturated byte copy cannot answer lcp >= 128
            elif whole:
                assert (s1, fl) == (1, 0), what  # a whole reload without a value above 127: the one-pass scan again
    finally:
        ctx.timing(False)
        drain(ctx)
        sh.close()


# ---------------------------------------------------------------------------------------------------------------------------
# (D) the context's cached shard
# ---------------------------------------------------------------------------------------------------------------------------
def host_call(ctx, d, soa=False, k=16, m=2, mcov=5):
    w = want(d, k, m, mcov)
    p = params(d, mcov)
    rec10 = np.empty((len(w.es) + 16) * 10, dtype=np.uint8)
    evbuf = (api.Event * (w.res.n_candidates + 16))()
    if soa:
        pair = np.empty(d.n, dtype=np.dtype([("suff", "<u4"), ("text", "<u4")]))
        pair["suff"], pair["text"] = d.suff, d.text
        res = ctx.pipeline_host_soa(np.ascontiguousarray(d.lcp).view(np.uint8), d.bwt, pair.view(np.uint8), d.n, d.reads.reshape(-1),
                                    d.off, p, k, m, rec10=rec10, events=evbuf)
    else:
        rec = synth.gesa_records(d.eg()).view(np.uint8).reshape(-1)
        res = ctx.pipeline_host(rec, d.n, d.reads.reshape(-1), d.off, p, k, m, rec10=rec10, events=evbuf)
    what = ("soa" if soa else "host", d.name, k, m, mcov)
    assert res.n_written == len(w.es) and rec10[:len(w.es) * 10].tobytes() == w.clusters, what
    assert (res.n_clust_out, res.max_clust_length) == (w.enc, w.mcl), what
    check_counts(res.snp, w, what)
    assert api.events_format(list(evbuf)[:res.snp.n_variants], p) == w.text, what


def test_cached_shard_sequence(ctx, monkeypatch):
    A, B = data(1), data(2)
    late = data(4, hi=(2 * T, data(4).n))
    chunk = {None: None, "16k": str(T), "100003": "100003"}

    def env(c):
        if chunk[c] is None:
            monkeypatch.delenv("E2S_CHUNK_POSITIONS", raising=False)
        else:
            monkeypatch.setenv("E2S_CHUNK_POSITIONS", chunk[c])

    env("16k")
    host_call(ctx, A)
    host_call(ctx, B)
    host_call(ctx, B, soa=True)
    host_call(ctx, A)  # (pipeline_host_soa must not have left its pairSA on the cached shard)
    host_call(ctx, A.cut(A.n - 12345))
    host_call(ctx, A)
    for c in ("100003", None, "16k"):
        env(c)
        host_call(ctx, B)
        host_call(ctx, A, soa=True)
    host_call(ctx, A, m=34)  # a resident shard in between
    host_call(ctx, B)
    host_call(ctx, A, m=34)
    host_call(ctx, A, m=34, mcov=3)
    host_call(ctx, B)
    # refused in a later chunk by the lean pipeline, then a normal call
    pair = np.zeros(late.n, dtype=np.uint64).view(np.uint8)
    with pytest.raises(api.E2SError) as ei:
        ctx.pipeline_host_soa(np.ascontiguousarray(late.lcp).view(np.uint8), late.bwt, pair, late.n, late.reads.reshape(-1), late.off,
                              params(late), 128, 2)
    assert ei.value.code == api.ERR_UNSUPPORTED
    host_call(ctx, B)
    # e2s_pipeline_host falls back to a resident shard for it.  With E2S_NO_FUSED_PREFILTER the calls below go to that cached
    # shard directly (pipeline_host_resident), reloaded each time from the first record: at -k 128 the scan must follow the
    # data -- the 4-byte stream over LCP values above 127, the one-pass scan over an index without any.
    host_call(ctx, late, k=128)
    monkeypatch.setenv("E2S_NO_FUSED_PREFILTER", "1")
    ctx.timing(True)
    try:
        drain(ctx)
        host_call(ctx, late, k=128)
        path(ctx, False)
        # an index whose LCP values all lie below 128 has no cluster at -k 128, so clust2snp refuses it as the reference does
        # (its statistics divide by zero) -- after the scan, which is what is checked here; ebwt2clust's output (no record) is
        # compared with the oracle on a resident shard in test_resident_reload
        assert len(want(A, k=128, phase1=True).es) == 0
        rec = synth.gesa_records(A.eg()).view(np.uint8).reshape(-1)
        with pytest.raises(api.E2SError) as ei:
            ctx.pipeline_host(rec, A.n, A.reads.reshape(-1), A.off, params(A), 128, 2, rec10=np.empty(160, dtype=np.uint8))
        assert ei.value.code == api.ERR_UNSUPPORTED and "no clusters" in str(ei.value)
        path(ctx, True)  # the reloaded cached shard forgot the old LCP > 127 verdict
        host_call(ctx, late, k=128)
        path(ctx, False)
        host_call(ctx, A)
        path(ctx, True)
    finally:
        ctx.timing(False)
        drain(ctx)
    monkeypatch.delenv("E2S_NO_FUSED_PREFILTER")
    host_call(ctx, B)


def test_fresh_context_lean_first(built, gesa_file):
    """A context whose first streamed call is the lean pipeline: the .gesa loads after it (e2s_pipeline_host's chunks, a
    resident shard loaded from a file descriptor) use the copy stream it made and the events they share with it."""
    d = data(1)
    c = api.Context(0)
    try:
        host_call(c, d, soa=True)
        host_call(c, d)
        sh = c.shard(d.n)
        try:
            load(sh, d, "gesa_fd", (4, 4, 4), 0, d.n, gesa_file)
            sh.seal()
            step(sh, d, what="resident from a file descriptor after the streamed calls")
        finally:
            sh.close()
    finally:
        c.close()


# ---------------------------------------------------------------------------------------------------------------------------
# (E) one chunked shard over several passes (the C4 loop)
# ---------------------------------------------------------------------------------------------------------------------------
CHUNK_E = 20 * T  # 5 chunks of the tiny dataset (1 616 000 positions)


def lean_arrays(d):
    pair = np.empty(d.n, dtype=np.dtype([("suff", "<u1"), ("text", "<u4")]))
    pair["suff"], pair["text"] = d.suff, d.text
    return d.lcp.astype(np.uint8), pair.view(np.uint8)


def load_chunk(sh, d, clo, cn, lean):
    a, b = max(0, clo - 176), min(d.n, clo + cn + 152)
    if lean:
        lcp1, _ = lean_arrays(d)
        sh.load_bcr(lcp1[a:b], d.bwt[a:b], None, 1, 4, 1, first=a)
        sh.set_layout(1, 4, 1, True)
    else:
        sh.load_soa(d.lcp[a:b], d.text[a:b], d.suff[a:b], d.bwt[a:b], first=a)


def scan_pass(sh, d, k=16, m=2, mcov=5, lean=False, stop_after=None, after_scan=None):
    """chunk_begin / load / chunk_scan over the range, the records fetched chunk by chunk; then finish -> merge -> finalize ->
    statistics -> find_events, all compared with the oracle.  stop_after: abandon the pass after that many chunks; after_scan:
    called after each chunk's scan"""
    w = want(d, k, m, mcov, xyz=(1, 4, 1) if lean else (4, 4, 4), bcr=lean)
    p = params(d, mcov)
    keep = None
    if lean:
        keep = lean_arrays(d)
        sh.host_gsa(keep[1], 4, 1)
    recs = []
    for i, (clo, cn) in enumerate(sh.chunks()):
        if i == stop_after:
            return
        sh.chunk_begin(clo, cn)
        load_chunk(sh, d, clo, cn, lean)
        m_ = sh.chunk_scan(k, m, mcov)
        if after_scan:
            after_scan()
        recs.append(sh.cluster_fetch_packed())
        assert len(recs[-1]) == 10 * m_
    sm = sh.chunked_finish(k, m)
    mg = api.cluster_merge([sm], 0)
    sh.cluster_finalize(mg)
    tail = O.clusters_to_bytes(np.array(mg.append_start[:mg.n_append], dtype=np.uint64), np.array(mg.append_len[:mg.n_append], dtype=np.uint16))
    what = (d.name, k, m, mcov, lean)
    assert b"".join(recs) + tail == w.clusters and mg.n_clust_out == w.enc and mg.total_written == len(w.es), what
    st, ost = sh.statistics(mcov, 0.99), O.statistics(w.es, w.el, mcov, 0.99)
    assert list(st.hist) == list(ost.hist) and (st.n_clust, st.n_bases) == (ost.n_clust, ost.n_bases), what
    assert st.max_clust_length == w.mcl, what
    cnt = sh.find_events(p, st.max_clust_length)
    check_counts(cnt, w, what)
    assert api.events_format(sh.events(), p) == w.text, what
    del keep


def stage_pass(sh, d, mcov=5):
    """clust2snp on the chunked shard: the .clusters records of each chunk staged, phase 2 on the captured survivors"""
    w = want(d, mcov=mcov)
    p = params(d, mcov)
    rec10 = np.frombuffer(w.clusters, dtype=np.uint8)
    for clo, cn in sh.chunks():
        sh.chunk_begin(clo, cn)
        load_chunk(sh, d, clo, cn, False)
        r0, r1 = np.searchsorted(w.es, clo), np.searchsorted(w.es, clo + cn)
        sh.chunk_stage_clusters(rec10[r0 * 10:r1 * 10], mcov, w.mcl)
    sh.chunked_clusters_finish()
    cnt = sh.find_events(p, w.mcl)
    check_counts(cnt, w, ("staged", d.name))
    assert api.events_format(sh.events(), p) == w.text, ("staged", d.name)


def test_chunked_reset_passes(ctx):
    A, B, C = data(1, tail=True), data(2), data(3)
    mid = data(4, hi=(2 * CHUNK_E + 100, 3 * CHUNK_E - 100))
    assert A.n == B.n == C.n == mid.n
    sh = ctx.shard(A.n, 0, A.n, chunk_positions=CHUNK_E)
    assert len(list(sh.chunks())) == 5

    def run(d, **kw):
        ctx.stage_reads(d.reads, d.off)
        sh.chunked_reset()
        scan_pass(sh, d, **kw)

    try:
        ctx.stage_reads(A.reads, A.off)
        scan_pass(sh, A)  # (a fresh shard: no reset before the first pass)
        run(B)
        run(C, mcov=3)
        run(A)
        # abandoned after 2 of 5 chunks
        sh.chunked_reset()
        scan_pass(sh, B, stop_after=2)
        run(A)
        # clust2snp's streamed mode between two scan passes
        sh.chunked_reset()
        ctx.stage_reads(B.reads, B.off)
        stage_pass(sh, B)
        run(C)
        # lean, then not lean (the caller takes its pairSA back)
        run(A, lean=True)
        sh.host_gsa(None, 4, 4)
        run(B)
        # an LCP value above 127 in the middle chunk under -k 16, then a pass without
        run(mid)
        run(C)
        run(A)
    finally:
        sh.close()


def test_chunked_scan_legacy_hook(ctx, monkeypatch):
    """E2S_SCAN_LEGACY=1 forces K1 + K2 on resident shards only: a chunked shard keeps the one-pass scan, which writes each
    chunk's records to its segments and starts from the open-cluster state the chunks before it left"""
    d = data(1, tail=True)
    monkeypatch.setenv("E2S_SCAN_LEGACY", "1")
    sh = ctx.shard(d.n, 0, d.n, chunk_positions=CHUNK_E)
    assert len(list(sh.chunks())) == 5
    ctx.stage_reads(d.reads, d.off)
    ctx.timing(True)
    try:
        drain(ctx)
        for i, m in enumerate((2, 33)):
            if i:
                sh.chunked_reset()
            scan_pass(sh, d, m=m, after_scan=lambda: path(ctx, True))
    finally:
        ctx.timing(False)
        drain(ctx)
        sh.close()


def test_chunked_reset_second_shard(ctx):
    """the last shard [cut, n) of two, streamed as one chunk that starts inside a cluster (a head END): after a pass that ended
    with a cluster open at the end of the eBWT, e2s_chunked_reset must bring the open-cluster state back to "unknown" (an
    earlier shard decides), or the next pass closes the stale open cluster at that head END"""
    d = data(1, tail=True)
    n = d.n
    w = want(d)
    j = int(np.searchsorted(w.es, n - 50_000))
    j += int(np.argmax(w.el[j:] >= 12))
    cut = int(w.es[j] + w.el[j] // 2)  # (range_n < 65 536: one chunk, every wrapped length stays long)
    ctx.stage_reads(d.reads, d.off)
    p = params(d)
    sh0 = ctx.shard(cut, 0, n)
    sh0.load_soa(d.lcp[:cut + 151], d.text[:cut + 151], d.suff[:cut + 151], d.bwt[:cut + 151])
    sh0.seal()
    sh1 = ctx.shard(n - cut, cut, n, chunk_positions=n - cut)
    try:
        for rnd in range(3):
            if rnd:
                sh1.chunked_reset()
            sh0.cluster_prefilter(5)
            sums = [sh0.cluster_run(16, 2)]
            recs = [sh0.cluster_fetch()]
            (clo, cn), = list(sh1.chunks())
            sh1.chunk_begin(clo, cn)
            load_chunk(sh1, d, clo, cn, False)
            sh1.chunk_scan(16, 2, 5)
            recs.append(sh1.cluster_fetch())
            sums.append(sh1.chunked_finish(16, 2))
            assert sums[1].head_end, rnd
            S, L, mg = H.assemble(sums, recs)
            assert mg.n_clust_out == w.enc and np.array_equal(S, w.es) and np.array_equal(L, w.el), rnd
            texts, first_id, tot = [], 1, np.zeros(3, dtype=np.int64)
            for g, sh in enumerate((sh0, sh1)):
                sh.cluster_finalize(api.cluster_merge(sums, g))
                cnt = sh.find_events(p, w.mcl)
                texts.append(api.events_format(sh.events(), p, first_id=first_id))
                first_id += cnt.n_events
                tot += (cnt.n_analysed, cnt.n_candidates, cnt.n_events)
            assert tuple(tot) == (w.res.n_analysed, w.res.n_candidates, w.res.n_events) and b"".join(texts) == w.text, rnd
    finally:
        sh0.close()
        sh1.close()


# ---------------------------------------------------------------------------------------------------------------------------
# (F) one-rank NCCL step
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def comm(ctx):
    try:
        cm = api.Comm(ctx, 0, 1, lambda b: b)
    except api.E2SError as e:
        pytest.skip(f"no one-rank communicator on this machine: {e}")
    yield cm
    cm.close()


def test_one_rank_sharded_steps(ctx, comm, monkeypatch):
    A, B = data(1, tail=True), data(2)
    ctx.stage_reads(A.reads, A.off)
    sh = resident(ctx, A)
    ctx.timing(True)
    try:
        # E2S_NO_FUSED_PREFILTER keeps the phases of the resident step apart, not those of the sharded step
        for no_fused in (False, True):
            if no_fused:
                monkeypatch.setenv("E2S_NO_FUSED_PREFILTER", "1")
            for i, mcov in enumerate((5, 3, 5)):
                w = want(A, mcov=mcov)
                p = params(A, mcov)
                drain(ctx)
                mg, st, cnt = sh.pipeline_sharded(comm, p, 16, 2)
                what = ("sharded", no_fused, i, mcov)
                assert ctx.kernel_time(api.KERNEL_SCAN)[1] == 0, what  # (phase 2 starts from the scan's survivors: no k_code_scan)
                assert (mg.total_written, mg.n_clust_out, st.max_clust_length) == (len(w.es), w.enc, w.mcl), what
                check_counts(cnt, w, what)
                assert sh.cluster_fetch_packed() == w.clusters and api.events_format(sh.events(), p) == w.text, what
                step(sh, A, mcov=mcov, what="resident after sharded")
        monkeypatch.delenv("E2S_NO_FUSED_PREFILTER")
    finally:
        ctx.timing(False)
        drain(ctx)
        sh.close()
    sh = ctx.shard(A.n, 0, A.n, chunk_positions=CHUNK_E)
    try:
        for i, d in enumerate((A, B, A)):
            if i:
                sh.chunked_reset()
            ctx.stage_reads(d.reads, d.off)
            w = want(d)
            recs = []
            for clo, cn in sh.chunks():
                sh.chunk_begin(clo, cn)
                load_chunk(sh, d, clo, cn, False)
                sh.chunk_scan(16, 2, 5)
                recs.append(sh.cluster_fetch_packed())
            mg, st = sh.chunked_exchange(comm, 16, 2, 5, 0.99)
            tail = O.clusters_to_bytes(np.array(mg.append_start[:mg.n_append], dtype=np.uint64),
                                       np.array(mg.append_len[:mg.n_append], dtype=np.uint16))
            what = ("chunked_exchange", i, d.name)
            assert b"".join(recs) + tail == w.clusters and mg.n_clust_out == w.enc and st.max_clust_length == w.mcl, what
            cnt = sh.find_events(params(d), st.max_clust_length)
            check_counts(cnt, w, what)
            assert api.events_format(sh.events(), params(d)) == w.text, what
    finally:
        sh.close()
    # e2s_pipeline_host_sharded twice on the context's cached shard, the second time with another chunk size
    rec = synth.gesa_records(A.eg()).view(np.uint8).reshape(-1)
    w, p = want(A), params(A)
    for chunk in (str(T), "100003"):
        monkeypatch.setenv("E2S_CHUNK_POSITIONS", chunk)
        rec10 = np.empty((len(w.es) + 16) * 10, dtype=np.uint8)
        evbuf = (api.Event * (w.res.n_candidates + 16))()
        res, mg, st, m = api.pipeline_host_sharded(ctx, comm, rec, 0, 0, A.n, A.n, A.reads.reshape(-1), A.off, p, 16, 2, rec10=rec10,
                                                   events=evbuf)
        what = ("host_sharded", chunk)
        assert m == len(w.es) and rec10[:m * 10].tobytes() == w.clusters, what
        assert (res.n_written, res.n_clust_out, res.max_clust_length) == (len(w.es), w.enc, w.mcl), what
        assert (mg.total_written, st.max_clust_length) == (len(w.es), w.mcl), what
        check_counts(res.snp, w, what)
        assert api.events_format(list(evbuf)[:res.snp.n_variants], p) == w.text, what


# ---------------------------------------------------------------------------------------------------------------------------
# (G) reads restaged between steps
# ---------------------------------------------------------------------------------------------------------------------------
def designed(name):
    case = next(c for c in P.reads_cases() if c.name == name)
    text, res = O.find_events(case.lcp, case.text, case.suff, case.bwt, *O.cluster_lm(case.lcp, case.bwt, P.K, P.MIN_LEN)[:2],
                              case.oparams(), case.max_clust_length, case.bases, case.off)
    return case, text, res


def test_reads_restaged(ctx):
    """big (tiny dataset), small (designed), big again, small with an N inside a context and IUPAC bytes, ragged, clean:
    K4's fast / general path and the read offsets follow the staged set"""
    seq = [data(1), "reads_upper_uniform", data(2), "reads_n_in_context", "reads_iupac_in_context", "reads_ragged_with_empty",
           "reads_upper_uniform", data(3)]
    for i, item in enumerate(seq):
        if isinstance(item, Data):
            d = item
            ctx.stage_reads(d.reads, d.off)
            sh = resident(ctx, d)
            try:
                res = step(sh, d, what=("restaged", i))
                assert bool(res.snp.saw_n) == bool(want(d).res.flags & O.FLAG_SAW_N)
            finally:
                sh.close()
            continue
        case, otext, ores = designed(item)
        assert bool(ores.flags & O.FLAG_SAW_N) == (item == "reads_n_in_context")
        ctx.stage_reads(case.bases, case.off)
        sh = ctx.shard(case.n)
        try:
            sh.load_soa(case.lcp, case.text, case.suff, case.bwt)
            sh.seal()
            p = api.default_params(case.nreads1, **case.params)
            p.pval = case.pval
            res = sh.pipeline_resident(p, P.K, P.MIN_LEN)
            got = (res.snp.n_analysed, res.snp.n_candidates, res.snp.n_variants, res.snp.n_events, bool(res.snp.saw_n))
            exp = (ores.n_analysed, ores.n_candidates, ores.n_variants, ores.n_events, bool(ores.flags & O.FLAG_SAW_N))
            assert got == exp, (i, item)
            assert api.events_format(sh.events(), p) == otext, (i, item)
        finally:
            sh.close()

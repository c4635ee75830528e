"""-m gpu: the sharded step at 2 to 64 ranks on ONE GPU.  Every rank is a thread with its own context and shard; the exchange
between the phases goes through a communicator whose all-gather the test performs (api.Comm.gather: a barrier and a shared
table), so k_merge_stats sees world > 1 rows, the retry agreement of the scan runs across ranks and e2s_pipeline_host_sharded
splices head and tail records, all without NCCL.  Each run is checked three ways: the device merge against the host merge of
the very rows the ranks exchanged, each rank against the host-driven sequence on the same cuts, and the whole against the
oracle's single pass."""
import threading

import numpy as np
import pytest

from ebwt2snp_b200 import api, synth
from oracle import oracle as O
from tests import helpers as H
from tests import phase2_cases as P
from tests.test_from_reads_gpu import case_reads, pipeline_outputs
from tests.test_from_reads_shards_gpu import host_sequence
from tests.test_grid_rounds_gpu import dense
from tests.test_range_edges_gpu import ACGT, NR1, R, L, index_arrays, phantom_input, wrapped_run

pytestmark = pytest.mark.gpu

MAX_WORLD = 64  # MERGE_MAX_SHARDS
TIMEOUT = 30    # seconds a rank waits at the fake's barrier (a step's scan takes milliseconds); twice that for a rank's thread
HALO_L, HALO_R = 2, api.MAX_C_LEN + 1
HOOKS = ("E2S_PF_CAPACITY", "E2S_SCAN_LEGACY", "E2S_CHUNK_POSITIONS", "E2S_NO_FUSED_PREFILTER", "E2S_SM_COUNT")


@pytest.fixture(autouse=True)
def clean_env(monkeypatch):
    for k in HOOKS:
        monkeypatch.delenv(k, raising=False)


class Pool:
    """one context per rank, made on first use and kept for the module; the reads staged on each as real ranks have them"""

    def __init__(self):
        self.ctxs, self.staged = [], [None] * (MAX_WORLD + 1)

    def get(self, world, reads):
        while len(self.ctxs) < world:
            self.ctxs.append(api.Context(0))
        for r in range(world):
            if self.staged[r] is not reads:
                self.ctxs[r].stage_reads(*reads)
                self.staged[r] = reads
        return self.ctxs[:world]

    def close(self):
        for c in self.ctxs:
            c.close()


@pytest.fixture(scope="module")
def pool(built):
    p = Pool()
    yield p
    p.close()


@pytest.fixture(scope="module")
def ctx(built):
    c = api.Context(0)
    yield c
    c.close()


class FakeGather:
    """the all-gather of `world` ranks that are threads of this process: every call writes its row to a shared table, waits for
    the others, copies the table and waits again.  A broken barrier (a rank that does not come) fails the call, never hangs it.
    Keeps every call's count and the rows each call delivered."""

    def __init__(self, world):
        self.world = world
        self.barrier = threading.Barrier(world, timeout=TIMEOUT)
        self.table = np.zeros((world, api.exchange_row_words()), dtype=np.uint64)
        self.calls = [0] * world
        self.delivered = [[] for _ in range(world)]

    def __call__(self, rank, send, recv):
        try:
            self.table[rank] = send
            self.barrier.wait()
            recv[:] = self.table
            self.barrier.wait()
        except threading.BrokenBarrierError:
            return False
        self.calls[rank] += 1
        self.delivered[rank].append(recv.copy())
        return True


def run_ranks(world, body):
    """body(rank) on `world` threads at once -> the results in rank order.  A rank that raises breaks the barrier of whatever
    fake it waits on (body's closure), so the others fail instead of waiting; every thread is joined before this returns."""
    out, errs = [None] * world, [None] * world

    def one(r):
        try:
            out[r] = body(r)
        except BaseException as e:  # noqa: BLE001 (re-raised below, on the test's thread)
            errs[r] = e
            for f in getattr(body, "fakes", ()):
                f.barrier.abort()

    th = [threading.Thread(target=one, args=(r,), daemon=True) for r in range(world)]
    for t in th:
        t.start()
    for t in th:
        t.join(timeout=2 * TIMEOUT)
    assert not any(t.is_alive() for t in th), "a rank is still running"
    return out, errs


# ---- inputs --------------------------------------------------------------------------------------------------------------------
class Input:
    """an index (lcp / text / suff / bwt), its reads and the options of one run, with the oracle's single pass"""

    def __init__(self, name, lcp, text, suff, bwt, bases, off, nreads1, k=16, m=2, params=None, pval=None, x=4):
        self.name, self.lcp, self.text, self.suff, self.bwt = name, lcp, text, suff, bwt
        self.reads = (np.ascontiguousarray(bases, dtype=np.uint8).reshape(-1), np.ascontiguousarray(off, dtype=np.uint64))
        self.nreads1, self.k, self.m, self.x = nreads1, k, m, x
        self.params, self.pval = dict(params or {}), pval
        self.n = len(lcp)
        self._oracle = None

    def p(self):
        p = api.default_params(self.nreads1, **self.params)
        if self.pval is not None:
            p.pval = self.pval
        return p

    def oracle(self):
        """(records es, el, n_clust_out, .snp text, n_candidates, max_clust_length)"""
        if self._oracle is None:
            es, el, enc, _ = O.cluster_lm(self.lcp, self.bwt, self.k, self.m, x=self.x)
            op = O.default_params(self.nreads1, **self.params)
            if self.pval is not None:
                op.pval = self.pval
            ost = O.statistics(es, el, op.mcov_out, op.pval)
            text, res = O.find_events(self.lcp, self.text, self.suff, self.bwt, es, el, op, ost.max_clust_length, self.reads[0],
                                      self.reads[1], x=self.x)
            self._oracle = (es, el, enc, text, int(res.n_candidates), ost.max_clust_length)
        return self._oracle

    def kept_cluster(self):
        """[s, e] of an analysable record of the oracle whose cluster yields a kept event"""
        es, el = self.oracle()[:2]
        p = self.p()
        mcl = self.oracle()[5]
        for s, ln in zip(es, el):
            s, ln = int(s), int(ln)
            if 2 * p.mcov_out <= ln <= mcl and self.event_in(s, s + ln - 1):
                return s, s + ln - 1
        raise AssertionError(f"{self.name}: no analysable cluster with a kept event")

    def event_in(self, s, e):
        if not hasattr(self, "_starts"):
            sh = None  # (the oracle's events carry no position: take them from one resident run)
            self._starts = set()
            c = api.Context(0)
            try:
                c.stage_reads(*self.reads)
                sh = load(c, self, 0, self.n)
                sh.pipeline_resident(self.p(), self.k, self.m)
                self._starts = {int(ev.cluster_start) for ev in sh.events() if ev.keep}
            finally:
                if sh is not None:
                    sh.close()
                c.close()
        return any(s <= q <= e for q in self._starts)


def load(c, inp, lo, hi):
    """the shard [lo, hi) of inp on context c, loaded with 2 / 151 positions of halo and sealed"""
    a, b = max(lo - HALO_L, 0), min(hi + HALO_R, inp.n)
    sh = c.shard(hi - lo, lo, inp.n)
    sh.load_soa(inp.lcp[a:b], inp.text[a:b], inp.suff[a:b], inp.bwt[a:b], first=a)
    if inp.x != 4:
        sh.set_layout(inp.x, 4, 4)
    sh.seal()
    return sh


_INPUTS = {}


def synth_input(name, seed):
    key = (name, seed)
    if key not in _INPUTS:
        rs, e = H.dataset(name, seed)
        _INPUTS[key] = Input(f"{name}{seed}", e["lcp"], e["text"], e["suff"], e["bwt"], rs.reads, O.uniform_read_offsets(*rs.reads.shape),
                             rs.nreads1)
    return _INPUTS[key]


def random_reads(seed):
    rng = np.random.default_rng(seed)
    rd = ACGT[rng.integers(0, 4, size=(R, L))]
    return rd, O.uniform_read_offsets(R, L)


DESIGNED = ("cand_c33", "dist_indels_kl32_g32", "ctx_L32_R30_g32")  # kept SNP events; INDEL events; short right contexts


def designed_input():
    """designed phase-2 cases (tests/phase2_cases.py) whose clusters keep SNP and INDEL events, each with its own options"""
    cases = [c for c in P.all_cases() if c.name in DESIGNED]
    assert len(cases) == len(DESIGNED)
    return [Input(f"designed:{c.name}", c.lcp, c.text, c.suff, c.bwt, c.bases, c.off, c.nreads1, P.K, P.MIN_LEN, c.params, c.pval)
            for c in cases]


def ragged_input():
    bases, off = case_reads("genome")
    want = O.build_egsa_ragged(bases, off)
    return Input("ragged", want["lcp"], want["text"], want["suff"], want["bwt"], bases, off, (len(off) - 1) // 2)


def nm2_input(n=32769, k=16, s=None, snps=True):
    """the n - 2 END / phantom input: a cluster [s, n - 2] closed by an END at n - 2, a START at n - 1"""
    rng = np.random.default_rng(n + (0 if snps else 1))
    s = n - 400 if s is None else s
    lcp, text, suff, bwt = phantom_input(rng, n, k, s)
    if not snps:  # nothing analysable anywhere but the tail (the records of 3 positions are below 2 mcov_out)
        lcp[:] = 0
        lcp[100:n - 500:5] = k + 1
        lcp[101:n - 500:5] = k + 1
        lcp[s - 1], lcp[s:n - 2], lcp[n - 2], lcp[n - 1] = 0, k + 6, k + 5, k + 5
    rd, off = random_reads(n)
    return Input(f"nm2:{n}:{s}:{snps}", lcp, text, suff, bwt, rd, off, NR1, k)


def wrapped_input():
    rd, lcp, text, suff, bwt = wrapped_run()
    return Input("wrapped", lcp, text, suff, bwt, rd, O.uniform_read_offsets(R, L), NR1)


def overflow_input():
    """a dense region of 40 tiles (a record every 4 positions) between two sparse ones: only the shard that holds it overflows
    its record segments"""
    T = 16384
    dn = 40 * T + 1
    lcpd, _ = dense(dn, 16, seed=5)
    rng = np.random.default_rng(77)
    sparse = np.minimum(rng.integers(0, 34, size=60_000), 255).astype(np.uint32)
    lcp = np.concatenate([sparse, lcpd[:-2], [0], sparse]).astype(np.uint32)
    text, suff, bwt = index_arrays(rng, lcp)
    rd, off = random_reads(78)
    return Input("overflow", lcp, text, suff, bwt, rd, off, NR1), (60_000, 60_000 + dn - 1)


# ---- cut layouts ---------------------------------------------------------------------------------------------------------------
def random_cuts(inp, world, seed):
    """world - 1 seeded cuts among the oracle's record boundaries (start, start + 1, end, end + 1) and random positions; every
    shard >= 2 positions"""
    es, el = inp.oracle()[:2]
    rng = np.random.default_rng(seed)
    cand = np.concatenate([es, es + 1, es + el.astype(np.uint64) - 1, es + el.astype(np.uint64), rng.integers(2, inp.n - 2, size=200)])
    cand = np.unique(cand[(cand >= 2) & (cand <= inp.n - 2)].astype(np.int64))
    for _ in range(1000):
        pick = np.sort(rng.choice(cand, size=world - 1, replace=False))
        cuts = [0] + [int(c) for c in pick] + [inp.n]
        if all(b - a >= 2 for a, b in zip(cuts[:-1], cuts[1:])):
            return cuts
    raise AssertionError("no cut layout")


def valid(cuts):
    return cuts[0] == 0 and all(b - a >= 2 for a, b in zip(cuts[:-1], cuts[1:]))


# ---- one run ---------------------------------------------------------------------------------------------------------------------
def sharded_run(pool, inp, cuts, repeat=False, timing=False):
    """pipeline_sharded on every rank (threads) through a FakeGather -> (per rank dict, fake)"""
    world = len(cuts) - 1
    ctxs = pool.get(world, inp.reads)
    p = inp.p()
    fake = FakeGather(world)
    comms = [api.Comm.gather(ctxs[r], r, world, fake) for r in range(world)]
    shards = [load(ctxs[r], inp, cuts[r], cuts[r + 1]) for r in range(world)]
    for c in ctxs:
        if timing:
            c.timing(True)
        for kk in range(9):
            c.kernel_time(kk)

    def body(r):
        out = []
        for _ in range(2 if repeat else 1):
            mg, st, cnt = shards[r].pipeline_sharded(comms[r], p, inp.k, inp.m)
            out.append(dict(mg=bytes(mg), st=bytes(st), cnt=bytes(cnt), recs=shards[r].cluster_fetch_packed(),
                            ev=[bytes(e) for e in shards[r].events()], mgs=mg, sts=st, cnts=cnt))
        return out
    body.fakes = (fake,)
    try:
        outs, errs = run_ranks(world, body)
        for r in range(world):
            res = {}
            for kk, name in ((api.KERNEL_SCAN1, "scan1"), (api.KERNEL_FLAGS, "flags")):
                res[name] = ctxs[r].kernel_time(kk)[1]
            if errs[r] is None:
                outs[r][0].update(res)
            if timing:
                ctxs[r].timing(False)
    finally:
        for sh in shards:
            sh.close()
        for cm in comms:
            cm.close()
    return outs, errs, fake


def check_run(ctx, pool, inp, cuts, repeat=False, timing=False):
    """the three checks of one layout (see the module doc) -> per rank results"""
    world = len(cuts) - 1
    assert valid(cuts), cuts
    outs, errs, fake = sharded_run(pool, inp, cuts, repeat, timing)
    for r, e in enumerate(errs):
        if e is not None:
            raise AssertionError(f"{inp.name} cuts={cuts}: rank {r} failed: {e}") from e
    where = (inp.name, cuts)
    p = inp.p()
    # 1. device merge = host merge of the rows the fake delivered
    for r in range(world):
        mg, st = api.exchange_rows_finish(fake.delivered[r][-1], r, inp.n, inp.k, inp.m, p.mcov_out, p.pval)
        assert (bytes(mg), bytes(st)) == (outs[r][0]["mg"], outs[r][0]["st"]), (where, r)
        assert all(np.array_equal(fake.delivered[r][-1], fake.delivered[0][-1]) for r in range(world))
    # 2. each rank = the host-driven sequence on the same cuts
    seq = host_sequence([load(ctx_host(ctx, inp), inp, cuts[g], cuts[g + 1]) for g in range(world)], p, inp.k, inp.m)
    for r in range(world):
        o = outs[r][0]
        assert (o["mg"], o["st"], o["cnt"], o["recs"], o["ev"]) == (seq[r][3], seq[r][4], seq[r][5], seq[r][1], seq[r][6]), (where, r)
    # 3. the whole = the oracle's single pass
    es, el, enc, otext, ocand, omcl = inp.oracle()
    recs = [outs[r][0]["recs"] for r in range(world)]
    assert b"".join(recs) == O.clusters_to_bytes(es, el), where
    assert [outs[r][0]["mgs"].record_offset for r in range(world)] == list(np.cumsum([0] + [len(x) // 10 for x in recs[:-1]])), where
    assert all(outs[r][0]["mgs"].n_clust_out & 0xFFFFFFFF == enc for r in range(world)), where
    assert all(outs[r][0]["sts"].max_clust_length == omcl for r in range(world)), where
    assert sum(outs[r][0]["cnts"].n_candidates for r in range(world)) == ocand, where
    text, first = b"", 1
    for r in range(world):
        evs = [api.Event.from_buffer_copy(e) for e in outs[r][0]["ev"]]
        text += api.events_format(evs, p, first_id=first)
        first += outs[r][0]["cnts"].n_events
    assert text == otext, where
    # 4. the same shards and communicators again: the same bytes
    if repeat:
        for r in range(world):
            a, b = outs[r]
            assert (a["mg"], a["st"], a["cnt"], a["recs"], a["ev"]) == (b["mg"], b["st"], b["cnt"], b["recs"], b["ev"]), (where, r)
    # retry agreement: every rank gathered, and scanned, as often as every other
    assert len(set(fake.calls)) == 1, (where, fake.calls)
    if timing:
        for kern in ("scan1", "flags"):  # (k_cluster_scan launches, or k_lcp_flags launches on the two-kernel path)
            assert len({outs[r][0][kern] for r in range(world)}) == 1, (where, kern, [outs[r][0][kern] for r in range(world)])
    return outs, fake


def row_dev(fake, r):
    """the scan accumulators in rank r's exchange row, as the ranks last exchanged them"""
    return api.ClusterDev.from_buffer_copy(fake.delivered[0][-1][r].tobytes())


def ctx_host(ctx, inp):
    ctx.stage_reads(*inp.reads)
    return ctx


# ---- random cuts at 2, 3, 8 and 64 ranks -------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3, 8])
def test_random_cuts_synth(ctx, pool, world):
    for name, seed in (("tiny", 3), ("small", 4)):
        inp = synth_input(name, seed)
        for rep in range(2):
            check_run(ctx, pool, inp, random_cuts(inp, world, 1000 * world + rep), repeat=rep == 0, timing=True)


def test_random_cuts_64_ranks(ctx, pool):
    inp = synth_input("tiny", 3)
    outs, fake = check_run(ctx, pool, inp, random_cuts(inp, MAX_WORLD, 64), repeat=True, timing=True)
    assert fake.calls == [2] * MAX_WORLD


@pytest.mark.parametrize("world", [2, 3, 8])
def test_random_cuts_designed_ragged(ctx, pool, world):
    for inp in designed_input() + [ragged_input()]:
        if inp.n < 4 * world:
            continue
        check_run(ctx, pool, inp, random_cuts(inp, world, 7 * world), timing=True)


# ---- around one analysable cluster with a kept event ---------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["designed", "tiny"])
def test_cuts_around_a_kept_cluster(ctx, pool, which):
    """a cut at s, s + 1, e - 1, e, e + 1 and at every position inside [s, e], at 2 ranks and (with one more cut well away) at
    3: head records at shard positions 0 and 1, and the adopted survivor entry phase 2 finds the event from"""
    inp = designed_input()[0] if which == "designed" else synth_input("tiny", 3)
    s, e = inp.kept_cluster()
    straddling = 0
    for c in sorted(set(range(s, e + 2)) | {s + 1, e - 1}):
        if not 2 <= c <= inp.n - 2:
            continue
        outs, _ = check_run(ctx, pool, inp, [0, c, inp.n])
        if s < c <= e:  # START on rank 0, END on rank 1: rank 0 owns the record's start, so it adopts the record for phase 2
            mg = outs[0][0]["mgs"]
            assert (s, e - s + 1) in [(mg.adopt_start[i], mg.adopt_len[i]) for i in range(mg.n_adopt)], (c, s, e)
            straddling += 1
        far = c // 2 if c >= 200 else (c + inp.n) // 2
        cuts = sorted({0, c, far, inp.n})
        if valid(cuts) and len(cuts) == 4:
            check_run(ctx, pool, inp, cuts)
    assert straddling == e - s


def test_chain_of_two_position_shards(ctx, pool):
    """the inside of one cluster cut into 2-position shards: shards with no event of their own between its START and its END"""
    inp = nm2_input(n=40_000, s=40_000 - 140)
    es, el = inp.oracle()[:2]
    s, ln = next((int(a), int(b)) for a, b in zip(es, el) if 40 <= b <= 150 and int(a) > 2000)
    cuts = [0] + list(range(s + 1, min(s + ln - 1, s + 1 + 2 * 60), 2)) + [inp.n]
    _, fake = check_run(ctx, pool, inp, cuts, timing=True)
    rows = [row_dev(fake, r) for r in range(len(cuts) - 1)]
    assert sum(1 for h in rows[1:-1] if h.any_event == 0) >= 2


# ---- the tail ----------------------------------------------------------------------------------------------------------------------
def tail_layouts(inp):
    """(name, cuts) of the tail layouts, on an input whose last record is no tail record (so the record statistics() counts twice
    is some shard's own or head record, and no record is appended to the last shard).  s1 / s0: the last / second-to-last record."""
    n = inp.n
    es, el = (a.astype(np.int64) for a in inp.oracle()[:2])
    assert int((es + el).max()) < n - 1 and len(es) >= 2, inp.name
    s0, l0, s1, l1 = int(es[-2]), int(el[-2]), int(es[-1]), int(el[-1])
    out = [("last2", [0, n // 2, n - 2, n]),
           ("last_no_record", [0, s1 // 2, s1 + l1 + 1, n]),          # the last record lives on the shard before the last
           ("head_plus_own", [0, max(2, s0 // 2), s0 + l0 // 2, n]),  # the last shard: a head record, then its own records
           ("head_only", [0, max(2, s1 // 2), s1 + l1 // 2, n])]      # the last shard's only record is its head record
    for name, cuts in out:
        assert valid(cuts) and len(set(cuts)) == len(cuts), (inp.name, name, cuts)
    return out


def test_tail_layouts(ctx, pool):
    """the last record of the file, which statistics() counts twice, on the last shard or on an earlier one, as a head record
    or an own record"""
    head_len_differs = 0
    for inp in designed_input()[:2] + [wrapped_input()]:
        for name, cuts in tail_layouts(inp):
            outs, fake = check_run(ctx, pool, inp, cuts, timing=True)
            mg, h = outs[-1][0]["mgs"], row_dev(fake, len(cuts) - 2)
            head = bool(mg.n_prepend and mg.prepend_written)
            assert mg.n_append == 0, (inp.name, name)
            assert {"last2": True, "last_no_record": h.n_written == 0 and not head, "head_plus_own": h.n_written > 0 and head,
                    "head_only": h.n_written == 0 and head}[name], (inp.name, name, h.n_written, head)
            head_len_differs += name == "head_plus_own" and mg.prepend_len != h.last_rec & 0xFFFF
    assert head_len_differs  # (a head record whose length differs from the shard's last own record)


@pytest.mark.parametrize("start", [3, 2])
def test_nm2_last_shard(ctx, pool, start):
    """END at n - 2: the last shard starts at n - 3 or n - 2 (2 ranks and 3)"""
    inp = nm2_input()
    n = inp.n
    check_run(ctx, pool, inp, [0, n - start, n], timing=True)
    check_run(ctx, pool, inp, [0, n - 1000, n - start, n], timing=True)


def test_wrapped_run_across_shards(ctx, pool):
    """a run of 65 560 positions (wrapped length 24) crossing 3 shards"""
    inp = wrapped_input()
    check_run(ctx, pool, inp, [0, 20_000, 45_000, 62_000, 100_000, inp.n], timing=True)


def test_65_ranks_refused(ctx, pool):
    inp = synth_input("tiny", 3)
    world = MAX_WORLD + 1
    cuts = random_cuts(inp, world, 65)
    outs, errs, fake = sharded_run(pool, inp, cuts)
    assert all(isinstance(e, api.E2SError) and e.code == api.ERR_UNSUPPORTED for e in errs), errs
    assert fake.calls == [0] * world and not any(fake.delivered)


# ---- the two-kernel scan --------------------------------------------------------------------------------------------------------
def two_kernel_inputs():
    long_ = case_reads("long")
    want = O.build_egsa_ragged(*long_)
    inp128 = Input("long_k128", want["lcp"], want["text"], want["suff"], want["bwt"], *long_, (len(long_[1]) - 1) // 2, k=128)
    assert int(want["lcp"].max()) > 127
    mr = case_reads("min_len_34")
    w34 = O.build_egsa_ragged(*mr)
    inp34 = Input("m34", w34["lcp"], w34["text"], w34["suff"], w34["bwt"], *mr, (len(mr[1]) - 1) // 2, m=34)
    return [inp128, inp34]


@pytest.mark.parametrize("world", [2, 3])
def test_two_kernel_scan(ctx, pool, monkeypatch, world):
    for inp in two_kernel_inputs():
        outs, _ = check_run(ctx, pool, inp, random_cuts(inp, world, 31 * world), timing=True)
        assert all(o[0]["scan1"] == 0 and o[0]["flags"] >= 1 for o in outs), inp.name
    monkeypatch.setenv("E2S_SCAN_LEGACY", "1")
    inp = synth_input("tiny", 3)
    outs, _ = check_run(ctx, pool, inp, random_cuts(inp, world, 37 * world), timing=True)
    assert all(o[0]["scan1"] == 0 and o[0]["flags"] >= 1 for o in outs)


# ---- retry agreement -----------------------------------------------------------------------------------------------------------
def test_segment_overflow_on_one_rank(ctx, pool):
    """only the middle shard overflows its record segments: every rank reruns the scan once"""
    inp, (lo, hi) = overflow_input()
    outs, fake = check_run(ctx, pool, inp, [0, lo - 1000, hi + 1000, inp.n], timing=True)
    assert fake.calls == [2, 2, 2] and [o[0]["scan1"] for o in outs] == [2, 2, 2]


def test_survivor_list_capacity_3(ctx, pool, monkeypatch):
    monkeypatch.setenv("E2S_PF_CAPACITY", "3")
    inp = synth_input("tiny", 3)
    outs, fake = check_run(ctx, pool, inp, random_cuts(inp, 3, 333), timing=True)
    assert fake.calls == [2, 2, 2] and [o[0]["scan1"] for o in outs] == [2, 2, 2]


def test_survivor_list_capacity_1_tail_adoption(ctx, pool, monkeypatch):
    """a survivor list of 1 entry (the scan keeps none) and no rank with survivors of its own, while the last shards adopt the
    records around the END at n - 2 and the phantom START at n - 1: every rank must still decide alike, and equal the oracle"""
    monkeypatch.setenv("E2S_PF_CAPACITY", "1")
    n = 32769
    s = n - 40
    inp = nm2_input(n=n, s=s, snps=False)  # (the cluster closed at n - 2 is short enough to be analysed)
    adopt = {}
    for last in (n - 3, n - 2, s - 1, s, s - 29):
        outs, fake = check_run(ctx, pool, inp, [0, n // 2, last, n], timing=True)
        adopt[last] = [o[0]["mgs"].n_adopt for o in outs]
    assert adopt[n - 3] == adopt[n - 2] == [0, 1, 1] and adopt[s] == adopt[s - 29] == [0, 0, 1], adopt


def test_survivor_list_capacity_1_two_tail_adoptions(ctx, pool, monkeypatch):
    """-m 1 and a survivor list of 1 entry: the last shard owns the start of the cluster still open at n - 1 and the phantom
    record [n, n] of length 1, so it adopts both tail records and no rank has survivors of its own.  Its adoptions must fit the
    room the scan leaves in the list; a rank that found its list full after the exchange would repeat the step alone"""
    monkeypatch.setenv("E2S_PF_CAPACITY", "1")
    n, k = 32769, 16
    inp = nm2_input(n=n, s=n - 40, snps=False)
    inp.lcp[n - 2], inp.lcp[n - 1] = k + 6, k + 5  # (no END at n - 2: the cluster [n - 40, n - 1] is open at the end)
    inp.m = 1
    es, el = inp.oracle()[:2]
    assert [(int(a), int(b)) for a, b in zip(es[-2:], el[-2:])] == [(n - 40, 40), (n, 1)]
    outs, fake = check_run(ctx, pool, inp, [0, n // 2, n - 40, n], timing=True)
    assert [o[0]["mgs"].n_adopt for o in outs] == [0, 0, 2] and fake.calls == [1, 1, 1]


# ---- streamed: e2s_pipeline_host_sharded ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("m", [2, 10])
@pytest.mark.parametrize("world", [2, 3, 8])
def test_host_sharded_equals_resident_step(ctx, pool, monkeypatch, world, m):
    """chunks of 16 384 positions, counted from each rank's range_lo.  A cut lies inside a cluster (a head record), or 16 384
    positions before the middle of one (that rank's first chunk boundary cuts the cluster).  At -m 10 the clusters cut are 4 to
    9 positions long, shorter than the minimum record length"""
    base = synth_input("tiny", 3)
    es, el = base.oracle()[:2]
    inp = Input(f"tiny3:m{m}", base.lcp, base.text, base.suff, base.bwt, *base.reads, base.nreads1, m=m) if m != 2 else base
    T = 16384
    mids = [int(a) + int(b) // 2 for a, b in zip(es, el) if 4 <= b < (m if m > 2 else 151)]
    rng = np.random.default_rng(world)
    cand = [c - T * int(rng.integers(0, 2)) for c in mids if c > T + 2]
    cuts = sorted(set([0, inp.n] + [int(c) for c in rng.choice(cand, size=world - 1, replace=False)]))
    while not (valid(cuts) and len(cuts) - 1 == world):
        cuts = sorted(set([0, inp.n] + [int(c) for c in rng.choice(cand, size=world - 1, replace=False)]))
    ref, _ = check_run(ctx, pool, inp, cuts)
    monkeypatch.setenv("E2S_CHUNK_POSITIONS", str(T))
    ctxs = pool.get(world, inp.reads)
    fake = FakeGather(world)
    comms = [api.Comm.gather(ctxs[r], r, world, fake) for r in range(world)]
    p = inp.p()
    rec_all = synth.gesa_records(dict(lcp=inp.lcp, text=inp.text, suff=inp.suff, bwt=inp.bwt, n=inp.n)).view(np.uint8).reshape(-1)
    rs = 13

    def body(r):
        lo, hi = cuts[r], cuts[r + 1]
        a, b = max(0, lo - 176), min(inp.n, hi + 152)
        rec10 = np.zeros((len(ref[r][0]["recs"]) // 10 + 16) * 10, dtype=np.uint8)
        ev = (api.Event * (len(ref[r][0]["ev"]) + 16))()
        res, mg, st, m = api.pipeline_host_sharded(ctxs[r], comms[r], rec_all[a * rs:b * rs], a, lo, hi - lo, inp.n, None, None, p,
                                                   inp.k, inp.m, rec10=rec10, events=ev)
        return bytes(mg), bytes(st), rec10[:m * 10].tobytes(), res, [bytes(e) for e in list(ev)[:res.snp.n_variants]]
    body.fakes = (fake,)
    try:
        outs, errs = run_ranks(world, body)
    finally:
        for cm in comms:
            cm.close()
    assert not any(errs), errs
    for r in range(world):
        mg, st, recs, res, ev = outs[r]
        o = ref[r][0]
        assert (mg, st, recs, ev) == (o["mg"], o["st"], o["recs"], o["ev"]), (cuts, r)
        c = o["cnts"]
        assert (res.snp.n_candidates, res.snp.n_variants, res.snp.n_events) == (c.n_candidates, c.n_variants, c.n_events), (cuts, r)
    assert fake.calls == [1] * world


# ---- reads to SNPs on W ranks ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 3, 8])
def test_reads_to_snps_ranks(ctx, pool, world):
    """stage the reads on every rank, key_cuts + build_egsa_range, halo rows exchanged, seal, pipeline_sharded through the fake:
    equals e2s_pipeline_reads on the whole index"""
    bases, off = case_reads("genome")
    reads = (np.ascontiguousarray(bases, dtype=np.uint8), np.ascontiguousarray(off, dtype=np.uint64))
    p = api.default_params((len(off) - 1) // 2)
    n = int(off[-1]) + len(off) - 1
    ctx.stage_reads(*reads)
    rc, whole = pipeline_outputs(ctx, lambda r, e: ctx.pipeline_reads(bases, off, p, 16, 2, 1, 4, 1, rec10=r, events=e), n)[:2]
    assert rc == 0, whole
    ctxs = pool.get(world, reads)
    cuts = [c.key_cuts(off, world) for c in ctxs]
    assert all(np.array_equal(cuts[0][0], k) and np.array_equal(cuts[0][1], q) for k, q in cuts)
    key_lo, pos = cuts[0]
    shards = []
    for r in range(world):
        sh = ctxs[r].shard(int(pos[r + 1]) - int(pos[r]), int(pos[r]), n)
        sh.build_egsa_range(off, int(key_lo[r]), int(key_lo[r + 1]) if r + 1 < world else 0, 1, 4, 1)
        shards.append(sh)
    rows = np.stack([sh.halo_row() for sh in shards])
    for r, sh in enumerate(shards):
        sh.halo_apply(rows, r)
        sh.seal()
    fake = FakeGather(world)
    comms = [api.Comm.gather(ctxs[r], r, world, fake) for r in range(world)]

    def body(r):
        mg, st, cnt = shards[r].pipeline_sharded(comms[r], p, 16, 2)
        return mg, st, cnt, shards[r].cluster_fetch_packed(), [bytes(e) for e in shards[r].events()]
    body.fakes = (fake,)
    try:
        outs, errs = run_ranks(world, body)
    finally:
        for sh in shards:
            sh.close()
        for cm in comms:
            cm.close()
    assert not any(errs), errs
    assert b"".join(o[3] for o in outs) == whole[1]
    assert sum((o[4] for o in outs), []) == whole[2]
    assert all((o[0].n_clust_out, o[1].max_clust_length) == (whole[0][1], whole[0][2]) for o in outs)

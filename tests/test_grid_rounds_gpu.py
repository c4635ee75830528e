"""-m gpu: parity with the oracle when CTAs loop -- scan chunks of many tiles, grid-stride rounds -- at any SM count.

Every grid of phase 1, the loaders and phase 2 is sized from the context's SM count, which E2S_SM_COUNT overrides when the
context is made.  At one SM the scan runs on 3-4 CTAs, so a 40-tile input gives each CTA 10-14 tiles: the state k_cluster_scan
carries from tile to tile, its tile-parity buffers and its stage / phase ring all run many rounds at sizes the oracle checks
quickly, and so do the grid-stride loops of the loaders, K1 and phase 2.  Where the chunks of the scan start depends on the
occupancy, which a test cannot see, so every feature is planted at every tile boundary in turn: whichever tiles start chunks,
each feature lands on a chunk's first, second and later tiles.

(A) the one-pass scan on planted tile boundaries at 1, 2, 3, 7 SMs and the device's own: records, n_clust_out, statistics;
    a segment that overflows in a chunk's later tile (the scan reruns on grown segments).
(B) the same inputs through K1 + K2 (E2S_SCAN_LEGACY), and -k > 127 over LCP values
    above 127, which takes that path by itself.
(C) shards cut anywhere and chunked shards at one SM: summaries against helpers.emulate_shard, the assembled .clusters.
(D) phase 2 on the designed cases of tests/phase2_cases.py at 1 and 3 SMs, the volume case over 183 tiles included.
(E) every loader at one SM, whole and in pieces, then both tools against the oracle.
(F) both builds of k_cluster_scan (E2S_SCAN_OCC=3 / 4): a subset of (A) and (D) in a child process per build.
(G) the default geometry at a size where every CTA scans four tiles or more, resident and streamed.
(H) the CLIs at one SM, streaming small chunks.
"""
import contextlib
import os
import subprocess
import sys

import numpy as np
import pytest

from ebwt2snp_b200 import api, synth
from oracle import oracle as O
from tests import helpers as H
from tests import phase2_cases as P
from tests import test_phase2_paths_gpu as PP
from tests import test_range_edges_gpu as RE
from tests import test_reuse_gpu as RU
from tests.test_reuse_gpu import gesa_file  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T = 16384            # positions per scan tile
SC_CAP = 512         # ENDs a scan tile keeps in shared memory before its window loop
SMS = [1, 2, 3, 7, 0]  # 0: the device's own SM count (E2S_SM_COUNT unset)
SM_IDS = [f"sm{s}" if s else "smdev" for s in SMS]
KS = (1, 2, 3, 16, 70, 127)
MS = (-3, 1, 2, 3, 33, 34, 200)
LENS = (1, 2, 3, 32, 33, 34)
RUNS = (65535, 65536, 65537, 65538, 131073)
CHILD = "E2S_GRID_ROUNDS_CHILD"  # set in the child processes of (F)


@contextlib.contextmanager
def sm_env(sm):
    """E2S_SM_COUNT set to sm (None / 0: unset) while a context is made; the environment is restored afterwards"""
    old = os.environ.pop("E2S_SM_COUNT", None)
    if sm:
        os.environ["E2S_SM_COUNT"] = str(sm)
    try:
        yield
    finally:
        os.environ.pop("E2S_SM_COUNT", None)
        if old is not None:
            os.environ["E2S_SM_COUNT"] = old


@pytest.fixture(scope="module")
def ctxs(built):
    """sm -> a context whose grids are sized for sm SMs (made once)"""
    made = {}

    def get(sm):
        if sm not in made:
            with sm_env(sm):
                made[sm] = api.Context(0)
        return made[sm]
    yield get
    for c in made.values():
        c.close()


def device_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------------
# inputs: features planted at every tile boundary, rotating by the boundary's index
# ---------------------------------------------------------------------------------------------------------------------------
def run(lcp, lo, hi, v):
    """one run of LCP v over [lo, hi) with 0 on both sides (inside the array)"""
    n = len(lcp)
    lo, hi = max(1, lo), min(hi, n - 1)
    lcp[lo - 1] = 0
    lcp[lo:hi] = v
    lcp[hi] = 0


def plant(lcp, k, rot=0):
    """at boundary t * T (t >= 1), feature (t + rot) % 6:
      0  a cluster open across the whole tile t;
      1  a run of LENS[...] positions whose END is the tile's first or second position;
      2  tile t dense: runs of 3, 4096 ENDs (> SC_CAP), only at t >= 2;
      3  a run of RUNS[...] positions from 7 before the boundary (4 or more tiles; its length wraps from 65536 on);
      4  an END at the tile's first position by the local-minimum rule (lcp[b-1] > lcp[b] <= lcp[b+1]), START carried to b + 1;
      5  none (the background crosses the boundary)
    and always a cluster closed by an END at n - 2 (a START follows at n - 1), opened in the tile before n - 2's."""
    n = len(lcp)
    v = k + 1
    free = 0
    for t in range(1, (n + T - 1) // T):
        b = t * T
        if b < free:
            continue
        f = (t + rot) % 6
        j = t // 6 + rot
        if f == 0:
            run(lcp, b - 3, b + T + 3, v)
            free = b + T + 4
        elif f == 1 or (f == 2 and t < 2):
            ln, d = LENS[j % len(LENS)], j % 2
            run(lcp, b + d + 1 - ln, b + d + 1, v + 1)
        elif f == 2:
            hi = min(b + T, n - 4)
            lcp[b:hi] = v
            lcp[b:hi:4] = 0
            free = hi
        elif f == 3:
            ln = RUNS[j % len(RUNS)]
            if b - 7 + ln < n - 8:
                run(lcp, b - 7, b - 7 + ln, v + 2)
                free = b - 7 + ln + 1
        elif f == 4 and b + 8 < n:
            run(lcp, b - 20 - j % 7, b + 6, v + 1)
            lcp[b - 20 - j % 7:b] = v + 3
    return end_nm2(lcp, k)


def end_nm2(lcp, k):
    """a cluster closed by an END at n - 2 (lcp[n-3] > lcp[n-2] <= lcp[n-1]), opened in the tile before n - 2's or in its own"""
    n = len(lcp)
    if n >= 8:
        s = max(2, n - 2 - T // 3 - (n % 977))
        lcp[s - 1] = 0
        lcp[s:n - 2] = k + 6
        lcp[n - 2] = k + 5
        lcp[n - 1] = k + 5
    return lcp


def planted(n, k, mode, seed, rot=0):
    rng = np.random.default_rng(seed)
    lcp = plant(H.random_lcp(rng, n, k, mode), k, rot)
    bwt = rng.choice(H.BWT_ALPHABET, size=n)
    return lcp, bwt


def sizes(tiles=(2, 3, 5, 8, 13, 21, 40), deltas=(-2, -1, 1, 2)):
    return [t * T + d for t in tiles for d in deltas]


def km_pairs(sm_index, count):
    """count (k, m) pairs: every pair of KS x MS within the first 42, in an order that differs per SM count"""
    pairs = [(k, m) for k in KS for m in MS]
    return [pairs[(5 * i + 11 * sm_index) % len(pairs)] for i in range(count)]


def check_scan(ctx, lcp, bwt, k, m, what):
    """cluster_lm + statistics on one resident shard against the oracle"""
    es, el, enc, _ = O.cluster_lm(lcp, bwt, k, m)
    sh = ctx.shard(len(lcp))
    try:
        sh.load_soa(lcp, None, None, bwt)
        sh.seal()
        nw, nc = sh.cluster_lm(k, m)
        s, l = sh.cluster_fetch()
        assert (nw, nc) == (len(es), enc), what
        assert np.array_equal(s, es) and np.array_equal(l, el), what
        if len(es):
            st, ost = sh.statistics(5, 0.99), O.statistics(es, el, 5, 0.99)
            assert list(st.hist) == list(ost.hist), what
            assert (st.n_clust, st.n_bases, st.max_len, st.max_clust_length) == (ost.n_clust, ost.n_bases, ost.max_len,
                                                                                  ost.max_clust_length), what
    finally:
        sh.close()
    return es, el


# ---------------------------------------------------------------------------------------------------------------------------
# the hook
# ---------------------------------------------------------------------------------------------------------------------------
def test_sm_count_hook_refuses_bad_values(built):
    dev = device_sms()
    for bad in ("0", str(dev + 1), "-4", "12x", ""):
        os.environ["E2S_SM_COUNT"] = bad
        try:
            with pytest.raises(api.E2SError) as ei:
                api.Context(0)
            assert ei.value.code == api.ERR_ARG and "E2S_SM_COUNT" in str(ei.value), bad
        finally:
            os.environ.pop("E2S_SM_COUNT", None)
    for good in (1, dev):
        with sm_env(good):
            api.Context(0).close()


# ---------------------------------------------------------------------------------------------------------------------------
# (A) the one-pass scan
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sm", SMS, ids=SM_IDS)
def test_scan_tile_boundaries(ctxs, sm):
    ctx = ctxs(sm)
    si = SMS.index(sm)
    ns = sizes()
    kms = km_pairs(si, 2 * len(ns))
    for i, n in enumerate(ns):
        for r in range(2):
            k, m = kms[2 * i + r]
            mode = (i + r + si) % 5
            lcp, bwt = planted(n, k, mode, seed=1000 * si + 2 * i + r, rot=i + r)
            check_scan(ctx, lcp, bwt, k, m, (sm, n, k, m, mode))


def dense(n, k, seed):
    """every tile dense (runs of 3 separated by one 0: 4096 records a tile), random bytes in the BWT, an END at n - 2"""
    rng = np.random.default_rng(seed)
    lcp = np.full(n, k + 1, dtype=np.uint32)
    lcp[::4] = 0
    return end_nm2(lcp, k), rng.choice(H.BWT_ALPHABET, size=n)


@pytest.mark.parametrize("sm", SMS, ids=SM_IDS)
def test_segment_overflow_in_later_tile(ctxs, sm):
    """n / 4 records, twice what the first segment guess holds: every chunk overflows its segment after its first tiles (at one
    SM a chunk of 10-14 tiles overflows in its 6th-8th tile) -- the scan reruns once on grown segments and equals the oracle"""
    ctx = ctxs(sm)
    n = 40 * T + 1
    k, m = 16, 2
    lcp, bwt = dense(n, k, seed=sm)
    ctx.timing(True)
    RU.drain(ctx)
    try:
        es, _ = check_scan(ctx, lcp, bwt, k, m, sm)
        assert len(es) > n // 8 + 4096 + 64 * 41  # (more than the segments of all chunks hold at first)
        s1, fl = RU.scans(ctx)
        assert (s1, fl) == (2, 0), (s1, fl)
    finally:
        ctx.timing(False)
        RU.drain(ctx)


# ---------------------------------------------------------------------------------------------------------------------------
# (B) K1 + K2
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [0, 1, 2])
def test_k1_k2_tile_boundaries(ctxs, case, monkeypatch):
    """E2S_SCAN_LEGACY=1 at every SM count, three sets of (k, -m) pairs and planted patterns"""
    monkeypatch.setenv("E2S_SCAN_LEGACY", "1")
    ns = sizes(tiles=(3, 13, 40), deltas=(-1, 2))
    for si, sm in enumerate(SMS):
        ctx = ctxs(sm)
        kms = km_pairs(si + 3 * case, len(ns))
        for i, n in enumerate(ns):
            k, m = kms[i]
            lcp, bwt = planted(n, k, (i + case) % 5, seed=5000 + 100 * case + 10 * si + i, rot=i + case)
            check_scan(ctx, lcp, bwt, k, m, (case, sm, n, k, m))


@pytest.mark.parametrize("sm", SMS, ids=SM_IDS)
def test_k_above_127_tile_boundaries(ctxs, sm):
    """-k 128 / 200 over LCP values up to 70 000: the byte copy cannot answer, the shard runs K1 + K2 on its own"""
    ctx = ctxs(sm)
    ctx.timing(True)
    RU.drain(ctx)
    try:
        for i, n in enumerate(sizes(tiles=(5, 40), deltas=(-2, 1))):
            for k, m in ((128, 2), (200, -3), (129, 33)):
                lcp, bwt = planted(n, k, 1 + (i % 2), seed=7000 + 10 * i + k, rot=i)
                check_scan(ctx, lcp, bwt, k, m, (sm, n, k, m))
                s1, fl = RU.scans(ctx)
                assert s1 == 0 and fl >= 1, (s1, fl)
    finally:
        ctx.timing(False)
        RU.drain(ctx)


# ---------------------------------------------------------------------------------------------------------------------------
# (C) shard layouts at one SM
# ---------------------------------------------------------------------------------------------------------------------------
def cut_shards(ctx, lcp, bwt, cuts, k, m, what):
    n = len(lcp)
    sums, recs = [], []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        sh = ctx.shard(hi - lo, lo, n)
        try:
            a, b = max(0, lo - 2), min(n, hi + 151)
            sh.load_soa(lcp[a:b], None, None, bwt[a:b], first=a)
            sh.seal()
            sums.append(sh.cluster_run(k, m))
            sh.cluster_finalize(api.ClusterMerged())
            recs.append(sh.cluster_fetch())
        finally:
            sh.close()
        want, ws, wl = H.emulate_shard(lcp, bwt, lo, hi, k, m)
        RE.summary_equals(sums[-1], want, (what, lo, hi))
        assert np.array_equal(recs[-1][0], ws) and np.array_equal(recs[-1][1], wl), (what, lo, hi)
    return H.assemble(sums, recs)


@pytest.mark.parametrize("n", [40 * T + 1, 21 * T - 2])
def test_shard_layouts_one_sm(ctxs, n):
    """shards cut at random positions (cluster_run -> merge) and chunked shards streaming chunks of 5 * 16384 + 1 and 7 * 16384
    positions: every chunk is scanned by CTAs of several tiles"""
    ctx = ctxs(1)
    rng = np.random.default_rng(n)
    for i, (k, m) in enumerate(((16, 2), (3, 3), (70, 33), (1, -3), (127, 1))):
        lcp, bwt = planted(n, k, i % 5, seed=n + i, rot=i)
        es, el, enc, _ = O.cluster_lm(lcp, bwt, k, m)
        cuts = [0] + sorted(int(c) for c in rng.choice(np.arange(1000, n - 1000), size=3, replace=False)) + [n]
        S, L, mg = cut_shards(ctx, lcp, bwt, cuts, k, m, (n, k, m, cuts))
        assert mg.n_clust_out == enc and np.array_equal(S, es) and np.array_equal(L, el), (n, k, m, cuts)
        want, _, _ = H.emulate_shard(lcp, bwt, 0, n, k, m)
        for chunk in (5 * T + 1, 7 * T):
            sm_, s_, l_, sh = RE.stream_range(ctx, lcp, bwt, k, m, chunk)
            sh.close()
            RE.summary_equals(sm_, want, (n, k, m, chunk))
            S, L, mg = H.assemble([sm_], [(s_, l_)])
            assert mg.n_clust_out == enc and np.array_equal(S, es) and np.array_equal(L, el), (n, k, m, chunk)


# ---------------------------------------------------------------------------------------------------------------------------
# (D) phase 2 on the designed cases
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def designed():
    """[(case, oracle)] of every designed case, the subset's flags and the volume case (3 000 000 positions, 183 tiles)"""
    out = [(c, PP.oracle(c), "subset" in c.groups) for c in PP.CASES]
    vol = P.volume_case()
    out.append((vol, PP.oracle(vol), True))
    return out


@pytest.mark.parametrize("sm", [1, 3], ids=["sm1", "sm3"])
def test_phase2_designed(ctxs, designed, sm, monkeypatch):
    """two-phase and e2s_pipeline_resident on every case; the subset also through e2s_pipeline_host / _soa streaming chunks of
    16384 positions and clust2snp on a chunked shard (lean and not)"""
    ctx = ctxs(sm)
    for case, want, sub in designed:
        PP.resident_and_fused(ctx, case, want)
    monkeypatch.setenv("E2S_CHUNK_POSITIONS", str(PP.CHUNK))
    for case, want, sub in designed:
        if sub:
            for lean in (False, True):
                PP.pipeline_host_chunked(ctx, (case, want), lean)
                PP.chunked_clust2snp(ctx, (case, want), lean)


# ---------------------------------------------------------------------------------------------------------------------------
# (E) the loaders at one SM
# ---------------------------------------------------------------------------------------------------------------------------
def load_soa_dev(sh, d, a, b):
    import torch
    arrs = [torch.from_numpy(np.ascontiguousarray(x[a:b])).cuda() for x in (d.lcp, d.text, d.suff, d.bwt)]
    torch.cuda.synchronize()
    sh.load_soa(*arrs, first=a, device=True)
    sh.ctx.synchronize()


@pytest.mark.parametrize("kind,xyz", RU.LOADERS + [("soa_dev", (4, 4, 4))],
                         ids=[f"{k}{''.join(map(str, x))}" for k, x in RU.LOADERS + [("soa_dev", (4, 4, 4))]])
def test_loaders_one_sm(ctxs, kind, xyz, gesa_file):  # noqa: F811
    """about 1 M positions loaded whole and in pieces with edges off every multiple of 64, then e2s_pipeline_resident"""
    ctx = ctxs(1)
    d = RU.data(3).cut(1_000_003)
    ctx.stage_reads(d.reads, d.off)
    w = RU.want(d, xyz=xyz, bcr=kind == "bcr")
    rng = np.random.default_rng(sum(xyz) + len(kind))
    sh = ctx.shard(d.n)
    try:
        for whole in (True, False):
            for a, b in ([(0, d.n)] if whole else RU.pieces(d.n, rng)):
                if kind == "soa_dev":
                    load_soa_dev(sh, d, a, b)
                else:
                    RU.load(sh, d, kind, xyz, a, b, gesa_file)
            sh.seal()
            res = sh.pipeline_resident(RU.params(d), 16, 2)
            RU.check_step(sh, res, d, w, 5, (kind, xyz, whole))
    finally:
        sh.close()


@pytest.mark.parametrize("lean", [False, True])
def test_chunked_loads_one_sm(ctxs, lean):
    """a chunked shard over the same index: e2s_shard_load_soa, or the lean e2s_shard_load_lcp_bwt with text / suff from the
    host's pairSA (e2s_shard_host_gsa), chunks of 5 * 16384 + 1 positions; both tools against the oracle"""
    ctx = ctxs(1)
    d = RU.data(3).cut(1_000_003)
    ctx.stage_reads(d.reads, d.off)
    sh = ctx.shard(d.n, 0, d.n, chunk_positions=5 * T + 1)
    try:
        RU.scan_pass(sh, d, lean=lean)
    finally:
        sh.close()


# ---------------------------------------------------------------------------------------------------------------------------
# (F) both builds of the scan
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("occ", [3, 4])
def test_both_scan_builds(built, occ):
    """k_cluster_scan<3> and <4>: the process keeps the build it picked first, so each runs in a child process of its own"""
    if os.environ.get(CHILD):
        pytest.skip("already in a child process")
    env = dict(os.environ, E2S_SCAN_OCC=str(occ))
    env[CHILD] = "1"
    sel = "(test_scan_tile_boundaries or test_phase2_designed or test_segment_overflow) and (sm1 or smdev)"
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "gpu", "-p", "no:cacheprovider", "-k", sel,
                        os.path.join(ROOT, "tests", "test_grid_rounds_gpu.py")], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and " failed" not in r.stdout, r.stdout[-2000:]


# ---------------------------------------------------------------------------------------------------------------------------
# (G) the default geometry at production size
# ---------------------------------------------------------------------------------------------------------------------------
def big_case():
    """n = 4 * 16384 * 1024 + 12 345: with at most 1024 scan CTAs each scans 4 tiles or more at any SM count.  A volume case
    of 600 000 designed clusters with the boundary features of (A) planted over it; rows outside clusters point inside reads."""
    n = 4 * T * 1024 + 12345
    case = P.volume_case(n_clusters=600_000, n_pos=n, seed=901)
    rng = np.random.default_rng(902)
    lcp = plant(case.lcp.copy(), P.K, rot=1)
    bg = case.lcp == 0
    text, suff = case.text.copy(), case.suff.copy()
    text[bg] = rng.integers(0, len(case.off) - 1, size=int(bg.sum()))
    suff[bg] = 40
    return P.Case("big", lcp, text, suff, case.bwt, case.bases, case.off, case.nreads1, case.params, case.pval, 0, [], {})


def test_default_geometry_production_size(ctxs, monkeypatch):
    ctx = ctxs(0)
    case = big_case()
    n = case.n
    es, el, enc, _ = O.cluster_lm(case.lcp, case.bwt, P.K, P.MIN_LEN)
    ost = O.statistics(es, el, case.params["mcov_out"], case.pval)
    otext, ores = O.find_events(case.lcp, case.text, case.suff, case.bwt, es, el, case.oparams(), ost.max_clust_length, case.bases,
                                case.off)
    assert ores.n_candidates > 50_000
    ctx.stage_reads(case.bases, case.off)
    p = PP.params(case)
    sh = PP.resident(ctx, case)
    try:
        res = sh.pipeline_resident(p, P.K, P.MIN_LEN)
        assert (res.n_written, res.n_clust_out, res.max_clust_length) == (len(es), enc, ost.max_clust_length)
        assert sh.cluster_fetch_packed() == O.clusters_to_bytes(es, el)
        PP.check(res.snp, api.events_format(sh.events(), p), (otext, ores), "resident")
    finally:
        sh.close()
    monkeypatch.setenv("E2S_CHUNK_POSITIONS", str(1 << 25))
    rec = synth.gesa_records(dict(lcp=case.lcp, text=case.text, suff=case.suff, bwt=case.bwt, n=n)).view(np.uint8).reshape(-1)
    rec10 = np.empty((len(es) + 16) * 10, dtype=np.uint8)
    evbuf = (api.Event * (ores.n_candidates + 16))()
    res = ctx.pipeline_host(rec, n, case.bases, case.off, p, P.K, P.MIN_LEN, rec10=rec10, events=evbuf)
    assert res.n_written == len(es) and rec10[: len(es) * 10].tobytes() == O.clusters_to_bytes(es, el)
    assert (res.n_clust_out, res.max_clust_length) == (enc, ost.max_clust_length)
    PP.check(res.snp, api.events_format(list(evbuf)[: res.snp.n_variants], p), (otext, ores), "pipeline_host")


# ---------------------------------------------------------------------------------------------------------------------------
# (H) the CLIs at one SM
# ---------------------------------------------------------------------------------------------------------------------------
def test_clis_one_sm(built, tmp_path, monkeypatch):
    """ebwt2clust + clust2snp streaming chunks of 16384 positions (E2S_CLI_STREAM=1) on the designed CLI case, and ebwt2clust
    on a 40-tile planted input: the files byte for byte against the oracle's"""
    monkeypatch.setenv("E2S_SM_COUNT", "1")
    monkeypatch.setenv("E2S_CLI_STREAM", "1")
    case, fa, snp = PP.cli_files(str(tmp_path / "designed"))
    want_cl = open(fa + ".clusters", "rb").read()
    os.remove(fa + ".clusters")
    cl, _ = RE.ebwt2clust(fa, P.K, P.MIN_LEN)
    assert cl == want_cl
    otext, ores, _, _ = PP.oracle(case)
    r = subprocess.run([os.path.join(PP.BIN, "clust2snp"), "-i", fa, "-n", str(case.nreads1), *PP.CLI_ARGS, "-x", "4", "-y", "4",
                        "-z", "4"], capture_output=True, text=True, env=dict(os.environ, E2S_CHUNK_POSITIONS=str(T)), timeout=600)
    assert r.returncode == 0, (r.stdout, r.stderr)
    assert open(snp, "rb").read() == otext

    n = 40 * T + 1
    lcp, bwt = planted(n, 16, 0, seed=77, rot=3)
    rng = np.random.default_rng(78)
    rd = RE.ACGT[rng.integers(0, 4, size=(RE.R, RE.L))]
    text, suff, _ = RE.index_arrays(rng, lcp)
    rs = synth.ReadSet(reads=rd, nreads1=RE.NR1, genome1=None, genome2=None, snp_pos=None, indels=[])
    fa = synth.write_dataset(str(tmp_path / "planted"), rs, {"n": n, "lcp": lcp, "text": text, "suff": suff, "bwt": bwt})
    for m in (2, 33):
        es, el, enc, _ = O.cluster_lm(lcp, bwt, 16, m)
        cl, done = RE.ebwt2clust(fa, 16, m)
        assert cl == O.clusters_to_bytes(es, el) and done == enc, m

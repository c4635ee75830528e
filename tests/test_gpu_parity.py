"""-m gpu: the CUDA path, called through the C ABI, against the oracle (bit-exact: all integer work)."""
import os

import numpy as np
import pytest

from ebwt2snp_b200 import api, synth
from oracle import oracle as O
from tests import golden_util as GU
from tests import helpers as H

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(built):
    c = api.Context(0)
    yield c
    c.close()


def run_cluster(ctx, lcp, bwt, k, m):
    n = len(lcp)
    sh = ctx.shard(n)
    sh.load_soa(lcp, None, None, bwt)
    sh.seal()
    nw, nc = sh.cluster_lm(k, m)
    s, l = sh.cluster_fetch()
    sh.close()
    assert nw == len(s)
    return s, l, nc


@pytest.mark.parametrize("case", [0, 1, 2])
def test_cluster_fuzz(ctx, case):
    rng = np.random.default_rng(100 + case)
    sizes = [2, 3, 4, 5, 17, 255, 256, 257, 4095, 4096, 4097, 8191, 8192, 8193, 12289, 40000, 70001, 300000]
    for it, n in enumerate(sizes * 2):
        k = int(rng.choice([1, 2, 3, 5, 16, 70]))
        m = int(rng.choice([1, 2, 3, 8, 33, 34, 200, -3]))  # <= 33: bit-parallel kept count, else the dense count path
        lcp = H.random_lcp(rng, n, k, it % 5)
        bwt = rng.choice(H.BWT_ALPHABET, size=n)
        es, el, enc, _ = O.cluster_lm(lcp, bwt, k, m)
        s, l, nc = run_cluster(ctx, lcp, bwt, k, m)
        assert nc == enc, (n, k, m, it)
        assert np.array_equal(s, es) and np.array_equal(l, el), (n, k, m, it)


def test_cluster_long_wrap(ctx):
    """a 70 000-long run: length wraps mod 2^16 (ref:ebwt2clust.cpp:104)"""
    n = 200000
    lcp = np.zeros(n, dtype=np.uint32)
    lcp[1000:71000] = 40
    lcp[100000:100010] = 20
    bwt = np.full(n, ord("A"), dtype=np.uint8)
    es, el, enc, _ = O.cluster_lm(lcp, bwt, 16, 2)
    s, l, nc = run_cluster(ctx, lcp, bwt, 16, 2)
    assert nc == enc and np.array_equal(s, es) and np.array_equal(l, el)
    assert 70000 - 65536 in set(el.tolist())
    # lengths 65536 (wraps to 0), 65537 (wraps to 1) and 65538 against every kind of min_len
    for run in (65535, 65536, 65537, 65538, 131072, 131073):
        for m in (-1, 1, 2, 3, 40):
            lcp = np.zeros(n, dtype=np.uint32)
            lcp[777:777 + run] = 40
            lcp[190000:190003] = 17
            es, el, enc, _ = O.cluster_lm(lcp, bwt, 16, m)
            s, l, nc = run_cluster(ctx, lcp, bwt, 16, m)
            assert nc == enc and np.array_equal(s, es) and np.array_equal(l, el), (run, m)


@pytest.mark.parametrize("wide", [0, 1])
def test_cluster_narrow_lcp(ctx, wide, monkeypatch):
    """K1 on the one-byte resident LCP (all values <= 127; built at seal) against the oracle, and the same inputs
    forced onto the 4-byte stream (E2S_LCP_WIDE=1): sizes around the 16384-position tiles of the narrow kernel,
    k on both sides of the byte range, single shards and shards cut at arbitrary positions."""
    monkeypatch.setenv("E2S_LCP_WIDE", str(wide))
    rng = np.random.default_rng(4242)
    sizes = [2, 3, 5, 63, 64, 65, 127, 129, 16383, 16384, 16385, 16387, 32768, 49153, 100003, 262144 + 7]
    for it, n in enumerate(sizes * 2):
        k = int(rng.choice([1, 2, 16, 30, 100, 127, 128, 129, 300]))
        m = int(rng.choice([1, 2, 3, 8, 34]))
        mode = it % 4
        if mode == 0:
            lcp = rng.integers(0, 128, size=n)
        elif mode == 1:
            lcp = np.clip(np.cumsum(rng.integers(-3, 4, size=n)) + min(k, 120), 0, 127)
        elif mode == 2:
            lcp = rng.integers(max(0, min(k, 125) - 1), min(k, 125) + 3, size=n)
        else:
            lcp = rng.choice(np.array([0, 1, 126, 127]), size=n)
        lcp = lcp.astype(np.uint32)
        bwt = rng.choice(H.BWT_ALPHABET, size=n)
        es, el, enc, _ = O.cluster_lm(lcp, bwt, k, m)
        sh = ctx.shard(n)
        sh.load_soa(lcp, None, None, bwt)
        sh.seal()
        assert sh.lcp_bytes_resident() == (4 if wide else 1)
        nw, nc = sh.cluster_lm(k, m)
        s, l = sh.cluster_fetch()
        sh.close()
        assert nc == enc and np.array_equal(s, es) and np.array_equal(l, el), (n, k, m, it)
        if n < 200:
            continue
        nsh = int(rng.integers(2, 5))
        cuts = sorted(set([0, n] + [int(c) for c in rng.integers(2, n - 2, size=nsh - 1)]))
        cuts = [c for i, c in enumerate(cuts) if i == 0 or c - cuts[i - 1] >= 2 or c == n]
        if n - cuts[-2] < 2:
            cuts.pop(-2)
        sums, recs = [], []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            sh = ctx.shard(hi - lo, lo, n)
            a, b = max(0, lo - 2), min(n, hi + 151)
            sh.load_soa(lcp[a:b], None, None, bwt[a:b], first=a)
            sh.seal()
            assert sh.lcp_bytes_resident() == (4 if wide else 1)
            sums.append(sh.cluster_run(k, m))
            sh.cluster_finalize(api.ClusterMerged())
            recs.append(sh.cluster_fetch())
            sh.close()
        S, L, mg = H.assemble(sums, recs)
        assert mg.n_clust_out == enc and np.array_equal(S, es) and np.array_equal(L, el), (it, cuts)


def test_lcp_above_127(ctx):
    """LCP values above 127 (reads of 128 bases and more) are saturated in the bit-sliced copy: the one-pass scan stays exact
    for -k <= 127 (the descent plane comes from the exact values); -k > 127 goes to the 4-byte kernels.  Both against the oracle."""
    n = 50000
    lcp = np.full(n, 20, dtype=np.uint32)
    bwt = np.full(n, ord("C"), dtype=np.uint8)
    for pos in (0, 1, 16384, n - 1):
        l2 = lcp.copy()
        l2[pos] = 128
        sh = ctx.shard(n)
        sh.load_soa(l2, None, None, bwt)
        sh.seal()
        assert sh.lcp_bytes_resident() == 1
        for k in (16, 128):
            es, el, enc, _ = O.cluster_lm(l2, bwt, k, 2)
            if len(es) == 0:
                continue
            nw, nc = sh.cluster_lm(k, 2)
            s, l = sh.cluster_fetch()
            assert nc == enc and np.array_equal(s, es) and np.array_equal(l, el), (pos, k)
        sh.close()
    rng = np.random.default_rng(128)
    for it, n in enumerate([16385, 100003, 262144 + 7, 300001]):
        for k in (1, 16, 100, 127, 128, 150, 260):
            m = int(rng.choice([1, 2, 3, 8, 33]))
            if it % 2:  # random walks around 127 / around k: runs above and below both thresholds, local minima among saturated values
                lcp = np.clip(np.cumsum(rng.integers(-3, 4, size=n)) + (125 if it == 1 else k), 0, 255).astype(np.uint32)
            else:
                lcp = rng.choice(np.array([0, 1, k - 1 if k > 1 else 0, k, k + 1, 126, 127, 128, 129, 200, 255, 70000], dtype=np.uint32), size=n)
            bwt = rng.choice(H.BWT_ALPHABET, size=n)
            es, el, enc, _ = O.cluster_lm(lcp, bwt, k, m)
            if len(es) == 0:
                continue
            sh = ctx.shard(n)
            sh.load_soa(lcp, None, None, bwt)
            sh.seal()
            nw, nc = sh.cluster_lm(k, m)
            s, l = sh.cluster_fetch()
            sh.close()
            assert nc == enc and np.array_equal(s, es) and np.array_equal(l, el), (it, n, k, m)


def test_cluster_sharded(ctx):
    """shards run one after the other on the same GPU + host merge == single pass (SURVEY.md §4 item 4)"""
    rng = np.random.default_rng(7)
    for it in range(24):
        n = int(rng.integers(30, 30000))
        k = int(rng.choice([2, 5, 16]))
        m = int(rng.choice([1, 2, 3, 40]))
        lcp = H.random_lcp(rng, n, k, it % 5)
        bwt = rng.choice(H.BWT_ALPHABET, size=n)
        es, el, enc, _ = O.cluster_lm(lcp, bwt, k, m)
        nsh = int(rng.integers(2, 6))
        cuts = sorted(set([0, n] + [int(c) for c in rng.integers(2, n - 2, size=nsh - 1)]))
        cuts = [c for i, c in enumerate(cuts) if i == 0 or c - cuts[i - 1] >= 2 or c == n]
        if n - cuts[-2] < 2:
            cuts.pop(-2)
        sums, recs = [], []
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            sh = ctx.shard(hi - lo, lo, n)
            a, b = max(0, lo - 2), min(n, hi + 151)
            sh.load_soa(lcp[a:b], None, None, bwt[a:b], first=a)
            sh.seal()
            sums.append(sh.cluster_run(k, m))
            mg1 = api.cluster_merge([sums[-1]], 0) if (lo == 0 and hi == n) else None
            # own records only (no merge applied yet)
            sh.cluster_finalize(api.ClusterMerged())
            recs.append(sh.cluster_fetch())
            # emulation agrees with the kernel's summary
            es_, rs_, rl_ = H.emulate_shard(lcp, bwt, lo, hi, k, m)
            for f, _ in api.ClusterSummary._fields_:
                assert getattr(sums[-1], f) == getattr(es_, f), (f, it, lo, hi)
            assert np.array_equal(recs[-1][0], rs_) and np.array_equal(recs[-1][1], rl_)
            sh.close()
        S, L, mg = H.assemble(sums, recs)
        assert mg.n_clust_out == enc, (it, cuts)
        assert np.array_equal(S, es) and np.array_equal(L, el), (it, cuts)


@pytest.mark.parametrize("name,seed", [("tiny", 1), ("tiny", 2), ("small", 1)])
def test_pipeline_vs_oracle(ctx, name, seed):
    rs, e = H.dataset(name, seed)
    n = e["n"]
    k, m = 16, 2
    es, el, enc, _ = O.cluster_lm(e["lcp"], e["bwt"], k, m)
    sh = ctx.shard(n)
    rec = synth.gesa_records(e)
    sh.load_gesa(rec.view(np.uint8).reshape(-1), 0, n)
    sh.seal()
    nw, nc = sh.cluster_lm(k, m)
    s, l = sh.cluster_fetch()
    assert nc == enc and np.array_equal(s, es) and np.array_equal(l, el)
    assert sh.cluster_fetch_packed() == O.clusters_to_bytes(es, el)

    # (k_left <= 32 takes K4's one-position-per-lane ballot paths, k_left > 32 the strided ones; 32 is the boundary)
    for kw in ({}, {"mcov_out": 3}, {"consensus_reads": 3, "max_gap": 4}, {"k_left": 25, "k_right": 20, "max_err": 1},
               {"k_left": 32, "max_gap": 32}, {"k_left": 40, "k_right": 35, "max_gap": 12}, {"k_left": 33, "max_err": 0}):
        p = api.default_params(rs.nreads1, **kw)
        op = O.default_params(rs.nreads1, **kw)
        st = sh.statistics(p.mcov_out, p.pval)
        ost = O.statistics(es, el, op.mcov_out, op.pval)
        assert list(st.hist) == list(ost.hist) and st.n_clust == ost.n_clust and st.n_bases == ost.n_bases
        assert st.max_clust_length == ost.max_clust_length and st.max_len == ost.max_len
        off = O.uniform_read_offsets(*rs.reads.shape)
        ctx.stage_reads(rs.reads, off)
        cnt = sh.find_events(p, st.max_clust_length)
        otext, ores = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], es, el, op, ost.max_clust_length, rs.reads, off)
        assert (cnt.n_analysed, cnt.n_candidates, cnt.n_variants, cnt.n_events) == (
            ores.n_analysed, ores.n_candidates, ores.n_variants, ores.n_events), kw
        text = api.events_format(sh.events(), p)
        assert text == otext, kw
    sh.close()


def _load_layout(ctx, e, lay):
    """shard loaded the way the CLI would for this index layout"""
    n = e["n"]
    sh = ctx.shard(n)
    if lay["bcr"]:
        sh.load_soa(e["lcp"], e["text"], e["suff"], e["bwt"])
        sh.set_layout(lay["x"], lay["y"], lay["z"], True)
    else:
        rec = synth.gesa_records(e, lay["x"], lay["y"], lay["z"])
        sh.load_gesa(rec.view(np.uint8).reshape(-1), 0, n, x=lay["x"], y=lay["y"], z=lay["z"])
    sh.seal()
    return sh


@pytest.mark.parametrize("name", ["micro_a", "micro_b"])
def test_golden_vs_reference_outputs(ctx, name):
    """the committed outputs of the UNMODIFIED reference (tests/golden): default layout x 6 option sets, and 5 other
    index layouts (narrow fields, 8-byte fields, BCR triple)"""
    g = GU.micro(name)
    e = g["egsa"]
    off = O.uniform_read_offsets(*g["reads"].shape)
    ctx.stage_reads(g["reads"], off)
    base = dict(x=4, y=4, z=4, bcr=False)
    sh = _load_layout(ctx, e, base)
    nw, nc = sh.cluster_lm(g["k"], g["m"])
    assert sh.cluster_fetch_packed() == g["clusters"] and (nc & 0xFFFFFFFF) == g["n_clust_out"]
    for v in g["variants"]:
        p = api.default_params(g["nreads1"], **GU.params_kw(v["args"]))
        st = sh.statistics(p.mcov_out, p.pval)
        assert (2 * p.mcov_out, st.max_clust_length) == v["allowed"]
        cnt = sh.find_events(p, st.max_clust_length)
        if v["rc"] == 0:
            assert cnt.n_candidates == v["ncand"] and api.events_format(sh.events(), p) == v["snp"], v["args"]
        else:
            assert cnt.n_candidates == 0
    sh.close()
    for lay in g["layouts"]:
        sh = _load_layout(ctx, e, lay)
        nw, nc = sh.cluster_lm(g["k"], g["m"])
        assert sh.cluster_fetch_packed() == lay["clusters"] and (nc & 0xFFFFFFFF) == lay["n_clust_out"], lay
        p = api.default_params(g["nreads1"])
        st = sh.statistics(p.mcov_out, p.pval)
        assert (2 * p.mcov_out, st.max_clust_length) == lay["allowed"]
        cnt = sh.find_events(p, st.max_clust_length)
        assert cnt.n_candidates == lay["ncand"] and api.events_format(sh.events(), p) == lay["snp"], lay
        sh.close()


def test_phantom_tail_vs_reference(ctx):
    """the post-EOF phantom record for 11 width combinations x {EGSA, BCR}: candidate counts printed by the reference"""
    reads = np.frombuffer(b"ACGT", dtype=np.uint8).reshape(1, 4)
    ctx.stage_reads(reads, O.uniform_read_offsets(1, 4))
    checked = 0
    for c in GU.phantom_tail_cases():
        n = len(c["lcp"])
        sh = ctx.shard(n)
        sh.load_soa(c["lcp"], c["text"], c["suff"], c["bwt"])
        sh.set_layout(c["x"], c["y"], c["z"], c["bcr"])
        sh.seal()
        sh.cluster_lm(16, 2)
        assert sh.cluster_fetch_packed() == c["clusters"], c["ci"]
        for n1, ncand in c["readouts"]:
            p = api.default_params(n1, k_left=1, k_right=1, max_gap=1)
            st = sh.statistics(p.mcov_out, p.pval)
            try:
                cnt = sh.find_events(p, st.max_clust_length)
            except api.E2SError as err:  # the candidate's reads do not exist (the reference goes on to crash there)
                assert err.code == api.ERR_UNSUPPORTED
                cnt = err.counts
            assert cnt.n_candidates == ncand, (c["x"], c["y"], c["z"], c["bcr"], n1)
            checked += 1
        sh.close()
    assert checked == 132


def test_phase1_golden_gpu(ctx):
    for c in list(GU.phase1_cases()) + list(GU.phase1_width_cases()):
        n = len(c["lcp"])
        sh = ctx.shard(n)
        sh.load_soa(c["lcp"], None, None, c["bwt"])
        sh.set_layout(c.get("x", 4), c.get("y", 4), c.get("z", 4), False)
        sh.seal()
        nw, nc = sh.cluster_lm(c["k"], c["m"])
        assert sh.cluster_fetch_packed() == c["clusters"] and (nc & 0xFFFFFFFF) == c["n_clust_out"], (n, c["k"], c["m"])
        sh.close()


def test_phase2_capacity_retry(ctx, monkeypatch):
    """the survivor / flagged lists start from a capacity guess; an overflow must be detected and the pass repeated"""
    rs, e = H.dataset("small", 1)
    n = e["n"]
    es, el, _, _ = O.cluster_lm(e["lcp"], e["bwt"], 16, 2)
    off = O.uniform_read_offsets(*rs.reads.shape)
    ctx.stage_reads(rs.reads, off)
    p, op = api.default_params(rs.nreads1), O.default_params(rs.nreads1)
    ost = O.statistics(es, el, op.mcov_out, op.pval)
    otext, ores = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], es, el, op, ost.max_clust_length, rs.reads, off)
    assert ores.n_candidates > 8
    for first_cap in ("1", "7"):
        monkeypatch.setenv("E2S_SNP_FIRST_CAPACITY", first_cap)
        sh = ctx.shard(n)
        sh.load_soa(e["lcp"], e["text"], e["suff"], e["bwt"])
        sh.seal()
        sh.cluster_lm(16, 2)
        st = sh.statistics(p.mcov_out, p.pval)
        cnt = sh.find_events(p, st.max_clust_length)
        assert cnt.n_candidates == ores.n_candidates and api.events_format(sh.events(), p) == otext
        sh.close()


def test_phase2_capacity_retry_fused(ctx, monkeypatch):
    """the same on the fused path (e2s_pipeline_resident: the survivor list comes from the scan, K3a does not run): the
    flagged list must be able to grow up to the length of THAT list, whatever the capacity guess was"""
    rs, e = H.dataset("small", 1)
    n = e["n"]
    es, el, _, _ = O.cluster_lm(e["lcp"], e["bwt"], 16, 2)
    off = O.uniform_read_offsets(*rs.reads.shape)
    ctx.stage_reads(rs.reads, off)
    p, op = api.default_params(rs.nreads1), O.default_params(rs.nreads1)
    ost = O.statistics(es, el, op.mcov_out, op.pval)
    otext, ores = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], es, el, op, ost.max_clust_length, rs.reads, off)
    for first_cap in ("1", "5"):
        monkeypatch.setenv("E2S_SNP_FIRST_CAPACITY", first_cap)
        sh = ctx.shard(n)
        sh.load_soa(e["lcp"], e["text"], e["suff"], e["bwt"])
        sh.seal()
        res = sh.pipeline_resident(p, 16, 2)
        assert res.snp.n_candidates == ores.n_candidates and api.events_format(sh.events(), p) == otext
        sh.close()


def test_rejects_unsorted_clusters(ctx):
    """the reference silently mis-joins unsorted / overlapping records (ref:clust2snp.cpp:818-833); here: E2S_ERR_UNSUPPORTED"""
    rs, e = H.dataset("tiny", 1)
    n = e["n"]
    ctx.stage_reads(rs.reads, O.uniform_read_offsets(*rs.reads.shape))
    sh = ctx.shard(n)
    sh.load_soa(e["lcp"], e["text"], e["suff"], e["bwt"])
    sh.seal()
    sh.stage_clusters(np.array([500, 100, 900], dtype=np.uint64), np.array([20, 20, 20], dtype=np.uint16))
    with pytest.raises(api.E2SError) as ei:
        sh.find_events(api.default_params(rs.nreads1), 150)
    assert ei.value.code == api.ERR_UNSUPPORTED
    sh.stage_clusters(np.array([100, 110], dtype=np.uint64), np.array([20, 20], dtype=np.uint16))  # overlap
    with pytest.raises(api.E2SError):
        sh.find_events(api.default_params(rs.nreads1), 150)
    sh.close()


@pytest.mark.parametrize("name,seed", [("tiny", 3), ("small", 2)])
def test_fused_prefilter_equals_two_phase(ctx, name, seed, monkeypatch):
    """e2s_pipeline_resident / e2s_cluster_prefilter: K2 runs clust2snp's BWT prefilter while writing the records.
    Same events as the two-phase path and as the oracle, for several -m, incl. sharded runs (adopted records)."""
    rs, e = H.dataset(name, seed)
    n = e["n"]
    es, el, _, _ = O.cluster_lm(e["lcp"], e["bwt"], 16, 2)
    off = O.uniform_read_offsets(*rs.reads.shape)
    ctx.stage_reads(rs.reads, off)
    for mcov in (5, 3, 8):
        p, op = api.default_params(rs.nreads1, mcov_out=mcov), O.default_params(rs.nreads1, mcov_out=mcov)
        ost = O.statistics(es, el, mcov, op.pval)
        otext, ores = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], es, el, op, ost.max_clust_length, rs.reads, off)
        sh = ctx.shard(n)
        sh.load_soa(e["lcp"], e["text"], e["suff"], e["bwt"])
        sh.seal()
        res = sh.pipeline_resident(p, 16, 2)
        assert sh.cluster_fetch_packed() == O.clusters_to_bytes(es, el)
        assert (res.snp.n_analysed, res.snp.n_candidates, res.snp.n_events) == (ores.n_analysed, ores.n_candidates, ores.n_events), mcov
        assert res.max_clust_length == ost.max_clust_length
        assert api.events_format(sh.events(), p) == otext, mcov
        # a different -m afterwards must not reuse the armed prefilter's list
        p2 = api.default_params(rs.nreads1, mcov_out=mcov + 1)
        st2 = sh.statistics(p2.mcov_out, p2.pval)
        sh.find_events(p2, st2.max_clust_length)
        op2 = O.default_params(rs.nreads1, mcov_out=mcov + 1)
        ost2 = O.statistics(es, el, mcov + 1, op2.pval)
        assert api.events_format(sh.events(), p2) == O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], es, el, op2, ost2.max_clust_length, rs.reads, off)[0]
        sh.close()
    # sharded, fused: every record is prefiltered by the shard that wrote it or adopted by the shard that analyses it
    p, op = api.default_params(rs.nreads1), O.default_params(rs.nreads1)
    ost = O.statistics(es, el, 5, op.pval)
    otext, ores = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], es, el, op, ost.max_clust_length, rs.reads, off)
    cuts = [0, n // 3 + 7, 2 * n // 3 - 11, n]
    shards, sums = [], []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        sh = ctx.shard(hi - lo, lo, n)
        a, b = max(0, lo - 2), min(n, hi + 151)
        sh.load_soa(e["lcp"][a:b], e["text"][a:b], e["suff"][a:b], e["bwt"][a:b], first=a)
        sh.seal()
        sh.cluster_prefilter(5)
        sums.append(sh.cluster_run(16, 2))
        shards.append(sh)
    texts, first_id, ncand = [], 1, 0
    for g, sh in enumerate(shards):
        sh.cluster_finalize(api.cluster_merge(sums, g))
        cnt = sh.find_events(p, ost.max_clust_length)
        texts.append(api.events_format(sh.events(), p, first_id=first_id))
        first_id += cnt.n_events
        ncand += cnt.n_candidates
        sh.close()
    assert ncand == ores.n_candidates and b"".join(texts) == otext


@pytest.mark.parametrize("fused", [False, True])
def test_non_acgt_bwt_bytes_use_exact_planes(ctx, fused):
    """bytes that are neither ACGT nor acgt ('#', 0xff, 'x', 'E') in the BWT: the resident base-code planes built at seal
    (k_bwt_planes) must give every such byte the code of 'A' (ref:include.hpp:277), for K3a and for the fused K2 alike"""
    rs, e = H.dataset("small", 3)
    n = e["n"]
    rng = np.random.default_rng(12)
    bwt = e["bwt"].copy()
    hit = rng.random(n) < 0.02
    bwt[hit] = rng.choice(np.frombuffer(b"#\xffxE", dtype=np.uint8), size=int(hit.sum()))
    es, el, _, _ = O.cluster_lm(e["lcp"], bwt, 16, 2)
    off = O.uniform_read_offsets(*rs.reads.shape)
    ctx.stage_reads(rs.reads, off)
    p, op = api.default_params(rs.nreads1), O.default_params(rs.nreads1)
    ost = O.statistics(es, el, op.mcov_out, op.pval)
    otext, ores = O.find_events(e["lcp"], e["text"], e["suff"], bwt, es, el, op, ost.max_clust_length, rs.reads, off)
    sh = ctx.shard(n)
    sh.load_soa(e["lcp"], e["text"], e["suff"], bwt)
    sh.seal()
    if fused:
        res = sh.pipeline_resident(p, 16, 2)
        cnt = res.snp
    else:
        sh.cluster_lm(16, 2)
        st = sh.statistics(p.mcov_out, p.pval)
        cnt = sh.find_events(p, st.max_clust_length)
    assert (cnt.n_analysed, cnt.n_candidates) == (ores.n_analysed, ores.n_candidates)
    assert api.events_format(sh.events(), p) == otext and ores.n_candidates > 0
    sh.close()


def test_fused_prefilter_overflow_falls_back(ctx, monkeypatch):
    """K2's survivor list is bounded; when it overflows, find_events must ignore it and run its own pass over the BWT"""
    rs, e = H.dataset("small", 1)
    n = e["n"]
    es, el, _, _ = O.cluster_lm(e["lcp"], e["bwt"], 16, 2)
    off = O.uniform_read_offsets(*rs.reads.shape)
    ctx.stage_reads(rs.reads, off)
    p, op = api.default_params(rs.nreads1), O.default_params(rs.nreads1)
    ost = O.statistics(es, el, op.mcov_out, op.pval)
    otext, ores = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], es, el, op, ost.max_clust_length, rs.reads, off)
    monkeypatch.setenv("E2S_PF_CAPACITY", "3")
    sh = ctx.shard(n)
    sh.load_soa(e["lcp"], e["text"], e["suff"], e["bwt"])
    sh.seal()
    launches0 = ctx.launches
    res = sh.pipeline_resident(p, 16, 2)
    assert res.snp.n_candidates == ores.n_candidates and res.snp.n_analysed == ores.n_analysed
    assert api.events_format(sh.events(), p) == otext
    monkeypatch.delenv("E2S_PF_CAPACITY")
    fused_launches = None
    sh2 = ctx.shard(n)
    sh2.load_soa(e["lcp"], e["text"], e["suff"], e["bwt"])
    sh2.seal()
    l0 = ctx.launches
    sh2.pipeline_resident(p, 16, 2)
    fused_launches = ctx.launches - l0
    assert api.events_format(sh2.events(), p) == otext
    sh.close()
    sh2.close()
    assert fused_launches >= 5  # scan, k_put?/K3x, K3b, K4 (+ the adopted-record helper)


@pytest.mark.parametrize("fused", [False, True])
def test_wrapped_length_cluster_in_phase2(ctx, fused):
    """a cluster of 65536 + 24 positions is stored with length 24 and clust2snp analyses [start, start + 24): the fused
    prefilter (which sees such a record far from where it starts) must hand it to the exact test"""
    rng = np.random.default_rng(31)
    n, R, L = 200_000, 400, 100
    reads = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=(R, L))]
    lcp = np.zeros(n, dtype=np.uint32)
    lcp[5000:5000 + 65536 + 24] = 40            # one giant run: wrapped length 24
    lcp[150_000:150_030] = 35                    # and an ordinary cluster
    text = rng.integers(0, R, size=n).astype(np.uint32)
    suff = rng.integers(31, 60, size=n).astype(np.uint32)
    bwt = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n)].copy()
    # make both analysed ranges look like SNP clusters: sample 0 (text < 200) all 'A', sample 1 all 'C'
    for lo_, hi_ in ((5000, 5024), (150_000, 150_030)):
        half = (hi_ - lo_) // 2
        text[lo_:lo_ + half] = rng.integers(0, 200, size=half)
        bwt[lo_:lo_ + half] = ord("A")
        text[lo_ + half:hi_] = rng.integers(200, R, size=hi_ - lo_ - half)
        bwt[lo_ + half:hi_] = ord("C")
    es, el, _, _ = O.cluster_lm(lcp, bwt, 16, 2)
    assert 24 in el.tolist()
    off = O.uniform_read_offsets(R, L)
    ctx.stage_reads(reads, off)
    p, op = api.default_params(200), O.default_params(200)
    ost = O.statistics(es, el, op.mcov_out, op.pval)
    otext, ores = O.find_events(lcp, text, suff, bwt, es, el, op, ost.max_clust_length, reads, off)
    assert ores.n_candidates >= 2
    sh = ctx.shard(n)
    sh.load_soa(lcp, text, suff, bwt)
    sh.seal()
    if fused:
        cnt = sh.pipeline_resident(p, 16, 2).snp
    else:
        sh.cluster_lm(16, 2)
        st = sh.statistics(p.mcov_out, p.pval)
        cnt = sh.find_events(p, st.max_clust_length)
    assert cnt.n_candidates == ores.n_candidates and api.events_format(sh.events(), p) == otext
    sh.close()


def test_events_fast_and_general_path_agree(ctx, monkeypatch):
    """K4 takes a short cut when the staged reads hold nothing but ACGT (k_reads_check) and k_left <= 32: same events as the
    general path (E2S_K4_GENERIC), and reads with an N keep it off by themselves"""
    rs, e = H.dataset("small", 2)
    off = O.uniform_read_offsets(*rs.reads.shape)
    p = api.default_params(rs.nreads1)

    def events(reads):
        ctx.stage_reads(reads, off)
        sh = ctx.shard(e["n"])
        sh.load_soa(e["lcp"], e["text"], e["suff"], e["bwt"])
        sh.seal()
        sh.cluster_lm(16, 2)
        st = sh.statistics(p.mcov_out, p.pval)
        cnt = sh.find_events(p, st.max_clust_length)
        text = api.events_format(sh.events(), p)
        sh.close()
        return cnt, text

    c1, t1 = events(rs.reads)
    monkeypatch.setenv("E2S_K4_GENERIC", "1")
    c2, t2 = events(rs.reads)
    monkeypatch.delenv("E2S_K4_GENERIC")
    assert c1.n_events > 0 and (c1.n_candidates, c1.n_events) == (c2.n_candidates, c2.n_events) and t1 == t2
    es, el, _, _ = O.cluster_lm(e["lcp"], e["bwt"], 16, 2)
    op = O.default_params(rs.nreads1)
    ost = O.statistics(es, el, op.mcov_out, op.pval)
    otext, _ = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], es, el, op, ost.max_clust_length, rs.reads, off)
    assert t1 == otext
    # a read that is never used as a context gets an N: the flag keeps K4 on the general path, the events stay the same
    dirty = rs.reads.copy()
    dirty[-1, -1] = ord("N")
    c3, t3 = events(dirty)
    if c3.saw_n == 0:
        assert t3 == t1

"""-m gpu: clust2snp's CUDA paths on the designed phase-2 cases (tests/phase2_cases.py) against the oracle.

Every case, the volume case included, runs the two-phase resident path (cluster_lm -> statistics -> find_events) and the fused
e2s_pipeline_resident.  A subset (every reads variant, -c 33, 100 and 150 with -m 1, k_left 32 / 33 / 128, the volume case)
also runs K4's general path (E2S_K4_GENERIC), three fused shards cut through designed clusters, e2s_pipeline_host /
e2s_pipeline_host_soa with chunk boundaries inside designed clusters, and clust2snp on a chunked shard (lean and not).
Compared: the counts, saw_n and the .snp bytes.  In the case with an N inside a context the reference draws rand() % 4 for it;
the oracle and the CUDA path both count it as 'A', so there only they are compared with each other, together with the saw_n
flag."""
import os
import subprocess

import numpy as np
import pytest

from ebwt2snp_b200 import api, synth
from oracle import oracle as O
from tests import phase2_cases as P

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "ebwt2snp_b200", "bin")
CASES = P.all_cases()
SUBSET = [c for c in CASES if "subset" in c.groups]
CHUNK = 16384


@pytest.fixture(scope="module")
def ctx(built):
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def volume():
    case = P.volume_case()
    return case, oracle(case)


def oracle(case):
    es, el, _, _ = O.cluster_lm(case.lcp, case.bwt, P.K, P.MIN_LEN)
    if case.refuse:
        with pytest.raises(ValueError):
            O.find_events(case.lcp, case.text, case.suff, case.bwt, es, el, case.oparams(), case.max_clust_length, case.bases, case.off)
        return None
    text, res = O.find_events(case.lcp, case.text, case.suff, case.bwt, es, el, case.oparams(), case.max_clust_length, case.bases,
                              case.off)
    return text, res, es, el


def params(case):
    p = api.default_params(case.nreads1, **case.params)
    p.pval = case.pval
    return p


def check(cnt, text, want, what):
    otext, ores = want[0], want[1]
    got = (cnt.n_analysed, cnt.n_candidates, cnt.n_variants, cnt.n_events, bool(cnt.saw_n))
    exp = (ores.n_analysed, ores.n_candidates, ores.n_variants, ores.n_events, bool(ores.flags & O.FLAG_SAW_N))
    assert got == exp, what
    assert text == otext, what


def resident(ctx, case):
    sh = ctx.shard(case.n)
    sh.load_soa(case.lcp, case.text, case.suff, case.bwt)
    sh.seal()
    return sh


def two_phase(ctx, case, want, what):
    ctx.stage_reads(case.bases, case.off)
    p = params(case)
    sh = resident(ctx, case)
    try:
        sh.cluster_lm(P.K, P.MIN_LEN)
        st = sh.statistics(p.mcov_out, p.pval)
        assert st.max_clust_length == case.max_clust_length
        if want is None:
            with pytest.raises(api.E2SError):
                sh.find_events(p, st.max_clust_length)
            return
        cnt = sh.find_events(p, st.max_clust_length)
        check(cnt, api.events_format(sh.events(), p), want, what)
    finally:
        sh.close()


def resident_and_fused(ctx, case, want):
    two_phase(ctx, case, want, "two-phase")
    p = params(case)
    sh = resident(ctx, case)
    try:
        if want is None:
            with pytest.raises(api.E2SError):
                sh.pipeline_resident(p, P.K, P.MIN_LEN)
            return
        res = sh.pipeline_resident(p, P.K, P.MIN_LEN)
        assert res.max_clust_length == case.max_clust_length
        check(res.snp, api.events_format(sh.events(), p), want, "fused")
    finally:
        sh.close()


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_resident_and_fused(ctx, case):
    resident_and_fused(ctx, case, oracle(case))


def test_volume_resident_and_fused(ctx, volume):
    resident_and_fused(ctx, *volume)


SUBSET_IDS = [c.name for c in SUBSET] + ["volume"]


@pytest.fixture(params=SUBSET_IDS)
def sub(request, volume):
    if request.param == "volume":
        return volume
    case = next(c for c in SUBSET if c.name == request.param)
    return case, oracle(case)


def test_subset_covers_the_paths():
    names = set(SUBSET_IDS)
    assert {"cand_c33", "cand_c100", "volume"} <= names
    assert {c.name for c in CASES if "reads" in c.groups} <= names
    for kl in (32, 33, 128):
        assert any(n.startswith(f"ctx_L{kl}_") for n in names)


def test_k4_general_path(ctx, sub, monkeypatch):
    case, want = sub
    monkeypatch.setenv("E2S_K4_GENERIC", "1")
    two_phase(ctx, case, want, "E2S_K4_GENERIC")


def cuts_through_clusters(case, parts=3):
    """shard boundaries at the middle of designed clusters (a third and two thirds into the cluster list)"""
    cl = case.clusters
    if len(cl) >= parts:
        picks = [cl[len(cl) * i // parts] for i in range(1, parts)]
        return [0] + [s + max(1, l // 2) for s, l in picks] + [case.n]
    s, l = cl[0]
    return [0, s + l // 3, s + 2 * l // 3, case.n]


def test_fused_shards_cut_through_clusters(ctx, sub):
    case, want = sub
    ctx.stage_reads(case.bases, case.off)
    p = params(case)
    n = case.n
    cuts = cuts_through_clusters(case)
    assert all(a < b for a, b in zip(cuts[:-1], cuts[1:]))
    shards, sums = [], []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        sh = ctx.shard(hi - lo, lo, n)
        a, b = max(0, lo - 2), min(n, hi + 151)
        sh.load_soa(case.lcp[a:b], case.text[a:b], case.suff[a:b], case.bwt[a:b], first=a)
        sh.seal()
        sh.cluster_prefilter(p.mcov_out)
        sums.append(sh.cluster_run(P.K, P.MIN_LEN))
        shards.append(sh)
    texts, first_id, tot = [], 1, np.zeros(4, dtype=np.int64)
    saw_n = False
    for g, sh in enumerate(shards):
        sh.cluster_finalize(api.cluster_merge(sums, g))
        cnt = sh.find_events(p, case.max_clust_length)
        texts.append(api.events_format(sh.events(), p, first_id=first_id))
        first_id += cnt.n_events
        tot += (cnt.n_analysed, cnt.n_candidates, cnt.n_variants, cnt.n_events)
        saw_n |= bool(cnt.saw_n)
        sh.close()
    otext, ores = want[0], want[1]
    assert tuple(tot) == (ores.n_analysed, ores.n_candidates, ores.n_variants, ores.n_events)
    assert saw_n == bool(ores.flags & O.FLAG_SAW_N)
    assert b"".join(texts) == otext


def shifted(case):
    """the case behind enough LCP-0 records that a chunk boundary (a multiple of CHUNK) falls inside its middle cluster"""
    s, l = case.clusters[len(case.clusters) // 2]
    if case.n > 4 * CHUNK:  # (the volume case: boundaries fall inside clusters by themselves)
        st = np.array([s_ for s_, _ in case.clusters])
        ln = np.array([l_ for _, l_ in case.clusters])
        b = np.arange(CHUNK, case.n, CHUNK)
        j = np.searchsorted(st, b) - 1
        assert np.sum((j >= 0) & (st[j] + ln[j] > b) & (st[j] < b)) > 20
        return case, 0
    pad = CHUNK - (s + l // 2)
    assert pad > 0

    def ext(a, v):
        return np.concatenate([np.full(pad, v, dtype=a.dtype), a])
    c = P.Case(case.name, ext(case.lcp, 0), ext(case.text, 0), ext(case.suff, 0), ext(case.bwt, ord("T")), case.bases, case.off,
               case.nreads1, case.params, case.pval, case.max_clust_length, [(s_ + pad, l_) for s_, l_ in case.clusters],
               case.expect, case.refuse, case.groups, case.note)
    assert c.clusters[len(c.clusters) // 2][0] < CHUNK < sum(c.clusters[len(c.clusters) // 2])
    return c, pad


@pytest.mark.parametrize("lean", [False, True])
def test_pipeline_host_chunk_inside_cluster(ctx, sub, lean, monkeypatch):
    monkeypatch.setenv("E2S_CHUNK_POSITIONS", str(CHUNK))
    pipeline_host_chunked(ctx, sub, lean)


def pipeline_host_chunked(ctx, sub, lean):
    """e2s_pipeline_host (lean: _soa) with a chunk boundary inside a designed cluster; E2S_CHUNK_POSITIONS set by the caller"""
    case, want = sub
    case, pad = shifted(case)
    if pad:
        want = oracle(case)
    otext, ores, es, el = want
    p = params(case)
    n = case.n
    rec10 = np.empty((len(es) + 16) * 10, dtype=np.uint8)
    evbuf = (api.Event * (ores.n_candidates + 16))()
    if lean:
        pair = np.empty(n, dtype=np.dtype([("suff", "<u4"), ("text", "<u4")]))
        pair["suff"], pair["text"] = case.suff, case.text
        res = ctx.pipeline_host_soa(case.lcp.view(np.uint8), case.bwt, pair.view(np.uint8), n, case.bases, case.off, p, P.K,
                                    P.MIN_LEN, 4, 4, 4, rec10=rec10, events=evbuf)
    else:
        rec = synth.gesa_records(dict(lcp=case.lcp, text=case.text, suff=case.suff, bwt=case.bwt, n=n)).view(np.uint8).reshape(-1)
        res = ctx.pipeline_host(rec, n, case.bases, case.off, p, P.K, P.MIN_LEN, rec10=rec10, events=evbuf)
    assert res.n_written == len(es) and rec10[: len(es) * 10].tobytes() == O.clusters_to_bytes(es, el)
    assert res.max_clust_length == case.max_clust_length
    check(res.snp, api.events_format(list(evbuf)[: res.snp.n_variants], p), want, ("pipeline_host_soa" if lean else "pipeline_host"))


@pytest.mark.parametrize("lean", [False, True])
def test_chunked_clust2snp(ctx, sub, lean):
    chunked_clust2snp(ctx, sub, lean)


def chunked_clust2snp(ctx, sub, lean):
    """clust2snp on a chunked shard of CHUNK positions (lean: text / suff from the host's pairSA)"""
    case, want = sub
    case, pad = shifted(case)
    if pad:
        want = oracle(case)
    otext, ores, es, el = want
    p = params(case)
    n = case.n
    ctx.stage_reads(case.bases, case.off)
    rec10 = np.frombuffer(O.clusters_to_bytes(es, el), dtype=np.uint8)
    pair = np.empty(n, dtype=np.dtype([("suff", "<u4"), ("text", "<u4")]))
    pair["suff"], pair["text"] = case.suff, case.text
    pair = pair.view(np.uint8)
    sh = ctx.shard(n, 0, n, chunk_positions=CHUNK)
    try:
        if lean:
            sh.host_gsa(pair, 4, 4)
        for clo, cn in sh.chunks():
            sh.chunk_begin(clo, cn)
            a, b = max(0, clo - 176), min(n, clo + cn + 152)
            if lean:
                sh.load_bcr(case.lcp[a:b].view(np.uint8), case.bwt[a:b], None, 4, 4, 4, first=a)
                sh.set_layout(4, 4, 4, True)
            else:
                sh.load_soa(case.lcp[a:b], case.text[a:b], case.suff[a:b], case.bwt[a:b], first=a)
            r0, r1 = np.searchsorted(es, clo), np.searchsorted(es, clo + cn)
            sh.chunk_stage_clusters(rec10[r0 * 10:r1 * 10], p.mcov_out, case.max_clust_length)
        sh.chunked_clusters_finish()
        cnt = sh.find_events(p, case.max_clust_length)
        check(cnt, api.events_format(sh.events(), p), want, "chunked clust2snp")
    finally:
        sh.close()


def test_volume_exceeds_one_round(ctx, volume):
    """the volume case needs several K3x / K3b / K4 rounds on this device and overflows the first flagged-list guess"""
    import torch
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    case, (otext, ores, es, el) = volume
    assert ores.n_candidates > sm * 16 * 32 and ores.n_candidates > sm * 8 * 8 and ores.n_candidates > sm * 16 * 4
    assert ores.n_candidates > len(es) // 256 + 2048


# ---- the clust2snp CLI ----------------------------------------------------------------------------------------------------
def write_fasta(path, case):
    with open(path, "wb") as f:
        for i in range(len(case.off) - 1):
            f.write(b">r%d\n" % i + case.bases[int(case.off[i]):int(case.off[i + 1])].tobytes() + b"\n")


CLI_ARGS = ["-c", "100", "-L", "40", "-R", "33", "-g", "12", "-e", "1", "-p", "1"]


def cli_files(d):
    case = P.cli_case()
    assert dict(consensus_reads=100, k_left=40, k_right=33, max_gap=12, max_err=1).items() <= case.params.items()
    os.makedirs(d, exist_ok=True)
    fa = os.path.join(d, "designed.fasta")
    write_fasta(fa, case)
    synth.write_gesa(fa + ".gesa", dict(lcp=case.lcp, text=case.text, suff=case.suff, bwt=case.bwt, n=case.n))
    es, el, _, _ = O.cluster_lm(case.lcp, case.bwt, P.K, P.MIN_LEN)
    with open(fa + ".clusters", "wb") as f:
        f.write(O.clusters_to_bytes(es, el))
    return case, fa, os.path.join(d, "designed.snp")


@pytest.mark.parametrize("stream", [False, True])
def test_cli_ragged_designed(built, tmp_path, stream):
    case, fa, snp = cli_files(str(tmp_path))
    otext, ores, _, _ = oracle(case)
    assert ores.n_events == 7
    env = dict(os.environ)
    if stream:
        env.update(E2S_CLI_STREAM="1", E2S_CHUNK_POSITIONS=str(CHUNK))
    r = subprocess.run([os.path.join(BIN, "clust2snp"), "-i", fa, "-n", str(case.nreads1), *CLI_ARGS, "-x", "4", "-y", "4", "-z", "4"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, (r.stdout, r.stderr)
    assert f"Done. {ores.n_candidates} potential variants" in r.stdout, r.stdout
    assert open(snp, "rb").read() == otext


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref not built")
def test_oracle_vs_reference_on_designed_set(built, tmp_path):
    case, fa, snp = cli_files(str(tmp_path))
    otext, ores, _, _ = oracle(case)
    r, info = O.ref_clust2snp(fa, case.nreads1, extra=CLI_ARGS)
    assert r.returncode == 0 and info.get("n_candidates") == ores.n_candidates
    assert open(snp, "rb").read() == otext

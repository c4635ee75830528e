"""-m gpu: one index over several shards, each built from the reads for its own key range (e2s_reads_key_cuts,
e2s_shard_build_egsa_range, the halo rows).  Checked against inputs the repository already trusts: the oracle's index keys, shards
loaded from the oracle's index with the same halos, e2s_pipeline_reads on the whole index, and the three-tool chain."""
import os
import socket

import numpy as np
import pytest
import torch.multiprocessing as mp

from ebwt2snp_b200 import api, sharding, synth
from oracle import oracle as O
from tests import golden_util as GU
from tests.test_builder_ranges_gpu import index_keys
from tests.test_from_reads_gpu import (BIN, ENV_HOOKS, ROOT, case_reads, chain_outputs, ebwt2snp_outputs, flat, micro_variants,
                                       pipeline_outputs, tool)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(built):
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(autouse=True)
def clean_env(monkeypatch):
    for k in ENV_HOOKS:
        monkeypatch.delenv(k, raising=False)


def ragged(bases, off):
    return int(off[-1]) != (len(off) - 1) * int(np.diff(off.astype(np.int64)).max())


def expected_cuts(bases, off, parts):
    """numpy restatement of e2s_reads_key_cuts' sample: slots k n / m, the builder's slot map, sorted, quantiles, bumped"""
    R = len(off) - 1
    n = int(off[-1]) + R
    m = min(n, 1 << 16)
    slots = np.arange(m, dtype=np.int64) * n // m
    if ragged(bases, off):
        slot0 = off.astype(np.int64) + np.arange(R + 1)
        rows = np.searchsorted(slot0, slots, side="right") - 1
        cols = slots - slot0[rows]
    else:
        L = int(off[1])
        q = slots // R
        rows, cols = slots - q * R, L - q
    keys = np.sort(sharding.first_key_words((bases, off), rows, cols))
    cuts = [0] + [int(keys[i * m // parts]) for i in range(1, parts)]
    for i in range(1, parts):
        cuts[i] = max(cuts[i], cuts[i - 1] + 1)
    return cuts


# ---- 1. key cuts -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("parts", [2, 3, 8])
@pytest.mark.parametrize("name", ["micro_a", "micro_b", "genome", "long"])
def test_key_cuts(ctx, name, parts):
    bases, off = case_reads(name)
    want = O.build_egsa_ragged(bases, off)
    n = want["n"]
    keys = np.sort(index_keys(bases, off, want))
    ctx.stage_reads(bases, off)
    key_lo, pos = ctx.key_cuts(off, parts)
    assert [int(v) for v in key_lo] == expected_cuts(bases, off, parts)
    assert all(int(a) < int(b) for a, b in zip(key_lo[:-1], key_lo[1:]))
    assert int(pos[-1]) == n and all(int(b) - int(a) >= 2 for a, b in zip(pos[:-1], pos[1:]))
    for i in range(parts):
        assert int(pos[i]) == int(np.searchsorted(keys, key_lo[i], side="left")), i
    again = ctx.key_cuts(off, parts)
    assert np.array_equal(again[0], key_lo) and np.array_equal(again[1], pos)
    with pytest.raises(api.E2SError) as ei:
        ctx.key_cuts(off, n // 2 + 1)
    assert ei.value.code == api.ERR_UNSUPPORTED


# ---- 2. built shards = loaded shards ----------------------------------------------------------------------------------------
def built_shards(ctx, off, key_lo, pos, x, y, z):
    """every shard built for its key range, the halo rows applied, sealed"""
    G, n = len(key_lo), int(pos[-1])
    shards = []
    for g in range(G):
        sh = ctx.shard(int(pos[g + 1]) - int(pos[g]), int(pos[g]), n)
        sh.build_egsa_range(off, int(key_lo[g]), int(key_lo[g + 1]) if g + 1 < G else 0, x, y, z)
        shards.append(sh)
    rows = np.stack([sh.halo_row() for sh in shards])
    for g, sh in enumerate(shards):
        sh.halo_apply(rows, g)
        sh.seal()
    return shards


def loaded_shards(ctx, want, pos, x, y, z):
    """the same positions of the oracle's index loaded with 2 positions of left and 151 of right halo"""
    rec = synth.gesa_records(want, x, y, z).view(np.uint8).reshape(-1)
    rs, n = x + y + z + 1, int(pos[-1])
    shards = []
    for g in range(len(pos) - 1):
        lo, hi = int(pos[g]), int(pos[g + 1])
        a, b = max(lo - 2, 0), min(hi + api.MAX_C_LEN + 1, n)
        sh = ctx.shard(hi - lo, lo, n)
        sh.load_gesa(rec[a * rs:b * rs], a, b - a, x, y, z)
        sh.seal()
        shards.append(sh)
    return shards


def host_sequence(shards, p, k, m):
    """the host-driven multi-shard sequence -> per shard: (summary, .clusters slice, lcp bytes, merged, statistics, counts, events)"""
    G = len(shards)
    sums, own = [], []
    for sh in shards:
        sh.cluster_prefilter(p.mcov_out)
        sums.append(sh.cluster_run(k, m))
        own.append(sh.statistics(finish=False))
    sum_rows, stat_rows = (api.ClusterSummary * G)(*sums), (api.Stats * G)(*own)
    out = []
    for g, sh in enumerate(shards):
        mg, st = api.exchange_finish(sum_rows, stat_rows, g, p.mcov_out, p.pval)
        sh.cluster_finalize(mg)
        cnt = sh.find_events(p, st.max_clust_length)
        out.append((bytes(sums[g]), sh.cluster_fetch_packed(), sh.lcp_bytes_resident(), bytes(mg), bytes(st), bytes(cnt),
                    [bytes(e) for e in sh.events()]))
    for sh in shards:
        sh.close()
    return out


def built_vs_loaded(ctx, bases, off, want, key_lo, pos, p, k, m, xyz=(4, 4, 4)):
    ctx.stage_reads(bases, off)
    got = host_sequence(built_shards(ctx, off, key_lo, pos, *xyz), p, k, m)
    ref = host_sequence(loaded_shards(ctx, want, pos, *xyz), p, k, m)
    for g, (a, b) in enumerate(zip(got, ref)):
        assert a == b, (g, xyz)
    return got


STEP_CASES = [("micro_a", 16, 2), ("micro_b", 16, 2), ("genome", 16, 2), ("long", 16, 2), ("long", 128, 2), ("min_len_34", 16, 34)]


@pytest.mark.parametrize("parts", [2, 3, 8])
@pytest.mark.parametrize("name,k,m", STEP_CASES)
def test_built_shards_equal_loaded_shards(ctx, name, k, m, parts):
    bases, off = case_reads(name)
    want = O.build_egsa_ragged(bases, off)
    p = api.default_params(max(1, (len(off) - 1) // 2))
    ctx.stage_reads(bases, off)
    key_lo, pos = ctx.key_cuts(off, parts)
    built_vs_loaded(ctx, bases, off, want, key_lo, pos, p, k, m)


@pytest.mark.parametrize("xyz", [(1, 4, 1), (2, 4, 2)])
@pytest.mark.parametrize("name", ["genome", "long"])
def test_built_shards_truncated_layouts(ctx, name, xyz):
    bases, off = case_reads(name)
    want = O.build_egsa_ragged(bases, off)
    p = api.default_params((len(off) - 1) // 2)
    ctx.stage_reads(bases, off)
    key_lo, pos = ctx.key_cuts(off, 3)
    built_vs_loaded(ctx, bases, off, want, key_lo, pos, p, 16, 2, xyz)


@pytest.mark.parametrize("name,vi", micro_variants())
def test_built_shards_micro_options(ctx, name, vi):
    g = GU.micro(name)
    bases, off = flat(g["reads"])
    want = O.build_egsa_ragged(bases, off)
    p = api.default_params(g["nreads1"], **GU.params_kw(g["variants"][vi]["args"]))
    ctx.stage_reads(bases, off)
    key_lo, pos = ctx.key_cuts(off, 3)
    for xyz in ((1, 4, 1), (4, 4, 4), (2, 4, 2)):
        built_vs_loaded(ctx, bases, off, want, key_lo, pos, p, g["k"], g["m"], xyz)


def explicit_cut_reads():
    """the genome reads and one read of 33 T: its two longest suffixes are the only ones with 32 T, so a last shard of 2 is possible"""
    bases, off = case_reads("genome")
    bases = np.concatenate([bases, np.frombuffer(b"T" * 33, dtype=np.uint8)])
    off = np.concatenate([off, [off[-1] + 33]]).astype(np.uint64)
    return bases, off


def test_built_shards_explicit_cuts(ctx, monkeypatch):
    """cuts picked from the oracle's index keys: (a) a cluster straddles a cut, (b) a shard of 2 positions, (c) shards shorter than
    the right halo, (d) a last shard of 2 positions; then with sub-ranges forced inside the shards and with 64-bit ids"""
    bases, off = explicit_cut_reads()
    want = O.build_egsa_ragged(bases, off)
    n, k = want["n"], 16
    keys = index_keys(bases, off, want)
    assert np.all(keys[1:] >= keys[:-1])
    ok = np.flatnonzero(keys[1:] != keys[:-1]) + 1  # positions where a cut can fall (a key value is never split)
    lcp = want["lcp"].astype(np.int64)
    okset = set(int(c) for c in ok)
    a = next(int(c) for c in ok[len(ok) // 5:] if lcp[c] >= k and lcp[c - 1] >= k)  # (a): inside a cluster
    b = next(int(c) for c in ok if c > a + 200 and c + 2 in okset)  # (b): [b, b + 2)
    cs = [int(c) for c in ok if c > b + 300][:40]
    c0 = cs[0]
    c1 = next(c for c in cs if 20 <= c - c0 < 140)
    c2 = next(c for c in cs if 20 <= c - c1 < 140)  # (c): [c0, c1) and [c1, c2) shorter than 151
    assert keys[n - 3] < keys[n - 2] and n - 2 > c2 + 200  # (d): [n - 2, n)
    pos = [0, a, b, b + 2, c0, c1, c2, n - 2, n]
    key_lo = [int(keys[q]) if q else 0 for q in pos[:-1]]
    p = api.default_params((len(off) - 1) // 2)
    ref = built_vs_loaded(ctx, bases, off, want, key_lo, pos, p, k, 2)
    head = [np.frombuffer(r[1], dtype=np.uint8) for r in ref]
    assert any(api.ClusterMerged.from_buffer_copy(r[3]).n_prepend for r in ref)  # a cluster did straddle a cut
    assert sum(h.size for h in head) > 0
    cap = max(4096, (b - a) // 3)
    launches = {}
    for env in ({}, {"E2S_BUILD_RANGE_RECORDS": str(cap)}, {"E2S_BUILD_IDS64": "1"}):
        for kk, v in env.items():
            monkeypatch.setenv(kk, v)
        ctx.stage_reads(bases, off)
        l0 = ctx.launches
        shards = built_shards(ctx, off, key_lo, pos, 4, 4, 4)
        launches[tuple(env)] = ctx.launches - l0
        got = host_sequence(shards, p, k, 2)
        for kk in env:
            monkeypatch.delenv(kk)
        assert got == ref, env
    assert launches[("E2S_BUILD_RANGE_RECORDS",)] > launches[()], launches  # the sub-ranges were taken


def test_range_mismatch_is_refused(ctx):
    bases, off = case_reads("genome")
    ctx.stage_reads(bases, off)
    key_lo, pos = ctx.key_cuts(off, 3)
    n = int(pos[-1])
    sh = ctx.shard(int(pos[2]) - int(pos[1]) + 1, int(pos[1]), n)  # one position too many for the key range
    with pytest.raises(api.E2SError) as ei:
        sh.build_egsa_range(off, int(key_lo[1]), int(key_lo[2]), 4, 4, 4)
    assert ei.value.code == api.ERR_ARG
    sh.close()


# ---- 3. sharded = whole ----------------------------------------------------------------------------------------------------
def whole_outputs(ctx, bases, off, p, k, m, xyz):
    n = int(off[-1]) + len(off) - 1
    rc, out = pipeline_outputs(ctx, lambda r, e: ctx.pipeline_reads(bases, off, p, k, m, *xyz, rec10=r, events=e), n)[:2]
    assert rc == 0, out
    return out


def sharded_outputs(ctx, bases, off, parts, p, k, m, xyz):
    ctx.stage_reads(bases, off)
    key_lo, pos = ctx.key_cuts(off, parts)
    out = host_sequence(built_shards(ctx, off, key_lo, pos, *xyz), p, k, m)
    st = api.Stats.from_buffer_copy(out[-1][4])
    mg = api.ClusterMerged.from_buffer_copy(out[-1][3])
    return ((mg.n_clust_out, st.max_clust_length), b"".join(o[1] for o in out), sum((o[6] for o in out), []))


@pytest.mark.parametrize("name,vi", micro_variants())
def test_sharded_equals_whole_micro(ctx, name, vi):
    g = GU.micro(name)
    bases, off = flat(g["reads"])
    p = api.default_params(g["nreads1"], **GU.params_kw(g["variants"][vi]["args"]))
    for xyz in ((1, 4, 1), (4, 4, 4), (2, 4, 2)):
        whole = whole_outputs(ctx, bases, off, p, g["k"], g["m"], xyz)
        for parts in (2, 3):
            mine = sharded_outputs(ctx, bases, off, parts, p, g["k"], g["m"], xyz)
            assert mine == ((whole[0][1], whole[0][2]), whole[1], whole[2]), (xyz, parts)


@pytest.mark.parametrize("name,k,m", [("genome", 16, 2), ("long", 16, 2), ("long", 128, 2), ("min_len_34", 16, 34)])
def test_sharded_equals_whole(ctx, name, k, m):
    bases, off = case_reads(name)
    p = api.default_params((len(off) - 1) // 2)
    for xyz in ((1, 4, 1), (4, 4, 4)):
        whole = whole_outputs(ctx, bases, off, p, k, m, xyz)
        for parts in (2, 3, 8):
            mine = sharded_outputs(ctx, bases, off, parts, p, k, m, xyz)
            assert mine == ((whole[0][1], whole[0][2]), whole[1], whole[2]), (xyz, parts)


# ---- 4. one process per shard --------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _rank(rank, world, port, bases, off, nreads1, q):
    import sys
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from ebwt2snp_b200 import api as A, sharding as S
        ctx = A.Context(0)
        sh = S.shard_from_reads(ctx, bases, off, 1, 4, 1, "cpu")
        p = A.default_params(nreads1)
        mg, st, cnt, ids = S.hot_path_step(sh, p, 16, 2, "cpu")
        first_id, _ = ids.resolve()
        q.put((rank, sh.cluster_fetch_packed(), [bytes(e) for e in sh.events()], first_id, mg.n_clust_out, st.max_clust_length))
        sh.close()
        ctx.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_processes_gloo(ctx, world):
    bases, off = case_reads("genome")
    nreads1 = (len(off) - 1) // 2
    p = api.default_params(nreads1)
    whole = whole_outputs(ctx, bases, off, p, 16, 2, (1, 4, 1))
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    port = _free_port()
    procs = [mpc.Process(target=_rank, args=(r, world, port, bases, off, nreads1, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    got = sorted([q.get(timeout=600) for _ in range(world)], key=lambda t: t[0])
    for pr in procs:
        pr.join(timeout=120)
    assert all(pr.exitcode == 0 for pr in procs)
    assert b"".join(g[1] for g in got) == whole[1]
    assert sum((g[2] for g in got), []) == whole[2]
    ids = [1]
    for g in got[:-1]:
        ids.append(ids[-1] + len(g[2]))
    assert [g[3] for g in got] == ids
    assert all((g[4], g[5]) == (whole[0][1], whole[0][2]) for g in got)


# ---- 5. the CLI -------------------------------------------------------------------------------------------------------------
def test_cli_shards_equal_one_shard_and_the_chain(built, tmp_path):
    z = np.load(os.path.join(ROOT, "tests", "golden", "snp_vs_vcf.npz"))
    rs = synth.make_config("tiny", seed=21)
    fa = str(tmp_path / "ALL.fasta")
    synth.write_fasta(fa, rs.reads)
    w = ["-x", 1, "-y", 4, "-z", 1]
    chain = chain_outputs(fa, rs.nreads1, w, 16, 2, [])
    for g in (1, 2, 3, 8):
        assert ebwt2snp_outputs(fa, rs.nreads1, w, 16, 2, ["-G", g]) == chain, g
    r = tool("ebwt2snp", "-i", fa, "-n", rs.nreads1, "-G", 3)
    assert r.returncode == 0, r.stdout + r.stderr
    snp = str(tmp_path / "ALL.snp")
    assert open(snp, "rb").read() == z["0_calls"].tobytes()
    ref_fa, vcf = str(tmp_path / "ref.fasta"), str(tmp_path / "truth.vcf")
    open(ref_fa, "wb").write(z["0_fasta"].tobytes())
    open(vcf, "wb").write(z["0_vcf"].tobytes())
    import subprocess
    r = subprocess.run([os.path.join(BIN, "snp_vs_vcf"), "-v", vcf, "-c", snp, "-f", ref_fa], capture_output=True, timeout=120)
    assert r.returncode == 0 and b"TP = 39" in r.stdout and b"FP = 0" in r.stdout


def test_cli_c1_shards(built, tmp_path):
    rs = synth.make_config("C1", seed=1)
    fa = str(tmp_path / "C1.fasta")
    synth.write_fasta(fa, rs.reads)
    w = ["-x", 1, "-y", 4, "-z", 1]
    one = ebwt2snp_outputs(fa, rs.nreads1, w, 16, 2, [])
    for g in (2, 3, 8):
        assert ebwt2snp_outputs(fa, rs.nreads1, w, 16, 2, ["-G", g]) == one, g


def test_cli_too_many_shards_leaves_no_files(built, tmp_path):
    fa = tmp_path / "s.fasta"
    fa.write_text(">a\nACGTACGTTACG\n>b\nACGTACGTTACGT\n")
    r = tool("ebwt2snp", "-i", fa, "-n", 1, "-k", 4, "-G", 20)
    assert r.returncode != 0 and "too many shards" in r.stderr, r.stderr
    assert not os.path.exists(str(fa) + ".clusters") and not os.path.exists(str(tmp_path / "s.snp"))


def test_ranks_nccl_comm(built):
    """one process per GPU under torchrun, NCCL and the library's communicator (needs >= 2 GPUs; skipped otherwise)"""
    import subprocess
    import sys

    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    for world in sorted({2, min(n, 4)}):
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
                            "--master-addr", "127.0.0.1", "--master-port", str(29560 + world),
                            os.path.join(ROOT, "tests", "shards_from_reads_worker.py")], capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        assert f"OK {world}" in r.stdout, r.stdout

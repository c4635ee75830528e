"""-m gpu: reads to SNPs without an index file.  e2s_shard_build_egsa builds the index straight into a resident shard, and
e2s_pipeline_reads / the ebwt2snp CLI run both tools on it.  Checked against inputs the repository already trusts: shards
loaded from the oracle's index, e2s_pipeline_host on the records of the same index, and the three-tool chain
build_gesa -> ebwt2clust -> clust2snp."""
import os
import subprocess

import numpy as np
import pytest

from ebwt2snp_b200 import api, synth
from oracle import oracle as O
from tests import golden_util as GU
from tests.test_builder_gpu import ragged_from_genome
from tests.test_builder_ranges_gpu import host_slices, index_keys

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "ebwt2snp_b200", "bin")
ENV_HOOKS = ("E2S_BUILD_RANGE_RECORDS", "E2S_BUILD_IDS64", "E2S_NO_FUSED_PREFILTER")


@pytest.fixture(scope="module")
def ctx(built):
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(autouse=True)
def clean_env(monkeypatch):
    for k in ENV_HOOKS:
        monkeypatch.delenv(k, raising=False)


def flat(reads):
    """(bases, off) of an (R, L) read array"""
    R, L = reads.shape
    return np.ascontiguousarray(reads, dtype=np.uint8).reshape(-1), O.uniform_read_offsets(R, L)


def micro_variants():
    out = []
    for name in ("micro_a", "micro_b"):
        for vi in range(len(GU.micro(name)["variants"])):
            out.append((name, vi))
    return out


# ---- 1. built shard = loaded shard ----------------------------------------------------------------------------------------
def step_outputs(sh, p, k, m):
    """everything e2s_pipeline_resident leaves: (result fields, records, events, lcp bytes resident)"""
    res = sh.pipeline_resident(p, k, m)
    return ((res.n_written, res.n_clust_out, res.max_clust_length, bytes(res.snp)), sh.cluster_fetch_packed(),
            [bytes(e) for e in sh.events()], sh.lcp_bytes_resident())


def loaded_step(ctx, bases, off, want, p, k, m):
    n = want["n"]
    ctx.stage_reads(bases, off)
    sh = ctx.shard(n)
    sh.load_soa(want["lcp"], want["text"], want["suff"], want["bwt"])
    sh.seal()
    out = step_outputs(sh, p, k, m)
    sh.close()
    return out


def built_step(ctx, bases, off, p, k, m):
    n = int(off[-1]) + len(off) - 1
    ctx.stage_reads(bases, off)
    sh = ctx.shard(n)
    l0 = ctx.launches
    sh.build_egsa(off, 4, 4, 4)
    launches = ctx.launches - l0
    sh.seal()
    out = step_outputs(sh, p, k, m)
    sh.close()
    return out, launches


def case_reads(name):
    if name in ("micro_a", "micro_b"):
        return flat(GU.micro(name)["reads"])
    rng = np.random.default_rng({"genome": 101, "long": 102, "min_len_34": 103}[name])
    if name == "genome":  # ragged, empty reads included
        return ragged_from_genome(rng, 5_000, 2_000, 0, 150)
    if name == "long":  # LCP values above 127: saturated byte copy, and -k 128 on the 4-byte kernels
        return ragged_from_genome(rng, 20_000, 1_200, 130, 300)
    return ragged_from_genome(rng, 4_000, 1_500, 60, 120)


STEP_CASES = [("micro_a", 16, 2), ("micro_b", 16, 2), ("genome", 16, 2), ("long", 16, 2), ("long", 128, 2), ("min_len_34", 16, 34)]


@pytest.mark.parametrize("name,k,m", STEP_CASES)
def test_built_shard_equals_loaded_shard(ctx, monkeypatch, name, k, m):
    bases, off = case_reads(name)
    want = O.build_egsa_ragged(bases, off)
    n = want["n"]
    p = api.default_params(max(1, (len(off) - 1) // 2))
    ref = loaded_step(ctx, bases, off, want, p, k, m)
    if name == "long":
        assert int(want["lcp"].max()) > 127 and ref[3] == 1  # the saturated byte copy
    got, whole_launches = built_step(ctx, bases, off, p, k, m)
    assert got == ref, name
    # key ranges: a cap at which at least one starting slice holds more records than the cap (cut in two on the way), then 64-bit ids
    keys = np.sort(index_keys(bases, off, want))
    k0 = int(np.count_nonzero(keys == 0))

    def splits(c):
        return c > k0 and any(int(np.searchsorted(keys, hi) - np.searchsorted(keys, lo)) > c for lo, hi in host_slices(n, c))
    cap = next(n // d for d in range(2, 200) if splits(n // d))
    for env in ({"E2S_BUILD_RANGE_RECORDS": str(cap)}, {"E2S_BUILD_RANGE_RECORDS": str(cap), "E2S_BUILD_IDS64": "1"}, {"E2S_BUILD_IDS64": "1"}):
        for kk, v in env.items():
            monkeypatch.setenv(kk, v)
        got, launches = built_step(ctx, bases, off, p, k, m)
        for kk in env:
            monkeypatch.delenv(kk)
        assert got == ref, (name, env)
        if "E2S_BUILD_RANGE_RECORDS" in env:
            assert launches > whole_launches, (env, launches, whole_launches)  # the ranges were taken


# ---- 2. e2s_pipeline_reads = e2s_pipeline_host ------------------------------------------------------------------------------
def run_pipeline(fn):
    try:
        return 0, fn()
    except api.E2SError as e:
        return e.code, str(e)


def pipeline_outputs(ctx, call, n):
    """(0, (result fields, records, events), result) of a pipeline call on an index of n positions, or (error code, message)"""
    rec10 = np.zeros((n // 2 + 16) * 10, dtype=np.uint8)
    evbuf = (api.Event * (n // 50 + 1000))()
    rc, res = run_pipeline(lambda: call(rec10, evbuf))
    if rc:
        return rc, res
    m = res.n_written
    return 0, ((m, res.n_clust_out, res.max_clust_length, bytes(res.snp)), rec10[: m * 10].tobytes(),
               [bytes(e) for e in list(evbuf)[: res.snp.n_variants]]), res


def reads_vs_host(ctx, bases, off, egsa, p, k, m, x, y, z):
    """(outputs of e2s_pipeline_reads, outputs of e2s_pipeline_host on the x/y/z records of egsa, reads-call result)"""
    n = int(egsa["n"])
    rec = synth.gesa_records(egsa, x, y, z).view(np.uint8)
    host = pipeline_outputs(ctx, lambda r, e: ctx.pipeline_host(rec, n, bases, off, p, k, m, x, y, z, rec10=r, events=e), n)
    mine = pipeline_outputs(ctx, lambda r, e: ctx.pipeline_reads(bases, off, p, k, m, x, y, z, rec10=r, events=e), n)
    return mine, host


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("name,vi", micro_variants())
def test_pipeline_reads_equals_pipeline_host(ctx, monkeypatch, name, vi, fused):
    g = GU.micro(name)
    if not fused:
        monkeypatch.setenv("E2S_NO_FUSED_PREFILTER", "1")
    bases, off = flat(g["reads"])
    p = api.default_params(g["nreads1"], **GU.params_kw(g["variants"][vi]["args"]))
    for x, y, z in ((1, 4, 1), (4, 4, 4), (2, 4, 2)):
        mine, host = reads_vs_host(ctx, bases, off, g["egsa"], p, g["k"], g["m"], x, y, z)
        assert mine[0] == host[0], (x, y, z, mine[1], host[1])
        if mine[0]:
            continue
        assert mine[1] == host[1], (x, y, z)
        assert mine[2].h2d_bytes == bases.size + 8 * len(off)
        if (x, y, z) == (4, 4, 4):  # the golden outputs of the reference, 4/4/4 layout
            assert mine[1][1] == g["clusters"]


# ---- 3. field widths --------------------------------------------------------------------------------------------------------
def test_truncated_fields_equal_the_build_gesa_file(ctx, tmp_path):
    """300-base reads at -x 1 -z 1: lcp and suff wrap mod 256 in the .gesa build_gesa writes; the built shard keeps the same values"""
    rs = synth.make_read_set(G=20_000, reads_per_sample=1_500, L=300, n_snps=20, seed=5)
    fa = str(tmp_path / "ALL.fasta")
    synth.write_fasta(fa, rs.reads)
    r = subprocess.run([os.path.join(BIN, "build_gesa"), "-i", fa, "-x", "1", "-y", "4", "-z", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Warning: values do not fit" in r.stdout
    rec = np.fromfile(fa + ".gesa", dtype=np.uint8)
    bases, off = flat(rs.reads)
    n = int(off[-1]) + len(off) - 1
    assert rec.size == n * 7
    p = api.default_params(rs.nreads1)
    host = pipeline_outputs(ctx, lambda a, e: ctx.pipeline_host(rec, n, bases, off, p, 16, 2, 1, 4, 1, rec10=a, events=e), n)
    mine = pipeline_outputs(ctx, lambda a, e: ctx.pipeline_reads(bases, off, p, 16, 2, 1, 4, 1, rec10=a, events=e), n)
    assert host[0] == 0 and mine[0] == 0
    assert mine[1] == host[1]
    assert host[1][0][3] != bytes(api.SnpCounts())  # phase 2 found something to compare


# ---- 4. reuse ------------------------------------------------------------------------------------------------------------
def test_reuse_on_one_context(ctx):
    rng = np.random.default_rng(77)
    # a first set, a second of another n, a third of the second's n (its read lengths) with other bases
    sets = [ragged_from_genome(rng, 6_000, 1_500, 40, 120), ragged_from_genome(rng, 6_000, 900, 40, 120)]
    other, _ = ragged_from_genome(rng, 6_000, 900, 40, 120)
    sets.append((np.resize(other, int(sets[1][1][-1])), sets[1][1].copy()))
    assert not np.array_equal(sets[2][0], sets[1][0])
    p = api.default_params(400)

    def fresh(bases, off):
        c = api.Context(0)
        try:
            return mine(bases, off, c)
        finally:
            c.close()

    def mine(bases, off, c=ctx):
        n = int(off[-1]) + len(off) - 1
        return pipeline_outputs(c, lambda a, e: c.pipeline_reads(bases, off, p, 16, 2, rec10=a, events=e), n)

    for bases, off in sets:
        got, want = mine(bases, off), fresh(bases, off)
        assert got[0] == 0 and got[1] == want[1]
    # after a pipeline_host call on the same context (its chunked shard replaces the resident one)
    egsa = O.build_egsa_ragged(*sets[0])
    rec = synth.gesa_records(egsa, 1, 4, 1).view(np.uint8)
    n = egsa["n"]
    rc = pipeline_outputs(ctx, lambda a, e: ctx.pipeline_host(rec, n, sets[0][0], sets[0][1], p, 16, 2, 1, 4, 1, rec10=a, events=e), n)[0]
    assert rc == 0
    for bases, off in sets[:2]:
        got, want = mine(bases, off), fresh(bases, off)
        assert got[0] == 0 and got[1] == want[1]


# ---- 5. refusals and a nearly full device ------------------------------------------------------------------------------------
def test_base_outside_acgt_is_refused(ctx):
    bases = np.frombuffer(b"ACGTACGTAC" + b"ACGNACGTAC" + b"TTTTACGTAC", dtype=np.uint8).copy()
    off = O.uniform_read_offsets(3, 10)
    p = api.default_params(1)
    res_box = []
    rc, msg = run_pipeline(lambda: res_box.append(ctx.pipeline_reads(bases, off, p, 4, 2)))
    assert rc == 4 and "outside ACGT" in msg, (rc, msg)  # E2S_ERR_UNSUPPORTED
    assert not res_box


def test_nearly_full_device_builds_by_key_ranges(ctx):
    import torch
    rng = np.random.default_rng(45)
    bases, off = ragged_from_genome(rng, 2_000_000, 300_000, 60, 140)
    R = len(off) - 1
    n = int(off[R]) + R
    p = api.default_params(R // 2)
    call = lambda a, e: ctx.pipeline_reads(bases, off, p, 16, 2, rec10=a, events=e)  # noqa: E731
    l0 = ctx.launches
    want = pipeline_outputs(ctx, call, n)  # also leaves the resident shard of this n cached on the context
    whole_launches = ctx.launches - l0
    assert want[0] == 0
    dev = torch.device("cuda", ctx.device)
    torch.cuda.synchronize(dev)
    torch.cuda.empty_cache()
    leave = 300 << 20
    assert n * 25 > leave / 0.92 + (64 << 20)  # the whole build's scratch does not fit what is left
    hold = None
    try:
        free, _ = torch.cuda.mem_get_info(dev)
        assert free > leave + (1 << 30), free
        hold = torch.empty(free - leave, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        l0 = ctx.launches
        got = pipeline_outputs(ctx, call, n)
        launches = ctx.launches - l0
    finally:
        del hold
        torch.cuda.empty_cache()
    assert got[0] == 0, got[1]
    assert launches > whole_launches, (launches, whole_launches)
    assert got[1] == want[1]


# ---- 6. the CLI -------------------------------------------------------------------------------------------------------------
def tool(name, *args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([os.path.join(BIN, name), *[str(a) for a in args]], capture_output=True, text=True, env=e, timeout=600)


def chain_outputs(fa, nreads1, w, k, m, opts):
    """(.clusters, .snp or None, stdout Done lines) of build_gesa -> ebwt2clust -> clust2snp, files removed afterwards"""
    snp = fa.rsplit(".fast", 1)[0] + ".snp"
    r0 = tool("build_gesa", "-i", fa, *w)
    assert r0.returncode == 0, r0.stdout + r0.stderr
    r1 = tool("ebwt2clust", "-i", fa, "-k", k, "-m", m, *w)
    assert r1.returncode == 0, r1.stderr
    r2 = tool("clust2snp", "-i", fa, "-n", nreads1, *w, *opts)
    out = (open(fa + ".clusters", "rb").read(), open(snp, "rb").read() if os.path.exists(snp) else None, r2.returncode,
           [ln for ln in (r1.stdout + r2.stdout).splitlines() if ln.startswith("Done. ") and ln != "Done. "])
    for f in (fa + ".gesa", fa + ".clusters", snp):
        if os.path.exists(f):
            os.remove(f)
    return out


def ebwt2snp_outputs(fa, nreads1, w, k, m, opts):
    snp = fa.rsplit(".fast", 1)[0] + ".snp"
    r = tool("ebwt2snp", "-i", fa, "-n", nreads1, "-k", k, "-l", m, *w, *opts)
    assert r.returncode in (0, 3), r.stdout + r.stderr
    assert not os.path.exists(fa + ".gesa")
    out = (open(fa + ".clusters", "rb").read(), open(snp, "rb").read() if os.path.exists(snp) else None, r.returncode,
           [ln for ln in r.stdout.splitlines() if ln.startswith("Done. ")])
    for f in (fa + ".clusters", snp):
        if os.path.exists(f):
            os.remove(f)
    return out


def write_fasta_ragged(path, bases, off, wrap=None):
    with open(path, "w") as f:
        for r in range(len(off) - 1):
            seq = bases[int(off[r]):int(off[r + 1])].tobytes().decode()
            f.write(f">read{r} description\n")
            step = wrap or max(len(seq), 1)
            for a in range(0, len(seq), step):
                f.write(seq[a:a + step] + "\n")
            if not seq:
                f.write("\n")


def test_cli_equals_the_three_tool_chain(built, tmp_path):
    g = GU.micro("micro_a")
    fa = str(tmp_path / "micro_a.fasta")
    synth.write_fasta(fa, g["reads"])
    option_sets = [[], g["variants"][-1]["args"]]
    for w in (["-x", 1, "-y", 4, "-z", 1], ["-x", 4, "-y", 4, "-z", 4]):
        for opts in option_sets:
            mine = ebwt2snp_outputs(fa, g["nreads1"], w, g["k"], g["m"], opts)
            assert mine == chain_outputs(fa, g["nreads1"], w, g["k"], g["m"], opts), (w, opts)
            assert mine[1] is not None or mine[2] == 3
    mine = ebwt2snp_outputs(fa, g["nreads1"], ["-x", 4, "-y", 4, "-z", 4], g["k"], g["m"], [])
    assert mine[0] == g["clusters"] and mine[1] == g["variants"][0]["snp"]
    # ragged reads with empty ones, then the same FASTA wrapped over several lines
    rng = np.random.default_rng(9)
    bases, off = ragged_from_genome(rng, 8_000, 2_400, 0, 150)
    for wrap in (None, 23):
        fa = str(tmp_path / f"ragged{wrap}.fasta")
        write_fasta_ragged(fa, bases, off, wrap)
        for w in (["-x", 1, "-y", 4, "-z", 1], ["-x", 4, "-y", 4, "-z", 4]):
            mine = ebwt2snp_outputs(fa, 1_200, w, 16, 2, [])
            assert mine == chain_outputs(fa, 1_200, w, 16, 2, []), (wrap, w)


def test_cli_against_the_reference_binaries(built, tmp_path):
    if not O.ref_available():
        pytest.skip("oracle/_ref not built")
    rs = synth.make_config("tiny", seed=11)
    fa = str(tmp_path / "ALL.fasta")
    synth.write_fasta(fa, rs.reads)
    mine = ebwt2snp_outputs(fa, rs.nreads1, ["-x", 1, "-y", 4, "-z", 1], 16, 2, [])
    assert tool("build_gesa", "-i", fa, "-x", 1, "-y", 4, "-z", 1).returncode == 0
    ref = os.path.join(ROOT, "oracle", "_ref")
    r1 = subprocess.run([os.path.join(ref, "ebwt2clust"), "-i", fa, "-x", "1", "-y", "4", "-z", "1"], capture_output=True, text=True, timeout=600)
    r2 = subprocess.run([os.path.join(ref, "clust2snp"), "-i", fa, "-n", str(rs.nreads1), "-x", "1", "-y", "4", "-z", "1"],
                        capture_output=True, text=True, timeout=600)
    assert r1.returncode == 0 and r2.returncode == 0
    assert open(fa + ".clusters", "rb").read() == mine[0]
    assert open(str(tmp_path / "ALL.snp"), "rb").read() == mine[1]


def test_cli_reads_to_scores(built, tmp_path):
    """the read set of the three-tool end-to-end test: ebwt2snp alone gives its golden .snp and the same snp_vs_vcf scores"""
    z = np.load(os.path.join(ROOT, "tests", "golden", "snp_vs_vcf.npz"))
    rs = synth.make_config("tiny", seed=21)
    fa = str(tmp_path / "ALL.fasta")
    synth.write_fasta(fa, rs.reads)
    r = tool("ebwt2snp", "-i", fa, "-n", rs.nreads1)
    assert r.returncode == 0, r.stdout + r.stderr
    assert not os.path.exists(fa + ".gesa")
    snp = str(tmp_path / "ALL.snp")
    assert open(snp, "rb").read() == z["0_calls"].tobytes()
    ref_fa, vcf = str(tmp_path / "ref.fasta"), str(tmp_path / "truth.vcf")
    open(ref_fa, "wb").write(z["0_fasta"].tobytes())
    open(vcf, "wb").write(z["0_vcf"].tobytes())
    r = subprocess.run([os.path.join(BIN, "snp_vs_vcf"), "-v", vcf, "-c", snp, "-f", ref_fa], capture_output=True, timeout=120)
    assert r.returncode == 0 and b"TP = 39" in r.stdout and b"FP = 0" in r.stdout


def test_cli_refusal_leaves_no_files(built, tmp_path):
    fa = tmp_path / "n.fasta"
    fa.write_text(">a\nACGTACGTNACGT\n>b\nACGTACGTTACGT\n")
    r = tool("ebwt2snp", "-i", fa, "-n", 1, "-k", 4)
    assert r.returncode != 0 and "outside ACGT" in r.stderr
    assert not os.path.exists(str(fa) + ".clusters") and not os.path.exists(str(tmp_path / "n.snp"))


# ---- 7. C1 whole ------------------------------------------------------------------------------------------------------------
def test_c1_from_reads(ctx):
    rs = synth.make_config("C1", seed=1)
    e = synth.build_egsa(rs.reads, device="cuda")
    eg = {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in e.items()}
    del e
    bases, off = flat(rs.reads)
    p = api.default_params(rs.nreads1)
    mine, host = reads_vs_host(ctx, bases, off, eg, p, 16, 2, 1, 4, 1)
    assert mine[0] == 0 and host[0] == 0
    assert mine[1] == host[1]
    assert mine[1][0][3] != bytes(api.SnpCounts())

"""-m gpu: the two drop-in CLIs, file against file, with the committed outputs of the UNMODIFIED reference
(tests/golden) and -- where oracle/_ref is present -- with the reference run live on the same files."""
import os
import subprocess

import numpy as np
import pytest

from ebwt2snp_b200 import synth
from oracle import oracle as O
from tests import golden_util as GU
from tests import helpers as H

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "ebwt2snp_b200", "bin")


def run(tool, *args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([os.path.join(BIN, tool), *[str(a) for a in args]], capture_output=True, text=True, env=e, timeout=600)


def write_index(d, g, lay):
    rs = synth.ReadSet(reads=g["reads"], nreads1=g["nreads1"], genome1=None, genome2=None, snp_pos=None, indels=[])
    return synth.write_dataset(str(d), rs, g["egsa"], name=g["name"] + ".fasta", x=lay["x"], y=lay["y"], z=lay["z"], bcr=lay["bcr"])


def stdout_value(out, prefix, cast=int, field=1):
    for line in out.splitlines():
        if line.startswith(prefix):
            return cast(line.split()[field])
    return None


@pytest.mark.parametrize("name", ["micro_a", "micro_b"])
def test_cli_default_layout_all_option_sets(built, tmp_path, name):
    g = GU.micro(name)
    lay = dict(x=4, y=4, z=4, bcr=False)
    fa = write_index(tmp_path, g, lay)
    r = run("ebwt2clust", "-i", fa, "-k", g["k"], "-m", g["m"], "-x", 4, "-y", 4, "-z", 4)
    assert r.returncode == 0, r.stderr
    assert open(fa + ".clusters", "rb").read() == g["clusters"]
    assert f"This is ebwt2clust. Input file: {fa}" in r.stdout
    assert stdout_value(r.stdout, "Done. ") == g["n_clust_out"]  # ref:ebwt2clust.cpp:137
    snp = os.path.join(str(tmp_path), name + ".snp")  # X cut at the last ".fast" + ".snp" (ref:clust2snp.cpp:1074-1076)
    for v in g["variants"]:
        if os.path.exists(snp):
            os.remove(snp)
        r = run("clust2snp", "-i", fa, "-n", g["nreads1"], "-x", 4, "-y", 4, "-z", 4, *v["args"])
        assert f"Cluster sizes allowed: [{v['allowed'][0]},{v['allowed'][1]}]" in r.stdout, v["args"]
        if v["rc"] == 0:
            assert r.returncode == 0, r.stderr
            assert stdout_value(r.stdout, "Done. ") == v["ncand"]
            assert open(snp, "rb").read() == v["snp"], v["args"]
            assert r.stdout.rstrip().endswith("Done.")
        else:  # the reference segfaults on zero candidates (ref:clust2snp.cpp:531): clean exit 3, no .snp
            assert r.returncode == 3 and not os.path.exists(snp)


@pytest.mark.parametrize("name", ["micro_a", "micro_b"])
def test_cli_other_layouts(built, tmp_path, name):
    """narrow / 8-byte field widths and the BCR triple (ref:include.hpp:157-188): same outputs as the reference"""
    g = GU.micro(name)
    for j, lay in enumerate(g["layouts"]):
        d = tmp_path / f"lay{j}"
        fa = write_index(d, g, lay)
        w = ["-x", lay["x"], "-y", lay["y"], "-z", lay["z"]]
        r = run("ebwt2clust", "-i", fa, "-k", g["k"], "-m", g["m"], *w)
        assert r.returncode == 0, r.stderr
        assert open(fa + ".clusters", "rb").read() == lay["clusters"], lay
        assert stdout_value(r.stdout, "Done. ") == lay["n_clust_out"]
        r = run("clust2snp", "-i", fa, "-n", g["nreads1"], *w)
        assert r.returncode == 0, r.stderr
        assert stdout_value(r.stdout, "Done. ") == lay["ncand"]
        assert open(os.path.join(str(d), name + ".snp"), "rb").read() == lay["snp"], lay


@pytest.mark.parametrize("name", ["micro_a", "micro_b"])
def test_cli_clust2snp_streamed(built, tmp_path, name):
    """clust2snp with the index STREAMED through a chunked shard (what it does for an index larger than device memory;
    E2S_CLI_STREAM=1 forces it): every option set and layout -- EGSA and the BCR triple, whose pairSA is then only read for the
    prefilter's survivors -- gives the reference's .snp"""
    g = GU.micro(name)
    env = {"E2S_CLI_STREAM": "1", "E2S_CHUNK_POSITIONS": "20000"}
    fa = write_index(tmp_path / "d", g, dict(x=4, y=4, z=4, bcr=False))
    assert run("ebwt2clust", "-i", fa, "-k", g["k"], "-m", g["m"], "-x", 4, "-y", 4, "-z", 4).returncode == 0
    snp = os.path.join(str(tmp_path / "d"), name + ".snp")
    for v in g["variants"]:
        if os.path.exists(snp):
            os.remove(snp)
        r = run("clust2snp", "-i", fa, "-n", g["nreads1"], "-x", 4, "-y", 4, "-z", 4, *v["args"], env=env)
        assert f"Cluster sizes allowed: [{v['allowed'][0]},{v['allowed'][1]}]" in r.stdout, v["args"]
        if v["rc"] == 0:
            assert r.returncode == 0, r.stderr
            assert stdout_value(r.stdout, "Done. ") == v["ncand"]
            assert open(snp, "rb").read() == v["snp"], v["args"]
        else:
            assert r.returncode == 3 and not os.path.exists(snp)
    for j, lay in enumerate(g["layouts"]):
        d = tmp_path / f"lay{j}"
        fa = write_index(d, g, lay)
        w = ["-x", lay["x"], "-y", lay["y"], "-z", lay["z"]]
        assert run("ebwt2clust", "-i", fa, "-k", g["k"], "-m", g["m"], *w, env=env).returncode == 0
        assert open(fa + ".clusters", "rb").read() == lay["clusters"], lay
        r = run("clust2snp", "-i", fa, "-n", g["nreads1"], *w, env=env)
        assert r.returncode == 0, (lay, r.stderr)
        assert stdout_value(r.stdout, "Done. ") == lay["ncand"]
        assert open(os.path.join(str(d), name + ".snp"), "rb").read() == lay["snp"], lay


def test_cli_sharded_on_one_box(built, tmp_path):
    """E2S_GPUS=N shards the eBWT over N devices; outputs must not depend on N (runs with every N the box offers)"""
    import torch
    g = GU.micro("micro_a")
    fa = write_index(tmp_path, g, dict(x=4, y=4, z=4, bcr=False))
    for n_gpu in sorted({1, min(2, torch.cuda.device_count()), torch.cuda.device_count()}):
        env = {"E2S_GPUS": str(n_gpu)}
        r = run("ebwt2clust", "-i", fa, "-k", g["k"], "-m", g["m"], "-x", 4, "-y", 4, "-z", 4, env=env)
        assert r.returncode == 0, r.stderr
        assert open(fa + ".clusters", "rb").read() == g["clusters"], n_gpu
        r = run("clust2snp", "-i", fa, "-n", g["nreads1"], "-x", 4, "-y", 4, "-z", 4, env=env)
        assert r.returncode == 0, r.stderr
        assert open(os.path.join(str(tmp_path), "micro_a.snp"), "rb").read() == g["variants"][0]["snp"], n_gpu


def test_cli_live_vs_reference(built, tmp_path):
    """a fresh seeded read set (not one of the fixtures): reference (oracle/_ref where it is built, else the oracle's
    restatement of it) and B200 CLIs on the same files"""
    rs = synth.make_read_set(G=30_000, reads_per_sample=6_000, L=100, n_snps=60, n_indels=10, rc=True, seed=321)
    e = synth.build_egsa(rs.reads)
    eg = {k: (v.numpy() if hasattr(v, "numpy") else v) for k, v in e.items()}
    ref_dir, our_dir = tmp_path / "ref", tmp_path / "b200"
    fa_ref = synth.write_dataset(str(ref_dir), rs, eg)
    fa_our = synth.write_dataset(str(our_dir), rs, eg)
    ref_cl, ref_snp, ncl, info = H.reference_outputs(fa_ref, eg, rs.reads, rs.nreads1)
    assert info["returncode"] == 0
    o1 = run("ebwt2clust", "-i", fa_our, "-x", 4, "-y", 4, "-z", 4)
    o2 = run("clust2snp", "-i", fa_our, "-n", rs.nreads1, "-x", 4, "-y", 4, "-z", 4)
    assert o1.returncode == 0 and o2.returncode == 0, (o1.stderr, o2.stderr)
    assert open(fa_our + ".clusters", "rb").read() == ref_cl
    assert open(os.path.join(str(our_dir), "ALL.snp"), "rb").read() == ref_snp
    assert stdout_value(o1.stdout, "Done. ") == ncl
    assert stdout_value(o2.stdout, "Done. ") == info["n_candidates"]
    assert f"Cluster sizes allowed: [{info['allowed'][0]},{info['allowed'][1]}]" in o2.stdout
    if "stdout" not in info:  # the restatement prints nothing
        return
    # the histogram block of statistics() is printed identically (ref:clust2snp.cpp:916-934)
    def hist_block(out):
        lines = out.splitlines()
        a = next(i for i, ln in enumerate(lines) if ln.startswith("cluster length"))
        b = next(i for i, ln in enumerate(lines) if ln.startswith("Cluster sizes allowed"))
        return lines[a:b + 1]
    assert hist_block(o2.stdout) == hist_block(info["stdout"])


def test_cli_multiline_fasta(built, tmp_path):
    """the FASTA may wrap its sequences over several lines (ref:clust2snp.cpp:166-171,187-192); same .snp"""
    g = GU.micro("micro_b")
    fa = write_index(tmp_path, g, dict(x=4, y=4, z=4, bcr=False))
    with open(fa, "w") as f:
        for i, r in enumerate(g["reads"]):
            seq = r.tobytes().decode()
            f.write(f">read{i} some description\n")
            for a in range(0, len(seq), 23):
                f.write(seq[a:a + 23] + "\n")
    assert run("ebwt2clust", "-i", fa, "-k", g["k"], "-m", g["m"], "-x", 4, "-y", 4, "-z", 4).returncode == 0
    r = run("clust2snp", "-i", fa, "-n", g["nreads1"], "-x", 4, "-y", 4, "-z", 4)
    assert r.returncode == 0, r.stderr
    assert open(os.path.join(str(tmp_path), "micro_b.snp"), "rb").read() == g["variants"][0]["snp"]


def test_build_gesa_cli_feeds_both_tool_chains(built, tmp_path):
    """build_gesa (index construction on the GPU, SURVEY.md 8(f) rank 1) writes the files the tools look for: byte-identical
    to the synthetic-data writer for the egsa default layout 4/1/1 (ref:pipeline.sh:30-32), 4/4/4 and the BCR triple; the
    UNMODIFIED reference tools run on its output give the same .clusters / .snp as this repository's tools."""
    rs = synth.make_config("tiny", seed=11)
    e = synth.build_egsa(rs.reads)
    for j, (x, y, z, bcr) in enumerate([(1, 4, 1, False), (4, 4, 4, False), (2, 4, 2, True)]):
        d = tmp_path / f"b{j}"
        want = synth.write_dataset(str(d / "want"), rs, e, x=x, y=y, z=z, bcr=bcr)
        os.makedirs(d / "got")
        fa = str(d / "got" / "ALL.fasta")
        synth.write_fasta(fa, rs.reads)
        r = run("build_gesa", "-i", fa, "-x", x, "-y", y, "-z", z, *(["-b"] if bcr else []))
        assert r.returncode == 0, r.stdout + r.stderr
        assert f"Done. {e['n']} suffixes of {rs.reads.shape[0]} reads indexed." in r.stdout
        for ext in ((".out", ".out.lcp", ".out.pairSA") if bcr else (".gesa",)):
            assert open(fa + ext, "rb").read() == open(want + ext, "rb").read(), (x, y, z, bcr, ext)
    # the 4/1/1 index through both tool chains
    fa = str(tmp_path / "b0" / "got" / "ALL.fasta")
    w = ["-x", 1, "-y", 4, "-z", 1]
    r = run("ebwt2clust", "-i", fa, *w)
    assert r.returncode == 0, r.stderr
    mine_cl = open(fa + ".clusters", "rb").read()
    r = run("clust2snp", "-i", fa, "-n", rs.nreads1, *w)
    assert r.returncode == 0, r.stderr
    mine_snp = open(str(tmp_path / "b0" / "got" / "ALL.snp"), "rb").read()
    assert len(mine_snp) > 0
    if O.ref_available():
        for f in (fa + ".clusters", str(tmp_path / "b0" / "got" / "ALL.snp")):
            os.remove(f)
        ref = os.path.join(ROOT, "oracle", "_ref")
        r1 = subprocess.run([os.path.join(ref, "ebwt2clust"), "-i", fa, "-x", "1", "-y", "4", "-z", "1"], capture_output=True, text=True, timeout=600)
        assert r1.returncode == 0
        assert open(fa + ".clusters", "rb").read() == mine_cl
        r2 = subprocess.run([os.path.join(ref, "clust2snp"), "-i", fa, "-n", str(rs.nreads1), "-x", "1", "-y", "4", "-z", "1"],
                            capture_output=True, text=True, timeout=600)
        assert r2.returncode == 0
        assert open(str(tmp_path / "b0" / "got" / "ALL.snp"), "rb").read() == mine_snp


def test_reads_to_scores_with_the_tools_alone(built, tmp_path):
    """the reference's pipeline.sh end to end with this repository's tools only (ref:pipeline.sh:98-140): reads FASTA ->
    build_gesa (4/1/1, egsa's default layout) -> ebwt2clust -> clust2snp -> snp_vs_vcf against the planted truth.  The .snp
    equals the one the snp_vs_vcf golden fixture was made from (the oracle's), so the scores equal the reference tool's."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "snp_vs_vcf.npz"))
    assert str(z["0_name"]) == "planted"
    rs = synth.make_config("tiny", seed=21)  # the read set of tests/golden/make_golden.py:snp_vs_vcf_inputs
    fa = str(tmp_path / "ALL.fasta")
    synth.write_fasta(fa, rs.reads)
    w = ["-x", 1, "-y", 4, "-z", 1]
    assert run("build_gesa", "-i", fa, *w).returncode == 0
    assert run("ebwt2clust", "-i", fa, *w).returncode == 0
    assert run("clust2snp", "-i", fa, "-n", rs.nreads1, *w).returncode == 0
    snp = str(tmp_path / "ALL.snp")
    assert open(snp, "rb").read() == z["0_calls"].tobytes()
    ref_fa, vcf = str(tmp_path / "ref.fasta"), str(tmp_path / "truth.vcf")
    open(ref_fa, "wb").write(z["0_fasta"].tobytes())
    open(vcf, "wb").write(z["0_vcf"].tobytes())
    r = subprocess.run([os.path.join(BIN, "snp_vs_vcf"), "-v", vcf, "-c", snp, "-f", ref_fa], capture_output=True, timeout=120)
    assert r.returncode == 0 and r.stdout == z["0_stdout"].tobytes()
    assert b"TP = 39" in r.stdout and b"FP = 0" in r.stdout

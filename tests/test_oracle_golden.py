"""not gpu: the oracle restatement (oracle/oracle.c) against the golden vectors produced by the unmodified
reference, against the reference's own two known answers, and -- where oracle/_ref is present -- live."""
import os
import tempfile

import numpy as np
import pytest

from oracle import oracle as O
from tests import golden_util as GU
from tests import helpers as H


def test_phase1_golden(built):
    n = 0
    for c in GU.phase1_cases():
        s, l, ncl, _ = O.cluster_lm(c["lcp"], c["bwt"], c["k"], c["m"])
        assert O.clusters_to_bytes(s, l) == c["clusters"]
        assert ncl == c["n_clust_out"]
        n += 1
    assert n == 72


def test_phase1_widths_golden(built):
    """-x 1 / 2 / 8: the phantom LCP is truncated to the field width"""
    n = 0
    for c in GU.phase1_width_cases():
        s, l, ncl, _ = O.cluster_lm(c["lcp"], c["bwt"], c["k"], c["m"], x=c["x"])
        assert O.clusters_to_bytes(s, l) == c["clusters"] and ncl == c["n_clust_out"], (c["x"], c["y"], c["z"], n)
        n += 1
    assert n == 96


def test_phantom_tail_golden(built):
    """the phantom record's fields for 11 width combinations x {EGSA, BCR}, read out of the reference through -n"""
    n = 0
    for c in GU.phantom_tail_cases():
        s, l, _, _ = O.cluster_lm(c["lcp"], c["bwt"], 16, 2, x=c["x"])
        assert O.clusters_to_bytes(s, l) == c["clusters"]
        reads = np.frombuffer(b"ACGT", dtype=np.uint8).reshape(1, 4)
        for n1, ncand in c["readouts"]:
            p = O.default_params(n1, k_left=1, k_right=1, max_gap=1)  # -g only matters after the count is printed
            st = O.statistics(s, l, p.mcov_out, p.pval)
            _, res = O.find_events(c["lcp"], c["text"], c["suff"], c["bwt"], s, l, p, st.max_clust_length, reads,
                                   O.uniform_read_offsets(1, 4), x=c["x"], y=c["y"], z=c["z"], bcr=c["bcr"], strict=False)
            assert res.n_candidates == ncand, (c["x"], c["y"], c["z"], c["bcr"], n1)
            n += 1
    assert n == 132


@pytest.mark.parametrize("name", ["micro_a", "micro_b"])
def test_micro_layouts_golden(built, name):
    """the same read sets through narrow-field .gesa files and the BCR triple (SURVEY.md 8(f) row 2)"""
    g = GU.micro(name)
    e = g["egsa"]
    off = O.uniform_read_offsets(*g["reads"].shape)
    for lay in g["layouts"]:
        s, l, ncl, _ = O.cluster_lm(e["lcp"], e["bwt"], g["k"], g["m"], x=lay["x"])
        assert O.clusters_to_bytes(s, l) == lay["clusters"] and ncl == lay["n_clust_out"], lay
        p = O.default_params(g["nreads1"])
        st = O.statistics(s, l, p.mcov_out, p.pval)
        assert (2 * p.mcov_out, st.max_clust_length) == lay["allowed"]
        text, res = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], s, l, p, st.max_clust_length, g["reads"], off,
                                  x=lay["x"], y=lay["y"], z=lay["z"], bcr=lay["bcr"])
        assert lay["rc"] == 0 and res.n_candidates == lay["ncand"] and text == lay["snp"]


@pytest.mark.parametrize("name", ["micro_a", "micro_b"])
def test_micro_golden(built, name):
    g = GU.micro(name)
    e = g["egsa"]
    s, l, ncl, _ = O.cluster_lm(e["lcp"], e["bwt"], g["k"], g["m"])
    assert O.clusters_to_bytes(s, l) == g["clusters"] and ncl == g["n_clust_out"]
    off = O.uniform_read_offsets(*g["reads"].shape)
    for v in g["variants"]:
        p = O.default_params(g["nreads1"], **GU.params_kw(v["args"]))
        st = O.statistics(s, l, p.mcov_out, p.pval)
        assert (2 * p.mcov_out, st.max_clust_length) == v["allowed"]
        text, res = O.find_events(e["lcp"], e["text"], e["suff"], e["bwt"], s, l, p, st.max_clust_length, g["reads"], off)
        if v["rc"] == 0:
            assert res.n_candidates == v["ncand"] and text == v["snp"], v["args"]
        else:  # the reference crashed: zero candidates (ref:clust2snp.cpp:531)
            assert res.n_candidates == 0


def test_distance_known_answers(built):
    # the only golden vectors in the reference tree: ref:clust2snp.cpp:250-251
    for g in (2, 3, 8):
        assert O.distance(b"ACCTACTG", b"TTACTTAC", g) == (1, 2)
        assert O.distance(b"TTACTTAC", b"ACCTACTG", g) == (1, -2)
    assert O.distance(b"ACGTACGT", b"ACGTACGT", 10 if False else 8) == (0, 0)


@pytest.mark.skipif(not O.ref_available(), reason="oracle/_ref not built")
def test_phase1_live_vs_reference(built):
    rng = np.random.default_rng(5)
    dt = np.dtype([("text", "<u4"), ("suff", "<u4"), ("lcp", "<u4"), ("bwt", "u1")])
    with tempfile.TemporaryDirectory() as d:
        fa = os.path.join(d, "X.fasta")
        open(fa, "w").write(">a\nA\n")
        for it in range(40):
            n = int(rng.integers(2, 2000))
            k = int(rng.choice([1, 2, 3, 5, 16, 70]))
            m = int(rng.choice([1, 2, 3, 8]))
            lcp = H.random_lcp(rng, n, k, it % 5)
            bwt = rng.choice(H.BWT_ALPHABET, size=n)
            rec = np.zeros(n, dtype=dt)
            rec["lcp"], rec["bwt"] = lcp, bwt
            rec.tofile(fa + ".gesa")
            r, ncl = O.ref_ebwt2clust(fa, k=k, m=m)
            s, l, nc, _ = O.cluster_lm(lcp, bwt, k, m)
            assert O.clusters_to_bytes(s, l) == open(fa + ".clusters", "rb").read() and nc == ncl


def test_reference_build_matches_the_goldens():
    """The phantom record (the one value of the goldens that depends on how the reference was compiled) is pinned for the
    compiler named in tests/golden/REFERENCE_BUILD.txt: with another g++ the live-reference comparisons of the tail may
    differ, which is the reference's undefined behaviour, not a regression -- warn loudly instead of failing."""
    import os
    import subprocess
    import warnings
    here = os.path.dirname(os.path.abspath(__file__))
    txt = open(os.path.join(here, "golden", "REFERENCE_BUILD.txt")).read()
    want = [l.split(":", 1)[1].strip() for l in txt.splitlines() if l.strip().startswith("compiler:")][0]
    try:
        have = subprocess.run(["g++", "--version"], capture_output=True, text=True, timeout=30).stdout.splitlines()[0].strip()
    except Exception:
        return  # no compiler here (the GPU box uses the prebuilt oracle/_ref)
    if have != want:
        warnings.warn(f"oracle/_ref would be built by '{have}', the goldens were made with '{want}': the post-EOF phantom record "
                      f"may differ (tests/golden/REFERENCE_BUILD.txt)")
    flags = [l.split(":", 1)[1].strip() for l in txt.splitlines() if l.strip().startswith("flags:")][0]
    mk = open(os.path.join(os.path.dirname(here), "oracle", "Makefile")).read()
    for f in flags.split("(")[0].split():
        assert f in mk, f


def test_reference_outputs_with_the_binaries(tmp_path, monkeypatch):
    """tests/helpers.py:reference_outputs where oracle/_ref is built: clust2snp reads the .clusters ebwt2clust wrote, its stdout
    comes back with the outputs, and both output files are gone afterwards (stand-in tools with the reference's file contract)"""
    ref = tmp_path / "_ref"
    ref.mkdir()
    tools = {
        "ebwt2clust": 'printf "CLUSTERS" > "$2.clusters"; echo "Done. 7 clusters saved to file."',
        "clust2snp": 'cat "$2.clusters" > /dev/null || exit 1; printf "SNP" > "${2%.fasta}.snp"; '
                     'echo "Cluster sizes allowed: [10,42]"; echo "Done. 3 potential variants found."',
    }
    for name, body in tools.items():
        (ref / name).write_text("#!/bin/sh\n" + body + "\n")
        (ref / name).chmod(0o755)
    monkeypatch.setattr(O, "REF_DIR", str(ref))
    assert O.ref_available()
    fa = str(tmp_path / "ALL.fasta")
    open(fa, "w").write(">r0\nACGT\n")
    cl, snp, ncl, info = H.reference_outputs(fa, None, None, 1)
    assert (cl, snp, ncl) == (b"CLUSTERS", b"SNP", 7)
    assert info["returncode"] == 0 and info["allowed"] == (10, 42) and info["n_candidates"] == 3
    assert "Cluster sizes allowed: [10,42]" in info["stdout"]
    assert not os.path.exists(fa + ".clusters") and not os.path.exists(str(tmp_path / "ALL.snp"))

"""not gpu: the parts of reads-to-SNPs over several shards that are decided before any GPU work: the CLI's -G option and the halo
row size the library reports."""
import os
import subprocess

from ebwt2snp_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "ebwt2snp_b200", "bin")


def run(*args):
    e = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    return subprocess.run([os.path.join(BIN, "ebwt2snp"), *[str(a) for a in args]], capture_output=True, text=True, env=e, timeout=120)


def test_help_lists_shards(built):
    h = run("-h").stdout
    assert "-G <arg>" in h and "E2S_GPUS is\nignored" in h


def test_bad_shard_count_exits_before_the_device(built, tmp_path):
    fa = tmp_path / "r.fasta"
    fa.write_text(">a\nACGT\n")
    for g in (0, -3):
        r = run("-i", fa, "-n", 1, "-G", g)
        assert r.returncode == 2 and "-G must be at least 1" in r.stderr, (g, r.stderr)
    assert not os.path.exists(str(fa) + ".clusters") and not os.path.exists(str(tmp_path / "r.snp"))


def test_halo_row_words(built):
    # n_local, global_off, first and last suffix ids, then the last 2 and the first 151 records at 2 words each
    assert api.HALO_ROW_WORDS == api.halo_row_words() == 4 + 2 * (2 + api.MAX_C_LEN + 1)

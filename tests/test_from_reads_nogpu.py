"""not gpu: ebwt2snp (reads to SNPs in one process) behaviour that is decided before any GPU work."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "ebwt2snp_b200", "bin")


def run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([os.path.join(BIN, "ebwt2snp"), *[str(a) for a in args]], capture_output=True, text=True, env=e, timeout=120)


def test_help_exits_zero(built):
    for args in ([], ["-h"], ["-Q"], ["-i", "x.fasta"], ["-n", "5"], ["-i", "x.fasta", "-n", "0"], ["-i", "x", "-n", "3", "-b"]):
        r = run(*args)
        assert r.returncode == 0 and "ebwt2snp [options]" in r.stdout, args
    h = run("-h").stdout
    for flag in ("-k <arg>", "-l <arg>", "-m <arg>", "-x <arg>", "E2S_GPUS is\nignored"):
        assert flag in h, flag


def test_missing_fasta_exits_one_without_a_device(built, tmp_path):
    fa = str(tmp_path / "none.fasta")
    r = run("-i", fa, "-n", 5, env={"CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode == 1 and f"Error: could not read {fa}" in r.stdout
    assert not os.path.exists(fa + ".clusters") and not os.path.exists(str(tmp_path / "none.snp"))


def test_bad_field_width_exits_before_the_device(built, tmp_path):
    fa = tmp_path / "r.fasta"
    fa.write_text(">a\nACGT\n")
    r = run("-i", fa, "-n", 1, "-x", 3, env={"CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode == 2 and "-x/-y/-z must be 1, 2, 4 or 8" in r.stderr
    assert not os.path.exists(str(fa) + ".clusters")
